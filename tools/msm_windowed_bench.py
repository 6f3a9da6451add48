"""Plain against windowed prepared MSM bases, side by side (B200).

    python tools/msm_windowed_bench.py OUT_DIR [--logn 10,16,20,22,24] [--c 16,18,20,21,22]

For every size n = 2^logn: P_i = a_i G (fixed-base kernel, projective Elements), seeded
random canonical scalars s_i.  One plain set (d377_msm_bases_create) and one windowed set per
window width (c = 0, the library's choice, plus every width of --c) are created and measured:

  create_ms          host wall clock around the creation (ends in a device synchronise)
  bytes              device bytes of the set (d377_msm_bases_info)
  blocking_ms        median host wall clock of device.msm (d377_msm_dev, one MSM at a time)
  b2b_ms             device time per MSM of K back-to-back device.msm_async(inputs_ready=True)
                     calls between CUDA events on the engine stream (as bench.py times them)
  e2e_ms             host wall clock per MSM of msm_submit / msm_wait over pinned host scalars,
                     2 (n >= 2^23) or 3 MSMs in flight
  stages_ms, c, W    d377_msm_stage_info of a blocking call

Every timed result is compared with compress((sum a_i s_i mod r) G) (bench.py's helpers); the
process exits 1 if any differs.  The GPU name, power limit and SM clock are read with a
read-only nvidia-smi query in the same run.  One JSON line is printed and written to
OUT_DIR/msm_windowed_bench.json.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info() -> dict:
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        return {"query": q, "rows": [ln.strip() for ln in r.stdout.splitlines() if ln.strip()]}
    except Exception as ex:  # noqa: BLE001
        return {"query": q, "error": repr(ex)}


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--logn", default="10,16,20,22,24")
    ap.add_argument("--c", default="", help="extra window widths of windowed sets (sweep)")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--seed", type=int, default=377)
    args = ap.parse_args()
    import torch

    import decaf377_b200 as d
    from bench import dot_mod_r, expected_encoding
    from decaf377_b200 import device as dev

    d.init(0)
    os.makedirs(args.out_dir, exist_ok=True)
    sweep = [int(x) for x in args.c.split(",") if x.strip()]
    res = {"tool": "tools/msm_windowed_bench.py", "gpu": gpu_info(), "seed": args.seed, "sizes": []}
    all_ok = True
    es = dev.engine_stream()
    for logn in [int(x) for x in args.logn.split(",")]:
        n = 1 << logn
        g = torch.Generator(device="cuda")
        g.manual_seed(args.seed + logn)
        a = torch.randint(0, 256, (n, 32), dtype=torch.uint8, device="cuda", generator=g)
        s = torch.randint(0, 256, (n, 32), dtype=torch.uint8, device="cuda", generator=g)
        a[:, 31] &= 0x03
        s[:, 31] &= 0x03
        pts = dev.fixed_base_mul(a, d.OUT_ELEMENT)
        d.sync()
        torch.cuda.synchronize()
        want = expected_encoding(dot_mod_r(torch, a, s))
        h_sc = d.pinned_copy(s.cpu().numpy())
        entry = {"logn": logn, "n": n, "sets": []}
        kinds = [("plain", None)] + [("windowed", c) for c in [0] + [c for c in sweep if c]]
        for kind, c in kinds:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            if kind == "plain":
                b = d.MsmBases(device_ptr=pts.data_ptr(), n=n, point_format=d.PT_ELEMENT)
            else:
                b = d.MsmBases(device_ptr=pts.data_ptr(), n=n, point_format=d.PT_ELEMENT, windowed=True, c=c)
            torch.cuda.synchronize()
            create_ms = (time.perf_counter() - t0) * 1e3
            ok = True
            # blocking call
            reps = max(5, min(50, (1 << 26) // (n * 8)))
            dev.msm(s, b)
            times = []
            for _ in range(reps):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                _, oc = dev.msm(s, b)
                torch.cuda.synchronize()
                times.append((time.perf_counter() - t0) * 1e3)
                ok = ok and bytes(oc.cpu().numpy().tobytes()) == want
            info = d.msm_stage_info()
            # back to back, device resident
            K = max(args.steps, min(200, (1 << 27) // (n * 8)))
            ring = [(torch.empty(128, dtype=torch.uint8, device="cuda"), torch.empty(32, dtype=torch.uint8, device="cuda"))
                    for _ in range(4)]
            for i in range(3):
                dev.msm_async(s, b, out_element=ring[i % 4][0], out_encoding=ring[i % 4][1], inputs_ready=True)
            d.sync()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(es):
                e0.record()
            for i in range(K):
                dev.msm_async(s, b, out_element=ring[i % 4][0], out_encoding=ring[i % 4][1], inputs_ready=True)
            d.join()
            with torch.cuda.stream(es):
                es.wait_stream(torch.cuda.current_stream())
                e1.record()
            d.sync()
            torch.cuda.synchronize()
            b2b_ms = e0.elapsed_time(e1) / K
            ok = ok and bytes(ring[(K - 1) % 4][1].cpu().numpy().tobytes()) == want
            # end to end over host scalars
            depth = 2 if n >= (1 << 23) else 3
            e2e_steps = max(args.steps, min(100, (1 << 26) // (n * 8)))

            def run():
                last = None
                for i in range(e2e_steps + depth):
                    if i >= depth:
                        last = d.msm_wait((i - depth) % 4)
                    if i < e2e_steps:
                        d.msm_submit(h_sc, b, slot=i % 4)
                return last
            run()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            last = run()
            torch.cuda.synchronize()
            e2e_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
            ok = ok and bytes(last[1].tobytes()) == want
            all_ok = all_ok and ok
            blk = statistics.median(times)
            entry["sets"].append({
                "kind": kind, "c_arg": c, "c": info["c"], "W": info["W"], "windowed": info["windowed"],
                "bytes": b.nbytes, "bytes_per_base": b.nbytes / n, "create_ms": create_ms,
                "blocking_ms": blk, "blocking_mpts": n / blk / 1e3,
                "b2b_ms": b2b_ms, "b2b_mpts": n / b2b_ms / 1e3, "b2b_calls": K,
                "e2e_ms": e2e_ms, "e2e_mpts": n / e2e_ms / 1e3, "e2e_steps": e2e_steps,
                "stages_ms": {k: round(v, 4) for k, v in info["ms"].items()}, "verified": ok})
            b.close()
            print("2^%d %-8s c=%-2d W=%-2d create %8.2f ms  blocking %8.3f ms  b2b %8.3f ms  e2e %8.3f ms  %s"
                  % (logn, kind, info["c"], info["W"], create_ms, blk, b2b_ms, e2e_ms, "ok" if ok else "MISMATCH"),
                  file=sys.stderr, flush=True)
        res["sizes"].append(entry)
        del pts, a, s, h_sc
        torch.cuda.empty_cache()
    res["verified"] = all_ok
    line = json.dumps(res)
    print(line)
    with open(os.path.join(args.out_dir, "msm_windowed_bench.json"), "w") as f:
        f.write(line + "\n")
    return 0 if all_ok else 1


if __name__ == "__main__":
    sys.exit(main())
