"""Many independent MSMs: d377_msm_segmented_dev against the two other routes (B200).

    python tools/msm_segmented_bench.py OUT_DIR [--steps 3] [--seed 377] [--per-msm-cap 1024]

Workload: nseg segments of m pairs each (nseg m = N), m = 64, 256, 1024, 4096, 16384, 65536 at
N = 2^22, and m = 1024, 16384 at N = 2^24.  Points P_i = a_i G from the fixed-base path
(a_i < 2^250 drawn on the device, seeded), batch-normalised to AffinePoint inputs; scalars
s_i < 2^250 (canonical, so that every route accepts them).  Outputs are encodings.

Device time per call on the engine stream (CUDA events around `steps` back-to-back calls after
one warm-up call), device-resident inputs and outputs, for the same inputs:

  segmented   d377_msm_segmented_dev (one segmented Pippenger)
  batch       d377_batch_msm_dev (signed-window ladder per pair, one warp per segment)
  per_msm     one d377_msm_dev_async per segment, then d377_join; timed over the first
              min(nseg, --per-msm-cap) segments (one pass) and scaled to nseg segments
              (`per_msm_ms` is that extrapolation, `per_msm_segments` the number timed)

Every timed result is checked: the segmented and batch outputs byte for byte against each
other, the per-MSM outputs against the segmented ones over the segments timed, and a sample of
segments (both ends included) against the known answer (sum s_i a_i mod r) G computed on the
host and encoded by the fixed-base path.  The process exits 1 on any mismatch.  The GPU name,
power limit and SM clock are read with a read-only nvidia-smi query in the same run.  One
JSON line is printed and written to OUT_DIR/msm_segmented_bench.json, a table to
OUT_DIR/msm_segmented_bench.txt.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CONFIGS = [(22, m) for m in (64, 256, 1024, 4096, 16384, 65536)] + [(24, 1024), (24, 16384)]


def gpu_info() -> dict:
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        return {"query": q, "rows": [ln.strip() for ln in r.stdout.splitlines() if ln.strip()]}
    except Exception as ex:  # noqa: BLE001
        return {"query": q, "error": repr(ex)}


def timed(es, torch, fn, steps, warm=True):
    """ms per call of `steps` back-to-back calls of fn (enqueued on the engine stream)."""
    if warm:
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(es):
        e0.record()
    for _ in range(steps):
        fn()
    with torch.cuda.stream(es):
        e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / steps


def to_int(row) -> int:
    return int.from_bytes(bytes(row), "little")


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--seed", type=int, default=377)
    ap.add_argument("--per-msm-cap", type=int, default=1024)
    args = ap.parse_args()
    os.makedirs(args.out_dir, exist_ok=True)

    import numpy as np
    import torch

    import decaf377_b200 as d
    from decaf377_b200 import _lib
    from decaf377_b200 import device as dev
    from oracle import decaf377_ref as o
    d.init(0)
    lib = _lib.load()
    es = dev.engine_stream()
    fmt, ofmt = d.PT_AFFINE, d.OUT_ENCODING
    res = {"tool": "tools/msm_segmented_bench.py", "gpu": gpu_info(), "steps": args.steps, "configs": []}
    all_ok = True
    cache = {}
    for logn, m in CONFIGS:
        n, nseg = 1 << logn, (1 << logn) // m
        if logn not in cache:
            cache.clear()
            torch.cuda.empty_cache()
            g = torch.Generator(device="cuda")
            g.manual_seed(args.seed + logn)
            a = torch.randint(0, 256, (n, 32), dtype=torch.uint8, device="cuda", generator=g)
            a[:, 31] &= 0x03
            s = torch.randint(0, 256, (n, 32), dtype=torch.uint8, device="cuda", generator=g)
            s[:, 31] &= 0x03
            pts = dev.normalize(dev.fixed_base_mul(a, d.OUT_ELEMENT))
            torch.cuda.synchronize()
            cache[logn] = (a, s, pts)
        a, s, pts = cache[logn]
        off = (np.arange(nseg + 1, dtype=np.int64) * m).astype(np.uint32)
        out_seg = torch.empty((nseg, 32), dtype=torch.uint8, device="cuda")
        out_bm = torch.empty((nseg, 32), dtype=torch.uint8, device="cuda")
        off_dev = torch.from_numpy(off).cuda()
        torch.cuda.synchronize()

        def seg():
            _lib.check(lib.d377_msm_segmented_dev(s.data_ptr(), pts.data_ptr(), fmt, off.ctypes.data, nseg,
                                                  out_seg.data_ptr(), ofmt, None))

        def bm():
            _lib.check(lib.d377_batch_msm_dev(s.data_ptr(), pts.data_ptr(), fmt, off_dev.data_ptr(), nseg, n,
                                              out_bm.data_ptr(), ofmt, None))

        row = {"n": n, "m": m, "nseg": nseg}
        row["segmented_ms"] = timed(es, torch, seg, args.steps)
        c, w, chunks = d.msm_segmented_last()
        row.update({"c": c, "W": w, "chunks": chunks})
        row["batch_ms"] = timed(es, torch, bm, args.steps)
        # per-MSM route over the first k segments, one pass (after a warm-up over a few)
        k = min(nseg, args.per_msm_cap)
        oc = torch.empty((k, 32), dtype=torch.uint8, device="cuda")
        oe = torch.empty((k, 128), dtype=torch.uint8, device="cuda")

        def per_msm(cnt=k):
            for j in range(cnt):
                lo = j * m
                _lib.check(lib.d377_msm_dev_async(s[lo].data_ptr(), pts[lo].data_ptr(), fmt, m, oe[j].data_ptr(),
                                                  oc[j].data_ptr(), 1))
            d.join()

        per_msm(min(k, 8))
        d.sync()
        t = timed(es, torch, per_msm, 1, warm=False)
        d.sync()
        row["per_msm_segments"] = k
        row["per_msm_ms"] = t * nseg / k
        row["speedup_vs_batch"] = row["batch_ms"] / row["segmented_ms"]
        row["speedup_vs_per_msm"] = row["per_msm_ms"] / row["segmented_ms"]
        # checks on the last timed results
        ok_bm = bool(torch.equal(out_seg, out_bm))
        ok_pm = bool(torch.equal(out_seg[:k], oc))
        samp = sorted({0, 1, nseg - 2, nseg - 1} | set(range(0, nseg, max(1, nseg // 12))))
        samp = [j for j in samp if 0 <= j < nseg]
        ks = []
        for j in samp:
            aa = a[j * m:(j + 1) * m].cpu().numpy()
            ss = s[j * m:(j + 1) * m].cpu().numpy()
            ks.append(sum(to_int(x) * to_int(y) for x, y in zip(aa, ss)) % o.R)
        want = d.fixed_base_mul(np.frombuffer(b"".join(v.to_bytes(32, "little") for v in ks), np.uint8).reshape(-1, 32),
                                d.OUT_ENCODING)
        ok_kat = bool(np.array_equal(out_seg[samp].cpu().numpy(), want))
        row["verified"] = {"batch_equal": ok_bm, "per_msm_equal": ok_pm, "known_answer_segments": len(samp),
                           "known_answer": ok_kat}
        all_ok = all_ok and ok_bm and ok_pm and ok_kat
        res["configs"].append(row)
        print(json.dumps(row), flush=True)
        del out_seg, out_bm, oc, oe
    res["verified"] = all_ok
    line = json.dumps(res)
    print(line)
    with open(os.path.join(args.out_dir, "msm_segmented_bench.json"), "w") as f:
        f.write(line + "\n")
    with open(os.path.join(args.out_dir, "msm_segmented_bench.txt"), "w") as f:
        f.write("gpu: %s\n" % json.dumps(res["gpu"]))
        f.write("device-resident, back to back, AffinePoint inputs, encoding outputs; ms per call\n")
        f.write("%10s %7s %7s %4s %4s %6s %12s %12s %12s %8s %8s %s\n" % (
            "pairs", "m", "nseg", "c", "W", "chunks", "segmented", "batch_msm", "per_msm*", "x batch", "x per", "ok"))
        for r in res["configs"]:
            v = r["verified"]
            f.write("%10d %7d %7d %4d %4d %6d %12.3f %12.3f %12.3f %8.2f %8.2f %s\n" % (
                r["n"], r["m"], r["nseg"], r["c"], r["W"], r["chunks"], r["segmented_ms"], r["batch_ms"],
                r["per_msm_ms"], r["speedup_vs_batch"], r["speedup_vs_per_msm"],
                v["batch_equal"] and v["per_msm_equal"] and v["known_answer"]))
        f.write("* per_msm: one d377_msm_dev_async per segment, timed over the first min(nseg, %d) segments and "
                "scaled to nseg\n" % args.per_msm_cap)
    return 0 if all_ok else 1


if __name__ == "__main__":
    sys.exit(main())
