"""Prepared fixed bases (d377_fixed_bases_*) against the route available without them (B200).

    python tools/fixed_bases_bench.py OUT_DIR [--steps 5] [--seed 377]
    python tools/fixed_bases_bench.py OUT_DIR --generator-only [--tree DIR] [--tag NAME]

Inputs: k bases P_j = encode_to_curve(seeded), scalars uniform over [0, 2^250) (seeded, on the
device; canonical Fr, as bench.py draws them: scalars at or above 2^252 would send the
generator's quartic kernel to its Edwards fallback).  Reported:

  create          host wall clock around FixedBases creation (ends in a device synchronise) and
                  its device bytes, k = 1, 2, 4
  b2b             device time per call (CUDA events on the engine stream around `steps`
                  back-to-back calls, after one warm-up call) of d377_fixed_bases_mul_dev, for
                  k = 1, 2, 4 x Element / encoding output x n = 2^20, 2^22 (and 2^24 for k <= 2),
                  beside today's route on the same inputs: k d377_batch_scalar_mul_dev over the
                  base repeated n times (Element out), k - 1 d377_batch_add_dev, and
                  d377_batch_compress_dev for encodings
  generator       k = 1 with B = G against d377_fixed_base_mul_dev, both formats, 2^20 and 2^24
                  (encodings of the generator call take the Jacobi-quartic path)
  e2e             host wall clock of FixedBases.mul over pinned host scalars and a pinned
                  output at 2^22, k = 2, encodings (median of `steps` calls)

Every timed result (the last call of each timed loop) is checked against the C oracle on a
strided sample that includes both ends (c_oracle.scalar_mul + add + compress); the process
exits 1 on any mismatch.  The GPU name, power limit and SM clock are read with a read-only
nvidia-smi query in the same run.  One JSON line is printed and written to
OUT_DIR/fixed_bases_bench.json, a table to OUT_DIR/fixed_bases_bench.txt.

--generator-only times the generator's Edwards kernels alone, back to back: d377_fixed_base_mul_dev
at 2^24 with Element output (k_fixed_base<0>) and at 2^17 with encoding output (below the
quartic threshold: k_fixed_base<1>), with the package found under --tree (default: this
checkout), so that two builds can be compared in one session.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def gpu_info() -> dict:
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        return {"query": q, "rows": [ln.strip() for ln in r.stdout.splitlines() if ln.strip()]}
    except Exception as ex:  # noqa: BLE001
        return {"query": q, "error": repr(ex)}


def timed(es, torch, fn, steps):
    """ms per call of `steps` back-to-back calls of fn (enqueued on the engine stream)."""
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


def sample_rows(n, m=256):
    step = max(1, n // m)
    return sorted(set(list(range(0, min(n, 16))) + list(range(0, n, step)) + list(range(max(0, n - 16), n))))


def oracle_encodings(co, wires, S):
    """compress(sum_j S[:, j] * P_j) by the C oracle; S: (m, k, 32) host array."""
    import numpy as np
    m, k = S.shape[0], S.shape[1]
    th = co.threads_default()
    acc = None
    for j in range(k):
        pts = np.repeat(wires[j:j + 1], m, axis=0)
        prod = co.scalar_mul(pts, np.ascontiguousarray(S[:, j]), threads=th)
        acc = prod if acc is None else co.add(acc, prod, threads=th)
    return co.compress(acc, threads=th)


def generator_only(args) -> int:
    import torch

    import decaf377_b200 as d
    from decaf377_b200 import _lib
    from decaf377_b200 import device as dev
    d.init(0)
    lib = _lib.load()
    es = dev.engine_stream()
    from oracle import c_oracle as co
    res = {"tool": "tools/fixed_bases_bench.py --generator-only", "tag": args.tag, "gpu": gpu_info()}
    ok = True
    for name, logn, fmt in (("k_fixed_base0_element", 24, d.OUT_ELEMENT), ("k_fixed_base1_encoding", 17, d.OUT_ENCODING)):
        n = 1 << logn
        g = torch.Generator(device="cuda")
        g.manual_seed(args.seed + logn)
        sc = torch.randint(0, 256, (n, 32), dtype=torch.uint8, device="cuda", generator=g)
        sc[:, 31] &= 0x03
        out = torch.empty((n, 128 if fmt == d.OUT_ELEMENT else 32), dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        steps = max(args.steps, 10) * (1 if logn >= 24 else 20)
        ms = timed(es, torch, lambda: _lib.check(lib.d377_fixed_base_mul_dev(sc.data_ptr(), n, out.data_ptr(), fmt)),
                   steps)
        rows = sample_rows(n)
        got = out[rows].cpu().numpy()
        if fmt == d.OUT_ELEMENT:
            got = co.compress(got)
        ok = ok and bool((got == co.fixed_base(sc[rows].cpu().numpy())).all())
        res[name] = {"n": n, "ms": ms, "melem_s": n / ms / 1e3, "steps": steps}
    res["verified"] = ok
    print(json.dumps(res))
    return 0 if ok else 1


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--seed", type=int, default=377)
    ap.add_argument("--generator-only", action="store_true")
    ap.add_argument("--tree", default=ROOT, help="checkout whose decaf377_b200 is imported")
    ap.add_argument("--tag", default="")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.abspath(args.tree))
    if args.generator_only:
        return generator_only(args)
    import numpy as np
    import torch

    import decaf377_b200 as d
    from decaf377_b200 import _lib
    from decaf377_b200 import device as dev
    from oracle import c_oracle as co
    from oracle import decaf377_ref as o
    from tests.util import np_bytes, oracle_points

    d.init(0)
    lib = _lib.load()
    chk = _lib.check
    os.makedirs(args.out_dir, exist_ok=True)
    es = dev.engine_stream()
    res = {"tool": "tools/fixed_bases_bench.py", "gpu": gpu_info(), "seed": args.seed, "steps": args.steps,
           "create": [], "b2b": [], "generator": [], "e2e": []}
    all_ok = True
    lines = []

    def log(s):
        lines.append(s)
        print(s, file=sys.stderr, flush=True)

    log("gpu: %s" % res["gpu"].get("rows"))
    P = oracle_points("fixed_bases_bench", 4)
    wires = np_bytes([o.point_to_wire(p) for p in P], 128)
    ks = (1, 2, 4)
    sets = {}
    for k in ks:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fb = d.FixedBases(wires[:k])
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t0) * 1e3
        sets[k] = fb
        res["create"].append({"k": k, "create_ms": ms, "bytes": fb.nbytes})
        log("create k=%d  %8.2f ms  %d bytes (%.1f MiB)" % (k, ms, fb.nbytes, fb.nbytes / 2**20))

    def check_rows(name, got_enc, S_dev, wire_rows, n):
        rows = sample_rows(n)
        want = oracle_encodings(co, wire_rows, S_dev[rows].cpu().numpy())
        ok = bool((got_enc[rows] == want).all())
        if not ok:
            log("MISMATCH %s" % name)
        return ok

    def enc_of(out, fmt):
        o_np = out.cpu().numpy() if fmt == d.OUT_ENCODING else dev.compress(out).cpu().numpy()
        return o_np

    # ---- back to back, device resident -------------------------------------------------------
    for logn in (20, 22, 24):
        n = 1 << logn
        for k in ks:
            if logn == 24 and k > 2:
                continue
            g = torch.Generator(device="cuda")
            g.manual_seed(args.seed + 31 * logn + k)
            S = torch.randint(0, 256, (n, k, 32), dtype=torch.uint8, device="cuda", generator=g)
            S[:, :, 31] &= 0x03
            cols = [S[:, j].contiguous() for j in range(k)]
            reps = [torch.from_numpy(wires[j:j + 1]).cuda().repeat(n, 1) for j in range(k)]
            prods = [torch.empty((n, 128), dtype=torch.uint8, device="cuda") for _ in range(k)]
            acc = torch.empty((n, 128), dtype=torch.uint8, device="cuda")
            for fmt in (d.OUT_ELEMENT, d.OUT_ENCODING):
                w = 128 if fmt == d.OUT_ELEMENT else 32
                out_new = torch.empty((n, w), dtype=torch.uint8, device="cuda")
                out_old = torch.empty((n, w), dtype=torch.uint8, device="cuda")
                fb = sets[k]

                def new():
                    chk(lib.d377_fixed_bases_mul_dev(C.c_void_p(fb.ptr), S.data_ptr(), n, out_new.data_ptr(), fmt))

                def old():
                    for j in range(k):
                        dst = out_old if (k == 1 and fmt == d.OUT_ELEMENT) else prods[j]
                        chk(lib.d377_batch_scalar_mul_dev(reps[j].data_ptr(), d.PT_ELEMENT, cols[j].data_ptr(), n,
                                                          dst.data_ptr(), d.OUT_ELEMENT, None))
                    last = prods[0]
                    for j in range(1, k):
                        dst = out_old if (fmt == d.OUT_ELEMENT and j == k - 1) else acc
                        chk(lib.d377_batch_add_dev(last.data_ptr(), prods[j].data_ptr(), n, dst.data_ptr()))
                        last = dst
                    if fmt == d.OUT_ENCODING:
                        chk(lib.d377_batch_compress_dev(last.data_ptr(), n, out_old.data_ptr()))

                old_steps = max(1, args.steps // 2) if logn == 24 else args.steps
                ms_new = timed(es, torch, new, args.steps)
                ms_old = timed(es, torch, old, old_steps)
                torch.cuda.synchronize()
                e_new, e_old = enc_of(out_new, fmt), enc_of(out_old, fmt)
                ok = bool((e_new == e_old).all()) and check_rows("b2b k=%d 2^%d fmt=%d" % (k, logn, fmt), e_new, S,
                                                                 wires[:k], n)
                all_ok = all_ok and ok
                res["b2b"].append({"k": k, "logn": logn, "n": n, "out": "element" if fmt == 0 else "encoding",
                                   "fixed_bases_ms": ms_new, "fixed_bases_mrows_s": n / ms_new / 1e3,
                                   "today_ms": ms_old, "today_mrows_s": n / ms_old / 1e3,
                                   "speedup": ms_old / ms_new, "verified": ok})
                log("b2b  k=%d 2^%d %-8s fixed_bases %9.3f ms (%7.1f Mrows/s)  today %9.3f ms (%6.1f Mrows/s)  x%5.1f  %s"
                    % (k, logn, "element" if fmt == 0 else "encoding", ms_new, n / ms_new / 1e3, ms_old,
                       n / ms_old / 1e3, ms_old / ms_new, "ok" if ok else "MISMATCH"))
                del out_new, out_old
            del S, cols, reps, prods, acc
            torch.cuda.empty_cache()

    # ---- generator: k = 1 over G against d377_fixed_base_mul_dev ------------------------------
    Gw = np.frombuffer(o.point_to_wire(o.GENERATOR), np.uint8).reshape(1, 128)
    fbg = d.FixedBases(Gw)
    for logn in (20, 24):
        n = 1 << logn
        g = torch.Generator(device="cuda")
        g.manual_seed(args.seed + 7 * logn)
        S = torch.randint(0, 256, (n, 32), dtype=torch.uint8, device="cuda", generator=g)
        S[:, 31] &= 0x03
        for fmt in (d.OUT_ELEMENT, d.OUT_ENCODING):
            w = 128 if fmt == d.OUT_ELEMENT else 32
            out_fb = torch.empty((n, w), dtype=torch.uint8, device="cuda")
            out_g = torch.empty((n, w), dtype=torch.uint8, device="cuda")
            ms_fb = timed(es, torch, lambda: chk(lib.d377_fixed_bases_mul_dev(C.c_void_p(fbg.ptr), S.data_ptr(), n,
                                                                              out_fb.data_ptr(), fmt)), args.steps)
            ms_g = timed(es, torch, lambda: chk(lib.d377_fixed_base_mul_dev(S.data_ptr(), n, out_g.data_ptr(), fmt)),
                         args.steps)
            torch.cuda.synchronize()
            same = bool(torch.equal(out_fb, out_g))
            rows = sample_rows(n)
            ok = same and bool((enc_of(out_fb, fmt)[rows] == co.fixed_base(S[rows].cpu().numpy())).all())
            all_ok = all_ok and ok
            res["generator"].append({"logn": logn, "n": n, "out": "element" if fmt == 0 else "encoding",
                                     "fixed_bases_ms": ms_fb, "fixed_base_mul_ms": ms_g, "byte_identical": same,
                                     "generator_path": "edwards" if fmt == 0 else "quartic", "verified": ok})
            log("gen  2^%d %-8s fixed_bases([G]) %9.3f ms  fixed_base_mul %9.3f ms (%s)  %s"
                % (logn, "element" if fmt == 0 else "encoding", ms_fb, ms_g,
                   "edwards, same kernel" if fmt == 0 else "quartic path", "ok" if ok else "MISMATCH"))
            del out_fb, out_g
        del S
        torch.cuda.empty_cache()
    fbg.close()

    # ---- end to end: pinned host buffers, 2^22, k = 2, encodings ------------------------------
    n, k = 1 << 22, 2
    rng = np.random.default_rng(args.seed)
    hS = rng.integers(0, 256, (n, k, 32), dtype=np.uint8)
    hS[:, :, 31] &= 0x03
    hS = d.pinned_copy(hS)
    hout = d.pinned_empty((n, 32))
    fb = sets[k]
    fb.mul(hS, d.OUT_ENCODING, out=hout)
    times = []
    for _ in range(args.steps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fb.mul(hS, d.OUT_ENCODING, out=hout)
        times.append((time.perf_counter() - t0) * 1e3)
    rows = sample_rows(n)
    ok = bool((hout[rows] == oracle_encodings(co, wires[:k], hS[rows])).all())
    all_ok = all_ok and ok
    e2e = statistics.median(times)
    res["e2e"].append({"k": k, "logn": 22, "n": n, "out": "encoding", "median_ms": e2e, "mrows_s": n / e2e / 1e3,
                       "times_ms": times, "verified": ok})
    log("e2e  k=2 2^22 encoding pinned host buffers  %9.3f ms (%6.1f Mrows/s)  %s"
        % (e2e, n / e2e / 1e3, "ok" if ok else "MISMATCH"))
    for fbk in sets.values():
        fbk.close()

    res["verified"] = all_ok
    line = json.dumps(res)
    print(line)
    with open(os.path.join(args.out_dir, "fixed_bases_bench.json"), "w") as f:
        f.write(line + "\n")
    with open(os.path.join(args.out_dir, "fixed_bases_bench.txt"), "w") as f:
        f.write("\n".join(lines) + "\n")
    return 0 if all_ok else 1


if __name__ == "__main__":
    sys.exit(main())
