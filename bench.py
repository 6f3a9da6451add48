#!/usr/bin/env python3
"""bench.py -- headline benchmark of the decaf377 batch engine on B200.

Metric (BASELINE.json): decaf377 Pippenger MSM throughput in Mpoints/s; batch
decompress / compress / Elligator / fixed-base throughput in Melem/s.

Default workload: `vartime_multiscalar_mul` over 2^24 (scalar, Element) pairs per GPU
(BASELINE.json configs[3]/[4]); with --gpus N every rank owns its own 2^24-pair slice
(weak scaling, 2^24 .. 2^27 points in total) and the 128-byte partial sums are combined
with one NCCL all-gather + N-1 point additions.  The one JSON line also carries

  * `configs` (N = 1): every other BASELINE config -- pipeline 2^16, encode 2^22, hash 2^22,
    fixed_base 2^24, compress / decompress 2^22, msm 2^20 -- each with value, roofline, e2e,
    cpu_baseline and an oracle check;
  * `strong_scaling_2p24` (N > 1): ONE 2^24-pair MSM cut into N slices, the north-star
    target, and `single_process` -- the same call through d377_msm_multi_dev, one process
    driving all N GPUs;
  * `verified_sharded`: the points are P_i = a_i G, so sum s_i P_i = (sum a_i s_i mod r) G;
    the encoding the TIMED calls produced is compared with the oracle's compress(k G).  The
    process exits non-zero if that check fails.

    python bench.py --gpus 1 --steps 10 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference        # CPU port of the reference path, same metric
    python bench.py --dump-outputs DIR      # also write the last timed step's outputs to DIR/*.npy

`--workload encode | hash | fixed_base | pipeline | decompress | compress` times one of the
other configs alone with the same harness.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FQ_OPS = {  # exact Fq multiplications + squarings per element (tools/count_ops.py, DESIGN.md 3);
    # products with a small curve constant (fq_mul_small, 16 wide multiplies) are not counted
    "isqrt": 308, "decompress": 320, "compress": 315, "encode": 323,
    "encode_compress": 338,   # fused: the encoding is read off the Jacobi-quartic pair (one isqrt)
    "hash_compress": 670,     # fused: two maps, the sum on the quartic, encoding from the sum
    # fixed base on the Jacobi quartic: 12 x (9 M + 2 S) + encoding tail 16 M + 4 S (DESIGN.md 3.3);
    # the Edwards path it replaces is 16 x 7 + 315 = 427
    "fixed_base_jq": 152,
    "scalar_mul": 3133, "pipeline": 320 + 3133 + 315,
}
IMAD_PER_FQ_OP = 128
# IMAD.WIDE.U32 actually issued per element (tools/count_ops.py): 120 per multiplication,
# 92 per squaring, 56 per from-Montgomery reduction.  `achieved` counts the reference's
# 128 per Fq-op (SURVEY 8d); `issued_frac` is this count against the same peak, i.e. the
# share of the multiply pipe's issue slots the kernel really fills.
WIDE_ISSUED = {"decompress": 31612, "compress": 31140, "encode": 33916, "hash": 66932,
               "fixed_base": 17760,
               # decompress + compress + the kernel's signed 4-bit ladder: 192 x (4S + 3M) + 64 x
               # (4S + 4M) doublings, 64 x 7M + 8M cached additions, 71 M for the table of 8 multiples
               "pipeline": 31612 + 31140 + 192 * 728 + 64 * 848 + 64 * 840 + 960 + 8520}
OPS_OF = {"encode": FQ_OPS["encode_compress"], "hash": FQ_OPS["hash_compress"],
          "fixed_base": FQ_OPS["fixed_base_jq"], "compress": FQ_OPS["compress"],
          "decompress": FQ_OPS["decompress"], "pipeline": FQ_OPS["pipeline"]}
WIDE_PER_MUL = 120
# DRAM bytes (read + write) per launch from the round-2 `ncu --set full` captures of the same
# kernels (profiles/r2_ncu_full_summary.csv); None where no capture is committed.
NCU_TRAFFIC = {
    # k_msm_accumulate<1>, 2^24 pairs, c = 18, the whole MSM as ONE launch (what the back-to-back
    # loop runs): 34.35 GB read + 0.46 GB written (profiles/r2_ncu_full_summary.csv, capture
    # msm24_one_group) against 31.9 GB algorithmic
    ("msm", 24, True): 34.81e9,
    # codec / fused kernels: DRAM bytes of the 2^20 captures (codec20) scaled to n
    ("compress", 22): 4 * 153.3e6, ("decompress", 22): 4 * 115.4e6, ("encode", 22): 4 * 34.7e6,
    ("hash", 22): 4 * 82.5e6, ("fixed_base", 24): 16 * 1881.6e6,
}

WORKLOADS = ["msm", "encode", "hash", "fixed_base", "pipeline", "decompress", "compress"]
DEFAULT_LOGN = {"msm": 24, "encode": 22, "hash": 22, "fixed_base": 24, "pipeline": 16, "decompress": 22,
                "compress": 22}
# CPU samples: about 1-4 s of work per step on 16 host threads (the bounded cpu_baseline leg)
CPU_SAMPLE_LOGN = {"msm": 21, "encode": 18, "hash": 17, "fixed_base": 15, "pipeline": 15, "decompress": 18,
                   "compress": 18}
UNIT = {"msm": "Mpoints/s"}
METRIC = {
    "msm": "decaf377 MSM throughput (vartime_multiscalar_mul, Pippenger)",
    "encode": "decaf377 batch encode_to_curve + vartime_compress throughput",
    "hash": "decaf377 batch hash_to_curve + vartime_compress throughput",
    "fixed_base": "decaf377 fixed-base (generator) scalar mul + compress throughput",
    "pipeline": "decaf377 vartime_decompress -> scalar mul -> vartime_compress throughput",
    "decompress": "decaf377 batch vartime_decompress throughput",
    "compress": "decaf377 batch vartime_compress throughput",
}
WORKLOAD_NAME = {
    "msm": "Pippenger vartime_multiscalar_mul, 2^{logn} (Fr, Element) pairs per GPU",
    "encode": "batch Elligator encode_to_curve + compress of 2^{logn} Fq elements per GPU",
    "hash": "batch hash_to_curve (two Elligator maps + add) + compress of 2^{logn} Fq pairs per GPU",
    "fixed_base": "fixed-base generator mul + compress of 2^{logn} Fr scalars per GPU",
    "pipeline": "2^{logn} encodings: vartime_decompress -> scalar mul -> vartime_compress",
    "decompress": "batch vartime_decompress of 2^{logn} encodings per GPU",
    "compress": "batch vartime_compress of 2^{logn} elements per GPU",
}
R_MODULUS = 0x04AAD957A68B2955982D1347970DEC005293A3AFC43C8AFEB95AEE9AC33FD9FF


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="msm", choices=WORKLOADS)
    ap.add_argument("--logn", type=int, default=None, help="log2 of units per GPU")
    ap.add_argument("--ref-logn", type=int, default=None, help="log2 of the CPU sample size")
    ap.add_argument("--ref-budget-s", type=float, default=900.0,
                    help="--impl reference: wall-clock budget for warm-up + timed steps")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the per-config block of the MSM line")
    ap.add_argument("--no-single-process", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed call returned in its last step to DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU arm; --impl reference has none")
    return a


DUMP_BUDGET = 64_000_000     # bytes written by --dump-outputs, .npy headers included


def dump_outputs(path: str, outputs: dict) -> None:
    """Write every output of the last timed step as <path>/<name>.npy in float32 (every value
    is a byte, so the conversion is exact).  When the outputs together would exceed 64 MB,
    all of them keep the same rows, a sample drawn with a fixed seed, and rows.npy (float64)
    lists the row indices kept.  `outputs` maps names to torch tensors on any device."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    total = sum(4 * t.numel() for t in outputs.values())
    if total > DUMP_BUDGET - (1 << 16):          # room for the .npy headers
        n = {t.shape[0] for t in outputs.values()}
        assert len(n) == 1, "sampled outputs must share their first dimension"
        n = n.pop()
        row_bytes = sum(4 * t[0].numel() for t in outputs.values()) + 8
        m = (DUMP_BUDGET - (1 << 16)) // row_bytes
        rows = np.sort(np.random.default_rng(377).choice(n, m, replace=False))
        np.save(os.path.join(path, "rows.npy"), rows.astype(np.float64))
        outputs = {k: t[torch.from_numpy(rows).to(t.device)] for k, t in outputs.items()}
    for k, t in outputs.items():
        np.save(os.path.join(path, k + ".npy"), t.cpu().numpy().astype(np.float32))


# ---------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md recipe)
# ---------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "power_w_max": max(pw),
                "samples": len(sm), "reasons": sorted(reasons)}


def measured_peaks() -> dict:
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        d["_source"] = "measured (MEASURED_PEAKS.json)"
        return d
    return {"hbm_gbs": 6650.0, "_source": "fallback (B200_PROFILING.md)"}


# ---------------------------------------------------------------------------
# CPU port of the reference path (oracle) -- cpu_baseline and --impl reference
# ---------------------------------------------------------------------------
def cpu_inputs(workload: str, n: int):
    import numpy as np
    from oracle import c_oracle as co
    from oracle import decaf377_ref as o
    threads = os.cpu_count() or 1
    raw = np.frombuffer(o.xof_bytes("bench_fq", n), np.uint8).reshape(n, 32).copy()
    sc = np.frombuffer(o.xof_bytes("bench_sc", n), np.uint8).reshape(n, 32).copy()
    sc[:, 31] &= 0x03
    if workload == "msm":
        return (sc, co.encode_to_curve(raw, threads=threads))
    if workload == "encode":
        return (raw,)
    if workload == "hash":
        raw2 = np.frombuffer(o.xof_bytes("bench_fq2", n), np.uint8).reshape(n, 32).copy()
        return (raw, raw2)
    if workload == "fixed_base":
        return (sc,)
    el = co.encode_to_curve(raw, threads=threads)
    if workload == "compress":
        return (el,)
    enc = co.compress(el, threads=threads)
    if workload == "decompress":
        return (enc,)
    return (enc, sc)


def cpu_step(workload: str, inputs, threads: int):
    from oracle import c_oracle as co
    if workload == "msm":
        return co.msm_pippenger(inputs[0], inputs[1], threads=threads)
    if workload == "encode":
        return co.encode_to_curve(inputs[0], out_enc=True, threads=threads)
    if workload == "hash":
        return co.hash_to_curve(inputs[0], inputs[1], out_enc=True, threads=threads)
    if workload == "fixed_base":
        return co.fixed_base(inputs[0], out_enc=True, threads=threads)
    if workload == "compress":
        return co.compress(inputs[0], threads=threads)
    if workload == "decompress":
        return co.decompress(inputs[0], threads=threads)
    return co.pipeline(inputs[0], inputs[1], threads=threads)


CPU_KIND_NOTE = ("C port of the reference algorithms (oracle/d377_oracle.c: 4x64 Montgomery, "
                 "Sarkar sqrt, ark-ec style Pippenger, pthreads); the Rust crate cannot be built here")


def run_cpu(workload: str, logn: int, steps: int, warmup: int, budget_s: float = 1e9):
    """W warm-up and K timed steps of the CPU port over 2^logn units; fewer when the budget
    (wall clock, warm-up included) would be exceeded.  Returns (value, ms, threads, n, steps, warmup)."""
    threads = os.cpu_count() or 1
    n = 1 << logn
    inputs = cpu_inputs(workload, n)
    t_start = time.perf_counter()
    t0 = time.perf_counter()
    cpu_step(workload, inputs, threads)          # first step: also the estimate of the step time
    est = time.perf_counter() - t0
    did_warm = 1
    while did_warm < warmup and (time.perf_counter() - t_start) + est * (steps + 1) < budget_s:
        cpu_step(workload, inputs, threads)
        did_warm += 1
    did = 0
    t0 = time.perf_counter()
    while did < steps and (did == 0 or (time.perf_counter() - t_start) + est < budget_s):
        cpu_step(workload, inputs, threads)
        did += 1
    dt = time.perf_counter() - t0
    return n * did / dt / 1e6, dt / did * 1e3, threads, n, did, did_warm


def cpu_baseline_of(wl: str, logn: int, steps: int = 2) -> dict:
    v, ms, threads, nn, did, _ = run_cpu(wl, logn, steps, 1)
    return {"value": v, "unit": UNIT.get(wl, "Melem/s"), "cores": threads, "kind": "port",
            "sample": "%d steps of 2^%d units on %d host threads (%.0f ms/step); %s"
                      % (did, logn, threads, ms, CPU_KIND_NOTE)}


def main_reference(args):
    """The reference arm: the reference's own CPU implementation of the path (here its C port,
    the Rust crate cannot be compiled in this image) on all host threads, at the SAME size the
    GPU arm names, for the same --steps / --warmup as long as the budget allows."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    wl = args.workload
    full = args.logn or DEFAULT_LOGN[wl]
    logn = args.ref_logn or full
    value, ms, threads, n, steps, warm = run_cpu(wl, logn, max(1, args.steps), max(1, args.warmup),
                                                 args.ref_budget_s)
    unit = UNIT.get(wl, "Melem/s")
    sample = "%d steps (+%d warm-up) of 2^%d units on %d host threads; %s" % (steps, warm, logn, threads,
                                                                             CPU_KIND_NOTE)
    line = {
        "impl": "reference", "metric": METRIC[wl], "value": value, "unit": unit,
        "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64 (4x64-bit limb Montgomery)",
        "data": "synthetic (SHAKE-256 bytes; points = encode_to_curve of random Fq)",
        "config": {"workload": WORKLOAD_NAME[wl].format(logn=full), "units_per_step": n,
                   "same_size_as_gpu_arm": logn == full,
                   "note": "the CPU path does not shard: rank 0 runs it once whatever --gpus is"},
        "cpu_baseline": {"value": value, "unit": unit, "cores": threads, "kind": "port",
                         "sample": sample},
        "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ---------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------
class Ctx:
    """Process-wide handles of the GPU arm."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist

        import decaf377_b200 as d
        from decaf377_b200 import device as dev
        from decaf377_b200 import dist as ddist
        self.torch, self.dist, self.d, self.dev, self.ddist = torch, dist, d, dev, ddist
        self.args = args
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        if self.world != args.gpus and self.world > 1:
            raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (args.gpus, self.world))
        if args.gpus > 1 and self.world == 1:
            raise SystemExit("launch with torch.distributed.run for --gpus > 1")
        if not torch.cuda.is_available():
            raise SystemExit("no CUDA device: decaf377_b200 has no CPU fallback (use --impl reference "
                             "for the CPU port)")
        torch.cuda.set_device(self.local_rank)
        self.cuda = torch.device("cuda", self.local_rank)
        self._hb = 0
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.cuda)
        d.init(self.local_rank)
        self.st = dev.engine_stream()
        self.flush_buf = None
        self.gen = torch.Generator(device=self.cuda).manual_seed(377 + self.rank)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()

    def host_barrier(self):
        """Barrier on the HOST, through the rendezvous TCP store (127.0.0.1): a rank that waits
        in an NCCL barrier keeps a spinning kernel on its GPU, and kernels of two processes on
        one GPU are time-sliced -- rank 0 drives every GPU during the single-process
        measurement, so the other ranks must leave theirs idle."""
        if self.world == 1:
            return
        self.torch.cuda.synchronize()
        store = self.dist.distributed_c10d._get_default_store()
        self._hb += 1
        key = "d377_host_barrier_%d" % self._hb
        store.add(key, 1)
        while int(store.add(key, 0)) < self.world:
            time.sleep(0.002)

    def rand(self, n, scalar=False):
        t = self.torch.randint(0, 256, (n, 32), dtype=self.torch.uint8, device=self.cuda, generator=self.gen)
        if scalar:
            t[:, 31] &= 0x03           # < 2^250 < r: canonical Fr
        return t

    def max_over_ranks(self, x: float) -> float:
        if self.world == 1:
            return x
        t = self.torch.tensor([x], device=self.cuda, dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def time_device(self, step, steps, warmup, flush_l2=False):
        """W untimed + K timed steps, CUDA events on the engine stream (the stream the kernels
        are launched on), barrier + synchronize on both sides, max over ranks.  The join
        before the closing event orders the engine stream behind the MSM tails that run on the
        result stream, so the interval covers every kernel of every step.

        `flush_l2` (workloads whose inputs fit the 126 MB L2): every step gets its own event
        pair and a 256 MiB write runs between the pairs, outside the timed intervals."""
        torch, d = self.torch, self.d
        for _ in range(warmup):
            step()
        d.sync()
        torch.cuda.synchronize()
        self.barrier()
        l0 = d.launch_count()
        if flush_l2:
            if self.flush_buf is None:
                self.flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=self.cuda)
            pairs = []
            for k in range(steps):
                with torch.cuda.stream(self.st):
                    self.flush_buf.fill_(k & 0xFF)
                    a = torch.cuda.Event(enable_timing=True)
                    b = torch.cuda.Event(enable_timing=True)
                    a.record()
                step()
                d.join()
                with torch.cuda.stream(self.st):
                    b.record()
                pairs.append((a, b))
            d.sync()
            torch.cuda.synchronize()
            self.barrier()
            ms = self.max_over_ranks(sum(a.elapsed_time(b) for a, b in pairs))
            return ms / steps, int(d.launch_count() - l0)
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(self.st):
            e0.record()
        for _ in range(steps):
            step()
        d.join()
        with torch.cuda.stream(self.st):
            self.st.wait_stream(torch.cuda.current_stream())
            e1.record()
        d.sync()
        torch.cuda.synchronize()
        self.barrier()
        ms = self.max_over_ranks(e0.elapsed_time(e1))
        return ms / steps, int(d.launch_count() - l0)

    def time_host(self, fn):
        """Wall clock around fn() with a device synchronize on both sides, max over ranks."""
        torch = self.torch
        torch.cuda.synchronize()
        self.barrier()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        return self.max_over_ranks(time.perf_counter() - t0)


def dot_mod_r(torch, a, s) -> int:
    """sum_i a_i s_i mod r for two (n, 32) uint8 device tensors of little-endian integers:
    16-bit limbs in int64 (a limb product is < 2^32, a sum of 2^24 of them < 2^56)."""
    a16 = a.view(torch.int16).to(torch.int64) & 0xFFFF
    s16 = s.view(torch.int16).to(torch.int64) & 0xFFFF
    k = 0
    for i in range(16):
        col = a16[:, i:i + 1] * s16                  # (n, 16)
        sums = col.sum(dim=0).cpu().tolist()
        for j in range(16):
            k += int(sums[j]) << (16 * (i + j))
    return k % R_MODULUS


def sum_over_ranks_mod_r(cx: Ctx, k: int) -> int:
    if cx.world == 1:
        return k % R_MODULUS
    torch = cx.torch
    mine = torch.tensor(list(k.to_bytes(32, "little")), dtype=torch.uint8, device=cx.cuda)
    allk = torch.empty((cx.world, 32), dtype=torch.uint8, device=cx.cuda)
    cx.dist.all_gather_into_tensor(allk, mine.reshape(1, 32))
    return sum(int.from_bytes(bytes(row), "little") for row in allk.cpu().tolist()) % R_MODULUS


def expected_encoding(k: int) -> bytes:
    """compress(k G) by the oracle (the checker; one scalar multiplication)."""
    from oracle import decaf377_ref as o
    return o.compress(o.scalar_mul(o.GENERATOR, k))


def msm_roofline(cx: Ctx, n: int, logn: int, ms_step: float, imad_peak: float, peaks: dict):
    """Roofline of the dominant kernel (k_msm_accumulate) of the most recent MSM of the timed
    loop, from the CUDA-event stage timers the engine keeps on its own streams."""
    d = cx.d
    info = d.msm_stage_info()
    stages = {k: round(v, 4) for k, v in info["ms"].items()}
    acc_ms = info["ms"]["accumulate"]
    adds = n * info["W"]                      # one bucket addition per non-zero digit
    # Fq multiplications per bucket addition: 7 for a mixed addition against an affine
    # point (SURVEY 8d "A = 7 (mixed)"), 8 against a cached projective point
    per_add = 7 if info["mixed"] else 8
    imads = adds * per_add * IMAD_PER_FQ_OP
    ach = imads / (acc_ms * 1e-3) / 1e9
    issued = adds * per_add * WIDE_PER_MUL / (acc_ms * 1e-3) / 1e9
    bytes_alg = adds * (128 + 4) + (n * info["W"] / 32) * 128
    ach_bw = bytes_alg / (acc_ms * 1e-3) / 1e9
    traffic = NCU_TRAFFIC.get(("msm", logn, info["mixed"]))
    # whole step against the same peak, SURVEY 8d's per-point formula 7 W + 18 2^(c-1) W / n
    per_point = 7 * info["W"] + 18 * (1 << (info["c"] - 1)) * info["W"] / n
    whole = n * per_point * IMAD_PER_FQ_OP / (ms_step * 1e-3) / 1e9 / imad_peak
    roofline = {"bound": "imad", "kernel": "k_msm_accumulate", "achieved": ach, "peak": imad_peak,
                "unit": "GIMAD/s (32x32->64 multiply-adds)", "frac": ach / imad_peak,
                "issued_frac": issued / imad_peak, "fq_mults_per_bucket_addition": per_add,
                "whole_step_frac": whole,
                "traffic": traffic, "algorithmic_bytes": bytes_alg,
                "launch_ms": acc_ms, "window_c": info["c"], "windows": info["W"],
                "peak_source": "IMAD.WIDE.U32 issue-rate microbenchmark run in this process",
                "note": "launch_ms is the engine-stream span of the bucket accumulation of the last "
                        "MSM of the timed loop; the next MSM's counting sort and the previous MSM's "
                        "tail run under it on their own streams"}
    roofline_hbm = {"bound": "hbm", "kernel": "k_msm_accumulate", "achieved": ach_bw,
                    "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": ach_bw / peaks["hbm_gbs"],
                    "traffic": traffic, "peak_source": peaks["_source"]}
    return roofline, roofline_hbm, stages


# ---- MSM -------------------------------------------------------------------------------------
def bench_msm(cx: Ctx, logn: int, steps: int, warmup: int, e2e: bool, extras: bool) -> dict:
    """One MSM workload: device-resident throughput, roofline, end-to-end forms, known-answer
    verification of the timed result.  `extras`: the additional e2e variants and the clock
    sampler (the headline line); the 2^20 config entry runs without them."""
    torch, d, dev, ddist = cx.torch, cx.d, cx.dev, cx.ddist
    world, rank = cx.world, cx.rank
    n = 1 << logn
    # Known-answer inputs (SURVEY 8d): P_i = a_i G from the fixed-base kernel (projective
    # Elements, Z != 1), random canonical scalars s_i.
    a = cx.rand(n, scalar=True)
    sc = cx.rand(n, scalar=True)
    pts = dev.fixed_base_mul(a, d.OUT_ELEMENT)
    d.sync()
    k_all = sum_over_ranks_mod_r(cx, dot_mod_r(torch, a, sc))
    want = expected_encoding(k_all)
    ring = steps + warmup + 4
    oe = torch.empty((ring, 128), dtype=torch.uint8, device=cx.cuda)
    oc = torch.empty((ring, 32), dtype=torch.uint8, device=cx.cuda)
    cnt = [0]
    last = [None]

    def step_dev():
        i = cnt[0] % ring
        cnt[0] += 1
        if world == 1:
            dev.msm_async(sc, pts, d.PT_ELEMENT, out_element=oe[i], out_encoding=oc[i], inputs_ready=True)
            last[0] = (oe[i], oc[i])
        else:
            last[0] = ddist.msm_sharded_async(sc, pts, d.PT_ELEMENT, inputs_ready=True)

    sampler = ClockSampler(cx.local_rank)
    if rank == 0:
        sampler.start()
    ms_step, launches = cx.time_device(step_dev, steps, warmup)
    clocks = sampler.stop() if rank == 0 else None
    value = world * n / (ms_step * 1e-3) / 1e6
    got = bytes(last[0][1].cpu().numpy().tobytes())
    verified = got == want
    out = {"value": value, "unit": "Mpoints/s", "ms_per_step": ms_step, "gpu_launches": launches,
           "clocks": clocks, "verified_known_answer": verified, "h2d": n * (32 + 128), "d2h": 160,
           "steps": steps, "l2": "inputs (%.0f MiB per GPU) exceed the 126 MB L2" % (n * 160 / 2**20),
           # the projective (X : Y : Z : T) of the sum depends on the order in which the counting
           # sort's atomic slot claims put each bucket's points; its affine (x, y) does not
           "outputs": {"element_xy": dev.normalize(last[0][0].reshape(1, 128))[0], "encoding": last[0][1]}}
    imad_peak = d.imad_peak()
    peaks = measured_peaks()
    out["roofline"], out["roofline_hbm"], out["stages"] = msm_roofline(cx, n, logn, ms_step, imad_peak, peaks)
    # the blocking call (one MSM at a time, host synchronisation per call) beside it
    if world == 1:
        ms_blk, _ = cx.time_device(lambda: dev.msm(sc, pts, d.PT_ELEMENT), max(2, steps // 2), 1)
        out["blocking_call"] = {"value": n / (ms_blk * 1e-3) / 1e6, "unit": "Mpoints/s", "ms_per_step": ms_blk,
                                "api": "d377_msm_dev (status read back after every call)"}

    # ---- strong scaling beside it (N > 1): ONE 2^24-pair MSM cut into N slices -----------------
    # BASELINE.json configs[4] / north star: "MSM at 2^24 points sharded across 8 GPUs".
    if world > 1 and logn == 24 and extras:
        ns = n // world
        sc_s, pts_s, a_s = sc[:ns], pts[:ns], a[:ns]
        want_s = expected_encoding(sum_over_ranks_mod_r(cx, dot_mod_r(torch, a_s, sc_s)))
        last_s = [None]

        def step_strong():
            last_s[0] = ddist.msm_sharded_async(sc_s, pts_s, d.PT_ELEMENT, inputs_ready=True)[1]

        ms_s, _ = cx.time_device(step_strong, steps, 3)
        ok_s = bytes(last_s[0].cpu().numpy().tobytes()) == want_s
        sinfo = d.msm_stage_info()
        s_adds = ns * sinfo["W"] * (7 if sinfo["mixed"] else 8) * IMAD_PER_FQ_OP
        per_point = 7 * sinfo["W"] + 18 * (1 << (sinfo["c"] - 1)) * sinfo["W"] / ns
        out["strong_scaling_2p24"] = {
            "scaling": "strong", "total_units": n, "units_per_gpu": ns, "ms_per_step": ms_s,
            "value": n / (ms_s * 1e-3) / 1e6, "unit": "Mpoints/s", "window_c": sinfo["c"],
            "accumulate_ms_rank0": sinfo["ms"]["accumulate"],
            "accumulate_imad_frac_rank0": s_adds / (sinfo["ms"]["accumulate"] * 1e-3) / 1e9 / imad_peak,
            "whole_step_imad_frac": ns * per_point * IMAD_PER_FQ_OP / (ms_s * 1e-3) / 1e9 / imad_peak,
            "verified_sharded": ok_s,
            "api": "dist.msm_sharded_async: d377_msm_dev_async + NCCL all-gather + "
                   "d377_element_sum_result_dev, back to back"}
        verified = verified and ok_s

    # ---- one process driving all N GPUs through the C ABI (d377_msm_multi_dev) ------------------
    if world > 1 and logn == 24 and extras and not cx.args.no_single_process:
        out["single_process"] = single_process_multi(cx, n, steps)
        if out["single_process"] and out["single_process"].get("verified_sharded") is False:
            verified = False
    out["verified"] = verified

    # ---- end to end through the host-buffer C ABI ------------------------------------------------
    # Every step copies that step's inputs from pinned host memory to the device and reads
    # the result back.  `e2e` is the pipelined form a throughput-oriented caller uses
    # (d377_msm_submit / d377_msm_wait, two slots: the upload of step i+1 overlaps the
    # MSM of step i) over the Element wire image X||Y||Z||T the reference type holds;
    # `e2e_sync` is the plain blocking call; the other variants shrink the wire.
    if e2e:
        e2e_steps = max(2, min(steps, 10 if world == 1 else 6))

        def finish_step(res):
            if world == 1:
                return res
            part = torch.from_numpy(res[0]).to(cx.cuda)
            gathered = ddist.gather_partials(part)
            o_e, o_c = dev.element_sum(gathered)
            d.sync()
            return o_e.cpu().numpy(), o_c.cpu().numpy()

        def pipelined(h_sc, h_pts, fmt):
            res = [None]

            # up to `depth` MSMs in flight: two keep the link busy for large MSMs, small ones
            # (whose result arrives a tail after their accumulation) need three
            depth = 2 if n >= (1 << 23) else 3

            def run():
                for i in range(e2e_steps + depth):
                    if i >= depth:
                        res[0] = finish_step(d.msm_wait((i - depth) % 4))
                    if i < e2e_steps:
                        d.msm_submit(h_sc, h_pts, fmt, slot=i % 4)
            run()                      # warm both slots and the staging buffers
            dt = cx.time_host(run)
            return dt, bytes(res[0][1].tobytes())

        def entry(dt, got_enc, h2d, api):
            return {"value": world * n * e2e_steps / dt / 1e6, "unit": "Mpoints/s",
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 160, "steps": e2e_steps,
                    "ms_per_step": dt / e2e_steps * 1e3, "api": api, "verified": got_enc == want}

        h_sc = d.pinned_copy(sc.cpu().numpy())
        h_el = d.pinned_copy(pts.cpu().numpy())
        dt, enc = pipelined(h_sc, h_el, d.PT_ELEMENT)
        out["e2e"] = entry(dt, enc, n * 160,
                           "d377_msm_submit/d377_msm_wait, 2-3 MSMs in flight, pinned host buffers, "
                           "Element wire image X||Y||Z||T (D377_PT_ELEMENT, 128 B)")
        verified = verified and out["e2e"]["verified"]
        if extras:
            def run_sync():
                for _ in range(e2e_steps):
                    finish_step(d.vartime_multiscalar_mul(h_sc, h_el, d.PT_ELEMENT))
            dt = cx.time_host(run_sync)
            out["e2e_sync"] = {"value": world * n * e2e_steps / dt / 1e6, "unit": "Mpoints/s",
                               "ms_per_step": dt / e2e_steps * 1e3, "api": "d377_msm, blocking call per step"}
            # T = XY/Z is redundant and the Rust shim copies the coordinates one by one anyway
            # (Projective is not repr(C)): the T-less image moves 128 instead of 160 B per pair
            h_xyz = d.pinned_copy(h_el[:, :96])
            del h_el
            dt, enc = pipelined(h_sc, h_xyz, d.PT_XYZ)
            out["e2e_xyz"] = entry(dt, enc, n * 128, "same, Element wire image X||Y||Z (D377_PT_XYZ, 96 B)")
            del h_xyz
            # AffinePoint bases (64 B), the input type of the reference's VariableBaseMSM::msm
            # (ark_curve/element.rs:22-37)
            aff = dev.normalize(pts)
            d.sync()
            h_aff = d.pinned_copy(aff.cpu().numpy())
            del aff
            dt, enc = pipelined(h_sc, h_aff, d.PT_AFFINE)
            out["e2e_affine"] = entry(dt, enc, n * 96, "same, D377_PT_AFFINE bases (64 B)")
            del h_aff
            # VariableBaseMSM::msm with LONG-LIVED bases (batch_convert_to_mul_base once,
            # ark_curve/element.rs:27-37): d377_msm_bases_create uploads and normalises the
            # bases once, untimed; every step then moves only the 32-byte scalars.
            bases = d.MsmBases(device_ptr=pts.data_ptr(), n=n, point_format=d.PT_ELEMENT)
            dt, enc = pipelined(h_sc, bases, d.PT_BASES)
            eb = entry(dt, enc, n * 32, "d377_msm_bases_create once (untimed), then d377_msm_submit/"
                                        "d377_msm_wait with D377_PT_BASES")
            if world == 1:
                ms_b, _ = cx.time_device(lambda: dev.msm_async(sc, bases, inputs_ready=True), steps, 2)
                eb["device_resident_value"] = n / (ms_b * 1e-3) / 1e6
                eb["device_resident_ms_per_step"] = ms_b
            out["e2e_prepared_bases"] = eb
            bases.close()
            for key in ("e2e_xyz", "e2e_affine", "e2e_prepared_bases"):
                verified = verified and out[key]["verified"]
        out["verified"] = verified
    return out


def single_process_multi(cx: Ctx, n_total: int, steps: int):
    """Rank 0 alone drives every GPU of the box through d377_msm_multi_dev (one host thread
    per GPU inside the library, partial sums by peer copy) while the other ranks wait at a
    barrier: the path a single Rust process takes.  Strong scaling: ONE 2^24-pair MSM."""
    torch, d, dev = cx.torch, cx.d, cx.dev
    world = cx.world
    res = None
    cx.host_barrier()
    if cx.rank == 0:
        try:
            d.init_multi(list(range(world)))
            ns = n_total // world
            a_k, s_k, p_k = [], [], []
            for k in range(world):
                d.set_device(k)
                with torch.cuda.device(k):
                    g = torch.Generator(device="cuda:%d" % k).manual_seed(9000 + k)
                    a = torch.randint(0, 256, (ns, 32), dtype=torch.uint8, device="cuda:%d" % k, generator=g)
                    s = torch.randint(0, 256, (ns, 32), dtype=torch.uint8, device="cuda:%d" % k, generator=g)
                    a[:, 31] &= 3
                    s[:, 31] &= 3
                    torch.cuda.synchronize()
                    p = dev.fixed_base_mul(a, d.OUT_ELEMENT)
                    d.sync()
                a_k.append(a); s_k.append(s); p_k.append(p)
            d.set_device(-1)
            k_all = sum(dot_mod_r(torch, a, s) for a, s in zip(a_k, s_k)) % R_MODULUS
            want = expected_encoding(k_all)
            for _ in range(2):
                got = dev.msm_multi(s_k, p_k, d.PT_ELEMENT)
            for k in range(world):
                torch.cuda.synchronize(k)
            t0 = time.perf_counter()
            for _ in range(steps):
                got = dev.msm_multi(s_k, p_k, d.PT_ELEMENT)
            dt_blk = (time.perf_counter() - t0) / steps
            ok_blk = bytes(got[1].tobytes()) == want
            # asynchronous form: K calls enqueued back to back, one d377_multi_sync at the end
            oc_ring = torch.empty((steps + 3, 32), dtype=torch.uint8, device="cuda:0")
            for i in range(3):
                dev.msm_multi_async(s_k, p_k, d.PT_ELEMENT, out_encoding=oc_ring[i])
            dev.multi_sync()
            t0 = time.perf_counter()
            for i in range(steps):
                dev.msm_multi_async(s_k, p_k, d.PT_ELEMENT, out_encoding=oc_ring[3 + i])
            dev.multi_sync()
            dt = (time.perf_counter() - t0) / steps
            ok_async = all(bytes(row) == want for row in oc_ring.cpu().numpy())
            # the same MSM from HOST memory: d377_msm_multi uploads every GPU's slice over that
            # GPU's own PCIe link (all out of one pinned buffer) inside the timed region
            e2e_host = None
            if not cx.args.no_e2e:
                import numpy as np
                h_s = d.pinned_copy(np.concatenate([t.cpu().numpy() for t in s_k]))
                h_p = d.pinned_copy(np.concatenate([t.cpu().numpy() for t in p_k]))
                got_h = d.msm_multi(h_s, h_p, d.PT_ELEMENT, ngpu=world)
                hs = max(2, min(steps, 6))
                t0 = time.perf_counter()
                for _ in range(hs):
                    got_h = d.msm_multi(h_s, h_p, d.PT_ELEMENT, ngpu=world)
                dt_h = (time.perf_counter() - t0) / hs
                e2e_host = {"ms_per_step": dt_h * 1e3, "value": n_total / dt_h / 1e6, "unit": "Mpoints/s",
                            "h2d_bytes_per_step": n_total * 160, "d2h_bytes_per_step": 160, "steps": hs,
                            "api": "d377_msm_multi, pinned host buffers, blocking call per step",
                            "verified": bytes(got_h[1].tobytes()) == want}
                ok_async = ok_async and e2e_host["verified"]
                del h_s, h_p
            res = {"scaling": "strong", "total_units": n_total, "units_per_gpu": ns,
                   "ms_per_step": dt * 1e3, "value": n_total / dt / 1e6, "unit": "Mpoints/s",
                   "e2e": e2e_host,
                   "parallelism": "single process, %d GPUs, one host thread per GPU, partial sums by peer stores over NVLink" % world,
                   "api": "d377_msm_multi_dev_async back to back + d377_multi_sync",
                   "timing": "host wall clock from the first enqueue to the return of d377_multi_sync",
                   "blocking_call": {"ms_per_step": dt_blk * 1e3, "value": n_total / dt_blk / 1e6,
                                     "api": "d377_msm_multi_dev (result in host memory after every call)"},
                   "verified_sharded": ok_blk and ok_async}
            del a_k, s_k, p_k
        except Exception as ex:   # report, never hide
            res = {"error": repr(ex), "verified_sharded": False}
    cx.host_barrier()
    return res


# ---- the element-wise configs ----------------------------------------------------------------
def bench_elementwise(cx: Ctx, wl: str, logn: int, steps: int, warmup: int, e2e: bool) -> dict:
    torch, d, dev = cx.torch, cx.d, cx.dev
    n = 1 << logn
    raw = cx.rand(n)
    sc = cx.rand(n, scalar=True)
    el = dev.encode_to_curve(raw, d.OUT_ELEMENT) if wl in ("compress", "decompress", "pipeline") else None
    enc = dev.compress(el) if wl in ("decompress", "pipeline") else None
    d.sync()
    # e2e: pinned inputs AND pinned result buffers (d377_host_alloc), so the chunked
    # host API overlaps upload, kernel and download
    if wl == "encode":
        ins, h2d, d2h = (raw,), n * 32, n * 32
        step_dev = lambda: dev.encode_to_curve(raw, d.OUT_ENCODING)
        make_out = lambda: (d.pinned_empty((n, 32)),)
        step_e2e = lambda h, o: d.batch_encode_to_curve(h[0], d.OUT_ENCODING, out=o[0])
    elif wl == "hash":
        raw2 = cx.rand(n)
        ins, h2d, d2h = (raw, raw2), n * 64, n * 32
        step_dev = lambda: dev.hash_to_curve(raw, raw2, d.OUT_ENCODING)
        make_out = lambda: (d.pinned_empty((n, 32)),)
        step_e2e = lambda h, o: d.batch_hash_to_curve(h[0], h[1], d.OUT_ENCODING, out=o[0])
    elif wl == "fixed_base":
        ins, h2d, d2h = (sc,), n * 32, n * 32
        step_dev = lambda: dev.fixed_base_mul(sc, d.OUT_ENCODING)
        make_out = lambda: (d.pinned_empty((n, 32)),)
        step_e2e = lambda h, o: d.fixed_base_mul(h[0], d.OUT_ENCODING, out=o[0])
    elif wl == "compress":
        ins, h2d, d2h = (el,), n * 128, n * 32
        step_dev = lambda: dev.compress(el)
        make_out = lambda: (d.pinned_empty((n, 32)),)
        step_e2e = lambda h, o: d.batch_compress(h[0], out=o[0])
    elif wl == "decompress":
        ins, h2d, d2h = (enc,), n * 32, n * 129
        step_dev = lambda: dev.decompress(enc)
        make_out = lambda: (d.pinned_empty((n, 128)), d.pinned_empty((n,)))
        step_e2e = lambda h, o: d.batch_decompress(h[0], out=o[0], ok=o[1])
    else:
        ins, h2d, d2h = (enc, sc), n * 64, n * 33
        step_dev = lambda: dev.scalar_mul(enc, sc, d.PT_ENCODING, d.OUT_ENCODING)
        make_out = lambda: (d.pinned_empty((n, 32)), d.pinned_empty((n,)))
        step_e2e = lambda h, o: d.batch_scalar_mul(h[0], h[1], d.PT_ENCODING, d.OUT_ENCODING,
                                                   return_ok=True, out=o[0], ok=o[1])
    last = [None]

    def step_last():
        last[0] = step_dev()

    # inputs + outputs below the 126 MB L2: flush it between the timed iterations
    small = (h2d + d2h) < (126 << 20)
    sampler = ClockSampler(cx.local_rank)
    if cx.rank == 0:
        sampler.start()
    ms_step, launches = cx.time_device(step_last, steps, warmup, flush_l2=small)
    clocks = sampler.stop() if cx.rank == 0 else None
    unit = "Melem/s"
    out = {"value": cx.world * n / (ms_step * 1e-3) / 1e6, "unit": unit, "ms_per_step": ms_step,
           "gpu_launches": launches, "h2d": h2d, "d2h": d2h, "units": n, "clocks": clocks, "steps": steps,
           "l2": ("flushed between timed iterations (256 MiB write outside the event pairs)" if small else
                  "inputs + outputs (%.0f MiB) exceed the 126 MB L2" % ((h2d + d2h) / 2**20)),
           "outputs": (dict(zip(("elements", "ok"), last[0])) if wl == "decompress"
                       else {"encodings": last[0]})}
    imad_peak = d.imad_peak()
    peaks = measured_peaks()
    ach = n * OPS_OF[wl] * IMAD_PER_FQ_OP / (ms_step * 1e-3) / 1e9
    ach_bw = (h2d + d2h) / (ms_step * 1e-3) / 1e9
    out["roofline"] = {"bound": "imad", "kernel": wl, "achieved": ach, "peak": imad_peak,
                       "unit": "GIMAD/s (32x32->64 multiply-adds)", "frac": ach / imad_peak,
                       "issued_frac": n * WIDE_ISSUED[wl] / (ms_step * 1e-3) / 1e9 / imad_peak,
                       "traffic": NCU_TRAFFIC.get((wl, logn)), "launch_ms": ms_step,
                       "peak_source": "IMAD.WIDE.U32 issue-rate microbenchmark run in this process"}
    out["roofline_hbm"] = {"bound": "hbm", "kernel": wl, "achieved": ach_bw, "peak": peaks["hbm_gbs"],
                           "unit": "GB/s", "frac": ach_bw / peaks["hbm_gbs"], "traffic": None,
                           "peak_source": peaks["_source"]}
    if e2e:
        host = tuple(d.pinned_copy(t.cpu().numpy()) for t in ins)
        outb = make_out()
        e2e_steps = max(2, min(steps, 10))
        step_e2e(host, outb)           # warm the staging buffers

        def run():
            for _ in range(e2e_steps):
                step_e2e(host, outb)
        dt = cx.time_host(run)
        out["e2e"] = {"value": cx.world * n * e2e_steps / dt / 1e6, "unit": unit,
                      "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                      "ms_per_step": dt / e2e_steps * 1e3,
                      "api": "host-buffer C ABI, blocking call per step, pinned in/out buffers, chunk-pipelined"}
        del host, outb

    # ---- correctness spot check against the oracle (untimed) ---------------------------
    verified = None
    if cx.rank == 0:
        try:
            from oracle import c_oracle as co
            m = 2048
            if wl == "encode":
                r_h = raw[:m].cpu().numpy()
                verified = bool((d.batch_encode_to_curve(r_h, d.OUT_ENCODING)
                                 == co.encode_to_curve(r_h, out_enc=True, threads=8)).all())
            elif wl == "hash":
                r_h, r2_h = raw[:m].cpu().numpy(), raw2[:m].cpu().numpy()
                verified = bool((d.batch_hash_to_curve(r_h, r2_h, d.OUT_ENCODING)
                                 == co.hash_to_curve(r_h, r2_h, out_enc=True, threads=8)).all())
            elif wl == "fixed_base":
                # the timed launch's own output on a sample (the quartic-table path), against the
                # oracle's plain double-and-add
                s_h = sc[:256].cpu().numpy()
                got = dev.fixed_base_mul(sc, d.OUT_ENCODING)[:256].cpu().numpy()
                verified = bool((got == co.fixed_base(s_h, threads=8)).all())
            elif wl == "compress":
                e_h = el[:m].cpu().numpy()
                verified = bool((d.batch_compress(e_h) == co.compress(e_h, threads=8)).all())
            elif wl == "decompress":
                e_h = enc[:m].cpu().numpy()
                a_, b_ = d.batch_decompress(e_h), co.decompress(e_h, threads=8)
                verified = bool((a_[1] == b_[1]).all() and (d.batch_compress(a_[0]) == e_h).all())
            else:
                e_h, s_h = enc[:256].cpu().numpy(), sc[:256].cpu().numpy()
                verified = bool((d.batch_scalar_mul(e_h, s_h, d.PT_ENCODING, d.OUT_ENCODING)
                                 == co.pipeline(e_h, s_h, threads=8)[0]).all())
        except Exception as ex:
            verified = "check failed to run: %r" % (ex,)
    out["verified"] = verified
    return out


def config_entry(res: dict, cpu) -> dict:
    """The per-config record of the headline line."""
    rf = res["roofline"]
    e = {"value": res["value"], "unit": res["unit"], "ms_per_step": res["ms_per_step"],
         "roofline": {"bound": rf["bound"], "frac": rf["frac"], "issued_frac": rf["issued_frac"],
                      "achieved": rf["achieved"], "peak": rf["peak"], "unit": rf["unit"],
                      "kernel": rf["kernel"], "traffic": rf.get("traffic")},
         "e2e": res.get("e2e"), "cpu_baseline": cpu, "verified_vs_oracle": res["verified"],
         "steps": res.get("steps"), "clocks": res.get("clocks"), "l2": res.get("l2")}
    if "whole_step_frac" in rf:
        e["roofline"]["whole_step_frac"] = rf["whole_step_frac"]
    if "blocking_call" in res:
        e["blocking_call"] = res["blocking_call"]
    return e


def main_ours(args):
    cx = Ctx(args)
    d, world, rank = cx.d, cx.world, cx.rank
    wl = args.workload
    logn = args.logn or DEFAULT_LOGN[wl]
    n = 1 << logn
    steps, warmup = max(1, args.steps), max(args.warmup, 3)
    want_cpu = rank == 0 and world == 1 and not args.no_cpu_baseline
    failed = False
    if wl == "msm":
        res = bench_msm(cx, logn, steps, warmup, not args.no_e2e, extras=True)
    else:
        res = bench_elementwise(cx, wl, logn, steps, warmup, not args.no_e2e)
    outputs = res.pop("outputs")
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, outputs)
    cpu = None
    if want_cpu:
        cpu = cpu_baseline_of(wl, args.ref_logn or CPU_SAMPLE_LOGN[wl], 3)

    # ---- every other BASELINE config, in the same line (N = 1, default workload) ----------
    configs = None
    if wl == "msm" and world == 1 and not args.no_configs:
        configs = {}
        csteps = max(3, min(steps, 10))
        plan = [("pipeline", "pipeline", 16), ("encode", "encode", 22), ("hash", "hash", 22),
                ("fixed_base", "fixed_base", 24), ("compress", "compress", 22),
                ("decompress", "decompress", 22)]
        for name, w, ln in plan:
            r = bench_elementwise(cx, w, ln, csteps, 3, not args.no_e2e)
            c = cpu_baseline_of(w, CPU_SAMPLE_LOGN[w]) if want_cpu else None
            configs[name] = config_entry(r, c)
            configs[name]["workload"] = WORKLOAD_NAME[w].format(logn=ln)
            del r
            cx.torch.cuda.empty_cache()
        r = bench_msm(cx, 20, max(10, csteps), 3, not args.no_e2e, extras=False)
        c = cpu_baseline_of("msm", 20) if want_cpu else None
        configs["msm20"] = config_entry(r, c)
        configs["msm20"]["workload"] = WORKLOAD_NAME["msm"].format(logn=20)
        for name, e in configs.items():
            if e["verified_vs_oracle"] is not True:
                failed = True

    if rank == 0:
        line = {
            "metric": METRIC[wl], "value": res["value"], "unit": UNIT.get(wl, "Melem/s"),
            "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u32 (8x32-bit limb Montgomery, IMAD.WIDE)",
            "data": ("synthetic (torch CUDA RNG scalars; points P_i = a_i G from the fixed-base kernel, so that "
                     "the result has a known answer)" if wl == "msm" else
                     "synthetic (torch CUDA RNG bytes; points = encode_to_curve of random Fq)"),
            "config": {"workload": WORKLOAD_NAME[wl].format(logn=logn), "units_per_gpu": n,
                       "total_units": world * n,
                       "point_format": "Element X||Y||Z||T 128 B" if wl == "msm" else None,
                       "parallelism": ("point-slice sharding x%d, one process per GPU, 128 B NCCL all-gather" % world
                                       if world > 1 else "single GPU"),
                       "timed_call": ("d377_msm_dev_async back to back (tail of MSM k and sort of MSM k+1 "
                                      "overlap the bucket accumulation)" if wl == "msm" else "device-resident _dev call"),
                       "l2": res.get("l2") or "inputs (%.0f MiB per GPU) exceed the 126 MB L2" % (res["h2d"] / 2**20)},
            "roofline": res["roofline"], "roofline_hbm": res["roofline_hbm"],
            "cpu_baseline": cpu, "e2e": res.get("e2e"),
            "gpu_launches": res["gpu_launches"], "clocks": res.get("clocks"),
            "verified_vs_oracle": res["verified"],
        }
        for key in ("e2e_sync", "e2e_xyz", "e2e_affine", "e2e_prepared_bases", "blocking_call",
                    "strong_scaling_2p24", "single_process"):
            if key in res:
                line[key] = res[key]
        if "stages" in res:
            line["msm_stage_ms"] = res["stages"]
        if wl == "msm":
            line["verified_sharded"] = bool(res["verified"]) if world > 1 else None
            line["verified_known_answer"] = res["verified_known_answer"]
        if configs is not None:
            line["configs"] = configs
        print(json.dumps(line), flush=True)
        if res["verified"] is not True:
            failed = True
    if world > 1:
        # every rank agrees on the exit code
        t = cx.torch.tensor([1 if failed or res["verified"] is not True else 0], device=cx.cuda)
        cx.dist.all_reduce(t, op=cx.dist.ReduceOp.MAX)
        failed = bool(t.item())
        cx.dist.destroy_process_group()
    return 1 if failed else 0


if __name__ == "__main__":
    a = parse_args()
    sys.exit(main_reference(a) if a.impl == "reference" else main_ours(a))
