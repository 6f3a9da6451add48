#!/usr/bin/env python3
"""MSM stage timings (developer tool): python tools/tune_msm.py LOGN [c ...]"""
import os
import sys

import torch

sys.path.insert(0, ".")
import decaf377_b200 as d
from decaf377_b200 import device as dev

logn = int(sys.argv[1]) if len(sys.argv) > 1 else 20
cs = [int(x) for x in sys.argv[2:]] or [0]
d.init(0)
n = 1 << logn
g = torch.Generator(device="cuda").manual_seed(1)
r = torch.randint(0, 256, (n, 32), dtype=torch.uint8, device="cuda", generator=g)
sc = r.clone()
sc[:, 31] &= 0x03
el = dev.encode_to_curve(r, d.OUT_ELEMENT)
d.sync()
st = dev.engine_stream()
for c in cs:
    d.msm_set_window(c)
    for _ in range(2):
        dev.msm(sc, el)
    d.sync()
    t0 = torch.cuda.Event(enable_timing=True)
    t1 = torch.cuda.Event(enable_timing=True)
    iters = 5
    with torch.cuda.stream(st):
        t0.record()
    for _ in range(iters):
        dev.msm(sc, el)
    with torch.cuda.stream(st):
        t1.record()
    d.sync()
    t1.synchronize()
    ms = t0.elapsed_time(t1) / iters
    info = d.msm_stage_info()
    print("n=2^%d c=%d W=%d: %.3f ms  %.1f Mpt/s  %s" % (
        logn, info["c"], info["W"], ms, n / ms / 1e3,
        " ".join("%s=%.3f" % (k, v) for k, v in info["ms"].items())), flush=True)
    if os.environ.get("D377_TIMELINE"):
        for k, g in enumerate(d.msm_timeline()):
            print("   group %d: sorted %.2f  acc %.2f -> %.2f  tail_end %.2f" % (
                k, g["sorted"], g["acc_start"], g["acc_end"], g["tail_end"]), flush=True)
