#!/usr/bin/env python3
"""Wave-quantisation probe of the one-element-per-thread kernels (developer tool):
decompress -> mul -> compress and compress at batch sizes around whole waves of
148 SMs x 4 CTAs x 128 threads = 75 776 elements."""
import sys

import torch

sys.path.insert(0, ".")
import decaf377_b200 as d
from decaf377_b200 import device as dev
from tools.quick_bench import timeit

d.init(0)
g = torch.Generator(device="cuda").manual_seed(1)
wave = 148 * 4 * 128
for n in (1 << 16, wave, wave + 128, 2 * wave, 1 << 18, 3 * wave, 4 * wave, 1 << 19):
    r = torch.randint(0, 256, (n, 32), dtype=torch.uint8, device="cuda", generator=g)
    sc = r.clone()
    sc[:, 31] &= 0x03
    el = dev.encode_to_curve(r, d.OUT_ELEMENT)
    enc = dev.compress(el)
    ms1 = timeit(lambda: dev.scalar_mul(enc, sc, d.PT_ENCODING, d.OUT_ENCODING), iters=3)
    ms2 = timeit(lambda: dev.compress(el), iters=10)
    print("n=%7d (%.3f waves): pipeline %.3f ms %.2f Melem/s   compress %.4f ms %.1f Melem/s" % (
        n, n / wave, ms1, n / ms1 / 1e3, ms2, n / ms2 / 1e3), flush=True)
