"""Windowed MSM bases (d377_msm_bases_create_windowed): the table of window multiples
2^(c j) * P_i and the single-bucket-set MSM over it, against the oracle and the plain
prepared path, through every entry point."""
import ctypes as C
import os
import random
import subprocess
import sys

import numpy as np
import pytest

from decaf377_b200._lib import D377Error
from oracle import decaf377_ref as o
from tests.util import canon, np_bytes, oracle_points, oracle_scalars

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R = o.R
Q = o.Q
IDENTITY = (0, 1, 1, 0)


def _windows(c):
    return (252 + c - 1) // c


def _edge_scalars(n, seed):
    """0, 1, r - 1 and values at the digit boundaries of the windows the tests use
    (2^(c k) - 1, 2^(c k), K 2^(c k), (K + 1) 2^(c k)): the signed-digit carry then crosses
    windows.  The rest is seeded random."""
    edge = [0, 1, R - 1]
    for c in (4, 7, 11, 16, 21):
        K = 1 << (c - 1)
        for k in (1, 2, 5, 11):
            if c * k + c > 250:
                continue
            edge += [(1 << (c * k)) - 1, 1 << (c * k), K << (c * k), (K + 1) << (c * k), (1 << (c * (k + 1))) - 1]
    rnd = random.Random(seed)
    s = oracle_scalars("win/s%d" % seed, n)
    for i in range(n):
        s[i] = edge[i] if i < len(edge) else s[i]
    rnd.shuffle(s)
    return s


def _edge_points(n, seed):
    """identities, P / -P pairs, and projective representatives with a non-trivial Z."""
    P = oracle_points("win/p%d" % seed, n)
    rnd = random.Random(seed + 1)
    for i in range(n):
        if i % 7 == 3:
            P[i] = IDENTITY
        elif i % 7 == 5 and i > 0:
            P[i] = o.point_neg(P[i - 1])
    out = []
    for p in P:
        lam = rnd.randrange(2, Q)
        out.append(tuple(v * lam % Q for v in p))   # (lX : lY : lZ : lT), T = XY / Z still holds
    return out


def _formats(P):
    """the same points in every input format of the bases: Element, Encoding, AffinePoint, XYZ"""
    wire = np_bytes([o.point_to_wire(p) for p in P], 128)
    enc = np_bytes([o.compress(p) for p in P], 32)
    aff = np_bytes([o.fq_to_mont_bytes(x) + o.fq_to_mont_bytes(y) for x, y in (o.to_affine(p) for p in P)], 64)
    return {0: wire, 1: enc, 2: aff, 3: np.ascontiguousarray(wire[:, :96])}


@pytest.mark.parametrize("n", [1, 3, 33, 1000])
def test_windowed_matches_oracle_every_format(engine, n):
    P, s = _edge_points(n, n), _edge_scalars(n, n)
    S = canon(s)
    want = o.compress(o.vartime_multiscalar_mul(s, P))
    for fmt, pts in _formats(P).items():
        plain = engine.MsmBases(pts, fmt)
        assert engine.vartime_multiscalar_mul(S, plain)[1].tobytes() == want, fmt
        assert not engine.msm_stage_info()["windowed"]
        plain.close()
        for c in (4, 7, 11, 16, 0):
            win = engine.MsmBases(pts, fmt, windowed=True, c=c)
            assert win.c == (c or win.c) and win.windows == _windows(win.c)
            try:
                for groups in (1, 2, 3):
                    engine.msm_set_groups(groups)
                    got = engine.vartime_multiscalar_mul(S, win)[1].tobytes()
                    assert got == want, (fmt, c, groups)
                    info = engine.msm_stage_info()
                    assert info["windowed"] and info["c"] == win.c and info["W"] == win.windows
            finally:
                engine.msm_set_groups(0)
                win.close()


def _mont_scalars(s):
    return canon([v * (1 << 256) % R for v in s])


def test_windowed_every_entry_point(engine):
    import torch
    from decaf377_b200 import device as dev
    n = 5000
    P, s = oracle_points("win/e", n), oracle_scalars("win/e", n)
    W, S = np_bytes([o.point_to_wire(p) for p in P], 128), canon(s)
    want = engine.vartime_multiscalar_mul(S, W)[1].tobytes()
    assert engine.vartime_multiscalar_mul(S[:64], W[:64])[1].tobytes() == \
        o.compress(o.vartime_multiscalar_mul(s[:64], P[:64]))
    for c in (0, 11):
        win = engine.MsmBases(W, windowed=True, c=c)
        assert engine.vartime_multiscalar_mul(S, win)[1].tobytes() == want
        # pipelined host-buffer form; sub-chunks start inside the set and keep its stride
        for k in (1, 2, 4):
            engine.msm_set_host_chunks(k)
            try:
                engine.msm_submit(S, win, slot=1)
                assert engine.msm_wait(1)[1].tobytes() == want, (c, k)
            finally:
                engine.msm_set_host_chunks(0)
        d_s = torch.from_numpy(S).cuda()
        assert dev.msm(d_s, win)[1].cpu().numpy().tobytes() == want
        # back to back, both workspace sets in flight
        outs = [dev.msm_async(d_s, win, inputs_ready=True) for _ in range(3)]
        engine.sync()
        for _, oc in outs:
            assert oc.cpu().numpy().tobytes() == want
        # scalars in Montgomery form
        SM = _mont_scalars(s)
        assert engine.vartime_multiscalar_mul(SM, win, scalars_montgomery=True)[1].tobytes() == want
        assert dev.msm(torch.from_numpy(SM).cuda(), win, scalars_montgomery=True)[1].cpu().numpy().tobytes() == want
        win.close()


def test_windowed_prefixes_and_registry(engine):
    from decaf377_b200 import _lib
    lib = _lib.load()
    n = 3000
    P, s = oracle_points("win/r", n), oracle_scalars("win/r", n)
    W, S = np_bytes([o.point_to_wire(p) for p in P], 128), canon(s)
    win = engine.MsmBases(W, windowed=True, c=16)
    assert (win.n, win.c, win.windows) == (n, 16, 16) and win.nbytes >= n * 16 * 128
    plain = engine.MsmBases(W)
    assert (plain.c, plain.windows) == (0, 1) and plain.nbytes >= n * 128
    for m in (1, 100, 2999):
        assert engine.vartime_multiscalar_mul(S[:m], win)[1].tobytes() == \
            engine.vartime_multiscalar_mul(S[:m], plain)[1].tobytes(), m
    assert engine.msm_stage_info()["windowed"] is False
    engine.vartime_multiscalar_mul(S[:7], win)
    assert engine.msm_stage_info()["windowed"] is True
    oe = np.empty(128, np.uint8)
    S2 = np.concatenate([S, S[:1]])
    rc = lib.d377_msm(S2.ctypes.data_as(C.c_void_p), C.c_void_p(win.ptr), engine.PT_BASES, n + 1,
                      oe.ctypes.data_as(C.c_void_p), None)
    assert rc == _lib.ERR_INVALID_ARG                                  # n' > N
    rc = lib.d377_msm(S.ctypes.data_as(C.c_void_p), C.c_void_p(win.ptr + 128 * 5), engine.PT_BASES, 8,
                      oe.ctypes.data_as(C.c_void_p), None)
    assert rc == _lib.ERR_INVALID_ARG                                  # not a handle
    # a scalar >= r
    bad = S[:10].copy()
    bad[4] = np.frombuffer(R.to_bytes(32, "little"), np.uint8)
    with pytest.raises(D377Error) as ei:
        engine.vartime_multiscalar_mul(bad, win)
    assert ei.value.code == _lib.ERR_SCALAR_RANGE
    ptr = win.ptr
    win.close()
    plain.close()
    assert lib.d377_msm_bases_destroy(C.c_void_p(ptr)) == _lib.ERR_INVALID_ARG   # second destroy
    sz = C.c_size_t(0)
    assert lib.d377_msm_bases_info(C.c_void_p(ptr), C.byref(sz), None, None, None) == _lib.ERR_INVALID_ARG
    # window widths outside [4, 22]
    for c in (3, 23, -1):
        with pytest.raises(D377Error) as ei:
            engine.MsmBases(W[:10], windowed=True, c=c)
        assert ei.value.code == _lib.ERR_INVALID_ARG


def test_windowed_dev_refuses_too_many_records_before_reading(engine):
    """n * W >= 2^31 is refused by the _dev twin before anything is allocated or read: the
    device buffer holds 4 points, n claims ~2^31 / 63 of them."""
    import torch
    from decaf377_b200 import _lib
    small = torch.zeros((4, 128), dtype=torch.uint8, device="cuda")
    n = (1 << 31) // 63 + 1
    with pytest.raises(D377Error) as ei:
        engine.MsmBases(device_ptr=small.data_ptr(), n=n, point_format=engine.PT_ELEMENT, windowed=True, c=4)
    assert ei.value.code == _lib.ERR_INVALID_ARG
    with pytest.raises(D377Error) as ei:
        engine.MsmBases(device_ptr=small.data_ptr(), n=(1 << 31) // 12 + 1, point_format=engine.PT_ELEMENT,
                        windowed=True, c=22)
    assert ei.value.code == _lib.ERR_INVALID_ARG
    engine.sync()


def test_windowed_known_answer_2p22(engine):
    """P_i = a_i G, 2^22 pairs: the result is (sum a_i s_i mod r) G (bench.py's check)."""
    import torch
    from bench import dot_mod_r, expected_encoding
    from decaf377_b200 import device as dev
    n = 1 << 22
    g = torch.Generator(device="cuda")
    g.manual_seed(2222)
    a = torch.randint(0, 256, (n, 32), dtype=torch.uint8, device="cuda", generator=g)
    s = torch.randint(0, 256, (n, 32), dtype=torch.uint8, device="cuda", generator=g)
    a[:, 31] &= 0x03
    s[:, 31] &= 0x03
    pts = dev.fixed_base_mul(a, engine.OUT_ELEMENT)
    engine.sync()
    want = expected_encoding(dot_mod_r(torch, a, s))
    win = engine.MsmBases(device_ptr=pts.data_ptr(), n=n, point_format=engine.PT_ELEMENT, windowed=True)
    plain = engine.MsmBases(device_ptr=pts.data_ptr(), n=n, point_format=engine.PT_ELEMENT)
    try:
        got = dev.msm(s, win)[1].cpu().numpy().tobytes()
        assert engine.msm_stage_info()["windowed"]
        assert got == want
        assert dev.msm(s, plain)[1].cpu().numpy().tobytes() == want
    finally:
        win.close()
        plain.close()


def test_c_host_program_drives_windowed_bases(tmp_path):
    exe = tmp_path / "abi_windowed_smoke"
    libdir = os.path.join(ROOT, "decaf377_b200")
    cmd = ["gcc", "-O1", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
           os.path.join(ROOT, "tests", "abi_windowed_smoke.c"), "-o", str(exe),
           "-L", libdir, "-ldecaf377_b200", "-Wl,-rpath," + libdir]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "abi_windowed_smoke: all checks passed" in r.stdout


def test_windowed_table_points_are_on_the_curve_in_the_debug_build():
    """k_msm_bases_double runs the on-curve predicate in the -DD377_DEBUG_ON_CURVE build."""
    if not os.path.exists(os.path.join(ROOT, "decaf377_b200", "libdecaf377_b200_dbg.so")):
        pytest.skip("debug library not built (python -m decaf377_b200.build --debug)")
    code = (
        "import numpy as np, decaf377_b200 as d\n"
        "from tests.util import np_bytes, oracle_points, oracle_scalars, canon\n"
        "from oracle import decaf377_ref as o\n"
        "d.init(0)\n"
        "P, s = oracle_points('win/dbg', 300), oracle_scalars('win/dbg', 300)\n"
        "W = np_bytes([o.point_to_wire(p) for p in P], 128)\n"
        "f0, c0 = d.debug_counts()\n"
        "b = d.MsmBases(W, windowed=True, c=5)\n"
        "assert d.vartime_multiscalar_mul(canon(s), b)[1].tobytes() == d.vartime_multiscalar_mul(canon(s), W)[1].tobytes()\n"
        "f1, c1 = d.debug_counts()\n"
        "assert d.debug_build() >= 1 and f1 == f0 and c1 - c0 >= 300 * (b.windows - 1), (f0, f1, c0, c1)\n"
        "print('debug ok', c1 - c0)\n")
    env = dict(os.environ, D377_DEBUG_LIB="1")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert r.returncode == 0 and "debug ok" in r.stdout, r.stdout + r.stderr
