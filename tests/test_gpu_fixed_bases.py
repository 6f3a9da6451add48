"""Prepared fixed bases (d377_fixed_bases_create / d377_fixed_bases_mul): window tables of k
caller-chosen points and out_i = sum_j s_ij B_j over them, against the oracle, the generator
path and per-base products, through every entry point, with every refusal of the ABI."""
import ctypes as C
import os
import random
import subprocess
import sys

import numpy as np
import pytest

from decaf377_b200._lib import D377Error
from oracle import c_oracle
from oracle import decaf377_ref as o
from tests.util import np_bytes, oracle_points

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R = o.R
Q = o.Q
IDENTITY = (0, 1, 1, 0)
M256 = (1 << 256) - 1
TABLE_BYTES = (16 * (1 << 15) + 1) * 96


def _edge_list():
    """Scalars that stress the signed 16-bit windows: 0, 1, r - 1, r, 2r, the carry out of the
    top window (2^256 - 1, 2^255), every window boundary and alternating +-2^15 digits."""
    edge = [0, 1, R - 1, R, 2 * R, M256, 1 << 255]
    for w in range(16):
        b = 1 << (16 * w)
        edge += [(b - 1) & M256, b, (1 << 15) * b, ((1 << 15) + 1) * b & M256]
    alt = sum(((1 << 15) if w % 2 == 0 else -(1 << 15)) << (16 * w) for w in range(16))
    edge += [alt & M256, alt % R, sum(0x8000 << (16 * w) for w in range(16)), sum(0x8001 << (16 * w) for w in range(16))]
    return edge


EDGE = _edge_list()


def _scalars(n, k, seed):
    """n rows of k 256-bit integers: the edge list spread over the rows (row i, column j gets
    edge[(i * k + j) % len] in the first rows), the rest uniform over [0, 2^256)."""
    rnd = random.Random(seed)
    rows = [[rnd.getrandbits(256) for _ in range(k)] for _ in range(n)]
    for t in range(min(len(EDGE) * k, n * k)):
        i, j = divmod(t, k)
        rows[i][j] = EDGE[(t + j) % len(EDGE)]
    return rows


def _sc_bytes(rows):
    k = len(rows[0])
    return np.frombuffer(b"".join(v.to_bytes(32, "little") for r in rows for v in r), np.uint8).reshape(-1, k, 32).copy()


def _bases(k, seed):
    """k bases covering: a random projective scale, the identity, a P / -P pair, G itself and
    the same point twice (as two different representatives)."""
    P = oracle_points("fb/b%d" % seed, 4)
    kinds = {1: [P[0]], 2: [P[1], o.point_neg(P[1])], 3: [o.GENERATOR, P[2], P[2]],
             5: [P[3], IDENTITY, P[0], o.point_neg(P[0]), o.GENERATOR]}[k]
    rnd = random.Random(seed)
    out = []
    for p in kinds:
        lam = rnd.randrange(2, Q)
        out.append(tuple(v * lam % Q for v in p))   # (lX : lY : lZ : lT)
    return out


def _formats(P):
    wire = np_bytes([o.point_to_wire(p) for p in P], 128)
    enc = np_bytes([o.compress(p) for p in P], 32)
    aff = np_bytes([o.fq_to_mont_bytes(x) + o.fq_to_mont_bytes(y) for x, y in (o.to_affine(p) for p in P)], 64)
    return {0: wire, 1: enc, 2: aff, 3: np.ascontiguousarray(wire[:, :96])}


def _ref_encodings(P, rows):
    """decaf377_ref: scalar_mul + point_add + compress, row by row."""
    out = []
    for r in rows:
        acc = IDENTITY
        for p, s in zip(P, r):
            acc = o.point_add(acc, o.scalar_mul(p, s))
        out.append(o.compress(acc))
    return out


def _c_oracle_encodings(P, S):
    """The C oracle over whole columns: scalar_mul per base, add, compress.  S: [n, k, 32]."""
    n, k = S.shape[0], S.shape[1]
    th = c_oracle.threads_default()
    acc = None
    for j, p in enumerate(P):
        pts = np.repeat(np.frombuffer(o.point_to_wire(p), np.uint8).reshape(1, 128), n, axis=0)
        prod = c_oracle.scalar_mul(pts, np.ascontiguousarray(S[:, j]), threads=th)
        acc = prod if acc is None else c_oracle.add(acc, prod, threads=th)
    return c_oracle.compress(acc, threads=th)


def _canonical_limbs(el):
    limbs = el.reshape(-1, 32)
    vals = [int.from_bytes(limbs[i].tobytes(), "little") for i in range(limbs.shape[0])]
    return all(v < Q for v in vals)


@pytest.mark.parametrize("n", [1, 127, 128, 129, 5000])
@pytest.mark.parametrize("k", [1, 2, 3, 5])
def test_fixed_bases_match_oracle_every_format(engine, k, n):
    P = _bases(k, 10 * k + n % 7)
    rows = _scalars(n, k, 1000 * k + n)
    S = _sc_bytes(rows)
    want = _c_oracle_encodings(P, S)
    m = min(n, 12)      # the first planted rows, against the Python reference
    assert [want[i].tobytes() for i in range(m)] == _ref_encodings(P, rows[:m])
    for fmt, pts in _formats(P).items():
        fb = engine.FixedBases(pts, fmt)
        try:
            assert (fb.k, len(fb), fb.nbytes) == (k, k, k * TABLE_BYTES)
            enc = fb.mul(S, engine.OUT_ENCODING)
            assert np.array_equal(enc, want), (fmt, np.nonzero((enc != want).any(axis=1))[0][:8])
            el = fb.mul(S, engine.OUT_ELEMENT)
            assert np.array_equal(c_oracle.compress(el, threads=c_oracle.threads_default()), want), fmt
            assert _canonical_limbs(el), fmt
        finally:
            fb.close()


def test_k1_over_special_bases(engine):
    """k = 1 over the identity, G and a P with a projective scale, every format."""
    rows = _scalars(300, 1, 7)
    S = _sc_bytes(rows)
    for p in (IDENTITY, o.GENERATOR, _bases(1, 3)[0]):
        want = _c_oracle_encodings([p], S)
        assert [want[i].tobytes() for i in range(20)] == _ref_encodings([p], rows[:20])
        for fmt, pts in _formats([p]).items():
            fb = engine.FixedBases(pts, fmt)
            assert np.array_equal(fb.mul(S[:, 0], engine.OUT_ENCODING), want), fmt
            fb.close()


def test_generator_set_is_byte_identical_to_fixed_base_mul(engine):
    """FixedBases([G]) walks the same table as d377_fixed_base_mul's Edwards path: Element
    outputs are the same bytes; encodings too (the generator call takes the quartic path at
    this size, which gives the reference's bytes as well)."""
    n = (1 << 20) + 7
    rng = np.random.default_rng(20)
    S = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    S[:len(EDGE)] = _sc_bytes([[v] for v in EDGE])[:, 0]
    S[-len(EDGE):] = _sc_bytes([[v] for v in EDGE])[:, 0]
    G = np.frombuffer(o.point_to_wire(o.GENERATOR), np.uint8).reshape(1, 128)
    fb = engine.FixedBases(G)
    try:
        for fmt in (engine.OUT_ELEMENT, engine.OUT_ENCODING):
            assert np.array_equal(fb.mul(S, fmt), engine.fixed_base_mul(S, fmt)), fmt
    finally:
        fb.close()
    idx = list(range(len(EDGE))) + list(range(0, n, 9973))
    want = c_oracle.fixed_base(S[idx])
    got = engine.fixed_base_mul(S[idx], engine.OUT_ENCODING)
    assert np.array_equal(got, want)


def test_linearity_at_scale(engine):
    """FixedBases([B, C]).mul([s, t]) == compress(FixedBases([B]).mul(s) + FixedBases([C]).mul(t))
    on every row of 2^22 + 3; the C oracle checks a strided sample and both ends."""
    n = (1 << 22) + 3
    B, Cp = oracle_points("fb/lin", 2)
    rng = np.random.default_rng(22)
    S = rng.integers(0, 256, (n, 2, 32), dtype=np.uint8)
    planted = _sc_bytes(_scalars(len(EDGE), 2, 5))
    S[:len(EDGE)] = planted
    S[-len(EDGE):] = planted
    wb = np.frombuffer(o.point_to_wire(B), np.uint8).reshape(1, 128)
    wc = np.frombuffer(o.point_to_wire(Cp), np.uint8).reshape(1, 128)
    both = engine.FixedBases(np.concatenate([wb, wc]))
    fb_b, fb_c = engine.FixedBases(wb), engine.FixedBases(wc)
    try:
        got = both.mul(S, engine.OUT_ENCODING)
        parts = engine.batch_add(fb_b.mul(np.ascontiguousarray(S[:, 0])), fb_c.mul(np.ascontiguousarray(S[:, 1])))
        assert np.array_equal(got, engine.batch_compress(parts))
        del parts
    finally:
        for f in (both, fb_b, fb_c):
            f.close()
    idx = np.array(list(range(64)) + list(range(64, n - 64, 65537)) + list(range(n - 64, n)))
    want = _c_oracle_encodings([B, Cp], np.ascontiguousarray(S[idx]))
    assert np.array_equal(got[idx], want)


def test_every_entry_point(engine):
    import torch
    from decaf377_b200 import device as dev
    n = (1 << 19) + 5           # three chunks of the host-buffer pipeline
    P = _bases(2, 77)
    pts = _formats(P)[0]
    rng = np.random.default_rng(5)
    S = rng.integers(0, 256, (n, 2, 32), dtype=np.uint8)
    S[:40] = _sc_bytes(_scalars(40, 2, 9))
    fb = engine.FixedBases(pts)
    try:
        want = fb.mul(S, engine.OUT_ENCODING)
        idx = list(range(40)) + list(range(40, n, 8191)) + [n - 1]
        assert np.array_equal(want[idx], _c_oracle_encodings(P, np.ascontiguousarray(S[idx])))
        want_el = fb.mul(S, engine.OUT_ELEMENT)
        # pinned buffers, and a caller-supplied out
        Sp = engine.pinned_copy(S)
        out = engine.pinned_empty((n, 32))
        assert np.array_equal(fb.mul(Sp, engine.OUT_ENCODING, out=out), want)
        outp = engine.pinned_empty((n, 128))
        assert np.array_equal(fb.mul(Sp, engine.OUT_ELEMENT, out=outp), want_el)
        # device-resident, through torch
        dS = torch.from_numpy(S).cuda()
        assert np.array_equal(dev.fixed_bases_mul(fb, dS, engine.OUT_ENCODING).cpu().numpy(), want)
        assert np.array_equal(dev.fixed_bases_mul(fb, dS, engine.OUT_ELEMENT).cpu().numpy(), want_el)
        # scalars in the reference's Montgomery form (the canonical value of each is s mod r)
        m = 3000
        rows = [[int.from_bytes(S[i, j].tobytes(), "little") for j in range(2)] for i in range(m)]
        SM = _sc_bytes([[v * (1 << 256) % R for v in r] for r in rows])
        SC = _sc_bytes([[v % R for v in r] for r in rows])
        ref = fb.mul(SC, engine.OUT_ENCODING)
        assert np.array_equal(ref, want[:m])       # s and s mod r: the same element
        assert np.array_equal(fb.mul(SM, engine.OUT_ENCODING, scalars_montgomery=True), ref)
        mont = engine.SCALARS_MONTGOMERY
        assert np.array_equal(dev.fixed_bases_mul(fb, torch.from_numpy(SM).cuda(), engine.OUT_ENCODING | mont)
                              .cpu().numpy(), ref)
        assert np.array_equal(engine.batch_compress(fb.mul(SM, engine.OUT_ELEMENT, scalars_montgomery=True)), ref)
        # n = 0
        assert fb.mul(np.zeros((0, 2, 32), np.uint8)).shape == (0, 128)
        assert dev.fixed_bases_mul(fb, torch.zeros((0, 2, 32), dtype=torch.uint8, device="cuda")).shape == (0, 128)
        # bases from device memory
        fb_dev = engine.FixedBases(device_ptr=torch.from_numpy(_formats(P)[1]).cuda().data_ptr(),
                                   point_format=engine.PT_ENCODING, k=2)
        engine.sync()
        assert np.array_equal(fb_dev.mul(S[:5000], engine.OUT_ENCODING), want[:5000])
        fb_dev.close()
    finally:
        fb.close()


def test_k1_accepts_flat_scalars_and_shapes_are_checked(engine):
    P = _bases(1, 4)
    fb = engine.FixedBases(_formats(P)[0])
    fb2 = engine.FixedBases(_formats(_bases(2, 4))[0])
    try:
        S = _sc_bytes(_scalars(10, 1, 4))
        assert np.array_equal(fb.mul(S[:, 0]), fb.mul(S))
        for bad in (np.zeros((10, 2, 32), np.uint8), np.zeros((10, 31), np.uint8), np.zeros((320,), np.uint8)):
            with pytest.raises(ValueError):
                fb.mul(bad)
        for bad in (np.zeros((10, 32), np.uint8), np.zeros((10, 1, 32), np.uint8), np.zeros((10, 2, 16), np.uint8)):
            with pytest.raises(ValueError):
                fb2.mul(bad)
    finally:
        fb.close()
        fb2.close()
    with pytest.raises(ValueError):
        fb.mul(S)                      # closed


def _info(lib, ptr):
    kk, nb = C.c_size_t(0), C.c_size_t(0)
    return lib.d377_fixed_bases_info(C.c_void_p(ptr), C.byref(kk), C.byref(nb))


def test_refusals_register_nothing(engine):
    import torch
    from decaf377_b200 import _lib
    lib = _lib.load()
    P = _bases(2, 11)
    W = _formats(P)[0]
    E = _formats(P)[1]
    sentinel = 0x5A5A5A5A00
    out = C.c_void_p(sentinel)

    def create(pts, fmt, k, handle=True):
        out.value = sentinel
        rc = lib.d377_fixed_bases_create(None if pts is None else pts.ctypes.data_as(C.c_void_p), fmt, k,
                                         C.byref(out) if handle else None)
        assert out.value == sentinel and _info(lib, sentinel) == _lib.ERR_INVALID_ARG
        return rc

    assert create(W, engine.PT_ELEMENT, 0) == _lib.ERR_INVALID_ARG                 # k = 0
    assert create(W, engine.PT_BASES, 2) == _lib.ERR_INVALID_ARG                   # bad format
    assert create(W, -1, 2) == _lib.ERR_INVALID_ARG
    assert create(None, engine.PT_ELEMENT, 2) == _lib.ERR_INVALID_ARG              # null points
    assert create(W, engine.PT_ELEMENT, 2, handle=False) == _lib.ERR_INVALID_ARG   # null handle slot
    assert create(W, engine.PT_ELEMENT, 1 << 60) == _lib.ERR_INVALID_ARG           # byte count overflows
    # an invalid encoding among the bases (tests/encoding.rs:28-52)
    Eb = E.copy()
    Eb[1] = 0
    Eb[1, 0] = 1
    assert create(Eb, engine.PT_ENCODING, 2) == _lib.ERR_INVALID_ENCODING
    with pytest.raises(D377Error) as ei:
        engine.FixedBases(Eb, engine.PT_ENCODING)
    assert ei.value.code == _lib.ERR_INVALID_ENCODING
    # k = 2^20 through _dev over a 4-point buffer: refused before anything is read
    small = torch.zeros((4, 128), dtype=torch.uint8, device="cuda")
    out.value = sentinel
    rc = lib.d377_fixed_bases_create_dev(C.c_void_p(small.data_ptr()), engine.PT_ELEMENT, 1 << 20, C.byref(out))
    assert rc == _lib.ERR_CUDA and out.value == sentinel
    assert str((1 << 20) * TABLE_BYTES) in lib.d377_last_error().decode()
    engine.sync()
    # mul / info / destroy on handles that are not live fixed-bases handles
    fb = engine.FixedBases(W)
    msm = engine.MsmBases(W)
    S = _sc_bytes(_scalars(8, 2, 1))
    sp = S.ctypes.data_as(C.c_void_p)
    res = np.empty((8, 32), np.uint8)
    rp = res.ctypes.data_as(C.c_void_p)
    for h in (msm.ptr, fb.ptr + 96, 0, sentinel):
        assert lib.d377_fixed_bases_mul(C.c_void_p(h), sp, 8, rp, engine.OUT_ENCODING) == _lib.ERR_INVALID_ARG
        assert lib.d377_fixed_bases_mul_dev(C.c_void_p(h), sp, 0, rp, engine.OUT_ENCODING) == _lib.ERR_INVALID_ARG
        assert _info(lib, h) == _lib.ERR_INVALID_ARG
        if h:
            assert lib.d377_fixed_bases_destroy(C.c_void_p(h)) == _lib.ERR_INVALID_ARG
    # bad out_format, null scalars / out
    for fmt in (2, -1):
        assert lib.d377_fixed_bases_mul(C.c_void_p(fb.ptr), sp, 8, rp, fmt) == _lib.ERR_INVALID_ARG
    assert lib.d377_fixed_bases_mul(C.c_void_p(fb.ptr), None, 8, rp, engine.OUT_ENCODING) == _lib.ERR_INVALID_ARG
    assert lib.d377_fixed_bases_mul(C.c_void_p(fb.ptr), sp, 8, None, engine.OUT_ENCODING) == _lib.ERR_INVALID_ARG
    # a fixed-bases handle is not a D377_PT_BASES handle of the MSM
    oe = np.empty(128, np.uint8)
    rc = lib.d377_msm(np.ascontiguousarray(S[:, 0]).ctypes.data_as(C.c_void_p), C.c_void_p(fb.ptr),
                      engine.PT_BASES, 2, oe.ctypes.data_as(C.c_void_p), None)
    assert rc == _lib.ERR_INVALID_ARG
    assert lib.d377_msm_bases_info(C.c_void_p(fb.ptr), None, None, None, None) == _lib.ERR_INVALID_ARG
    assert lib.d377_msm_bases_destroy(C.c_void_p(fb.ptr)) == _lib.ERR_INVALID_ARG
    assert _info(lib, fb.ptr) == _lib.OK
    # destroy twice; a destroyed handle is dead everywhere
    ptr = fb.ptr
    fb.close()
    msm.close()
    assert lib.d377_fixed_bases_destroy(C.c_void_p(ptr)) == _lib.ERR_INVALID_ARG
    assert _info(lib, ptr) == _lib.ERR_INVALID_ARG
    assert lib.d377_fixed_bases_mul(C.c_void_p(ptr), sp, 8, rp, engine.OUT_ENCODING) == _lib.ERR_INVALID_ARG
    assert lib.d377_fixed_bases_destroy(None) == _lib.OK


def test_shutdown_returns_the_tables_memory():
    """A child process creates 4 tables (192 MiB), shuts the library down without destroying
    them, and sees the device memory come back."""
    code = (
        "import numpy as np, torch, decaf377_b200 as d\n"
        "from oracle import decaf377_ref as o\n"
        "from tests.util import np_bytes, oracle_points\n"
        "d.init(0)\n"
        "W = np_bytes([o.point_to_wire(p) for p in oracle_points('fb/shut', 4)], 128)\n"
        "f0 = torch.cuda.mem_get_info(0)[0]\n"
        "fb = d.FixedBases(W)\n"
        "f1 = torch.cuda.mem_get_info(0)[0]\n"
        "d.shutdown()\n"
        "f2 = torch.cuda.mem_get_info(0)[0]\n"
        "mib = 1 << 20\n"
        "assert f0 - f1 >= 190 * mib and f2 - f1 >= 190 * mib, (f0 // mib, f1 // mib, f2 // mib)\n"
        "print('shutdown ok', (f0 - f1) // mib, (f2 - f1) // mib)\n")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0 and "shutdown ok" in r.stdout, r.stdout + r.stderr


def test_handle_of_another_device_is_refused(engine):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from decaf377_b200 import _lib
    lib = _lib.load()
    engine.init_multi([0, 1])
    W = _formats(_bases(1, 12))[0]
    engine.set_device(1)
    try:
        fb1 = engine.FixedBases(W)
    finally:
        engine.set_device(-1)
    S = _sc_bytes(_scalars(4, 1, 2))
    res = np.empty((4, 32), np.uint8)
    rc = lib.d377_fixed_bases_mul(C.c_void_p(fb1.ptr), S.ctypes.data_as(C.c_void_p), 4,
                                  res.ctypes.data_as(C.c_void_p), engine.OUT_ENCODING)
    assert rc == _lib.ERR_INVALID_ARG
    assert _info(lib, fb1.ptr) == _lib.ERR_INVALID_ARG
    engine.set_device(1)
    try:
        assert _info(lib, fb1.ptr) == _lib.OK
        fb1.close()
    finally:
        engine.set_device(-1)


def test_c_host_program_drives_fixed_bases(tmp_path):
    exe = tmp_path / "abi_fixed_bases_smoke"
    libdir = os.path.join(ROOT, "decaf377_b200")
    cmd = ["gcc", "-O1", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
           os.path.join(ROOT, "tests", "abi_fixed_bases_smoke.c"), "-o", str(exe),
           "-L", libdir, "-ldecaf377_b200", "-Wl,-rpath," + libdir]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "abi_fixed_bases_smoke: all checks passed" in r.stdout


def test_fixed_bases_points_are_on_the_curve_in_the_debug_build():
    """k_fb_load and k_fixed_base run the on-curve predicate in the -DD377_DEBUG_ON_CURVE build."""
    if not os.path.exists(os.path.join(ROOT, "decaf377_b200", "libdecaf377_b200_dbg.so")):
        pytest.skip("debug library not built (python -m decaf377_b200.build --debug)")
    code = (
        "import numpy as np, decaf377_b200 as d\n"
        "from tests.test_gpu_fixed_bases import _bases, _formats, _scalars, _sc_bytes, _c_oracle_encodings\n"
        "d.init(0)\n"
        "P = _bases(3, 1)\n"
        "S = _sc_bytes(_scalars(200, 3, 1))\n"
        "want = _c_oracle_encodings(P, S)\n"
        "f0, c0 = d.debug_counts()\n"
        "for fmt, pts in _formats(P).items():\n"
        "    fb = d.FixedBases(pts, fmt)\n"
        "    assert np.array_equal(fb.mul(S, d.OUT_ENCODING), want), fmt\n"
        "    assert np.array_equal(d.batch_compress(fb.mul(S, d.OUT_ELEMENT)), want), fmt\n"
        "    fb.close()\n"
        "f1, c1 = d.debug_counts()\n"
        "assert d.debug_build() >= 1 and f1 == f0 and c1 - c0 >= 4 * (3 + 2 * 200), (f0, f1, c0, c1)\n"
        "print('debug ok', c1 - c0)\n")
    env = dict(os.environ, D377_DEBUG_LIB="1")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert r.returncode == 0 and "debug ok" in r.stdout, r.stdout + r.stderr
