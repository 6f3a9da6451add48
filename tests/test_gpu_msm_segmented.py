"""Many independent MSMs in one segmented Pippenger (d377_msm_segmented / _dev): against the
oracle and an exact known answer, at every window width, across chunk boundaries, against
d377_batch_msm and d377_msm, through every entry point, with every refusal of the ABI."""
import ctypes as C
import os
import random
import subprocess
import sys

import numpy as np
import pytest

from decaf377_b200._lib import D377Error
from oracle import c_oracle as co
from oracle import decaf377_ref as o
from tests.util import canon, oracle_points, wire

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R = o.R
M256 = (1 << 256) - 1
BUDGET = 1 << 30          # bytes of bucket sums per chunk


def _geom(c):
    return c, -(-257 // c), 1 << (c - 1)


def _mont(vals):
    return canon([v % R * (1 << 256) % R for v in vals])


def _window_edges(c):
    """Scalars for width c: all ones in a window, digits +K and -(K - 1) (raw K and K + 1), the
    carry through every window (2^256 - 1) and the top windows."""
    _, W, K = _geom(c)
    out = [0, 1, R - 1, R, 2 * R, 1 << 255, M256]
    for w in (0, 1, W // 2, W - 2, W - 1):
        sh = w * c
        out += [(((1 << c) - 1) << sh) & M256, (K << sh) & M256, ((K + 1) << sh) & M256]
    return out


def _kat(d, n, tag):
    """Known-answer pairs: P_i = a_i G (fixed-base path), so a segment's MSM is
    (sum s_i a_i mod r) G whatever the scalars are."""
    rnd = random.Random(tag)
    a = [rnd.randrange(1, R) for _ in range(n)]
    return a, d.fixed_base_mul(canon(a), d.OUT_ELEMENT)


def _expected(d, s, a, off):
    ks = [sum(s[i] * a[i] for i in range(int(off[j]), int(off[j + 1]))) % R for j in range(len(off) - 1)]
    return d.fixed_base_mul(canon(ks), d.OUT_ENCODING)


def _place(s, off, vals):
    """Put `vals` on the first and last pair of the segments, round robin."""
    k = 0
    for j in range(len(off) - 1):
        lo, hi = int(off[j]), int(off[j + 1])
        for i in {lo, hi - 1} if hi > lo else ():
            s[i] = vals[k % len(vals)]
            k += 1
    return s


SIZES = [0, 1, 3, 0, 2, 31, 32, 33, 64, 100, 1, 0, 7]


def test_oracle_parity_every_input_format(engine):
    """Encodings byte for byte against the C oracle's Pippenger, segment by segment, for
    Element, Encoding, AffinePoint and X||Y||Z inputs, with and without Montgomery scalars."""
    d = engine
    n = sum(SIZES)
    off = np.cumsum([0] + SIZES).astype(np.uint32)
    P = oracle_points("seg/parity", n)
    rnd = random.Random(5)
    s = [rnd.randrange(0, 1 << 256) for _ in range(n)]
    s = _place(s, off, _window_edges(8))
    W = wire(P)
    want = [co.msm_pippenger(canon([v % R for v in s[int(off[j]):int(off[j + 1])]]),
                             W[int(off[j]):int(off[j + 1])])[1].tobytes() for j in range(len(SIZES))]
    S, SM = canon(s), _mont(s)
    E = d.batch_compress(W)
    inputs = {d.PT_ELEMENT: W, d.PT_ENCODING: E, d.PT_AFFINE: d.batch_normalize(W), d.PT_XYZ: W[:, :96].copy()}
    for fmt, pts in inputs.items():
        for mont in (False, True):
            enc, ok = d.msm_segmented(SM if mont else S, pts, off, fmt, d.OUT_ENCODING, return_ok=True,
                                      scalars_montgomery=mont)
            assert [enc[j].tobytes() for j in range(len(SIZES))] == want, (fmt, mont)
            assert ok.all()
        el = d.msm_segmented(S, pts, off, fmt, d.OUT_ELEMENT)
        assert [e.tobytes() for e in d.batch_compress(el)] == want, fmt
    # an all-empty call gives identities
    empty = np.zeros(5, np.uint32)
    enc, ok = d.msm_segmented(S[:0], W[:0], empty, d.PT_ELEMENT, d.OUT_ENCODING, return_ok=True)
    assert ok.all() and not enc.any()
    el = d.msm_segmented(S[:0], W[:0], empty, d.PT_ELEMENT, d.OUT_ELEMENT)
    assert d.batch_element_eq(el, np.tile(wire([o.IDENTITY]), (4, 1))).all()


@pytest.mark.parametrize("c", list(range(4, 17)))
def test_every_window_width(engine, c):
    """Each width 4..16, forced and read back; c = 4, 8, 16 have their top window at bit 256.
    Edge scalars sit on the first and last pair of every segment."""
    d = engine
    sizes = [5, 1, 0, 40, 33, 2, 17]
    off = np.cumsum([0] + sizes).astype(np.uint32)
    n = int(off[-1])
    a, pts = _kat(d, n, "w%d" % c)
    rnd = random.Random(c)
    s = _place([rnd.randrange(0, 1 << 256) for _ in range(n)], off, _window_edges(c))
    d.msm_set_window(c)
    try:
        enc = d.msm_segmented(canon(s), pts, off, d.PT_ELEMENT, d.OUT_ENCODING)
        assert d.msm_segmented_last() == (_geom(c)[0], _geom(c)[1], 1)
    finally:
        d.msm_set_window(0)
    assert np.array_equal(enc, _expected(d, s, a, off))


def test_skew_and_one_bucket_segments(engine):
    """One segment of 2^16 pairs among single pairs, and a segment whose scalars are all
    equal (every entry of each window in one bucket, across many accumulation runs)."""
    d = engine
    sizes = [1] * 50 + [1 << 16] + [1] * 50 + [5000, 1, 0, 1]
    off = np.cumsum([0] + sizes).astype(np.uint32)
    n = int(off[-1])
    a, pts = _kat(d, n, "skew")
    rnd = random.Random(11)
    s = [rnd.randrange(0, 1 << 256) for _ in range(n)]
    lo = int(off[101])
    for i in range(lo, lo + 5000):
        s[i] = M256 - 12345
    s = _place(s, off, _window_edges(11))
    want = _expected(d, s, a, off)
    aff = d.batch_normalize(pts)
    enc = d.msm_segmented(canon(s), aff, off, d.PT_AFFINE, d.OUT_ENCODING)
    assert np.array_equal(enc, want)
    el = d.msm_segmented(canon(s), pts, off, d.PT_ELEMENT, d.OUT_ELEMENT)
    assert np.array_equal(d.batch_compress(el), want)


def test_parity_with_batch_msm_and_msm(engine):
    """The same inputs through d377_batch_msm: identical encodings, equal Elements; one
    segment against d377_msm with canonical scalars."""
    d = engine
    rnd = random.Random(23)
    sizes = [rnd.choice([0, 1, 2, 63, 64, 65, 300, 1000]) for _ in range(200)]
    off = np.cumsum([0] + sizes).astype(np.uint32)
    n = int(off[-1])
    _, pts = _kat(d, n, "bm")
    s = canon(_place([rnd.randrange(0, 1 << 256) for _ in range(n)], off, _window_edges(9)))
    aff = d.batch_normalize(pts)
    for fmt, p in ((d.PT_AFFINE, aff), (d.PT_ENCODING, d.batch_compress(pts))):
        assert np.array_equal(d.msm_segmented(s, p, off, fmt, d.OUT_ENCODING),
                              d.batch_msm(s, p, off, fmt, d.OUT_ENCODING))
        assert d.batch_element_eq(d.msm_segmented(s, p, off, fmt), d.batch_msm(s, p, off, fmt)).all()
    m = 3000
    sc = canon([rnd.randrange(0, R) for _ in range(m)])
    one = np.array([0, m], np.uint32)
    el, enc = d.vartime_multiscalar_mul(sc, pts[:m])
    assert d.msm_segmented(sc, pts[:m], one, d.PT_ELEMENT, d.OUT_ENCODING)[0].tobytes() == enc.tobytes()
    assert d.batch_element_eq(d.msm_segmented(sc, pts[:m], one), el[None, :]).all()


def test_several_chunks(engine):
    """2^16 segments of 8 pairs at c = 4: ~4.4 GB of bucket sums, cut into chunks of
    floor(2^30 / (W K 128)) segments; every segment against the known answer and against
    d377_batch_msm, with edge scalars on the segments around every chunk boundary."""
    d = engine
    c, W, K = _geom(4)
    nseg, m = 1 << 16, 8
    per_chunk = BUDGET // (W * K * 128)
    off = (np.arange(nseg + 1) * m).astype(np.uint32)
    n = nseg * m
    a, pts = _kat(d, n, "chunks")
    rnd = random.Random(31)
    s = [rnd.randrange(0, 1 << 256) for _ in range(n)]
    edges = _window_edges(c)
    k = 0
    for b in range(per_chunk, nseg, per_chunk):
        for j in (b - 1, b):
            for i in (j * m, j * m + m - 1):
                s[i] = edges[k % len(edges)]
                k += 1
    d.msm_set_window(4)
    try:
        enc = d.msm_segmented(canon(s), pts, off, d.PT_ELEMENT, d.OUT_ENCODING)
        assert d.msm_segmented_last() == (4, W, -(-nseg // per_chunk))
    finally:
        d.msm_set_window(0)
    assert d.msm_segmented_last()[2] > 1
    assert np.array_equal(enc, _expected(d, s, a, off))
    assert np.array_equal(enc, d.batch_msm(canon(s), pts, off, d.PT_ELEMENT, d.OUT_ENCODING))


def test_invalid_encoding_clears_only_its_segment(engine):
    d = engine
    off = np.cumsum([0] + SIZES).astype(np.uint32)
    n = int(off[-1])
    _, pts = _kat(d, n, "bad")
    s = canon([random.Random(3).randrange(0, R) for _ in range(n)])
    E = d.batch_compress(pts)
    good, ok0 = d.msm_segmented(s, E, off, d.PT_ENCODING, d.OUT_ENCODING, return_ok=True)
    assert ok0.all()
    bad = E.copy()
    for j in (5, 9):                          # first pair of 5, last of 9
        i = int(off[j]) if j == 5 else int(off[j + 1]) - 1
        bad[i] = 0
        bad[i, 0] = 1                         # s = 1: not a valid encoding
    enc, ok = d.msm_segmented(s, bad, off, d.PT_ENCODING, d.OUT_ENCODING, return_ok=True)
    assert [int(v) for v in ok] == [0 if j in (5, 9) else 1 for j in range(len(SIZES))]
    assert all(np.array_equal(enc[j], good[j]) for j in range(len(SIZES)) if j not in (5, 9))
    # the invalid pair counts as the identity, as in d377_batch_msm
    assert np.array_equal(enc, d.batch_msm(s, bad, off, d.PT_ENCODING, d.OUT_ENCODING))
    # other formats report every segment good
    assert d.msm_segmented(s, pts, off, d.PT_ELEMENT, d.OUT_ENCODING, return_ok=True)[1].all()


def test_entry_points_agree(engine):
    """Host buffers (pageable, pinned) against _dev through torch, byte for byte; _dev
    interleaved with d377_msm_dev_async; the offsets array reused right after the call."""
    import torch
    from decaf377_b200 import device as dev
    d = engine
    rnd = random.Random(41)
    sizes = [rnd.choice([0, 1, 31, 32, 33, 500]) for _ in range(100)]
    off = np.cumsum([0] + sizes).astype(np.uint32)
    n = int(off[-1])
    a, pts = _kat(d, n, "entry")
    s = [rnd.randrange(0, 1 << 256) for _ in range(n)]
    S = canon(s)
    want = _expected(d, s, a, off)
    E = d.batch_compress(pts)
    assert np.array_equal(d.msm_segmented(S, E, off, d.PT_ENCODING, d.OUT_ENCODING), want)
    assert np.array_equal(d.msm_segmented(d.pinned_copy(S), d.pinned_copy(E), d.pinned_copy(off),
                                          d.PT_ENCODING, d.OUT_ENCODING), want)
    el_host = d.msm_segmented(S, E, off, d.PT_ENCODING, d.OUT_ELEMENT)
    tS, tE = torch.from_numpy(S).cuda(), torch.from_numpy(E).cuda()
    tok = torch.zeros(len(sizes), dtype=torch.uint8, device="cuda")
    host_off = off.copy()
    got = dev.msm_segmented(tS, tE, host_off, d.PT_ENCODING, d.OUT_ENCODING, ok=tok)
    host_off[:] = 0                           # the library has its own copy
    got_el = dev.msm_segmented(tS, tE, torch.from_numpy(off), d.PT_ENCODING, d.OUT_ELEMENT)
    torch.cuda.synchronize()
    assert np.array_equal(got.cpu().numpy(), want) and bool(tok.all())
    # Elements: the same points (their projective limbs follow the order of the bucket sort)
    assert d.batch_element_eq(got_el.cpu().numpy(), el_host).all()
    # _dev between asynchronous single MSMs
    m = 2048
    tsc = torch.from_numpy(canon([rnd.randrange(0, R) for _ in range(m)])).cuda()
    tp = torch.from_numpy(pts[:m].copy()).cuda()
    want_one = d.vartime_multiscalar_mul(tsc.cpu().numpy(), pts[:m])[1]
    _, oc1 = dev.msm_async(tsc, tp)
    seg = dev.msm_segmented(tS, tE, off, d.PT_ENCODING, d.OUT_ENCODING)
    _, oc2 = dev.msm_async(tsc, tp)
    d.sync()
    torch.cuda.synchronize()
    assert np.array_equal(seg.cpu().numpy(), want)
    assert oc1.cpu().numpy().tobytes() == want_one.tobytes() == oc2.cpu().numpy().tobytes()


def test_refusals_leave_outputs_untouched(engine):
    d = engine
    lib = d._lib.load()
    off = np.array([0, 3, 5], np.uint32)
    S, P = canon([1, 2, 3, 4, 5]), wire(oracle_points("seg/ref", 5))
    out = np.full((2, 128), 0xAB, np.uint8)
    ok = np.full((2,), 0xCD, np.uint8)

    def call(sc, pts, fmt, offs, nmsm, o, ofmt, okp):
        p = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)   # noqa: E731
        return lib.d377_msm_segmented(p(sc), p(pts), fmt, p(offs), nmsm, p(o), ofmt, p(okp))

    cases = [
        (S, P, d.PT_BASES, off, 2, out, 0, ok),                  # prepared bases
        (S, P, 5, off, 2, out, 0, ok),
        (S, P, -1, off, 2, out, 0, ok),
        (S, P, 0x200, off, 2, out, 0, ok),
        (S, P, 0, off, 2, out, 2, ok),                           # out format
        (S, P, 0, off, 2, out, d.SCALARS_MONTGOMERY, ok),
        (None, P, 0, off, 2, out, 0, ok),                        # null pointers
        (S, None, 0, off, 2, out, 0, ok),
        (S, P, 0, None, 2, out, 0, ok),
        (S, P, 0, off, 2, None, 0, ok),
        (S, P, 0, np.array([1, 3, 5], np.uint32), 2, out, 0, ok),    # offsets
        (S, P, 0, np.array([0, 4, 3], np.uint32), 2, out, 0, ok),
        (S, P, 0, np.array([0, 3, 0xfffffff1], np.uint32), 2, out, 0, ok),
    ]
    for k, args in enumerate(cases):
        assert call(*args) == d._lib.ERR_INVALID_ARG, k
        assert (out == 0xAB).all() and (ok == 0xCD).all(), k
    # a width whose bucket set exceeds the chunk budget, and a segment too long for one chunk
    # (2^27 pairs x 65 windows at c = 4): refused before any input is read
    for c, offs in ((21, off), (22, off), (4, np.array([0, 1 << 27], np.uint32))):
        d.msm_set_window(c)
        try:
            assert call(S, P, 0, offs, len(offs) - 1, out, 0, ok) == d._lib.ERR_INVALID_ARG, c
        finally:
            d.msm_set_window(0)
        assert (out == 0xAB).all() and (ok == 0xCD).all(), c
    # nmsm = 0: nothing happens, even with null pointers
    assert call(None, None, 0, None, 0, None, 0, None) == 0
    assert call(S, P, 0, off, 0, out, 0, ok) == 0 and (out == 0xAB).all()
    # the largest widths that still fit run
    d.msm_set_window(20)
    try:
        enc = d.msm_segmented(S, P, off, d.PT_ELEMENT, d.OUT_ENCODING)
        assert d.msm_segmented_last()[:2] == (20, 13)
    finally:
        d.msm_set_window(0)
    assert np.array_equal(enc, d.batch_msm(S, P, off, d.PT_ELEMENT, d.OUT_ENCODING))
    with pytest.raises(D377Error):
        d.msm_segmented(S, P, np.array([0, 4, 3], np.uint32))


def test_parity_under_the_on_curve_debug_build():
    lib = os.path.join(ROOT, "decaf377_b200", "libdecaf377_b200_dbg.so")
    if not os.path.exists(lib):
        pytest.skip("debug library not built (python -m decaf377_b200.build --debug)")
    env = dict(os.environ, D377_DEBUG_LIB="1", D377_DEBUG_REPORT="1")
    r = subprocess.run([sys.executable, "-m", "pytest", "-x", "-q", "-m", "gpu", "-p", "no:cacheprovider",
                        os.path.join(ROOT, "tests", "test_gpu_msm_segmented.py"),
                        "-k", "oracle_parity or skew"],
                       capture_output=True, text=True, timeout=1200, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-2000:]
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("D377_DEBUG ")]
    assert line, r.stdout[-2000:]
    fields = dict(kv.split("=") for kv in line[-1].split()[1:])
    assert int(fields["build"]) == 2
    assert int(fields["checked"]) > 1000 and int(fields["failures"]) == 0, line[-1]
