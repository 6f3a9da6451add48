"""GPU parity: every C-ABI entry point against the CPU oracle, bit-exact.

Mirrors the reference's own tests: tests/encoding.rs (KATs, round trips),
src/ark_curve/elligator.rs:86-208, tests/operations.rs:19-61,
src/ark_curve/invsqrt.rs:182-211, plus the edge cases of SURVEY Appendix B.
"""
import random

import numpy as np
import pytest

from oracle import decaf377_ref as o
from tests import golden_vectors as gv
from tests.util import canon, mont, np_bytes, oracle_points, oracle_scalars, unmont, unwire, wire

pytestmark = pytest.mark.gpu

Q, R = o.Q, o.R


def rand_fq(rnd, n):
    edge = [0, 1, 2, Q - 1, Q - 2, (Q - 1) // 2, (Q + 1) // 2, o.ZETA, 1 << 252, (1 << 253) - 1 - Q]
    return (edge + [rnd.randrange(Q) for _ in range(n)])[:max(n, len(edge))]


# ---- field layer (rows a2-a5) ------------------------------------------------
def test_fq_ops(engine):
    rnd = random.Random(1)
    a = rand_fq(rnd, 4096)
    b = list(reversed(rand_fq(rnd, 4096)))
    A, B = mont(a), mont(b)
    assert unmont(engine.fq_batch_op(0, A, B)) == [x * y % Q for x, y in zip(a, b)]
    assert unmont(engine.fq_batch_op(1, A)) == [x * x % Q for x in a]
    assert unmont(engine.fq_batch_op(2, A, B)) == [(x + y) % Q for x, y in zip(a, b)]
    assert unmont(engine.fq_batch_op(3, A, B)) == [(x - y) % Q for x, y in zip(a, b)]
    assert unmont(engine.fq_batch_op(4, A)) == [(-x) % Q for x in a]
    # to / from Montgomery are exact byte conversions
    assert np.array_equal(engine.fq_batch_op(5, canon(a)), A)
    assert np.array_equal(engine.fq_batch_op(6, A), canon(a))
    # inversion (binary extended Euclid of the batched normalisations, and Fermat), 0 -> 0;
    # the small-constant products of the curve formulas (2d = 6042, 2(2d - a) = 12086)
    inv = [pow(x, -1, Q) if x else 0 for x in a]
    assert unmont(engine.fq_batch_op(8, A)) == inv
    assert unmont(engine.fq_batch_op(9, A)) == inv
    assert unmont(engine.fq_batch_op(10, A)) == [x * 6042 % Q for x in a]
    assert unmont(engine.fq_batch_op(11, A)) == [x * 12086 % Q for x in a]


def test_fq_from_le_bytes_mod_order(engine):
    # fq/arkworks.rs:586-620: any 32 bytes reduce mod q (p + 1 -> 1 etc.)
    rnd = random.Random(2)
    raw = [Q, Q + 1, (1 << 256) - 1, 0, 2 * Q + 5] + [rnd.getrandbits(256) for _ in range(2000)]
    out = engine.fq_batch_op(7, canon(raw))
    assert unmont(out) == [v % Q for v in raw]


def test_isqrt_matches_reference_root(engine):
    rnd = random.Random(3)
    xs = rand_fq(rnd, 3000)
    out, ws = engine.fq_batch_isqrt(mont(xs))
    got = unmont(out)
    for x, g, w in zip(xs, got, ws):
        ok, root = o.isqrt(x)
        assert bool(w) == ok and g == root, hex(x)
        # invsqrt.rs:182-211 contract
        if x:
            assert g * g % Q * x % Q == (1 if ok else o.ZETA)


# ---- codec (rows a6-a9) --------------------------------------------------------
def test_generator_multiples_kat(engine):
    enc = np_bytes([bytes.fromhex(h) for h in gv.GENERATOR_MULTIPLES], 32)
    el, ok = engine.batch_decompress(enc)
    assert ok.all()
    assert np.array_equal(engine.batch_compress(el), enc)
    # running sum accumulator += basepoint (tests/encoding.rs:80-94)
    acc = engine.Element.IDENTITY
    for i in range(16):
        assert acc == engine.Element(el[i].tobytes())
        assert acc.vartime_compress().bytes.hex() == gv.GENERATOR_MULTIPLES[i]
        acc = acc + engine.Element.GENERATOR


def test_identity_and_generator(engine):
    ident = engine.Element.default()
    assert ident.vartime_compress().bytes == bytes(32)
    assert engine.Encoding(bytes(32)).vartime_decompress() == ident
    # tests/encoding.rs:28-52: first decodable [b,0,...] is b = 8 and it is the generator
    first = None
    for b in range(1, 256):
        try:
            el = engine.Encoding(bytes([b]) + bytes(31)).vartime_decompress()
            first = b
            break
        except engine.EncodingError:
            pass
    assert first == 8
    assert el == engine.Element.GENERATOR
    assert el.vartime_compress().bytes == bytes([8]) + bytes(31)


def test_decompress_matches_oracle_including_invalid(engine):
    raw = o.xof_blocks("raw", 3000)
    raw = [b[:31] + bytes([b[31] & 0x1F]) for b in raw] + o.xof_blocks("raw2", 200)
    raw += [bytes(x) for x in gv.EDGE_ENCODINGS]
    enc = np_bytes(raw, 32)
    el, ok = engine.batch_decompress(enc)
    pts = unwire(el)
    n_ok = 0
    for i, b in enumerate(raw):
        ref = o.decompress(b)
        assert bool(ok[i]) == (ref is not None), b.hex()
        if ref is not None:
            n_ok += 1
            assert o.on_curve(pts[i])
            assert o.to_affine(pts[i]) == o.to_affine(ref), b.hex()
    assert 200 < n_ok < 1500
    # round trip (tests/encoding.rs:97-106)
    good = enc[ok.astype(bool)]
    assert np.array_equal(engine.batch_compress(el[ok.astype(bool)]), good)


def test_compress_projective_inputs(engine):
    pts = oracle_points("pt", 300)
    sc = oracle_scalars("sc", 300)
    # non-trivial Z: use oracle scalar multiples in projective form
    proj = [o.scalar_mul(p, s % 1000 + 2) for p, s in zip(pts, sc)] + [o.IDENTITY, (0, Q - 1, 1, 0)]
    got = engine.batch_compress(wire(proj))
    for i, p in enumerate(proj):
        assert got[i].tobytes() == o.compress(p)


# ---- Elligator (row a10) ----------------------------------------------------------
def test_elligator_kat(engine):
    inp = np_bytes([bytes(v) for v in gv.ELLIGATOR_INPUTS], 32)
    el = unwire(engine.batch_encode_to_curve(inp))
    for p, (x, y) in zip(el, gv.ELLIGATOR_XY):
        assert o.on_curve(p)
        assert o.to_affine(p) == (x, y)


def test_encode_and_hash_to_curve(engine):
    r1 = o.xof_blocks("fq", 2000) + [bytes(32), (Q - 1).to_bytes(32, "little"), b"\xff" * 32]
    r2 = o.xof_blocks("fq2", len(r1))
    a1, a2 = np_bytes(r1, 32), np_bytes(r2, 32)
    enc = engine.batch_encode_to_curve(a1, engine.OUT_ENCODING)
    el = engine.batch_encode_to_curve(a1, engine.OUT_ELEMENT)
    assert np.array_equal(engine.batch_compress(el), enc)
    henc = engine.batch_hash_to_curve(a1, a2, engine.OUT_ENCODING)
    # the fused kernels (encoding read off the Jacobi-quartic pair / sum) against the
    # two-step path of the engine itself, every element
    hel = engine.batch_hash_to_curve(a1, a2, engine.OUT_ELEMENT)
    assert np.array_equal(engine.batch_compress(hel), henc)
    # r2 = r1 and r2 = -r1 style inputs: doubling and inverse pairs on the quartic
    same = engine.batch_hash_to_curve(a1, a1, engine.OUT_ENCODING)
    assert np.array_equal(engine.batch_compress(engine.batch_hash_to_curve(a1, a1, engine.OUT_ELEMENT)), same)
    negs = np_bytes([((Q - o.fq_from_le_bytes_mod_order(b)) % Q).to_bytes(32, "little") for b in r1], 32)
    opp = engine.batch_hash_to_curve(a1, negs, engine.OUT_ENCODING)
    assert np.array_equal(engine.batch_compress(engine.batch_hash_to_curve(a1, negs, engine.OUT_ELEMENT)), opp)
    for i in range(len(r1)):
        x1 = o.fq_from_le_bytes_mod_order(r1[i])
        x2 = o.fq_from_le_bytes_mod_order(r2[i])
        assert enc[i].tobytes() == o.compress(o.encode_to_curve(x1)), i
        if i % 8 == 0:
            assert henc[i].tobytes() == o.compress(o.hash_to_curve(x1, x2)), i


def test_elligator_zero_input_among_neighbours(engine):
    """r0 = 0 is the Elligator input with a degenerate Jacobi-quartic pair, (s, t) = (0, -1),
    so 1 / (s t) = 0 in k_elligator_encode's CTA-wide inversion; (0, 0) takes k_hash_encode's
    generic fallback after the warp-wide inversion.  Planted at lanes 0, 15 and 31 of the last
    warp of a CTA, across the first warp of the next, over one whole CTA and at both ends of
    the batch (the padding lanes re-read index 0), between random inputs: every element is
    the oracle's, the zero lanes and their good neighbours alike.  (The Elligator denominator
    itself never vanishes: tests/test_jacobi_shortcuts_cpu.py.)"""
    from oracle import c_oracle as co
    n = 5 * 128 + 77
    rng = np.random.default_rng(168)
    r1 = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    r2 = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    zero = [0, 224, 239, 255] + list(range(256, 288)) + list(range(384, 512)) + [n - 1]
    r1[zero] = 0
    r2[zero] = 0
    r2[[100, 600]] = 0                           # (x, 0): one degenerate map in the sum
    r1[[101, 601]] = 0                           # (0, x)
    enc = engine.batch_encode_to_curve(r1, engine.OUT_ENCODING)
    henc = engine.batch_hash_to_curve(r1, r2, engine.OUT_ENCODING)
    want = co.encode_to_curve(r1, out_enc=True, threads=4)
    hwant = co.hash_to_curve(r1, r2, out_enc=True, threads=4)
    for i in range(n):
        assert enc[i].tobytes() == want[i].tobytes(), i
        assert henc[i].tobytes() == hwant[i].tobytes(), i
    assert want[0].tobytes() == o.compress(o.encode_to_curve(0)) == bytes(32)
    assert hwant[0].tobytes() == o.compress(o.hash_to_curve(0, 0)) == bytes(32)


# ---- group ops (rows a11, a12, a16) -------------------------------------------------
def test_scalar_mul_matches_oracle(engine):
    n = 256
    pts = oracle_points("pt", n)
    sc = oracle_scalars("sc", n)
    sc[:4] = [0, 1, R - 1, 2]
    got = engine.batch_scalar_mul(wire(pts), canon(sc), out_format=engine.OUT_ENCODING)
    for i in range(n):
        assert got[i].tobytes() == o.compress(o.scalar_mul(pts[i], sc[i])), i
    # config 1 pipeline: decompress -> mul -> compress from encodings
    encs = np_bytes([o.compress(p) for p in pts], 32)
    got2, ok = engine.batch_scalar_mul(encs, canon(sc), engine.PT_ENCODING, engine.OUT_ENCODING,
                                       return_ok=True)
    assert ok.all() and np.array_equal(got, got2)


def test_scalar_mul_homomorphism(engine):
    # tests/operations.rs:19-43
    n = 64
    P = wire(oracle_points("ptH", n))
    a, b = oracle_scalars("a", n), oracle_scalars("b", n)
    aP = engine.batch_scalar_mul(P, canon(a))
    bP = engine.batch_scalar_mul(P, canon(b))
    abP = engine.batch_scalar_mul(P, canon([(x + y) % R for x, y in zip(a, b)]))
    assert engine.batch_element_eq(engine.batch_add(aP, bP), abP).all()
    baP = engine.batch_scalar_mul(aP, canon(b))
    mP = engine.batch_scalar_mul(P, canon([x * y % R for x, y in zip(a, b)]))
    assert engine.batch_element_eq(baP, mP).all()


def test_fixed_base_matches_oracle(engine):
    n = 300
    sc = oracle_scalars("fb", n)
    sc[:6] = [0, 1, R - 1, 2, 1 << 15, (1 << 16) - 1]
    # digit boundaries of the quartic table's signed 21-bit windows (encoding output), all
    # digits at their extremes, and non-canonical scalars >= 2^252 (Edwards fallback)
    sc[6:18] = [1 << 20, (1 << 20) + 1, (1 << 21) - 1, 1 << 21, (1 << 231) - 1, 1 << 231,
                int("1" + "0" * 20, 2) * sum(1 << (21 * w) for w in range(12)) % R,
                sum(((1 << 20) + 1) << (21 * w) for w in range(11)),
                1 << 252, (1 << 252) + 5, (1 << 255) - 19, (1 << 256) - 1]
    got = engine.fixed_base_mul(canon(sc), engine.OUT_ENCODING)
    el = engine.fixed_base_mul(canon(sc), engine.OUT_ELEMENT)
    assert np.array_equal(engine.batch_compress(el), got)
    for i in range(n):
        assert got[i].tobytes() == o.compress(o.scalar_mul(o.GENERATOR, sc[i])), i
    # the quartic path against the Edwards path on a batch with several elements per thread
    # and a ragged tail
    big = np.frombuffer(o.xof_bytes("fb_big", 32 * 70001), np.uint8).reshape(-1, 32).copy()
    big[:, 31] &= 0x03
    assert np.array_equal(engine.fixed_base_mul(big, engine.OUT_ENCODING),
                          engine.batch_compress(engine.fixed_base_mul(big, engine.OUT_ELEMENT)))


# ---- MSM (rows a14, a15) ------------------------------------------------------------
@pytest.mark.parametrize("n", [0, 1, 3, 33, 1000])
def test_msm_matches_oracle_fold(engine, n):
    pts = oracle_points("msm_pt", n)
    sc = oracle_scalars("msm_sc", n)
    el, enc = engine.vartime_multiscalar_mul(canon(sc) if n else np.zeros((0, 32), np.uint8),
                                             wire(pts) if n else np.zeros((0, 128), np.uint8))
    want = o.vartime_multiscalar_mul(sc, pts)
    assert enc.tobytes() == o.compress(want)
    assert o.point_eq(o.point_from_wire(el.tobytes()), want)


def test_msm_edge_inputs(engine):
    # repeated points, P and -P, identity points, zero scalars (SURVEY appendix B)
    base = oracle_points("msm_e", 8)
    pts = base + base + [o.point_neg(p) for p in base] + [o.IDENTITY] * 4 + base[:4]
    sc = oracle_scalars("msm_es", len(pts))
    sc[0] = 0
    sc[9] = R - 1
    sc[-1] = 0
    _, enc = engine.vartime_multiscalar_mul(canon(sc), wire(pts))
    assert enc.tobytes() == o.compress(o.vartime_multiscalar_mul(sc, pts))
    # all scalars equal: one bucket per window holds everything
    sc2 = [sc[3]] * len(pts)
    _, enc2 = engine.vartime_multiscalar_mul(canon(sc2), wire(pts))
    assert enc2.tobytes() == o.compress(o.vartime_multiscalar_mul(sc2, pts))


@pytest.mark.parametrize("c", [4, 7, 11, 16])
def test_msm_window_widths(engine, c):
    n = 500
    pts = oracle_points("msm_w", n)
    sc = oracle_scalars("msm_ws", n)
    want = o.compress(o.vartime_multiscalar_mul(sc, pts))
    engine.msm_set_window(c)
    try:
        _, enc = engine.vartime_multiscalar_mul(canon(sc), wire(pts))
    finally:
        engine.msm_set_window(0)
    assert enc.tobytes() == want


def test_msm_point_formats(engine):
    n = 200
    pts = oracle_points("msm_f", n)
    sc = canon(oracle_scalars("msm_fs", n))
    want = o.compress(o.vartime_multiscalar_mul(oracle_scalars("msm_fs", n), pts))
    encs = np_bytes([o.compress(p) for p in pts], 32)
    aff = np_bytes([o.fq_to_mont_bytes(c) for p in pts for c in o.to_affine(p)], 64)
    assert engine.vartime_multiscalar_mul(sc, encs, engine.PT_ENCODING)[1].tobytes() == want
    assert engine.vartime_multiscalar_mul(sc, aff, engine.PT_AFFINE)[1].tobytes() == want
    assert engine.vartime_multiscalar_mul(sc, wire(pts), engine.PT_ELEMENT)[1].tobytes() == want
    # X||Y||Z without the redundant T, on both addition paths
    xyz = np.ascontiguousarray(wire(pts)[:, :96])
    for mode in (1, -1):
        engine.msm_set_normalize(mode)
        try:
            assert engine.vartime_multiscalar_mul(sc, xyz, engine.PT_XYZ)[1].tobytes() == want
        finally:
            engine.msm_set_normalize(0)


@pytest.mark.parametrize("mode,mixed", [(1, True), (-1, False)])
@pytest.mark.parametrize("n", [1, 31, 257, 3000])
def test_msm_element_inputs_normalised_or_not(engine, mode, mixed, n):
    """Element inputs: batch-normalised (7M mixed bucket additions, one inversion per CTA)
    and projective (8M cached additions) give the oracle's result; identity points, P / -P
    pairs and non-trivial Z included."""
    pts = oracle_points("msm_n", n)
    # re-scale some representatives (Z != 1 in various sizes) and plant identities
    rnd = random.Random(n)
    pts = [tuple(c * lam % Q for c in p) for p, lam in ((p, rnd.randrange(1, Q)) for p in pts)]
    if n > 8:
        pts[3] = o.IDENTITY
        pts[5] = o.point_neg(pts[4])
        pts[n - 1] = o.IDENTITY
    sc = oracle_scalars("msm_ns", n)
    want = o.compress(o.vartime_multiscalar_mul(sc, pts))
    engine.msm_set_normalize(mode)
    try:
        _, enc = engine.vartime_multiscalar_mul(canon(sc), wire(pts))
        assert engine.msm_stage_info()["mixed"] is mixed
    finally:
        engine.msm_set_normalize(0)
    assert enc.tobytes() == want


@pytest.mark.parametrize("groups", [1, 2, 3, 8])
@pytest.mark.parametrize("fmt", ["element", "affine"])
def test_msm_window_group_pipeline(engine, groups, fmt):
    """The two-stream pipeline (sort of window group k+1 under the accumulation of group k)
    gives the same result for every group count, including more groups than make sense."""
    n = 700
    pts = oracle_points("msm_g", n)
    sc = oracle_scalars("msm_gs", n)
    sc[0], sc[1], sc[2] = 0, R - 1, 1
    want = o.compress(o.vartime_multiscalar_mul(sc, pts))
    engine.msm_set_groups(groups)
    try:
        for c in (0, 5):
            engine.msm_set_window(c)
            if fmt == "element":
                _, enc = engine.vartime_multiscalar_mul(canon(sc), wire(pts))
            else:
                aff = np_bytes([o.fq_to_mont_bytes(c_) for p in pts for c_ in o.to_affine(p)], 64)
                _, enc = engine.vartime_multiscalar_mul(canon(sc), aff, engine.PT_AFFINE)
            assert enc.tobytes() == want, (groups, c)
    finally:
        engine.msm_set_window(0)
        engine.msm_set_groups(0)


def test_msm_prepared_bases(engine):
    """d377_msm_bases_create + D377_PT_BASES: batch_convert_to_mul_base once, msm many times
    (ark_curve/element.rs:27-37).  Same result as passing the points with every call, from
    every input format, through the host, the submit / wait and the device entry points, and
    for a prefix of the bases."""
    import torch
    from decaf377_b200 import device as dev
    n = 3000
    rng = np.random.default_rng(9)
    pts = oracle_points("pb_pt", 40) + [o.IDENTITY, o.GENERATOR]
    W = wire(pts)[rng.integers(0, len(pts), n)]
    sc = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    sc[:, 31] &= 0x03
    want = engine.vartime_multiscalar_mul(sc, W)[1].tobytes()
    aff = engine.batch_normalize(W)
    enc = engine.batch_compress(W)
    for fmt, arr in ((engine.PT_ELEMENT, W), (engine.PT_XYZ, np.ascontiguousarray(W[:, :96])),
                     (engine.PT_AFFINE, aff), (engine.PT_ENCODING, enc)):
        bases = engine.MsmBases(arr, fmt)
        assert len(bases) == n
        assert engine.vartime_multiscalar_mul(sc, bases)[1].tobytes() == want
        engine.msm_submit(sc, bases, slot=1)
        assert engine.msm_wait(1)[1].tobytes() == want
        got = dev.msm(torch.from_numpy(sc).cuda(), bases)[1].cpu().numpy().tobytes()
        assert got == want
        # a prefix of the bases
        m = 1234
        assert engine.vartime_multiscalar_mul(sc[:m], bases)[1].tobytes() == \
            engine.vartime_multiscalar_mul(sc[:m], W[:m])[1].tobytes()
        bases.close()
    # an invalid encoding among the bases is reported at creation
    bad = enc.copy()
    bad[7] = np.frombuffer(bytes([1] + [0] * 31), np.uint8)
    with pytest.raises(Exception):
        engine.MsmBases(bad, engine.PT_ENCODING)
    # large enough for the batch normalisation with several elements per thread
    n2 = 200000
    W2 = wire(pts)[rng.integers(0, len(pts), n2)]
    sc2 = rng.integers(0, 256, (n2, 32), dtype=np.uint8)
    sc2[:, 31] &= 0x03
    b2 = engine.MsmBases(W2, engine.PT_ELEMENT)
    assert engine.vartime_multiscalar_mul(sc2, b2)[1].tobytes() == engine.vartime_multiscalar_mul(sc2, W2)[1].tobytes()
    b2.close()


def test_msm_timeline_reports_every_group(engine):
    """d377_msm_timeline: one record per window group of the last MSM, in stream order."""
    n = 5000
    rng = np.random.default_rng(5)
    sc = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    sc[:, 31] &= 0x03
    pts = wire(oracle_points("tl_pt", 8))[rng.integers(0, 8, n)]
    engine.msm_set_groups(3)
    try:
        engine.vartime_multiscalar_mul(sc, pts)
        tl = engine.msm_timeline()
    finally:
        engine.msm_set_groups(0)
    assert len(tl) == 3
    for g in tl:
        assert 0.0 <= g["sorted"] <= g["acc_start"] <= g["acc_end"] <= g["tail_end"]
    assert tl[0]["acc_end"] <= tl[1]["acc_start"] <= tl[2]["acc_start"]


def test_outputs_are_canonical_montgomery(engine):
    """Lazy reduction is internal: every Fq that crosses the ABI is the canonical
    Montgomery representative (< q), whatever path produced it."""
    n = 300
    pts = oracle_points("canon", n)
    sc = canon(oracle_scalars("canon_s", n))
    def assert_canonical(arr):
        for row in np.asarray(arr).reshape(-1, 32):
            assert int.from_bytes(row.tobytes(), "little") < Q
    assert_canonical(engine.batch_add(wire(pts), wire(list(reversed(pts)))))
    assert_canonical(engine.batch_scalar_mul(wire(pts), sc, engine.PT_ELEMENT, engine.OUT_ELEMENT))
    assert_canonical(engine.fixed_base_mul(sc, engine.OUT_ELEMENT))
    assert_canonical(engine.vartime_multiscalar_mul(sc, wire(pts))[0])
    encs = np_bytes([o.compress(p) for p in pts], 32)
    assert_canonical(engine.batch_decompress(encs)[0])
    raw = np.frombuffer(o.xof_bytes("canon_r", n), np.uint8).reshape(n, 32)
    assert_canonical(engine.batch_encode_to_curve(raw, engine.OUT_ELEMENT))
    assert_canonical(engine.batch_normalize(wire(pts)))
    # extreme field operands
    ext = [0, 1, Q - 1, Q - 2, (Q - 1) // 2]
    A = mont([a for a in ext for _ in ext]); B = mont([b for _ in ext for b in ext])
    for op in (0, 2, 3):
        assert_canonical(engine.fq_batch_op(op, A, B))
    assert_canonical(engine.fq_batch_op(1, A)); assert_canonical(engine.fq_batch_op(4, A))


def test_msm_rejects_noncanonical_scalar_and_bad_encoding(engine):
    from decaf377_b200._lib import D377Error, ERR_INVALID_ENCODING, ERR_SCALAR_RANGE
    pts = wire(oracle_points("msm_r", 4))
    sc = canon([1, 2, R, 3])
    with pytest.raises(D377Error) as ei:
        engine.vartime_multiscalar_mul(sc, pts)
    assert ei.value.code == ERR_SCALAR_RANGE
    encs = np_bytes([bytes([1]) + bytes(31)] * 4, 32)
    with pytest.raises(D377Error) as ei:
        engine.vartime_multiscalar_mul(canon([1, 2, 3, 4]), encs, engine.PT_ENCODING)
    assert ei.value.code == ERR_INVALID_ENCODING


def test_msm_known_answer_large(engine):
    """P_i = a_i G  =>  sum s_i P_i = (sum s_i a_i mod r) G   (SURVEY 8d)."""
    n = 1 << 16
    a = np.frombuffer(o.xof_bytes("dl", n), np.uint8).reshape(n, 32).copy()
    s = np.frombuffer(o.xof_bytes("sc", n), np.uint8).reshape(n, 32).copy()
    a[:, 31] &= 0x03
    s[:, 31] &= 0x03           # < 2^250 < r: canonical
    P = engine.fixed_base_mul(a, engine.OUT_ELEMENT)
    _, enc = engine.vartime_multiscalar_mul(s, P)
    ai = [int.from_bytes(a[i].tobytes(), "little") for i in range(n)]
    si = [int.from_bytes(s[i].tobytes(), "little") for i in range(n)]
    k = sum(x * y for x, y in zip(ai, si)) % R
    assert enc.tobytes() == o.compress(o.scalar_mul(o.GENERATOR, k))


def test_element_sum(engine):
    pts = oracle_points("sum", 100)
    want = o.IDENTITY
    for p in pts:
        want = o.point_add(want, p)
    _, enc = engine.element_sum(wire(pts))
    assert enc.tobytes() == o.compress(want)
    assert engine.element_sum(np.zeros((0, 128), np.uint8))[1].tobytes() == bytes(32)


def test_msm_submit_wait_pipeline(engine):
    """d377_msm_submit / d377_msm_wait: two MSMs in flight, results and errors per slot."""
    from decaf377_b200._lib import D377Error, ERR_SCALAR_RANGE
    n = 300
    pts = wire(oracle_points("msm_p", n))
    s0 = oracle_scalars("msm_p0", n)
    s1 = oracle_scalars("msm_p1", n)
    a0, a1 = canon(s0), canon(s1)
    engine.msm_submit(a0, pts, slot=0)
    engine.msm_submit(a1, pts, slot=1)
    with pytest.raises(D377Error):
        engine.msm_submit(a0, pts, slot=1)          # still in flight
    P = oracle_points("msm_p", n)
    assert engine.msm_wait(0)[1].tobytes() == o.compress(o.vartime_multiscalar_mul(s0, P))
    assert engine.msm_wait(1)[1].tobytes() == o.compress(o.vartime_multiscalar_mul(s1, P))
    with pytest.raises(D377Error):
        engine.msm_wait(1)                          # nothing in flight
    bad = canon([R] * n)
    engine.msm_submit(bad, pts, slot=0)
    with pytest.raises(D377Error) as ei:
        engine.msm_wait(0)
    assert ei.value.code == ERR_SCALAR_RANGE
    engine.msm_submit(a0, pts, slot=0)              # slot usable again after an error
    assert engine.msm_wait(0)[1].tobytes() == o.compress(o.vartime_multiscalar_mul(s0, P))


def test_msm_skewed_scalars_large(engine):
    """All-equal and tiny scalars: one bucket per window holds every point (stitching depth)."""
    n = 1 << 15
    a = np.frombuffer(o.xof_bytes("skew_dl", n), np.uint8).reshape(n, 32).copy()
    a[:, 31] &= 0x03
    P = engine.fixed_base_mul(a, engine.OUT_ELEMENT)
    ai = [int.from_bytes(a[i].tobytes(), "little") for i in range(n)]
    for k in (1, 5, (1 << 250) - 3):
        s = canon([k] * n)
        _, enc = engine.vartime_multiscalar_mul(s, P)
        assert enc.tobytes() == o.compress(o.scalar_mul(o.GENERATOR, k * sum(ai) % R)), k
    # half zeros, half one value
    sc = [0 if i % 2 else 12345 for i in range(n)]
    _, enc = engine.vartime_multiscalar_mul(canon(sc), P)
    assert enc.tobytes() == o.compress(o.scalar_mul(o.GENERATOR, sum(x * y for x, y in zip(sc, ai)) % R))


# ---- chunk-pipelined host API -------------------------------------------------------
def test_host_api_chunk_pipeline_matches_device_path(engine):
    """The host entry points cut a batch into chunks that overlap upload / kernel /
    download; the stitched result must equal the one-kernel device path, ragged tail
    included, with pinned and with pageable buffers."""
    import torch
    from decaf377_b200 import device as dev
    from oracle import c_oracle as co
    n = (1 << 20) + 12345            # 5 chunks of 2^18, the last one ragged
    rng = np.random.default_rng(77)
    raw = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    raw_d = torch.from_numpy(raw).cuda()
    enc_dev = dev.encode_to_curve(raw_d, engine.OUT_ENCODING)
    torch.cuda.synchronize()
    want = enc_dev.cpu().numpy()
    # pageable in / out
    got = engine.batch_encode_to_curve(raw, engine.OUT_ENCODING)
    assert np.array_equal(got, want)
    # pinned in / out
    raw_p = engine.pinned_copy(raw)
    out_p = engine.pinned_empty((n, 32))
    res = engine.batch_encode_to_curve(raw_p, engine.OUT_ENCODING, out=out_p)
    assert res is out_p and np.array_equal(out_p, want)
    # two outputs, some invalid inputs: decompress of (encodings with every 7th one damaged)
    enc = want.copy()
    enc[::7, 0] |= 1                 # odd s: InvalidEncoding
    el, ok = engine.batch_decompress(enc, out=engine.pinned_empty((n, 128)), ok=engine.pinned_empty((n,)))
    assert not ok[::7].any() and ok.sum() == n - len(range(0, n, 7))
    back = engine.batch_compress(el)
    good = ok.astype(bool)
    assert np.array_equal(back[good], enc[good]) and not back[~good].any()
    # and a sample against the oracle
    idx = rng.integers(0, n, 512)
    assert np.array_equal(co.encode_to_curve(raw[idx], out_enc=True, threads=4), want[idx])


@pytest.mark.parametrize("chunks", [2, 3, 8])
def test_msm_host_chunks_same_result(engine, chunks):
    """d377_msm over host buffers as k overlapped sub-MSMs == one Pippenger."""
    n = 70001
    pts = wire(oracle_points("chunk_pt", 64))
    rng = np.random.default_rng(5)
    P = pts[rng.integers(0, 64, n)]
    sc = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    sc[:, 31] &= 0x03
    engine.msm_set_host_chunks(1)
    _, want = engine.vartime_multiscalar_mul(sc, P)
    try:
        engine.msm_set_host_chunks(chunks)
        _, got = engine.vartime_multiscalar_mul(sc, P)
        assert got.tobytes() == want.tobytes()
        engine.msm_submit(sc, P, slot=1)
        engine.msm_submit(sc[:1000], P[:1000], slot=0)
        _, a = engine.msm_wait(1)
        assert a.tobytes() == want.tobytes()
        engine.msm_wait(0)
    finally:
        engine.msm_set_host_chunks(0)


# ---- SURVEY 8f rows: normalize_batch, general sqrt_ratio_zeta, wire formats ------------
def test_normalize_batch_matches_oracle(engine):
    """CurveGroup::normalize_batch / batch_convert_to_mul_base (ark_curve/element.rs:27-34,
    74-81): x = X/Z, y = Y/Z, bit-exact, for sizes around the per-thread chunking."""
    pts = oracle_points("norm_pt", 300)
    # projective representatives with Z != 1 (elligator outputs), plus identity and generator
    pts += [o.IDENTITY, o.GENERATOR, o.scalar_mul(o.GENERATOR, 5)]
    W = wire(pts)
    for n in (1, 2, 33, len(pts)):
        aff = engine.batch_normalize(W[:n])
        for i in range(n):
            x, y = o.to_affine(pts[i])
            assert aff[i, :32].tobytes() == o.fq_to_mont_bytes(x), i
            assert aff[i, 32:].tobytes() == o.fq_to_mont_bytes(y), i
    # large batch: several elements per thread (more than one resident wave of threads) and
    # many per inversion; check through the MSM affine input path
    n = 300000
    rng = np.random.default_rng(11)
    big = W[rng.integers(0, len(pts), n)]
    aff = engine.batch_normalize(big)
    idx = rng.integers(0, n, 200)
    for i in idx:
        p = o.point_from_wire(big[i].tobytes())
        x, y = o.to_affine(p)
        assert aff[i].tobytes() == o.fq_to_mont_bytes(x) + o.fq_to_mont_bytes(y)
    sc = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    sc[:, 31] &= 0x03
    _, e1 = engine.vartime_multiscalar_mul(sc, big)
    _, e2 = engine.vartime_multiscalar_mul(sc, aff, engine.PT_AFFINE)
    assert e1.tobytes() == e2.tobytes()
    # host mirror
    els = [engine.Element(W[i].tobytes()) for i in range(4)]
    affs = engine.Element.normalize_batch(els)
    assert all(a.into_element() == e for a, e in zip(affs, els))
    assert engine.AffinePoint.deserialize_compressed(affs[1].serialize_compressed()) == affs[1]


def test_sqrt_ratio_zeta_general_matches_reference_root(engine):
    """Fq::sqrt_ratio_zeta(num, den), ark_curve/invsqrt.rs:69-166: the 4-way contract of
    invsqrt.rs:182-211 and the very root the reference's algorithm returns."""
    rnd = random.Random(9)
    nums = rand_fq(rnd, 1500)
    dens = list(reversed(rand_fq(rnd, 1500)))
    nums += [1, 1, 0, 0, 5]
    dens += [1, 0, 0, 7, 0]          # proptest-regressions/invsqrt.txt:7 and the zero cases
    out, ws = engine.fq_batch_sqrt_ratio_zeta(mont(nums), mont(dens))
    got = unmont(out)
    for nu, de, g, w in zip(nums, dens, got, ws):
        ok, root = o.sqrt_ratio_zeta(nu, de)
        assert bool(w) == ok and g == root, (hex(nu), hex(de))
        if nu and de:
            lhs = g * g % Q * de % Q
            assert lhs == (nu if ok else o.ZETA * nu % Q)
    ok, r = engine.Fq.sqrt_ratio_zeta(engine.Fq(4), engine.Fq(9))
    assert ok and (r * r * engine.Fq(9)) == engine.Fq(4)


def test_field_deserialize_batch(engine):
    """CanonicalDeserialize for Fq / Fr (fq/arkworks.rs:189-229; fq.rs:149-153, fr.rs:129-133;
    proptest-regressions/fields/fr/arkworks.txt): values >= modulus are rejected."""
    rnd = random.Random(10)
    vals = [0, 1, Q - 1, Q, Q + 1, R - 1, R, R + 1, (1 << 256) - 1] + [rnd.getrandbits(256) for _ in range(500)] \
        + [rnd.randrange(Q) for _ in range(500)]
    raw = canon(vals)
    out, ok = engine.field_batch_deserialize(engine.FIELD_FQ, raw)
    assert [bool(x) for x in ok] == [v < Q for v in vals]
    assert unmont(out) == [v if v < Q else 0 for v in vals]
    out, ok = engine.field_batch_deserialize(engine.FIELD_FR, raw)
    assert [bool(x) for x in ok] == [v < R for v in vals]
    assert [int.from_bytes(out[i].tobytes(), "little") for i in range(len(vals))] == [v if v < R else 0 for v in vals]
    # serialize is the exact inverse on valid values
    good = [v for v in vals if v < Q]
    m, _ = engine.field_batch_deserialize(engine.FIELD_FQ, canon(good))
    assert np.array_equal(engine.fq_batch_op(6, m), canon(good))
    assert engine.Fq.deserialize_compressed(engine.Fq(5).serialize_compressed()) == engine.Fq(5)
    el = engine.Element.GENERATOR
    assert engine.Element.deserialize_compressed(el.serialize_compressed()) == el


def test_scalar_mul_all_256_bit_scalars(engine):
    """The windowed scalar multiplication handles any 256-bit k (the carry of the signed
    recoding is a 65th digit): [k]P == [k mod r]P, including k = 2^256 - 1."""
    pts = oracle_points("smul_pt", 6)
    ks = [0, 1, R - 1, R, (1 << 256) - 1, (1 << 255) + 12345]
    out = engine.batch_scalar_mul(wire(pts), canon(ks), engine.PT_ELEMENT, engine.OUT_ENCODING)
    for i, (p, k) in enumerate(zip(pts, ks)):
        assert out[i].tobytes() == o.compress(o.scalar_mul(p, k % R)), i
