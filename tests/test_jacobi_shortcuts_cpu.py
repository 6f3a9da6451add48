"""CPU checks of the algebra behind the square-root-free encodings (DESIGN.md 3.3).

The CUDA kernels k_elligator_encode, k_hash_encode and k_fixed_base_jq read the decaf377
encoding of a point off a preimage on the Jacobi quartic
    J:  t^2 = s^4 - 2 (2d - a) s^2 + 1,     (s, t) |-> (2s / (1 + a s^2), (1 - a s^2) / t)
instead of running vartime_compress (ark_curve/encoding.rs:91-128).  These tests restate the
three shortcuts with Python integers and compare them with the oracle's compress of the
reference path, so the identities are pinned without a GPU.
"""
import random

from oracle import decaf377_ref as o

Q, R = o.Q, o.R
A, D = o.COEFF_A, o.COEFF_D
DELTA = (2 * D - A) % Q            # t^2 = s^4 - 2 DELTA s^2 + 1


def inv(x):
    return pow(x, -1, Q) if x % Q else 0


def elligator_st(r0):
    """ark_curve/elligator.rs:15-54 up to the Jacobi-quartic pair (pt_elligator_st)."""
    r = o.ZETA * r0 * r0 % Q
    den = (D * r - (D - A)) * ((D - A) * r - D) % Q
    num = (r + 1) * (A - 2 * D) % Q
    iss, isri = o.isqrt(num * den % Q)
    sgn, tw = (1, 1) if iss else (Q - 1, r0)
    isri = isri * tw % Q
    s = isri * num % Q
    t = (-sgn * isri * s * (r - 1) * pow(A - 2 * D, 2, Q) - 1) % Q
    if o.is_negative(s) == iss:
        s = (-s) % Q
    return s, t


def encoding_from_projective(S, T, Z):
    """jq_encoding_with_inverse: s = S / Z, t = T / Z^2; None where the shortcut does not apply."""
    prod = S * T % Q * Z % Q
    if prod == 0:
        return None
    i = inv(prod)
    u = 2 * pow(S * Z, 2, Q) * i % Q                    # 2 s / t
    ti = T * i % Q
    s3, is3 = S * S % Q * ti % Q, Z * Z % Q * ti % Q    # s, 1 / s
    if (1 - s3 * s3) % Q == 0:
        return None
    return o.fq_abs(is3 if o.is_negative(u) else s3)


def jq_madd(P, s2, t2):
    """jq_madd (point.cuh): projective + affine on J, unified Billet-Joye law."""
    S1, T1, Z1 = P
    a, b, c, s2sq = S1 * S1 % Q, Z1 * Z1 % Q, S1 * Z1 % Q, s2 * s2 % Q
    dd, h = a * s2sq % Q, c * s2 % Q
    return ((c * t2 + T1 * s2) % Q,
            ((b + dd) * (T1 * t2 - 2 * DELTA * h) + 2 * h * (a + s2sq * b)) % Q,
            (b - dd) % Q)


def jq_dbl(P):
    S, T, Z = P
    a, b = S * S % Q, Z * Z % Q
    a2, b2 = a * a % Q, b * b % Q
    return (2 * S * T % Q * Z % Q, ((b2 + a2) * (T * T - 2 * DELTA * a * b) + 4 * a2 * b2) % Q, (b2 - a2) % Q)


def test_elligator_pair_lies_on_the_quartic_and_maps_to_the_point():
    rnd = random.Random(1)
    for r0 in [0, 1, 2, Q - 1, o.ZETA] + [rnd.randrange(Q) for _ in range(40)]:
        s, t = elligator_st(r0)
        assert (t * t - (pow(s, 4, Q) - 2 * DELTA * s * s + 1)) % Q == 0
        X, Y, Z, T = o.elligator_map(r0)
        assert (X, Z) == (2 * s * t % Q, (1 - s * s) * t % Q)


def test_elligator_denominator_never_vanishes():
    """den = (d r - (d - a)) ((d - a) r - d), r = zeta r0^2, is zero only where zeta r0^2 is
    (d - a) / d or d / (d - a).  Both targets are squares and zeta is not, so target / zeta
    has no root in Fq: no r0 reaches a zero denominator.  The degenerate Jacobi-quartic pair
    the kernels do meet is the one of r0 = 0, (s, t) = (0, -1)."""
    for target in ((D - A) * inv(D) % Q, D * inv(D - A) % Q):
        r0sq = target * inv(o.ZETA) % Q
        assert pow(r0sq, (Q - 1) // 2, Q) == Q - 1           # Euler: not a square
        assert o.sqrt_ratio_zeta(r0sq, 1)[0] is False
    assert elligator_st(0) == (0, Q - 1)


def test_encoding_of_elligator_output_is_abs_s_or_abs_inverse_s():
    """compress(encode_to_curve(r0)) = |s| if 2s/t is non-negative else |1/s|."""
    rnd = random.Random(2)
    for r0 in [0, 1, 2, Q - 1, Q - 2, o.ZETA, (Q - 1) // 2] + [rnd.randrange(Q) for _ in range(300)]:
        s, t = elligator_st(r0)
        want = o.compress_to_field(o.elligator_map(r0))
        if (1 - s * s) * t % Q == 0:
            continue                       # projective Z = 0: the kernel takes the generic path
        ip = inv(s * t % Q)
        u = 2 * s * s % Q * ip % Q
        got = o.fq_abs(t * ip % Q if o.is_negative(u) else s)
        assert got == want, hex(r0)
        assert encoding_from_projective(s, t, 1) in (want, None)


def test_hash_to_curve_encoding_through_the_quartic_addition_law():
    rnd = random.Random(3)
    for _ in range(200):
        r1, r2 = rnd.randrange(Q), rnd.randrange(Q)
        (s1, t1), (s2, t2) = elligator_st(r1), elligator_st(r2)
        p = s1 * s2 % Q
        w = (1 - p * p) % Q
        ns = (s1 * t2 + t1 * s2) % Q
        nt = ((1 + p * p) * (t1 * t2 - 2 * DELTA * p) + 2 * p * (s1 * s1 + s2 * s2)) % Q
        got = encoding_from_projective(ns, nt, w)
        want = o.compress_to_field(o.hash_to_curve(r1, r2))
        assert got in (want, None)
        assert got is not None            # random inputs never hit the exceptional set


def test_fixed_base_on_the_quartic_with_signed_21_bit_windows():
    """compress(k G) = encoding of k G_J, G_J = (8, 65 / y_G); 12 signed 21-bit windows."""
    G = o.decompress((8).to_bytes(32, "little"))
    xg, yg = o.to_affine(G)
    assert (xg, yg) == (o.B_X, o.B_Y)
    sG, tG = 8, 65 * inv(yg) % Q
    assert (tG * tG - (pow(sG, 4, Q) - 2 * DELTA * sG * sG + 1)) % Q == 0
    C_, W_, K_ = 21, 12, 1 << 20
    bases, P = [], (sG, tG, 1)
    for _ in range(W_):
        iz = inv(P[2])
        bases.append((P[0] * iz % Q, P[1] * iz * iz % Q))
        for _ in range(C_):
            P = jq_dbl(P)

    def entry(w, m):
        acc = (0, 1, 1)
        for i in reversed(range(C_)):
            acc = jq_dbl(acc)
            if (m >> i) & 1:
                acc = jq_madd(acc, *bases[w])
        iz = inv(acc[2])
        return acc[0] * iz % Q, acc[1] * iz * iz % Q

    rnd = random.Random(4)
    ks = [1, 2, R - 1, (R - 1) // 2, 1 << 20, (1 << 20) + 1, (1 << 21) - 1, (1 << 251) - 1]
    ks += [rnd.randrange(R) for _ in range(6)]
    for k in ks:
        acc, carry, bad = (0, 1, 1), 0, False
        for w in range(W_):
            raw = ((k >> (C_ * w)) & ((1 << C_) - 1)) + carry
            carry = 1 if raw > K_ else 0
            dg = raw - (carry << C_)
            s2, t2 = (0, 1) if dg == 0 else entry(w, abs(dg))
            if dg < 0:
                s2 = (-s2) % Q
            acc = jq_madd(acc, s2, t2)
            bad = bad or acc[2] == 0
        assert not carry and not bad
        assert encoding_from_projective(*acc) == o.compress_to_field(o.scalar_mul(o.GENERATOR, k)), hex(k)
