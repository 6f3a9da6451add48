// decaf377 group layer on the GPU: extended twisted-Edwards points over Fq
// (a = -1, d = 3021), decaf compress / decompress, Elligator 2 map.
//
// Formulas restated from the reference's arkworks-free twin
// (src/min_curve/element.rs) and its arkworks build (src/ark_curve/*):
//   add        min_curve/element.rs:291-322   (8M + 1 mul by K = 2d)
//   double     min_curve/element.rs:119-136   (4S + 4M)
//   neg        min_curve/element.rs:324-332
//   eq         min_curve/element.rs:334-340
//   compress   ark_curve/encoding.rs:91-128
//   decompress ark_curve/encoding.rs:32-83
//   elligator  ark_curve/elligator.rs:15-62
// The addition law is complete (a = -1 is a square, d a non-square mod q), so
// none of these has exceptional inputs and every thread runs the same code.
#pragma once
#include "engine.h"
#include "isqrt.cuh"

// Every coordinate kept in a pt_t / niels_t / cached_t is a storage-class value (< 2q,
// fq.cuh); the formulas below are arranged so that their outputs are again < 2q without
// any reduction on the hot paths (the static bounds in the comments are in units of q
// and are enforced by the types).
struct pt_t {
  fq_t x, y, z, t;
};

// K = 2d = 6042 (min_curve/constants.rs:34-39): small enough for fq_mul_small
constexpr uint32_t D377_K = 6042;

// Affine point cached for mixed addition: (y - x, y + x, 2d * x * y), Z = 1; canonical
// (< q) because the entries come from tables built once.
struct niels_t {
  fq_r ymx, ypx, kt;
};

D377_DI pt_t pt_identity() {
  pt_t p;
  p.x = fq_zero();
  p.y = fq_one();
  p.z = fq_one();
  p.t = fq_zero();
  return p;
}

D377_DI niels_t niels_identity() {
  niels_t n;
  n.ymx = fq_one();
  n.ypx = fq_one();
  n.kt = fq_zero();
  return n;
}

// General addition (min_curve/element.rs:291-322).  Not on a hot path (tree sums, tails):
// E is folded once so that the four output products stay below 2q.
D377_DI pt_t pt_add(const pt_t& p, const pt_t& o) {
  auto a = fq_mul(fq_sub(p.y, p.x), fq_sub(o.y, o.x));   // 4 * 4      -> 2.17
  auto b = fq_mul(fq_add(p.y, p.x), fq_add(o.y, o.x));   // 4 * 4      -> 2.17
  auto c = fq_mul(fq_mul_small<D377_K>(p.t), o.t);       // 3 * 2      -> 1.44
  auto d = fq_mul(fq_dbl(p.z), o.z);                     // 4 * 2      -> 1.59
  auto e = fq_fold(fq_sub(b, a));                        // 5.17       -> 2
  auto f = fq_sub(d, c);                                 // 3.59
  auto g = fq_add(d, c);                                 // 2.76
  auto h = fq_add(b, a);                                 // 4.34
  pt_t r;
  r.x = fq_mul(e, f);                                    // 1.53
  r.y = fq_mul(g, h);                                    // 1.88
  r.t = fq_mul(e, h);                                    // 1.64
  r.z = fq_mul(f, g);                                    // 1.73
  return r;
}

// p + n where n is a cached affine point (7M).  2 Z1 would be 4q; Z1 is folded to < q
// first (one conditional subtraction instead of a multiplication).
D377_DI pt_t pt_add_affine_fwd(const pt_t& p, const fq_r& ymx, const fq_r& ypx, const fq_r& kt);
D377_DI pt_t pt_add_niels(const pt_t& p, const niels_t& n) {
  return pt_add_affine_fwd(p, n.ymx, n.ypx, n.kt);
}

// p + n for a canonical affine cached point (y-x, y+x, 2d*x*y), 7M.  A subtraction is the
// same call with (y+x, y-x, -2d*x*y): callers that keep both signs of kt in memory apply
// the sign of a bucket entry purely by choosing load addresses.
template <bool kNeedT = true>
D377_DI pt_t pt_add_affine(const pt_t& p, const fq_r& ymx, const fq_r& ypx, const fq_r& kt) {
  auto a = fq_mul(fq_sub(p.y, p.x), ymx);                // 4 * 1 -> 1.30
  auto b = fq_mul(fq_add(p.y, p.x), ypx);                // 4 * 1 -> 1.30
  auto c = fq_mul(p.t, kt);                              // 2 * 1 -> 1.15
  auto d = fq_dbl(fq_reduce(p.z));                       // 2
  auto e = fq_sub(b, a);                                 // 3.30
  auto h = fq_add(b, a);                                 // 2.59
  auto f = fq_sub(d, c);                                 // 4
  auto g = fq_add(d, c);                                 // 3.15
  pt_t r;
  r.x = fq_mul(e, f);                                    // 1.97
  r.y = fq_mul(g, h);                                    // 1.60
  if (kNeedT) r.t = fq_mul(e, h); else r.t = p.t;        // 1.62
  r.z = fq_mul(f, g);                                    // 1.92
  return r;
}

D377_DI pt_t pt_add_affine_fwd(const pt_t& p, const fq_r& ymx, const fq_r& ypx, const fq_r& kt) {
  return pt_add_affine<true>(p, ymx, ypx, kt);
}

// -n: swap (y-x, y+x), negate kt.
D377_DI niels_t niels_cneg(const niels_t& n, bool neg) {
  niels_t r;
  r.ymx = fq_select(neg, n.ypx, n.ymx);
  r.ypx = fq_select(neg, n.ymx, n.ypx);
  r.kt = fq_select(neg, fq_reduce(fq_neg(n.kt)), n.kt);   // q - 0 = q -> 0
  return r;
}

// Doubling (min_curve/element.rs:119-136, 4S + 4M) with a = -1: D = -A, so G = B - A,
// H = -(A + B), F = G - C.  The signs of F and H are flipped together (F' = C - G,
// H' = A + B): that negates all four output coordinates, i.e. the same projective point.
// kNeedT = false skips T3 = E*H (7 instead of 8 multiplications): a doubling that is
// followed by another doubling never reads T.
template <bool kNeedT = true>
D377_DI pt_t pt_dbl(const pt_t& p) {
  auto a = fq_sqr(p.x);                                  // 1.30
  auto b = fq_sqr(p.y);                                  // 1.30
  auto c = fq_dbl(fq_sqr(p.z));                          // 2.59
  auto hh = fq_add(a, b);                                // 2.59   H' = A + B
  auto s = fq_sqr(fq_add(p.x, p.y));                     // 4^2 -> 2.17
  auto e = fq_fold(fq_sub(s, hh));                       // 5.17 -> 2     E = 2XY
  auto g = fq_fold(fq_sub(b, a));                        // 3.30 -> 2     G = B - A
  auto ff = fq_sub(c, g);                                // 4.59          F' = C - G
  pt_t r;
  r.x = fq_mul(e, ff);                                   // 1.67
  r.y = fq_mul(g, hh);                                   // 1.38
  if (kNeedT) r.t = fq_mul(e, hh); else r.t = p.t;       // 1.38
  r.z = fq_mul(ff, g);                                   // 1.67
  return r;
}

// The same doubling with the T decision taken at run time (warp-uniform): ONE instance of
// the code for loops whose body must stay inside the instruction cache (pt_scalar_mul).
D377_DI pt_t pt_dbl_flag(const pt_t& p, bool need_t) {
  auto a = fq_sqr(p.x);
  auto b = fq_sqr(p.y);
  auto c = fq_dbl(fq_sqr(p.z));
  auto hh = fq_add(a, b);
  auto s = fq_sqr(fq_add(p.x, p.y));
  auto e = fq_fold(fq_sub(s, hh));
  auto g = fq_fold(fq_sub(b, a));
  auto ff = fq_sub(c, g);
  pt_t r;
  r.x = fq_mul(e, ff);
  r.y = fq_mul(g, hh);
  r.t = p.t;
  if (need_t) r.t = fq_mul(e, hh);
  r.z = fq_mul(ff, g);
  return r;
}

// Projective point cached for repeated addition: (Y - X, Y + X, 2d * T, 2Z); an
// addition against it costs 8 multiplications (7 when the sum's T is not needed).
struct cached_t {
  fq_t ymx, ypx, kt, z2;
};

D377_DI cached_t cached_from(const pt_t& p) {
  cached_t c;
  c.ymx = fq_fold(fq_sub(p.y, p.x));
  c.ypx = fq_fold(fq_add(p.y, p.x));
  c.kt = fq_fold(fq_mul_small<D377_K>(p.t));
  c.z2 = fq_fold(fq_dbl(p.z));
  return c;
}

D377_DI cached_t cached_identity() {
  cached_t c;
  c.ymx = fq_one();
  c.ypx = fq_one();
  c.kt = fq_zero();
  c.z2 = fq_const(FQ_TWO);
  return c;
}

// p + n or p - n for a cached projective n (8M).  The sign costs no arithmetic:
// -n swaps (Y-X, Y+X) and negates 2dT, and negating C just swaps F = D - C and G = D + C.
// kSwapped: the caller already exchanged n.ymx / n.ypx for a negative sign (by choosing
// the load addresses), so only the F/G exchange is left.
template <bool kNeedT = true, bool kSwapped = false>
D377_DI pt_t pt_add_cached(const pt_t& p, const cached_t& n, bool neg) {
  auto a = fq_mul(fq_sub(p.y, p.x), fq_select(neg && !kSwapped, n.ypx, n.ymx));   // 4 * 2 -> 1.59
  auto b = fq_mul(fq_add(p.y, p.x), fq_select(neg && !kSwapped, n.ymx, n.ypx));   // 4 * 2 -> 1.59
  auto c = fq_mul(p.t, n.kt);                                        // 2 * 2 -> 1.30
  auto d = fq_mul(p.z, n.z2);                                        // 2 * 2 -> 1.30
  auto e = fq_sub(b, a);                                             // 3.59
  auto h = fq_add(b, a);                                             // 3.17
  auto f0 = fq_sub(d, c);                                            // 3.30
  auto g0 = fq_add(d, c);                                            // 2.59
  auto f = fq_select(neg, g0, f0), g = fq_select(neg, f0, g0);       // 3.30
  pt_t r;
  r.x = fq_mul(e, f);                                                // 1.87
  r.y = fq_mul(g, h);                                                // 1.77
  if (kNeedT) r.t = fq_mul(e, h); else r.t = p.t;                    // 1.83
  r.z = fq_mul(f, g);                                                // 1.80
  return r;
}

// run-time T decision, see pt_dbl_flag
D377_DI pt_t pt_add_cached_flag(const pt_t& p, const cached_t& n, bool neg, bool need_t) {
  auto a = fq_mul(fq_sub(p.y, p.x), fq_select(neg, n.ypx, n.ymx));
  auto b = fq_mul(fq_add(p.y, p.x), fq_select(neg, n.ymx, n.ypx));
  auto c = fq_mul(p.t, n.kt);
  auto d = fq_mul(p.z, n.z2);
  auto e = fq_sub(b, a);
  auto h = fq_add(b, a);
  auto f0 = fq_sub(d, c);
  auto g0 = fq_add(d, c);
  auto f = fq_select(neg, g0, f0), g = fq_select(neg, f0, g0);
  pt_t r;
  r.x = fq_mul(e, f);
  r.y = fq_mul(g, h);
  r.t = p.t;
  if (need_t) r.t = fq_mul(e, h);
  r.z = fq_mul(f, g);
  return r;
}

D377_DI pt_t pt_neg(const pt_t& p) {
  pt_t r = p;
  r.x = fq_neg(fq_reduce(p.x));
  r.t = fq_neg(fq_reduce(p.t));
  return r;
}

D377_DI pt_t pt_select(bool c, const pt_t& a, const pt_t& b) {
  pt_t r;
  r.x = fq_select(c, a.x, b.x);
  r.y = fq_select(c, a.y, b.y);
  r.z = fq_select(c, a.z, b.z);
  r.t = fq_select(c, a.t, b.t);
  return r;
}

// affine (Z = 1) extended point -> cached form, canonical
D377_DI niels_t niels_from_affine(const fq_t& x, const fq_t& y) {
  niels_t n;
  n.ymx = fq_reduce(fq_sub(y, x));
  n.ypx = fq_reduce(fq_add(y, x));
  n.kt = fq_reduce(fq_mul_small<D377_K>(fq_mul(x, y)));
  return n;
}

// ---- wire I/O: X||Y||Z||T, 32-byte Montgomery LE each (SURVEY 8b) ----------
D377_DI pt_t pt_load(const uint8_t* p) {
  pt_t r;
  r.x = fq_load(p);
  r.y = fq_load(p + 32);
  r.z = fq_load(p + 64);
  r.t = fq_load(p + 96);
  return r;
}

// caller-supplied Elements (untrusted limbs, see fq_load_wire)
D377_DI pt_t pt_load_wire(const uint8_t* p) {
  pt_t r;
  r.x = fq_load_wire(p);
  r.y = fq_load_wire(p + 32);
  r.z = fq_load_wire(p + 64);
  r.t = fq_load_wire(p + 96);
  return r;
}

// internal workspaces (bucket sums, partial sums): lazily reduced
D377_DI void pt_store(uint8_t* p, const pt_t& a) {
  fq_store(p, a.x);
  fq_store(p + 32, a.y);
  fq_store(p + 64, a.z);
  fq_store(p + 96, a.t);
}

// ABI outputs: canonical Montgomery limbs, as the reference's Fq holds them
D377_DI void pt_store_canon(uint8_t* p, const pt_t& a) {
  fq_store_canon(p, a.x);
  fq_store_canon(p + 32, a.y);
  fq_store_canon(p + 64, a.z);
  fq_store_canon(p + 96, a.t);
}

// ---- codec -----------------------------------------------------------------

// ark_curve/encoding.rs:91-114.  Returns the CANONICAL bytes of |s| as limbs.
D377_DI fq_r pt_compress_to_field(const pt_t& p, const isqrt_smem_t& sm) {
  auto u1 = fq_mul(fq_add(p.x, p.t), fq_sub(p.x, p.t));
  fq_t v;
  // a - d = -3022: small-constant products (fq_mul_small) instead of Montgomery ones
  fq_isqrt(v, fq_mul(fq_neg(fq_mul_small<3022>(u1)), fq_sqr(p.x)), sm);
  auto u2 = fq_abs(fq_mul(v, u1));
  auto u3 = fq_sub(fq_mul(u2, p.z), p.t);
  auto s = fq_mul(fq_mul(fq_neg(fq_mul_small<3022>(v)), u3), p.x);
  // abs() and serialisation both need the canonical value: reduce once, then
  // negate in the canonical domain.
  fq_r sc = fq_from_mont(s);
  bool neg = sc.l[0] & 1u;
  fq_r sn = fq_assume<1000>(fq_neg(sc));  // only used when sc is odd: sc != 0, so q - sc < q
  return fq_select(neg, sn, sc);
}

// ark_curve/encoding.rs:32-83.  `s_raw` are the 32 encoding bytes as limbs.
D377_DI bool pt_decompress(pt_t& out, const fq_raw_t& s_raw, const isqrt_smem_t& sm) {
  bool ok = (s_raw.l[7] >> 29) == 0;        // top three bits clear
  ok = ok && fq_raw_is_canonical(s_raw);    // from_bytes_checked
  ok = ok && !(s_raw.l[0] & 1u);            // s non-negative
  fq_t s = fq_to_mont(s_raw);
  auto ss = fq_sqr(s);
  auto u1 = fq_sub(fq_one(), ss);
  auto u1sq = fq_sqr(u1);
  auto u2 = fq_sub(u1sq, fq_mul_small<2 * D377_K>(ss));   // 4d = 12084
  fq_t v0;
  bool was_square = fq_isqrt(v0, fq_mul(u2, u1sq), sm);
  ok = ok && was_square;
  auto two_s_u1 = fq_mul(fq_dbl(s), u1);
  auto check = fq_mul(two_s_u1, v0);
  auto v = fq_select(fq_is_negative(check), fq_neg(v0), v0);
  out.x = fq_mul(fq_mul(two_s_u1, fq_sqr(v)), u2);
  out.y = fq_mul(fq_mul(fq_add(fq_one(), ss), v), u1);
  out.z = fq_one();
  out.t = fq_mul(out.x, out.y);
  return ok;
}

// Element i of a caller's point array in format kFmt (D377_PT_ELEMENT, _ENCODING, _AFFINE or
// _XYZ) -> extended coordinates.  An invalid encoding reads as the identity and returns false;
// `sm` is used by encodings only.
template <int kFmt>
D377_DI bool pt_load_fmt(pt_t& p, const uint8_t* pts, size_t i, const isqrt_smem_t& sm) {
  const uint8_t* b = pts + d377::pt_bytes(kFmt) * i;
  if (kFmt == D377_PT_ENCODING) {
    const bool good = pt_decompress(p, fq_load_raw(b), sm);
    p = pt_select(good, p, pt_identity());
    return good;
  }
  if (kFmt == D377_PT_ELEMENT) {
    p = pt_load_wire(b);
  } else if (kFmt == D377_PT_AFFINE) {
    p.x = fq_load_wire(b);
    p.y = fq_load_wire(b + 32);
    p.z = fq_one();
    p.t = fq_mul(p.x, p.y);
  } else {
    // (X : Y : Z) without T: (XZ : YZ : Z^2 : XY) is the same point in extended coordinates
    fq_t x = fq_load_wire(b), y = fq_load_wire(b + 32), z = fq_load_wire(b + 64);
    p.x = fq_mul(x, z);
    p.y = fq_mul(y, z);
    p.z = fq_sqr(z);
    p.t = fq_mul(x, y);
  }
  return true;
}

// ark_curve/elligator.rs:15-54: r0 (Montgomery form) -> the Jacobi-quartic pair (s, t).
D377_DI void pt_elligator_st(fq_t& s_out, fq_t& t_out, const fq_t& r0, const isqrt_smem_t& sm) {
  const fq_r one = fq_one();
  const fq_r D = fq_const(FQ_D);
  const fq_r dma = fq_const(FQ_D_MINUS_A);
  auto r = fq_mul(fq_const(FQ_ZETA), fq_sqr(r0));
  auto den = fq_mul(fq_sub(fq_mul_small<3021>(r), dma), fq_sub(fq_mul_small<3022>(r), D));   // d = 3021, d - a = 3022
  auto num = fq_fold(fq_neg(fq_mul_small<6043>(fq_add(r, one))));   // a - 2d = -6043
  fq_t isri0;
  bool iss = fq_isqrt(isri0, fq_mul(num, den), sm);
  // sgn = iss ? 1 : -1 ; twiddle = iss ? 1 : r0
  auto isri = fq_mul(isri0, fq_select(iss, one, r0));
  auto s0 = fq_mul(isri, num);
  // t = -sgn * isri * s * (r - 1) * (a - 2d)^2 - 1
  auto tt = fq_mul(fq_mul(fq_mul(isri, s0), fq_sub(r, one)), fq_const(FQ_A_MINUS_2D_SQ));
  auto t = fq_sub(fq_select(iss, fq_neg(tt), tt), one);
  bool sneg = fq_is_negative(s0);
  auto s = fq_select(sneg == iss, fq_neg(s0), s0);
  s_out = fq_fold(s);
  t_out = fq_fold(t);
}

// ark_curve/elligator.rs:56-62: (s, t) -> (E*H : F*G : F*H : E*G) with a = -1:
// E = 2s, F = 1 - s^2, G = 1 + s^2, H = t.
D377_DI pt_t pt_from_jacobi(const fq_t& s, const fq_t& t) {
  const fq_r one = fq_one();
  auto s2 = fq_sqr(s);
  auto E = fq_dbl(s);
  auto F = fq_sub(one, s2);
  auto G = fq_add(one, s2);
  pt_t p;
  p.x = fq_mul(E, t);
  p.y = fq_mul(F, G);
  p.z = fq_mul(F, t);
  p.t = fq_mul(E, G);
  return p;
}

D377_DI pt_t pt_elligator(const fq_t& r0, const isqrt_smem_t& sm) {
  fq_t s, t;
  pt_elligator_st(s, t, r0, sm);
  return pt_from_jacobi(s, t);
}

// ---- 1 / x for every thread of a CTA with ONE field inversion (Montgomery's trick) -------
// Warp-level inclusive prefix / suffix products by shuffles, the kWarps warp totals through
// shared memory, warp 0 inverts the CTA product (fq_inv_vartime: no multiplications, so the
// other CTAs of the SM keep the multiply pipe busy meanwhile), every thread assembles its
// own inverse: ~15 multiplications per thread.  0 -> 0.  Every thread of the CTA must call
// it (two barriers); sh: kWarps + 1 entries of shared memory.
D377_DI fq_t fq_shfl_up(const fq_t& v, int d) {
  fq_t r;
#pragma unroll
  for (int i = 0; i < 8; i++) r.l[i] = __shfl_up_sync(0xffffffffu, v.l[i], d);
  return r;
}
D377_DI fq_t fq_shfl_down(const fq_t& v, int d) {
  fq_t r;
#pragma unroll
  for (int i = 0; i < 8; i++) r.l[i] = __shfl_down_sync(0xffffffffu, v.l[i], d);
  return r;
}

template <int kWarps>
D377_DI fq_t fq_cta_inverse(const fq_t& x_in, fq_t* sh) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const bool zero = fq_is_zero(x_in);
  const fq_t x = fq_select(zero, fq_t(fq_one()), x_in);
  fq_t pre = x, suf = x;
#pragma unroll 1
  for (int o = 1; o < 32; o <<= 1) {
    fq_t y = fq_shfl_up(pre, o);
    fq_t m = fq_mul(pre, y);
    pre = fq_select(lane >= o, m, pre);
    fq_t w = fq_shfl_down(suf, o);
    fq_t m2 = fq_mul(suf, w);
    suf = fq_select(lane + o < 32, m2, suf);
  }
  if (lane == 31) sh[wid] = pre;
  __syncthreads();
  if (wid == 0) {
    fq_t tot = sh[0];
#pragma unroll 1
    for (int v = 1; v < kWarps; v++) tot = fq_mul(tot, sh[v]);
    fq_t inv = fq_inv_vartime(tot);
    if (lane == 0) sh[kWarps] = inv;
  }
  __syncthreads();
  // 1 / (this warp's total) = inv(CTA total) * product of the other warps' totals
  fq_t inv = sh[kWarps];
#pragma unroll 1
  for (int v = 0; v < kWarps; v++)
    if (v != wid) inv = fq_mul(inv, sh[v]);
  // 1 / x = that * (product of the lanes before) * (product of the lanes after)
  fq_t ex_pre = fq_shfl_up(pre, 1), ex_suf = fq_shfl_down(suf, 1);
  inv = fq_mul(inv, fq_select(lane == 0, fq_t(fq_one()), ex_pre));
  inv = fq_mul(inv, fq_select(lane == 31, fq_t(fq_one()), ex_suf));
  return fq_select(zero, fq_t(fq_zero()), inv);
}

// The same per WARP: no shared memory and no barrier.  The warp total is broadcast and every
// lane runs the (multiplication-free) binary-GCD inversion on the same value, i.e. the warp
// executes it once in lockstep.  Four times the inversions of the CTA-wide form, but they
// are ALU work next to kernels bound by the multiply pipe, and a warp that inverts stalls
// only itself: with the CTA-wide form the other three warps of the CTA sit at the barrier
// for the ~50 us of the inversion (14-24 % of the stall samples of the fused kernels,
// profiles/r2_stalls_codec20.txt).  Measured per kernel: hash_to_curve + compress gains
// (104.3 -> 108.5 Melem/s at 2^22), encode_to_curve + compress and the quartic fixed base
// do not (206 / 204, 442 / 440) -- those keep the CTA-wide form.
D377_DI fq_t fq_warp_inverse(const fq_t& x_in) {
  const int lane = threadIdx.x & 31;
  const bool zero = fq_is_zero(x_in);
  const fq_t x = fq_select(zero, fq_t(fq_one()), x_in);
  fq_t pre = x, suf = x;
#pragma unroll 1
  for (int o = 1; o < 32; o <<= 1) {
    fq_t y = fq_shfl_up(pre, o);
    fq_t m = fq_mul(pre, y);
    pre = fq_select(lane >= o, m, pre);
    fq_t w = fq_shfl_down(suf, o);
    fq_t m2 = fq_mul(suf, w);
    suf = fq_select(lane + o < 32, m2, suf);
  }
  fq_t tot;
#pragma unroll
  for (int i = 0; i < 8; i++) tot.l[i] = __shfl_sync(0xffffffffu, pre.l[i], 31);
  fq_t inv = fq_inv_vartime(tot);
  fq_t ex_pre = fq_shfl_up(pre, 1), ex_suf = fq_shfl_down(suf, 1);
  inv = fq_mul(inv, fq_select(lane == 0, fq_t(fq_one()), ex_pre));
  inv = fq_mul(inv, fq_select(lane == 31, fq_t(fq_one()), ex_suf));
  return fq_select(zero, fq_t(fq_zero()), inv);
}

// vartime_compress(encode_to_curve(r0)) WITHOUT the second inverse square root.
// For a point that comes from the Jacobi quartic, x = 2s / (1 - s^2), y = (1 + s^2) / t with
// t^2 = s^4 - (2 + 4d) s^2 + 1, the radicand of compress (ark_curve/encoding.rs:94-101) is
// a perfect square whose root is known:  (a - d)(1 - y^2) = (2 (a - d) s / t)^2.  Following
// encoding.rs:98-111 with that root w, u2 = |2s / t| and
//   s_enc = | sigma (1 - s^2) / (2s) - (1 + s^2) / (2s) |,  sigma = +1 if 2s/t is
//   non-negative, -1 otherwise,
// i.e. the encoding is |s| when 2s/t is non-negative and |1/s| when it is negative.  Only
// the sign test and 1/s need a division, and divisions batch (fq_cta_inverse of s t):
// ~20 multiplications instead of the 315 of a compress.  Bit-exact with the reference path
// (20 000 random and edge inputs against the oracle in Python; the parity suite compares
// this kernel with compress(elligator) of the oracle).  A projective Z = (1 - s^2) t of
// zero (no such r0 is known) takes the generic path.
// ip = 1 / (s t) supplied by the caller (0 if s t = 0)
D377_DI fq_r pt_jacobi_encoding_with_inverse(const fq_t& s, const fq_t& t, const fq_t& ip) {
  const auto u = fq_mul(fq_dbl(fq_sqr(s)), ip);                    // 2s / t
  const bool flip = fq_is_negative(u);
  const fq_t cand = fq_select(flip, fq_t(fq_mul(t, ip)), s);       // 1/s or s
  const fq_r c = fq_from_mont(cand);
  const fq_r cn = fq_assume<1000>(fq_neg(c));   // only used when c is odd: c != 0, so q - c < q
  return fq_select((c.l[0] & 1u) != 0, cn, c);
}

// vartime_compress(hash_to_curve(r1, r2)) the same way.  The map from the Jacobi quartic
// J: t^2 = s^4 - 2 delta s^2 + 1 (delta = 2d - a = 6043) to the curve is a 2-isogeny, hence a
// homomorphism: E(r1) + E(r2) is the image of (s1, t1) + (s2, t2) under the quartic's own
// addition law (Billet-Joye, epsilon = a^2 = 1):
//   s3 = (s1 t2 + t1 s2) / w,   w = 1 - (s1 s2)^2,
//   t3 = ((1 + (s1 s2)^2)(t1 t2 - 2 delta s1 s2) + 2 s1 s2 (s1^2 + s2^2)) / w^2,
// and the encoding is read off the projective quartic point (ns : nt : w) of the two
// numerators and the denominator (jq_encoding_with_inverse below): ONE batched inversion of
// w ns nt serves the sign test, s3 and 1 / s3.
// The encoding of the image of a PROJECTIVE quartic point (S : T : Z), s = S / Z,
// t = T / Z^2: 2s / t = 2 S Z / T, s = S / Z, 1 / s = Z / S -- one batched inversion of S T Z
// serves all three.  Returns false where the shortcut does not apply (S T Z = 0, or an image
// with projective Z = (1 - s^2) t = 0); the caller then takes a generic path.
// I = 1 / (S T Z) supplied by the caller (0 if the product is 0).
D377_DI bool jq_encoding_with_inverse(fq_r& enc, const fq_t& S, const fq_t& T, const fq_t& Z,
                                      const fq_t& I) {
  const fq_r one = fq_one();
  const fq_t sz = fq_mul(S, Z);
  const auto u = fq_mul(fq_dbl(fq_sqr(sz)), I);          // 2 S Z / T = 2 s / t
  const fq_t TI = fq_mul(T, I);                          // 1 / (S Z)
  const fq_t s3 = fq_mul(fq_sqr(S), TI);                 // S / Z
  const fq_t is3 = fq_mul(fq_sqr(Z), TI);                // Z / S
  const bool flip = fq_is_negative(u);
  const fq_t cand = fq_select(flip, is3, s3);
  const fq_r c = fq_from_mont(cand);
  const fq_r cn = fq_assume<1000>(fq_neg(c));   // only used when c is odd: c != 0, so q - c < q
  enc = fq_select((c.l[0] & 1u) != 0, cn, c);
  return !(fq_is_zero(I) || fq_is_zero(fq_sub(one, fq_sqr(s3))));
}

D377_DI void pt_jacobi_sum(fq_t& ns, fq_t& nt, fq_t& w, const fq_t& s1, const fq_t& t1, const fq_t& s2,
                           const fq_t& t2) {
  const fq_r one = fq_one();
  const fq_t p = fq_mul(s1, s2);
  const fq_t p2 = fq_sqr(p);
  w = fq_fold(fq_sub(one, p2));
  ns = fq_fold(fq_add(fq_mul(s1, t2), fq_mul(t1, s2)));
  const fq_t inner = fq_fold(fq_sub(fq_mul(t1, t2), fq_mul_small<12086>(p)));        // 2 delta = 12086
  const fq_t sq = fq_fold(fq_add(fq_sqr(s1), fq_sqr(s2)));
  nt = fq_fold(fq_add(fq_mul(fq_fold(fq_add(one, p2)), inner), fq_mul(fq_fold(fq_dbl(p)), sq)));
  // (s3, t3) = (ns / w, nt / w^2): the projective quartic point (ns : nt : w)
}

// ---- arithmetic on the Jacobi quartic itself (fixed-base multiplication, scalar.cu) --------
// Projective point (S : T : Z), s = S / Z, t = T / Z^2; neutral element (0 : 1 : 1); the
// negative of (s, t) is (-s, t).
struct jq_t {
  fq_t S, T, Z;
};

D377_DI jq_t jq_identity() {
  jq_t p;
  p.S = fq_zero();
  p.T = fq_one();
  p.Z = fq_one();
  return p;
}

// p + (s2, t2) for an affine, canonical (s2, t2, s2^2): the unified Billet-Joye law in
// projective form,  S3 = S1 Z1 t2 + T1 s2,  Z3 = Z1^2 - S1^2 s2^2,
//   T3 = (Z1^2 + S1^2 s2^2)(T1 t2 - 2 delta S1 Z1 s2) + 2 S1 Z1 s2 (S1^2 + s2^2 Z1^2):
// 9 M + 2 S + 1 K.  Z3 = 0 marks the exceptional pairs (s1 s2 = +-1); callers check it.
D377_DI jq_t jq_madd(const jq_t& p, const fq_r& s2, const fq_r& t2, const fq_r& s2sq) {
  auto A = fq_sqr(p.S);                                  // 1.29
  auto B = fq_sqr(p.Z);                                  // 1.29
  auto C = fq_mul(p.S, p.Z);                             // 1.29
  auto D = fq_mul(A, s2sq);                              // 1.09
  auto H = fq_mul(C, s2);                                // 1.09
  auto I = fq_sub(fq_mul(p.T, t2), fq_mul_small<12086>(H));   // 1.15 + 3
  auto J = fq_add(A, fq_mul(s2sq, B));                   // 2.38
  jq_t r;
  r.S = fq_fold(fq_add(fq_mul(C, t2), fq_mul(p.T, s2))); // 2.24 -> 2
  r.Z = fq_fold(fq_sub(B, D));                           // 3.29 -> 2
  r.T = fq_fold(fq_add(fq_mul(fq_add(B, D), I), fq_mul(fq_dbl(H), J)));   // 1.72 + 1.38 -> 2
  return r;
}

// 2 p (table building only): S3 = 2 S T Z, Z3 = Z^4 - S^4,
//   T3 = (Z^4 + S^4)(T^2 - 2 delta S^2 Z^2) + 4 S^4 Z^4
D377_DI jq_t jq_dbl(const jq_t& p) {
  auto A = fq_sqr(p.S), B = fq_sqr(p.Z);
  auto A2 = fq_sqr(A), B2 = fq_sqr(B);
  auto inner = fq_sub(fq_sqr(p.T), fq_mul_small<12086>(fq_mul(A, B)));
  jq_t r;
  r.S = fq_mul(fq_mul(p.S, p.T), fq_dbl(p.Z));
  r.Z = fq_fold(fq_sub(B2, A2));
  r.T = fq_fold(fq_add(fq_mul(fq_add(B2, A2), inner), fq_dbl(fq_dbl(fq_mul(A2, B2)))));
  return r;
}

// 251-bit scalar as 8 little-endian limbs; canonical (< r) check, fr.rs:108-115
D377_DI bool fr_raw_is_canonical(const fq_raw_t& s) {
  uint32_t bw = 0;
  // s - r borrow chain
  uint64_t acc = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    uint64_t d = (uint64_t)s.l[i] - (uint64_t)FR_MOD[i] - bw;
    bw = (uint32_t)(d >> 63);
    acc |= d;
  }
  (void)acc;
  return bw != 0;
}

// Fr::into_bigint on the device: the in-memory form of the reference's Fr is Montgomery
// (fr/u64/wrapper.rs, fr/u32/wrapper.rs: x * 2^256 mod r); callers that hand those limbs
// over unconverted (D377_SCALARS_MONTGOMERY) get the canonical integer here -- one
// word-serial Montgomery reduction, -r^-1 mod 2^32 = 0x70e3da01 (fr/u32/fiat.rs).  Any
// 256-bit input gives (s + M r) / 2^256 <= r, so one conditional subtraction canonicalises.
D377_DI fq_raw_t fr_from_mont(const fq_raw_t& s) {
  uint32_t t[8];
#pragma unroll
  for (int i = 0; i < 8; i++) t[i] = s.l[i];
  uint32_t top = 0;
#pragma unroll 1
  for (int i = 0; i < 8; i++) {
    const uint32_t m = t[0] * 0x70e3da01u;
    uint64_t c = ((uint64_t)m * FR_MOD[0] + t[0]) >> 32;
#pragma unroll
    for (int j = 1; j < 8; j++) {
      c += (uint64_t)m * FR_MOD[j] + t[j];
      t[j - 1] = (uint32_t)c;
      c >>= 32;
    }
    c += top;
    t[7] = (uint32_t)c;
    top = (uint32_t)(c >> 32);
  }
  // subtract r when t >= r
  uint32_t d[8];
  uint64_t bw = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    const uint64_t x = (uint64_t)t[i] - FR_MOD[i] - bw;
    d[i] = (uint32_t)x;
    bw = (x >> 63) & 1u;
  }
  const bool ge = top != 0 || bw == 0;
  fq_raw_t r;
#pragma unroll
  for (int i = 0; i < 8; i++) r.l[i] = ge ? d[i] : t[i];
  return r;
}

// [k]P for a 256-bit little-endian k (min_curve/element.rs:138-153 and ark-ec's
// mul_bigint, ops/projective.rs:123-131, give the same group element; the result is
// compared through its encoding).  Signed 4-bit fixed windows: with
// k' = k + 0x88...8 the digits are d_i = nibble_i(k') - 8 in [-8, 8), plus the carry
// out of that addition as a 65th digit, so every 256-bit k is handled (canonical
// scalars never produce it).  The table {1..8}P sits in per-thread local memory in
// cached form; every lane runs the same 4 doublings + 1 addition per digit (a zero
// digit adds the cached identity), so a warp never diverges on scalar bits.
// Cost: 256 doublings (7M, every 4th 8M) + 65 additions (7M) + 71 for the table.
D377_DI pt_t pt_scalar_mul(const pt_t& p, const fq_raw_t& k) {
  cached_t tab[9];
  tab[0] = cached_identity();
  {
    pt_t m = p;
    tab[1] = cached_from(m);
#pragma unroll 1
    for (int j = 2; j <= 8; j++) {
      m = pt_add_cached<true>(m, tab[1], false);
      tab[j] = cached_from(m);
    }
  }
  // k' = k + 0x8888...8
  uint32_t kp[8], top;
  asm("add.cc.u32 %0, %9, 0x88888888;\n\t"
      "addc.cc.u32 %1, %10, 0x88888888;\n\t"
      "addc.cc.u32 %2, %11, 0x88888888;\n\t"
      "addc.cc.u32 %3, %12, 0x88888888;\n\t"
      "addc.cc.u32 %4, %13, 0x88888888;\n\t"
      "addc.cc.u32 %5, %14, 0x88888888;\n\t"
      "addc.cc.u32 %6, %15, 0x88888888;\n\t"
      "addc.cc.u32 %7, %16, 0x88888888;\n\t"
      "addc.u32 %8, 0, 0;"
      : "=r"(kp[0]), "=r"(kp[1]), "=r"(kp[2]), "=r"(kp[3]), "=r"(kp[4]), "=r"(kp[5]), "=r"(kp[6]),
        "=r"(kp[7]), "=r"(top)
      : "r"(k.l[0]), "r"(k.l[1]), "r"(k.l[2]), "r"(k.l[3]), "r"(k.l[4]), "r"(k.l[5]), "r"(k.l[6]),
        "r"(k.l[7]));
  // digit 64 (weight 16^64) is the carry: acc = top * P
  pt_t acc = pt_identity();
  acc = pt_add_cached<false>(acc, tab[top & 1u], false);
#pragma unroll 1
  for (int i = 63; i >= 0; i--) {
    // One doubling body and one addition body, T decided at run time: unrolled (three
    // doublings without T, one with, two additions) the loop was ~44 multiplication bodies,
    // more than the SM's instruction cache holds, and 19 % of the kernel's stall samples were
    // "no instruction" (profiles/r2_stalls_codec20_final.txt).
#pragma unroll 1
    for (int j = 0; j < 4; j++) acc = pt_dbl_flag(acc, j == 3);
    uint32_t limb = 0;
#pragma unroll
    for (int j = 0; j < 8; j++) limb = (i >> 3) == j ? kp[j] : limb;
    int d = (int)((limb >> ((i & 7) * 4)) & 15u) - 8;
    int mag = d < 0 ? -d : d;
    // the result's T (i == 0) is read by compress / the caller
    acc = pt_add_cached_flag(acc, tab[mag], d < 0, i == 0);
  }
  return acc;
}

// ---- on-curve predicate (ark_curve/on_curve.rs:17-38) ------------------------
// curve equation (a = -1: Y^2 - X^2 = Z^2 + d T^2), Segre embedding T Z = X Y, Z != 0.
D377_DI bool pt_on_curve(const pt_t& p) {
  auto xx = fq_sqr(p.x), yy = fq_sqr(p.y), zz = fq_sqr(p.z), tt = fq_sqr(p.t);
  const bool curve = fq_eq(fq_sub(yy, xx), fq_add(zz, fq_mul_small<3021>(tt)));
  const bool segre = fq_eq(fq_mul(p.t, p.z), fq_mul(p.x, p.y));
  return curve && segre && !fq_is_zero(p.z);
}

// [2r]P == Projective::zero()  (on_curve.rs:25-34; arkworks compares (X : Y : Z) with
// (0 : 1 : 1), i.e. X = 0 and Y = Z)
D377_DI bool pt_order_divides_2r(const pt_t& p) {
  fq_raw_t two_r;
  uint32_t cy = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    two_r.l[i] = (FR_MOD[i] << 1) | cy;
    cy = FR_MOD[i] >> 31;
  }
  const pt_t m = pt_scalar_mul(p, two_r);
  return fq_is_zero(m.x) && fq_eq(m.y, m.z);
}

// Debug builds (-DD377_DEBUG_ON_CURVE, the reference keeps the same predicate alive in CI
// through debug assertions) check every point a kernel produces and count the failures in a
// per-translation-unit device word read back by d377_debug_failures; -DD377_DEBUG_ORDER
// adds the [2r]P test (one scalar multiplication per point).
#ifdef D377_DEBUG_ON_CURVE
static __device__ unsigned long long g_dbg_fail = 0ull;
static __device__ unsigned long long g_dbg_checked = 0ull;
D377_DI void pt_debug_check(const pt_t& p) {
  bool good = pt_on_curve(p);
#ifdef D377_DEBUG_ORDER
  good = good && pt_order_divides_2r(p);
#endif
  atomicAdd(&g_dbg_checked, 1ull);
  if (!good) atomicAdd(&g_dbg_fail, 1ull);
}
#define D377_DBG_POINT(p) pt_debug_check(p)
#define D377_DBG_READER(name)                                                          \
  void name(unsigned long long* fail, unsigned long long* checked) {                   \
    cudaMemcpyFromSymbol(fail, g_dbg_fail, sizeof(unsigned long long));               \
    cudaMemcpyFromSymbol(checked, g_dbg_checked, sizeof(unsigned long long));         \
  }
#else
#define D377_DBG_POINT(p) ((void)0)
#define D377_DBG_READER(name)                                                          \
  void name(unsigned long long* fail, unsigned long long* checked) { *fail = 0; *checked = 0; }
#endif
