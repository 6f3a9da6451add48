// Batch codec kernels, one element per thread: vartime_decompress, vartime_compress,
// Elligator encode_to_curve / hash_to_curve, and the batch inverse square roots.
// Reference items replaced are cited per kernel; the device arithmetic lives in
// fq.cuh / isqrt.cuh / point.cuh.  (Own translation unit so that the heavy kernels of
// the library compile in parallel.)
#include "engine.h"
#include "point.cuh"

namespace d377 {

constexpr int kCodecBlock = 128;  // 8 isqrt slots * 32 B * 128 = 32 KB shared / CTA
static size_t codec_smem() { return ISQRT_SMEM_WORDS(kCodecBlock) * sizeof(uint32_t); }

// Fq input of the Elligator kernels: `width` bytes per element, reduced exactly like
// Fq::from_le_bytes_mod_order (fields/fq.rs:90-102).  32 bytes -- what the reference's own
// tests feed (tests/operations.rs:6-11) -- is one Montgomery product; wider inputs (64-byte
// hash outputs are the usual hash_to_curve input) take the out-of-line Horner.
__device__ __noinline__ fq_t fq_input_wide(const uint8_t* p, size_t width) {
  return fq_from_le_bytes_wide(p, width);
}
D377_DI fq_t fq_input(const uint8_t* base, size_t width, size_t i) {
  if (width == 32) return fq_to_mont(fq_load_raw(base + 32 * i));
  return fq_input_wide(base + width * i, width);
}

// Encoding::vartime_decompress, ark_curve/encoding.rs:32-83.  kAffine: the AffinePoint form
// of the same point (CanonicalDeserialize for AffinePoint, ark_curve/serialize.rs:8-28:
// decompress, then Element -> AffinePoint); decompression produces Z = 1, so x||y IS the
// affine point and no inversion is needed.
template <bool kAffine>
__global__ void __launch_bounds__(kCodecBlock)
k_decompress(const uint8_t* __restrict__ enc, size_t n, uint8_t* __restrict__ out,
             uint8_t* __restrict__ ok) {
  extern __shared__ uint32_t smem[];
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  isqrt_smem_t sm = isqrt_smem(smem);
  fq_raw_t s = fq_load_raw(enc + 32 * i);
  pt_t p;
  bool good = pt_decompress(p, s, sm);
  p = pt_select(good, p, pt_identity());
  D377_DBG_POINT(p);
  if (kAffine) {
    fq_store_canon(out + 64 * i, p.x);
    fq_store_canon(out + 64 * i + 32, p.y);
  } else {
    pt_store_canon(out + 128 * i, p);
  }
  if (ok) ok[i] = good ? 1 : 0;
}

// Element::vartime_compress, ark_curve/encoding.rs:116-128.  kFmt = D377_PT_AFFINE:
// CanonicalSerialize for AffinePoint (ark_curve/serialize.rs:30-46: AffinePoint -> Element,
// then compress), i.e. Z = 1, T = xy.  kFmt = D377_PT_XYZ: the representative
// (XZ : YZ : Z^2 : XY) of the same point, whose T needs no division.
template <int kFmt>
__global__ void __launch_bounds__(kCodecBlock)
k_compress(const uint8_t* __restrict__ in, size_t n, uint8_t* __restrict__ enc) {
  extern __shared__ uint32_t smem[];
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  isqrt_smem_t sm = isqrt_smem(smem);
  pt_t p;
  pt_load_fmt<kFmt>(p, in, i, sm);
  fq_store(enc + 32 * i, pt_compress_to_field(p, sm));
}

// Element::encode_to_curve / hash_to_curve, ark_curve/elligator.rs:67-76
template <bool kHash, bool kEncode>
__global__ void __launch_bounds__(kCodecBlock)
k_elligator(const uint8_t* __restrict__ r1, const uint8_t* __restrict__ r2, size_t width, size_t n,
            uint8_t* __restrict__ out) {
  extern __shared__ uint32_t smem[];
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  isqrt_smem_t sm = isqrt_smem(smem);
  // from_le_bytes_mod_order on 32 bytes == to_mont of the raw 256-bit value
  fq_t a = fq_input(r1, width, i);
  pt_t p = pt_elligator(a, sm);
  if (kHash) {
    fq_t b = fq_input(r2, width, i);
    pt_t q = pt_elligator(b, sm);
    p = pt_add(p, q);
  }
  D377_DBG_POINT(p);
  if (kEncode)
    fq_store(out + 32 * i, pt_compress_to_field(p, sm));
  else
    pt_store_canon(out + 128 * i, p);
}

// vartime_compress(encode_to_curve(r0)) fused: the encoding is read off the Jacobi-quartic
// pair (s, t) of the Elligator map (pt_jacobi_encoding_with_inverse, point.cuh) -- one inverse
// square root per element instead of two, plus one field inversion per CTA.  Every thread of
// the CTA takes part in the batched inversion, so out-of-range threads run on a dummy input.
// (Several elements per thread before one inversion, as in the fixed-base kernel, were
// measured here: 1, 2 and 4 give the same throughput or less -- the parked pairs cost what
// the shorter bubble saves.)
__global__ void __launch_bounds__(kCodecBlock)
k_elligator_encode(const uint8_t* __restrict__ r1, size_t width, size_t n, uint8_t* __restrict__ out) {
  extern __shared__ uint32_t smem[];
  __shared__ fq_t inv_sh[kCodecBlock / 32 + 1];
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool valid = i < n;
  isqrt_smem_t sm = isqrt_smem(smem);
  fq_t a = fq_input(r1, width, valid ? i : 0);
  fq_t s, t;
  pt_elligator_st(s, t, a, sm);
  const fq_t ip = fq_cta_inverse<kCodecBlock / 32>(fq_mul(s, t), inv_sh);   // 1 / (s t), 0 if s t = 0
  fq_r enc = pt_jacobi_encoding_with_inverse(s, t, ip);
  // Z = (1 - s^2) t = 0: not a point the shortcut's derivation covers
  const bool degenerate = fq_is_zero(t) || fq_is_zero(fq_sub(fq_one(), fq_sqr(s)));
  if (degenerate) enc = pt_compress_to_field(pt_from_jacobi(s, t), sm);
  if (valid) fq_store(out + 32 * i, enc);
}

// vartime_compress(hash_to_curve(r1, r2)) fused: two Elligator maps, the sum on the Jacobi
// quartic (pt_jacobi_sum), the encoding read off the sum: two inverse square roots instead
// of three, one batched inversion per warp.  The rare inputs the
// shortcut does not cover take the generic path (map both pairs to the curve, add, compress).
// The maps are out of line on purpose: with both (each carries an inlined inverse square
// root) and the generic fallback inlined, the hot path no longer fits the instruction cache
// once the CTAs of an SM have drifted apart (71 instead of 98 Melem/s at 2^22, and falling
// with the batch size).

// (no reference parameters: an fq_t& across a call boundary is a stack slot, i.e. local
// memory -- input comes as a pointer into the batch, output goes to shared-memory columns)
__device__ __noinline__ void elligator_st_to_smem(const uint8_t* __restrict__ r, size_t width, size_t i,
                                                  isqrt_smem_t sm, int slot) {
  fq_t s, t;
  pt_elligator_st(s, t, fq_input(r, width, i), sm);
  sm.put(slot, s);
  sm.put(slot + 1, t);
}
__device__ __noinline__ fq_r hash_generic_encoding(const uint8_t* __restrict__ r1,
                                                   const uint8_t* __restrict__ r2, size_t width,
                                                   size_t i, isqrt_smem_t sm) {
  fq_t s1, t1, s2, t2;
  pt_elligator_st(s1, t1, fq_input(r1, width, i), sm);
  pt_elligator_st(s2, t2, fq_input(r2, width, i), sm);
  return pt_compress_to_field(pt_add(pt_from_jacobi(s1, t1), pt_from_jacobi(s2, t2)), sm);
}

// One element per thread (two per thread before one inversion was measured: 99 against
// 103 Melem/s).  Values that have to survive an out-of-line call or the CTA-wide inversion
// are parked in SHARED memory, not left to the register allocator: the maps' (s, t) pairs
// in four extra columns behind the isqrt slots (passed by reference across the calls they
// lived in local memory, 77 local loads per thread), the sum (S : T : Z) in the isqrt
// slots themselves -- idle by then -- while the warp inverts.
constexpr int kHashSlots = ISQRT_SLOTS + 4;
static size_t hash_smem() { return (size_t)kHashSlots * 8 * kCodecBlock * sizeof(uint32_t); }

__global__ void __launch_bounds__(kCodecBlock, 4)
k_hash_encode(const uint8_t* __restrict__ r1, const uint8_t* __restrict__ r2, size_t width, size_t n,
              uint8_t* __restrict__ out) {
  extern __shared__ uint32_t smem[];
  isqrt_smem_t sm = isqrt_smem(smem);
  const size_t i = (size_t)blockIdx.x * kCodecBlock + threadIdx.x;
  const size_t ii = i < n ? i : 0;
  elligator_st_to_smem(r1, width, ii, sm, ISQRT_SLOTS);
  elligator_st_to_smem(r2, width, ii, sm, ISQRT_SLOTS + 2);
  {
    fq_t ns, nt, w;
    pt_jacobi_sum(ns, nt, w, sm.get(ISQRT_SLOTS), sm.get(ISQRT_SLOTS + 1), sm.get(ISQRT_SLOTS + 2),
                  sm.get(ISQRT_SLOTS + 3));
    sm.put(0, ns);
    sm.put(1, nt);
    sm.put(2, w);
  }
  const fq_t prod = fq_mul(fq_mul(sm.get(0), sm.get(2)), sm.get(1));
  const bool zero = fq_is_zero(prod);
  const fq_t inv = fq_warp_inverse(fq_select(zero, fq_t(fq_one()), prod));   // per warp: no barrier
  const fq_t I = fq_select(zero, fq_t(fq_zero()), inv);
  fq_r enc;
  const bool ok = jq_encoding_with_inverse(enc, sm.get(0), sm.get(1), sm.get(2), I);
  if (!ok) enc = hash_generic_encoding(r1, r2, width, ii, sm);
  if (i < n) fq_store(out + 32 * i, enc);
}

__global__ void __launch_bounds__(kCodecBlock)
k_fq_isqrt(const uint8_t* __restrict__ x, size_t n, uint8_t* __restrict__ out,
           uint8_t* __restrict__ wsq) {
  extern __shared__ uint32_t smem[];
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  isqrt_smem_t sm = isqrt_smem(smem);
  fq_t r;
  bool s = fq_isqrt(r, fq_load_wire(x + 32 * i), sm);
  fq_store_canon(out + 32 * i, r);
  wsq[i] = s ? 1 : 0;
}

// Fq::sqrt_ratio_zeta(num, den) for a general ratio, ark_curve/invsqrt.rs:75-166
__global__ void __launch_bounds__(kCodecBlock)
k_fq_sqrt_ratio(const uint8_t* __restrict__ num, const uint8_t* __restrict__ den, size_t n,
                uint8_t* __restrict__ out, uint8_t* __restrict__ wsq) {
  extern __shared__ uint32_t smem[];
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  isqrt_smem_t sm = isqrt_smem(smem);
  fq_t r;
  bool s = fq_sqrt_ratio_zeta(r, fq_load_wire(num + 32 * i), fq_load_wire(den + 32 * i), sm);
  fq_store_canon(out + 32 * i, r);
  wsq[i] = s ? 1 : 0;
}


void launch_decompress(const uint8_t* enc, size_t n, uint8_t* out, uint8_t* ok, cudaStream_t st,
                       int out_format) {
  if (out_format == D377_PT_AFFINE)
    k_decompress<true><<<grid_for(n, kCodecBlock), kCodecBlock, codec_smem(), st>>>(enc, n, out, ok);
  else
    k_decompress<false><<<grid_for(n, kCodecBlock), kCodecBlock, codec_smem(), st>>>(enc, n, out, ok);
}

void launch_compress(const uint8_t* in, size_t n, uint8_t* enc, cudaStream_t st, int in_format) {
  const unsigned g = grid_for(n, kCodecBlock);
  if (in_format == D377_PT_AFFINE)
    k_compress<D377_PT_AFFINE><<<g, kCodecBlock, codec_smem(), st>>>(in, n, enc);
  else if (in_format == D377_PT_XYZ)
    k_compress<D377_PT_XYZ><<<g, kCodecBlock, codec_smem(), st>>>(in, n, enc);
  else
    k_compress<D377_PT_ELEMENT><<<g, kCodecBlock, codec_smem(), st>>>(in, n, enc);
}

void launch_elligator(bool hash, bool encode, const uint8_t* r1, const uint8_t* r2, size_t width, size_t n,
                      uint8_t* out, cudaStream_t st) {
  dim3 g(grid_for(n, kCodecBlock));
  size_t sm = codec_smem();
  if (hash) {
    if (encode) {
      // 48 KB of dynamic shared memory + the static words: above the default limit, opt in
      // (per device, so on every launch; the call is a table lookup in the driver)
      cudaFuncSetAttribute(k_hash_encode, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)hash_smem());
      k_hash_encode<<<g, kCodecBlock, hash_smem(), st>>>(r1, r2, width, n, out);
    }
    else k_elligator<true, false><<<g, kCodecBlock, sm, st>>>(r1, r2, width, n, out);
  } else {
    if (encode) k_elligator_encode<<<g, kCodecBlock, sm, st>>>(r1, width, n, out);
    else k_elligator<false, false><<<g, kCodecBlock, sm, st>>>(r1, nullptr, width, n, out);
  }
}

// OnCurve::is_on_curve over a batch (ark_curve/on_curve.rs:17-38): curve equation, Segre
// embedding, Z != 0 and -- with check_order -- [2r]P = 0.
__global__ void __launch_bounds__(kCodecBlock)
k_on_curve(const uint8_t* __restrict__ el, size_t n, int check_order, uint8_t* __restrict__ ok) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const pt_t p = pt_load_wire(el + 128 * i);
  bool good = pt_on_curve(p);
  if (check_order) good = good && pt_order_divides_2r(p);
  ok[i] = good ? 1 : 0;
}

void launch_on_curve(const uint8_t* el, size_t n, int check_order, uint8_t* ok, cudaStream_t st) {
  k_on_curve<<<grid_for(n, kCodecBlock), kCodecBlock, 0, st>>>(el, n, check_order, ok);
}

D377_DBG_READER(codec_debug_counts)

void launch_fq_isqrt(const uint8_t* x, size_t n, uint8_t* out, uint8_t* wsq, cudaStream_t st) {
  k_fq_isqrt<<<grid_for(n, kCodecBlock), kCodecBlock, codec_smem(), st>>>(x, n, out, wsq);
}

void launch_fq_sqrt_ratio(const uint8_t* num, const uint8_t* den, size_t n, uint8_t* out,
                          uint8_t* wsq, cudaStream_t st) {
  k_fq_sqrt_ratio<<<grid_for(n, kCodecBlock), kCodecBlock, codec_smem(), st>>>(num, den, n, out, wsq);
}

}  // namespace d377
