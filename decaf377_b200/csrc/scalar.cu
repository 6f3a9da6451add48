// Scalar-multiplication kernels, one element per thread: variable-base &Element * &Fr,
// fixed-base GENERATOR * s and sum_j s_j * B_j over GPU-built window tables (normalize_batch
// lives with the MSM normalisation kernel in msm.cu).  Own translation unit so that the
// heavy kernels of the library compile in parallel.
#include "engine.h"
#include "point.cuh"

namespace d377 {

constexpr int kCodecBlock = 128;
static size_t codec_smem() { return ISQRT_SMEM_WORDS(kCodecBlock) * sizeof(uint32_t); }

// &Element * &Fr, ark_curve/ops/projective.rs:106-191
// 128 registers: four CTAs per SM, so that the 512 CTAs of configuration 1 (2^16 elements)
// are ONE wave on 148 SMs (at 130 registers they were 1.15 waves of three CTAs per SM).
template <int kFmt, bool kEncode>
__global__ void __launch_bounds__(kCodecBlock, 4)
k_scalar_mul(const uint8_t* __restrict__ pts, const uint8_t* __restrict__ scalars, size_t n,
             uint8_t* __restrict__ out, uint8_t* __restrict__ ok) {
  extern __shared__ uint32_t smem[];
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  isqrt_smem_t sm = isqrt_smem(smem);
  pt_t p;
  const bool good = pt_load_fmt<kFmt>(p, pts, i, sm);
  // only encodings can fail to decode; the host entry point fills `ok` for the other formats
  if (kFmt == D377_PT_ENCODING && ok) ok[i] = good ? 1 : 0;
  fq_raw_t k = fq_load_raw(scalars + 32 * i);
  pt_t r = pt_scalar_mul(p, k);
  D377_DBG_POINT(r);
  if (kEncode)
    fq_store(out + 32 * i, pt_compress_to_field(r, sm));
  else
    pt_store_canon(out + 128 * i, r);
}

// ---- fixed-base tables ------------------------------------------------------
// Table of a base B: T[w][j] = (j+1) * 2^(16 w) * B in cached affine form, w < 16, j < 2^15,
// followed by one extra entry 2^256 * B: the carry out of the top window of a scalar >= 2^255
// (never a canonical Fr, but the entry points accept any 256-bit string).  A set of k bases
// (d377_fixed_bases_create*) holds k such tables back to back, kFbStride records apart; the
// generator's table is the set {G}.
constexpr int kFbC = 16;
constexpr int kFbW = 16;
constexpr int kFbK = 1 << (kFbC - 1);
constexpr size_t kFbStride = (size_t)kFbW * kFbK + 1;

size_t fixed_bases_bytes_per_base() { return kFbStride * sizeof(niels_t); }

// Element::GENERATOR, the starting point of the generator's table
__global__ void k_fb_generator(pt_t* start) {
  pt_t p;
  p.x = fq_const(FQ_BX);
  p.y = fq_const(FQ_BY);
  p.z = fq_one();
  p.t = fq_const(FQ_BT);
  start[0] = p;
}

// The caller's bases in point_format 0..3 -> extended points, one thread per base.  An
// invalid encoding sets bit 0 of *flags (the base then reads as the identity).
template <int kFmt>
__global__ void __launch_bounds__(kCodecBlock)
k_fb_load(const uint8_t* __restrict__ pts, size_t k, pt_t* __restrict__ start, uint32_t* __restrict__ flags) {
  extern __shared__ uint32_t smem[];
  size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= k) return;
  pt_t p;
  if (!pt_load_fmt<kFmt>(p, pts, j, isqrt_smem(smem))) atomicOr(flags, 1u);
  D377_DBG_POINT(p);
  start[j] = p;
}

// 2^(16 w) * B_j for w <= kFbW, one thread per base: bases[j * (kFbW + 1) + w]
__global__ void k_fb_bases(const pt_t* __restrict__ start, size_t k, pt_t* __restrict__ bases) {
  size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= k) return;
  pt_t p = start[j];
  for (int w = 0; w <= kFbW; w++) {
    bases[j * (kFbW + 1) + w] = p;
    for (int c = 0; c < kFbC; c++) p = pt_dbl(p);
  }
}

// All k tables in one launch; the entries are normalised affine, so a table depends on its
// base only, not on the representative it was built from.
__global__ void k_fb_fill(const pt_t* __restrict__ bases, size_t k, niels_t* __restrict__ table) {
  size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= k * kFbStride) return;
  size_t j = idx / kFbStride, r = idx % kFbStride;   // r = kFbW * kFbK: the carry entry 1 * bases[kFbW]
  int w = (int)(r / kFbK);
  uint32_t m = (uint32_t)(r % kFbK) + 1;
  pt_t base = bases[j * (kFbW + 1) + w];
  pt_t acc = pt_identity();
#pragma unroll 1
  for (int i = kFbC - 1; i >= 0; i--) {
    acc = pt_dbl(acc);
    if ((m >> i) & 1u) acc = pt_add(acc, base);
  }
  fq_t zi = fq_inv(acc.z);
  table[idx] = niels_from_affine(fq_mul(acc.x, zi), fq_mul(acc.y, zi));
}

D377_DI niels_t niels_load(const niels_t* p) {
  const uint8_t* b = reinterpret_cast<const uint8_t*>(p);   // 96-byte records, 32-byte aligned
  niels_t n;
  n.ymx = fq_assume<1000>(fq_load(b));
  n.ypx = fq_assume<1000>(fq_load(b + 32));
  n.kt = fq_assume<1000>(fq_load(b + 64));
  return n;
}

// acc + s * B with signed 16-bit windows over the table of B.
D377_DI pt_t fixed_base_edwards(const niels_t* __restrict__ table, const fq_raw_t& k, pt_t acc) {
  uint32_t carry = 0;
#pragma unroll 1
  for (int w = 0; w < kFbW; w++) {
    uint32_t limb = k.l[w >> 1];
    uint32_t raw = ((w & 1) ? (limb >> 16) : (limb & 0xffffu)) + carry;
    carry = raw > (uint32_t)kFbK ? 1u : 0u;
    int32_t d = (int32_t)raw - (int32_t)(carry << kFbC);
    uint32_t mag = d < 0 ? (uint32_t)(-d) : (uint32_t)d;
    niels_t nl = niels_identity();
    if (mag) nl = niels_cneg(niels_load(table + (size_t)w * kFbK + (mag - 1)), d < 0);
    acc = pt_add_niels(acc, nl);
  }
  // a carry out of the top window only happens for scalars >= 2^255 (never canonical)
  if (carry) acc = pt_add_niels(acc, niels_load(table + (size_t)kFbW * kFbK));
  return acc;
}

// out[i] = sum_j s_ij * B_j over the k tables of a set, ONE accumulator through all of them:
// 16 k mixed additions per row.  The generator is the set {G} (k = 1).
template <bool kEncode>
__global__ void __launch_bounds__(kCodecBlock)
k_fixed_base(const niels_t* __restrict__ tables, size_t k, const uint8_t* __restrict__ scalars, size_t n,
             uint8_t* __restrict__ out) {
  extern __shared__ uint32_t smem[];
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  pt_t acc = pt_identity();
#pragma unroll 1
  for (size_t j = 0; j < k; j++)
    acc = fixed_base_edwards(tables + j * kFbStride, fq_load_raw(scalars + 32 * (i * k + j)), acc);
  D377_DBG_POINT(acc);
  if (kEncode) {
    isqrt_smem_t sm = isqrt_smem(smem);
    fq_store(out + 32 * i, pt_compress_to_field(acc, sm));
  } else {
    pt_store_canon(out + 128 * i, acc);
  }
}

// ---- vartime_compress(GENERATOR * s) on the Jacobi quartic ---------------------------------
// The decaf encoding s of a point IS the s-coordinate of a preimage under the 2-isogeny from
// the Jacobi quartic J: t^2 = s^4 - 2(2d - a) s^2 + 1 (that is what decompress inverts), and
// for a point of J the encoding can be read off (s, t) without a square root
// (jq_encoding_with_inverse, point.cuh).  So when only the encoding of s * G is wanted, the
// whole multiplication runs on J: G_J = (8, 65 / y_G) is the preimage of the basepoint
// (encoding 08 00 ... 00), the isogeny is a homomorphism, and
//   compress(s * G) = encoding of s * G_J
// with 12 mixed quartic additions (9 M + 2 S + 1 K each) over a second window table and
// ~20 multiplications for the encoding -- 152 Fq-ops instead of 16 * 7 + 315 = 427, and no
// inverse square root at all.  Table record (128 B, one cache line): s | t | s^2 | -s, so a
// negative digit only changes the load address of the first field.  The quartic's unified
// addition law has exceptional pairs (Z3 = 0); a thread that meets one, or whose result the
// encoding shortcut does not cover (S T Z = 0, e.g. the identity for s = 0), recomputes its
// element on the Edwards path, so the output is the reference's for EVERY scalar.
struct jq_rec_t {
  fq_r s, t, s2, ns;
};

// The quartic table has its own geometry: 12 signed 21-bit windows (12 * 21 = 252 bits
// cover every canonical scalar), 2^20 entries each: 1.6 GB, built once in ~0.1 s.  Twelve
// additions instead of sixteen; the entries are gathered from HBM (12 lines per element),
// which 16 resident warps per SM hide.  Scalars with a bit at or above 2^252 take the
// Edwards path.
constexpr int kJqC = 21;
constexpr int kJqW = 12;
constexpr int kJqK = 1 << (kJqC - 1);

D377_DI fq_r fq_load_canon(const void* p) { return fq_assume<1000>(fq_load(p)); }

__device__ __noinline__ fq_r fixed_base_generic_encoding(const niels_t* __restrict__ table,
                                                         const fq_raw_t& k, isqrt_smem_t sm) {
  return pt_compress_to_field(fixed_base_edwards(table, k, pt_identity()), sm);
}

// Every thread computes kPer elements before the CTA inverts once (Montgomery's trick per
// thread on top of fq_cta_inverse): the lone-warp inversion is a ~60 us bubble in a kernel
// whose per-element work is only ~150 multiplications, so it is amortised over kPer x 128
// elements -- 284 (one element, 16-bit windows) -> 398 (kPer = 4) -> 434 (8) -> 447 Melem/s
// (16) at 2^24.  Large kPer needs a large batch (a launch should still be several waves of
// CTAs), so the launcher picks it from n.  Finished (S, T, Z) and the running prefix
// products are parked in local memory (dynamically indexed, L1-resident).
template <int kFbPer>
__global__ void __launch_bounds__(kCodecBlock, 4)
k_fixed_base_jq(const jq_rec_t* __restrict__ jtable, const niels_t* __restrict__ etable,
                const uint8_t* __restrict__ scalars, size_t n, uint8_t* __restrict__ out) {
  extern __shared__ uint32_t smem[];
  __shared__ fq_t inv_sh[kCodecBlock / 32 + 1];
  fq_t pS[kFbPer], pT[kFbPer], pZ[kFbPer], pre[kFbPer];
  uint32_t badmask = 0;
  fq_t run = fq_one();
#pragma unroll 1
  for (int e = 0; e < kFbPer; e++) {
    const size_t i = ((size_t)blockIdx.x * kFbPer + e) * kCodecBlock + threadIdx.x;
    const fq_raw_t k = fq_load_raw(scalars + 32 * (i < n ? i : 0));
    jq_t acc = jq_identity();
    bool bad = (k.l[7] >> 28) != 0;                       // bits >= 2^252: not covered by 12 windows
    // signed digit of window w given the carry into it
    auto digit = [&](int w, uint32_t& carry) -> int32_t {
      const int bit = w * kJqC, limb = bit >> 5, off = bit & 31;
      uint64_t v = k.l[limb];
      if (limb + 1 < 8) v |= (uint64_t)k.l[limb + 1] << 32;
      uint32_t raw = ((uint32_t)(v >> off) & ((1u << kJqC) - 1u)) + carry;
      carry = raw > (uint32_t)kJqK ? 1u : 0u;
      return (int32_t)raw - (int32_t)(carry << kJqC);
    };
    auto record = [&](int w, int32_t d) -> const uint8_t* {
      uint32_t mag = d < 0 ? (uint32_t)(-d) : (uint32_t)d;
      return reinterpret_cast<const uint8_t*>(jtable + (size_t)w * kJqK + (mag ? mag - 1 : 0));
    };
    uint32_t carry = 0;
    int32_t d_next = digit(0, carry);
#pragma unroll 1
    for (int w = 0; w < kJqW; w++) {
      const int32_t d = d_next;
      const uint32_t mag = d < 0 ? (uint32_t)(-d) : (uint32_t)d;
      const uint8_t* rec = record(w, d);
      // the table entries are gathered from HBM: fetch the next window's line while this
      // window's addition runs (measured neutral: 16 resident warps already hide the gather)
      if (w + 1 < kJqW) {
        d_next = digit(w + 1, carry);
        asm volatile("prefetch.global.L1 [%0];" ::"l"(record(w + 1, d_next)));
      }
      // a zero digit adds the neutral element (0, 1)
      const fq_r s2 = fq_select(mag != 0, fq_load_canon(rec + (d < 0 ? 96 : 0)), fq_zero());
      const fq_r t2 = fq_select(mag != 0, fq_load_canon(rec + 32), fq_one());
      const fq_r s2sq = fq_select(mag != 0, fq_load_canon(rec + 64), fq_zero());
      acc = jq_madd(acc, s2, t2, s2sq);
      bad = bad || fq_is_zero(acc.Z);
    }
    bad = bad || carry != 0;
    const fq_t prod = fq_mul(fq_mul(acc.S, acc.Z), acc.T);
    bad = bad || fq_is_zero(prod);
    if (bad) badmask |= 1u << e;
    pS[e] = acc.S;
    pT[e] = acc.T;
    pZ[e] = acc.Z;
    pre[e] = run;                                         // product of the elements before e
    run = fq_mul(run, fq_select(bad, fq_t(fq_one()), prod));
  }
  fq_t inv = fq_cta_inverse<kCodecBlock / 32>(run, inv_sh);   // 1 / (product of this thread's elements)
#pragma unroll 1
  for (int e = kFbPer - 1; e >= 0; e--) {
    const size_t i = ((size_t)blockIdx.x * kFbPer + e) * kCodecBlock + threadIdx.x;
    const bool bad = (badmask >> e) & 1u;
    const fq_t S = pS[e], T = pT[e], Z = pZ[e];
    const fq_t I = fq_mul(inv, pre[e]);                   // 1 / (S T Z) of element e
    inv = fq_mul(inv, fq_select(bad, fq_t(fq_one()), fq_t(fq_mul(fq_mul(S, Z), T))));
    fq_r enc;
    const bool ok = jq_encoding_with_inverse(enc, S, T, Z, I);
    if (bad || !ok)
      enc = fixed_base_generic_encoding(etable, fq_load_raw(scalars + 32 * (i < n ? i : 0)), isqrt_smem(smem));
    if (i < n) fq_store(out + 32 * i, enc);
  }
}

// Quartic table: bases B_w = 2^(16 w) G_J (affine), then T[w][j] = (j + 1) B_w.
__global__ void k_jq_bases(fq_t* bases /* kJqW x (s, t) */) {
  // G_J = (8, (1 + 8^2) / y_G)
  jq_t p;
  p.S = fq_fold(fq_mul_small<8>(fq_one()));
  p.T = fq_mul(fq_fold(fq_mul_small<65>(fq_one())), fq_inv(fq_const(FQ_BY)));
  p.Z = fq_one();
  for (int w = 0; w < kJqW; w++) {
    fq_t iz = fq_inv(p.Z);
    bases[2 * w] = fq_mul(p.S, iz);
    bases[2 * w + 1] = fq_mul(p.T, fq_sqr(iz));
    for (int k = 0; k < kJqC; k++) p = jq_dbl(p);
  }
}

__global__ void k_jq_fill(const fq_t* __restrict__ bases, jq_rec_t* __restrict__ table) {
  size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (size_t)kJqW * kJqK) return;
  int w = (int)(idx / kJqK);
  uint32_t m = (uint32_t)(idx % kJqK) + 1;
  const fq_r bs = fq_reduce(bases[2 * w]), bt = fq_reduce(bases[2 * w + 1]);
  const fq_r bs2 = fq_reduce(fq_sqr(bs));
  jq_t acc = jq_identity();
#pragma unroll 1
  for (int i = kJqC - 1; i >= 0; i--) {
    acc = jq_dbl(acc);
    if ((m >> i) & 1u) acc = jq_madd(acc, bs, bt, bs2);
  }
  fq_t iz = fq_inv(acc.Z);
  fq_r s = fq_reduce(fq_mul(acc.S, iz));
  fq_r t = fq_reduce(fq_mul(acc.T, fq_sqr(iz)));
  uint8_t* rec = reinterpret_cast<uint8_t*>(table + idx);
  fq_store(rec, s);
  fq_store(rec + 32, t);
  fq_store(rec + 64, fq_reduce(fq_sqr(s)));
  fq_store(rec + 96, fq_reduce(fq_neg(s)));
}

// k_fb_bases + k_fb_fill for the k start points at work[0, k); work[k, k + k (kFbW + 1)) holds
// the window bases
static void fb_build(pt_t* work, size_t k, niels_t* table, cudaStream_t st) {
  k_fb_bases<<<grid_for(k, 32), 32, 0, st>>>(work, k, work + k);
  D377_LAUNCHED();
  k_fb_fill<<<grid_for(k * kFbStride, 128), 128, 0, st>>>(work + k, k, table);
  D377_LAUNCHED();
}

int ensure_fb_table() {
  Engine& e = engine();
  if (e.fb_table) return D377_OK;
  pt_t* work = nullptr;
  niels_t* table = nullptr;
  D377_CUDA(cudaMalloc(&work, sizeof(pt_t) * (kFbW + 2)));
  D377_CUDA(cudaMalloc(&table, sizeof(niels_t) * kFbStride));
  k_fb_generator<<<1, 1, 0, e.stream>>>(work);
  D377_LAUNCHED();
  fb_build(work, 1, table, e.stream);
  D377_CUDA(cudaGetLastError());
  D377_CUDA(cudaStreamSynchronize(e.stream));
  D377_CUDA(cudaFree(work));
  e.fb_table = table;
  return D377_OK;
}

// The tables of k caller-chosen bases (device memory, point_format 0..3) into `table`
// (k * fixed_bases_bytes_per_base() bytes).  Synchronises the engine stream.
int fixed_bases_fill(const uint8_t* points, int point_format, size_t k, void* table) {
  Engine& e = engine();
  uint32_t* dflags = (uint32_t*)(e.d_small + kSmallFlags);
  uint32_t* hflags = (uint32_t*)(e.h_small + kSmallFlags);
  pt_t* work = nullptr;
  D377_CUDA(cudaMalloc(&work, sizeof(pt_t) * k * (kFbW + 2)));
  cudaError_t ce = cudaMemsetAsync(dflags, 0, 4, e.stream);
  if (ce == cudaSuccess) {
    dim3 g(grid_for(k, kCodecBlock));
    switch (point_format) {
      case D377_PT_ELEMENT: k_fb_load<D377_PT_ELEMENT><<<g, kCodecBlock, 0, e.stream>>>(points, k, work, dflags); break;
      case D377_PT_ENCODING:
        k_fb_load<D377_PT_ENCODING><<<g, kCodecBlock, codec_smem(), e.stream>>>(points, k, work, dflags);
        break;
      case D377_PT_AFFINE: k_fb_load<D377_PT_AFFINE><<<g, kCodecBlock, 0, e.stream>>>(points, k, work, dflags); break;
      default: k_fb_load<D377_PT_XYZ><<<g, kCodecBlock, 0, e.stream>>>(points, k, work, dflags); break;
    }
    D377_LAUNCHED();
    fb_build(work, k, (niels_t*)table, e.stream);
    ce = cudaGetLastError();
  }
  if (ce == cudaSuccess) ce = cudaMemcpyAsync(hflags, dflags, 4, cudaMemcpyDeviceToHost, e.stream);
  cudaError_t se = cudaStreamSynchronize(e.stream);
  if (ce == cudaSuccess) ce = se;
  cudaFree(work);
  if (ce != cudaSuccess) return cuda_fail(ce, "fixed bases: table build", __FILE__, __LINE__);
  if (*hflags & 1u) {
    set_error("fixed bases: a base is not a valid encoding");
    return D377_ERR_INVALID_ENCODING;
  }
  return D377_OK;
}

// second table (1.6 GB): multiples of the basepoint's preimage on the Jacobi quartic
int ensure_fb_table_jq() {
  Engine& e = engine();
  if (e.fb_table_jq) return D377_OK;
  fq_t* bases = nullptr;
  jq_rec_t* table = nullptr;
  D377_CUDA(cudaMalloc(&bases, sizeof(fq_t) * 2 * kJqW));
  D377_CUDA(cudaMalloc(&table, sizeof(jq_rec_t) * (size_t)kJqW * kJqK));
  k_jq_bases<<<1, 1, 0, e.stream>>>(bases);
  D377_LAUNCHED();
  k_jq_fill<<<grid_for((size_t)kJqW * kJqK, 128), 128, 0, e.stream>>>(bases, table);
  D377_LAUNCHED();
  D377_CUDA(cudaGetLastError());
  D377_CUDA(cudaStreamSynchronize(e.stream));
  D377_CUDA(cudaFree(bases));
  e.fb_table_jq = table;
  return D377_OK;
}

void launch_scalar_mul(int point_format, bool encode, const uint8_t* points, const uint8_t* scalars,
                       size_t n, uint8_t* out, uint8_t* ok, cudaStream_t st) {
  // CTA size / residency at 2^16 elements (configuration 1: 512 CTAs of 128 threads are 0.86 of
  // one wave, 68 SMs hold four CTAs and 80 hold three).  Smaller CTAs, with or without a
  // shared-memory request that caps the CTAs per SM at an even 14 warps, do not pay
  // (profiles/r2_scalar_mul_cta_sweep.txt): 20.5 Melem/s with 128 threads, 20.3 with 96,
  // 20.3 / 20.2 with 64, 20.2 with 32 -- the kernel is bound by each thread's dependent chain,
  // not by the warps an SM holds.
  dim3 g(grid_for(n, kCodecBlock));
#define SM_LAUNCH(F, E) k_scalar_mul<F, E><<<g, kCodecBlock, codec_smem(), st>>>(points, scalars, n, out, ok)
  switch (point_format) {
    case D377_PT_ELEMENT: if (encode) SM_LAUNCH(D377_PT_ELEMENT, true); else SM_LAUNCH(D377_PT_ELEMENT, false); break;
    case D377_PT_ENCODING: if (encode) SM_LAUNCH(D377_PT_ENCODING, true); else SM_LAUNCH(D377_PT_ENCODING, false); break;
    default: if (encode) SM_LAUNCH(D377_PT_AFFINE, true); else SM_LAUNCH(D377_PT_AFFINE, false); break;
  }
#undef SM_LAUNCH
}

// table: a set of k tables (k = 1 for the generator); table_jq: the generator's quartic table
// (only with k = 1), or null
void launch_fixed_base(bool encode, const void* table, size_t k, const void* table_jq, const uint8_t* scalars,
                       size_t n, uint8_t* out, cudaStream_t st) {
  dim3 g(grid_for(n, kCodecBlock));
  const niels_t* tab = (const niels_t*)table;
  if (encode && table_jq) {
    const jq_rec_t* jt = (const jq_rec_t*)table_jq;
    // elements per thread: >= ~1000 CTAs per launch
    if (n >= ((size_t)1 << 22))
      k_fixed_base_jq<16><<<grid_for(n, kCodecBlock * 16), kCodecBlock, codec_smem(), st>>>(jt, tab, scalars, n, out);
    else if (n >= ((size_t)1 << 19))
      k_fixed_base_jq<8><<<grid_for(n, kCodecBlock * 8), kCodecBlock, codec_smem(), st>>>(jt, tab, scalars, n, out);
    else if (n >= ((size_t)1 << 16))
      k_fixed_base_jq<4><<<grid_for(n, kCodecBlock * 4), kCodecBlock, codec_smem(), st>>>(jt, tab, scalars, n, out);
    else
      k_fixed_base_jq<1><<<grid_for(n, kCodecBlock), kCodecBlock, codec_smem(), st>>>(jt, tab, scalars, n, out);
  }
  else if (encode) k_fixed_base<true><<<g, kCodecBlock, codec_smem(), st>>>(tab, k, scalars, n, out);
  else k_fixed_base<false><<<g, kCodecBlock, codec_smem(), st>>>(tab, k, scalars, n, out);
}

D377_DBG_READER(scalar_debug_counts)

}  // namespace d377
