// Pippenger multiscalar multiplication  Q = sum_i s_i * P_i  on one GPU.
//
// Replaces Element::vartime_multiscalar_mul (reference
// src/ark_curve/element/projective.rs:99-117, a serial fold of scalar-muls) and
// the ark-ec default `VariableBaseMSM::msm` the reference inherits at
// src/ark_curve/element.rs:37 (not in the reference tree).  The result is the
// same group element; tests compare its 32-byte encoding with the oracle's.
//
// Pipeline (no host synchronisation inside; the scalar side 2-4 runs on a second stream,
// window group by window group, under the accumulation of the group before):
//   1. k_msm_normalize / k_msm_points*   input points -> 128-byte bucket operands
//                      (affine (y-x, y+x, 2dxy, -2dxy), or cached projective for small n)
//   2. k_msm_count     scalars -> signed c-bit digits; per-(window,|digit|) bucket
//                      histogram with fire-and-forget atomics
//   3. scan            bucket counts -> offsets
//   4. k_msm_scatter   counting-sort scatter of (point index | sign) by bucket,
//                      window-major so the target stays in L2
//   5. k_msm_accumulate  every thread adds a fixed-length run of the sorted list
//                      (load balance independent of the scalar distribution);
//                      runs covering a whole bucket store the bucket sum, pieces
//                      of buckets that straddle threads are stitched by
//   6. k_msm_seg_reduce / k_msm_seg_reduce_warp (log-depth, so one huge bucket costs no
//                      serial walk)
//   7. k_msm_bucket_reduce_ap  per 16-bucket segment: running sums (A, P)
//   8. k_wsum_tree     weighted tree over the segments -> one sum per window;
//      k_msm_finish    Horner over the windows, optional fused compress.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <vector>

#include "engine.h"
#include "point.cuh"

namespace d377 {

D377_DI cached_t cached_load(const cached_t* p) {
  const uint8_t* b = reinterpret_cast<const uint8_t*>(p);
  cached_t c;
  c.ymx = fq_load(b);
  c.ypx = fq_load(b + 32);
  c.kt = fq_load(b + 64);
  c.z2 = fq_load(b + 96);
  return c;
}

D377_DI void cached_store(cached_t* p, const cached_t& c) {
  uint8_t* b = reinterpret_cast<uint8_t*>(p);
  fq_store(b, c.ymx);
  fq_store(b + 32, c.ypx);
  fq_store(b + 64, c.kt);
  fq_store(b + 96, c.z2);
}

// Affine bucket operand as the accumulation kernel reads it: 128 bytes, one cache line,
// (y-x | y+x | 2d*x*y | -2d*x*y), all canonical.  Adding -P reads the first pair in the
// opposite order and the fourth field instead of the third, so the sign of a bucket entry
// costs no instruction beyond the address computation; and a 128-byte aligned record is one
// DRAM fetch, where a 96-byte one straddles two 128-byte lines half of the time (ncu:
// 1.97x the algorithmic bytes with 96-byte records).
struct aff4_t {
  fq_r ymx, ypx, kt, nkt;
};

D377_DI void aff4_store(aff4_t* p, const niels_t& c) {
  uint8_t* b = reinterpret_cast<uint8_t*>(p);
  fq_store(b, c.ymx);
  fq_store(b + 32, c.ypx);
  fq_store(b + 64, c.kt);
  fq_store(b + 96, fq_reduce(fq_neg(c.kt)));
}

D377_DI pt_t ptv_load(const pt_t* p) { return pt_load(reinterpret_cast<const uint8_t*>(p)); }
D377_DI void ptv_store(pt_t* p, const pt_t& v) { pt_store(reinterpret_cast<uint8_t*>(p), v); }

// ---- 1. points -> cached ---------------------------------------------------
constexpr int kBlk = 128;

// Element / XYZ inputs -> cached projective records (small MSMs, no batch normalisation)
template <int kFmt>
__global__ void __launch_bounds__(kBlk)
k_msm_points(const uint8_t* __restrict__ pts, size_t n, cached_t* __restrict__ out) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  pt_t p;
  pt_load_fmt<kFmt>(p, pts, i, isqrt_smem_t{});
  cached_store(out + i, cached_from(p));
}

// Inputs that already have Z = 1 (AffinePoint, Encoding) -> canonical (y-x, y+x, 2d*x*y),
// 96 B each: the bucket additions then cost 7 multiplications instead of 8.
// Only an encoding can fail to load (it is stored as the identity).  With `ok` the kernel
// writes the decode status of every pair there; otherwise a failure sets bit 1 of `flags`
// (if given).
template <int kFmt>
__global__ void __launch_bounds__(kBlk)
k_msm_points_affine(const uint8_t* __restrict__ pts, size_t n, aff4_t* __restrict__ out,
                    uint32_t* __restrict__ flags, uint8_t* __restrict__ ok) {
  extern __shared__ uint32_t smem[];
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  pt_t p;
  const bool good = pt_load_fmt<kFmt>(p, pts, i, isqrt_smem(smem));
  if (kFmt == D377_PT_ENCODING && ok) ok[i] = good ? 1 : 0;
  else if (!good && flags) atomicOr(flags, 2u);
  aff4_store(out + i, niels_from_affine(p.x, p.y));
}

// Element inputs (projective) -> the same 96 B affine form, by Montgomery's trick with ONE
// field inversion per CTA: thread t multiplies the Z of its strided elements
// {t, t + T, ...} (prefix products parked in `scratch`, n x 32 B), the CTA combines the
// per-thread products (warp shuffles, then the eight warp totals through shared memory),
// warp 0 alone inverts the CTA product while the other warps wait at the barrier (the
// multiply pipe is free for other CTAs meanwhile), and every thread unwinds its own
// chain backwards.  Per element: 3 M (trick) + 2 M (x, y) + 2 M (2d x y); the inversion
// costs ~380 M per CTA.  (normalize_batch of the reference, ark_curve/element.rs:74-81,
// is the same computation; see k_normalize for the ABI entry point.)
constexpr int kNormBlk = 256;

// kStride: 128 for Elements (X||Y||Z||T), 96 for the T-less D377_PT_XYZ records; T is
// never read -- the affine form recomputes 2d*x*y from x and y.
// kXY: write the AffinePoint wire image x || y (64 B, canonical; Z = 0 gives (0, 0)) instead
// of the bucket operand -- the batch_normalize entry point (ark_curve/element.rs:74-81).
template <int kStride, bool kXY = false>
__global__ void __launch_bounds__(kNormBlk)
k_msm_normalize(const uint8_t* __restrict__ pts, size_t n, size_t T, uint8_t* __restrict__ scratch,
                void* __restrict__ out_v) {
  aff4_t* out = reinterpret_cast<aff4_t*>(out_v);
  uint8_t* out_xy = reinterpret_cast<uint8_t*>(out_v);
  __shared__ fq_t sh[kNormBlk / 32 + 1];
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  fq_t acc = fq_one();
  size_t cnt = 0;
#pragma unroll 1
  for (size_t i = t; i < n; i += T, cnt++) {
    fq_t z = fq_load_wire(pts + (size_t)kStride * i + 64);
    fq_store(scratch + 32 * i, acc);
    // Z = 0 never occurs for a curve point; keep the chain alive anyway
    acc = fq_mul(acc, fq_select(fq_is_zero(z), fq_t(fq_one()), z));
  }
  // inclusive prefix / suffix products of `acc` across the warp
  fq_t pre = acc, suf = acc;
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
    for (int v = 1; v < kNormBlk / 32; v++) tot = fq_mul(tot, sh[v]);
    fq_t inv = fq_inv_vartime(tot);
    if (lane == 0) sh[kNormBlk / 32] = inv;
  }
  __syncthreads();
  // 1 / (this warp's total) = inv(CTA total) * product of the other warps' totals
  fq_t inv = sh[kNormBlk / 32];
#pragma unroll 1
  for (int v = 0; v < kNormBlk / 32; v++)
    if (v != wid) inv = fq_mul(inv, sh[v]);
  // 1 / acc = that * (product of the lanes before) * (product of the lanes after)
  fq_t ex_pre = fq_shfl_up(pre, 1), ex_suf = fq_shfl_down(suf, 1);
  inv = fq_mul(inv, fq_select(lane == 0, fq_t(fq_one()), ex_pre));
  inv = fq_mul(inv, fq_select(lane == 31, fq_t(fq_one()), ex_suf));
#pragma unroll 1
  for (size_t k = cnt; k-- > 0;) {
    const size_t i = t + k * T;
    fq_t z = fq_load_wire(pts + (size_t)kStride * i + 64);
    const bool zz = fq_is_zero(z);
    fq_t zi = fq_mul(inv, fq_load_rw(scratch + 32 * i));
    inv = fq_mul(inv, fq_select(zz, fq_t(fq_one()), z));
    fq_t x = fq_mul(fq_load_wire(pts + (size_t)kStride * i), zi);
    fq_t y = fq_mul(fq_load_wire(pts + (size_t)kStride * i + 32), zi);
    if (kXY) {
      fq_store_canon(out_xy + 64 * i, fq_select(zz, fq_t(fq_zero()), x));
      fq_store_canon(out_xy + 64 * i + 32, fq_select(zz, fq_t(fq_zero()), y));
    } else {
      niels_t nl = niels_from_affine(x, y);
      aff4_store(out + i, zz ? niels_identity() : nl);
    }
  }
}

// Thread count T of a batch normalisation of n points: every thread walks per >= min_per
// strided points, per = n / 2^17 so that >= 2^17 threads stay busy, and T is capped at one
// wave: every CTA is resident from the start (3 per SM at <= 80 registers), so the kernel has
// no ragged last wave and the CTA-wide inversion bubble occurs once.
constexpr size_t kNormCtasPerSm = 3;

static size_t normalize_threads(size_t n, size_t min_per, int sm_count) {
  const size_t per = std::max(n >> 17, min_per);
  const size_t T = ((n + per - 1) / per + kNormBlk - 1) / kNormBlk * kNormBlk;
  return std::min(T, (size_t)sm_count * kNormCtasPerSm * kNormBlk);
}

// d377_batch_normalize: same kernel, one resident wave of CTAs (or fewer for small batches).
void launch_normalize(const uint8_t* el, size_t n, uint8_t* scratch, uint8_t* out, cudaStream_t st) {
  const size_t T = normalize_threads(n, 1, engine().sm_count);
  k_msm_normalize<128, true><<<(unsigned)(T / kNormBlk), kNormBlk, 0, st>>>(el, n, T, scratch, out);
}

static bool projective_format(int fmt) { return fmt == D377_PT_ELEMENT || fmt == D377_PT_XYZ; }

// n input points of any wire format -> bucket operands in `out` (n x 128 B) on `st`.  Affine
// records where `affine`: Element / XYZ by batch normalisation (normalize_threads(n, min_per),
// `scratch` n x 32 B), AffinePoint / Encoding one point per thread (an invalid encoding is
// reported in `ok` or `flags`, see k_msm_points_affine).  Otherwise cached projective records
// (Element / XYZ only).
static void launch_operands(const Engine& e, int fmt, bool affine, size_t min_per, const uint8_t* pts, size_t n,
                            uint8_t* scratch, uint8_t* out, uint32_t* flags, uint8_t* ok, cudaStream_t st) {
  aff4_t* aff = (aff4_t*)out;
  if (!affine) {
    auto k = fmt == D377_PT_ELEMENT ? k_msm_points<D377_PT_ELEMENT> : k_msm_points<D377_PT_XYZ>;
    k<<<grid_for(n, kBlk), kBlk, 0, st>>>(pts, n, (cached_t*)out);
  } else if (projective_format(fmt)) {
    const size_t T = normalize_threads(n, min_per, e.sm_count);
    auto k = fmt == D377_PT_ELEMENT ? k_msm_normalize<128> : k_msm_normalize<96>;
    k<<<(unsigned)(T / kNormBlk), kNormBlk, 0, st>>>(pts, n, T, scratch, aff);
  } else if (fmt == D377_PT_AFFINE) {
    k_msm_points_affine<D377_PT_AFFINE><<<grid_for(n, kBlk), kBlk, 0, st>>>(pts, n, aff, flags, ok);
  } else {
    k_msm_points_affine<D377_PT_ENCODING><<<grid_for(n, kBlk), kBlk, ISQRT_SMEM_WORDS(kBlk) * 4, st>>>(pts, n, aff,
                                                                                                        flags, ok);
  }
  D377_LAUNCHED();
}

// Windowed bases: the running points 2^(c j) * P_i, projective in `run` (n x 128 B), move on
// to the next window: c doublings in place, one base per thread.  With `first` (slab 0 of
// the table, the bucket operands (y-x, y+x, ...) of P_i) the running point is taken from
// there instead: (X' : Y' : Z) = (2x : 2y : 2), in extended coordinates (2X' : 2Y' : 4 : X'Y').
__global__ void __launch_bounds__(kBlk)
k_msm_bases_double(uint8_t* __restrict__ run, const aff4_t* __restrict__ first, size_t n, int c) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  pt_t p;
  if (first) {
    const uint8_t* rec = reinterpret_cast<const uint8_t*>(first + i);
    const fq_r ymx = fq_assume<1000>(fq_load(rec)), ypx = fq_assume<1000>(fq_load(rec + 32));
    const fq_t x2 = fq_sub(ypx, ymx), y2 = fq_add(ypx, ymx);
    p.x = fq_fold(fq_dbl(x2));
    p.y = fq_fold(fq_dbl(y2));
    p.z = fq_fold(fq_dbl(fq_dbl(fq_one())));
    p.t = fq_mul(x2, y2);
  } else {
    p = pt_load(run + 128 * i);
  }
#pragma unroll 1
  for (int k = 1; k < c; k++) p = pt_dbl<false>(p);
  p = pt_dbl<true>(p);
  D377_DBG_POINT(p);
  pt_store(run + 128 * i, p);
}

// ---- 2./4. signed-digit recoding ------------------------------------------
struct MsmGeom {
  int c;        // window width
  int W;        // number of windows = ceil(252 / c) (ceil(257 / c) for any 256-bit scalar)
  uint32_t K;   // buckets per window = 2^(c-1)
};

static MsmGeom geom(int c, int W) { return MsmGeom{c, W, 1u << (c - 1)}; }

// bits [w*c, w*c + c) of the 256-bit little-endian scalar; bits at or above 256 read 0 (when
// c divides 256 the top window of a 257-bit recoding starts at bit 256)
D377_DI uint32_t scalar_window(const fq_raw_t& s, int w, int c) {
  const int bit = w * c;
  if (bit >= 256) return 0u;
  const int limb = bit >> 5, off = bit & 31;
  uint64_t v = s.l[limb];
  if (limb + 1 < 8) v |= (uint64_t)s.l[limb + 1] << 32;
  return (uint32_t)(v >> off) & ((1u << c) - 1u);
}

// One signed-digit step: window w of s plus the carry in -> digit d in (-K, K] and the carry
// out.  A nonzero digit (when `take`) bumps the count of bucket id0 + |d| - 1 and returns that
// id with the sign in bit 31; otherwise the entry is 0xffffffff.
D377_DI uint32_t digit_entry(const fq_raw_t& s, int w, const MsmGeom& g, uint32_t& carry, uint32_t id0, bool take,
                             uint32_t* __restrict__ counts) {
  const uint32_t raw = scalar_window(s, w, g.c) + carry;
  carry = raw > g.K ? 1u : 0u;
  const int32_t d = (int32_t)raw - (int32_t)(carry << g.c);
  uint32_t e = 0xffffffffu;
  if (d != 0 && take) {
    const uint32_t id = id0 + (d < 0 ? (uint32_t)(-d) : (uint32_t)d) - 1;
    atomicAdd(&counts[id], 1u);   // result unused: compiles to RED.E.ADD
    e = id | (d < 0 ? 0x80000000u : 0u);
  }
  return e;
}

// Pass 1 (one thread per scalar): range check, signed-digit recoding, bucket histogram.
// For every (window, scalar) it records the entry's bucket id (sign in bit 31, 0xffffffff
// for a zero digit) in `dig` -- 4 bytes, the only per-entry state the sort keeps -- and
// bumps the bucket's count with a fire-and-forget reduction (RED: no return value, so no
// round trip to L2 stalls the warp).
// The kernel handles the windows [wa, wb) of one window group (`counts` and `dig` are the
// group's own arrays, bucket ids are local to the group); the signed-digit carry into
// window wa is recomputed from the windows below it.
// `wstride`: bucket ids of consecutive windows lie this far apart -- g.K (one bucket set per
// window) or 0 (windowed bases: every window of the group adds into ONE set of K buckets).
__global__ void __launch_bounds__(256, 8)   // <= 32 registers: fits beside 4 accumulation CTAs
k_msm_count(const uint8_t* __restrict__ scalars, size_t n, MsmGeom g, int wa, int wb, uint32_t wstride,
            uint32_t* __restrict__ counts, uint32_t* __restrict__ dig, uint32_t* __restrict__ flags) {
  // grid-stride: when the kernel shares the SMs with an accumulation it is launched with
  // one CTA per SM (the registers an accumulation CTA set leaves over) and walks the batch
#pragma unroll 1
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    fq_raw_t s = fq_load_raw(scalars + 32 * i);
    const bool ok = fr_raw_is_canonical(s);
    if (!ok) atomicOr(flags, 1u);  // contributes nothing; the call reports D377_ERR_SCALAR_RANGE
    uint32_t carry = 0;
    // W = ceil(252 / c): every window starts below bit 252 (scalar_window's bit-256 test folds away)
#pragma unroll 1
    for (int w = 0; w < wa; w++) {
      __builtin_assume(w * g.c < 252);
      carry = (scalar_window(s, w, g.c) + carry) > g.K ? 1u : 0u;
    }
    uint32_t* row = dig + i;
#pragma unroll 1
    for (int w = wa; w < wb; w++, row += n) {
      __builtin_assume(w * g.c < 252);
      *row = digit_entry(s, w, g, carry, (uint32_t)(w - wa) * wstride, ok, counts);
    }
  }
}

// Pass 2: counting-sort scatter.  `cursor` starts as a copy of the bucket offsets; every
// entry claims its slot with one atomicAdd on its bucket's cursor and stores (point index |
// sign) there.  The walk is window-major: one window at a time keeps the destination region
// (n * 4 B) and its cursors resident in L2, so the random 4-byte stores merge there instead
// of becoming DRAM read-modify-writes.  Every thread moves kScatterIlp entries so that as
// many (digit -> atomic -> store) chains are in flight.
// The stored index of entry i in row r is rec_base + r * rec_stride + i: the point index
// (both 0), or the record (w, i) = w * N + i of a windowed set (rec_base = wa * N,
// rec_stride = N).
constexpr int kScatterIlp = 4;

__global__ void __launch_bounds__(256, 8)
k_msm_scatter(const uint32_t* __restrict__ dig, size_t n, uint32_t rows, uint32_t* __restrict__ cursor,
              uint32_t* __restrict__ sorted, uint32_t rec_base, uint32_t rec_stride) {
  const size_t tiles_per_row = (n + 256 * kScatterIlp - 1) / (256 * kScatterIlp);
  const size_t total = tiles_per_row * rows;
  // row-major walk: all CTAs work on the same window at (almost) the same time
#pragma unroll 1
  for (size_t tile = blockIdx.x; tile < total; tile += gridDim.x) {
    const size_t r = tile / tiles_per_row;
    const size_t base = (tile - r * tiles_per_row) * (256 * kScatterIlp) + threadIdx.x;
    const uint32_t* row = dig + r * n;
    const uint32_t rec0 = rec_base + (uint32_t)r * rec_stride;
    uint32_t e[kScatterIlp], pos[kScatterIlp];
#pragma unroll
    for (int k = 0; k < kScatterIlp; k++) {
      const size_t i = base + (size_t)k * 256;
      e[k] = i < n ? row[i] : 0xffffffffu;
    }
#pragma unroll
    for (int k = 0; k < kScatterIlp; k++)
      pos[k] = e[k] != 0xffffffffu ? atomicAdd(&cursor[e[k] & 0x7fffffffu], 1u) : 0u;
#pragma unroll
    for (int k = 0; k < kScatterIlp; k++) {
      const size_t i = base + (size_t)k * 256;
      if (e[k] != 0xffffffffu) sorted[pos[k]] = (rec0 + (uint32_t)i) | (e[k] & 0x80000000u);
    }
  }
}

// ---- 3. exclusive scan (three small kernels) ---------------------------------
// 256-thread CTAs with few registers: they have to fit beside a resident accumulation
constexpr int kScanBlock = 256;
constexpr int kScanItems = 16;
constexpr int kScanTile = kScanBlock * kScanItems;

__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t v, uint32_t* total) {
  __shared__ uint32_t warp_sums[32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  uint32_t x = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) warp_sums[wid] = x;
  __syncthreads();
  if (wid == 0) {
    uint32_t s = lane < kScanBlock / 32 ? warp_sums[lane] : 0u;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      uint32_t y = __shfl_up_sync(0xffffffffu, s, o);
      if (lane >= o) s += y;
    }
    warp_sums[lane] = s;
  }
  __syncthreads();
  uint32_t before = wid ? warp_sums[wid - 1] : 0u;
  *total = warp_sums[31];
  __syncthreads();
  return before + x - v;
}

__global__ void __launch_bounds__(kScanBlock, 8)
k_scan_tiles(uint32_t* __restrict__ data, size_t n, uint32_t* __restrict__ tile_sums) {
  size_t base = (size_t)blockIdx.x * kScanTile + (size_t)threadIdx.x * kScanItems;
  uint32_t v[kScanItems], sum = 0;
#pragma unroll
  for (int k = 0; k < kScanItems; k++) {
    v[k] = base + k < n ? data[base + k] : 0u;
    sum += v[k];
  }
  uint32_t total;
  uint32_t ex = block_exclusive_scan(sum, &total);
#pragma unroll
  for (int k = 0; k < kScanItems; k++) {
    if (base + k < n) data[base + k] = ex;
    ex += v[k];
  }
  if (threadIdx.x == 0) tile_sums[blockIdx.x] = total;
}

__global__ void __launch_bounds__(kScanBlock)
k_scan_sums(uint32_t* __restrict__ tile_sums, size_t ntiles, uint32_t* __restrict__ grand_total) {
  uint32_t running = 0;
  for (size_t base = 0; base < ntiles; base += kScanBlock) {
    size_t i = base + threadIdx.x;
    uint32_t v = i < ntiles ? tile_sums[i] : 0u;
    uint32_t total;
    uint32_t ex = block_exclusive_scan(v, &total);
    if (i < ntiles) tile_sums[i] = running + ex;
    running += total;
  }
  if (threadIdx.x == 0) *grand_total = running;
}

__global__ void __launch_bounds__(kScanBlock, 8)
k_scan_apply(uint32_t* __restrict__ data, size_t n, const uint32_t* __restrict__ tile_sums,
             uint32_t* __restrict__ copy) {
  size_t base = (size_t)blockIdx.x * kScanTile + (size_t)threadIdx.x * kScanItems;
  uint32_t add = tile_sums[blockIdx.x];
#pragma unroll
  for (int k = 0; k < kScanItems; k++)
    if (base + k < n) {
      uint32_t v = data[base + k] + add;
      data[base + k] = v;
      copy[base + k] = v;   // the scatter's cursors
    }
}

// ---- 5. bucket accumulation -------------------------------------------------
// `offsets` has nb + 1 entries (offsets[nb] = total number of sorted entries).
// Thread t owns sorted[t*L, (t+1)*L).
// kAffine: `pts` holds canonical affine records (aff4_t) and an addition costs 7
// multiplications; otherwise cached projective records (cached_t, 8 multiplications).
// Both are 128 bytes.
// 112 registers: four CTAs (57 344 registers) leave room for one 256-thread, 32-register
// sort CTA of the second stream on every SM.
template <bool kAffine>
__global__ void __maxnreg__(112)
k_msm_accumulate(const void* __restrict__ pts_v, const uint32_t* __restrict__ sorted,
                 const uint32_t* __restrict__ offsets, uint32_t nb, int L,
                 pt_t* __restrict__ bsum, pt_t* __restrict__ part, int32_t* __restrict__ part_bucket,
                 int32_t bucket_base) {
  const uint8_t* pts = reinterpret_cast<const uint8_t*>(pts_v);
  constexpr uint32_t kRec = 128u;
  // (n W < 2^32 entries, so thread ids and positions fit 32 bits; the few scalars the loop
  // keeps live are chosen so that the kernel fits its 112 registers without a spill)
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t lo, hi;
  {
    const uint32_t total = offsets[nb];
    const uint64_t lo64 = (uint64_t)t * (uint64_t)L;
    if (lo64 >= total) return;
    lo = (uint32_t)lo64;
    hi = (uint32_t)min((uint64_t)total, lo64 + (uint64_t)L);
  }
  // bucket containing position lo: the last b with offsets[b] <= lo
  uint32_t b = 0;
  {
    uint32_t z = nb;  // invariant: offsets[b] <= lo < offsets[z]
    while (z - b > 1) {
      uint32_t m = b + ((z - b) >> 1);
      if (offsets[m] <= lo) b = m; else z = m;
    }
  }
  // does the current bucket begin inside this thread's range?
  bool starts_here = offsets[b] >= lo;
  uint32_t next = offsets[b + 1];
  pt_t acc = pt_identity();
  // Software pipeline on the sorted list and on the operands.  The index of entry pos + 2
  // is loaded while entry pos is added.  Affine records: the first two fields of the operand
  // of entry pos + 1 are loaded into REGISTERS before the addition of entry pos starts (16
  // more live registers), so the gather has a whole addition (~5 us) to arrive -- with a
  // prefetch into L1 and a load at the point of use, 9 % of the stall samples were the first
  // multiply of an addition waiting for its operand (profiles/; the kernel being pipe-bound,
  // removing them is worth < 1 % of its time).  Projective records (four fields) keep the
  // L1 prefetch: a register copy would cost a resident CTA.
  uint32_t e_next = sorted[lo];
  uint32_t e_next2 = lo + 1 < hi ? sorted[lo + 1] : 0u;
  fq_r n_ymx, n_ypx;
  if (kAffine) {
    const uint8_t* rec = pts + (size_t)(e_next & 0x7fffffffu) * kRec;
    const int o = (e_next >> 31) ? 32 : 0;
    n_ymx = fq_assume<1000>(fq_load_stream(rec + o));
    n_ypx = fq_assume<1000>(fq_load_stream(rec + (32 - o)));
  }
#pragma unroll 1
  for (uint32_t pos = lo; pos < hi; pos++) {
    const uint32_t e = e_next;
    e_next = e_next2;
    if (pos + 2 < hi) e_next2 = sorted[pos + 2];
    if (kAffine) {
      // written canonical by aff4_store; the sign of the entry picks the load addresses of
      // (y-x, y+x) and of (2dxy, -2dxy): no selects on limbs
      const fq_r ymx = n_ymx, ypx = n_ypx;
      // third field of the current record: its line came into L1 with the two fields above,
      // and it is not needed before the third multiplication
      const fq_r kt = fq_assume<1000>(
          fq_load_stream(pts + (size_t)(e & 0x7fffffffu) * kRec + 64 + ((e >> 31) ? 32 : 0)));
      if (pos + 1 < hi) {
        const uint8_t* rec = pts + (size_t)(e_next & 0x7fffffffu) * kRec;
        const int o = (e_next >> 31) ? 32 : 0;
        n_ymx = fq_assume<1000>(fq_load_stream(rec + o));
        n_ypx = fq_assume<1000>(fq_load_stream(rec + (32 - o)));
      }
      acc = pt_add_affine<true>(acc, ymx, ypx, kt);
    } else {
      if (pos + 1 < hi)
        asm volatile("prefetch.global.L1 [%0];" ::"l"(pts + (size_t)(e_next & 0x7fffffffu) * kRec));
      const bool neg = (e >> 31) != 0;
      const uint8_t* rec = pts + (size_t)(e & 0x7fffffffu) * kRec;
      const int o = neg ? 32 : 0;
      cached_t c;
      c.ymx = fq_load_stream(rec + o);
      c.ypx = fq_load_stream(rec + (32 - o));
      c.kt = fq_load_stream(rec + 64);
      c.z2 = fq_load_stream(rec + 96);
      acc = pt_add_cached<true, true>(acc, c, neg);
    }
    const bool bucket_ends = (pos + 1 == next);
    if (bucket_ends || pos + 1 == hi) {
      // The slot address is recomputed HERE from the special registers (opaque to the
      // optimiser): hoisted out of the loop it is a 64-bit value the compiler keeps alive
      // across every addition, and at 112 registers that meant a spill reloaded per entry.
      uint32_t tt = blockIdx.x * blockDim.x + threadIdx.x;
      asm volatile("" : "+r"(tt));
      if (starts_here && bucket_ends) {
        ptv_store(bsum + b, acc);
      } else if (!starts_here) {
        // piece of a bucket that began in an earlier thread's range
        ptv_store(part + 2 * (size_t)tt, acc);
        part_bucket[2 * (size_t)tt] = bucket_base + (int32_t)b;
      } else {
        // bucket begins here and continues into later ranges: this thread owns it
        ptv_store(part + 2 * (size_t)tt + 1, acc);
        part_bucket[2 * (size_t)tt + 1] = bucket_base + (int32_t)b;
      }
      acc = pt_identity();
      if (bucket_ends && pos + 1 < hi) {
        do {
          b++;
          next = offsets[b + 1];
        } while (next <= pos + 1);
        starts_here = true;   // every later bucket begins at or after pos + 1 > lo
      }
    }
  }
}

// ---- 6. stitch buckets that straddle accumulation ranges -------------------
// `keys`/`pts` is a list of slots, each either empty (key < 0) or a partial sum
// of bucket `key`; all pieces of one bucket are consecutive non-empty slots.
// Every thread folds kSegG slots.  A run of equal keys whose neighbours on both
// sides (looked up across the range boundary) belong to other buckets is the
// whole bucket and is stored; a run that may continue in an adjacent range is
// handed to the next level (two output slots per thread), so a bucket that
// holds N entries is finished after ~log_16(N/L) levels whatever the scalar
// distribution is.
constexpr int kSegG = 32;
constexpr int kSegLook = 64;
// stitch levels of at most this many slots use the warp-scan kernel below
constexpr size_t kStitchWarpSlots = (size_t)1 << 18;

__global__ void __launch_bounds__(kBlk)
k_msm_seg_reduce(const int32_t* __restrict__ keys, const pt_t* __restrict__ pts, size_t nslots,
                 pt_t* __restrict__ bsum, int32_t* __restrict__ out_keys, pt_t* __restrict__ out_pts,
                 size_t nthreads) {
  size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nthreads) return;
  const size_t lo = t * kSegG, hi = min(nslots, lo + (size_t)kSegG);
  int32_t cur = -1;
  int nruns = 0;
  bool out0_used = false;
  pt_t acc = pt_identity();
  // left neighbour: nearest non-empty slot before lo (bounded look-back)
  int32_t left = -2;  // -2: unknown (treat as possibly the same bucket)
  if (lo == 0) {
    left = -1;
  } else {
    for (size_t s = lo, k = 0; s-- > 0 && k < (size_t)kSegLook; k++) {
      int32_t v = keys[s];
      if (v >= 0) { left = v; break; }
      if (s == 0) left = -1;
    }
  }
  out_keys[2 * t] = -1;
  out_keys[2 * t + 1] = -1;
  for (size_t s = lo; s <= hi; s++) {
    int32_t k = s < hi ? keys[s] : -3;  // -3: end-of-range sentinel
    if (k == -1) continue;
    if (k != cur) {
      if (cur >= 0) {
        // close run `cur`
        nruns++;
        bool left_done = nruns > 1 || (left != -2 && left != cur);
        bool right_done;
        if (k != -3) {
          right_done = true;  // another bucket follows inside this range
        } else {
          // look ahead past hi
          int32_t right = -2;
          if (hi >= nslots) {
            right = -1;
          } else {
            for (size_t q = hi, c = 0; q < nslots && c < (size_t)kSegLook; q++, c++) {
              int32_t v = keys[q];
              if (v >= 0) { right = v; break; }
              if (q + 1 == nslots) right = -1;
            }
          }
          right_done = (right != -2 && right != cur);
        }
        if (left_done && right_done) {
          ptv_store(bsum + cur, acc);
        } else {
          size_t o = out0_used ? 2 * t + 1 : 2 * t;
          out0_used = true;
          ptv_store(out_pts + o, acc);
          out_keys[o] = cur;
        }
      }
      if (k == -3) break;
      cur = k;
      acc = ptv_load(pts + s);
    } else {
      acc = pt_add(acc, ptv_load(pts + s));
    }
  }
}

// Warp-parallel form of the same stitching step: one slot per lane, a segmented inclusive
// scan over the warp's 32 slots (empty slots are transparent), so a level costs at most five
// dependent point additions instead of up to 31 -- and usually one, because a scan step
// that no lane needs is skipped by a warp vote (the common layout is [tail piece][head
// piece] pairs: only the distance-1 step has work).  Segments that touch the warp's first
// or last slot and whose neighbour beyond it is, or may be, the same bucket go to the next
// level (two output slots per warp); everything else is a finished bucket.
D377_DI pt_t pt_shfl_up(const pt_t& p, int delta) {
  pt_t r;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    r.x.l[i] = __shfl_up_sync(0xffffffffu, p.x.l[i], delta);
    r.y.l[i] = __shfl_up_sync(0xffffffffu, p.y.l[i], delta);
    r.z.l[i] = __shfl_up_sync(0xffffffffu, p.z.l[i], delta);
    r.t.l[i] = __shfl_up_sync(0xffffffffu, p.t.l[i], delta);
  }
  return r;
}

// nearest non-empty key in keys[from], keys[from + step], ... (step = +1 / -1), looking at
// most kSegLook slots; -1: ran off the list (no neighbour), -2: not found (unknown)
D377_DI int32_t seg_neighbour(const int32_t* __restrict__ keys, size_t nslots, size_t from, bool forward,
                              bool exists, int lane) {
  if (!exists) return -1;
  int32_t res = -2;
#pragma unroll 1
  for (int round = 0; round < kSegLook / 32 && res == -2; round++) {
    const size_t d = (size_t)round * 32 + lane;
    bool in_range;
    size_t s;
    if (forward) { s = from + d; in_range = s < nslots; }
    else { in_range = d <= from; s = from - d; }
    int32_t k = in_range ? keys[s] : -1;
    uint32_t found = __ballot_sync(0xffffffffu, in_range && k >= 0);
    uint32_t off = __ballot_sync(0xffffffffu, !in_range);
    if (found) {
      res = __shfl_sync(0xffffffffu, k, __ffs(found) - 1);
    } else if (off) {
      res = -1;
    }
  }
  return res;
}

__global__ void __launch_bounds__(kBlk)
k_msm_seg_reduce_warp(const int32_t* __restrict__ keys, const pt_t* __restrict__ pts, size_t nslots,
                      pt_t* __restrict__ bsum, int32_t* __restrict__ out_keys, pt_t* __restrict__ out_pts,
                      size_t nwarps) {
  const size_t gw = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (gw >= nwarps) return;   // warp-uniform
  const size_t lo = gw * 32, s = lo + lane;
  const int32_t key = s < nslots ? keys[s] : -1;
  const bool ne = key >= 0;
  const uint32_t nemask = __ballot_sync(0xffffffffu, ne);
  if (lane < 2) out_keys[2 * gw + lane] = -1;
  if (nemask == 0) return;
  __syncwarp();
  pt_t p = ne ? ptv_load(pts + s) : pt_identity();
  // key of the last non-empty slot at or before this lane
  const uint32_t below = nemask & (0xffffffffu >> (31 - lane));
  int32_t fkey = __shfl_sync(0xffffffffu, key, below ? 31 - __clz(below) : 0);
  if (!below) fkey = -1;
  const int32_t pkey = __shfl_up_sync(0xffffffffu, fkey, 1);
  const bool head = ne && (lane == 0 || pkey != key);
  const uint32_t H = __ballot_sync(0xffffffffu, head);
#pragma unroll 1
  for (int d = 1; d < 32; d <<= 1) {
    // lane i takes the partial sum ending at lane i - d unless a segment starts in (i - d, i]
    const bool need = lane >= d && ((H >> (lane - d + 1)) & ((1u << d) - 1u)) == 0;
    if (!__any_sync(0xffffffffu, need)) continue;
    pt_t q = pt_shfl_up(p, d);
    pt_t sum = pt_add(p, q);
    p = pt_select(need, sum, p);
  }
  const bool is_end = fkey >= 0 && (lane == 31 || ((H >> (lane + 1)) & 1u));
  const uint32_t hs = H & (0xffffffffu >> (31 - lane));   // heads at or before this lane
  const bool first = (hs & (hs - 1)) == 0;                // this lane's segment is the warp's first
  const bool last = lane == 31;
  const int32_t left = seg_neighbour(keys, nslots, lo - 1, false, lo > 0, lane);
  const int32_t right = seg_neighbour(keys, nslots, lo + 32, true, lo + 32 < nslots, lane);
  if (is_end) {
    const bool left_done = !first || (left != -2 && left != fkey);
    const bool right_done = !last || (right != -2 && right != fkey);
    if (left_done && right_done) {
      ptv_store(bsum + fkey, p);
    } else {
      const size_t o = first ? 2 * gw : 2 * gw + 1;
      ptv_store(out_pts + o, p);
      out_keys[o] = fkey;
    }
  }
}

// ---- 7. bucket reduction ------------------------------------------------------
// For window w the sum  sum_j (j + 1) * B_j  over its K buckets, segment by segment and
// window group by window group (the groups finish at different times, see msm_once).
// Same running sums without the per-segment scalar multiplication.  Segment s of a window
// yields A_s = sum_j (j - base + 1) * B_j and P_s = Lseg * sum_j B_j (log2 Lseg doublings);
// the window sum  sum_s (A_s + s * P_s)  is then formed by k_wsum_tree, which carries the
// weight in the node itself: a node that covers 2^k segments holds
//   A = sum_s (A_s + (s - first) * P_s)   and   P = 2^k * sum_s P_s,
// so two neighbours combine as  A = A_l + A_r + P_r,  P = 2 (P_l + P_r)  at every level.
// Segments can therefore be short (many threads, short dependent chains) at no extra cost.
// The bucket offsets (consulted for "is this bucket empty") belong to the window groups.
struct GroupTab {
  int ng;
  int wlo[8], whi[8];
  const uint32_t* offs[8];
};

__global__ void __launch_bounds__(kBlk)
k_msm_bucket_reduce_ap(const pt_t* __restrict__ bsum, GroupTab gt, MsmGeom g, uint32_t Lseg, int log_lseg,
                       uint32_t S, pt_t* __restrict__ out_a, pt_t* __restrict__ out_p) {
  // out_a / out_p: [W][S]
  size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (size_t)g.W * S) return;
  const int w = (int)(idx / S);
  const uint32_t s = (uint32_t)(idx % S);
  int grp = 0;
  while (grp + 1 < gt.ng && !(w >= gt.wlo[grp] && w < gt.whi[grp])) grp++;
  const uint32_t* __restrict__ offsets = gt.offs[grp] + (size_t)(w - gt.wlo[grp]) * g.K;
  const pt_t* __restrict__ bw = bsum + (size_t)w * g.K;
  uint32_t base = s * Lseg;
  uint32_t end = min(base + Lseg, g.K);
  pt_t run = pt_identity(), acc = pt_identity();
  bool any = false;
#pragma unroll 1
  for (uint32_t j = end; j-- > base;) {
    if (offsets[j + 1] > offsets[j]) {
      run = pt_add(run, ptv_load(bw + j));
      any = true;
    }
    if (any) acc = pt_add(acc, run);
  }
  ptv_store(out_a + idx, acc);
  if (any) {
#pragma unroll 1
    for (int k = 0; k < log_lseg; k++) run = pt_dbl<true>(run);
  }
  ptv_store(out_p + idx, run);
}

// ---- 8. tree sums and the final combine ------------------------------------
// in: [groups][len] points; out[groups][ceil(len/G)]: every thread folds G consecutive
// points (used while the list is long enough to fill the machine that way)
// kWire: `in` is a caller's buffer (untrusted limbs, pt_load_wire)
template <bool kWire = false>
__global__ void __launch_bounds__(kBlk)
k_sum_groups(const pt_t* __restrict__ in, uint32_t groups, uint32_t len, uint32_t G,
             pt_t* __restrict__ out) {
  uint32_t olen = (len + G - 1) / G;
  size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (size_t)groups * olen) return;
  uint32_t gi = (uint32_t)(idx / olen), o = (uint32_t)(idx % olen);
  uint32_t lo = o * G, hi = min(lo + G, len);
  auto ld = [&](size_t k) {
    const uint8_t* q = reinterpret_cast<const uint8_t*>(in + k);
    return kWire ? pt_load_wire(q) : pt_load(q);
  };
  pt_t acc = ld((size_t)gi * len + lo);
#pragma unroll 1
  for (uint32_t j = lo + 1; j < hi; j++) acc = pt_add(acc, ld((size_t)gi * len + j));
  ptv_store(out + idx, acc);
}

D377_DI fq_t fq_shfl(const fq_t& v, int src) {
  fq_t r;
#pragma unroll
  for (int i = 0; i < 8; i++) r.l[i] = __shfl_sync(0xffffffffu, v.l[i], src);
  return r;
}

D377_DI pt_t pt_shfl_down(const pt_t& p, int delta) {
  pt_t r;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    r.x.l[i] = __shfl_down_sync(0xffffffffu, p.x.l[i], delta);
    r.y.l[i] = __shfl_down_sync(0xffffffffu, p.y.l[i], delta);
    r.z.l[i] = __shfl_down_sync(0xffffffffu, p.z.l[i], delta);
    r.t.l[i] = __shfl_down_sync(0xffffffffu, p.t.l[i], delta);
  }
  return r;
}

// Latency-oriented sum for short lists: one point per thread, log-depth shuffle tree
// (5 dependent additions per 32 points instead of 31), then the four warp results of a
// CTA through shared memory.  grid = (ceil(len / 128), groups); out[groups][gridDim.x].
__global__ void __launch_bounds__(kBlk)
k_sum_tree(const pt_t* __restrict__ in, uint32_t len, pt_t* __restrict__ out) {
  __shared__ pt_t warp_sum[kBlk / 32];
  const uint32_t gi = blockIdx.y;
  const uint32_t j = blockIdx.x * kBlk + threadIdx.x;
  pt_t p = j < len ? ptv_load(in + (size_t)gi * len + j) : pt_identity();
#pragma unroll 1
  for (int d = 16; d >= 1; d >>= 1) p = pt_add(p, pt_shfl_down(p, d));
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) warp_sum[wid] = p;
  __syncthreads();
  if (wid == 0) {
    p = lane < kBlk / 32 ? warp_sum[lane] : pt_identity();
#pragma unroll 1
    for (int d = kBlk / 64; d >= 1; d >>= 1) p = pt_add(p, pt_shfl_down(p, d));
    if (lane == 0) ptv_store(out + (size_t)gi * gridDim.x + blockIdx.x, p);
  }
}

// Four lanes share one point operation: every lane holds the whole point, computes one
// of the four independent products of each half of the formula and the results are
// exchanged by shuffles, so a doubling costs the latency of 1S + 1M instead of 4S + 4M
// and an addition 3M instead of 9M.  Used by the serial Horner tail only.
D377_DI pt_t pt_gather4(const fq_t& m, int base) {
  pt_t r;
  r.x = fq_shfl(m, base + 0);
  r.y = fq_shfl(m, base + 1);
  r.z = fq_shfl(m, base + 2);
  r.t = fq_shfl(m, base + 3);
  return r;
}

D377_DI pt_t pt_dbl4(const pt_t& p, int role, int base) {
  auto in = fq_select(role == 0, p.x, fq_select(role == 1, p.y, fq_select(role == 2, p.z, fq_add(p.x, p.y))));
  pt_t s = pt_gather4(fq_fold(fq_sqr(in)), base);  // s.x = X^2, s.y = Y^2, s.z = Z^2, s.t = (X+Y)^2
  // same sign arrangement as pt_dbl: F' = C - G, H' = A + B
  auto c = fq_dbl(s.z);
  auto hh = fq_add(s.x, s.y);
  auto e = fq_fold(fq_sub(s.t, hh));
  auto g = fq_fold(fq_sub(s.y, s.x));
  auto ff = fq_sub(c, g);
  // role 0: X3 = E F', 1: Y3 = G H', 2: Z3 = F' G, 3: T3 = E H'
  auto u = fq_select(role == 0 || role == 3, e, fq_select(role == 1, g, ff));
  auto v = fq_select(role == 0, ff, fq_select(role == 2, g, hh));
  return pt_gather4(fq_fold(fq_mul(u, v)), base);
}

D377_DI pt_t pt_add4(const pt_t& p, const pt_t& o, int role, int base) {
  // role 0: A = (Y1-X1)(Y2-X2), 1: B = (Y1+X1)(Y2+X2), 2: D = 2 Z1 Z2, 3: C = K T1 T2
  auto u = fq_select(role == 0, fq_sub(p.y, p.x), fq_select(role == 1, fq_add(p.y, p.x),
           fq_select(role == 2, fq_dbl(p.z), p.t)));
  auto v = fq_select(role == 0, fq_sub(o.y, o.x), fq_select(role == 1, fq_add(o.y, o.x),
           fq_select(role == 2, o.z, fq_fold(fq_mul_small<D377_K>(o.t)))));
  pt_t m = pt_gather4(fq_fold(fq_mul(u, v)), base);  // m.x = A, m.y = B, m.z = D, m.t = C
  auto e = fq_sub(m.y, m.x), f = fq_sub(m.z, m.t);
  auto g = fq_add(m.z, m.t), h = fq_add(m.y, m.x);
  auto uu = fq_select(role == 0 || role == 3, e, fq_select(role == 1, g, f));
  auto vv = fq_select(role == 0, f, fq_select(role == 2, g, h));
  return pt_gather4(fq_fold(fq_mul(uu, vv)), base);
}

// One CTA folds kWT consecutive nodes of one group (missing ones count as empty).  A lone
// warp is bound by its own issue rate (one IMAD.WIDE per 4 clocks), not by the pipe, so a
// node is computed by FOUR lanes (pt_add4 / pt_dbl4: 11 multiplications per lane and node
// instead of 35); levels exchange nodes through shared memory.
// grid = (ceil(len / kWT), groups); out[groups][gridDim.x].
constexpr int kWT = 128;

D377_DI void wnode_combine4(pt_t& a, pt_t& p, const pt_t& al, const pt_t& pl, const pt_t& ar,
                            const pt_t& pr, int role, int base) {
  a = pt_add4(pt_add4(al, ar, role, base), pr, role, base);
  p = pt_dbl4(pt_add4(pl, pr, role, base), role, base);
}

__global__ void __launch_bounds__(2 * kWT)
k_wsum_tree(const pt_t* __restrict__ a_in, const pt_t* __restrict__ p_in, uint32_t len,
            pt_t* __restrict__ a_out, pt_t* __restrict__ p_out) {
  __shared__ pt_t sa[2][kWT / 2], sp[2][kWT / 2];
  const uint32_t gi = blockIdx.y;
  const int lane = threadIdx.x & 31, role = lane & 3, base = lane & ~3;
  const uint32_t grp = threadIdx.x >> 2, wid = threadIdx.x >> 5;
  const size_t row = (size_t)gi * len;
  const uint32_t l = blockIdx.x * kWT + 2 * grp, r = l + 1;
  pt_t a, p;
  {
    pt_t al = l < len ? ptv_load(a_in + row + l) : pt_identity();
    pt_t pl = l < len ? ptv_load(p_in + row + l) : pt_identity();
    pt_t ar = r < len ? ptv_load(a_in + row + r) : pt_identity();
    pt_t pr = r < len ? ptv_load(p_in + row + r) : pt_identity();
    wnode_combine4(a, p, al, pl, ar, pr, role, base);
  }
  int cur = 0;
  if (role == 0) {
    sa[0][grp] = a;
    sp[0][grp] = p;
  }
  __syncthreads();
#pragma unroll 1
  for (uint32_t n = kWT / 4; n >= 1; n >>= 1) {
    // whole warps only: the four-lane operations shuffle with a full mask
    if (wid * 8 < n) {
      const uint32_t j = min(grp, n - 1);
      wnode_combine4(a, p, sa[cur][2 * j], sp[cur][2 * j], sa[cur][2 * j + 1], sp[cur][2 * j + 1], role, base);
      if (role == 0 && grp < n) {
        sa[cur ^ 1][grp] = a;
        sp[cur ^ 1][grp] = p;
      }
    }
    __syncthreads();
    cur ^= 1;
  }
  if (threadIdx.x == 0) {
    const size_t o = (size_t)gi * gridDim.x + blockIdx.x;
    ptv_store(a_out + o, a);
    ptv_store(p_out + o, p);
  }
}

// Horner over the W window sums of each of J segments: Q_j = sum_w 2^(c w) * S_jw, with
// wsums[j W + w] = S_jw; W = 0 means identity.  One four-lane group per segment (pt_dbl4 /
// pt_add4), eight per warp; a single result (J = 1) is one warp whose other groups compute the
// same thing.  Stores the canonical Element (out_el + 128 j) and / or the encoding
// (out_enc + 32 j); ok_out[j] (if wanted) is the AND of the segment's per-pair decode status
// ok_in[offs[j] .. offs[j + 1]) (all good when ok_in is null).
constexpr int kFinishBlk = 128;

__global__ void __launch_bounds__(kFinishBlk)
k_msm_finish(const pt_t* __restrict__ wsums, uint32_t J, int W, int c, const uint32_t* __restrict__ offs,
             const uint8_t* __restrict__ ok_in, uint8_t* __restrict__ out_el, uint8_t* __restrict__ out_enc,
             uint8_t* __restrict__ ok_out) {
  extern __shared__ uint32_t smem[];
  const int lane = threadIdx.x & 31, role = lane & 3, base = lane & ~3;
  const size_t seg = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 2;
  // groups past the end repeat the last segment: the four-lane operations shuffle with a
  // full mask, so whole warps stay in the loop; only real segments store
  const bool real = seg < J;
  const size_t j = real ? seg : (size_t)J - 1;
  const pt_t* __restrict__ ws = wsums + j * (size_t)W;
  pt_t r = pt_identity();
  if (W > 0) {
    r = ptv_load(ws + (W - 1));
#pragma unroll 1
    for (int w = W - 2; w >= 0; w--) {
#pragma unroll 1
      for (int k = 0; k < c; k++) r = pt_dbl4(r, role, base);
      r = pt_add4(r, ptv_load(ws + w), role, base);
    }
  }
  if (real && role == 0) {
    D377_DBG_POINT(r);
    if (out_el) pt_store_canon(out_el + 128 * seg, r);
  }
  if (out_enc) {
    isqrt_smem_t sm = isqrt_smem(smem);
    fq_t s = pt_compress_to_field(r, sm);
    if (real && role == 0) fq_store(out_enc + 32 * seg, s);
  }
  if (ok_out) {
    bool good = true;
    if (ok_in) {
#pragma unroll 4
      for (uint32_t i = offs[j] + role; i < offs[j + 1]; i += 4) good = good && ok_in[i] != 0;
    }
    const uint32_t bad = __ballot_sync(0xffffffffu, !good);
    if (real && role == 0) ok_out[seg] = ((bad >> base) & 0xfu) == 0 ? 1 : 0;
  }
}


// ---- many small MSMs in one call ------------------------------------------------------
// Segment j of `prods` (the products s_i * P_i, 128 B each, written by k_scalar_mul) is
// summed by one warp: lanes stride over the segment, then a shuffle tree.  `okp` (may be
// null) holds the decode status of encoding inputs; a segment with an invalid encoding
// reports ok = 0 (and still gets the sum of its valid pairs, the invalid ones count as the
// identity).  Empty segments give the identity (Element::default()).
__global__ void __launch_bounds__(kBlk)
k_seg_sum(const uint8_t* __restrict__ prods, const uint8_t* __restrict__ okp, const uint32_t* __restrict__ offs,
          size_t nseg, uint8_t* __restrict__ out_el, uint8_t* __restrict__ ok_out) {
  const size_t seg = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (seg >= nseg) return;   // warp-uniform
  const uint32_t lo = offs[seg], hi = offs[seg + 1];
  pt_t acc = pt_identity();
  bool good = true;
#pragma unroll 1
  for (uint32_t i = lo + lane; i < hi; i += 32) {
    acc = pt_add(acc, pt_load(prods + 128 * (size_t)i));
    if (okp) good = good && okp[i] != 0;
  }
#pragma unroll 1
  for (int d = 16; d >= 1; d >>= 1) acc = pt_add(acc, pt_shfl_down(acc, d));
  const bool all_good = __all_sync(0xffffffffu, good);
  if (lane == 0) {
    D377_DBG_POINT(acc);
    pt_store_canon(out_el + 128 * seg, acc);
    if (ok_out) ok_out[seg] = all_good ? 1 : 0;
  }
}

void launch_seg_sum(const uint8_t* prods, const uint8_t* okp, const uint32_t* offs, size_t nseg,
                    uint8_t* out_el, uint8_t* ok_out, cudaStream_t st) {
  k_seg_sum<<<grid_for(nseg * 32, kBlk), kBlk, 0, st>>>(prods, okp, offs, nseg, out_el, ok_out);
  D377_LAUNCHED();
}

// ---- many independent MSMs in one segmented Pippenger (d377_msm_segmented*) ---------------
// Segment j of a chunk owns the "virtual windows" j W .. j W + W - 1: its window w adds into
// the bucket set of virtual window j W + w, so sort, accumulation, stitch, bucket reduction
// and weighted tree run over a flat bucket space exactly as for one MSM with J W windows.
// Scalars are any 256-bit integers, so the recoding covers 257 bits: W = ceil(257 / c)
// leaves no carry out of the top window.

// One thread per pair of a chunk of J segments.  `offs` (J + 1 entries) are the chunk's
// segment bounds as absolute pair indices; pair i of the chunk is pair offs[0] + i.  The
// entry of window w goes to row w of `dig` (window-major, as k_msm_count) with the bucket id
// (seg W + w) K + |d| - 1 (sign in bit 31, 0xffffffff for a zero digit).  No range check:
// every 256-bit integer is a valid scalar here.
__global__ void __launch_bounds__(256, 8)
k_msm_count_seg(const uint8_t* __restrict__ scalars, size_t n, const uint32_t* __restrict__ offs, uint32_t J,
                MsmGeom g, uint32_t* __restrict__ counts, uint32_t* __restrict__ dig) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t p = offs[0] + (uint32_t)i;
  // the segment holding pair p: the last j < J with offs[j] <= p (empty segments before it
  // have offs[j] = offs[j + 1] <= p and are passed over)
  uint32_t lo = 0, hi = J;   // invariant: offs[lo] <= p < offs[hi]
  while (hi - lo > 1) {
    const uint32_t m = lo + ((hi - lo) >> 1);
    if (offs[m] <= p) lo = m; else hi = m;
  }
  const fq_raw_t s = fq_load_raw(scalars + 32 * i);
  uint32_t carry = 0;
  uint32_t id = lo * (uint32_t)g.W * g.K;
  uint32_t* row = dig + i;
#pragma unroll 1
  for (int w = 0; w < g.W; w++, row += n, id += g.K) *row = digit_entry(s, w, g, carry, id, true, counts);
}

D377_DBG_READER(msm_debug_counts)

// ---------------------------------------------------------------------------
// host orchestration
// ---------------------------------------------------------------------------
static MsmGeom choose_geom(Engine& e, size_t n) {
  int best_c = 4;
  double best = 1e300;
  for (int c = 4; c <= 22; c++) {
    if (e.msm_window_override && c != e.msm_window_override) continue;
    int W = (252 + c - 1) / c;
    double K = std::ldexp(1.0, c - 1);
    // accumulate: 8M per (point, window); reduce: 2 adds (9M) per bucket + the tree;
    // fixed per-window latency of the serial tails.
    double cost = (double)W * (double)n * 8.0 + (double)W * K * 32.0 + (double)W * 3000.0;
    if (cost < best) { best = cost; best_c = c; }
  }
  // From 2^20 pairs the choice is the measured one (tools/tune_msm.py sweeps on B200,
  // gpurun_out/s4n_tune.log): the model above is right up to 2^24 but prefers c = 21 a
  // factor two too early -- with 2^20 buckets per window the accumulation itself slows down
  // (a warp handles a bucket end in almost every iteration) and the bucket reduction takes
  // 3.5 ms.  c = 19, 20 never win (no or one window fewer, twice / four times the buckets).
  // Re-swept in round 2 with the tails hidden under the next MSM (tools/sweep_c_r2.sh,
  // profiles/r2_msm_window_sweep_pipelined.txt): same winners -- 2^20 2.59 / 2.46 / 2.47 ms for
  // c = 15 / 16 / 17, 2^21 4.31 / 4.16 / 4.19 for 16 / 17 / 18, 2^22 7.56 / 7.36 / 8.47 for
  // 17 / 18 / 19, 2^24 26.8 / 30.5 / 28.3 / 27.8 for 18 / 19 / 20 / 21.
  if (!e.msm_window_override && n >= ((size_t)1 << 20)) {
    if (n < ((size_t)3 << 19)) best_c = 16;        // 2^20:        16 (3.53 ms; 17: 3.54, 15: 3.60)
    else if (n < ((size_t)3 << 20)) best_c = 17;   // 2^21:        17 (5.34 ms; 16: 5.46, 18: 5.45)
    else if (n < ((size_t)3 << 24)) best_c = 18;   // 2^22 - 2^25: 18 (2^25: 55.7 ms; 21: 59.8)
    else best_c = 21;                              // 2^26:        21 (113.3 ms; 18: 114.4)
  }
  MsmGeom g;
  g.c = best_c;
  g.W = (252 + best_c - 1) / best_c;
  g.K = 1u << (best_c - 1);
  return g;
}

static size_t align_up(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }

// Streams and events of the pipeline, created on first use (the engine's device is current).
static int msm_state_init(Engine& e) {
  MsmState& ms = e.msm;
  if (ms.ready) return D377_OK;
  int least = 0, greatest = 0;
  D377_CUDA(cudaDeviceGetStreamPriorityRange(&least, &greatest));
  D377_CUDA(cudaStreamCreateWithPriority(&ms.sort_stream, cudaStreamNonBlocking, greatest));
  // The tail kernels are short and latency-bound; at the greatest priority their CTAs take
  // the first slots that the long accumulation CTAs of the next MSM vacate instead of
  // queueing behind them.
  D377_CUDA(cudaStreamCreateWithPriority(&ms.tail_stream, cudaStreamNonBlocking, greatest));
  // (Measured back to back, greatest against least priority: 2.73 / 3.04 ms at 2^20,
  // 7.9 / 8.2 ms at 2^22, 27.5 / 29.6 ms at 2^24 with the single-group sort prefetch.)
  // the points stream at the least priority: see pts_prefetch in msm_once
  D377_CUDA(cudaStreamCreateWithPriority(&ms.points_stream, cudaStreamNonBlocking, least));
  for (int k = 0; k < 2; k++) D377_CUDA(cudaEventCreateWithFlags(&ms.ev_points_done[k], cudaEventDisableTiming));
  D377_CUDA(cudaEventCreateWithFlags(&ms.ev_fork, cudaEventDisableTiming));
  D377_CUDA(cudaEventCreateWithFlags(&ms.ev_acc_done, cudaEventDisableTiming));
  D377_CUDA(cudaEventCreateWithFlags(&ms.ev_join, cudaEventDisableTiming));
  for (int k = 0; k < 2; k++) D377_CUDA(cudaEventCreateWithFlags(&ms.ev_tail_done[k], cudaEventDisableTiming));
  // per-group events carry timestamps: d377_msm_timeline reads them
  for (int k = 0; k < kMaxGroups; k++) {
    D377_CUDA(cudaEventCreate(&ms.ev_sorted[k]));
    D377_CUDA(cudaEventCreate(&ms.ev_acc0[k]));
    D377_CUDA(cudaEventCreate(&ms.ev_acc[k]));
  }
  D377_CUDA(cudaEventCreate(&ms.ev_sort0));
  D377_CUDA(cudaEventCreate(&ms.ev_sort1));
  for (int k = 0; k <= kMsmStages; k++) D377_CUDA(cudaEventCreate(&ms.ev_stage[k]));
  ms.ready = true;
  return D377_OK;
}

// The stream on which MSM results become complete.  Whoever asks is about to enqueue work
// there, so the engine stream has to be ordered behind it at the next join.
cudaStream_t result_stream(Engine& e) {
  if (!e.msm_tail_overlap_override || msm_state_init(e) != D377_OK) return e.stream;
  e.msm.tail_pending = true;
  return e.msm.tail_stream;
}

int msm_join(Engine& e) {
  MsmState& ms = e.msm;
  if (!ms.ready || !ms.tail_pending) return D377_OK;
  D377_CUDA(cudaEventRecord(ms.ev_join, ms.tail_stream));
  D377_CUDA(cudaStreamWaitEvent(e.stream, ms.ev_join, 0));
  ms.tail_pending = false;
  return D377_OK;
}

// One result: Horner over W window sums (W = 0: the identity) on one warp.
static int finish(cudaStream_t st, const pt_t* wsums, int W, int c, uint8_t* out_element, uint8_t* out_encoding) {
  k_msm_finish<<<1, 32, ISQRT_SMEM_WORDS(32) * sizeof(uint32_t), st>>>(wsums, 1, W, c, nullptr, nullptr, out_element,
                                                                       out_encoding, nullptr);
  D377_LAUNCHED();
  D377_CUDA(cudaGetLastError());
  return D377_OK;
}

// reduce [groups][len] -> [groups][1] in place inside two ping-pong buffers
static int tree_sum(cudaStream_t st, pt_t*& cur, pt_t*& other, uint32_t groups, uint32_t len) {
  while (len > 1) {
    uint32_t olen;
    if ((size_t)groups * len >= ((size_t)1 << 18)) {
      const uint32_t G = 32;
      olen = (len + G - 1) / G;
      size_t total = (size_t)groups * olen;
      k_sum_groups<false><<<grid_for(total, kBlk), kBlk, 0, st>>>(cur, groups, len, G, other);
    } else {
      olen = (len + kBlk - 1) / kBlk;
      k_sum_tree<<<dim3(olen, groups), kBlk, 0, st>>>(cur, len, other);
    }
    D377_LAUNCHED();
    D377_CUDA(cudaGetLastError());
    std::swap(cur, other);
    len = olen;
  }
  return D377_OK;
}

// Sum<Element> (element/projective.rs:131-140) on stream `st` (the engine stream or the
// result stream; each has its own scratch).
int element_sum_on(Engine& e, cudaStream_t st, const uint8_t* elements, size_t n, uint8_t* out_element,
                   uint8_t* out_encoding) {
  if (n == 0) return finish(st, nullptr, 0, 0, out_element, out_encoding);
  if (n > 0xffffffffull) { set_error("element_sum: n too large"); return D377_ERR_INVALID_ARG; }
  DevBuf& ws = e.sum_ws[st == e.stream ? 0 : 1];
  size_t half = align_up(((n + 31) / 32) * sizeof(pt_t));
  int rc = ensure(ws, 2 * half);
  if (rc) return rc;
  pt_t* a = (pt_t*)ws.p;
  pt_t* b = (pt_t*)((uint8_t*)ws.p + half);
  // first level reads the caller's buffer
  const uint32_t G = 32;
  uint32_t len = (uint32_t)n;
  uint32_t olen = (len + G - 1) / G;
  k_sum_groups<true><<<grid_for(olen, kBlk), kBlk, 0, st>>>((const pt_t*)elements, 1, len, G, a);
  D377_LAUNCHED();
  D377_CUDA(cudaGetLastError());
  rc = tree_sum(st, a, b, 1, olen);
  if (rc) return rc;
  return finish(st, a, 1, 0, out_element, out_encoding);
}

// Prepared bases (D377_PT_BASES): any input format -> the affine bucket operands, once.
// Projective inputs are always batch-normalised here, whatever the batch size.
int msm_bases_prepare(const uint8_t* points, int point_format, size_t n, uint8_t* records) {
  Engine& e = engine();
  if (n == 0) return D377_OK;
  uint32_t* dflags = (uint32_t*)(e.d_small + kSmallFlags);
  uint32_t* hflags = (uint32_t*)(e.h_small + kSmallFlags);
  D377_CUDA(cudaMemsetAsync(dflags, 0, 4, e.stream));
  if (projective_format(point_format)) {
    int rc = ensure(e.scratch, n * 32);
    if (rc) return rc;
  }
  launch_operands(e, point_format, true, 1, points, n, (uint8_t*)e.scratch.p, records, dflags, nullptr, e.stream);
  D377_CUDA(cudaGetLastError());
  D377_CUDA(cudaMemcpyAsync(hflags, dflags, 4, cudaMemcpyDeviceToHost, e.stream));
  D377_CUDA(cudaStreamSynchronize(e.stream));
  return msm_check_flags(*hflags);
}

// Windowed bases: slab j of `table` (n records at table + j * n * 128) gets the bucket
// operands of 2^(c j) * P_i.  Slab 0 (P_i itself) has been written by msm_bases_prepare; the
// running points are kept projective in a scratch of n x 128 B and every slab is one
// k_msm_bases_double (c doublings) plus one batch normalisation (k_msm_normalize<128>).
int msm_bases_fill_windows(uint8_t* table, size_t n, int c, int W) {
  Engine& e = engine();
  if (n == 0 || W <= 1) return D377_OK;
  int rc = ensure(e.scratch, n * 32);
  if (rc) return rc;
  uint8_t* run = nullptr;
  D377_CUDA(cudaMalloc(&run, n * 128));
  const size_t T = normalize_threads(n, 1, e.sm_count);
  cudaError_t ce = cudaSuccess;
  for (int j = 1; j < W && ce == cudaSuccess; j++) {
    k_msm_bases_double<<<grid_for(n, kBlk), kBlk, 0, e.stream>>>(run, j == 1 ? (const aff4_t*)table : nullptr, n, c);
    D377_LAUNCHED();
    k_msm_normalize<128><<<(unsigned)(T / kNormBlk), kNormBlk, 0, e.stream>>>(
        run, n, T, (uint8_t*)e.scratch.p, table + (size_t)j * n * 128);
    D377_LAUNCHED();
    ce = cudaGetLastError();
  }
  if (ce == cudaSuccess) ce = cudaStreamSynchronize(e.stream);
  else cudaStreamSynchronize(e.stream);
  cudaFree(run);
  if (ce != cudaSuccess) return cuda_fail(ce, "windowed bases", __FILE__, __LINE__);
  return D377_OK;
}

// Window width of a windowed set created with c = 0.  Cost model as in choose_geom, with one
// set of K buckets per MSM and no Horner tail: n W mixed additions (7 M) + the reduction of K
// buckets (two additions each, ~32 M with the tree).  From 2^20 bases the choice is the
// measured one (tools/msm_windowed_bench.py --c 16,18,20,21,22 on B200,
// profiles/r3_msm_windowed_bench.json): c = 21 (W = 12) wins there -- back to back 2.01 /
// 6.26 / 23.6 ms at 2^20 / 2^22 / 2^24 against 2.03 / 6.57 / 26.7 for c = 18 and 2.58 / 7.69 /
// 27.2 for c = 22 -- where the model would still take 18 at 2^20.  Below 2^20 the model
// decides (11 at 2^10, 15 at 2^16); at 2^16 the sweep measured c = 16 a little faster (blocking
// 0.70 against 0.72 ms, back to back 0.47 against 0.55 ms), a point not swept densely enough yet
// to change the model for.
int msm_windowed_c(size_t n) {
  if (n >= ((size_t)1 << 20)) return 21;
  int best_c = 4;
  double best = 1e300;
  for (int c = 4; c <= 22; c++) {
    const int W = (252 + c - 1) / c;
    const double K = std::ldexp(1.0, c - 1);
    const double cost = (double)W * (double)n * 7.0 + K * 32.0;
    if (cost < best) { best = cost; best_c = c; }
  }
  return best_c;
}

// Window groups of an MSM over W windows: wlo[k] .. whi[k] are the windows of the k-th group
// processed, taken from the top down.  Group sizes in processing order, weights 2, 3, 4, ...:
// the first sort has only the point conversion to hide under, every later one the
// accumulation of the group before it.
static void group_windows(int W, int ngroups, int* wlo, int* whi) {
  int wsum = 0, acc = 0, cut[kMaxGroups + 1];
  // three groups: 2 : 5 : 7 (measured: the first sort then ends with the normalisation
  // and every later one just before the accumulation that waits for it)
  auto weight = [&](int k) { return ngroups == 3 ? (k == 0 ? 2 : k == 1 ? 5 : 7) : k + 2; };
  for (int k = 0; k < ngroups; k++) wsum += weight(k);
  cut[0] = 0;
  for (int k = 0; k < ngroups; k++) {
    acc += weight(k);
    cut[k + 1] = std::max(cut[k] + 1, (int)((long long)acc * W / wsum));
  }
  cut[ngroups] = W;
  for (int k = ngroups - 1; k > 0; k--) cut[k] = std::min(cut[k], cut[k + 1] - 1);
  for (int k = 0; k < ngroups; k++) {
    whi[k] = W - cut[k];
    wlo[k] = W - cut[k + 1];
  }
}

// ---- one Pippenger pass (sort, accumulation, tail), shared by msm_once and the segmented MSM ----
struct PassPlan {
  int L;              // sorted entries per accumulation thread
  int log_lseg;       // buckets per bucket-reduction thread: Lseg = 2^log_lseg
  uint32_t Lseg, S;   // S = ceil(K / Lseg) segments per bucket set
};

// The run lengths of a pass whose sort holds at most `max_entries` entries.
static PassPlan pass_plan(MsmGeom g, size_t max_entries) {
  PassPlan pl;
  // Run length per accumulate thread.  Every run boundary splits a bucket into pieces
  // that k_msm_seg_reduce has to stitch (one extra addition each), so runs are as long
  // as the thread count allows: >= ~2 full waves of 128-thread CTAs on 148 SMs.
  pl.L = max_entries >= ((size_t)1 << 27) ? 128 : max_entries >= ((size_t)1 << 25) ? 64 : 32;
  // Buckets per bucket-reduce thread.  With the weighted tree (k_wsum_tree) a segment
  // costs no scalar multiplication, so segments can be short: many threads, short
  // dependent chains.
  // With the tails hidden under the next MSM's head, their pipe work matters
  // more than their latency: longer segments (fewer doublings and tree nodes) win once a
  // window has many buckets -- measured back to back: 2^22 7.64 / 7.49 / 7.42 ms and 2^24
  // 27.08 / 26.97 / 27.00 ms with 16 / 32 / 64, 2^20 (c = 16) 2.43 / 2.48 / 2.64 ms.
  pl.log_lseg = g.c >= 18 ? 6 : g.c == 17 ? 5 : 4;
  pl.Lseg = 1u << pl.log_lseg;   // power of two: P_s = Lseg * R_s by doublings
  pl.S = (g.K + pl.Lseg - 1) / pl.Lseg;
  return pl;
}

// Bucket additions against affine records cost 7 M instead of 8: free when the input
// already has Z = 1; Element inputs are normalised first when the batch is large enough
// for the one-inversion-per-CTA trick to pay (7 M + one inversion per CTA against W
// multiplications saved).
// d377_msm_set_normalize: -1 never, 1 always (at least 4 points per thread), 0 from 2^20 pairs
static bool affine_operands(const Engine& e, int fmt, size_t n) {
  const int want = e.msm_normalize_override;
  return !projective_format(fmt) || want > 0 || (want == 0 && (n >> 17) >= 8);
}
static size_t normalize_min_per(const Engine& e) { return e.msm_normalize_override > 0 ? 4 : 1; }

// Cuts a workspace into 256-byte aligned arrays.  With base = 0 it only sizes them: a driver
// lays its workspace out once to learn the bytes to ensure() and once over the buffer.
struct Carver {
  uintptr_t base;
  size_t off = 0;
  template <class T = uint8_t>
  T* take(size_t bytes) {
    T* p = reinterpret_cast<T*>(base + off);
    off += align_up(bytes);
    return p;
  }
};

struct PassWs {
  uint32_t *dig, *sorted;   // digit entries and sorted list, window-major
  uint32_t *counts[kMaxGroups], *cursor[kMaxGroups], *tiles[kMaxGroups];   // per window group
  pt_t* bsum;               // bucket sums
  pt_t* part;               // two piece slots per accumulation thread, and their keys
  int32_t* pb;
  int32_t* kbuf[2];         // second and third stitch level (the levels ping-pong between them)
  pt_t* pbuf[2];
  pt_t *a, *p, *a2, *p2;    // segment nodes of the bucket reduction and of the weighted tree
};

static size_t scan_tiles(size_t nb) { return (nb + 1 + kScanTile - 1) / kScanTile; }

// A pass over `entries` sorted entries, `ngroups` window groups of gnb[k] buckets, `nthreads`
// accumulation threads and `rows` bucket sets of g.K buckets, each reduced in S segments.
static PassWs carve_pass(Carver& cv, size_t entries, int ngroups, const size_t* gnb, size_t nthreads, size_t rows,
                         MsmGeom g, uint32_t S) {
  PassWs w;
  w.dig = cv.take<uint32_t>(entries * 4);
  w.sorted = cv.take<uint32_t>(entries * 4);
  for (int k = 0; k < ngroups; k++) {
    w.counts[k] = cv.take<uint32_t>((gnb[k] + 1) * 4);
    w.cursor[k] = cv.take<uint32_t>((gnb[k] + 1) * 4);
    w.tiles[k] = cv.take<uint32_t>(scan_tiles(gnb[k]) * 4 + 4);
  }
  w.bsum = cv.take<pt_t>(rows * g.K * sizeof(pt_t));
  w.part = cv.take<pt_t>(2 * nthreads * sizeof(pt_t));
  w.pb = cv.take<int32_t>(2 * nthreads * 4);
  const size_t nthreads2 = (2 * nthreads + kSegG - 1) / kSegG;
  const size_t nthreads3 = (2 * nthreads2 + kSegG - 1) / kSegG;
  w.pbuf[0] = cv.take<pt_t>(2 * nthreads2 * sizeof(pt_t));
  w.kbuf[0] = cv.take<int32_t>(2 * nthreads2 * 4);
  w.pbuf[1] = cv.take<pt_t>(2 * nthreads3 * sizeof(pt_t));
  w.kbuf[1] = cv.take<int32_t>(2 * nthreads3 * 4);
  const size_t seg_n = rows * S, seg_n2 = rows * ((S + kWT - 1) / kWT);
  w.a = cv.take<pt_t>(seg_n * sizeof(pt_t));
  w.p = cv.take<pt_t>(seg_n * sizeof(pt_t));
  w.a2 = cv.take<pt_t>(seg_n2 * sizeof(pt_t));
  w.p2 = cv.take<pt_t>(seg_n2 * sizeof(pt_t));
  return w;
}

static unsigned grid_cap(size_t want, unsigned cap) { return (unsigned)(cap ? std::min<size_t>(want, cap) : want); }

// The counting sort after a count kernel has filled `counts` (nb + 1 words) and the rows x n
// entries of `dig`: scan of the counts into bucket offsets (copied into `cursor`), then the
// scatter into `sorted`.  `cap` (0: none) bounds the scatter's grid; n = 0 (a chunk of empty
// segments) only computes the offsets.
static void launch_sort(cudaStream_t s, uint32_t* counts, uint32_t* cursor, uint32_t* tiles, size_t nb,
                        const uint32_t* dig, size_t n, uint32_t rows, uint32_t* sorted, uint32_t rec_base,
                        uint32_t rec_stride, unsigned cap) {
  const size_t ntiles = scan_tiles(nb);
  k_scan_tiles<<<(unsigned)ntiles, kScanBlock, 0, s>>>(counts, nb + 1, tiles);
  D377_LAUNCHED();
  k_scan_sums<<<1, kScanBlock, 0, s>>>(tiles, ntiles, tiles + ntiles);
  D377_LAUNCHED();
  k_scan_apply<<<(unsigned)ntiles, kScanBlock, 0, s>>>(counts, nb + 1, tiles, cursor);
  D377_LAUNCHED();
  if (n == 0) return;
  k_msm_scatter<<<grid_cap((size_t)grid_for(n, 256 * kScatterIlp) * rows, cap), 256, 0, s>>>(
      dig, n, rows, cursor, sorted, rec_base, rec_stride);
  D377_LAUNCHED();
}

// Bucket accumulation of `nthreads` runs of L sorted entries; the nb buckets start at bucket b0
// of `bsum`.
static void launch_accumulate(cudaStream_t s, bool affine, const void* ops, const uint32_t* sorted,
                              const uint32_t* offsets, size_t nb, int L, size_t nthreads, pt_t* bsum, size_t b0,
                              pt_t* part, int32_t* pb) {
  auto k = affine ? k_msm_accumulate<true> : k_msm_accumulate<false>;
  k<<<grid_for(nthreads, kBlk), kBlk, 0, s>>>(ops, sorted, offsets, (uint32_t)nb, L, bsum + b0, part, pb, (int32_t)b0);
  D377_LAUNCHED();
}

// The tail of a pass on `s`: reduction of the `rows` bucket sets (their offsets in `gt`) to
// *sums, one point per row.  `marks` (may be null): two events recorded after the stitch and
// after the bucket reduction.
static int launch_tail(cudaStream_t s, const PassWs& w, size_t nthreads, const GroupTab& gt, MsmGeom g, size_t rows,
                       const PassPlan& pl, const cudaEvent_t* marks, pt_t** sums) {
  // Stitch the bucket pieces the accumulation left in 2 * nthreads slots (none: nothing to
  // stitch) into `bsum`; the slot lists of the later levels rotate through (kbuf, pbuf)[0]
  // and [1].  Work-efficient serial fold while a level is large, warp scan (log depth) below.
  const int32_t* kin = w.pb;
  const pt_t* pin = w.part;
  for (size_t nslots = 2 * nthreads, lvl = 0; nslots; lvl++) {
    const size_t nt = (nslots + kSegG - 1) / kSegG;
    int32_t* kout = w.kbuf[lvl & 1];
    pt_t* pout = w.pbuf[lvl & 1];
    if (nslots <= kStitchWarpSlots)
      k_msm_seg_reduce_warp<<<grid_for(nt * 32, kBlk), kBlk, 0, s>>>(kin, pin, nslots, w.bsum, kout, pout, nt);
    else
      k_msm_seg_reduce<<<grid_for(nt, kBlk), kBlk, 0, s>>>(kin, pin, nslots, w.bsum, kout, pout, nt);
    D377_LAUNCHED();
    nslots = nt == 1 ? 0 : 2 * nt;
    kin = kout;
    pin = pout;
  }
  if (marks) D377_CUDA(cudaEventRecord(marks[0], s));
  k_msm_bucket_reduce_ap<<<grid_for(rows * pl.S, kBlk), kBlk, 0, s>>>(w.bsum, gt, geom(g.c, (int)rows), pl.Lseg,
                                                                       pl.log_lseg, pl.S, w.a, w.p);
  D377_LAUNCHED();
  D377_CUDA(cudaGetLastError());
  if (marks) D377_CUDA(cudaEventRecord(marks[1], s));
  // Weighted tree over the rows of S segment nodes (a, p), ping-ponging with (a2, p2).  The
  // row is gridDim.y, so a launch covers at most 65 535 rows; more rows are launched in slices.
  constexpr size_t kMaxRows = 65535;
  pt_t *a = w.a, *p = w.p, *a2 = w.a2, *p2 = w.p2;
  for (uint32_t len = pl.S; len > 1;) {
    const uint32_t olen = (len + kWT - 1) / kWT;
    for (size_t r0 = 0; r0 < rows; r0 += kMaxRows) {
      const unsigned nr = (unsigned)std::min(kMaxRows, rows - r0);
      k_wsum_tree<<<dim3(olen, nr), 2 * kWT, 0, s>>>(a + r0 * len, p + r0 * len, len, a2 + r0 * olen, p2 + r0 * olen);
      D377_LAUNCHED();
    }
    std::swap(a, a2);
    std::swap(p, p2);
    len = olen;
  }
  *sums = a;
  return D377_OK;
}

// One Pippenger.  Head (point conversion, sort, bucket accumulation) on the engine and sort
// streams; tail (stitch, bucket reduction, weighted tree, Horner, compress) on the tail
// stream, over one of two tail-side workspace sets: the head of the next MSM starts right
// behind this MSM's last accumulation and the ~1 ms of latency-bound tail kernels run under
// it.  The result is complete on result_stream(e).
// `scalars_ready`: nullptr = the scalars are ordered on the engine stream like everything
// else (the sort stream forks from it); otherwise the scalars depend on nothing but that
// event (or on nothing at all if *scalars_ready is null), and the scalar side of this MSM
// is NOT ordered behind the engine stream: it starts as soon as its workspace set is free,
// i.e. under the bucket accumulation of the previous MSM.
//
// `bases` (D377_PT_BASES only): the layout of the set `points` points into.  A windowed set
// fixes c and W, and every window group then owns ONE set of K buckets: window w of the group
// adds the record w * N + i (= 2^(c w) P_i, N = the set's stride) into bucket |d| - 1, the
// groups' bucket sets are reduced like windows, and the tail sums the group results without
// any doubling.
static int msm_once(const uint8_t* scalars, const uint8_t* points, int point_format, bool sc_mont, size_t n,
                    uint8_t* out_element, uint8_t* out_encoding, uint32_t* flags /* device, OR-ed */,
                    const cudaEvent_t* scalars_ready = nullptr, const cudaEvent_t* points_ready = nullptr,
                    const BasesLayout* bases = nullptr) {
  Engine& e = engine();
  int rc = msm_state_init(e);
  if (rc) return rc;
  MsmState& ms = e.msm;
  const bool windowed = point_format == D377_PT_BASES && bases && bases->c > 0;
  const MsmGeom g = windowed ? geom(bases->c, bases->W) : choose_geom(e, n);
  const size_t max_entries = n * (size_t)g.W;
  if (max_entries >= 0xfffffff0ull) { set_error("msm chunk too large"); return D377_ERR_INVALID_ARG; }
  const PassPlan pl = pass_plan(g, max_entries);

  // Window groups: group k+1 is sorted (sort stream) while group k is accumulated (engine
  // stream).  Small MSMs run as one group: the extra launches would cost more than the
  // overlap hides.
  int ngroups = 1;
  if (g.W >= 6) {
    // measured on B200 (tools/tune_msm.py)
    if (max_entries >= ((size_t)3 << 26)) ngroups = std::min(3, g.W / 3);
    else if (max_entries >= ((size_t)1 << 24)) ngroups = 2;
  }
  // When this MSM's sort can run under the accumulation of the MSM before it (its scalars
  // are ready and that accumulation is still in flight), there is nothing left for window
  // groups to hide: one group, a third of the launches (2^24 back to back: 28.14 -> 27.76 ms).
  const bool may_prefetch = scalars_ready != nullptr && e.msm_tail_overlap_override;
  if (may_prefetch && ms.tail_used[0] && cudaEventQuery(ms.ev_acc_done) == cudaErrorNotReady) ngroups = 1;
  cudaGetLastError();
  if (e.msm_groups_override > 0) ngroups = std::min(std::min(e.msm_groups_override, kMaxGroups), g.W);
  int wlo[kMaxGroups], whi[kMaxGroups];
  group_windows(g.W, ngroups, wlo, whi);
  // sort kernels beside a resident accumulation: one 256-thread CTA per SM
  const unsigned sort_cap = ngroups > 1 || may_prefetch ? (unsigned)e.sm_count : 0u;
  // Buckets of group k: one set per window, or one merged set (windowed bases).  g_bucket[k]
  // is the group's first bucket in `bsum`; `rows` are the bucket sets the bucket reduction
  // sees (a merged set is reduced like one window).
  size_t g_nthreads[kMaxGroups], g_tbase[kMaxGroups + 1];
  size_t g_nb[kMaxGroups], g_bucket[kMaxGroups];
  g_tbase[0] = 0;
  for (int k = 0; k < ngroups; k++) {
    size_t ent_k = (size_t)(whi[k] - wlo[k]) * n;
    g_nthreads[k] = (ent_k + pl.L - 1) / pl.L;
    g_tbase[k + 1] = g_tbase[k] + g_nthreads[k];
    g_nb[k] = windowed ? (size_t)g.K : (size_t)(whi[k] - wlo[k]) * g.K;
    g_bucket[k] = windowed ? (size_t)k * g.K : (size_t)wlo[k] * g.K;
  }
  const size_t nthreads = g_tbase[ngroups];
  const size_t rows = windowed ? (size_t)ngroups : (size_t)g.W;

  const bool prepared = point_format == D377_PT_BASES;   // `points` already holds the bucket operands
  const bool affine = affine_operands(e, point_format, n);

  // ---- workspaces -----------------------------------------------------------------
  // Two complete sets (bucket operands, digits, sorted lists, offsets, bucket sums, piece
  // slots): the conversion of the points and the sort of the NEXT MSM run under this MSM's
  // bucket accumulation, and the tail of this MSM under the next MSM's accumulation.
  // The other set is only needed while the previous MSM is still in flight: a caller that
  // waits for every result (d377_msm_dev, d377_msm) keeps using set 0 and pays for one.
  int set = 0;
  if (e.msm_tail_overlap_override && ms.tail_used[ms.cur_set] &&
      cudaEventQuery(ms.ev_tail_done[ms.cur_set]) == cudaErrorNotReady)
    set = ms.cur_set ^ 1;
  cudaGetLastError();
  ms.cur_set = set;
  uint8_t *ops = nullptr, *norm = nullptr, *sc = nullptr;
  PassWs w;
  auto layout = [&](uintptr_t base) {
    Carver cv{base};
    ops = cv.take(prepared ? 0 : n * sizeof(cached_t));
    norm = cv.take(affine && projective_format(point_format) ? n * 32 : 0);
    sc = cv.take(sc_mont ? n * 32 : 0);
    w = carve_pass(cv, max_entries, ngroups, g_nb, nthreads, rows, g, pl.S);
    return cv.off;
  };
  rc = ensure(ms.tail_ws[set], layout(0));
  if (rc) return rc;
  layout((uintptr_t)ms.tail_ws[set].p);
  const void* ops_in = prepared ? (const void*)points : ops;
  cudaStream_t st = e.stream, ss = ms.sort_stream;
  // point conversion / normalisation: on the engine stream, or -- when the inputs are known to
  // be ready -- on a stream of its own, so that it runs under the previous MSM's accumulation
  // (its CTA-wide inversion bubble and its two passes over the points are then hidden; the
  // engine stream holds nothing but bucket accumulations)
  // Measured back to back (ms per MSM at 2^20 / 2^21 / 2^22 / 2^24): on the engine stream
  // 2.44 / 4.16 / 7.44 / 27.03, on its own stream at the least priority 2.57 / 4.09 / 7.36 /
  // 26.81, at the greatest 2.75 / 4.19 / 7.43 / 27.01 -- the conversion is multiply-pipe work
  // like the accumulation it runs under, so only its bubbles are hidden: ~1 % from 2^21 pairs
  // on one GPU.  In the 8-GPU strong-scaling loop (2^21 pairs per GPU, an all-gather per
  // step) it costs 4 % instead (4.28 -> 4.45 ms), so it is used from 2^22 pairs.
  const bool pts_prefetch = may_prefetch && !prepared && n >= ((size_t)1 << 22);
  cudaStream_t ps = pts_prefetch ? ms.points_stream : st;
  cudaStream_t ts = e.msm_tail_overlap_override ? ms.tail_stream : e.stream;

  ms.last_geom.c = g.c;
  ms.last_geom.W = g.W;
  ms.last_n = n;
  ms.last_affine = affine;
  ms.last_windowed = windowed;
  ms.last_groups = ngroups;
  ms.stage_valid = true;
  auto stage_mark = [&](int i, cudaStream_t s) { return cudaEventRecord(ms.ev_stage[i], s); };
  D377_CUDA(stage_mark(0, st));
  // The scalar side needs its inputs and its workspace set (the tail that last used the set
  // has to be done).  By default the inputs are ordered on the engine stream, so the sort
  // stream forks from it -- behind the previous MSM's accumulation.  With `scalars_ready`
  // the only dependency is that event.
  const bool prefetch = may_prefetch;
  if (prefetch) {
    if (*scalars_ready) D377_CUDA(cudaStreamWaitEvent(ss, *scalars_ready, 0));
  } else {
    D377_CUDA(cudaEventRecord(ms.ev_fork, st));
    D377_CUDA(cudaStreamWaitEvent(ss, ms.ev_fork, 0));
  }
  // (the points of a host-buffer MSM arrive after its scalars: the sort above only waits for
  // the scalars, the point conversion for the whole chunk)
  if (pts_prefetch) {
    const cudaEvent_t* pr = points_ready ? points_ready : scalars_ready;
    if (*pr) D377_CUDA(cudaStreamWaitEvent(ps, *pr, 0));
  }
  if (ms.tail_used[set]) {
    D377_CUDA(cudaStreamWaitEvent(ss, ms.ev_tail_done[set], 0));
    D377_CUDA(cudaStreamWaitEvent(st, ms.ev_tail_done[set], 0));
    if (pts_prefetch) D377_CUDA(cudaStreamWaitEvent(ps, ms.ev_tail_done[set], 0));
  }
  D377_CUDA(cudaEventRecord(ms.ev_sort0, ss));
  // scalars as the reference holds them in memory (Montgomery limbs): converted on the sort
  // stream into the workspace set before the digits are cut
  if (sc_mont) {
    launch_fr_from_mont(scalars, n, sc, ss);
    scalars = sc;
  }

  // ---- scalar side, all groups, on the sort stream (2, 3, 4) ----
  for (int k = 0; k < ngroups; k++) {
    const int wa = wlo[k], wb = whi[k];
    D377_CUDA(cudaMemsetAsync(w.counts[k], 0, (g_nb[k] + 1) * 4, ss));
    k_msm_count<<<grid_cap(grid_for(n, 256), sort_cap), 256, 0, ss>>>(scalars, n, g, wa, wb, windowed ? 0u : g.K,
                                                                      w.counts[k], w.dig + (size_t)wa * n, flags);
    D377_LAUNCHED();
    launch_sort(ss, w.counts[k], w.cursor[k], w.tiles[k], g_nb[k], w.dig + (size_t)wa * n, n, (uint32_t)(wb - wa),
                w.sorted + (size_t)wa * n, windowed ? (uint32_t)((size_t)wa * bases->n) : 0u,
                windowed ? (uint32_t)bases->n : 0u, sort_cap);
    D377_CUDA(cudaEventRecord(ms.ev_sorted[k], ss));
  }
  D377_CUDA(cudaEventRecord(ms.ev_sort1, ss));

  // ---- point side on the engine stream ----
  D377_CUDA(cudaMemsetAsync(w.pb, 0xff, 2 * nthreads * 4, st));
  // 1
  if (!prepared) {
    launch_operands(e, point_format, affine, normalize_min_per(e), points, n, norm, ops, flags, nullptr, ps);
    if (pts_prefetch) {
      D377_CUDA(cudaEventRecord(ms.ev_points_done[set], ps));
      D377_CUDA(cudaStreamWaitEvent(st, ms.ev_points_done[set], 0));
    }
  }
  for (int i = 1; i <= 4; i++) D377_CUDA(stage_mark(i, st));
  // 5: bucket accumulation, group by group as the sorted lists arrive.
  // 128 threads, ~106 registers, 4 CTAs/SM: measured flat from 4 to 7 CTAs/SM (the
  // fmaheavy pipe, not latency, is the limiter), slower at 8 (spills).
  for (int k = 0; k < ngroups; k++) {
    D377_CUDA(cudaStreamWaitEvent(st, ms.ev_sorted[k], 0));
    D377_CUDA(cudaEventRecord(ms.ev_acc0[k], st));
    launch_accumulate(st, affine, ops_in, w.sorted + (size_t)wlo[k] * n, w.counts[k], g_nb[k], pl.L, g_nthreads[k],
                      w.bsum, g_bucket[k], w.part + 2 * g_tbase[k], w.pb + 2 * g_tbase[k]);
    D377_CUDA(cudaEventRecord(ms.ev_acc[k], st));
  }
  D377_CUDA(stage_mark(5, st));
  // ---- tail: everything below runs on the tail stream ----
  D377_CUDA(cudaEventRecord(ms.ev_acc_done, st));
  if (ts != st) D377_CUDA(cudaStreamWaitEvent(ts, ms.ev_acc_done, 0));
  // 6: stitch the bucket pieces of all groups (stage 6 ends), 7: bucket reduction of every
  // window (stage 7 ends), 8: weighted tree -> one sum per window, Horner over the windows
  GroupTab gt;
  gt.ng = ngroups;
  for (int k = 0; k < ngroups; k++) {
    gt.wlo[k] = windowed ? k : wlo[k];
    gt.whi[k] = windowed ? k + 1 : whi[k];
    gt.offs[k] = w.counts[k];
  }
  pt_t* sums = nullptr;
  rc = launch_tail(ts, w, nthreads, gt, g, rows, pl, &ms.ev_stage[6], &sums);
  if (rc) return rc;
  // windowed: the group sums are already weighted by 2^(c w), k_msm_finish only adds them
  rc = finish(ts, sums, (int)rows, windowed ? 0 : g.c, out_element, out_encoding);
  if (rc) return rc;
  D377_CUDA(stage_mark(8, ts));
  D377_CUDA(cudaEventRecord(ms.ev_tail_done[set], ts));
  ms.tail_used[set] = true;
  if (ts != st) ms.tail_pending = true;
  return D377_OK;
}

// Enqueue a whole MSM (no host synchronisation).  `flags` (device word, reset by the
// caller) collects bit 0 = non-canonical scalar, bit 1 = invalid encoding.  The result is
// complete on result_stream(e).
int msm_enqueue(const uint8_t* scalars, const uint8_t* points, int point_format, bool sc_mont, size_t n,
                uint8_t* out_element, uint8_t* out_encoding, uint32_t* flags, size_t chunk,
                const cudaEvent_t* chunk_ready, bool inputs_ready, const cudaEvent_t* scalars_ready_ev) {
  Engine& e = engine();
  const cudaEvent_t no_event = nullptr;
  if (n == 0) return finish(result_stream(e), nullptr, 0, 0, out_element, out_encoding);
  const size_t kMax = (size_t)1 << 26;  // keeps n * W below 2^32
  if (chunk == 0 || chunk > kMax) chunk = kMax;
  size_t nchunks = (n + chunk - 1) / chunk;
  if (nchunks > 16) { set_error("msm: too many chunks (n = %zu, chunk = %zu)", n, chunk); return D377_ERR_INVALID_ARG; }
  // prepared bases: the set's layout (a windowed set keeps its stride N in every chunk, whose
  // records start at points + 128 * lo)
  BasesLayout layout;
  if (point_format == D377_PT_BASES) {
    int rc = check_bases(e, points, n, &layout);
    if (rc) return rc;
  }
  const BasesLayout* bl = point_format == D377_PT_BASES ? &layout : nullptr;
  // inputs_ready: the inputs depend on nothing but chunk_ready[k] (or on nothing)
  auto ready_of = [&](size_t k) -> const cudaEvent_t* {
    return !inputs_ready ? nullptr : chunk_ready ? &chunk_ready[k] : &no_event;
  };
  // scalars_ready_ev[k] (optional): the scalars of chunk k alone are uploaded -- the scalar
  // side starts on it, ahead of the chunk's points
  auto sc_ready_of = [&](size_t k) -> const cudaEvent_t* {
    return inputs_ready && scalars_ready_ev ? &scalars_ready_ev[k] : ready_of(k);
  };
  if (nchunks == 1) {
    if (chunk_ready) D377_CUDA(cudaStreamWaitEvent(e.stream, chunk_ready[0], 0));
    return msm_once(scalars, points, point_format, sc_mont, n, out_element, out_encoding, flags, sc_ready_of(0),
                    ready_of(0), bl);
  }
  pt_t* partials = (pt_t*)(e.d_small + kSmallPartials);  // up to 16 chunk results
  for (size_t k = 0; k < nchunks; k++) {
    size_t lo = k * chunk, len = std::min(chunk, n - lo);
    if (chunk_ready) D377_CUDA(cudaStreamWaitEvent(e.stream, chunk_ready[k], 0));
    int rc = msm_once(scalars + 32 * lo, points + pt_bytes(point_format) * lo, point_format, sc_mont, len,
                      (uint8_t*)(partials + k), nullptr, flags, sc_ready_of(k), ready_of(k), bl);
    if (rc) return rc;
  }
  cudaStream_t rs = result_stream(e);
  pt_t* tmp = (pt_t*)(e.d_small + kSmallTmp);
  k_sum_groups<false><<<1, kBlk, 0, rs>>>(partials, 1, (uint32_t)nchunks, 32, tmp);
  D377_LAUNCHED();
  D377_CUDA(cudaGetLastError());
  return finish(rs, tmp, 1, 0, out_element, out_encoding);
}

int msm_check_flags(uint32_t flags) {
  if (flags & 1u) {
    set_error("msm: a scalar is not canonical (>= r)");
    return D377_ERR_SCALAR_RANGE;
  }
  if (flags & 2u) {
    set_error("msm: an input encoding is invalid");
    return D377_ERR_INVALID_ENCODING;
  }
  return D377_OK;
}

int msm_args_ok(Engine& e, const char* who, const uint8_t* scalars, const uint8_t* points, int point_format,
                size_t n, int* fmt, bool* sc_mont) {
  int rc = parse_format(who, point_format, kPointFormats | fmt_set(D377_PT_BASES), fmt, sc_mont);
  if (rc) return rc;
  if (n && (!scalars || !points)) { set_error("null pointer"); return D377_ERR_INVALID_ARG; }
  if (*fmt == D377_PT_BASES && n) return check_bases(e, points, n);
  return D377_OK;
}

int msm_dev(const uint8_t* scalars, const uint8_t* points, int point_format, size_t n,
            uint8_t* out_element, uint8_t* out_encoding) {
  Engine& e = engine();
  int fmt = 0;
  bool sc_mont = false;
  int rc = msm_args_ok(e, "d377_msm_dev", scalars, points, point_format, n, &fmt, &sc_mont);
  if (rc) return rc;
  uint32_t* dflags = (uint32_t*)(e.d_small + kSmallFlags);
  uint32_t* hflags = (uint32_t*)(e.h_small + kSmallFlags);
  D377_CUDA(cudaMemsetAsync(dflags, 0, 4, e.stream));
  rc = msm_enqueue(scalars, points, fmt, sc_mont, n, out_element, out_encoding, dflags);
  if (rc) return rc;
  // status word: the only host read-back of the pipeline
  cudaStream_t rs = result_stream(e);
  D377_CUDA(cudaMemcpyAsync(hflags, dflags, 4, cudaMemcpyDeviceToHost, rs));
  D377_CUDA(cudaStreamSynchronize(rs));
  return msm_check_flags(*hflags);
}

// Same, without the host synchronisation: the status word is sticky and d377_sync reports
// it.  Back-to-back calls overlap the tail of one MSM with the head of the next.
int msm_dev_async(const uint8_t* scalars, const uint8_t* points, int point_format, size_t n,
                  uint8_t* out_element, uint8_t* out_encoding, int flags) {
  Engine& e = engine();
  int fmt = 0;
  bool sc_mont = false;
  int rc = msm_args_ok(e, "d377_msm_dev_async", scalars, points, point_format, n, &fmt, &sc_mont);
  if (rc) return rc;
  e.async_status_dirty = true;
  return msm_enqueue(scalars, points, fmt, sc_mont, n, out_element, out_encoding,
                     (uint32_t*)(e.d_small + kSmallAsyncFlags), 0, nullptr,
                     (flags & D377_MSM_INPUTS_READY) != 0);
}

// ---- many independent MSMs in one segmented Pippenger (d377_msm_segmented*) --------------
// A chunk's bucket sums (J W K x 128 B) stay under this budget; chunks are cut at segment
// bounds and run one after the other over one workspace.
constexpr size_t kSegBucketBudget = (size_t)1 << 30;
constexpr size_t kSegMaxEntries = 0xfffffff0ull;   // entries (pairs x W) of a chunk, as msm_once

// any 256-bit scalar: no carry out of the top window
static MsmGeom seg_geom(int c) { return geom(c, (257 + c - 1) / c); }

int msm_segmented_width(Engine& e, int fmt, const uint32_t* offsets, size_t nmsm, int* c_out) {
  const size_t n = offsets[nmsm];
  size_t longest = 0;
  for (size_t j = 0; j < nmsm; j++) longest = std::max<size_t>(longest, offsets[j + 1] - offsets[j]);
  // bucket operands as msm_once's, over all pairs of the call
  const double madd = affine_operands(e, fmt, n) ? 7.0 : 8.0;
  const int lo = e.msm_window_override ? e.msm_window_override : 4;
  const int hi = e.msm_window_override ? e.msm_window_override : 16;
  int best_c = 0;
  double best = 1e300;
  for (int c = lo; c <= hi; c++) {
    const MsmGeom g = seg_geom(c);
    // every segment must fit a chunk of its own
    if ((size_t)g.W * g.K * sizeof(pt_t) > kSegBucketBudget || longest * (size_t)g.W >= kSegMaxEntries) continue;
    // one bucket addition per (pair, window); two additions (~32 M with the tree) per bucket,
    // empty or not; the four-lane Horner tail of every segment
    const double K = (double)g.K, W = (double)g.W;
    const double cost = (double)n * W * madd + (double)nmsm * W * K * 32.0 + (double)nmsm * W * (c + 1) * 8.0;
    if (cost < best) { best = cost; best_c = c; }
  }
  if (!best_c) {
    set_error("d377_msm_segmented: a segment of %zu pairs does not fit one chunk at window width %s%d", longest,
              e.msm_window_override ? "" : "<= ", hi);
    return D377_ERR_INVALID_ARG;
  }
  *c_out = best_c;
  return D377_OK;
}

// Enqueue on the engine stream; arguments checked, `offsets` in host memory, c from
// msm_segmented_width.  Device pointers: scalars, points, out, ok (may be null).
int msm_segmented_enqueue(const uint8_t* scalars, const uint8_t* points, int fmt, bool sc_mont,
                          const uint32_t* offsets, size_t nmsm, int c, uint8_t* out, int out_format, uint8_t* ok) {
  Engine& e = engine();
  const MsmGeom g = seg_geom(c);
  const size_t n = offsets[nmsm];
  const size_t WK = (size_t)g.W * g.K;
  // chunks of whole segments: J W K x 128 B of buckets within the budget (so J W K < 2^31
  // too) and fewer than kSegMaxEntries entries
  struct Chunk { size_t j0, J; };
  std::vector<Chunk> chunks;
  size_t max_pairs = 0, max_J = 0;
  for (size_t j0 = 0; j0 < nmsm;) {
    size_t J = 1;
    while (j0 + J < nmsm && (J + 1) * WK * sizeof(pt_t) <= kSegBucketBudget &&
           (size_t)(offsets[j0 + J + 1] - offsets[j0]) * g.W < kSegMaxEntries)
      J++;
    chunks.push_back({j0, J});
    max_pairs = std::max<size_t>(max_pairs, offsets[j0 + J] - offsets[j0]);
    max_J = std::max(max_J, J);
    j0 += J;
  }
  const size_t max_entries = max_pairs * g.W;
  const PassPlan pl = pass_plan(g, max_entries);
  const bool affine = affine_operands(e, fmt, n);

  // ---- workspace: the call's offsets, scalars, bucket operands and decode status, then one
  // chunk's pass ----
  uint32_t* d_offs = nullptr;
  uint8_t *sc = nullptr, *ops = nullptr, *norm = nullptr, *okp = nullptr;
  PassWs w;
  const size_t max_nb = max_J * WK;
  auto layout = [&](uintptr_t base) {
    Carver cv{base};
    d_offs = cv.take<uint32_t>((nmsm + 1) * 4);
    sc = cv.take(sc_mont ? n * 32 : 0);
    ops = cv.take(n * 128);
    norm = cv.take(affine && projective_format(fmt) ? n * 32 : 0);
    okp = fmt == D377_PT_ENCODING ? cv.take(n) : nullptr;
    w = carve_pass(cv, max_entries, 1, &max_nb, (max_entries + pl.L - 1) / pl.L, max_J * g.W, g, pl.S);
    return cv.off;
  };
  int rc = ensure(e.seg_ws, layout(0));
  if (rc) return rc;
  layout((uintptr_t)e.seg_ws.p);
  cudaStream_t st = e.stream;

  // The offsets go up through a pinned staging copy, so that the caller may reuse its array
  // as soon as the call returns; the previous call's upload must have left the staging buffer.
  const size_t off_bytes = (nmsm + 1) * 4;
  if (!e.ev_seg_off) D377_CUDA(cudaEventCreateWithFlags(&e.ev_seg_off, cudaEventDisableTiming));
  else D377_CUDA(cudaEventSynchronize(e.ev_seg_off));
  if (e.seg_off_cap < off_bytes) {
    if (e.seg_off_host) D377_CUDA(cudaFreeHost(e.seg_off_host));
    e.seg_off_host = nullptr;
    e.seg_off_cap = 0;
    D377_CUDA(cudaHostAlloc(&e.seg_off_host, off_bytes, cudaHostAllocDefault));
    e.seg_off_cap = off_bytes;
  }
  memcpy(e.seg_off_host, offsets, off_bytes);
  D377_CUDA(cudaMemcpyAsync(d_offs, e.seg_off_host, off_bytes, cudaMemcpyHostToDevice, st));
  D377_CUDA(cudaEventRecord(e.ev_seg_off, st));

  // ---- once per call: canonical scalars, bucket operands (and per-pair decode status) ----
  if (n) {
    if (sc_mont) {
      launch_fr_from_mont(scalars, n, sc, st);
      scalars = sc;
    }
    // no flags word: affine inputs never fail to load, normalisation reports nothing and
    // encodings report per pair in okp
    launch_operands(e, fmt, affine, normalize_min_per(e), points, n, norm, ops, nullptr, okp, st);
  }

  // ---- chunk by chunk ----
  const size_t ob = out_bytes(out_format);
  for (const Chunk& ch : chunks) {
    const size_t p0 = offsets[ch.j0], np = offsets[ch.j0 + ch.J] - p0;
    const size_t nb = ch.J * WK, nthreads = (np * g.W + pl.L - 1) / pl.L;
    const uint32_t* offs = d_offs + ch.j0;
    D377_CUDA(cudaMemsetAsync(w.counts[0], 0, (nb + 1) * 4, st));
    if (np) {
      k_msm_count_seg<<<grid_for(np, 256), 256, 0, st>>>(scalars + 32 * p0, np, offs, (uint32_t)ch.J, g, w.counts[0],
                                                         w.dig);
      D377_LAUNCHED();
    }
    // stored index: the pair within the chunk, whose bucket operands start at p0
    launch_sort(st, w.counts[0], w.cursor[0], w.tiles[0], nb, w.dig, np, (uint32_t)g.W, w.sorted, 0u, 0u, 0u);
    if (np) {
      D377_CUDA(cudaMemsetAsync(w.pb, 0xff, 2 * nthreads * 4, st));
      launch_accumulate(st, affine, ops + 128 * p0, w.sorted, w.counts[0], nb, pl.L, nthreads, w.bsum, 0, w.part, w.pb);
    }
    // bucket reduction: one group of J W virtual windows
    const size_t rows = ch.J * g.W;
    const GroupTab gt{1, {0}, {(int)rows}, {w.counts[0]}};
    pt_t* sums = nullptr;
    rc = launch_tail(st, w, nthreads, gt, g, rows, pl, nullptr, &sums);
    if (rc) return rc;
    k_msm_finish<<<grid_for(ch.J * 4, kFinishBlk), kFinishBlk,
                   out_format == D377_OUT_ENCODING ? ISQRT_SMEM_WORDS(kFinishBlk) * 4 : 0, st>>>(
        sums, (uint32_t)ch.J, g.W, g.c, offs, okp, out_format == D377_OUT_ELEMENT ? out + ob * ch.j0 : nullptr,
        out_format == D377_OUT_ENCODING ? out + ob * ch.j0 : nullptr, ok ? ok + ch.j0 : nullptr);
    D377_LAUNCHED();
    D377_CUDA(cudaGetLastError());
  }
  e.seg_last_c = g.c;
  e.seg_last_W = g.W;
  e.seg_last_chunks = chunks.size();
  return D377_OK;
}

int msm_segmented_last(int* c, int* W, size_t* chunks) {
  Engine& e = engine();
  if (!e.seg_last_c) { set_error("no segmented msm has run yet"); return D377_ERR_INVALID_ARG; }
  if (c) *c = e.seg_last_c;
  if (W) *W = e.seg_last_W;
  if (chunks) *chunks = e.seg_last_chunks;
  return D377_OK;
}

bool msm_last_mixed() { return engine().msm.last_affine; }
bool msm_last_windowed() { return engine().msm.last_windowed; }

// d377_shutdown: the streams and events above belong to the device being released
void msm_shutdown(Engine& e) {
  MsmState& ms = e.msm;
  if (ms.ready) {
    cudaStreamSynchronize(ms.sort_stream);
    cudaStreamSynchronize(ms.tail_stream);
    cudaStreamSynchronize(ms.points_stream);
    cudaStreamDestroy(ms.points_stream);
    for (int k = 0; k < 2; k++) cudaEventDestroy(ms.ev_points_done[k]);
    cudaStreamDestroy(ms.sort_stream);
    cudaStreamDestroy(ms.tail_stream);
    ms.sort_stream = ms.tail_stream = nullptr;
    cudaEventDestroy(ms.ev_fork);
    cudaEventDestroy(ms.ev_acc_done);
    cudaEventDestroy(ms.ev_join);
    for (int k = 0; k < 2; k++) cudaEventDestroy(ms.ev_tail_done[k]);
    for (int k = 0; k < kMaxGroups; k++) {
      cudaEventDestroy(ms.ev_sorted[k]);
      cudaEventDestroy(ms.ev_acc0[k]);
      cudaEventDestroy(ms.ev_acc[k]);
    }
    cudaEventDestroy(ms.ev_sort0);
    cudaEventDestroy(ms.ev_sort1);
    for (int k = 0; k <= kMsmStages; k++) cudaEventDestroy(ms.ev_stage[k]);
  }
  for (int k = 0; k < 2; k++) {
    if (ms.tail_ws[k].p) cudaFree(ms.tail_ws[k].p);
    ms.tail_ws[k] = DevBuf();
  }
  ms = MsmState();
}

int msm_stage_info(float* ms_out, int* c, int* W, uint64_t* n) {
  MsmState& ms = engine().msm;
  if (!ms.ready || !ms.stage_valid) { set_error("no msm has run yet"); return D377_ERR_INVALID_ARG; }
  D377_CUDA(cudaEventSynchronize(ms.ev_stage[kMsmStages]));
  for (int k = 0; k < kMsmStages; k++) D377_CUDA(cudaEventElapsedTime(&ms_out[k], ms.ev_stage[k], ms.ev_stage[k + 1]));
  // the scalar side runs on its own stream, overlapped with `points` and `accumulate`:
  // its whole span (count + scan + scatter of every window group) is reported as `count`
  D377_CUDA(cudaEventElapsedTime(&ms_out[1], ms.ev_sort0, ms.ev_sort1));
  if (c) *c = ms.last_geom.c;
  if (W) *W = ms.last_geom.W;
  if (n) *n = ms.last_n;
  return D377_OK;
}

// Per window group of the most recent single-chunk MSM, in ms after its start: sorted list
// ready (sort stream), accumulation start / end (engine stream), end of the MSM.
int msm_timeline(float* out, int cap, int* ngroups) {
  MsmState& ms = engine().msm;
  if (!ms.ready || !ms.stage_valid) { set_error("no msm has run yet"); return D377_ERR_INVALID_ARG; }
  D377_CUDA(cudaEventSynchronize(ms.ev_stage[kMsmStages]));
  const int ng = ms.last_groups;
  if (ngroups) *ngroups = ng;
  for (int k = 0; k < ng && 4 * k + 3 < cap; k++) {
    D377_CUDA(cudaEventElapsedTime(&out[4 * k + 0], ms.ev_stage[0], ms.ev_sorted[k]));
    D377_CUDA(cudaEventElapsedTime(&out[4 * k + 1], ms.ev_stage[0], ms.ev_acc0[k]));
    D377_CUDA(cudaEventElapsedTime(&out[4 * k + 2], ms.ev_stage[0], ms.ev_acc[k]));
    D377_CUDA(cudaEventElapsedTime(&out[4 * k + 3], ms.ev_stage[0], ms.ev_stage[kMsmStages]));
  }
  return D377_OK;
}

}  // namespace d377
