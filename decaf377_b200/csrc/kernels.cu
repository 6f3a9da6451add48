// Engine plumbing, the light element-wise kernels and the C ABI of
// include/decaf377_b200.h.  The heavy kernels live in codec.cu (decompress / compress /
// Elligator / isqrt), scalar.cu (scalar multiplication, fixed base) and
// msm.cu (Pippenger, batch normalisation); this file launches them through the functions of engine.h.
#include <algorithm>
#include <cstdarg>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "engine.h"
#include "point.cuh"

namespace d377 {

// ---------------------------------------------------------------------------
// engine plumbing
// ---------------------------------------------------------------------------
static thread_local std::string g_err;
static thread_local Engine* tl_engine = nullptr;   // d377_set_device
static std::mutex g_reg_mu;                         // guards the registry below
static constexpr int kMaxDevices = 64;
static Engine* g_engines[kMaxDevices] = {};
static Engine* g_default = nullptr;
static int g_order[kMaxDevices];                    // devices in initialisation order
static int g_norder = 0;
static std::atomic<uint64_t> g_launches{0};

Engine& engine() {
  static Engine none;   // never ready: what the entry points see before d377_init
  Engine* e = tl_engine ? tl_engine : g_default;
  return e ? *e : none;
}

Engine* engine_for(int device) {
  if (device < 0 || device >= kMaxDevices) return nullptr;
  std::lock_guard<std::mutex> lk(g_reg_mu);
  Engine* e = g_engines[device];
  return e && e->ready ? e : nullptr;
}

void select_engine(Engine* e) { tl_engine = e; }
Engine* selected_engine() { return tl_engine; }

void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

void set_error(const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
}

const char* last_error() { return g_err.c_str(); }

int cuda_fail(cudaError_t e, const char* what, const char* file, int line) {
  set_error("CUDA error %d (%s) at %s:%d in `%s`", (int)e, cudaGetErrorString(e), file, line, what);
  return D377_ERR_CUDA;
}

int ensure(DevBuf& b, size_t bytes) {
  if (bytes <= b.cap) return D377_OK;
  if (b.p) D377_CUDA(cudaFree(b.p));
  b.p = nullptr;
  b.cap = 0;
  size_t cap = bytes + (bytes >> 3) + 256;
  D377_CUDA(cudaMalloc(&b.p, cap));
  b.cap = cap;
  return D377_OK;
}

// ---------------------------------------------------------------------------
// kernels
// ---------------------------------------------------------------------------

// Element (+ | - | neg | double), ark_curve/ops/projective.rs:5-104 (the arkworks group
// law behind them is min_curve/element.rs:119-136, 291-332).
//   0: a + b   1: a - b   2: -a   3: 2a
template <int kOp>
__global__ void k_binop(const uint8_t* __restrict__ a, const uint8_t* __restrict__ b, size_t n,
                        uint8_t* __restrict__ out) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  pt_t p = pt_load_wire(a + 128 * i), r;
  if (kOp == 0) r = pt_add(p, pt_load_wire(b + 128 * i));
  else if (kOp == 1) r = pt_add(p, pt_neg(pt_load_wire(b + 128 * i)));
  else if (kOp == 2) r = pt_neg(p);
  else r = pt_dbl<true>(p);
  D377_DBG_POINT(r);
  pt_store_canon(out + 128 * i, r);
}

// PartialEq, element/projective.rs:65-70: x1*y2 == x2*y1
__global__ void k_eq(const uint8_t* __restrict__ a, const uint8_t* __restrict__ b, size_t n,
                     uint8_t* __restrict__ eq) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  fq_t x1 = fq_load_wire(a + 128 * i), y1 = fq_load_wire(a + 128 * i + 32);
  fq_t x2 = fq_load_wire(b + 128 * i), y2 = fq_load_wire(b + 128 * i + 32);
  eq[i] = fq_eq(fq_mul(x1, y2), fq_mul(x2, y1)) ? 1 : 0;
}

// field-layer test entry (rows a2-a4)
__global__ void k_fq_op(int op, const uint8_t* __restrict__ a, const uint8_t* __restrict__ b,
                        size_t n, uint8_t* __restrict__ out) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  // ops 5 and 7 take arbitrary bytes; the others Montgomery limbs (brought below 2q on load)
  fq_raw_t xr = fq_load_raw(a + 32 * i);
  fq_t x = fq_load_wire(a + 32 * i);
  fq_t y = b ? fq_load_wire(b + 32 * i) : fq_t(fq_zero());
  fq_r r;
  switch (op) {
    case 0: r = fq_reduce(fq_mul(x, y)); break;
    case 1: r = fq_reduce(fq_sqr(x)); break;
    case 2: r = fq_reduce(fq_add(x, y)); break;
    case 3: r = fq_reduce(fq_sub(x, y)); break;
    case 4: r = fq_reduce(fq_neg(x)); break;
    case 6: r = fq_from_mont(x); break;
    case 8: r = fq_reduce(fq_inv_vartime(x)); break;            // binary-GCD inverse, 0 -> 0
    case 9: r = fq_reduce(fq_inv(x)); break;                    // Fermat inverse, 0 -> 0
    case 10: r = fq_reduce(fq_mul_small<6042>(x)); break;       // small-constant products
    case 11: r = fq_reduce(fq_mul_small<12086>(x)); break;
    default: r = fq_reduce(fq_to_mont(xr)); break;  // 5 to_montgomery, 7 from_le_bytes_mod_order
  }
  fq_store(out + 32 * i, r);
}

// Fq::from_le_bytes_mod_order for inputs of ANY length (fields/fq.rs:90-102): the bytes
// are cut into 32-byte little-endian chunks (the last one zero-padded) and folded from the
// most significant chunk down, acc = acc * 2^256 + chunk.  In Montgomery form a
// multiplication by 2^256 = R is a Montgomery product with R^2, and chunk -> Montgomery is
// the same product (fq_to_mont), so every step is one fq_mul and one addition.
__global__ void k_fq_from_wide(const uint8_t* __restrict__ in, size_t width, size_t n,
                               uint8_t* __restrict__ out) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  fq_store_canon(out + 32 * i, fq_from_le_bytes_wide(in + width * i, width));
}

// Fq / Fr CanonicalDeserialize (fq/arkworks.rs:189-229, fr/arkworks.rs): 32 canonical
// LE bytes -> Montgomery form, ok = 0 (and a zero element) when the value is >= modulus.
// kField: 0 = Fq (converted to Montgomery), 1 = Fr (range check only; scalars stay
// canonical on this ABI).
template <int kField>
__global__ void k_field_deserialize(const uint8_t* __restrict__ in, size_t n, uint8_t* __restrict__ out,
                                    uint8_t* __restrict__ ok) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  fq_raw_t x = fq_load_raw(in + 32 * i);
  bool good;
  if (kField == 0) {
    good = fq_raw_is_canonical(x);
    if (out) fq_store_canon(out + 32 * i, fq_select(good, fq_to_mont(x), fq_zero()));
  } else {
    good = fr_raw_is_canonical(x);
    // a canonical scalar is < r < q: the bytes pass through unchanged
    if (out) fq_store(out + 32 * i, fq_assume<2000>(fq_select(good, x, fq_zero())));
  }
  ok[i] = good ? 1 : 0;
}

// D377_SCALARS_MONTGOMERY: Fr limbs as the reference keeps them in memory -> canonical
// little-endian integers (Fr::into_bigint, fields/fr/arkworks.rs:36-57)
__global__ void k_fr_from_mont(const uint8_t* __restrict__ in, size_t n, uint8_t* __restrict__ out) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  fq_store(out + 32 * i, fq_assume<2000>(fr_from_mont(fq_load_raw(in + 32 * i))));
}

void launch_fr_from_mont(const uint8_t* in, size_t n, uint8_t* out, cudaStream_t st) {
  k_fr_from_mont<<<grid_for(n, 256), 256, 0, st>>>(in, n, out);
  D377_LAUNCHED();
}

// ---- IMAD.WIDE issue-rate microbenchmark --------------------------------
// Eight independent IMAD.WIDE.U32 (with carry-out, the form fq_mul issues) per
// step; every multiplicand is another accumulator's limb so that ptxas can
// neither hoist nor strength-reduce the products.  Counts 8 wide multiply-adds
// per step; 2048 resident threads per SM.  The achieved rate depends on the
// register-bank pattern ptxas happens to pick for the four source registers, so
// a few operand arrangements are timed and the best one is reported.
template <int kVariant>
__global__ void __launch_bounds__(256) k_imad_peak(uint32_t* out, uint32_t seed, int iters) {
  uint32_t b0 = seed * 3 + threadIdx.x * 5 + 7, b1 = b0 ^ 0x5bd1e995u;
  uint32_t x[16];
#pragma unroll
  for (int j = 0; j < 16; j++) x[j] = j * seed + threadIdx.x;
#pragma unroll 1
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int r = 0; r < 8; r++) {
#pragma unroll
      for (int j = 0; j < 8; j++) {
        const int src = kVariant == 0 ? ((2 * j + 3) & 15) : kVariant == 1 ? ((2 * j + 2) & 15)
                                                                          : ((2 * j + 5) & 15);
        asm volatile("mad.lo.cc.u32 %0, %2, %3, %0;\n\tmadc.hi.u32 %1, %2, %3, %1;"
                     : "+r"(x[2 * j]), "+r"(x[2 * j + 1])
                     : "r"(x[src]), "r"(kVariant == 3 ? ((j & 1) ? b1 : b0) : b0));
      }
    }
  }
  uint32_t s = 0;
#pragma unroll
  for (int j = 0; j < 16; j++) s ^= x[j];
  if (s == 0x1234567u) out[0] = s + b1;
}

D377_DBG_READER(kernels_debug_counts)

// ---------------------------------------------------------------------------
// host side of the API
// ---------------------------------------------------------------------------

// D377_SCALARS_MONTGOMERY rides on the format word of every call that takes scalars
int parse_format(const char* who, int word, unsigned accepted, int* fmt, bool* sc_mont) {
  const bool m = sc_mont && word >= 0 && (word & D377_SCALARS_MONTGOMERY) != 0;
  const int f = m ? word & ~D377_SCALARS_MONTGOMERY : word;
  if (f < 0 || f > 31 || !((accepted >> f) & 1u)) {
    set_error("%s: format word %d is not accepted", who, word);
    return D377_ERR_INVALID_ARG;
  }
  if (fmt) *fmt = f;
  if (sc_mont) *sc_mont = m;
  return D377_OK;
}
// point formats of the calls that multiply caller's points by scalars one by one
constexpr unsigned kMulFormats = fmt_set(D377_PT_ELEMENT, D377_PT_ENCODING, D377_PT_AFFINE);
// scalars in the reference's Montgomery form -> canonical, into the engine's scratch
static int canonical_scalars(Engine& e, const uint8_t*& scalars, size_t n) {
  int rc = ensure(e.sc_canon, n * 32 + 32);
  if (rc) return rc;
  launch_fr_from_mont(scalars, n, (uint8_t*)e.sc_canon.p, e.stream);
  scalars = (const uint8_t*)e.sc_canon.p;
  return D377_OK;
}

void codec_debug_counts(unsigned long long*, unsigned long long*);
void scalar_debug_counts(unsigned long long*, unsigned long long*);
void msm_debug_counts(unsigned long long*, unsigned long long*);

// Create the engine of `device` (idempotent).  Called with g_reg_mu held.
static int engine_create(int device) {
  if (g_engines[device] && g_engines[device]->ready) return D377_OK;
  cudaDeviceProp prop;
  int prev = -1;
  cudaGetDevice(&prev);
  D377_CUDA(cudaSetDevice(device));
  D377_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) {
    set_error("device %d is sm_%d%d; this library contains sm_100a code only", device, prop.major,
              prop.minor);
    return D377_ERR_CUDA;
  }
  if (!g_engines[device]) g_engines[device] = new Engine();
  Engine& e = *g_engines[device];
  e.device = device;
  e.sm_count = prop.multiProcessorCount;
  D377_CUDA(cudaStreamCreateWithFlags(&e.stream, cudaStreamNonBlocking));
  D377_CUDA(cudaMalloc(&e.d_small, kSmallBytes));
  D377_CUDA(cudaMemset(e.d_small, 0, kSmallBytes));
  D377_CUDA(cudaHostAlloc(&e.h_small, kSmallBytes, cudaHostAllocPortable));
  memset(e.h_small, 0, kSmallBytes);
  D377_CUDA(cudaStreamCreateWithFlags(&e.copy_stream, cudaStreamNonBlocking));
  D377_CUDA(cudaStreamCreateWithFlags(&e.out_stream, cudaStreamNonBlocking));
  for (int k = 0; k < Engine::kSlots; k++) {
    D377_CUDA(cudaEventCreateWithFlags(&e.ev_h2d[k], cudaEventDisableTiming));
    D377_CUDA(cudaEventCreateWithFlags(&e.ev_done[k], cudaEventDisableTiming));
    for (int c = 0; c < Engine::kMsmHostChunks; c++) {
      D377_CUDA(cudaEventCreateWithFlags(&e.ev_chunk[k][c], cudaEventDisableTiming));
      D377_CUDA(cudaEventCreateWithFlags(&e.ev_chunk_sc[k][c], cudaEventDisableTiming));
    }
    e.slot_busy[k] = false;
  }
  for (int b = 0; b < 2; b++) {
    D377_CUDA(cudaEventCreateWithFlags(&e.pe_in[b], cudaEventDisableTiming));
    D377_CUDA(cudaEventCreateWithFlags(&e.pe_k[b], cudaEventDisableTiming));
    D377_CUDA(cudaEventCreateWithFlags(&e.pe_out[b], cudaEventDisableTiming));
  }
  D377_CUDA(cudaEventCreateWithFlags(&e.ev_partial, cudaEventDisableTiming));
  e.ready = true;
  bool known = false;
  for (int k = 0; k < g_norder; k++) known = known || g_order[k] == device;
  if (!known) g_order[g_norder++] = device;
  if (prev >= 0 && prev != device) cudaSetDevice(prev);
  return D377_OK;
}

static void worker_stop(Engine& e) {
  if (!e.worker.joinable()) return;
  {
    std::lock_guard<std::mutex> lk(e.wmu);
    e.wquit = true;
  }
  e.wcv.notify_all();
  e.worker.join();
  e.wquit = false;
}

static void engine_destroy(Engine& e) {
  if (!e.ready) return;
  worker_stop(e);
  std::lock_guard<std::recursive_mutex> lk(e.mu);
  cudaSetDevice(e.device);
  cudaStreamSynchronize(e.stream);
  msm_shutdown(e);
  if (e.out_stream) cudaStreamSynchronize(e.out_stream);
  if (e.copy_stream) cudaStreamSynchronize(e.copy_stream);
  for (DevBuf* b : {&e.in0, &e.in1, &e.out0, &e.out1, &e.scratch, &e.sc_canon, &e.slot_sc[0], &e.slot_sc[1],
                    &e.slot_pt[0], &e.slot_pt[1], &e.st_in[0][0], &e.st_in[0][1], &e.st_in[0][2],
                    &e.st_in[1][0], &e.st_in[1][1], &e.st_in[1][2], &e.st_out[0][0], &e.st_out[0][1],
                    &e.st_out[1][0], &e.st_out[1][1], &e.sum_ws[0], &e.sum_ws[1], &e.bm_prod, &e.bm_ok,
                    &e.bm_sum, &e.bm_sc, &e.bm_pt, &e.bm_off, &e.bm_out, &e.bm_okout, &e.seg_ws}) {
    if (b->p) cudaFree(b->p);
    b->p = nullptr;
    b->cap = 0;
  }
  if (e.seg_off_host) cudaFreeHost(e.seg_off_host);
  e.seg_off_host = nullptr;
  e.seg_off_cap = 0;
  if (e.ev_seg_off) cudaEventDestroy(e.ev_seg_off);
  e.ev_seg_off = nullptr;
  e.seg_last_c = e.seg_last_W = 0;
  e.seg_last_chunks = 0;
  // prepared bases still alive belong to the library (header contract): release them
  for (auto& kv : e.bases) cudaFree(const_cast<void*>(kv.first));
  e.bases.clear();
  for (auto& kv : e.fixed_bases) cudaFree(const_cast<void*>(kv.first));
  e.fixed_bases.clear();
  if (e.fb_table) cudaFree(e.fb_table);
  e.fb_table = nullptr;
  if (e.fb_table_jq) cudaFree(e.fb_table_jq);
  e.fb_table_jq = nullptr;
  if (e.d_small) cudaFree(e.d_small);
  if (e.h_small) cudaFreeHost(e.h_small);
  e.d_small = e.h_small = nullptr;
  for (int k = 0; k < Engine::kSlots; k++) {
    if (e.ev_h2d[k]) cudaEventDestroy(e.ev_h2d[k]);
    if (e.ev_done[k]) cudaEventDestroy(e.ev_done[k]);
    e.ev_h2d[k] = e.ev_done[k] = nullptr;
    for (int c = 0; c < Engine::kMsmHostChunks; c++) {
      if (e.ev_chunk[k][c]) cudaEventDestroy(e.ev_chunk[k][c]);
      if (e.ev_chunk_sc[k][c]) cudaEventDestroy(e.ev_chunk_sc[k][c]);
      e.ev_chunk[k][c] = e.ev_chunk_sc[k][c] = nullptr;
    }
    e.slot_busy[k] = false;
  }
  for (int b = 0; b < 2; b++) {
    for (cudaEvent_t* ev : {&e.pe_in[b], &e.pe_k[b], &e.pe_out[b]}) {
      if (*ev) cudaEventDestroy(*ev);
      *ev = nullptr;
    }
  }
  if (e.ev_partial) cudaEventDestroy(e.ev_partial);
  e.ev_partial = nullptr;
  if (e.copy_stream) cudaStreamDestroy(e.copy_stream);
  e.copy_stream = nullptr;
  if (e.out_stream) cudaStreamDestroy(e.out_stream);
  e.out_stream = nullptr;
  cudaStreamDestroy(e.stream);
  e.stream = nullptr;
  e.async_status_dirty = false;
  e.ready = false;
}

// Wait (on the host) for everything the host-buffer pipelines of this engine have in
// flight.  Error paths call it before they report failure, so that no copy into or out of
// the caller's buffers is still running when the caller gets control back.
static void drain(Engine& e) {
  if (e.copy_stream) cudaStreamSynchronize(e.copy_stream);
  if (e.stream) cudaStreamSynchronize(e.stream);
  if (e.out_stream) cudaStreamSynchronize(e.out_stream);
  if (e.msm.sort_stream) cudaStreamSynchronize(e.msm.sort_stream);
  if (e.msm.points_stream) cudaStreamSynchronize(e.msm.points_stream);
  if (e.msm.tail_stream) cudaStreamSynchronize(e.msm.tail_stream);
}

}  // namespace d377

using namespace d377;

#define TRY(x) do { int _rc = (x); if (_rc) return _rc; } while (0)

// recursive lock already held by the scope of D377_REQUIRE_READY; kept for the helpers
#define LOCK() std::lock_guard<std::recursive_mutex> _lk(engine().mu)

extern "C" {

static int init_common(const int* devices, int ndev) {
  int count = 0;
  cudaError_t ce = cudaGetDeviceCount(&count);
  if (ce != cudaSuccess || count == 0) {
    set_error("no CUDA device available (%s); decaf377_b200 has no CPU fallback",
              ce == cudaSuccess ? "device count is 0" : cudaGetErrorString(ce));
    return D377_ERR_CUDA;
  }
  for (int k = 0; k < ndev; k++) {
    if (devices[k] < 0 || devices[k] >= count || devices[k] >= kMaxDevices) {
      set_error("device %d out of range (have %d)", devices[k], count);
      return D377_ERR_INVALID_ARG;
    }
    for (int j = 0; j < k; j++)
      if (devices[j] == devices[k]) { set_error("device %d listed twice", devices[k]); return D377_ERR_INVALID_ARG; }
  }
  std::lock_guard<std::mutex> lk(g_reg_mu);
  for (int k = 0; k < ndev; k++) {
    int rc = engine_create(devices[k]);
    if (rc) return rc;
  }
  g_default = g_engines[devices[0]];
  return D377_OK;
}

int d377_init(int device) { return init_common(&device, 1); }

int d377_init_multi(const int* devices, int ndev) {
  if (!devices || ndev < 1 || ndev > 8) { set_error("d377_init_multi: 1..8 devices"); return D377_ERR_INVALID_ARG; }
  int rc = init_common(devices, ndev);
  if (rc) return rc;
  // peer access lets the 128-byte partial sums travel GPU to GPU over NVLink; without it
  // cudaMemcpyPeerAsync stages through the host, which is still correct
  int prev = -1;
  cudaGetDevice(&prev);
  for (int a = 0; a < ndev; a++) {
    cudaSetDevice(devices[a]);
    for (int b = 0; b < ndev; b++) {
      if (a == b) continue;
      int can = 0;
      if (cudaDeviceCanAccessPeer(&can, devices[a], devices[b]) == cudaSuccess && can) {
        cudaError_t pe = cudaDeviceEnablePeerAccess(devices[b], 0);
        if (pe == cudaSuccess || pe == cudaErrorPeerAccessAlreadyEnabled) {
          if (Engine* ea = engine_for(devices[a])) ea->peer_mask |= 1ull << devices[b];
        }
        if (pe != cudaSuccess) cudaGetLastError();   // already enabled, or unsupported: fine
      }
    }
  }
  if (prev >= 0) cudaSetDevice(prev);
  return D377_OK;
}

int d377_set_device(int device) {
  if (device < 0) { select_engine(nullptr); return D377_OK; }
  Engine* e = engine_for(device);
  if (!e) { set_error("device %d has not been initialised (d377_init / d377_init_multi)", device); return D377_ERR_NOT_INITIALISED; }
  select_engine(e);
  return D377_OK;
}

int d377_get_device(void) { return engine().ready ? engine().device : -1; }

int d377_device_list(int* devices, int cap) {
  std::lock_guard<std::mutex> lk(g_reg_mu);
  int k = 0;
  for (int i = 0; i < g_norder; i++)
    if (g_engines[g_order[i]] && g_engines[g_order[i]]->ready) {
      if (devices && k < cap) devices[k] = g_order[i];
      k++;
    }
  return k;
}

int d377_shutdown(void) {
  select_engine(nullptr);
  std::lock_guard<std::mutex> lk(g_reg_mu);
  int prev = -1;
  cudaGetDevice(&prev);
  if (g_default && g_default->ready) {
    cudaSetDevice(g_default->device);
    multi_shutdown();
  }
  for (int d = 0; d < kMaxDevices; d++)
    if (g_engines[d]) engine_destroy(*g_engines[d]);
  g_default = nullptr;
  g_norder = 0;
  if (prev >= 0) cudaSetDevice(prev);
  return D377_OK;
}

void* d377_stream(void) { return (void*)engine().stream; }
void* d377_result_stream(void) { return engine().ready ? (void*)result_stream(engine()) : nullptr; }

int d377_join(void) {
  D377_REQUIRE_READY();
  return D377_OK;
}

int d377_sync(void) {
  D377_REQUIRE_READY();
  Engine& e = _eng;
  if (e.async_status_dirty) {
    // status of the asynchronous MSMs enqueued since the last sync
    uint32_t* dflags = (uint32_t*)(e.d_small + kSmallAsyncFlags);
    uint32_t* hflags = (uint32_t*)(e.h_small + kSmallAsyncFlags);
    D377_CUDA(cudaMemcpyAsync(hflags, dflags, 4, cudaMemcpyDeviceToHost, e.stream));
    D377_CUDA(cudaMemsetAsync(dflags, 0, 4, e.stream));
    D377_CUDA(cudaStreamSynchronize(e.stream));
    e.async_status_dirty = false;
    return msm_check_flags(*hflags);
  }
  D377_CUDA(cudaStreamSynchronize(e.stream));
  return D377_OK;
}

const char* d377_last_error(void) { return last_error(); }

uint64_t d377_launch_count(void) { return g_launches.load(); }

int d377_debug_build(void) {
#ifdef D377_DEBUG_ON_CURVE
#ifdef D377_DEBUG_ORDER
  return 2;
#else
  return 1;
#endif
#else
  return 0;
#endif
}

int d377_debug_counts(uint64_t* failures, uint64_t* checked) {
  D377_REQUIRE_READY();
  if (!failures || !checked) { set_error("null pointer"); return D377_ERR_INVALID_ARG; }
  D377_CUDA(cudaDeviceSynchronize());
  unsigned long long f = 0, c = 0, tf = 0, tc = 0;
  kernels_debug_counts(&f, &c); tf += f; tc += c;
  codec_debug_counts(&f, &c); tf += f; tc += c;
  scalar_debug_counts(&f, &c); tf += f; tc += c;
  msm_debug_counts(&f, &c); tf += f; tc += c;
  *failures = tf;
  *checked = tc;
  D377_CUDA(cudaGetLastError());
  return D377_OK;
}

int d377_msm_stage_info(float ms[8], int* c, int* W, uint64_t* n) {
  D377_REQUIRE_READY();
  if (!ms) { set_error("null pointer"); return D377_ERR_INVALID_ARG; }
  return msm_stage_info(ms, c, W, n);
}

int d377_msm_timeline(float* ms, int cap, int* ngroups) {
  D377_REQUIRE_READY();
  if (!ms || cap < 4) { set_error("timeline buffer too small"); return D377_ERR_INVALID_ARG; }
  return msm_timeline(ms, cap, ngroups);
}

int d377_msm_last_mode(int* mixed) {
  D377_REQUIRE_READY();
  if (!mixed) { set_error("null pointer"); return D377_ERR_INVALID_ARG; }
  *mixed = msm_last_mixed() ? 1 : 0;
  return D377_OK;
}

int d377_msm_set_normalize(int mode) {
  if (mode < -1 || mode > 1) { set_error("normalize mode %d out of range [-1, 1]", mode); return D377_ERR_INVALID_ARG; }
  engine().msm_normalize_override = mode;
  return D377_OK;
}

int d377_msm_set_groups(int groups) {
  if (groups < 0 || groups > 8) { set_error("group count %d out of range [0, 8]", groups); return D377_ERR_INVALID_ARG; }
  engine().msm_groups_override = groups;
  return D377_OK;
}

int d377_msm_set_window(int c) {
  // choose_geom evaluates c = 4 .. 22
  if (c != 0 && (c < 4 || c > 22)) {
    set_error("window width %d out of range [4, 22]", c);
    return D377_ERR_INVALID_ARG;
  }
  engine().msm_window_override = c;
  return D377_OK;
}

int d377_msm_set_host_chunks(int k) {
  if (k < 0 || k > Engine::kMsmHostChunks) {
    set_error("host chunk count %d out of range [0, %d]", k, Engine::kMsmHostChunks);
    return D377_ERR_INVALID_ARG;
  }
  engine().msm_host_chunks_override = k;
  return D377_OK;
}

int d377_msm_set_tail_overlap(int on) {
  D377_REQUIRE_READY();
  _eng.msm_tail_overlap_override = on ? 1 : 0;
  return D377_OK;
}

void* d377_host_alloc(size_t bytes) {
  if (!engine().ready) { set_error("d377_init has not been called"); return nullptr; }
  EngineScope scope(engine());
  void* p = nullptr;
  // portable: usable by every device of a multi-GPU call
  cudaError_t ce = cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable);
  if (ce != cudaSuccess) {
    set_error("cudaHostAlloc(%zu) failed: %s", bytes, cudaGetErrorString(ce));
    return nullptr;
  }
  return p;
}

int d377_host_free(void* p) {
  if (!p) return D377_OK;
  D377_CUDA(cudaFreeHost(p));
  return D377_OK;
}

// ---- device-pointer entry points -------------------------------------------

int d377_batch_decompress_dev(const uint8_t* enc, size_t n, uint8_t* elements, uint8_t* ok) {
  D377_REQUIRE_READY();
  if (n == 0) return D377_OK;
  if (!enc || !elements) { set_error("null pointer"); return D377_ERR_INVALID_ARG; }
  launch_decompress(enc, n, elements, ok, _eng.stream);
  D377_LAUNCHED();
  D377_CUDA(cudaGetLastError());
  return D377_OK;
}

int d377_batch_compress_dev(const uint8_t* elements, size_t n, uint8_t* enc) {
  D377_REQUIRE_READY();
  if (n == 0) return D377_OK;
  if (!enc || !elements) { set_error("null pointer"); return D377_ERR_INVALID_ARG; }
  launch_compress(elements, n, enc, _eng.stream);
  D377_LAUNCHED();
  D377_CUDA(cudaGetLastError());
  return D377_OK;
}

static int null_pointer() {
  set_error("null pointer");
  return D377_ERR_INVALID_ARG;
}

static int decompress_fmt_args(const uint8_t* enc, size_t n, int out_format, const uint8_t* out) {
  TRY(parse_format("d377_batch_decompress_fmt", out_format, fmt_set(D377_PT_ELEMENT, D377_PT_AFFINE), nullptr));
  return n && (!enc || !out) ? null_pointer() : D377_OK;
}

int d377_batch_decompress_fmt_dev(const uint8_t* enc, size_t n, int out_format, uint8_t* out,
                                  uint8_t* ok) {
  D377_REQUIRE_READY();
  TRY(decompress_fmt_args(enc, n, out_format, out));
  if (n == 0) return D377_OK;
  launch_decompress(enc, n, out, ok, _eng.stream, out_format);
  D377_LAUNCHED();
  D377_CUDA(cudaGetLastError());
  return D377_OK;
}

static int compress_fmt_args(const uint8_t* points, int point_format, size_t n, const uint8_t* enc) {
  TRY(parse_format("d377_batch_compress_fmt", point_format, fmt_set(D377_PT_ELEMENT, D377_PT_AFFINE, D377_PT_XYZ),
                   nullptr));
  return n && (!enc || !points) ? null_pointer() : D377_OK;
}

int d377_batch_compress_fmt_dev(const uint8_t* points, int point_format, size_t n, uint8_t* enc) {
  D377_REQUIRE_READY();
  TRY(compress_fmt_args(points, point_format, n, enc));
  if (n == 0) return D377_OK;
  launch_compress(points, n, enc, _eng.stream, point_format);
  D377_LAUNCHED();
  D377_CUDA(cudaGetLastError());
  return D377_OK;
}

static int check_width(size_t w) {
  if (w == 0 || w > 256) { set_error("input width %zu out of range [1, 256] bytes", w); return D377_ERR_INVALID_ARG; }
  return D377_OK;
}

// encode_to_curve (r1) and hash_to_curve (r1, r2)
static int elligator_args(bool hash, const uint8_t* r1, const uint8_t* r2, size_t in_width, size_t n,
                          const uint8_t* out, int out_format) {
  TRY(parse_format(hash ? "d377_batch_hash_to_curve" : "d377_batch_encode_to_curve", out_format, kOutFormats,
                   nullptr));
  TRY(check_width(in_width));
  return n && (!r1 || (hash && !r2) || !out) ? null_pointer() : D377_OK;
}

int d377_batch_encode_to_curve_wide_dev(const uint8_t* r, size_t in_width, size_t n, uint8_t* out,
                                        int out_format) {
  D377_REQUIRE_READY();
  TRY(elligator_args(false, r, nullptr, in_width, n, out, out_format));
  if (n == 0) return D377_OK;
  launch_elligator(false, out_format == D377_OUT_ENCODING, r, nullptr, in_width, n, out, _eng.stream);
  D377_LAUNCHED();
  D377_CUDA(cudaGetLastError());
  return D377_OK;
}

int d377_batch_encode_to_curve_dev(const uint8_t* r, size_t n, uint8_t* out, int out_format) {
  return d377_batch_encode_to_curve_wide_dev(r, 32, n, out, out_format);
}

int d377_batch_hash_to_curve_wide_dev(const uint8_t* r1, const uint8_t* r2, size_t in_width, size_t n,
                                      uint8_t* out, int out_format) {
  D377_REQUIRE_READY();
  TRY(elligator_args(true, r1, r2, in_width, n, out, out_format));
  if (n == 0) return D377_OK;
  launch_elligator(true, out_format == D377_OUT_ENCODING, r1, r2, in_width, n, out, _eng.stream);
  D377_LAUNCHED();
  D377_CUDA(cudaGetLastError());
  return D377_OK;
}

int d377_batch_hash_to_curve_dev(const uint8_t* r1, const uint8_t* r2, size_t n, uint8_t* out,
                                 int out_format) {
  return d377_batch_hash_to_curve_wide_dev(r1, r2, 32, n, out, out_format);
}

static int from_le_bytes_args(const uint8_t* bytes, size_t in_width, size_t n, const uint8_t* out) {
  TRY(check_width(in_width));
  return n && (!bytes || !out) ? null_pointer() : D377_OK;
}

int d377_fq_batch_from_le_bytes_mod_order_dev(const uint8_t* bytes, size_t in_width, size_t n,
                                              uint8_t* out) {
  D377_REQUIRE_READY();
  TRY(from_le_bytes_args(bytes, in_width, n, out));
  if (n == 0) return D377_OK;
  k_fq_from_wide<<<grid_for(n, 128), 128, 0, _eng.stream>>>(bytes, in_width, n, out);
  D377_LAUNCHED();
  D377_CUDA(cudaGetLastError());
  return D377_OK;
}

// *pf, *sc_mont: the point format and the scalar form the format word carries
static int scalar_mul_args(const uint8_t* points, int point_format, const uint8_t* scalars, size_t n,
                           const uint8_t* out, int out_format, int* pf, bool* sc_mont) {
  TRY(parse_format("d377_batch_scalar_mul", point_format, kMulFormats, pf, sc_mont));
  TRY(parse_format("d377_batch_scalar_mul", out_format, kOutFormats, nullptr));
  return n && (!points || !scalars || !out) ? null_pointer() : D377_OK;
}

int d377_batch_scalar_mul_dev(const uint8_t* points, int point_format, const uint8_t* scalars,
                              size_t n, uint8_t* out, int out_format, uint8_t* ok) {
  D377_REQUIRE_READY();
  int pf = 0;
  bool sc_mont = false;
  TRY(scalar_mul_args(points, point_format, scalars, n, out, out_format, &pf, &sc_mont));
  if (n == 0) return D377_OK;
  if (sc_mont) TRY(canonical_scalars(_eng, scalars, n));
  launch_scalar_mul(pf, out_format == D377_OUT_ENCODING, points, scalars, n, out, ok, _eng.stream);
  D377_LAUNCHED();
  D377_CUDA(cudaGetLastError());
  return D377_OK;
}

// *of, *sc_mont: the output format and the scalar form the format word carries
static int fixed_base_args(const uint8_t* scalars, size_t n, const uint8_t* out, int out_format, int* of,
                           bool* sc_mont) {
  TRY(parse_format("d377_fixed_base_mul", out_format, kOutFormats, of, sc_mont));
  return n && (!scalars || !out) ? null_pointer() : D377_OK;
}

int d377_fixed_base_mul_dev(const uint8_t* scalars, size_t n, uint8_t* out, int out_format) {
  D377_REQUIRE_READY();
  int of = 0;
  bool sc_mont = false;
  TRY(fixed_base_args(scalars, n, out, out_format, &of, &sc_mont));
  if (n == 0) return D377_OK;
  Engine& e = _eng;
  TRY(ensure_fb_table());
  if (sc_mont) TRY(canonical_scalars(e, scalars, n));
  // The quartic table is 1.6 GB and takes ~0.15 s to build: only a batch large enough to
  // win that back builds it (or finds it built); smaller calls take the Edwards table +
  // compress, whose output is bit-identical.  The host-buffer entry point passes the size of
  // the whole batch through fb_batch_hint so that its chunks agree.
  constexpr size_t kFbQuarticMin = (size_t)1 << 18;
  const size_t batch = std::max(n, e.fb_batch_hint);
  bool quartic = of == D377_OUT_ENCODING && (e.fb_table_jq != nullptr || batch >= kFbQuarticMin);
  if (quartic && ensure_fb_table_jq() != D377_OK) {
    // no room for the quartic table: the Edwards path gives the same bytes
    cudaGetLastError();
    quartic = false;
  }
  launch_fixed_base(of == D377_OUT_ENCODING, e.fb_table, 1, quartic ? e.fb_table_jq : nullptr, scalars, n,
                    out, e.stream);
  D377_LAUNCHED();
  D377_CUDA(cudaGetLastError());
  return D377_OK;
}

// The table set must be a live set of fixed bases of this engine (checked before n = 0 is
// looked at; *k receives its size); n rows of k 32-byte scalars must stay addressable.
static int fixed_bases_mul_args(Engine& e, const uint8_t* tables, const uint8_t* scalars, size_t n,
                                const uint8_t* out, int out_format, size_t* k, int* of, bool* sc_mont) {
  TRY(parse_format("d377_fixed_bases_mul", out_format, kOutFormats, of, sc_mont));
  auto it = e.fixed_bases.find(tables);
  if (it == e.fixed_bases.end()) {
    set_error("d377_fixed_bases_mul: %p is not a live set of fixed bases of device %d", (const void*)tables,
              e.device);
    return D377_ERR_INVALID_ARG;
  }
  *k = it->second.k;
  if (n && (!scalars || !out)) return null_pointer();
  if (n > SIZE_MAX / 32 / *k) {
    set_error("fixed bases: %zu rows of %zu scalars overflow the address space", n, *k);
    return D377_ERR_INVALID_ARG;
  }
  return D377_OK;
}

int d377_fixed_bases_mul_dev(const uint8_t* tables, const uint8_t* scalars, size_t n, uint8_t* out, int out_format) {
  D377_REQUIRE_READY();
  Engine& e = _eng;
  size_t k = 0;
  int of = 0;
  bool sc_mont = false;
  TRY(fixed_bases_mul_args(e, tables, scalars, n, out, out_format, &k, &of, &sc_mont));
  if (n == 0) return D377_OK;
  if (sc_mont) TRY(canonical_scalars(e, scalars, n * k));
  launch_fixed_base(of == D377_OUT_ENCODING, tables, k, nullptr, scalars, n, out, e.stream);
  D377_LAUNCHED();
  D377_CUDA(cudaGetLastError());
  return D377_OK;
}

static int binop_dev(int op, const uint8_t* a, const uint8_t* b, size_t n, uint8_t* out) {
  D377_REQUIRE_READY();
  if (n == 0) return D377_OK;
  if (!a || (op < 2 && !b) || !out) { set_error("null pointer"); return D377_ERR_INVALID_ARG; }
  cudaStream_t st = _eng.stream;
  switch (op) {
    case 0: k_binop<0><<<grid_for(n, 128), 128, 0, st>>>(a, b, n, out); break;
    case 1: k_binop<1><<<grid_for(n, 128), 128, 0, st>>>(a, b, n, out); break;
    case 2: k_binop<2><<<grid_for(n, 128), 128, 0, st>>>(a, nullptr, n, out); break;
    default: k_binop<3><<<grid_for(n, 128), 128, 0, st>>>(a, nullptr, n, out); break;
  }
  D377_LAUNCHED();
  D377_CUDA(cudaGetLastError());
  return D377_OK;
}

int d377_batch_add_dev(const uint8_t* a, const uint8_t* b, size_t n, uint8_t* out) { return binop_dev(0, a, b, n, out); }
int d377_batch_sub_dev(const uint8_t* a, const uint8_t* b, size_t n, uint8_t* out) { return binop_dev(1, a, b, n, out); }
int d377_batch_neg_dev(const uint8_t* a, size_t n, uint8_t* out) { return binop_dev(2, a, nullptr, n, out); }
int d377_batch_double_dev(const uint8_t* a, size_t n, uint8_t* out) { return binop_dev(3, a, nullptr, n, out); }

int d377_batch_element_eq_dev(const uint8_t* a, const uint8_t* b, size_t n, uint8_t* eq) {
  D377_REQUIRE_READY();
  if (n == 0) return D377_OK;
  if (!a || !b || !eq) { set_error("null pointer"); return D377_ERR_INVALID_ARG; }
  k_eq<<<grid_for(n, 128), 128, 0, _eng.stream>>>(a, b, n, eq);
  D377_LAUNCHED();
  D377_CUDA(cudaGetLastError());
  return D377_OK;
}

int d377_batch_on_curve_dev(const uint8_t* elements, size_t n, int check_order, uint8_t* ok) {
  D377_REQUIRE_READY();
  if (n == 0) return D377_OK;
  if (!elements || !ok) { set_error("null pointer"); return D377_ERR_INVALID_ARG; }
  launch_on_curve(elements, n, check_order, ok, _eng.stream);
  D377_LAUNCHED();
  D377_CUDA(cudaGetLastError());
  return D377_OK;
}

int d377_element_sum_dev(const uint8_t* elements, size_t n, uint8_t* out_element,
                         uint8_t* out_encoding) {
  D377_REQUIRE_READY();
  if (n && !elements) { set_error("null pointer"); return D377_ERR_INVALID_ARG; }
  return element_sum_on(_eng, _eng.stream, elements, n, out_element, out_encoding);
}

int d377_element_sum_result_dev(const uint8_t* elements, size_t n, uint8_t* out_element,
                                uint8_t* out_encoding) {
  D377_REQUIRE_READY_NOJOIN();
  if (n && !elements) { set_error("null pointer"); return D377_ERR_INVALID_ARG; }
  return element_sum_on(_eng, result_stream(_eng), elements, n, out_element, out_encoding);
}

int d377_msm_dev(const uint8_t* scalars, const uint8_t* points, int point_format, size_t n,
                 uint8_t* out_element, uint8_t* out_encoding) {
  D377_REQUIRE_READY();
  return msm_dev(scalars, points, point_format, n, out_element, out_encoding);
}

int d377_msm_dev_async(const uint8_t* scalars, const uint8_t* points, int point_format, size_t n,
                       uint8_t* out_element, uint8_t* out_encoding, int flags) {
  D377_REQUIRE_READY_NOJOIN();
  return msm_dev_async(scalars, points, point_format, n, out_element, out_encoding, flags);
}

// ---- many independent small MSMs (Element::vartime_multiscalar_mul in a loop) -----------
// The host offsets of a segmented call (`who` names the entry point in the error text): at
// most 2^31 - 1 segments, offsets[0] = 0, non-decreasing.
static int segment_offsets_ok(const char* who, const uint32_t* offsets, size_t nmsm) {
  if (nmsm > 0x7fffffffull) { set_error("%s: too many segments", who); return D377_ERR_INVALID_ARG; }
  if (offsets[0] != 0) { set_error("%s: offsets[0] must be 0", who); return D377_ERR_INVALID_ARG; }
  for (size_t j = 0; j < nmsm; j++)
    if (offsets[j + 1] < offsets[j]) {
      set_error("%s: offsets must not decrease (segment %zu)", who, j);
      return D377_ERR_INVALID_ARG;
    }
  return D377_OK;
}

// Host-buffer form of a segmented call: the n scalars and points (format pf) go up into
// bm_sc / bm_pt, `run(scalars, points, out, ok)` enqueues the device-side call on the engine
// stream, and the nmsm results (and decode status, if wanted) come back.  Blocks until they
// have landed; on an error the streams are drained first.
using SegmentedRun = std::function<int(const uint8_t*, const uint8_t*, uint8_t*, uint8_t*)>;

static int staged_segments(Engine& e, const uint8_t* scalars, const uint8_t* points, int pf, size_t n, size_t nmsm,
                           uint8_t* out, int out_format, uint8_t* ok, const SegmentedRun& run) {
  const size_t pb = pt_bytes(pf), ob = out_bytes(out_format);
  TRY(ensure(e.bm_sc, n * 32 + 32));
  TRY(ensure(e.bm_pt, n * pb + 128));
  TRY(ensure(e.bm_out, nmsm * ob));
  TRY(ensure(e.bm_okout, nmsm + 16));
  auto body = [&]() -> int {
    if (n) {
      D377_CUDA(cudaMemcpyAsync(e.bm_sc.p, scalars, n * 32, cudaMemcpyHostToDevice, e.stream));
      D377_CUDA(cudaMemcpyAsync(e.bm_pt.p, points, n * pb, cudaMemcpyHostToDevice, e.stream));
    }
    TRY(run((const uint8_t*)e.bm_sc.p, (const uint8_t*)e.bm_pt.p, (uint8_t*)e.bm_out.p,
            ok ? (uint8_t*)e.bm_okout.p : nullptr));
    D377_CUDA(cudaMemcpyAsync(out, e.bm_out.p, nmsm * ob, cudaMemcpyDeviceToHost, e.stream));
    if (ok) D377_CUDA(cudaMemcpyAsync(ok, e.bm_okout.p, nmsm, cudaMemcpyDeviceToHost, e.stream));
    D377_CUDA(cudaStreamSynchronize(e.stream));
    return D377_OK;
  };
  int rc = body();
  if (rc) drain(e);
  return rc;
}

static int batch_msm_formats(int point_format, int out_format, int* pf, bool* sc_mont) {
  TRY(parse_format("d377_batch_msm", point_format, kMulFormats, pf, sc_mont));
  return parse_format("d377_batch_msm", out_format, kOutFormats, nullptr);
}

int d377_batch_msm_dev(const uint8_t* scalars, const uint8_t* points, int point_format,
                       const uint32_t* offsets, size_t nmsm, size_t n, uint8_t* out, int out_format,
                       uint8_t* ok) {
  D377_REQUIRE_READY();
  int pf = 0;
  bool sc_mont = false;
  TRY(batch_msm_formats(point_format, out_format, &pf, &sc_mont));
  if (nmsm == 0) return D377_OK;
  if (n > 0xfffffff0ull) { set_error("d377_batch_msm: too many pairs"); return D377_ERR_INVALID_ARG; }
  if (!offsets || !out || (n && (!scalars || !points))) { set_error("null pointer"); return D377_ERR_INVALID_ARG; }
  Engine& e = _eng;
  TRY(ensure(e.bm_prod, n * 128 + 128));
  TRY(ensure(e.bm_ok, n + 16));
  uint8_t* prod = (uint8_t*)e.bm_prod.p;
  uint8_t* okp = pf == D377_PT_ENCODING ? (uint8_t*)e.bm_ok.p : nullptr;
  if (n) {
    if (sc_mont) TRY(canonical_scalars(e, scalars, n));
    launch_scalar_mul(pf, false, points, scalars, n, prod, okp, e.stream);
    D377_LAUNCHED();
  }
  uint8_t* sums = out;
  if (out_format == D377_OUT_ENCODING) {
    TRY(ensure(e.bm_sum, nmsm * 128));
    sums = (uint8_t*)e.bm_sum.p;
  }
  launch_seg_sum(prod, okp, offsets, nmsm, sums, ok, e.stream);
  if (out_format == D377_OUT_ENCODING) {
    launch_compress(sums, nmsm, out, e.stream);
    D377_LAUNCHED();
  }
  D377_CUDA(cudaGetLastError());
  return D377_OK;
}

int d377_batch_msm(const uint8_t* scalars, const uint8_t* points, int point_format, const uint32_t* offsets,
                   size_t nmsm, uint8_t* out, int out_format, uint8_t* ok) {
  D377_REQUIRE_READY();
  int pf = 0;
  bool sc_mont = false;
  TRY(batch_msm_formats(point_format, out_format, &pf, &sc_mont));
  if (nmsm == 0) return D377_OK;
  if (!offsets || !out) { set_error("null pointer"); return D377_ERR_INVALID_ARG; }
  TRY(segment_offsets_ok("d377_batch_msm", offsets, nmsm));
  const size_t n = offsets[nmsm];
  if (n && (!scalars || !points)) { set_error("null pointer"); return D377_ERR_INVALID_ARG; }
  Engine& e = _eng;
  TRY(ensure(e.bm_off, (nmsm + 1) * 4));
  return staged_segments(e, scalars, points, pf, n, nmsm, out, out_format, ok,
                         [&](const uint8_t* sc, const uint8_t* pt, uint8_t* dout, uint8_t* dok) -> int {
                           D377_CUDA(cudaMemcpyAsync(e.bm_off.p, offsets, (nmsm + 1) * 4, cudaMemcpyHostToDevice,
                                                     e.stream));
                           return d377_batch_msm_dev(sc, pt, point_format, (const uint32_t*)e.bm_off.p, nmsm, n, dout,
                                                     out_format, dok);
                         });
}

// ---- many independent MSMs in one segmented Pippenger ---------------------------------------
// Both forms: formats, null pointers (n = offsets[nmsm]), the host offsets (offsets[0] = 0,
// non-decreasing, n <= 0xfffffff0) and the window width.  Nothing is read or launched before
// this passes; nmsm = 0 passes with nothing else checked but the formats.
static int msm_segmented_args(Engine& e, const uint8_t* scalars, const uint8_t* points, int point_format,
                              const uint32_t* offsets, size_t nmsm, const uint8_t* out, int out_format, int* pf,
                              bool* sc_mont, int* c) {
  TRY(parse_format("d377_msm_segmented", point_format, kPointFormats, pf, sc_mont));
  TRY(parse_format("d377_msm_segmented", out_format, kOutFormats, nullptr));
  if (nmsm == 0) return D377_OK;
  if (!offsets || !out) return null_pointer();
  TRY(segment_offsets_ok("d377_msm_segmented", offsets, nmsm));
  const size_t n = offsets[nmsm];
  if (n > 0xfffffff0ull) { set_error("d377_msm_segmented: too many pairs"); return D377_ERR_INVALID_ARG; }
  if (n && (!scalars || !points)) return null_pointer();
  return msm_segmented_width(e, *pf, offsets, nmsm, c);
}

int d377_msm_segmented_dev(const uint8_t* scalars, const uint8_t* points, int point_format, const uint32_t* offsets,
                           size_t nmsm, uint8_t* out, int out_format, uint8_t* ok) {
  D377_REQUIRE_READY();
  int pf = 0, c = 0;
  bool sc_mont = false;
  TRY(msm_segmented_args(_eng, scalars, points, point_format, offsets, nmsm, out, out_format, &pf, &sc_mont, &c));
  if (nmsm == 0) return D377_OK;
  return msm_segmented_enqueue(scalars, points, pf, sc_mont, offsets, nmsm, c, out, out_format, ok);
}

int d377_msm_segmented(const uint8_t* scalars, const uint8_t* points, int point_format, const uint32_t* offsets,
                       size_t nmsm, uint8_t* out, int out_format, uint8_t* ok) {
  D377_REQUIRE_READY();
  Engine& e = _eng;
  int pf = 0, c = 0;
  bool sc_mont = false;
  TRY(msm_segmented_args(e, scalars, points, point_format, offsets, nmsm, out, out_format, &pf, &sc_mont, &c));
  if (nmsm == 0) return D377_OK;
  return staged_segments(e, scalars, points, pf, offsets[nmsm], nmsm, out, out_format, ok,
                         [&](const uint8_t* sc, const uint8_t* pt, uint8_t* dout, uint8_t* dok) {
                           return msm_segmented_enqueue(sc, pt, pf, sc_mont, offsets, nmsm, c, dout, out_format, dok);
                         });
}

int d377_msm_segmented_last(int* c, int* windows, size_t* chunks) {
  D377_REQUIRE_READY();
  return msm_segmented_last(c, windows, chunks);
}

int d377_batch_normalize_dev(const uint8_t* elements, size_t n, uint8_t* affine) {
  D377_REQUIRE_READY();
  if (n == 0) return D377_OK;
  if (!elements || !affine) { set_error("null pointer"); return D377_ERR_INVALID_ARG; }
  Engine& e = _eng;
  int rc = ensure(e.scratch, n * 32);
  if (rc) return rc;
  launch_normalize(elements, n, (uint8_t*)e.scratch.p, affine, e.stream);
  D377_LAUNCHED();
  D377_CUDA(cudaGetLastError());
  return D377_OK;
}

int d377_fq_batch_sqrt_ratio_zeta_dev(const uint8_t* num, const uint8_t* den, size_t n, uint8_t* out,
                                      uint8_t* was_square) {
  D377_REQUIRE_READY();
  if (n == 0) return D377_OK;
  if (!num || !den || !out || !was_square) { set_error("null pointer"); return D377_ERR_INVALID_ARG; }
  launch_fq_sqrt_ratio(num, den, n, out, was_square, _eng.stream);
  D377_LAUNCHED();
  D377_CUDA(cudaGetLastError());
  return D377_OK;
}

int d377_fq_batch_isqrt_dev(const uint8_t* x, size_t n, uint8_t* out, uint8_t* was_square) {
  D377_REQUIRE_READY();
  if (n == 0) return D377_OK;
  if (!x || !out || !was_square) { set_error("null pointer"); return D377_ERR_INVALID_ARG; }
  launch_fq_isqrt(x, n, out, was_square, _eng.stream);
  D377_LAUNCHED();
  D377_CUDA(cudaGetLastError());
  return D377_OK;
}

static int deserialize_args(int field, const uint8_t* bytes, size_t n, const uint8_t* ok) {
  if (field != 0 && field != 1) { set_error("field must be 0 (Fq) or 1 (Fr)"); return D377_ERR_INVALID_ARG; }
  return n && (!bytes || !ok) ? null_pointer() : D377_OK;
}

int d377_field_batch_deserialize_dev(int field, const uint8_t* bytes, size_t n, uint8_t* out, uint8_t* ok) {
  D377_REQUIRE_READY();
  TRY(deserialize_args(field, bytes, n, ok));
  if (n == 0) return D377_OK;
  Engine& e = _eng;
  if (field == 0)
    k_field_deserialize<0><<<grid_for(n, 256), 256, 0, e.stream>>>(bytes, n, out, ok);
  else
    k_field_deserialize<1><<<grid_for(n, 256), 256, 0, e.stream>>>(bytes, n, out, ok);
  D377_LAUNCHED();
  D377_CUDA(cudaGetLastError());
  return D377_OK;
}

// ---- host-pointer entry points -------------------------------------------
// The batch is cut into chunks that flow through two sets of device staging
// buffers: chunk k+1 goes up on the copy stream while chunk k is computed on the
// engine stream and chunk k-1 comes back on the out stream, so a call costs about
// max(H2D, kernel, D2H) instead of their sum (pinned host memory assumed; pageable
// buffers still work, the driver then stages the copies itself).  The call blocks
// until the last result byte has landed.

}  // extern "C"

namespace d377 {

struct HostIn { const uint8_t* h; size_t w; };
struct HostOut { uint8_t* h; size_t w; };

// Chunks of 2^18 elements (>= 3 full waves of the one-element-per-thread kernels, 8-32 MB
// per transfer); a batch below 2^19 runs as one chunk, because a kernel over less than a
// wave costs the same time as over a full one and the transfers are then negligible.
// From 2^24 elements the chunks are 2^20 (still >= 16 of them): the fixed-base kernel with its
// four elements per thread and one inversion per CTA needs several waves per launch to keep
// the multiply pipe busy across its barrier (e2e 274 -> 382 Melem/s at 2^24); smaller batches
// keep 2^18 so that the pipeline has enough stages to overlap (4 chunks of 2^20 at 2^22 cost
// compress / decompress 12 % end to end).
static size_t pipe_chunk(size_t n) {
  if (n >= ((size_t)1 << 24)) return (size_t)1 << 20;
  return n >= ((size_t)1 << 19) ? (size_t)1 << 18 : n;
}

// launch(din, dout, len) enqueues the kernel(s) of one chunk on the engine stream.
template <class Launch>
static int run_pipelined_inner(size_t n, const HostIn* ins, int nin, const HostOut* outs, int nout,
                               Launch&& launch) {
  Engine& e = engine();
  const size_t chunk = pipe_chunk(n);
  for (int b = 0; b < 2; b++) {
    for (int i = 0; i < nin; i++) TRY(ensure(e.st_in[b][i], chunk * ins[i].w));
    for (int j = 0; j < nout; j++) TRY(ensure(e.st_out[b][j], chunk * outs[j].w));
  }
  size_t k = 0;
  for (size_t lo = 0; lo < n; lo += chunk, k++) {
    const int b = (int)(k & 1);
    const size_t len = std::min(chunk, n - lo);
    uint8_t* din[3] = {nullptr, nullptr, nullptr};
    uint8_t* dout[2] = {nullptr, nullptr};
    // inputs of buffer set b are free once the kernel of chunk k-2 has run
    if (k >= 2) D377_CUDA(cudaStreamWaitEvent(e.copy_stream, e.pe_k[b], 0));
    for (int i = 0; i < nin; i++) {
      din[i] = (uint8_t*)e.st_in[b][i].p;
      D377_CUDA(cudaMemcpyAsync(din[i], ins[i].h + lo * ins[i].w, len * ins[i].w,
                                cudaMemcpyHostToDevice, e.copy_stream));
    }
    D377_CUDA(cudaEventRecord(e.pe_in[b], e.copy_stream));
    D377_CUDA(cudaStreamWaitEvent(e.stream, e.pe_in[b], 0));
    // outputs of buffer set b are free once chunk k-2 has been copied back
    if (k >= 2) D377_CUDA(cudaStreamWaitEvent(e.stream, e.pe_out[b], 0));
    for (int j = 0; j < nout; j++) dout[j] = (uint8_t*)e.st_out[b][j].p;
    TRY(launch(din, dout, len));
    D377_CUDA(cudaEventRecord(e.pe_k[b], e.stream));
    D377_CUDA(cudaStreamWaitEvent(e.out_stream, e.pe_k[b], 0));
    for (int j = 0; j < nout; j++) {
      if (!outs[j].h) continue;
      D377_CUDA(cudaMemcpyAsync(outs[j].h + lo * outs[j].w, dout[j], len * outs[j].w,
                                cudaMemcpyDeviceToHost, e.out_stream));
    }
    D377_CUDA(cudaEventRecord(e.pe_out[b], e.out_stream));
  }
  D377_CUDA(cudaStreamSynchronize(e.out_stream));
  D377_CUDA(cudaStreamSynchronize(e.stream));
  return D377_OK;
}

template <class Launch>
static int run_pipelined(size_t n, const HostIn* ins, int nin, const HostOut* outs, int nout,
                         Launch&& launch) {
  int rc = run_pipelined_inner(n, ins, nin, outs, nout, launch);
  // a failure in the middle of the pipeline leaves copies in flight: wait for them before
  // the caller is told that its buffers are its own again
  if (rc) drain(engine());
  return rc;
}

}  // namespace d377

extern "C" {

int d377_batch_decompress(const uint8_t* enc, size_t n, uint8_t* elements, uint8_t* ok) {
  D377_REQUIRE_READY();
  if (n == 0) return D377_OK;
  if (!enc || !elements) { set_error("null pointer"); return D377_ERR_INVALID_ARG; }
  HostIn ins[] = {{enc, 32}};
  HostOut outs[] = {{elements, 128}, {ok, 1}};
  return run_pipelined(n, ins, 1, outs, 2, [&](uint8_t* const* di, uint8_t* const* dout, size_t len) {
    return d377_batch_decompress_dev(di[0], len, dout[0], dout[1]);
  });
}

int d377_batch_compress(const uint8_t* elements, size_t n, uint8_t* enc) {
  D377_REQUIRE_READY();
  if (n == 0) return D377_OK;
  if (!enc || !elements) { set_error("null pointer"); return D377_ERR_INVALID_ARG; }
  HostIn ins[] = {{elements, 128}};
  HostOut outs[] = {{enc, 32}};
  return run_pipelined(n, ins, 1, outs, 1, [&](uint8_t* const* di, uint8_t* const* dout, size_t len) {
    return d377_batch_compress_dev(di[0], len, dout[0]);
  });
}

int d377_batch_decompress_fmt(const uint8_t* enc, size_t n, int out_format, uint8_t* out,
                              uint8_t* ok) {
  D377_REQUIRE_READY();
  TRY(decompress_fmt_args(enc, n, out_format, out));
  if (n == 0) return D377_OK;
  HostIn ins[] = {{enc, pt_bytes(D377_PT_ENCODING)}};
  HostOut outs[] = {{out, pt_bytes(out_format)}, {ok, 1}};
  return run_pipelined(n, ins, 1, outs, 2, [&](uint8_t* const* di, uint8_t* const* dout, size_t len) {
    return d377_batch_decompress_fmt_dev(di[0], len, out_format, dout[0], dout[1]);
  });
}

int d377_batch_compress_fmt(const uint8_t* points, int point_format, size_t n, uint8_t* enc) {
  D377_REQUIRE_READY();
  TRY(compress_fmt_args(points, point_format, n, enc));
  if (n == 0) return D377_OK;
  HostIn ins[] = {{points, pt_bytes(point_format)}};
  HostOut outs[] = {{enc, pt_bytes(D377_PT_ENCODING)}};
  return run_pipelined(n, ins, 1, outs, 1, [&](uint8_t* const* di, uint8_t* const* dout, size_t len) {
    return d377_batch_compress_fmt_dev(di[0], point_format, len, dout[0]);
  });
}

int d377_batch_encode_to_curve_wide(const uint8_t* r, size_t in_width, size_t n, uint8_t* out,
                                    int out_format) {
  D377_REQUIRE_READY();
  TRY(elligator_args(false, r, nullptr, in_width, n, out, out_format));
  if (n == 0) return D377_OK;
  HostIn ins[] = {{r, in_width}};
  HostOut outs[] = {{out, out_bytes(out_format)}};
  return run_pipelined(n, ins, 1, outs, 1, [&](uint8_t* const* di, uint8_t* const* dout, size_t len) {
    return d377_batch_encode_to_curve_wide_dev(di[0], in_width, len, dout[0], out_format);
  });
}

int d377_batch_encode_to_curve(const uint8_t* r, size_t n, uint8_t* out, int out_format) {
  return d377_batch_encode_to_curve_wide(r, 32, n, out, out_format);
}

int d377_batch_hash_to_curve_wide(const uint8_t* r1, const uint8_t* r2, size_t in_width, size_t n,
                                  uint8_t* out, int out_format) {
  D377_REQUIRE_READY();
  TRY(elligator_args(true, r1, r2, in_width, n, out, out_format));
  if (n == 0) return D377_OK;
  HostIn ins[] = {{r1, in_width}, {r2, in_width}};
  HostOut outs[] = {{out, out_bytes(out_format)}};
  return run_pipelined(n, ins, 2, outs, 1, [&](uint8_t* const* di, uint8_t* const* dout, size_t len) {
    return d377_batch_hash_to_curve_wide_dev(di[0], di[1], in_width, len, dout[0], out_format);
  });
}

int d377_batch_hash_to_curve(const uint8_t* r1, const uint8_t* r2, size_t n, uint8_t* out,
                             int out_format) {
  return d377_batch_hash_to_curve_wide(r1, r2, 32, n, out, out_format);
}

int d377_fq_batch_from_le_bytes_mod_order(const uint8_t* bytes, size_t in_width, size_t n, uint8_t* out) {
  D377_REQUIRE_READY();
  TRY(from_le_bytes_args(bytes, in_width, n, out));
  if (n == 0) return D377_OK;
  HostIn ins[] = {{bytes, in_width}};
  HostOut outs[] = {{out, 32}};
  return run_pipelined(n, ins, 1, outs, 1, [&](uint8_t* const* di, uint8_t* const* dout, size_t len) {
    return d377_fq_batch_from_le_bytes_mod_order_dev(di[0], in_width, len, dout[0]);
  });
}

int d377_batch_scalar_mul(const uint8_t* points, int point_format, const uint8_t* scalars,
                          size_t n, uint8_t* out, int out_format, uint8_t* ok) {
  D377_REQUIRE_READY();
  int pf = 0;
  bool sc_mont = false;
  TRY(scalar_mul_args(points, point_format, scalars, n, out, out_format, &pf, &sc_mont));
  if (n == 0) return D377_OK;
  HostIn ins[] = {{points, pt_bytes(pf)}, {scalars, 32}};
  HostOut outs[] = {{out, out_bytes(out_format)}, {ok, 1}};
  return run_pipelined(n, ins, 2, outs, 2, [&](uint8_t* const* di, uint8_t* const* dout, size_t len) {
    // only encodings can fail to decode; every other format is always Ok
    D377_CUDA(cudaMemsetAsync(dout[1], 1, len, engine().stream));
    return d377_batch_scalar_mul_dev(di[0], point_format, di[1], len, dout[0], out_format, dout[1]);
  });
}

int d377_fixed_base_mul(const uint8_t* scalars, size_t n, uint8_t* out, int out_format) {
  D377_REQUIRE_READY();
  int of = 0;
  bool sc_mont = false;
  TRY(fixed_base_args(scalars, n, out, out_format, &of, &sc_mont));
  if (n == 0) return D377_OK;
  HostIn ins[] = {{scalars, 32}};
  HostOut outs[] = {{out, out_bytes(of)}};
  _eng.fb_batch_hint = n;
  int rc = run_pipelined(n, ins, 1, outs, 1, [&](uint8_t* const* di, uint8_t* const* dout, size_t len) {
    return d377_fixed_base_mul_dev(di[0], len, dout[0], out_format);
  });
  _eng.fb_batch_hint = 0;
  return rc;
}

int d377_fixed_bases_mul(const uint8_t* tables, const uint8_t* scalars, size_t n, uint8_t* out, int out_format) {
  D377_REQUIRE_READY();
  size_t k = 0;
  int of = 0;
  bool sc_mont = false;
  TRY(fixed_bases_mul_args(_eng, tables, scalars, n, out, out_format, &k, &of, &sc_mont));
  if (n == 0) return D377_OK;
  HostIn ins[] = {{scalars, 32 * k}};
  HostOut outs[] = {{out, out_bytes(of)}};
  return run_pipelined(n, ins, 1, outs, 1, [&](uint8_t* const* di, uint8_t* const* dout, size_t len) {
    return d377_fixed_bases_mul_dev(tables, di[0], len, dout[0], out_format);
  });
}

static int binop_host(int op, const uint8_t* a, const uint8_t* b, size_t n, uint8_t* out) {
  D377_REQUIRE_READY();
  if (n == 0) return D377_OK;
  if (!a || (op < 2 && !b) || !out) { set_error("null pointer"); return D377_ERR_INVALID_ARG; }
  HostIn ins[] = {{a, 128}, {b, 128}};
  HostOut outs[] = {{out, 128}};
  return run_pipelined(n, ins, op < 2 ? 2 : 1, outs, 1, [&](uint8_t* const* di, uint8_t* const* dout, size_t len) {
    return binop_dev(op, di[0], op < 2 ? di[1] : nullptr, len, dout[0]);
  });
}

int d377_batch_add(const uint8_t* a, const uint8_t* b, size_t n, uint8_t* out) { return binop_host(0, a, b, n, out); }
int d377_batch_sub(const uint8_t* a, const uint8_t* b, size_t n, uint8_t* out) { return binop_host(1, a, b, n, out); }
int d377_batch_neg(const uint8_t* a, size_t n, uint8_t* out) { return binop_host(2, a, nullptr, n, out); }
int d377_batch_double(const uint8_t* a, size_t n, uint8_t* out) { return binop_host(3, a, nullptr, n, out); }

int d377_batch_element_eq(const uint8_t* a, const uint8_t* b, size_t n, uint8_t* eq) {
  D377_REQUIRE_READY();
  if (n == 0) return D377_OK;
  if (!a || !b || !eq) { set_error("null pointer"); return D377_ERR_INVALID_ARG; }
  HostIn ins[] = {{a, 128}, {b, 128}};
  HostOut outs[] = {{eq, 1}};
  return run_pipelined(n, ins, 2, outs, 1, [&](uint8_t* const* di, uint8_t* const* dout, size_t len) {
    return d377_batch_element_eq_dev(di[0], di[1], len, dout[0]);
  });
}

int d377_batch_on_curve(const uint8_t* elements, size_t n, int check_order, uint8_t* ok) {
  D377_REQUIRE_READY();
  if (n == 0) return D377_OK;
  if (!elements || !ok) { set_error("null pointer"); return D377_ERR_INVALID_ARG; }
  HostIn ins[] = {{elements, 128}};
  HostOut outs[] = {{ok, 1}};
  return run_pipelined(n, ins, 1, outs, 1, [&](uint8_t* const* di, uint8_t* const* dout, size_t len) {
    return d377_batch_on_curve_dev(di[0], len, check_order, dout[0]);
  });
}

#define H2D(dst, src, bytes) D377_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, e.stream))
#define D2H(dst, src, bytes) D377_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, e.stream))

static int small_results_back(uint8_t* out_element, uint8_t* out_encoding) {
  Engine& e = engine();
  D2H(e.h_small, e.d_small, 160);
  D377_CUDA(cudaStreamSynchronize(e.stream));
  if (out_element) memcpy(out_element, e.h_small, 128);
  if (out_encoding) memcpy(out_encoding, e.h_small + 128, 32);
  return D377_OK;
}

int d377_element_sum(const uint8_t* elements, size_t n, uint8_t out_element[128],
                     uint8_t out_encoding[32]) {
  D377_REQUIRE_READY();
  if (n && !elements) { set_error("null pointer"); return D377_ERR_INVALID_ARG; }
  Engine& e = _eng;
  TRY(ensure(e.in0, n * 128 + 128));
  if (n) H2D(e.in0.p, elements, n * 128);
  int rc = element_sum_on(e, e.stream, (uint8_t*)e.in0.p, n, e.d_small, e.d_small + 128);
  if (rc) { drain(e); return rc; }
  return small_results_back(out_element, out_encoding);
}

// d377_msm_bases_create* (windowed = false: a plain set, c = 0, W = 1) and
// d377_msm_bases_create_windowed* (windowed = true, c = 0: the width is chosen from n).  Every
// argument is checked before anything is allocated or read.  `host`: `points` is host memory,
// uploaded once the set is allocated.
static int msm_bases_create(const uint8_t* points, int point_format, size_t n, bool windowed, int c,
                            uint8_t** bases, bool host) {
  Engine& e = engine();
  int fmt = 0, W = 1;
  TRY(parse_format("d377_msm_bases_create", point_format, kPointFormats, &fmt));
  if (!bases || (n && !points)) return null_pointer();
  if (windowed) {
    if (c != 0 && (c < 4 || c > 22)) { set_error("window width %d out of range [4, 22]", c); return D377_ERR_INVALID_ARG; }
    if (c == 0) c = msm_windowed_c(n);
    W = (252 + c - 1) / c;
    // the scatter stores a record index and a sign bit in 32 bits
    if ((double)n * (double)W >= 2147483648.0) {
      set_error("windowed bases: n * W = %zu * %d records reach 2^31", n, W);
      return D377_ERR_INVALID_ARG;
    }
  } else {
    c = 0;
  }
  const size_t bytes = (n * (size_t)W + 1) * pt_bytes(D377_PT_BASES);
  uint8_t* tab = nullptr;
  cudaError_t ce = cudaMalloc(&tab, bytes);
  if (ce != cudaSuccess) {
    cudaGetLastError();
    set_error("msm bases: cannot allocate %zu bytes of device memory (%s)", bytes, cudaGetErrorString(ce));
    return D377_ERR_CUDA;
  }
  int rc = D377_OK;
  uint8_t* tmp = nullptr;
  if (host) {
    ce = cudaMalloc(&tmp, n * pt_bytes(fmt) + 128);
    if (ce == cudaSuccess) ce = cudaMemcpyAsync(tmp, points, n * pt_bytes(fmt), cudaMemcpyHostToDevice, e.stream);
    if (ce != cudaSuccess) rc = cuda_fail(ce, "upload of the bases", __FILE__, __LINE__);
  }
  // slab 0 = the plain set (synchronises the stream), then the upper slabs of a windowed set
  if (!rc) rc = msm_bases_prepare(host ? tmp : points, fmt, n, tab);
  if (!rc) rc = msm_bases_fill_windows(tab, n, c, W);
  if (rc) cudaStreamSynchronize(e.stream);
  if (tmp) cudaFree(tmp);
  if (rc) {
    cudaFree(tab);
    return rc;
  }
  BasesLayout bl;
  bl.n = n;
  bl.c = c;
  bl.W = W;
  bl.bytes = bytes;
  e.bases[tab] = bl;
  *bases = tab;
  return D377_OK;
}

int d377_msm_bases_create(const uint8_t* points, int point_format, size_t n, uint8_t** bases) {
  D377_REQUIRE_READY();
  return msm_bases_create(points, point_format, n, false, 0, bases, true);
}

int d377_msm_bases_create_dev(const uint8_t* points, int point_format, size_t n, uint8_t** bases) {
  D377_REQUIRE_READY();
  return msm_bases_create(points, point_format, n, false, 0, bases, false);
}

int d377_msm_bases_create_windowed(const uint8_t* points, int point_format, size_t n, int c, uint8_t** bases) {
  D377_REQUIRE_READY();
  return msm_bases_create(points, point_format, n, true, c, bases, true);
}

int d377_msm_bases_create_windowed_dev(const uint8_t* points, int point_format, size_t n, int c, uint8_t** bases) {
  D377_REQUIRE_READY();
  return msm_bases_create(points, point_format, n, true, c, bases, false);
}

int d377_msm_bases_info(const uint8_t* bases, size_t* n, int* c, int* windows, size_t* bytes) {
  D377_REQUIRE_READY_NOJOIN();
  auto it = _eng.bases.find(bases);
  if (it == _eng.bases.end()) {
    set_error("d377_msm_bases_info: %p is not a live set of prepared bases of device %d", (const void*)bases, _eng.device);
    return D377_ERR_INVALID_ARG;
  }
  if (n) *n = it->second.n;
  if (c) *c = it->second.c;
  if (windows) *windows = it->second.W;
  if (bytes) *bytes = it->second.bytes;
  return D377_OK;
}

int d377_msm_last_windowed(int* windowed) {
  D377_REQUIRE_READY();
  if (!windowed) { set_error("null pointer"); return D377_ERR_INVALID_ARG; }
  *windowed = msm_last_windowed() ? 1 : 0;
  return D377_OK;
}

int d377_msm_bases_destroy(uint8_t* bases) {
  if (!bases) return D377_OK;
  D377_REQUIRE_READY();
  Engine& e = _eng;
  auto it = e.bases.find(bases);
  if (it == e.bases.end()) {
    set_error("d377_msm_bases_destroy: %p is not a live set of prepared bases of device %d", (void*)bases, e.device);
    return D377_ERR_INVALID_ARG;
  }
  D377_CUDA(cudaStreamSynchronize(e.stream));
  e.bases.erase(it);
  D377_CUDA(cudaFree(bases));
  return D377_OK;
}

// ---- prepared fixed bases ----------------------------------------------------
// Arguments of d377_fixed_bases_create*, checked before anything is allocated or read;
// *fmt receives the point format, *bytes the size of the k tables.
static int fixed_bases_args(int point_format, size_t k, uint8_t** tables, const uint8_t* points, int* fmt,
                            size_t* bytes) {
  TRY(parse_format("d377_fixed_bases_create", point_format, kPointFormats, fmt));
  if (!tables || !points) return null_pointer();
  if (k == 0) { set_error("fixed bases: k = 0"); return D377_ERR_INVALID_ARG; }
  const size_t per = fixed_bases_bytes_per_base();
  if (k > SIZE_MAX / per) {
    set_error("fixed bases: %zu tables of %zu bytes overflow the address space", k, per);
    return D377_ERR_INVALID_ARG;
  }
  *bytes = k * per;
  return D377_OK;
}

// `host`: `points` is host memory, uploaded once the tables are allocated
static int fixed_bases_create(const uint8_t* points, int point_format, size_t k, uint8_t** tables, bool host) {
  Engine& e = engine();
  int fmt = 0;
  size_t bytes = 0;
  TRY(fixed_bases_args(point_format, k, tables, points, &fmt, &bytes));
  uint8_t* tab = nullptr;
  cudaError_t ce = cudaMalloc(&tab, bytes);
  if (ce != cudaSuccess) {
    cudaGetLastError();
    set_error("fixed bases: cannot allocate %zu bytes of device memory (%s)", bytes, cudaGetErrorString(ce));
    return D377_ERR_CUDA;
  }
  int rc = D377_OK;
  uint8_t* tmp = nullptr;
  if (host) {
    ce = cudaMalloc(&tmp, k * pt_bytes(fmt));
    if (ce == cudaSuccess) ce = cudaMemcpyAsync(tmp, points, k * pt_bytes(fmt), cudaMemcpyHostToDevice, e.stream);
    if (ce != cudaSuccess) rc = cuda_fail(ce, "upload of the fixed bases", __FILE__, __LINE__);
  }
  if (!rc) rc = fixed_bases_fill(host ? tmp : points, fmt, k, tab);   // synchronises the stream
  if (rc) cudaStreamSynchronize(e.stream);
  if (tmp) cudaFree(tmp);
  if (rc) {
    cudaFree(tab);
    return rc;
  }
  FixedBasesInfo info;
  info.k = k;
  info.bytes = bytes;
  e.fixed_bases[tab] = info;
  *tables = tab;
  return D377_OK;
}

int d377_fixed_bases_create(const uint8_t* points, int point_format, size_t k, uint8_t** tables) {
  D377_REQUIRE_READY();
  return fixed_bases_create(points, point_format, k, tables, true);
}

int d377_fixed_bases_create_dev(const uint8_t* points, int point_format, size_t k, uint8_t** tables) {
  D377_REQUIRE_READY();
  return fixed_bases_create(points, point_format, k, tables, false);
}

int d377_fixed_bases_info(const uint8_t* tables, size_t* k, size_t* bytes) {
  D377_REQUIRE_READY_NOJOIN();
  auto it = _eng.fixed_bases.find(tables);
  if (it == _eng.fixed_bases.end()) {
    set_error("d377_fixed_bases_info: %p is not a live set of fixed bases of device %d", (const void*)tables, _eng.device);
    return D377_ERR_INVALID_ARG;
  }
  if (k) *k = it->second.k;
  if (bytes) *bytes = it->second.bytes;
  return D377_OK;
}

int d377_fixed_bases_destroy(uint8_t* tables) {
  if (!tables) return D377_OK;
  D377_REQUIRE_READY();
  Engine& e = _eng;
  auto it = e.fixed_bases.find(tables);
  if (it == e.fixed_bases.end()) {
    set_error("d377_fixed_bases_destroy: %p is not a live set of fixed bases of device %d", (void*)tables, e.device);
    return D377_ERR_INVALID_ARG;
  }
  D377_CUDA(cudaStreamSynchronize(e.stream));
  e.fixed_bases.erase(it);
  D377_CUDA(cudaFree(tables));
  return D377_OK;
}

}  // extern "C"

namespace d377 {
// D377_PT_BASES: `points` must be a live handle of this engine holding at least n bases
int check_bases(Engine& e, const uint8_t* points, size_t n, BasesLayout* layout) {
  auto it = e.bases.find(points);
  if (it == e.bases.end()) {
    set_error("msm: D377_PT_BASES needs the pointer d377_msm_bases_create returned (on device %d)", e.device);
    return D377_ERR_INVALID_ARG;
  }
  if (n > it->second.n) {
    set_error("msm: %zu scalars for %zu prepared bases", n, it->second.n);
    return D377_ERR_INVALID_ARG;
  }
  if (layout) *layout = it->second;
  return D377_OK;
}
}  // namespace d377

extern "C" {

static int msm_submit_inner(Engine& e, const uint8_t* scalars, const uint8_t* points, int point_format,
                            bool sc_mont, size_t n, int slot) {
  const bool prepared = point_format == D377_PT_BASES;
  size_t pb = pt_bytes(point_format);
  TRY(ensure(e.slot_sc[slot], n * 32 + 32));
  if (!prepared) TRY(ensure(e.slot_pt[slot], n * pb + 128));
  uint8_t* dres = e.d_small + kSmallSlots + 256 * slot;
  // Inputs go up on the copy stream, cut into sub-MSM chunks: the Pippenger of chunk k
  // (engine stream) overlaps the upload of chunk k+1, and the uploads of this slot
  // overlap whatever the other slot is computing.  Chunks stay >= 2^21 pairs so that
  // the window width (and with it the work per point) barely changes.
  size_t nch = 1;
  while (nch < 4 && n / (nch * 2) >= ((size_t)1 << 21)) nch *= 2;
  // With the other slot still in flight this upload already overlaps that MSM's kernels,
  // and one big Pippenger is cheaper than several small ones (wider windows, one tail) --
  // unless the call is bound by the link anyway (measured on B200: 55 GB/s H2D, ~0.5 G
  // pairs/s of Pippenger), where sub-chunks still shorten the drain of the pipeline.
  bool other_busy = false;
  for (int k = 0; k < Engine::kSlots; k++) other_busy = other_busy || (k != slot && e.slot_busy[k]);
  if (other_busy && (double)n * (double)((prepared ? 0 : pb) + 32) / 55e9 < (double)n / 0.5e9) nch = 1;
  if (e.msm_host_chunks_override > 0) nch = (size_t)e.msm_host_chunks_override;
  if (nch > (size_t)Engine::kMsmHostChunks) nch = Engine::kMsmHostChunks;
  size_t chunk = n ? ((n + nch - 1) / nch + 255) / 256 * 256 : 1;
  nch = n ? (n + chunk - 1) / chunk : 1;
  // The status word is reset on the copy stream, ahead of the first chunk event: the scalar
  // side of this MSM (which sets it) depends on the chunk events only, not on the engine
  // stream.  The slot's previous MSM has been waited for, so nobody else uses the word.
  D377_CUDA(cudaMemsetAsync(dres + 192, 0, 4, e.copy_stream));
  for (size_t k = 0; k < nch; k++) {
    if (n) {
      size_t lo = k * chunk, len = std::min(chunk, n - lo);
      D377_CUDA(cudaMemcpyAsync((uint8_t*)e.slot_sc[slot].p + lo * 32, scalars + lo * 32, len * 32,
                                cudaMemcpyHostToDevice, e.copy_stream));
      // the scalars go first and get an event of their own: the counting sort of this chunk
      // starts on it, while the (4x larger) points are still on the link
      D377_CUDA(cudaEventRecord(e.ev_chunk_sc[slot][k], e.copy_stream));
      if (!prepared)
        D377_CUDA(cudaMemcpyAsync((uint8_t*)e.slot_pt[slot].p + lo * pb, points + lo * pb, len * pb,
                                  cudaMemcpyHostToDevice, e.copy_stream));
    }
    D377_CUDA(cudaEventRecord(e.ev_chunk[slot][k], e.copy_stream));
  }
  TRY(msm_enqueue((uint8_t*)e.slot_sc[slot].p, prepared ? points : (const uint8_t*)e.slot_pt[slot].p, point_format,
                  sc_mont, n, dres, dres + 128, (uint32_t*)(dres + 192), nch > 1 ? chunk : 0, e.ev_chunk[slot],
                  true, n ? e.ev_chunk_sc[slot] : nullptr));
  cudaStream_t rs = result_stream(e);
  D377_CUDA(cudaMemcpyAsync(e.h_small + kSmallSlots + 256 * slot, dres, 256, cudaMemcpyDeviceToHost, rs));
  D377_CUDA(cudaEventRecord(e.ev_done[slot], rs));
  e.slot_busy[slot] = true;
  return D377_OK;
}

int d377_msm_submit(const uint8_t* scalars, const uint8_t* points, int point_format, size_t n,
                    int slot) {
  D377_REQUIRE_READY_NOJOIN();
  Engine& e = _eng;
  int fmt = 0;
  bool sc_mont = false;
  TRY(msm_args_ok(e, "d377_msm_submit", scalars, points, point_format, n, &fmt, &sc_mont));
  if (slot < 0 || slot >= Engine::kSlots) { set_error("slot %d out of range", slot); return D377_ERR_INVALID_ARG; }
  if (e.slot_busy[slot]) { set_error("slot %d still in flight: call d377_msm_wait first", slot); return D377_ERR_INVALID_ARG; }
  int rc = msm_submit_inner(e, scalars, points, fmt, sc_mont, n, slot);
  if (rc) drain(e);   // uploads from the caller's buffers may still be running
  return rc;
}

int d377_msm_wait(int slot, uint8_t out_element[128], uint8_t out_encoding[32]) {
  D377_REQUIRE_READY_NOJOIN();
  if (slot < 0 || slot >= Engine::kSlots) { set_error("slot %d out of range", slot); return D377_ERR_INVALID_ARG; }
  Engine& e = _eng;
  if (!e.slot_busy[slot]) { set_error("slot %d has no MSM in flight", slot); return D377_ERR_INVALID_ARG; }
  cudaError_t ce = cudaEventSynchronize(e.ev_done[slot]);
  e.slot_busy[slot] = false;
  if (ce != cudaSuccess) { drain(e); return cuda_fail(ce, "cudaEventSynchronize(ev_done)", __FILE__, __LINE__); }
  const uint8_t* h = e.h_small + kSmallSlots + 256 * slot;
  uint32_t flags;
  memcpy(&flags, h + 192, 4);
  TRY(msm_check_flags(flags));
  if (out_element) memcpy(out_element, h, 128);
  if (out_encoding) memcpy(out_encoding, h + 128, 32);
  return D377_OK;
}

int d377_msm(const uint8_t* scalars, const uint8_t* points, int point_format, size_t n,
             uint8_t out_element[128], uint8_t out_encoding[32]) {
  D377_REQUIRE_READY_NOJOIN();
  int slot = 0;
  while (slot + 1 < Engine::kSlots && _eng.slot_busy[slot]) slot++;
  TRY(d377_msm_submit(scalars, points, point_format, n, slot));
  return d377_msm_wait(slot, out_element, out_encoding);
}

int d377_fq_batch_op(int op, const uint8_t* a, const uint8_t* b, size_t n, uint8_t* out) {
  D377_REQUIRE_READY();
  if (op < 0 || op > 11) { set_error("bad op %d", op); return D377_ERR_INVALID_ARG; }
  if (n == 0) return D377_OK;
  if (!a || !out) { set_error("null pointer"); return D377_ERR_INVALID_ARG; }
  bool binary = (op == 0 || op == 2 || op == 3);
  if (binary && !b) { set_error("op %d needs b", op); return D377_ERR_INVALID_ARG; }
  Engine& e = _eng;
  TRY(ensure(e.in0, n * 32));
  TRY(ensure(e.in1, n * 32));
  TRY(ensure(e.out0, n * 32));
  auto body = [&]() -> int {
    H2D(e.in0.p, a, n * 32);
    if (binary) H2D(e.in1.p, b, n * 32);
    k_fq_op<<<grid_for(n, 128), 128, 0, e.stream>>>(op, (uint8_t*)e.in0.p,
                                                    binary ? (uint8_t*)e.in1.p : nullptr, n,
                                                    (uint8_t*)e.out0.p);
    D377_LAUNCHED();
    D377_CUDA(cudaGetLastError());
    D2H(out, e.out0.p, n * 32);
    D377_CUDA(cudaStreamSynchronize(e.stream));
    return D377_OK;
  };
  int rc = body();
  if (rc) drain(e);
  return rc;
}

int d377_fq_batch_isqrt(const uint8_t* x, size_t n, uint8_t* out, uint8_t* was_square) {
  D377_REQUIRE_READY();
  if (n == 0) return D377_OK;
  if (!x || !out || !was_square) { set_error("null pointer"); return D377_ERR_INVALID_ARG; }
  HostIn ins[] = {{x, 32}};
  HostOut outs[] = {{out, 32}, {was_square, 1}};
  return run_pipelined(n, ins, 1, outs, 2, [&](uint8_t* const* di, uint8_t* const* dout, size_t len) {
    return d377_fq_batch_isqrt_dev(di[0], len, dout[0], dout[1]);
  });
}

int d377_fq_batch_sqrt_ratio_zeta(const uint8_t* num, const uint8_t* den, size_t n, uint8_t* out,
                                  uint8_t* was_square) {
  D377_REQUIRE_READY();
  if (n == 0) return D377_OK;
  if (!num || !den || !out || !was_square) { set_error("null pointer"); return D377_ERR_INVALID_ARG; }
  HostIn ins[] = {{num, 32}, {den, 32}};
  HostOut outs[] = {{out, 32}, {was_square, 1}};
  return run_pipelined(n, ins, 2, outs, 2, [&](uint8_t* const* di, uint8_t* const* dout, size_t len) {
    return d377_fq_batch_sqrt_ratio_zeta_dev(di[0], di[1], len, dout[0], dout[1]);
  });
}

int d377_batch_normalize(const uint8_t* elements, size_t n, uint8_t* affine) {
  D377_REQUIRE_READY();
  if (n == 0) return D377_OK;
  if (!elements || !affine) { set_error("null pointer"); return D377_ERR_INVALID_ARG; }
  HostIn ins[] = {{elements, 128}};
  HostOut outs[] = {{affine, 64}};
  return run_pipelined(n, ins, 1, outs, 1, [&](uint8_t* const* di, uint8_t* const* dout, size_t len) {
    return d377_batch_normalize_dev(di[0], len, dout[0]);
  });
}

int d377_field_batch_deserialize(int field, const uint8_t* bytes, size_t n, uint8_t* out, uint8_t* ok) {
  D377_REQUIRE_READY();
  TRY(deserialize_args(field, bytes, n, ok));
  if (n == 0) return D377_OK;
  HostIn ins[] = {{bytes, 32}};
  HostOut outs[] = {{out, 32}, {ok, 1}};
  return run_pipelined(n, ins, 1, outs, 2, [&](uint8_t* const* di, uint8_t* const* dout, size_t len) {
    return d377_field_batch_deserialize_dev(field, di[0], len, out ? dout[0] : nullptr, dout[1]);
  });
}

int d377_imad_peak(double* gimad_per_s) {
  D377_REQUIRE_READY();
  if (!gimad_per_s) { set_error("null pointer"); return D377_ERR_INVALID_ARG; }
  Engine& e = _eng;
  const int iters = 2048, block = 256;
  const int grid = e.sm_count * 8;
  cudaEvent_t t0, t1;
  D377_CUDA(cudaEventCreate(&t0));
  D377_CUDA(cudaEventCreate(&t1));
  uint32_t* sink = (uint32_t*)(e.d_small + kSmallTmp);
  double best = 0;
  for (int rep = 0; rep < 12; rep++) {
    D377_CUDA(cudaEventRecord(t0, e.stream));
    switch (rep & 3) {
      case 0: k_imad_peak<0><<<grid, block, 0, e.stream>>>(sink, 12345u + rep, iters); break;
      case 1: k_imad_peak<1><<<grid, block, 0, e.stream>>>(sink, 12345u + rep, iters); break;
      case 2: k_imad_peak<2><<<grid, block, 0, e.stream>>>(sink, 12345u + rep, iters); break;
      default: k_imad_peak<3><<<grid, block, 0, e.stream>>>(sink, 12345u + rep, iters); break;
    }
    D377_CUDA(cudaEventRecord(t1, e.stream));
    D377_CUDA(cudaEventSynchronize(t1));
    float ms = 0;
    D377_CUDA(cudaEventElapsedTime(&ms, t0, t1));
    double ops = (double)grid * block * iters * 64.0;
    double g = ops / (ms * 1e-3) / 1e9;
    if (rep >= 4 && g > best) best = g;
  }
  cudaEventDestroy(t0);
  cudaEventDestroy(t1);
  *gimad_per_s = best;
  return D377_OK;
}

}  // extern "C"
