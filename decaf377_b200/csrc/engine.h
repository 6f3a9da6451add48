// Engine state shared by the translation units of libdecaf377_b200.so.
//
// One `Engine` per CUDA device (streams, scratch arenas, MSM pipeline state).  A process
// may hold several (d377_init_multi); every C-ABI entry point acts on the engine the
// calling thread has selected (d377_set_device) or, by default, on the one d377_init chose.
// Entry points take the engine's lock and make its device current for the duration of the
// call (EngineScope), so the library can be called from any host thread.
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <condition_variable>
#include <cstdint>
#include <cstdio>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <unordered_map>

#include "../../include/decaf377_b200.h"

namespace d377 {

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
};

constexpr int kMsmStages = 8;  // points, count, scan, scatter, accumulate, stitch, bucket_reduce, tail
constexpr int kMaxGroups = 8;

struct MsmGeomInfo {
  int c = 0, W = 0;
};

// Layout of a set of prepared bases (d377_msm_bases_create*).  Plain sets: c = 0, W = 1, one
// bucket operand per base.  Windowed sets (d377_msm_bases_create_windowed*): W slabs of n
// operands, window-major with stride n; record j*n + i holds 2^(c*j) * P_i.
struct BasesLayout {
  size_t n = 0;
  int c = 0, W = 1;
  size_t bytes = 0;
};

// A set of prepared fixed bases (d377_fixed_bases_create*): k window tables back to back.
struct FixedBasesInfo {
  size_t k = 0;
  size_t bytes = 0;
};

// Per-device state of the Pippenger pipeline (msm.cu).
struct MsmState {
  bool ready = false;
  // second stream: the scalar side (digit recoding, histogram, scan, scatter) of window
  // group k+1 runs here while the engine stream accumulates group k
  cudaStream_t sort_stream = nullptr;
  // third stream: the latency-bound tail of an MSM (stitch, bucket reduction, weighted tree,
  // Horner, compress) runs here, so that the head of the NEXT MSM (normalisation, first sort,
  // first accumulation) starts on the engine stream right behind the last accumulation.
  // The tail owns one of two workspace sets; see msm_once.
  cudaStream_t tail_stream = nullptr;
  // fourth stream: point conversion / batch normalisation of the NEXT MSM (inputs known ready)
  cudaStream_t points_stream = nullptr;
  cudaEvent_t ev_points_done[2] = {};
  cudaEvent_t ev_fork = nullptr, ev_sorted[kMaxGroups] = {}, ev_sort0 = nullptr, ev_sort1 = nullptr;
  cudaEvent_t ev_acc0[kMaxGroups] = {}, ev_acc[kMaxGroups] = {};
  cudaEvent_t ev_stage[kMsmStages + 1] = {};
  cudaEvent_t ev_acc_done = nullptr;        // engine stream: last accumulation of the current MSM
  cudaEvent_t ev_tail_done[2] = {};         // tail stream: the tail that used workspace set k
  cudaEvent_t ev_join = nullptr;
  bool tail_used[2] = {false, false};       // set k has been used by some tail (event valid)
  bool tail_pending = false;                // a tail has been enqueued since the last join
  int cur_set = 0;                          // the set the most recent MSM used
  DevBuf tail_ws[2];
  MsmGeomInfo last_geom;
  bool last_affine = false;
  bool last_windowed = false;
  int last_groups = 1;
  size_t last_n = 0;
  bool stage_valid = false;
};

struct Engine {
  bool ready = false;
  int device = -1;
  int sm_count = 148;
  cudaStream_t stream = nullptr;
  std::recursive_mutex mu;
  // set through the ABI (d377_msm_set_*); the defaults are the library's own choices
  int msm_window_override = 0;
  int msm_host_chunks_override = 0;
  int msm_groups_override = 0;        // window groups of the sort / accumulate pipeline
  int msm_normalize_override = 0;     // Element / XYZ inputs: -1 never normalised, 1 always, 0 auto
  int msm_tail_overlap_override = 1;  // 0 = MSM tails on the engine stream
  // host-API staging
  DevBuf in0, in1, out0, out1;
  // prefix products of k_normalize
  DevBuf scratch;
  // canonical copy of scalars handed over in Montgomery form (D377_SCALARS_MONTGOMERY)
  DevBuf sc_canon;
  // d377_batch_msm: products, their decode status, segment sums; host-call staging
  DevBuf bm_prod, bm_ok, bm_sum, bm_sc, bm_pt, bm_off, bm_out, bm_okout;
  // d377_msm_segmented*: workspace (converted points, one chunk's sort and tail), pinned
  // staging of the host offsets with the event after their upload, and the geometry of the
  // most recent call (d377_msm_segmented_last)
  DevBuf seg_ws;
  void* seg_off_host = nullptr;
  size_t seg_off_cap = 0;
  cudaEvent_t ev_seg_off = nullptr;
  int seg_last_c = 0, seg_last_W = 0;
  size_t seg_last_chunks = 0;
  // fixed-base table (niels, affine) and its geometry
  void* fb_table = nullptr;
  void* fb_table_jq = nullptr;   // the same multiples on the Jacobi quartic (encoding output)
  size_t fb_batch_hint = 0;      // size of the host-buffer batch whose chunks are being launched
  // scratch of element_sum_on: [0] engine stream, [1] result stream
  DevBuf sum_ws[2];
  // small device result + pinned host mirror (8 KiB each; layout in kernels.cu)
  uint8_t* d_small = nullptr;
  uint8_t* h_small = nullptr;
  // pipelined host-buffer MSM (d377_msm_submit / d377_msm_wait)
  static constexpr int kSlots = 4;
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t ev_h2d[kSlots] = {};
  cudaEvent_t ev_done[kSlots] = {};
  DevBuf slot_sc[kSlots], slot_pt[kSlots];
  bool slot_busy[kSlots] = {};
  // host-buffer MSMs are cut into up to kMsmHostChunks sub-MSMs so that the upload of
  // chunk k+1 overlaps the Pippenger of chunk k (one event per chunk and slot)
  static constexpr int kMsmHostChunks = 8;
  cudaEvent_t ev_chunk[kSlots][kMsmHostChunks] = {};
  cudaEvent_t ev_chunk_sc[kSlots][kMsmHostChunks] = {};   // the chunk's scalars alone are up
  // chunk-pipelined host API of the batch kernels: H2D on copy_stream, kernels on
  // `stream`, D2H on out_stream, two staging sets
  cudaStream_t out_stream = nullptr;
  cudaEvent_t pe_in[2] = {nullptr, nullptr}, pe_k[2] = {nullptr, nullptr}, pe_out[2] = {nullptr, nullptr};
  DevBuf st_in[2][3], st_out[2][2];
  // prepared MSM bases handed out by d377_msm_bases_create*: device pointer -> layout
  std::unordered_map<const void*, BasesLayout> bases;
  // prepared fixed bases handed out by d377_fixed_bases_create*: device pointer -> {k, bytes}
  std::unordered_map<const void*, FixedBasesInfo> fixed_bases;
  // asynchronous MSMs (d377_msm_dev_async): sticky status word, reported by d377_sync
  bool async_status_dirty = false;
  MsmState msm;
  // multi-GPU calls (d377_msm_multi*): one persistent host thread per engine
  std::thread worker;
  std::mutex wmu;
  std::condition_variable wcv;
  std::function<int()> wtask;
  bool whas = false, wdone = false, wquit = false;
  int wrc = 0;
  std::string werr;
  cudaEvent_t ev_partial = nullptr;  // this engine's partial sum has landed on the gathering device
  uint64_t peer_mask = 0;            // bit d: this device may store into device d's memory (peer access enabled)
};

// d_small / h_small layout (kSmallBytes each)
constexpr size_t kSmallBytes = 16384;
constexpr size_t kSmallResult = 0;      // [0,160) result of the synchronous calls
constexpr size_t kSmallTmp = 512;       // [512,640) tmp
constexpr size_t kSmallGather = 1024;   // [1024,2048) partial sums of up to 8 devices (d377_msm_multi*)
constexpr size_t kSmallPartials = 2048; // [2048,4096) MSM chunk partials
constexpr size_t kSmallFlags = 4096;    // status word of the synchronous MSM
constexpr size_t kSmallAsyncFlags = 4100;  // sticky status word of d377_msm_dev_async
constexpr size_t kSmallDebug = 4104;    // on-curve debug predicate failures (D377_DEBUG_ON_CURVE builds)
constexpr size_t kSmallSlots = 4352;    // [4352 + 256 k, ...) slot k
constexpr size_t kSmallGatherRing = 8192;  // [8192,12288) four gather areas of d377_msm_multi_dev_async
// [4352, 5376): the four slots; [8192, 11264): three more gather areas of
// d377_msm_multi_dev_async (multi.cu)

Engine& engine();              // the calling thread's engine (selected or default); never null
Engine* engine_for(int device);  // nullptr if that device has not been initialised
void select_engine(Engine* e);   // thread-local selection (nullptr = default)
Engine* selected_engine();       // the calling thread's explicit selection (may be nullptr)
void multi_shutdown();           // multi.cu
void set_error(const char* fmt, ...);
const char* last_error();
int cuda_fail(cudaError_t e, const char* what, const char* file, int line);
int ensure(DevBuf& b, size_t bytes);
void count_launch();

// Lock the engine and make its device current; restores the previous device on exit.
struct EngineScope {
  Engine& e;
  int prev = -1;
  explicit EngineScope(Engine& en) : e(en) {
    e.mu.lock();
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (prev != e.device) cudaSetDevice(e.device);
  }
  ~EngineScope() {
    if (prev >= 0 && prev != e.device) cudaSetDevice(prev);
    e.mu.unlock();
  }
  EngineScope(const EngineScope&) = delete;
  EngineScope& operator=(const EngineScope&) = delete;
};

#define D377_CUDA(expr)                                                        \
  do {                                                                         \
    cudaError_t _e = (expr);                                                   \
    if (_e != cudaSuccess) return ::d377::cuda_fail(_e, #expr, __FILE__, __LINE__); \
  } while (0)

// Entry-point prologue: fails when no engine is ready, otherwise locks it and selects its
// device.  The _NOJOIN form leaves MSM tails running on the tail stream; the plain form
// first orders the engine stream behind them (so that anything enqueued by this call sees
// the results of every earlier call).
#define D377_REQUIRE_READY_NOJOIN()                                            \
  ::d377::Engine& _eng = ::d377::engine();                                     \
  if (!_eng.ready) {                                                           \
    ::d377::set_error("d377_init has not been called (or failed): no GPU path available"); \
    return D377_ERR_NOT_INITIALISED;                                           \
  }                                                                            \
  ::d377::EngineScope _scope(_eng)

#define D377_REQUIRE_READY()                                                   \
  D377_REQUIRE_READY_NOJOIN();                                                 \
  do {                                                                         \
    int _jrc = ::d377::msm_join(_eng);                                         \
    if (_jrc) return _jrc;                                                     \
  } while (0)

#define D377_LAUNCHED() (::d377::count_launch())

inline unsigned grid_for(size_t n, unsigned block) { return (unsigned)((n + block - 1) / block); }

// Bytes per element of a point array in format D377_PT_* (D377_PT_BASES: one prepared record)
// and of a result in format D377_OUT_*.
__host__ __device__ constexpr size_t pt_bytes(int fmt) {
  return fmt == D377_PT_ENCODING ? 32 : fmt == D377_PT_AFFINE ? 64 : fmt == D377_PT_XYZ ? 96 : 128;
}
constexpr size_t out_bytes(int fmt) { return pt_bytes(fmt == D377_OUT_ENCODING ? D377_PT_ENCODING : D377_PT_ELEMENT); }

// The set of format values an entry point accepts, as the `accepted` mask of parse_format.
template <class... F>
constexpr unsigned fmt_set(F... f) { return ((1u << f) | ...); }
constexpr unsigned kPointFormats = fmt_set(D377_PT_ELEMENT, D377_PT_ENCODING, D377_PT_AFFINE, D377_PT_XYZ);
constexpr unsigned kOutFormats = fmt_set(D377_OUT_ELEMENT, D377_OUT_ENCODING);

// The format word of entry point `who` -> the format value (*fmt, if wanted) and, for a call
// that takes scalars (sc_mont not null), the D377_SCALARS_MONTGOMERY flag riding on it
// (*sc_mont).  A value outside `accepted` is refused with D377_ERR_INVALID_ARG.
int parse_format(const char* who, int word, unsigned accepted, int* fmt, bool* sc_mont = nullptr);

// kernels.cu
void launch_fr_from_mont(const uint8_t* in, size_t n, uint8_t* out, cudaStream_t st);
// codec.cu
void launch_decompress(const uint8_t* enc, size_t n, uint8_t* out, uint8_t* ok, cudaStream_t st,
                       int out_format = D377_PT_ELEMENT);
void launch_compress(const uint8_t* in, size_t n, uint8_t* enc, cudaStream_t st,
                     int in_format = D377_PT_ELEMENT);
void launch_elligator(bool hash, bool encode, const uint8_t* r1, const uint8_t* r2, size_t width, size_t n,
                      uint8_t* out, cudaStream_t st);
void launch_fq_isqrt(const uint8_t* x, size_t n, uint8_t* out, uint8_t* wsq, cudaStream_t st);
void launch_fq_sqrt_ratio(const uint8_t* num, const uint8_t* den, size_t n, uint8_t* out,
                          uint8_t* wsq, cudaStream_t st);
void launch_on_curve(const uint8_t* el, size_t n, int check_order, uint8_t* ok, cudaStream_t st);
// scalar.cu
void launch_scalar_mul(int point_format, bool encode, const uint8_t* points, const uint8_t* scalars,
                       size_t n, uint8_t* out, uint8_t* ok, cudaStream_t st);
int ensure_fb_table();
int ensure_fb_table_jq();
void launch_fixed_base(bool encode, const void* table, size_t k, const void* table_jq, const uint8_t* scalars,
                       size_t n, uint8_t* out, cudaStream_t st);
size_t fixed_bases_bytes_per_base();
int fixed_bases_fill(const uint8_t* points, int point_format, size_t k, void* table);

// msm.cu
void launch_seg_sum(const uint8_t* prods, const uint8_t* okp, const uint32_t* offs, size_t nseg,
                    uint8_t* out_el, uint8_t* ok_out, cudaStream_t st);
void launch_normalize(const uint8_t* el, size_t n, uint8_t* scratch, uint8_t* out, cudaStream_t st);
// Order the engine stream behind every MSM tail enqueued so far (no host synchronisation).
int msm_join(Engine& e);
int msm_dev(const uint8_t* scalars, const uint8_t* points, int point_format, size_t n,
            uint8_t* out_element, uint8_t* out_encoding);
int msm_dev_async(const uint8_t* scalars, const uint8_t* points, int point_format, size_t n,
                  uint8_t* out_element, uint8_t* out_encoding, int flags);
// Arguments of the single-device MSM calls: the format word (any D377_PT_* format, split by
// parse_format), null pointers and, for prepared bases, the handle.
int msm_args_ok(Engine& e, const char* who, const uint8_t* scalars, const uint8_t* points, int point_format,
                size_t n, int* fmt, bool* sc_mont);
// `point_format`: a D377_PT_* value; `sc_mont`: the scalars are in Montgomery form.
// `inputs_ready`: the inputs depend on nothing but chunk_ready[k] (nothing at all without
// chunk_ready): the scalar side may then start under the previous MSM's accumulation.
// `chunk` = 0: one Pippenger (split only above 2^26 pairs).  Otherwise the input is
// processed as ceil(n / chunk) sub-MSMs whose partial sums are added at the end; the
// engine stream waits for chunk_ready[k] (if given) before it touches chunk k.
// The result is complete on result_stream(): the tail stream, or the engine stream when the
// tail overlap is switched off.
int msm_enqueue(const uint8_t* scalars, const uint8_t* points, int point_format, bool sc_mont, size_t n,
                uint8_t* out_element, uint8_t* out_encoding, uint32_t* flags, size_t chunk = 0,
                const cudaEvent_t* chunk_ready = nullptr, bool inputs_ready = false,
                const cudaEvent_t* scalars_ready_ev = nullptr);
cudaStream_t result_stream(Engine& e);
int msm_check_flags(uint32_t flags);
// kernels.cu; *layout (may be null) receives the set's layout
int check_bases(Engine& e, const uint8_t* points, size_t n, BasesLayout* layout = nullptr);
int msm_bases_prepare(const uint8_t* points, int point_format, size_t n, uint8_t* records);
// the W - 1 upper slabs of a windowed set whose slab 0 msm_bases_prepare has written
int msm_bases_fill_windows(uint8_t* table, size_t n, int c, int W);
int msm_windowed_c(size_t n);    // window width of a windowed set when the caller passes c = 0
bool msm_last_windowed();
// d377_msm_segmented*: the window width for these (validated, host) offsets -- refused with
// D377_ERR_INVALID_ARG when some segment does not fit a chunk of its own -- and the enqueue
// on the engine stream (device scalars, points, out, ok; host offsets)
int msm_segmented_width(Engine& e, int fmt, const uint32_t* offsets, size_t nmsm, int* c);
int msm_segmented_enqueue(const uint8_t* scalars, const uint8_t* points, int fmt, bool sc_mont,
                          const uint32_t* offsets, size_t nmsm, int c, uint8_t* out, int out_format, uint8_t* ok);
int msm_segmented_last(int* c, int* W, size_t* chunks);
int msm_stage_info(float* ms, int* c, int* W, uint64_t* n);
int msm_timeline(float* ms, int cap, int* ngroups);
bool msm_last_mixed();
void msm_shutdown(Engine& e);
int element_sum_on(Engine& e, cudaStream_t st, const uint8_t* elements, size_t n, uint8_t* out_element,
                   uint8_t* out_encoding);

}  // namespace d377
