// Multi-GPU MSM inside ONE process (d377_msm_multi, d377_msm_multi_dev): the C-ABI form of
// SURVEY 8(e) that a Rust host can call -- Element::vartime_multiscalar_mul
// (element/projective.rs:99-117) over the GPUs of one box.
//
// The (scalar, point) pairs are cut into `ngpu` contiguous slices.  Every initialised
// engine owns one persistent host thread; the threads enqueue their slices concurrently (a
// Pippenger is ~100 launches, so one thread driving eight GPUs would start the last one
// ~2 ms late), each GPU runs a complete Pippenger whose last kernel stores the 128-byte
// partial sum straight into the first GPU's gather area (a peer store over NVLink from
// inside the compute kernel; cudaMemcpyPeerAsync where peer access is unavailable), and the
// first GPU adds the partial sums and compresses.  Elliptic-curve addition is not a
// reduction operator NCCL knows, and 128 bytes per GPU is latency, not bandwidth: a peer
// copy per GPU is the whole exchange step.  The multi-process form of the same path is
// decaf377_b200/dist.py (one process per GPU, NCCL all-gather).
#include <algorithm>
#include <cstring>
#include <vector>

#include "engine.h"

namespace d377 {

// One multi-GPU call at a time, blocking or asynchronous: every worker holds one task, and the
// gather ring below is advanced under this lock.
static std::mutex g_multi_mu;

static void worker_main(Engine* e) {
  select_engine(e);
  std::unique_lock<std::mutex> lk(e->wmu);
  for (;;) {
    e->wcv.wait(lk, [&] { return e->whas || e->wquit; });
    if (e->wquit) return;
    std::function<int()> task = std::move(e->wtask);
    e->whas = false;
    lk.unlock();
    int rc = task();
    std::string err = rc ? last_error() : "";
    lk.lock();
    e->wrc = rc;
    e->werr = err;
    e->wdone = true;
    e->wcv.notify_all();
  }
}

static void worker_post(Engine& e, std::function<int()> task) {
  std::unique_lock<std::mutex> lk(e.wmu);
  if (!e.worker.joinable()) e.worker = std::thread(worker_main, &e);
  e.wtask = std::move(task);
  e.wdone = false;
  e.whas = true;
  e.wcv.notify_all();
}

static int worker_wait(Engine& e) {
  std::unique_lock<std::mutex> lk(e.wmu);
  e.wcv.wait(lk, [&] { return e.wdone; });
  if (e.wrc) set_error("device %d: %s", e.device, e.werr.c_str());
  return e.wrc;
}

// One GPU's share: a Pippenger over its slice, the partial sum sent to the gathering
// engine.  Runs on the engine's worker thread; returns after the GPU has finished (the
// status word has to be read anyway).
static int leg(Engine& e, Engine& root, int index, bool host, const uint8_t* scalars,
               const uint8_t* points, int point_format, bool sc_mont, size_t n) {
  EngineScope scope(e);
  uint8_t* dres = e.d_small + kSmallResult;
  uint32_t* dflags = (uint32_t*)(e.d_small + kSmallFlags);
  uint32_t* hflags = (uint32_t*)(e.h_small + kSmallFlags);
  const uint8_t *dsc = scalars, *dpt = points;
  const cudaEvent_t* ready = nullptr;
  size_t chunk = 0;
  int rc;
  auto fail = [&](int code) {
    cudaStreamSynchronize(e.copy_stream);
    cudaStreamSynchronize(e.stream);
    return code;
  };
  if (host && e.slot_busy[0]) {
    set_error("an MSM submitted with d377_msm_submit is still in flight on slot 0: d377_msm_wait first");
    return D377_ERR_INVALID_ARG;
  }
  if (host && n) {
    // same upload pipeline as d377_msm_submit: sub-MSM chunks, the Pippenger of chunk k
    // overlaps the upload of chunk k+1
    const size_t pb = pt_bytes(point_format);
    if ((rc = ensure(e.slot_sc[0], n * 32 + 32))) return rc;
    if ((rc = ensure(e.slot_pt[0], n * pb + 128))) return rc;
    // A slice of a multi-GPU call is link-bound (all GPUs pull from the same host memory),
    // so its upload is cut finer than a single-GPU call's: sub-MSMs down to 2^19 pairs.
    size_t nch = 1;
    while (nch < 4 && n / (nch * 2) >= ((size_t)1 << 19)) nch *= 2;
    if (e.msm_host_chunks_override > 0) nch = std::min<size_t>(e.msm_host_chunks_override, Engine::kMsmHostChunks);
    chunk = ((n + nch - 1) / nch + 255) / 256 * 256;
    nch = (n + chunk - 1) / chunk;
    // status word: reset ahead of the chunk events (the scalar side depends on those only)
    if (cudaMemsetAsync(dflags, 0, 4, e.copy_stream) != cudaSuccess)
      return fail(cuda_fail(cudaGetLastError(), "cudaMemsetAsync", __FILE__, __LINE__));
    for (size_t k = 0; k < nch; k++) {
      size_t lo = k * chunk, len = std::min(chunk, n - lo);
      cudaError_t ce = cudaMemcpyAsync((uint8_t*)e.slot_sc[0].p + lo * 32, scalars + lo * 32, len * 32,
                                       cudaMemcpyHostToDevice, e.copy_stream);
      if (ce == cudaSuccess) ce = cudaEventRecord(e.ev_chunk_sc[0][k], e.copy_stream);
      if (ce == cudaSuccess)
        ce = cudaMemcpyAsync((uint8_t*)e.slot_pt[0].p + lo * pb, points + lo * pb, len * pb,
                             cudaMemcpyHostToDevice, e.copy_stream);
      if (ce == cudaSuccess) ce = cudaEventRecord(e.ev_chunk[0][k], e.copy_stream);
      if (ce != cudaSuccess) return fail(cuda_fail(ce, "upload of a slice", __FILE__, __LINE__));
    }
    dsc = (const uint8_t*)e.slot_sc[0].p;
    dpt = (const uint8_t*)e.slot_pt[0].p;
    ready = e.ev_chunk[0];
    if (nch == 1) chunk = 0;
  }
  cudaError_t ce = cudaSuccess;
  if (!ready) ce = cudaMemsetAsync(dflags, 0, 4, e.stream);
  if (ce != cudaSuccess) return fail(cuda_fail(ce, "cudaMemsetAsync", __FILE__, __LINE__));
  // With peer access the MSM's last kernel (Horner over the windows) stores the partial sum
  // STRAIGHT into the first GPU's gather area -- a 128-byte store over NVLink from inside the
  // compute kernel, no copy in between; without it the sum lands locally and is copied.
  uint8_t* dst = root.d_small + kSmallGather + 128 * index;
  const bool direct = &e == &root || ((e.peer_mask >> root.device) & 1ull);
  rc = msm_enqueue(dsc, dpt, point_format, sc_mont, n, direct ? dst : dres, nullptr, dflags, chunk, ready,
                   ready != nullptr, ready ? e.ev_chunk_sc[0] : nullptr);
  if (rc) return fail(rc);
  cudaStream_t rs = result_stream(e);
  if (!direct) ce = cudaMemcpyPeerAsync(dst, root.device, dres, e.device, 128, rs);
  if (ce == cudaSuccess) ce = cudaEventRecord(e.ev_partial, rs);
  if (ce == cudaSuccess) ce = cudaMemcpyAsync(hflags, dflags, 4, cudaMemcpyDeviceToHost, rs);
  if (ce == cudaSuccess) ce = cudaStreamSynchronize(rs);
  if (ce != cudaSuccess) return fail(cuda_fail(ce, "partial sum exchange", __FILE__, __LINE__));
  return msm_check_flags(*hflags);
}

static int msm_multi(bool host, const uint8_t* const* scalars, const uint8_t* const* points,
                     int point_format, const size_t* n, int ngpu, uint8_t* out_element,
                     uint8_t* out_encoding) {
  int devs[8];
  const int have = d377_device_list(devs, 8);
  if (ngpu < 1 || ngpu > 8 || ngpu > have) {
    set_error("d377_msm_multi: ngpu = %d but %d device(s) initialised (d377_init_multi)", ngpu, have);
    return have ? D377_ERR_INVALID_ARG : D377_ERR_NOT_INITIALISED;
  }
  // prepared bases belong to one device: d377_msm takes them
  int pf = 0;
  bool sc_mont = false;
  int rc = parse_format("d377_msm_multi", point_format, kPointFormats, &pf, &sc_mont);
  if (rc) return rc;
  Engine* eng[8];
  for (int k = 0; k < ngpu; k++) {
    eng[k] = engine_for(devs[k]);
    if (!eng[k]) { set_error("device %d is not initialised", devs[k]); return D377_ERR_NOT_INITIALISED; }
    if (n[k] && (!scalars[k] || !points[k])) { set_error("null pointer"); return D377_ERR_INVALID_ARG; }
  }
  Engine& root = *eng[0];
  std::lock_guard<std::mutex> multi_lock(g_multi_mu);
  for (int k = 0; k < ngpu; k++) {
    Engine* e = eng[k];
    const uint8_t *s = scalars[k], *p = points[k];
    const size_t nk = n[k];
    worker_post(*e, [=, &root]() { return leg(*e, root, k, host, s, p, pf, sc_mont, nk); });
  }
  for (int k = 0; k < ngpu; k++) {
    int r = worker_wait(*eng[k]);
    if (r && !rc) rc = r;
  }
  if (rc) return rc;
  // every partial sum has landed (the legs synchronised their result streams): add them up
  EngineScope scope(root);
  cudaStream_t rs = result_stream(root);
  for (int k = 1; k < ngpu; k++) D377_CUDA(cudaStreamWaitEvent(rs, eng[k]->ev_partial, 0));
  rc = element_sum_on(root, rs, root.d_small + kSmallGather, (size_t)ngpu, root.d_small + kSmallResult,
                      root.d_small + kSmallResult + 128);
  if (rc) return rc;
  D377_CUDA(cudaMemcpyAsync(root.h_small + kSmallResult, root.d_small + kSmallResult, 160,
                            cudaMemcpyDeviceToHost, rs));
  D377_CUDA(cudaStreamSynchronize(rs));
  if (out_element) memcpy(out_element, root.h_small + kSmallResult, 128);
  if (out_encoding) memcpy(out_encoding, root.h_small + kSmallResult + 128, 32);
  return D377_OK;
}

// ---- asynchronous form ------------------------------------------------------------------
// Only enqueues: every GPU's Pippenger goes through the same overlapped pipeline as
// d377_msm_dev_async (tail of call k and sort of call k+1 under the bucket accumulation),
// the partial sums travel into one of kGatherRing gather areas on the first GPU, and the
// final sum + compress is enqueued on the first GPU's result stream behind the events the
// legs recorded.  Status words are sticky per engine; d377_multi_sync reports them.
constexpr int kGatherRing = 4;
// The ring has areas of its own: the blocking call's area (kSmallGather) is rewritten by the
// next blocking call straight away, which must not hit a sum of an earlier asynchronous call
// that is still waiting for its slowest leg.
static const size_t kGatherOff[kGatherRing] = {kSmallGatherRing, kSmallGatherRing + 1024,
                                               kSmallGatherRing + 2048, kSmallGatherRing + 3072};
static cudaEvent_t g_gather_free[kGatherRing] = {};   // on the root: the sum that read area k is done
static bool g_gather_used[kGatherRing] = {};
static Engine* g_gather_root = nullptr;
static int g_ring = 0;

static int leg_async(Engine& e, Engine& root, int index, int ring, const uint8_t* scalars,
                     const uint8_t* points, int point_format, bool sc_mont, size_t n) {
  EngineScope scope(e);
  uint8_t* dres = e.d_small + kSmallResult;
  uint8_t* dst = root.d_small + kGatherOff[ring] + 128 * index;
  const bool direct = &e == &root || ((e.peer_mask >> root.device) & 1ull);
  e.async_status_dirty = true;
  cudaStream_t rs = result_stream(e);
  // the gather area may still be read by the sum of the call that used it last (the tail that
  // writes it runs on the result stream, so the wait goes there before the MSM is enqueued)
  if (g_gather_used[ring]) D377_CUDA(cudaStreamWaitEvent(rs, g_gather_free[ring], 0));
  int rc = msm_enqueue(scalars, points, point_format, sc_mont, n, direct ? dst : dres, nullptr,
                       (uint32_t*)(e.d_small + kSmallAsyncFlags), 0, nullptr, true);
  if (rc) return rc;
  if (!direct) D377_CUDA(cudaMemcpyPeerAsync(dst, root.device, dres, e.device, 128, rs));
  D377_CUDA(cudaEventRecord(e.ev_partial, rs));
  return D377_OK;
}

static int msm_multi_async(const uint8_t* const* scalars, const uint8_t* const* points, int point_format,
                           const size_t* n, int ngpu, uint8_t* out_element_dev, uint8_t* out_encoding_dev) {
  int devs[8];
  const int have = d377_device_list(devs, 8);
  if (ngpu < 1 || ngpu > 8 || ngpu > have) {
    set_error("d377_msm_multi_dev_async: ngpu = %d but %d device(s) initialised (d377_init_multi)", ngpu, have);
    return have ? D377_ERR_INVALID_ARG : D377_ERR_NOT_INITIALISED;
  }
  int pf = 0;
  bool sc_mont = false;
  int rc = parse_format("d377_msm_multi_dev_async", point_format, kPointFormats, &pf, &sc_mont);
  if (rc) return rc;
  Engine* eng[8];
  for (int k = 0; k < ngpu; k++) {
    eng[k] = engine_for(devs[k]);
    if (!eng[k]) { set_error("device %d is not initialised", devs[k]); return D377_ERR_NOT_INITIALISED; }
    if (n[k] && (!scalars[k] || !points[k])) { set_error("null pointer"); return D377_ERR_INVALID_ARG; }
  }
  Engine& root = *eng[0];
  std::lock_guard<std::mutex> multi_lock(g_multi_mu);
  {
    EngineScope scope(root);
    if (g_gather_root != &root) {   // first use on this root device: events live there
      for (int k = 0; k < kGatherRing; k++) {
        if (g_gather_free[k]) cudaEventDestroy(g_gather_free[k]);
        D377_CUDA(cudaEventCreateWithFlags(&g_gather_free[k], cudaEventDisableTiming));
        g_gather_used[k] = false;
      }
      g_gather_root = &root;
      g_ring = 0;
    }
  }
  const int ring = g_ring;
  g_ring = (g_ring + 1) % kGatherRing;
  for (int k = 0; k < ngpu; k++) {
    Engine* e = eng[k];
    const uint8_t *sp = scalars[k], *pp = points[k];
    const size_t nk = n[k];
    worker_post(*e, [=, &root]() { return leg_async(*e, root, k, ring, sp, pp, pf, sc_mont, nk); });
  }
  for (int k = 0; k < ngpu; k++) {
    int r = worker_wait(*eng[k]);
    if (r && !rc) rc = r;
  }
  if (rc) return rc;
  // every leg has recorded its event: the sum waits for them on the root's result stream
  EngineScope scope(root);
  cudaStream_t rs = result_stream(root);
  for (int k = 0; k < ngpu; k++) D377_CUDA(cudaStreamWaitEvent(rs, eng[k]->ev_partial, 0));
  rc = element_sum_on(root, rs, root.d_small + kGatherOff[ring], (size_t)ngpu, out_element_dev, out_encoding_dev);
  if (rc) return rc;
  D377_CUDA(cudaEventRecord(g_gather_free[ring], rs));
  g_gather_used[ring] = true;
  return D377_OK;
}

void multi_shutdown() {
  for (int k = 0; k < kGatherRing; k++) {
    if (g_gather_free[k]) cudaEventDestroy(g_gather_free[k]);
    g_gather_free[k] = nullptr;
    g_gather_used[k] = false;
  }
  g_gather_root = nullptr;
}

}  // namespace d377

using namespace d377;

extern "C" {

int d377_msm_multi_dev_async(const uint8_t* const* scalars, const uint8_t* const* points, int point_format,
                             const size_t* n, int ngpu, uint8_t* out_element_dev, uint8_t* out_encoding_dev) {
  if (!scalars || !points || !n) { set_error("null pointer"); return D377_ERR_INVALID_ARG; }
  return msm_multi_async(scalars, points, point_format, n, ngpu, out_element_dev, out_encoding_dev);
}

int d377_multi_sync(void) {
  int devs[8];
  const int have = d377_device_list(devs, 8);
  if (!have) { set_error("d377_init_multi has not been called"); return D377_ERR_NOT_INITIALISED; }
  Engine* prev = selected_engine();
  int rc = D377_OK;
  for (int k = 0; k < have; k++) {
    Engine* e = engine_for(devs[k]);
    if (!e) continue;
    select_engine(e);
    int r = d377_sync();   // joins the result stream, waits, reports the sticky status word
    if (r && !rc) rc = r;
  }
  select_engine(prev);
  return rc;
}

int d377_msm_multi(const uint8_t* scalars, const uint8_t* points, int point_format, size_t n, int ngpu,
                   uint8_t out_element[128], uint8_t out_encoding[32]) {
  if (ngpu < 1 || ngpu > 8) { set_error("d377_msm_multi: ngpu must be 1..8"); return D377_ERR_INVALID_ARG; }
  int pf = 0;
  bool sc_mont = false;   // passed on in the format word
  const int rc = parse_format("d377_msm_multi", point_format, kPointFormats, &pf, &sc_mont);
  if (rc) return rc;
  if (n && (!scalars || !points)) { set_error("null pointer"); return D377_ERR_INVALID_ARG; }
  const uint8_t *sc[8], *pt[8];
  size_t cnt[8];
  const size_t pb = pt_bytes(pf);
  // contiguous slices whose sizes differ by at most one (dist.shard_range)
  const size_t base = n / (size_t)ngpu, rem = n % (size_t)ngpu;
  size_t lo = 0;
  for (int k = 0; k < ngpu; k++) {
    cnt[k] = base + ((size_t)k < rem ? 1 : 0);
    sc[k] = scalars + 32 * lo;
    pt[k] = points + pb * lo;
    lo += cnt[k];
  }
  return msm_multi(true, sc, pt, point_format, cnt, ngpu, out_element, out_encoding);
}

int d377_msm_multi_dev(const uint8_t* const* scalars, const uint8_t* const* points, int point_format,
                       const size_t* n, int ngpu, uint8_t out_element[128], uint8_t out_encoding[32]) {
  if (!scalars || !points || !n) { set_error("null pointer"); return D377_ERR_INVALID_ARG; }
  return msm_multi(false, scalars, points, point_format, n, ngpu, out_element, out_encoding);
}

}  // extern "C"
