// Library plumbing: error string, launch counter, version, FP32 probe, host-buffer entry points.
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <vector>

#include "fo_common.cuh"

namespace fo {

static thread_local char g_err[512] = "";
static std::atomic<uint64_t> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
void count_launch(uint64_t n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

// 8 independent FFMA chains per thread; 2 flops per FFMA.
__global__ void __launch_bounds__(256) fp32_probe_kernel(int iters, float seed, float* sink) {
  float a0 = seed + threadIdx.x, a1 = a0 + 1.f, a2 = a0 + 2.f, a3 = a0 + 3.f;
  float a4 = a0 + 4.f, a5 = a0 + 5.f, a6 = a0 + 6.f, a7 = a0 + 7.f;
  const float m = 0.999f, c = 0.001f;
#pragma unroll 32
  for (int i = 0; i < iters; ++i) {      // 256 FFMAs per loop-control triple: the loop overhead stays below 1.5 %
    a0 = fmaf(a0, m, c); a1 = fmaf(a1, m, c); a2 = fmaf(a2, m, c); a3 = fmaf(a3, m, c);
    a4 = fmaf(a4, m, c); a5 = fmaf(a5, m, c); a6 = fmaf(a6, m, c); a7 = fmaf(a7, m, c);
  }
  float r = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
  if (r == 123456.789f) sink[0] = r;
}

// per-thread device workspace of the host-buffer entry points
constexpr int kHostChunksMax = 16;
struct HostWs {
  void* dev = nullptr;
  size_t bytes = 0;
  cudaStream_t stream = nullptr;        // compute (+ result copies)
  cudaStream_t copy = nullptr;          // host -> device copies of the bundle
  cudaEvent_t ready[kHostChunksMax] = {};
};
static thread_local HostWs g_ws;

static int ws_reserve(size_t bytes) {
  if (!g_ws.stream) {
    FO_CUDA_TRY(cudaStreamCreateWithFlags(&g_ws.stream, cudaStreamNonBlocking));
    FO_CUDA_TRY(cudaStreamCreateWithFlags(&g_ws.copy, cudaStreamNonBlocking));
    for (int i = 0; i < kHostChunksMax; ++i) FO_CUDA_TRY(cudaEventCreateWithFlags(&g_ws.ready[i], cudaEventDisableTiming));
  }
  if (bytes <= g_ws.bytes) return FO_OK;
  if (g_ws.dev) FO_CUDA_TRY(cudaFree(g_ws.dev));
  g_ws.dev = nullptr; g_ws.bytes = 0;
  size_t want = bytes + bytes / 4;
  FO_CUDA_TRY(cudaMalloc(&g_ws.dev, want));
  g_ws.bytes = want;
  return FO_OK;
}

// Error exits of the host-buffer entry points happen with copies / kernels possibly still queued on the workspace
// streams: wait for them before handing the caller's buffers back (the message of the first failure is kept).
static int ws_fail(int code) {
  char keep[sizeof(g_err)];
  memcpy(keep, g_err, sizeof(keep));
  cudaStreamSynchronize(g_ws.copy);
  cudaStreamSynchronize(g_ws.stream);
  cudaGetLastError();
  memcpy(g_err, keep, sizeof(keep));
  return code;
}

// Upload chunks of N rows of row_bytes each: chunk c is rows [bound[c], bound[c + 1]); returns the chunk count.  The
// first chunk is small (its copy cannot be hidden), every following one four times larger; rows that take less than two
// first chunks go in one.
static int host_chunks(size_t N, size_t row_bytes, size_t bound[kHostChunksMax + 1]) {
  static const char* chunk_env = getenv("FO_HOST_CHUNK_MB");           // measurement switch: size of the first chunk
  const size_t first_bytes = (size_t)(chunk_env && atoi(chunk_env) > 0 ? atoi(chunk_env) : 16) << 20;
  bound[0] = 0; bound[1] = N;
  if (N * row_bytes < 2 * first_bytes || row_bytes == 0) return 1;
  size_t step = (first_bytes + row_bytes - 1) / row_bytes, at = 0;
  int chunks = 0;
  while (at < N && chunks < kHostChunksMax - 1) {
    at = (at + step < N) ? at + step : N;
    bound[++chunks] = at;
    step *= 4;
  }
  if (at < N) bound[++chunks] = N;
  return chunks;
}

}  // namespace fo

#define FO_HOST_TRY(expr)                                                                          \
  do {                                                                                             \
    cudaError_t _e = (expr);                                                                       \
    if (_e != cudaSuccess) {                                                                       \
      fo::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__);   \
      return fo::ws_fail(FO_ERR_CUDA);                                                             \
    }                                                                                              \
  } while (0)

extern "C" int fo_version(void) { return FO_ABI_VERSION; }
extern "C" const char* fo_last_error(void) { return fo::g_err; }
extern "C" uint64_t fo_launch_count(void) { return fo::g_launches.load(std::memory_order_relaxed); }

// ---- peer-mapped buffers (CUDA IPC) ---------------------------------------------------------------------------------
static_assert(sizeof(FoPeerHandle) == sizeof(cudaIpcMemHandle_t), "FoPeerHandle carries a cudaIpcMemHandle_t");

extern "C" int fo_peer_alloc(size_t bytes, void** dev_ptr, FoPeerHandle* handle) {
  if (!dev_ptr || !handle || bytes == 0) { fo::set_error("fo_peer_alloc: bad argument"); return FO_ERR_INVALID_ARG; }
  void* p = nullptr;
  FO_CUDA_TRY(cudaMalloc(&p, bytes));
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaMemset(p, 0, bytes);
  if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, p);
  if (e != cudaSuccess) {
    cudaFree(p);
    fo::set_error("fo_peer_alloc: %s", cudaGetErrorString(e));
    return FO_ERR_CUDA;
  }
  memcpy(handle->bytes, &h, sizeof(h));
  *dev_ptr = p;
  return FO_OK;
}

extern "C" int fo_peer_open(const FoPeerHandle* handle, void** dev_ptr) {
  if (!dev_ptr || !handle) { fo::set_error("fo_peer_open: bad argument"); return FO_ERR_INVALID_ARG; }
  cudaIpcMemHandle_t h;
  memcpy(&h, handle->bytes, sizeof(h));
  FO_CUDA_TRY(cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return FO_OK;
}

extern "C" int fo_peer_close(void* dev_ptr) {
  if (dev_ptr) FO_CUDA_TRY(cudaIpcCloseMemHandle(dev_ptr));
  return FO_OK;
}

extern "C" int fo_peer_free(void* dev_ptr) {
  if (dev_ptr) FO_CUDA_TRY(cudaFree(dev_ptr));
  return FO_OK;
}

extern "C" int fo_probe_fp32_peak(int32_t iters, float* ms, double* flops, void* stream) {
  if (iters <= 0 || !ms || !flops) { fo::set_error("fo_probe_fp32_peak: bad argument"); return FO_ERR_INVALID_ARG; }
  int dev = 0, sms = 0;
  FO_CUDA_TRY(cudaGetDevice(&dev));
  FO_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  float* sink = nullptr;
  FO_CUDA_TRY(cudaMalloc(&sink, 4));
  cudaEvent_t e0, e1;
  FO_CUDA_TRY(cudaEventCreate(&e0));
  FO_CUDA_TRY(cudaEventCreate(&e1));
  cudaStream_t st = (cudaStream_t)stream;
  const int grid = sms * 8;
  fo::fp32_probe_kernel<<<grid, 256, 0, st>>>(iters / 8 + 1, 1.0f, sink);  // warm-up
  FO_CUDA_TRY(cudaEventRecord(e0, st));
  fo::fp32_probe_kernel<<<grid, 256, 0, st>>>(iters, 1.0f, sink);
  FO_CUDA_TRY(cudaEventRecord(e1, st));
  fo::count_launch(2);
  FO_CUDA_TRY(cudaEventSynchronize(e1));
  FO_CUDA_TRY(cudaEventElapsedTime(ms, e0, e1));
  *flops = 2.0 * 8.0 * (double)iters * 256.0 * (double)grid;
  cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(sink);
  return FO_OK;
}

extern "C" int fo_metric_bundle_host(const float* ego_host, int32_t n_traj, int32_t n_states, const FoAgentsRaw* ag,
                                     const FoMetricArgs* params, uint8_t* out_valid, float* out_summary,
                                     uint32_t* out_flags, float* out_pair, float* out_step) {
  if (!params || !ag || (n_traj > 0 && (!ego_host || !out_valid))) {
    fo::set_error("fo_metric_bundle_host: NULL argument");
    return FO_ERR_INVALID_ARG;
  }
  if (n_traj < 0 || n_states < 0 || ag->n_agents < 0 || ag->t_stride < 0) {
    fo::set_error("fo_metric_bundle_host: negative size");
    return FO_ERR_INVALID_ARG;
  }
  if (n_traj == 0) return FO_OK;
  const size_t N = n_traj, T = n_states, A = ag->n_agents, Tp = ag->t_stride;
  auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
  const size_t b_ego = al(N * T * 5 * 4), b_f = al(A * Tp * 4), b_a = al(A * 4 + 4);
  const size_t b_tab = al(fo::agent_table_bytes((int)A, (int)Tp) + 16);
  const size_t b_valid = al(N), b_sum = al(N * FO_SUMMARY_K * 4), b_flags = al(N * 4);
  const size_t b_pair = out_pair ? al(N * A * FO_PAIR_K * 4 + 4) : 0;
  const size_t b_step = (out_step && T > 1) ? al(N * A * (T - 1) * FO_STEP_K * 4 + 4) : 0;
  const size_t total = b_ego + 6 * b_f + 6 * b_a + b_tab + b_valid + b_sum + b_flags + b_pair + b_step;
  int rc = fo::ws_reserve(total);
  if (rc != FO_OK) return rc;
  cudaStream_t st = fo::g_ws.stream;
  char* p = (char*)fo::g_ws.dev;
  auto take = [&](size_t b) { char* r = p; p += b; return r; };
  float* d_ego = (float*)take(b_ego);
  FoAgentsRaw d = *ag;
  const float* hsrc[6] = {ag->x, ag->y, ag->yaw, ag->v, ag->var_x, ag->var_y};
  const float** hdst[6] = {&d.x, &d.y, &d.yaw, &d.v, &d.var_x, &d.var_y};
  for (int i = 0; i < 6; ++i) {
    float* dp = (float*)take(b_f);
    if (A * Tp) {
      if (!hsrc[i]) { fo::set_error("fo_metric_bundle_host: NULL agent array"); return fo::ws_fail(FO_ERR_INVALID_ARG); }
      FO_HOST_TRY(cudaMemcpyAsync(dp, hsrc[i], A * Tp * 4, cudaMemcpyHostToDevice, st));
    }
    *hdst[i] = dp;
  }
  const void* asrc[6] = {ag->n_states, ag->kind, ag->length, ag->width, ag->buf_length, ag->buf_width};
  const void** adst[6] = {(const void**)&d.n_states, (const void**)&d.kind, (const void**)&d.length,
                          (const void**)&d.width, (const void**)&d.buf_length, (const void**)&d.buf_width};
  for (int i = 0; i < 6; ++i) {
    void* dp = take(b_a);
    if (A) {
      if (!asrc[i]) { fo::set_error("fo_metric_bundle_host: NULL agent array"); return fo::ws_fail(FO_ERR_INVALID_ARG); }
      FO_HOST_TRY(cudaMemcpyAsync(dp, asrc[i], A * 4, cudaMemcpyHostToDevice, st));
    }
    *adst[i] = dp;
  }
  void* d_tab = take(b_tab);
  FoMetricArgs m = *params;
  m.ego = d_ego; m.n_traj = n_traj; m.n_states = n_states; m.n_agents = (int32_t)A; m.t_stride = (int32_t)Tp;
  m.agent_table = d_tab;
  // Results go to the library's workspace -- or, when the caller names all three DEVICE destinations in `params`, there
  // (a rank's slice of a gather buffer: n_peers / peer_delta then apply as in fo_metric_bundle), and from there to the host.
  const bool dev_out = params->valid && params->summary && params->flags && !out_pair && !out_step;
  uint8_t* ws_valid = (uint8_t*)take(b_valid);
  float* ws_sum = (float*)take(b_sum);
  uint32_t* ws_flags = (uint32_t*)take(b_flags);
  if (dev_out) {
    m.valid = params->valid; m.summary = params->summary; m.flags = params->flags;
  } else {
    m.valid = ws_valid; m.summary = ws_sum; m.flags = ws_flags;
    m.n_peers = 0;
  }
  m.pair = out_pair ? (float*)take(b_pair) : nullptr;
  m.step = (out_step && T > 1) ? (float*)take(b_step) : nullptr;
  if (A > 0) {
    rc = fo_agents_pack(&d, &m.vehicle, d_tab, b_tab, st);
    if (rc != FO_OK) return fo::ws_fail(rc);
  }
  // Large bundles are pipelined: the trajectory range is cut into chunks, chunk k+1 crosses PCIe on the copy stream
  // while chunk k is evaluated (trajectories are independent), results follow each chunk back on the compute stream.
  // The first chunk is small (its copy cannot be hidden), every following one four times larger: copying is several
  // times faster than evaluating, and every launch costs a tail of about one trajectory time per warp.
  const size_t traj_bytes = T * 5 * 4;
  size_t bound[fo::kHostChunksMax + 1] = {0, N};
  const int chunks = (!m.pair && !m.step) ? fo::host_chunks(N, traj_bytes, bound) : 1;
  for (int c = 0; c < chunks; ++c) {
    const size_t lo = bound[c], hi = bound[c + 1], n = hi - lo;
    if (n == 0) continue;
    FO_HOST_TRY(cudaMemcpyAsync(d_ego + lo * T * 5, ego_host + lo * T * 5, n * traj_bytes, cudaMemcpyHostToDevice,
                                fo::g_ws.copy));
    FO_HOST_TRY(cudaEventRecord(fo::g_ws.ready[c], fo::g_ws.copy));
    FO_HOST_TRY(cudaStreamWaitEvent(st, fo::g_ws.ready[c], 0));
    FoMetricArgs mc = m;
    mc.ego = d_ego + lo * T * 5;
    mc.n_traj = (int32_t)n;
    mc.valid = m.valid + lo;
    mc.summary = m.summary + lo * FO_SUMMARY_K;
    mc.flags = m.flags + lo;
    if (m.pair) mc.pair = m.pair + lo * A * FO_PAIR_K;
    if (m.step) mc.step = m.step + lo * A * (T - 1) * FO_STEP_K;
    rc = fo_metric_bundle(&mc, st);
    if (rc != FO_OK) return fo::ws_fail(rc);
    FO_HOST_TRY(cudaMemcpyAsync(out_valid + lo, mc.valid, n, cudaMemcpyDeviceToHost, st));
    if (out_summary)
      FO_HOST_TRY(cudaMemcpyAsync(out_summary + lo * FO_SUMMARY_K, mc.summary, n * FO_SUMMARY_K * 4, cudaMemcpyDeviceToHost, st));
    if (out_flags) FO_HOST_TRY(cudaMemcpyAsync(out_flags + lo, mc.flags, n * 4, cudaMemcpyDeviceToHost, st));
  }
  if (m.pair) FO_HOST_TRY(cudaMemcpyAsync(out_pair, m.pair, N * A * FO_PAIR_K * 4, cudaMemcpyDeviceToHost, st));
  if (m.step) FO_HOST_TRY(cudaMemcpyAsync(out_step, m.step, N * A * (T - 1) * FO_STEP_K * 4, cudaMemcpyDeviceToHost, st));
  FO_HOST_TRY(cudaStreamSynchronize(st));
  return FO_OK;
}

namespace fo {

// Page-locked host buffers of fo_metric_batch_host_select, per calling thread, grown on demand: `in` holds a round's
// window table and, for pageable callers, the window rows the device reads; `out` receives a round's results.
struct PinnedBuf {
  unsigned char* p = nullptr;
  size_t bytes = 0;
};
static thread_local PinnedBuf g_pin_in, g_pin_out;

static int pin_reserve(PinnedBuf& b, size_t bytes) {
  if (bytes <= b.bytes) return FO_OK;
  if (b.p) FO_CUDA_TRY(cudaFreeHost(b.p));
  b.p = nullptr; b.bytes = 0;
  const size_t want = bytes + bytes / 4 > 4096 ? bytes + bytes / 4 : 4096;
  FO_CUDA_TRY(cudaMallocHost(&b.p, want));
  b.bytes = want;
  return FO_OK;
}

// The rounds of fo_metric_batch_host_select (DESIGN.md 5.15), after the agents are packed: b is the whole batch with the
// library's arena in place (problems pr = b->problems, n_run of them with rows, the fewest agents among those a_min);
// corr / veh per problem (corr NULL = none correlated); d_e32 room for n_traj float32 rows, d_win for n_run windows,
// d_res for n_traj result rows and n_run selections.
static int host_select_rounds(const char* fn, const double* ego_host, const double* origins_host,
                              const FoMetricBatchArgs* b, int n_run, int a_min, const uint8_t* corr, const FoVehicle* veh,
                              float* d_e32, IngestWindow* d_win, unsigned char* d_res, int32_t* out_selected,
                              uint8_t* out_valid, float* out_summary, uint32_t* out_flags) {
  const FoMetricArgs& c = b->common;
  const int P = b->n_problems, T = c.n_states;
  const FoBatchProblem* pr = b->problems;
  const size_t row_elems = (size_t)T * 5;
  cudaStream_t st = g_ws.stream;
  // every round's team size and shape classes are those fo_metric_batch_host_corr picks for the whole batch
  int W = 1, teams = 1;
  int rc = batch_team_shape(c.n_traj, T, a_min, &W, &teams);
  if (rc != FO_OK) return rc;
  // page-locked or registered rows are read in place; pageable ones are copied window by window into g_pin_in
  const double* mapped = nullptr;
  {
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, ego_host) == cudaSuccess && at.devicePointer)
      mapped = static_cast<const double*>(at.devicePointer);
    cudaGetLastError();
  }
  // round 0 gives every problem w0 ranks: together at least one per resident team
  const int w0 = std::max(32, (teams + n_run - 1) / n_run);
  std::vector<int> active, start(P, 0), next_len(P, w0);
  for (int p = 0; p < P; ++p) {
    out_selected[p] = pr[p].n_traj;                  // N_p; 0 for a problem without rows
    if (pr[p].n_traj > 0) active.push_back(p);
  }
  memset(out_valid, FO_VALID_SKIPPED, (size_t)c.n_traj);
  std::vector<FoBatchProblem> wp;
  std::vector<uint8_t> wcorr;
  std::vector<FoVehicle> wveh;
  const size_t tab_bytes = ((size_t)n_run * sizeof(IngestWindow) + 255) & ~(size_t)255;
  while (!active.empty()) {
    const int n_win = (int)active.size();
    // ---- the window table: problem p's ranks [start, start + len) become compact rows [rows, rows + len)
    int rows = 0;
    for (int i = 0; i < n_win; ++i) {
      const int p = active[i];
      rows += std::min(next_len[p], pr[p].n_traj - start[p]);
    }
    rc = pin_reserve(g_pin_in, tab_bytes + (mapped ? 0 : (size_t)rows * row_elems * sizeof(double)));
    if (rc != FO_OK) return rc;
    IngestWindow* win = reinterpret_cast<IngestWindow*>(g_pin_in.p);
    double* staged = reinterpret_cast<double*>(g_pin_in.p + tab_bytes);
    wp.assign(n_win, FoBatchProblem{});
    wcorr.assign(n_win, 0);
    wveh.assign(n_win, FoVehicle{});
    for (int i = 0, at = 0; i < n_win; ++i) {
      const int p = active[i];
      const int len = std::min(next_len[p], pr[p].n_traj - start[p]);
      const long long src_row = pr[p].traj_begin + start[p];
      if (!mapped) memcpy(staged + (size_t)at * row_elems, ego_host + (size_t)src_row * row_elems, (size_t)len * row_elems * 8);
      win[i] = IngestWindow{mapped ? src_row : at, at, len, make_double2(origins_host[2 * p], origins_host[2 * p + 1])};
      wp[i] = pr[p];
      wp[i].traj_begin = at;
      wp[i].n_traj = len;
      wcorr[i] = corr ? corr[p] : 0;
      wveh[i] = veh[p];
      at += len;
    }
    // ---- the window rows in float32, then the select launches over them (one descriptor per window)
    FO_CUDA_TRY(cudaMemcpyAsync(d_win, win, (size_t)n_win * sizeof(IngestWindow), cudaMemcpyHostToDevice, st));
    const double* src = mapped;
    if (!mapped) FO_CUDA_TRY(cudaHostGetDevicePointer((void**)&src, staged, 0));
    rc = launch_ego_window_ingest(src, d_e32, rows, T, d_win, n_win, st);
    if (rc != FO_OK) return rc;
    // results of the round back to back, for one read-back: summary, flags, selections, valid bytes
    const size_t sum_bytes = out_summary ? (size_t)rows * FO_SUMMARY_K * 4 : 0, flag_bytes = out_flags ? (size_t)rows * 4 : 0;
    const size_t sel_off = sum_bytes + flag_bytes, valid_off = sel_off + (size_t)n_win * 4, res_bytes = valid_off + rows;
    FoMetricBatchArgs rb = *b;
    rb.common.ego = d_e32;
    rb.common.n_traj = rows;
    rb.common.summary = out_summary ? reinterpret_cast<float*>(d_res) : nullptr;
    rb.common.flags = out_flags ? reinterpret_cast<uint32_t*>(d_res + sum_bytes) : nullptr;
    rb.common.valid = d_res + valid_off;
    rb.n_problems = n_win;
    rb.problems = wp.data();
    rc = metric_batch_select_w(fn, &rb, corr ? wcorr.data() : nullptr, wveh.data(), W,
                               reinterpret_cast<int32_t*>(d_res + sel_off), st);
    if (rc != FO_OK) return rc;
    rc = pin_reserve(g_pin_out, res_bytes);
    if (rc != FO_OK) return rc;
    FO_CUDA_TRY(cudaMemcpyAsync(g_pin_out.p, d_res, res_bytes, cudaMemcpyDeviceToHost, st));
    FO_CUDA_TRY(cudaStreamSynchronize(st));
    // ---- scatter: an assessed row's results go to its place; a window with a valid row finishes its problem
    const float* h_sum = reinterpret_cast<const float*>(g_pin_out.p);
    const uint32_t* h_flags = reinterpret_cast<const uint32_t*>(g_pin_out.p + sum_bytes);
    const int32_t* h_sel = reinterpret_cast<const int32_t*>(g_pin_out.p + sel_off);
    const uint8_t* h_valid = g_pin_out.p + valid_off;
    int kept = 0;
    for (int i = 0; i < n_win; ++i) {
      const int p = active[i], at = (int)wp[i].traj_begin, len = wp[i].n_traj;
      const size_t dst = (size_t)pr[p].traj_begin + start[p];
      for (int r = 0; r < len; ++r) {
        const uint8_t v = h_valid[at + r];
        out_valid[dst + r] = v;
        if (v == FO_VALID_SKIPPED) continue;
        if (out_summary) memcpy(out_summary + (dst + r) * FO_SUMMARY_K, h_sum + (size_t)(at + r) * FO_SUMMARY_K, FO_SUMMARY_K * 4);
        if (out_flags) out_flags[dst + r] = h_flags[at + r];
      }
      if (h_sel[i] < len) {
        out_selected[p] = start[p] + h_sel[i];
      } else if (start[p] + len < pr[p].n_traj) {      // no valid row in the window: the next, four times longer
        start[p] += len;
        next_len[p] = (int)std::min<long long>(4ll * next_len[p], pr[p].n_traj);
        active[kept++] = p;
      }
    }
    active.resize(kept);
  }
  return FO_OK;
}

}  // namespace fo

// fo_metric_batch_host, fo_metric_batch_host_corr and (select) fo_metric_batch_host_select.  corr: NULL = every table
// diagonal; else corr[p] != 0 = problem p's table is a correlated one, its off-diagonal terms in cov_xy (host, aligned
// with ag->var_x / var_y).  The pack and metric calls are the *_corr ones either way.
static int metric_batch_host_impl(const char* fn, const double* ego_host, int32_t n_traj, int32_t n_states,
                                  const double* origins_host, const FoAgentsRaw* ag, const float* cov_xy, int32_t n_problems,
                                  const FoBatchProblem* problems_host, const uint8_t* corr, const FoVehicle* vehicles_host,
                                  const FoMetricArgs* params, uint8_t* out_valid, float* out_summary, uint32_t* out_flags,
                                  float* out_pair, float* out_step, bool select = false, int32_t* out_selected = nullptr) {
  const int P = n_problems;
  // ---- every check before any device work
  if (!params) { fo::set_error("%s: NULL params", fn); return FO_ERR_INVALID_ARG; }
  if (params->n_peers != 0) { fo::set_error("%s: peer stores exist on the device entry points only", fn); return FO_ERR_UNSUPPORTED; }
  if (select && P > 0 && !out_selected) { fo::set_error("%s: out_selected must not be NULL with %d problems", fn, P); return FO_ERR_INVALID_ARG; }
  if (P > 0 && (!problems_host || !origins_host || !ag)) {
    fo::set_error("%s: NULL problems / origins / agents with %d problems", fn, P);
    return FO_ERR_INVALID_ARG;
  }
  if (n_traj > 0 && (!ego_host || !out_valid)) { fo::set_error("%s: NULL ego / out_valid", fn); return FO_ERR_INVALID_ARG; }
  // The library owns the arena: problem p's table goes where fo_agent_batch_layout[_corr] puts it.  Sizes out of range
  // take no bytes here; the batch calls' own checks below reject them.
  std::vector<FoBatchProblem> pr(P > 0 ? P : 0);
  size_t arena_bytes = 0;
  for (int p = 0; p < P; ++p) {
    pr[p] = problems_host[p];
    pr[p].table_offset = (int64_t)arena_bytes;
    const int A = pr[p].n_agents, Tp = pr[p].t_stride;
    if (A > 0 && Tp > 0 && Tp <= FO_MAX_STATES)
      arena_bytes += ((corr && corr[p] ? fo::agent_table_bytes_corr(A, Tp) : fo::agent_table_bytes(A, Tp)) + 15) & ~(size_t)15;
  }
  // the workspace is not placed yet: an aligned stand-in takes the place of its buffers in the checks
  alignas(16) static float stand_in[4];
  FoMetricBatchArgs b{};
  b.common = *params;
  b.common.ego = stand_in; b.common.n_traj = n_traj; b.common.n_states = n_states;
  b.common.agent_table = stand_in; b.common.n_agents = 0; b.common.t_stride = 1;
  b.common.valid = (uint8_t*)stand_in; b.common.summary = stand_in; b.common.flags = (uint32_t*)stand_in;
  b.common.pair = b.common.step = nullptr;
  b.n_problems = P; b.problems = pr.data(); b.arena_bytes = arena_bytes;
  int n_run = 0, a_min = 0, n_packed = 0, max_cells = 0;
  int rc = fo::check_batch(fn, &b, corr, false, &n_run, &a_min);
  if (rc != FO_OK) return rc;
  const FoAgentsRaw no_agents{};
  rc = fo::check_pack_batch(fn, P > 0 ? ag : &no_agents, P, pr.data(), corr, stand_in, arena_bytes, &n_packed, &max_cells);
  if (rc != FO_OK) return rc;
  // The correlated problems with agents: their covariances are in host memory here, so the states the correlation pack
  // reads (covariance i-1 of every state i < min(n_states, t_stride_p), as fo_agents_corr_kernel) are checked now, with
  // its own predicate, and a covariance that would give NaN collision probabilities on the device is an error.
  int n_corr = 0;
  for (int p = 0, a0 = 0; corr && p < P; a0 += pr[p].n_agents, ++p) {
    if (!corr[p] || pr[p].n_agents == 0) continue;
    if (!cov_xy) { fo::set_error("%s: cov_xy must not be NULL with correlated problems (problem %d)", fn, p); return FO_ERR_INVALID_ARG; }
    ++n_corr;
    const int Tp = pr[p].t_stride;
    for (int a = 0; a < pr[p].n_agents; ++a) {
      const int n = ag->n_states[a0 + a] < Tp ? ag->n_states[a0 + a] : Tp;
      const size_t row = (size_t)(a0 + a) * ag->t_stride;
      for (int i = 0; i < n; ++i) {
        const size_t ip = row + (i > 0 ? i - 1 : 0);
        double sx, sy, rho;
        if (!fo::corr_terms(ag->var_x[ip], ag->var_y[ip], cov_xy[ip], &sx, &sy, &rho)) {
          fo::set_error("%s: problem %d, agent %d: covariance %d is not positive definite", fn, p, a, i > 0 ? i - 1 : 0);
          return FO_ERR_INVALID_ARG;
        }
      }
    }
  }
  if (n_traj == 0) {                             // every N_p is 0
    for (int q = 0; select && q < P; ++q) out_selected[q] = 0;
    return FO_OK;
  }

  // ---- workspace: float64 rows, float32 bundle, raw agents (with cov_xy when correlated), arena, per-problem ingest
  // table, outputs (select: no float64 rows; a window table, and the outputs hold one round's results in one block)
  const size_t N = n_traj, T = n_states, A = ag->n_agents, S = ag->t_stride;
  long long pairs = 0;                           // sum of N_p A_p: the rows of the pair / step blocks
  for (int p = 0; p < P; ++p) pairs += (long long)pr[p].n_traj * pr[p].n_agents;
  // as MetricEngine.assess_batch: with no pair or step left to write the summary path runs
  const bool want_pair = out_pair && pairs > 0, want_step = out_step && pairs > 0 && T > 1;
  auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
  const size_t b_e64 = select ? 0 : al(N * T * 5 * 8), b_e32 = al(N * T * 5 * 4), b_f = al(A * S * 4), b_a = al(A * 4 + 4);
  const size_t b_first = ((size_t)n_run * 4 + 15) & ~(size_t)15, b_idx = al(b_first + (size_t)n_run * 16);
  const size_t b_arena = al(arena_bytes), b_valid = al(N), b_sum = al(N * FO_SUMMARY_K * 4), b_flags = al(N * 4);
  const size_t b_pair = want_pair ? al((size_t)pairs * FO_PAIR_K * 4) : 0;
  const size_t b_step = want_step ? al((size_t)pairs * (T - 1) * FO_STEP_K * 4) : 0;
  const size_t b_cov = corr ? b_f : 0;
  const size_t b_win = select ? al((size_t)n_run * sizeof(fo::IngestWindow)) : 0, b_sel = select ? al((size_t)n_run * 4) : 0;
  rc = fo::ws_reserve(b_e64 + b_e32 + 6 * b_f + b_cov + 6 * b_a + b_idx + b_arena + b_valid + b_sum + b_flags + b_pair +
                      b_step + b_win + b_sel);
  if (rc != FO_OK) return rc;
  cudaStream_t st = fo::g_ws.stream;
  char* p = (char*)fo::g_ws.dev;
  auto take = [&](size_t b) { char* r = p; p += b; return r; };
  double* d_e64 = (double*)take(b_e64);
  float* d_e32 = (float*)take(b_e32);

  // ---- agents: upload, then one pack call into the library's arena (overlaps the first ego chunk's upload)
  FoAgentsRaw d = *ag;
  const float* hsrc[6] = {ag->x, ag->y, ag->yaw, ag->v, ag->var_x, ag->var_y};
  const float** hdst[6] = {&d.x, &d.y, &d.yaw, &d.v, &d.var_x, &d.var_y};
  const void* asrc[6] = {ag->n_states, ag->kind, ag->length, ag->width, ag->buf_length, ag->buf_width};
  const void** adst[6] = {(const void**)&d.n_states, (const void**)&d.kind, (const void**)&d.length,
                          (const void**)&d.width, (const void**)&d.buf_length, (const void**)&d.buf_width};
  for (int i = 0; i < 6; ++i) {
    float* dp = (float*)take(b_f);
    if (n_packed) FO_HOST_TRY(cudaMemcpyAsync(dp, hsrc[i], A * S * 4, cudaMemcpyHostToDevice, st));
    *hdst[i] = dp;
  }
  for (int i = 0; i < 6; ++i) {
    void* dp = take(b_a);
    if (n_packed) FO_HOST_TRY(cudaMemcpyAsync(dp, asrc[i], A * 4, cudaMemcpyHostToDevice, st));
    *adst[i] = dp;
  }
  float* d_cov = corr ? (float*)take(b_cov) : nullptr;
  if (n_corr) FO_HOST_TRY(cudaMemcpyAsync(d_cov, cov_xy, A * S * 4, cudaMemcpyHostToDevice, st));
  // the ingest table: first rows and origins of the problems with trajectories
  std::vector<unsigned char> idx(b_first + (size_t)n_run * 16);
  int* first = (int*)idx.data();
  double* org = (double*)(idx.data() + b_first);
  for (int q = 0, i = 0; q < P; ++q) {
    if (pr[q].n_traj == 0) continue;
    first[i] = (int)pr[q].traj_begin;
    org[2 * i] = origins_host[2 * q];
    org[2 * i + 1] = origins_host[2 * q + 1];
    ++i;
  }
  char* d_idx = take(b_idx);
  FO_HOST_TRY(cudaMemcpyAsync(d_idx, idx.data(), idx.size(), cudaMemcpyHostToDevice, st));
  void* d_arena = take(b_arena);
  // the *_corr calls take a flag and a vehicle per problem: without corr none is correlated, without vehicles_host every
  // problem has params->vehicle (with every flag 0 they make the launches of the diagonal calls)
  const std::vector<uint8_t> no_corr(corr ? 0 : P, 0);
  const uint8_t* corr_flags = corr ? corr : no_corr.data();
  const std::vector<FoVehicle> shared(vehicles_host ? 0 : P, params->vehicle);
  const FoVehicle* veh = vehicles_host ? vehicles_host : shared.data();
  if (n_packed) {
    rc = fo_agents_pack_batch_corr(&d, n_corr ? d_cov : nullptr, P, pr.data(), corr_flags, veh, d_arena, arena_bytes, st);
    if (rc != FO_OK) return fo::ws_fail(rc);
  }
  b.common.agent_table = arena_bytes ? d_arena : nullptr;
  if (select) {                                  // rank windows in rounds instead of every row at once
    fo::IngestWindow* d_win = (fo::IngestWindow*)take(b_win);
    unsigned char* d_res = (unsigned char*)take(b_valid + b_sum + b_flags + b_sel);
    rc = fo::host_select_rounds(fn, ego_host, origins_host, &b, n_run, a_min, corr, veh, d_e32, d_win, d_res, out_selected,
                                out_valid, out_summary, out_flags);
    if (rc != FO_OK) return fo::ws_fail(rc);
    return FO_OK;
  }

  // ---- ego: chunk k+1 crosses PCIe on the copy stream while chunk k is converted on the compute stream
  const size_t row_bytes = T * 5 * 8;
  size_t bound[fo::kHostChunksMax + 1];
  const int chunks = fo::host_chunks(N, row_bytes, bound);
  for (int c = 0; c < chunks; ++c) {
    const size_t lo = bound[c], n = bound[c + 1] - lo;
    if (n == 0) continue;
    FO_HOST_TRY(cudaMemcpyAsync(d_e64 + lo * T * 5, ego_host + lo * T * 5, n * row_bytes, cudaMemcpyHostToDevice,
                                fo::g_ws.copy));
    FO_HOST_TRY(cudaEventRecord(fo::g_ws.ready[c], fo::g_ws.copy));
    FO_HOST_TRY(cudaStreamWaitEvent(st, fo::g_ws.ready[c], 0));
    rc = fo::launch_ego_ingest(d_e64 + lo * T * 5, d_e32 + lo * T * 5, (int)lo, (int)n, (int)T, (const int*)d_idx,
                               (const double2*)(d_idx + b_first), n_run, st);
    if (rc != FO_OK) return fo::ws_fail(rc);
  }

  // ---- the batch call itself, after the last chunk is converted (one W for the whole batch)
  b.common.ego = d_e32;
  b.common.valid = (uint8_t*)take(b_valid);
  b.common.summary = (float*)take(b_sum);
  b.common.flags = (uint32_t*)take(b_flags);
  b.common.pair = want_pair ? (float*)take(b_pair) : nullptr;
  b.common.step = want_step ? (float*)take(b_step) : nullptr;
  rc = (want_pair || want_step) ? fo_metric_batch_detail_corr(&b, corr_flags, veh, st)
                                 : fo_metric_batch_corr(&b, corr_flags, veh, st);
  if (rc != FO_OK) return fo::ws_fail(rc);

  // ---- results back, then synchronise
  FO_HOST_TRY(cudaMemcpyAsync(out_valid, b.common.valid, N, cudaMemcpyDeviceToHost, st));
  if (out_summary)
    FO_HOST_TRY(cudaMemcpyAsync(out_summary, b.common.summary, N * FO_SUMMARY_K * 4, cudaMemcpyDeviceToHost, st));
  if (out_flags) FO_HOST_TRY(cudaMemcpyAsync(out_flags, b.common.flags, N * 4, cudaMemcpyDeviceToHost, st));
  if (want_pair)
    FO_HOST_TRY(cudaMemcpyAsync(out_pair, b.common.pair, (size_t)pairs * FO_PAIR_K * 4, cudaMemcpyDeviceToHost, st));
  if (want_step)
    FO_HOST_TRY(cudaMemcpyAsync(out_step, b.common.step, (size_t)pairs * (T - 1) * FO_STEP_K * 4, cudaMemcpyDeviceToHost, st));
  FO_HOST_TRY(cudaStreamSynchronize(st));
  return FO_OK;
}

extern "C" int fo_metric_batch_host(const double* ego_host, int32_t n_traj, int32_t n_states, const double* origins_host,
                                    const FoAgentsRaw* ag, int32_t n_problems, const FoBatchProblem* problems_host,
                                    const FoVehicle* vehicles_host, const FoMetricArgs* params, uint8_t* out_valid,
                                    float* out_summary, uint32_t* out_flags, float* out_pair, float* out_step) {
  return metric_batch_host_impl("fo_metric_batch_host", ego_host, n_traj, n_states, origins_host, ag, nullptr, n_problems,
                                problems_host, nullptr, vehicles_host, params, out_valid, out_summary, out_flags, out_pair,
                                out_step);
}

extern "C" int fo_metric_batch_host_corr(const double* ego_host, int32_t n_traj, int32_t n_states,
                                         const double* origins_host, const FoAgentsRaw* ag, const float* cov_xy_host,
                                         int32_t n_problems, const FoBatchProblem* problems_host, const uint8_t* corr_host,
                                         const FoVehicle* vehicles_host, const FoMetricArgs* params, uint8_t* out_valid,
                                         float* out_summary, uint32_t* out_flags, float* out_pair, float* out_step) {
  const char* fn = "fo_metric_batch_host_corr";
  if (n_problems > 0 && !corr_host) { fo::set_error("%s: corr_host must not be NULL", fn); return FO_ERR_INVALID_ARG; }
  // (with no problems there is nothing to assess: NULL flags reach no pack or metric call)
  return metric_batch_host_impl(fn, ego_host, n_traj, n_states, origins_host, ag, cov_xy_host, n_problems, problems_host,
                                corr_host, vehicles_host, params, out_valid, out_summary, out_flags, out_pair, out_step);
}

extern "C" int fo_metric_batch_host_select(const double* ego_host, int32_t n_traj, int32_t n_states,
                                           const double* origins_host, const FoAgentsRaw* ag, const float* cov_xy_host,
                                           int32_t n_problems, const FoBatchProblem* problems_host, const uint8_t* corr_host,
                                           const FoVehicle* vehicles_host, const FoMetricArgs* params, int32_t* out_selected,
                                           uint8_t* out_valid, float* out_summary, uint32_t* out_flags) {
  return metric_batch_host_impl("fo_metric_batch_host_select", ego_host, n_traj, n_states, origins_host, ag, cov_xy_host,
                                n_problems, problems_host, corr_host, vehicles_host, params, out_valid, out_summary,
                                out_flags, nullptr, nullptr, true, out_selected);
}
