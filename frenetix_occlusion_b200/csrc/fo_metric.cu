// Host entry points of the dense metric core: agent-table packing and kernel dispatch.
#include <math.h>
#include <stdlib.h>

#include <algorithm>
#include <atomic>
#include <vector>

#include "fo_metric_dev.cuh"

namespace fo {

// ---------------------------------------------------------------------------------------------
// fo_agents_pack kernel: one thread per (agent, state).
__device__ __forceinline__ float obstacle_mass(int kind, float size) {  // harm_model.py:158-190
  switch (kind) {
    case FO_KIND_CAR: case FO_KIND_PRIORITY_VEHICLE: case FO_KIND_PARKED_VEHICLE: case FO_KIND_TAXI:
      return -1333.5f + 526.9f * powf(size, 0.8f);
    case FO_KIND_TRUCK: return 25000.0f;
    case FO_KIND_BUS: return 13000.0f;
    case FO_KIND_BICYCLE: return 90.0f;
    case FO_KIND_PEDESTRIAN: return 75.0f;
    case FO_KIND_TRAIN: return 118800.0f;
    case FO_KIND_MOTORCYCLE: return 250.0f;
    default: return 0.0f;
  }
}
__device__ __forceinline__ int protection_model(int kind) {  // harm_model.py:15-32
  switch (kind) {
    case FO_KIND_BICYCLE: case FO_KIND_PEDESTRIAN: case FO_KIND_MOTORCYCLE: case FO_KIND_UNKNOWN: return 0;
    default: return 1;
  }
}

// One problem of a packing launch: its agents are rows [a_begin, a_begin + A) of the raw arrays (row stride
// raw.t_stride), its table (stride Tp) starts table_off bytes into the arena, m_ego is its ego vehicle's mass (harm
// mass split).  fo_agents_pack is the one-problem case.
struct PackProblem {
  int a_begin, A, Tp;
  float m_ego;
  long long table_off;
};

// Slot order: stable sort by harm model.  One CTA per problem; A is a few hundred at most, so the O(A^2) rank count is free.
__global__ void fo_agents_order_kernel(const int32_t* __restrict__ kind_all, PackProblem one, const PackProblem* many,
                                       unsigned char* arena) {
  const PackProblem pp = many ? many[blockIdx.x] : one;
  const int A = pp.A;
  const AgentTableView v = agent_table_view(arena + pp.table_off, A, pp.Tp);
  const int Ap = v.Ap;
  int32_t* orig = const_cast<int32_t*>(v.orig);
  int32_t* slot = const_cast<int32_t*>(v.slot);
  const int32_t* kind = kind_all + pp.a_begin;
  for (int a = threadIdx.x; a < Ap; a += blockDim.x) {
    if (a >= A) { orig[a] = -1; slot[a] = a; continue; }      // padding slots keep their place behind the real ones
#ifdef FO_NO_SORT
    slot[a] = a; orig[a] = a; continue;
#endif
    const int m = protection_model(kind[a]);
    int rank = 0;
    for (int b = 0; b < A; ++b) {
      const int mb = protection_model(kind[b]);
      rank += (mb < m) | ((mb == m) & (b < a));
    }
    slot[a] = rank;
    orig[rank] = a;
  }
}

// one thread per (agent slot, state) of a problem; blockIdx.y strides over the problems
__global__ void fo_agents_pack_kernel(FoAgentsRaw raw, PackProblem one, const PackProblem* many, int P,
                                      unsigned char* arena) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const int S = raw.t_stride;
  for (int p = blockIdx.y; p < P; p += gridDim.y) {
    const PackProblem pp = many ? many[p] : one;
    const int A = pp.A, Tp = pp.Tp;
    const AgentTableView v = agent_table_view(arena + pp.table_off, A, Tp);
    const int Ap = v.Ap;
    float4* s0 = const_cast<float4*>(v.s0);
    float4* s1 = const_cast<float4*>(v.s1);
    float2* s2 = const_cast<float2*>(v.s2);
    float4* t0 = const_cast<float4*>(v.t0);
    float* tv = const_cast<float*>(v.tv);
    float* tpsi = const_cast<float*>(v.tpsi);
    const int32_t* orig = v.orig;
    const int32_t* slot = v.slot;
    const size_t r0 = (size_t)pp.a_begin * S;     // raw element of (agent 0, state 0) of this problem
    const int nW = agent_windows(Tp);
    if (idx < Ap * nW) {                       // window boxes for the summary kernel's filter (slot order)
      const int sl = idx / nW, wi = idx - sl * nW;
      float xl = 1e30f, xh = -1e30f, yl = 1e30f, yh = -1e30f, vm = 0.0f;
      if (sl < A) {
        const int a = orig[sl];
        const int nS = min(raw.n_states[pp.a_begin + a], Tp);
        const int lo = wi * kWinSteps;
        for (int i = max(lo - 1, 0); i < min(lo + kWinSteps, nS); ++i) {
          const size_t r = r0 + (size_t)a * S + i;
          const float x = raw.x[r], y = raw.y[r];
          xl = fminf(xl, x); xh = fmaxf(xh, x); yl = fminf(yl, y); yh = fmaxf(yh, y);
          if (i >= lo) vm = fmaxf(vm, fabsf(raw.v[r]));
        }
      }
      const_cast<float4*>(v.aw)[(size_t)wi * Ap + sl] = make_float4(xl, xh, yl, yh);
      const_cast<float*>(v.avw)[(size_t)wi * Ap + sl] = vm;
    }
    if (idx >= A * Tp && idx < Ap * Tp) {      // padding slots of the time-major copies
      const int sl = idx / Tp, i = idx - sl * Tp;
      t0[(size_t)i * Ap + sl] = make_float4(0, 0, 1, 0);
      tv[(size_t)i * Ap + sl] = 0.0f;
      tpsi[(size_t)i * Ap + sl] = 0.0f;
    }
    if (idx < A * Tp) {
      const int a = idx / Tp, i = idx - a * Tp;
      const int sl = slot[a];
      const size_t r = r0 + (size_t)a * S + i;
      float4 o0 = make_float4(0, 0, 1, 0), o1 = make_float4(0, 0, 0, 0);
      float2 o2 = make_float2(1, 1);
      if (i < raw.n_states[pp.a_begin + a]) {
        float yaw = raw.yaw[r];
        float sn, cs;
        sincosf(yaw, &sn, &cs);
        const size_t ip = i > 0 ? r - 1 : r;   // state i-1 (CP pairs ego step i with agent position / covariance i-1)
        float vx = raw.var_x[ip], vy = raw.var_y[ip];
        if (vx == 0.0f && vy == 0.0f) { vx = 0.1f; vy = 0.1f; }  // collision_probability.py:85-87
        o0 = make_float4(raw.x[r], raw.y[r], cs, sn);
        o1 = make_float4(yaw, raw.v[r], raw.x[ip], raw.y[ip]);
        o2 = make_float2(rsqrtf(2.0f * vx), rsqrtf(2.0f * vy));
      }
      const size_t am = (size_t)sl * Tp + i, tm = (size_t)i * Ap + sl;
      s0[am] = o0;
      s1[am] = o1;
      s2[am] = o2;
      t0[tm] = o0;
      tv[tm] = o1.y;
      tpsi[tm] = o1.x;
    }
    if (idx < A) {
      const int g = pp.a_begin + idx;
      AgentParams q;
      q.n_states = raw.n_states[g];
      q.model = protection_model(raw.kind[g]);
      q.hl = 0.5f * raw.length[g];
      q.hw = 0.5f * raw.width[g];
      q.hlb = 0.5f * raw.buf_length[g];
      float mo = obstacle_mass(raw.kind[g], raw.buf_length[g] * raw.buf_width[g]);  // harm_model.py:73,78
      q.ke = mo / (pp.m_ego + mo);
      q.ko = pp.m_ego / (pp.m_ego + mo);
      q.pad = sqrtf(q.hl * q.hl + q.hw * q.hw);   // circumradius of the unbuffered rectangle (distance lower bound)
      const_cast<AgentParams*>(v.prm)[slot[idx]] = q;
    }
  }
}
static void launch_pack(const FoAgentsRaw& raw, const PackProblem& one, const PackProblem* many, int P, int max_cells,
                        unsigned char* arena, cudaStream_t st) {
  fo_agents_order_kernel<<<P, 256, 0, st>>>(raw.kind, one, many, arena);
  const dim3 grid((max_cells + 255) / 256, P < 65535 ? P : 65535);
  fo_agents_pack_kernel<<<grid, 256, 0, st>>>(raw, one, many, P, arena);
}

// The s3 section of a correlated table (fo_agents_pack_corr), one thread per (agent, state), after the two launches of
// launch_pack (it reads their slot map): (1/sigma_x, 1/sigma_y, rho) of covariance i-1 in float64, then rounded.  The
// zero rule of the diagonal pack applies to the all-zero matrix; a covariance that is not positive definite gets
// rho = NaN (|rho| >= 1, a zero variance with a non-zero covariance: +-inf / NaN here), so its CP values are NaN.
// Problems as in fo_agents_pack_kernel (blockIdx.y strides over them); fo_agents_pack_corr is the one-problem case.
__global__ void fo_agents_corr_kernel(FoAgentsRaw raw, const float* __restrict__ cov_xy, PackProblem one,
                                      const PackProblem* many, int P, unsigned char* arena) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  for (int p = blockIdx.y; p < P; p += gridDim.y) {
    const PackProblem pp = many ? many[p] : one;
    const int A = pp.A, Tp = pp.Tp;
    if (idx >= A * Tp) continue;
    const int a = idx / Tp, i = idx - a * Tp;
    unsigned char* const table = arena + pp.table_off;
    const int32_t* slot = agent_table_view(table, A, Tp).slot;
    float4 o = make_float4(1, 1, 0, 0);
    if (i < raw.n_states[pp.a_begin + a]) {
      const size_t r = ((size_t)pp.a_begin + a) * raw.t_stride + i, ip = i > 0 ? r - 1 : r;
      double sx, sy, rho;
      if (!corr_terms(raw.var_x[ip], raw.var_y[ip], cov_xy[ip], &sx, &sy, &rho)) rho = CUDART_NAN;
      o = make_float4((float)(1.0 / sx), (float)(1.0 / sy), (float)rho, 0.0f);
    }
    const_cast<float4*>(agent_corr_view(table, A, Tp))[(size_t)slot[a] * Tp + i] = o;
  }
}
static void launch_corr(const FoAgentsRaw& raw, const float* cov_xy, const PackProblem& one, const PackProblem* many,
                        int P, int max_cells, unsigned char* arena, cudaStream_t st) {
  const dim3 grid((max_cells + 255) / 256, P < 65535 ? P : 65535);
  fo_agents_corr_kernel<<<grid, 256, 0, st>>>(raw, cov_xy, one, many, P, arena);
}

// ---------------------------------------------------------------------------------------------
// fo_metric_batch_host's ego ingest: float64 rows in the caller's world frame -> the float32 bundle of the metric kernels.
// x and y lose their problem's origin in float64 and are rounded once; theta, v and a are rounded.  The operations are
// explicit round-to-nearest intrinsics, so no contraction can change a bit: every value equals numpy's float64 difference
// cast to float32, which is what MetricEngine.assess_batch stages on the host.  A CTA takes a tile of whole rows, finds
// each row's problem once (find_problem, as the batch kernels do), then streams the tile: coalesced 8-byte loads and
// 4-byte stores.
constexpr int kIngestThreads = 256, kIngestTileRows = 256;

__global__ void __launch_bounds__(kIngestThreads)
fo_ego_ingest_kernel(const double* __restrict__ src, float* __restrict__ dst, int row0, int n_rows, int row_elems,
                     int tile_rows, const int* __restrict__ first, const double2* __restrict__ origin, int n_first) {
  __shared__ double2 org[kIngestTileRows];
  const int n_tiles = (n_rows + tile_rows - 1) / tile_rows;
  for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
    const int r_lo = t * tile_rows, rows = min(tile_rows, n_rows - r_lo);
    if ((int)threadIdx.x < rows) org[threadIdx.x] = origin[find_problem(first, n_first, row0 + r_lo + threadIdx.x)];
    __syncthreads();
    const double* s = src + (size_t)r_lo * row_elems;
    float* d = dst + (size_t)r_lo * row_elems;
    const int m = rows * row_elems;
    for (int j = threadIdx.x; j < m; j += kIngestThreads) {
      const double v = s[j];
      const int col = j % 5;                     // row_elems = 5 T: every row starts at a multiple of 5
      float o;
      if (col < 2) {
        const double2 g = org[j / row_elems];
        o = __double2float_rn(__dsub_rn(v, col == 0 ? g.x : g.y));
      } else {
        o = __double2float_rn(v);
      }
      d[j] = o;
    }
    __syncthreads();
  }
}

int launch_ego_ingest(const double* src, float* dst, int row0, int n_rows, int T, const int* first_dev,
                      const double2* origin_dev, int n_first, cudaStream_t st) {
  if (n_rows <= 0) return FO_OK;
  const int row_elems = 5 * T;
  // about 2048 elements per tile, so short horizons still give every thread several
  const int tile_rows = max(1, min(kIngestTileRows, 2048 / row_elems));
  const int n_tiles = (n_rows + tile_rows - 1) / tile_rows;
  fo_ego_ingest_kernel<<<min(n_tiles, 4096), kIngestThreads, 0, st>>>(src, dst, row0, n_rows, row_elems, tile_rows,
                                                                     first_dev, origin_dev, n_first);
  count_launch();
  FO_CUDA_TRY(cudaGetLastError());
  return FO_OK;
}

// The ego vehicle in kernel units; the single-problem path and every batch descriptor take it from here, so a problem
// of a batch sees the same float values as alone.
static void fill_ego_const(const FoVehicle& v, EgoConst& e) {
  e.hEx = 0.5f * v.length; e.hEy = 0.5f * v.width;
  e.wb = v.wb_rear_axle; e.a_max = v.a_max;
  e.L3 = v.length / 3.0f; e.L6 = v.length / 6.0f; e.W2 = v.width / 2.0f;
}

// Staging of the per-problem descriptors of the batch entry points, per calling thread and device: a ring of slots, each
// a page-locked host buffer and a device buffer.  A slot is refilled only after the event recorded behind its last use
// (the upload from the host buffer and the launches that read the device copy) has completed.
constexpr int kStageRing = 4, kStageMaxDev = 64;
struct StageSlot {
  unsigned char* host = nullptr;
  unsigned char* dev = nullptr;
  size_t bytes = 0;
  cudaEvent_t done = nullptr;
};
struct StageRing {
  StageSlot slot[kStageRing];
  int next = 0;
};
static thread_local StageRing g_stage[kStageMaxDev];

static int stage_acquire(size_t bytes, StageSlot** out) {
  int dev = 0;
  FO_CUDA_TRY(cudaGetDevice(&dev));
  if (dev < 0 || dev >= kStageMaxDev) { set_error("batch staging: device ordinal %d out of range", dev); return FO_ERR_UNSUPPORTED; }
  StageRing& ring = g_stage[dev];
  StageSlot& s = ring.slot[ring.next];
  ring.next = (ring.next + 1) % kStageRing;
  if (!s.done) FO_CUDA_TRY(cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming));
  FO_CUDA_TRY(cudaEventSynchronize(s.done));
  if (bytes > s.bytes) {
    if (s.host) FO_CUDA_TRY(cudaFreeHost(s.host));
    if (s.dev) FO_CUDA_TRY(cudaFree(s.dev));
    s.host = s.dev = nullptr;
    s.bytes = 0;
    const size_t want = bytes + bytes / 4 > 4096 ? bytes + bytes / 4 : 4096;
    FO_CUDA_TRY(cudaMallocHost(&s.host, want));
    FO_CUDA_TRY(cudaMalloc(&s.dev, want));
    s.bytes = want;
  }
  *out = &s;
  return FO_OK;
}

static int stage_upload(StageSlot* s, size_t bytes, cudaStream_t st) {
  FO_CUDA_TRY(cudaMemcpyAsync(s->dev, s->host, bytes, cudaMemcpyHostToDevice, st));
  return FO_OK;
}

// Checks the table of one problem against the arena (A > 0): stride range, 16-byte alignment, bounds (of a correlated
// table when corr).
static int check_table(const char* fn, int p, int A, int Tp, int64_t off, size_t arena_bytes, bool corr) {
  if (Tp < 1) { set_error("%s: problem %d has agents but t_stride %d", fn, p, Tp); return FO_ERR_INVALID_ARG; }
  if (Tp > FO_MAX_STATES) { set_error("%s: problem %d t_stride %d > FO_MAX_STATES", fn, p, Tp); return FO_ERR_UNSUPPORTED; }
  const size_t need = corr ? agent_table_bytes_corr(A, Tp) : agent_table_bytes(A, Tp);
  if (off < 0 || (off & 15) || (size_t)off > arena_bytes || arena_bytes - (size_t)off < need) {
    set_error("%s: %stable of problem %d (offset %lld, %zu bytes) misaligned or outside the arena (%zu bytes)", fn,
              corr ? "correlated " : "", p, (long long)off, need, arena_bytes);
    return FO_ERR_INVALID_ARG;
  }
  return FO_OK;
}

}  // namespace fo

// =============================================================================================
extern "C" size_t fo_agent_table_bytes(int32_t n_agents, int32_t t_stride) {
  if (n_agents < 0 || t_stride < 0) return 0;
  return fo::agent_table_bytes(n_agents, t_stride);
}

extern "C" int fo_agents_pack(const FoAgentsRaw* raw, const FoVehicle* vehicle, void* table_dev, size_t table_bytes,
                              void* stream) {
  if (!raw || !vehicle) { fo::set_error("fo_agents_pack: NULL argument"); return FO_ERR_INVALID_ARG; }
  const int A = raw->n_agents, Tp = raw->t_stride;
  if (A < 0 || Tp < 0) { fo::set_error("fo_agents_pack: negative size"); return FO_ERR_INVALID_ARG; }
  if (A == 0 || Tp == 0) return FO_OK;
  if (Tp > FO_MAX_STATES) { fo::set_error("fo_agents_pack: t_stride %d > FO_MAX_STATES", Tp); return FO_ERR_UNSUPPORTED; }
  if (!table_dev || table_bytes < fo::agent_table_bytes(A, Tp)) {
    fo::set_error("fo_agents_pack: table buffer too small (%zu < %zu)", table_bytes, fo::agent_table_bytes(A, Tp));
    return FO_ERR_INVALID_ARG;
  }
  if (!raw->x || !raw->y || !raw->yaw || !raw->v || !raw->var_x || !raw->var_y || !raw->n_states || !raw->kind ||
      !raw->length || !raw->width || !raw->buf_length || !raw->buf_width) {
    fo::set_error("fo_agents_pack: NULL array in FoAgentsRaw");
    return FO_ERR_INVALID_ARG;
  }
  const fo::PackProblem one{0, A, Tp, vehicle->mass, 0};
  fo::launch_pack(*raw, one, nullptr, 1, fo::agent_pad(A) * Tp, (unsigned char*)table_dev, (cudaStream_t)stream);
  fo::count_launch(2);
  FO_CUDA_TRY(cudaGetLastError());
  return FO_OK;
}

extern "C" size_t fo_agent_table_bytes_corr(int32_t n_agents, int32_t t_stride) {
  if (n_agents < 0 || t_stride < 0) return 0;
  return fo::agent_table_bytes_corr(n_agents, t_stride);
}

extern "C" int fo_agents_pack_corr(const FoAgentsRaw* raw, const float* cov_xy, const FoVehicle* vehicle, void* table_dev,
                                   size_t table_bytes, void* stream) {
  const char* fn = "fo_agents_pack_corr";
  if (!raw || !vehicle || !cov_xy) { fo::set_error("%s: NULL argument", fn); return FO_ERR_INVALID_ARG; }
  const int A = raw->n_agents, Tp = raw->t_stride;
  if (A < 0 || Tp < 0) { fo::set_error("%s: negative size", fn); return FO_ERR_INVALID_ARG; }
  if (A == 0 || Tp == 0) return FO_OK;
  if (Tp > FO_MAX_STATES) { fo::set_error("%s: t_stride %d > FO_MAX_STATES", fn, Tp); return FO_ERR_UNSUPPORTED; }
  if (!table_dev || table_bytes < fo::agent_table_bytes_corr(A, Tp)) {
    fo::set_error("%s: table buffer too small (%zu < %zu)", fn, table_bytes, fo::agent_table_bytes_corr(A, Tp));
    return FO_ERR_INVALID_ARG;
  }
  const int rc = fo_agents_pack(raw, vehicle, table_dev, table_bytes, stream);   // the diagonal table, byte for byte
  if (rc != FO_OK) return rc;
  fo::launch_corr(*raw, cov_xy, fo::PackProblem{0, A, Tp, vehicle->mass, 0}, nullptr, 1, A * Tp, (unsigned char*)table_dev,
                  (cudaStream_t)stream);
  fo::count_launch();
  FO_CUDA_TRY(cudaGetLastError());
  return FO_OK;
}

// corr: NULL = every table diagonal (fo_agent_batch_layout)
static size_t batch_layout(const char* fn, int32_t n_problems, const int32_t* n_agents, const int32_t* t_stride,
                           const uint8_t* corr, int64_t* table_offset) {
  if (n_problems < 0 || (n_problems > 0 && (!n_agents || !t_stride || !table_offset))) {
    fo::set_error("%s: bad argument", fn);
    return 0;
  }
  size_t off = 0;
  for (int p = 0; p < n_problems; ++p) {
    const int A = n_agents[p], Tp = t_stride[p];
    if (A < 0 || Tp < 0 || Tp > FO_MAX_STATES) {
      fo::set_error("%s: problem %d: n_agents %d / t_stride %d out of range", fn, p, A, Tp);
      return 0;
    }
    table_offset[p] = (int64_t)off;
    if (A > 0 && Tp > 0)
      off += ((corr && corr[p] ? fo::agent_table_bytes_corr(A, Tp) : fo::agent_table_bytes(A, Tp)) + 15) & ~(size_t)15;
  }
  return off;
}

extern "C" size_t fo_agent_batch_layout(int32_t n_problems, const int32_t* n_agents, const int32_t* t_stride,
                                        int64_t* table_offset) {
  return batch_layout("fo_agent_batch_layout", n_problems, n_agents, t_stride, nullptr, table_offset);
}

extern "C" size_t fo_agent_batch_layout_corr(int32_t n_problems, const int32_t* n_agents, const int32_t* t_stride,
                                             const uint8_t* corr_host, int64_t* table_offset) {
  const char* fn = "fo_agent_batch_layout_corr";
  if (n_problems > 0 && !corr_host) { fo::set_error("%s: corr_host must not be NULL", fn); return 0; }
  return batch_layout(fn, n_problems, n_agents, t_stride, corr_host, table_offset);
}

int fo::check_pack_batch(const char* fn, const FoAgentsRaw* raw, int32_t n_problems, const FoBatchProblem* problems,
                         const uint8_t* corr, const void* arena_dev, size_t arena_bytes, int* n_packed_out,
                         int* max_cells_out) {
  if (!raw || n_problems < 0 || (n_problems > 0 && !problems)) { fo::set_error("%s: bad argument", fn); return FO_ERR_INVALID_ARG; }
  if (raw->n_agents < 0 || raw->t_stride < 0) { fo::set_error("%s: negative size", fn); return FO_ERR_INVALID_ARG; }
  if (reinterpret_cast<uintptr_t>(arena_dev) & 15) { fo::set_error("%s: arena must be 16-byte aligned", fn); return FO_ERR_INVALID_ARG; }
  long long total = 0;
  int n_packed = 0, max_cells = 0;
  *n_packed_out = 0;
  for (int p = 0; p < n_problems; ++p) {
    const FoBatchProblem& q = problems[p];
    if (q.n_agents < 0) { fo::set_error("%s: problem %d has %d agents", fn, p, q.n_agents); return FO_ERR_INVALID_ARG; }
    total += q.n_agents;
    if (q.n_agents == 0) continue;
    const int rc = fo::check_table(fn, p, q.n_agents, q.t_stride, q.table_offset, arena_dev ? arena_bytes : 0,
                                   corr && corr[p]);
    if (rc != FO_OK) return rc;
    if (q.t_stride > raw->t_stride) { fo::set_error("%s: problem %d t_stride %d > raw row stride %d", fn, p, q.t_stride, raw->t_stride); return FO_ERR_INVALID_ARG; }
    ++n_packed;
    const int cells = fo::agent_pad(q.n_agents) * q.t_stride;
    if (cells > max_cells) max_cells = cells;
  }
  if (total != raw->n_agents) {
    fo::set_error("%s: the problems hold %lld agents, raw->n_agents is %d", fn, total, raw->n_agents);
    return FO_ERR_INVALID_ARG;
  }
  if (n_packed == 0) return FO_OK;
  if (!raw->x || !raw->y || !raw->yaw || !raw->v || !raw->var_x || !raw->var_y || !raw->n_states || !raw->kind ||
      !raw->length || !raw->width || !raw->buf_length || !raw->buf_width) {
    fo::set_error("%s: NULL array in FoAgentsRaw", fn);
    return FO_ERR_INVALID_ARG;
  }
  *n_packed_out = n_packed;
  *max_cells_out = max_cells;
  return FO_OK;
}

// Problem p is packed with the mass of vehicles[per_problem ? p : 0]; corr / cov_xy: the correlated problems
// (fo_agents_pack_batch_corr), NULL for none.
static int pack_batch_impl(const char* fn, const FoAgentsRaw* raw, int32_t n_problems, const FoBatchProblem* problems,
                           const FoVehicle* vehicles, bool per_problem, const uint8_t* corr, const float* cov_xy,
                           void* arena_dev, size_t arena_bytes, void* stream) {
  if (!vehicles) { fo::set_error("%s: bad argument", fn); return FO_ERR_INVALID_ARG; }
  int n_packed = 0, max_cells = 0;
  {
    const int rc = fo::check_pack_batch(fn, raw, n_problems, problems, corr, arena_dev, arena_bytes, &n_packed, &max_cells);
    if (rc != FO_OK || n_packed == 0) return rc;
  }
  int n_corr = 0, corr_cells = 0;               // the correlated problems with agents, the most (agent, state) cells of one
  for (int p = 0; corr && p < n_problems; ++p) {
    const FoBatchProblem& q = problems[p];
    if (!corr[p] || q.n_agents == 0) continue;
    ++n_corr;
    if (q.n_agents * q.t_stride > corr_cells) corr_cells = q.n_agents * q.t_stride;
  }
  if (n_corr > 0 && !cov_xy) { fo::set_error("%s: cov_xy must not be NULL with correlated problems", fn); return FO_ERR_INVALID_ARG; }
  cudaStream_t st = (cudaStream_t)stream;
  // staged: the descriptors of all packed problems, then those of the correlated ones again (the s3 launch)
  const size_t bytes = (size_t)(n_packed + n_corr) * sizeof(fo::PackProblem);
  fo::StageSlot* slot = nullptr;
  int rc = fo::stage_acquire(bytes, &slot);
  if (rc != FO_OK) return rc;
  fo::PackProblem* pp = reinterpret_cast<fo::PackProblem*>(slot->host);
  int a_begin = 0, j = 0, jc = n_packed;
  for (int p = 0; p < n_problems; ++p) {
    const FoBatchProblem& q = problems[p];
    if (q.n_agents > 0) {
      pp[j++] = fo::PackProblem{a_begin, q.n_agents, q.t_stride, vehicles[per_problem ? p : 0].mass, (long long)q.table_offset};
      if (corr && corr[p]) pp[jc++] = pp[j - 1];
    }
    a_begin += q.n_agents;
  }
  rc = fo::stage_upload(slot, bytes, st);
  if (rc != FO_OK) return rc;
  const fo::PackProblem* pp_dev = reinterpret_cast<const fo::PackProblem*>(slot->dev);
  fo::launch_pack(*raw, fo::PackProblem{}, pp_dev, n_packed, max_cells, (unsigned char*)arena_dev, st);
  fo::count_launch(2);
  if (n_corr > 0) {
    fo::launch_corr(*raw, cov_xy, fo::PackProblem{}, pp_dev + n_packed, n_corr, corr_cells, (unsigned char*)arena_dev, st);
    fo::count_launch();
  }
  FO_CUDA_TRY(cudaGetLastError());
  FO_CUDA_TRY(cudaEventRecord(slot->done, st));
  return FO_OK;
}

extern "C" int fo_agents_pack_batch(const FoAgentsRaw* raw, int32_t n_problems, const FoBatchProblem* problems,
                                    const FoVehicle* vehicle, void* arena_dev, size_t arena_bytes, void* stream) {
  return pack_batch_impl("fo_agents_pack_batch", raw, n_problems, problems, vehicle, false, nullptr, nullptr, arena_dev,
                         arena_bytes, stream);
}

extern "C" int fo_agents_pack_batch_vehicles(const FoAgentsRaw* raw, int32_t n_problems, const FoBatchProblem* problems,
                                             const FoVehicle* vehicles_host, void* arena_dev, size_t arena_bytes,
                                             void* stream) {
  const char* fn = "fo_agents_pack_batch_vehicles";
  if (n_problems > 0 && !vehicles_host) { fo::set_error("%s: vehicles_host must not be NULL", fn); return FO_ERR_INVALID_ARG; }
  static const FoVehicle none{};                 // no problems: nothing is read
  return pack_batch_impl(fn, raw, n_problems, problems, vehicles_host ? vehicles_host : &none, true, nullptr, nullptr,
                         arena_dev, arena_bytes, stream);
}

extern "C" int fo_agents_pack_batch_corr(const FoAgentsRaw* raw, const float* cov_xy, int32_t n_problems,
                                         const FoBatchProblem* problems, const uint8_t* corr_host,
                                         const FoVehicle* vehicles_host, void* arena_dev, size_t arena_bytes,
                                         void* stream) {
  const char* fn = "fo_agents_pack_batch_corr";
  if (n_problems > 0 && (!corr_host || !vehicles_host)) {
    fo::set_error("%s: corr_host and vehicles_host must not be NULL", fn);
    return FO_ERR_INVALID_ARG;
  }
  static const FoVehicle none{};                 // no problems: nothing is read
  return pack_batch_impl(fn, raw, n_problems, problems, vehicles_host ? vehicles_host : &none, true, corr_host, cov_xy,
                         arena_dev, arena_bytes, stream);
}

// SM count per device (a process may drive several GPUs, one per planner thread): cached per ordinal, racing
// first calls store the same value
static int num_sms_of_current_device(int* out) {
  constexpr int kMaxDev = 64;
  static std::atomic<int> cache[kMaxDev];
  int dev = 0;
  FO_CUDA_TRY(cudaGetDevice(&dev));
  int n = (dev >= 0 && dev < kMaxDev) ? cache[dev].load(std::memory_order_relaxed) : 0;
  if (n == 0) {
    FO_CUDA_TRY(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev));
    if (dev >= 0 && dev < kMaxDev) cache[dev].store(n, std::memory_order_relaxed);
  }
  *out = n;
  return FO_OK;
}
// Kernel arguments of a validated FoMetricArgs: inputs, vehicle / harm constants and the threshold clauses in kernel units.
static void fill_kargs(const FoMetricArgs* a, fo::MetricKArgs& k) {
  k.ego = a->ego; k.N = a->n_traj; k.T = a->n_states; k.A = a->n_agents; k.Tp = a->t_stride;
  k.tab = fo::agent_table_view(a->agent_table, a->n_agents, a->t_stride);
  fo::fill_ego_const(a->vehicle, k.veh);
  k.hc = a->harm; k.dt = (float)a->dt; k.dtd = a->dt;
  k.mmask = a->metric_mask; k.tmask = a->threshold_mask;
  k.thr_harm = a->thr_harm; k.thr_risk = a->thr_risk; k.thr_be = a->thr_be; k.thr_cp = a->thr_cp;
  k.thr_ttc = a->thr_ttc; k.thr_dce = a->thr_dce;
  {
    // smallest r with r / 1000.0 >= thr_dce (the reference compares np.round(d, 3) = r / 1000.0 in float64)
    long long c = (long long)ceil(a->thr_dce * 1000.0);
    if (!(a->thr_dce > 0.0)) c = 0;
    if (c > 0xffffff) c = 0xffffff;
    while (c > 0 && (double)(c - 1) / 1000.0 >= a->thr_dce) --c;
    while (c < 0xffffff && (double)c / 1000.0 < a->thr_dce) ++c;
    k.thr_dce_mm = (uint32_t)c;
    // smallest step with np.round(step * dt, 3) >= thr_ttc
    uint32_t q = 0;
    while (q < (uint32_t)FO_MAX_STATES + 1u && rint((double)q * a->dt * 1000.0) / 1000.0 < a->thr_ttc) ++q;
    k.thr_ttc_col = q;
  }
  k.valid = a->valid; k.summary = a->summary; k.flags = a->flags; k.pair = a->pair; k.step = a->step;
  k.stats = nullptr;
  { const char* e = getenv("FO_EXACT_DCE"); k.exact_dce = e && e[0] == '1'; }
  k.claim = nullptr;
  k.n_peers = 0;
  for (int p = 0; p < FO_MAX_PEERS; ++p) k.peer_delta[p] = 0;
  k.corr = false;
}

static int metric_bundle_impl(const FoMetricArgs* a, unsigned long long* stats, void* stream, bool corr = false);

// Peer stores: n_peers in [0, FO_MAX_PEERS], and only on the summary path (no pair / step, no work counters).
static int check_peers(const char* fn, const FoMetricArgs* a, bool stats) {
  if (a->n_peers < 0 || a->n_peers > FO_MAX_PEERS) { fo::set_error("%s: n_peers %d outside [0, %d]", fn, a->n_peers, FO_MAX_PEERS); return FO_ERR_INVALID_ARG; }
  if (a->n_peers > 0 && (a->pair || a->step || stats)) { fo::set_error("%s: peer stores exist on the summary path only", fn); return FO_ERR_UNSUPPORTED; }
  return FO_OK;
}

extern "C" int fo_metric_bundle(const FoMetricArgs* a, void* stream) { return metric_bundle_impl(a, nullptr, stream); }

extern "C" int fo_metric_bundle_corr(const FoMetricArgs* a, void* stream) {
  if (a && a->n_peers != 0) { fo::set_error("fo_metric_bundle_corr: no peer stores on correlated tables"); return FO_ERR_UNSUPPORTED; }
  return metric_bundle_impl(a, nullptr, stream, true);
}

// The peer checks run here before any device query, so a bad n_peers is reported without a device.
extern "C" int fo_metric_bundle_corr_peers(const FoMetricArgs* a, void* stream) {
  const int rc = a ? check_peers("fo_metric_bundle_corr_peers", a, false) : FO_OK;
  return rc != FO_OK ? rc : metric_bundle_impl(a, nullptr, stream, true);
}

static int metric_stats_impl(const char* fn, const FoMetricArgs* a, uint64_t* counters_dev, void* stream, bool corr) {
  if (!counters_dev) { fo::set_error("%s: counters_dev must not be NULL", fn); return FO_ERR_INVALID_ARG; }
  if (a && (a->pair || a->step)) { fo::set_error("%s: summary outputs only", fn); return FO_ERR_INVALID_ARG; }
  FO_CUDA_TRY(cudaMemsetAsync(counters_dev, 0, FO_STATS_K * sizeof(uint64_t), (cudaStream_t)stream));
  return metric_bundle_impl(a, reinterpret_cast<unsigned long long*>(counters_dev), stream, corr);
}

extern "C" int fo_metric_stats(const FoMetricArgs* a, uint64_t* counters_dev, void* stream) {
  return metric_stats_impl("fo_metric_stats", a, counters_dev, stream, false);
}

extern "C" int fo_metric_stats_corr(const FoMetricArgs* a, uint64_t* counters_dev, void* stream) {
  return metric_stats_impl("fo_metric_stats_corr", a, counters_dev, stream, true);
}

static int metric_bundle_impl(const FoMetricArgs* a, unsigned long long* stats, void* stream, bool corr) {
  if (!a) { fo::set_error("fo_metric_bundle: NULL args"); return FO_ERR_INVALID_ARG; }
  if (a->n_traj < 0 || a->n_states < 0 || a->n_agents < 0) { fo::set_error("fo_metric_bundle: negative size"); return FO_ERR_INVALID_ARG; }
  if (a->n_traj == 0) return FO_OK;
  if (!a->ego || !a->valid) { fo::set_error("fo_metric_bundle: ego/valid must not be NULL"); return FO_ERR_INVALID_ARG; }
  if (a->n_states < 1 || a->n_states > FO_MAX_STATES) {
    fo::set_error("fo_metric_bundle: n_states %d outside [1, %d]", a->n_states, FO_MAX_STATES);
    return FO_ERR_UNSUPPORTED;
  }
  if (a->n_agents > 0 && (!a->agent_table || a->t_stride < 1 || a->t_stride > FO_MAX_STATES)) {
    fo::set_error("fo_metric_bundle: agent table missing or t_stride out of range");
    return FO_ERR_INVALID_ARG;
  }
  if ((a->metric_mask & FO_M_BE) && !(a->metric_mask & FO_M_TTC)) {
    fo::set_error("fo_metric_bundle: 'be' needs 'ttc' (reference raises KeyError, be.py:39)");
    return FO_ERR_INVALID_ARG;
  }
  int g_num_sms = 0;
  { const int rc = num_sms_of_current_device(&g_num_sms); if (rc != FO_OK) return rc; }
  fo::MetricKArgs k;
  fill_kargs(a, k);
  k.stats = stats;
  if (a->summary && (reinterpret_cast<uintptr_t>(a->summary) & 7u)) { fo::set_error("fo_metric_bundle: summary must be 8-byte aligned"); return FO_ERR_INVALID_ARG; }
  { const int rc = check_peers("fo_metric_bundle", a, stats != nullptr); if (rc != FO_OK) return rc; }
  k.n_peers = a->n_peers;
  for (int p = 0; p < FO_MAX_PEERS; ++p) k.peer_delta[p] = p < a->n_peers ? (long long)a->peer_delta[p] : 0;
  k.corr = corr;

  cudaStream_t st = (cudaStream_t)stream;
  if (k.pair || k.step) return fo::launch_metric_detail(k, g_num_sms, st);
  return fo::launch_metric_sweep(k, g_num_sms, st);
}

// Host-side checks of the batch entry points, before any device work: the outputs each one accepts, row order and
// contiguity, rows inside n_traj, tables inside the arena, alignment, stride and T limits, 'be' needs 'ttc'.  On success
// *n_run = the problems with trajectories and *a_min = the fewest agents among them.
int fo::check_batch(const char* fn, const FoMetricBatchArgs* b, const uint8_t* corr, bool detail, int* n_run, int* a_min) {
  if (!b) { fo::set_error("%s: NULL args", fn); return FO_ERR_INVALID_ARG; }
  const FoMetricArgs& c = b->common;
  const int P = b->n_problems;
  if (P < 0 || c.n_traj < 0 || (P > 0 && !b->problems)) { fo::set_error("%s: bad problem list", fn); return FO_ERR_INVALID_ARG; }
  if (detail) {
    if (!c.pair && !c.step) { fo::set_error("%s: pair or step is required (summary outputs only: fo_metric_batch)", fn); return FO_ERR_INVALID_ARG; }
    if (c.n_peers != 0) { fo::set_error("%s: peer stores exist on the summary path only", fn); return FO_ERR_UNSUPPORTED; }
    if (reinterpret_cast<uintptr_t>(c.pair) & 15u) { fo::set_error("%s: pair must be 16-byte aligned", fn); return FO_ERR_INVALID_ARG; }
    if (reinterpret_cast<uintptr_t>(c.step) & 3u) { fo::set_error("%s: step must be 4-byte aligned", fn); return FO_ERR_INVALID_ARG; }
  } else if (c.pair || c.step || c.n_peers != 0) {
    fo::set_error("%s: batches have summary outputs only (no pair / step, no peer stores)", fn);
    return FO_ERR_UNSUPPORTED;
  }
  if (c.n_states < 1 || c.n_states > FO_MAX_STATES) {
    fo::set_error("%s: n_states %d outside [1, %d]", fn, c.n_states, FO_MAX_STATES);
    return FO_ERR_UNSUPPORTED;
  }
  if ((c.metric_mask & FO_M_BE) && !(c.metric_mask & FO_M_TTC)) {
    fo::set_error("%s: 'be' needs 'ttc' (reference raises KeyError, be.py:39)", fn);
    return FO_ERR_INVALID_ARG;
  }
  if (reinterpret_cast<uintptr_t>(c.agent_table) & 15) { fo::set_error("%s: arena must be 16-byte aligned", fn); return FO_ERR_INVALID_ARG; }
  // problems in order, their rows contiguous and together exactly [0, n_traj); tables inside the arena
  long long next_row = 0;
  *n_run = 0;
  *a_min = 1 << 30;
  for (int p = 0; p < P; ++p) {
    const FoBatchProblem& q = b->problems[p];
    if (q.n_traj < 0 || q.n_agents < 0) { fo::set_error("%s: problem %d: negative size", fn, p); return FO_ERR_INVALID_ARG; }
    if (q.traj_begin != next_row) {
      fo::set_error("%s: problem %d starts at row %lld, expected %lld (rows are contiguous, in problem order)", fn, p,
                    (long long)q.traj_begin, next_row);
      return FO_ERR_INVALID_ARG;
    }
    next_row += q.n_traj;
    if (next_row > c.n_traj) { fo::set_error("%s: problem %d ends at row %lld > n_traj %d", fn, p, next_row, c.n_traj); return FO_ERR_INVALID_ARG; }
    if (q.n_agents > 0) {
      const bool qc = corr && corr[p];
      const int rc = fo::check_table(fn, p, q.n_agents, q.t_stride, q.table_offset, c.agent_table ? b->arena_bytes : 0, qc);
      if (rc != FO_OK) return rc;
      // the detail descriptor holds the s3 section's place as a 32-bit offset from s0 in 16-byte units
      if (qc && detail && (fo::agent_corr_offset(q.n_agents, q.t_stride) >> 4) > 0xffffffffull) {
        fo::set_error("%s: correlated table of problem %d too large for a batch", fn, p);
        return FO_ERR_UNSUPPORTED;
      }
    }
    if (q.n_traj > 0) {
      ++*n_run;
      if (q.n_agents < *a_min) *a_min = q.n_agents;
    }
  }
  if (next_row != c.n_traj) { fo::set_error("%s: the problems cover %lld of %d rows", fn, next_row, c.n_traj); return FO_ERR_INVALID_ARG; }
  if (c.n_traj == 0) return FO_OK;
  if (!c.ego || !c.valid) { fo::set_error("%s: ego/valid must not be NULL", fn); return FO_ERR_INVALID_ARG; }
  if (c.summary && (reinterpret_cast<uintptr_t>(c.summary) & 7u)) { fo::set_error("%s: summary must be 8-byte aligned", fn); return FO_ERR_INVALID_ARG; }
  return FO_OK;
}

// The staged descriptors of a summary batch call (metric_batch_impl): one team size for the whole batch, as
// fo_metric_bundle picks it; with W = 1 problems with >= 17 agents run the window-filter shape, the others the team
// shape with their own lane grouping.  Classes: 0 / 1 diagonal window-filter / team shape, 2 / 3 the same for
// correlated tables; one launch per non-empty class, each numbering its trajectories.
struct BatchStage {
  int W = 1;
  int cnt[4] = {0, 0, 0, 0}, start[4] = {0, 0, 0, 0}, n_cls[4] = {0, 0, 0, 0};
  fo::StageSlot* slot = nullptr;
  size_t prob_off = 0;              // offset of the descriptors behind first[]
  size_t bytes = 0;                 // first[] and the descriptors; a caller's own data follows at this offset
  std::vector<int> problem;         // problem of each descriptor
};

// vehicles: problem p's ego vehicle is vehicles[p]; NULL = common.vehicle for every problem.  corr: problem p's table is a
// correlated one when corr[p] != 0; NULL = none is.  by_size: within a class the descriptors are sorted by N_p in
// descending order (stable), else they are in problem order.  Stages first[] of all classes, then their descriptors
// (16-byte aligned), class by class, and reserves extra_bytes behind them; the caller uploads.
static int stage_batch(const FoMetricBatchArgs* b, const uint8_t* corr, const FoVehicle* vehicles, int n_run, int a_min,
                       int num_sms, bool by_size, size_t extra_bytes, BatchStage& s) {
  const FoMetricArgs& c = b->common;
  const int P = b->n_problems;
  s.W = fo::pick_team_warps(c.n_traj, c.n_states, a_min, num_sms);
  const auto class_of = [&](int p) {
    return (corr && corr[p] ? 2 : 0) + (s.W == 1 && fo::lane_group_log2(b->problems[p].n_agents) == 5 ? 0 : 1);
  };
  s.problem.clear();
  for (int p = 0; p < P; ++p)
    if (b->problems[p].n_traj > 0) {
      ++s.cnt[class_of(p)];
      s.problem.push_back(p);
    }
  std::stable_sort(s.problem.begin(), s.problem.end(), [&](int p, int q) {
    const int cp = class_of(p), cq = class_of(q);
    if (cp != cq) return cp < cq;
    return by_size && b->problems[p].n_traj > b->problems[q].n_traj;
  });
  s.start[1] = s.cnt[0]; s.start[2] = s.start[1] + s.cnt[1]; s.start[3] = s.start[2] + s.cnt[2];
  s.prob_off = ((size_t)n_run * sizeof(int) + 15) & ~(size_t)15;
  s.bytes = s.prob_off + (size_t)n_run * sizeof(fo::BatchProb);
  int rc = fo::stage_acquire(s.bytes + extra_bytes, &s.slot);
  if (rc != FO_OK) return rc;
  int* first = reinterpret_cast<int*>(s.slot->host);
  fo::BatchProb* prob = reinterpret_cast<fo::BatchProb*>(s.slot->host + s.prob_off);
  const unsigned char* arena = reinterpret_cast<const unsigned char*>(c.agent_table);
  for (int i = 0; i < n_run; ++i) {
    const int p = s.problem[i];
    const FoBatchProblem& q = b->problems[p];
    const int cl = class_of(p);
    int& n = s.n_cls[cl];
    fo::BatchProb& d = prob[i];
    const int Tp = q.n_agents > 0 ? q.t_stride : 1;
    const unsigned char* tab = arena + (q.n_agents > 0 ? q.table_offset : 0);
    const fo::AgentTableView v = fo::agent_table_view(tab, q.n_agents, Tp);
    d.t0 = v.t0; d.tv = v.tv; d.aw = v.aw; d.avw = v.avw; d.s0 = v.s0; d.s1 = v.s1; d.s2 = v.s2; d.prm = v.prm;
    d.first = n; d.row0 = (int)q.traj_begin; d.A = q.n_agents; d.Tp = Tp; d.Ap = v.Ap; d.lg = fo::lane_group_log2(q.n_agents);
    fo::fill_ego_const(vehicles ? vehicles[p] : c.vehicle, d.veh);
    d.s3 = cl >= 2 && q.n_agents > 0 ? fo::agent_corr_view(tab, q.n_agents, Tp) : nullptr;
    first[i] = n;
    n += q.n_traj;
  }
  return FO_OK;
}

// Kernel arguments shared by the classes of a summary batch call: the tables are per problem.
static void batch_kargs(const FoMetricArgs& c, fo::MetricKArgs& k) {
  FoMetricArgs ca = c;
  ca.n_agents = 0;
  ca.agent_table = nullptr;
  fill_kargs(&ca, k);
}

// select (fo_metric_batch_select): the descriptors are sorted by N_p within each class, and staged behind them are the
// rank segments of every class (at most one per descriptor), the problem index of each descriptor and N_p of every
// problem, which is copied into selected_dev before the launches.
static int metric_batch_impl(const char* fn, const FoMetricBatchArgs* b, const uint8_t* corr, const FoVehicle* vehicles,
                             bool select, int32_t* selected_dev, void* stream) {
  int n_run = 0, a_min = 0;
  {
    const int rc = fo::check_batch(fn, b, corr, false, &n_run, &a_min);
    if (rc != FO_OK) return rc;
  }
  const int P = b->n_problems;
  if (select && P > 0 && (!selected_dev || (reinterpret_cast<uintptr_t>(selected_dev) & 3u))) {
    fo::set_error("%s: selected_dev must be a 4-byte aligned device array of n_problems int32", fn);
    return FO_ERR_INVALID_ARG;
  }
  cudaStream_t st = (cudaStream_t)stream;
  if (b->common.n_traj == 0) {                     // every N_p is 0
    if (select && P > 0) FO_CUDA_TRY(cudaMemsetAsync(selected_dev, 0, (size_t)P * sizeof(int32_t), st));
    return FO_OK;
  }
  int num_sms = 0;
  { const int rc = num_sms_of_current_device(&num_sms); if (rc != FO_OK) return rc; }
  const size_t seg_bytes = select ? (size_t)n_run * sizeof(int4) : 0;
  const size_t out_bytes = select ? ((size_t)n_run * sizeof(int) + 15) & ~(size_t)15 : 0;
  const size_t init_bytes = select ? (size_t)P * sizeof(int32_t) : 0;
  BatchStage s;
  int rc = stage_batch(b, corr, vehicles, n_run, a_min, num_sms, select, seg_bytes + out_bytes + init_bytes, s);
  if (rc != FO_OK) return rc;
  // class cl: descriptors start[cl] .. with N descending; the ranks in [N of descriptor m, N of descriptor m - 1) have
  // the first m descriptors active
  int seg_start[4] = {0, 0, 0, 0}, n_seg[4] = {0, 0, 0, 0};
  if (select) {
    int4* seg = reinterpret_cast<int4*>(s.slot->host + s.bytes);
    int* out = reinterpret_cast<int*>(s.slot->host + s.bytes + seg_bytes);
    int32_t* init = reinterpret_cast<int32_t*>(s.slot->host + s.bytes + seg_bytes + out_bytes);
    for (int p = 0; p < P; ++p) init[p] = b->problems[p].n_traj;
    for (int i = 0; i < n_run; ++i) out[i] = s.problem[i];
    int ns = 0;
    for (int cl = 0; cl < 4; ++cl) {
      seg_start[cl] = ns;
      int claims = 0, prev = 0;
      for (int m = s.cnt[cl]; m >= 1; --m) {
        const int hi = b->problems[s.problem[s.start[cl] + m - 1]].n_traj;
        if (hi <= prev) continue;
        seg[ns++] = make_int4(claims, prev, m, 0);
        claims += (hi - prev) * m;
        prev = hi;
      }
      n_seg[cl] = ns - seg_start[cl];
    }
  }
  rc = fo::stage_upload(s.slot, s.bytes + seg_bytes + out_bytes + init_bytes, st);
  if (rc != FO_OK) return rc;
  if (select)
    FO_CUDA_TRY(cudaMemcpyAsync(selected_dev, s.slot->dev + s.bytes + seg_bytes + out_bytes, init_bytes,
                                cudaMemcpyDeviceToDevice, st));
  fo::MetricKArgs k;
  batch_kargs(b->common, k);
  const int* first_dev = reinterpret_cast<const int*>(s.slot->dev);
  const fo::BatchProb* prob_dev = reinterpret_cast<const fo::BatchProb*>(s.slot->dev + s.prob_off);
  const int4* seg_dev = reinterpret_cast<const int4*>(s.slot->dev + s.bytes);
  const int* out_dev = reinterpret_cast<const int*>(s.slot->dev + s.bytes + seg_bytes);
  for (int cl = 0; cl < 4; ++cl) {
    if (s.cnt[cl] == 0) continue;
    k.N = s.n_cls[cl];
    k.corr = cl >= 2;
    const fo::SelectView sv = select ? fo::SelectView{seg_dev + seg_start[cl], out_dev + s.start[cl], selected_dev, n_seg[cl]}
                                     : fo::SelectView{};
    rc = fo::launch_metric_batch(k, num_sms, s.W, (cl & 1) == 0,
                                 fo::BatchView{first_dev + s.start[cl], prob_dev + s.start[cl], s.cnt[cl]}, sv, st);
    if (rc != FO_OK) return rc;
  }
  FO_CUDA_TRY(cudaEventRecord(s.slot->done, st));
  return FO_OK;
}

extern "C" int fo_metric_batch(const FoMetricBatchArgs* b, void* stream) {
  return metric_batch_impl("fo_metric_batch", b, nullptr, nullptr, false, nullptr, stream);
}

extern "C" int fo_metric_batch_vehicles(const FoMetricBatchArgs* b, const FoVehicle* vehicles_host, void* stream) {
  const char* fn = "fo_metric_batch_vehicles";
  if (b && b->n_problems > 0 && !vehicles_host) { fo::set_error("%s: vehicles_host must not be NULL", fn); return FO_ERR_INVALID_ARG; }
  return metric_batch_impl(fn, b, nullptr, vehicles_host, false, nullptr, stream);
}

// corr as in metric_batch_impl.  The diagonal problems run fo_metric_batch_detail_kernel, which takes its launch's rows
// to be [0, k.N) with the problems' first rows in first[]: where correlated problems sit between diagonal ones, their rows
// enter that launch as problems without agents (valid / summary / flags only), and the correlated launch that follows on
// the stream writes them again with their own results.  The correlated launch numbers its trajectories itself
// (fo_metric_batch_detail_corr_kernel), so it touches its own rows only.
static int metric_batch_detail_impl(const char* fn, const FoMetricBatchArgs* b, const uint8_t* corr,
                                    const FoVehicle* vehicles, void* stream) {
  int n_run = 0, a_min = 0;
  {
    const int rc = fo::check_batch(fn, b, corr, true, &n_run, &a_min);
    if (rc != FO_OK || b->common.n_traj == 0) return rc;
  }
  const FoMetricArgs& c = b->common;
  const int P = b->n_problems, Tm1 = c.n_states - 1;
  int num_sms = 0;
  { const int rc = num_sms_of_current_device(&num_sms); if (rc != FO_OK) return rc; }
  // the diagonal launch covers the rows up to the end of its last problem; its descriptors: every problem with
  // trajectories up to there (the correlated ones as stand-ins without agents).  The correlated launch: its problems.
  long long diag_rows = 0;
  int n_diag = 0, n_corr = 0;
  for (int p = 0; p < P; ++p) {
    const FoBatchProblem& q = b->problems[p];
    if (q.n_traj == 0) continue;
    if (corr && corr[p]) { ++n_corr; continue; }
    diag_rows = q.traj_begin + q.n_traj;
  }
  for (int p = 0; p < P; ++p)
    if (b->problems[p].n_traj > 0 && b->problems[p].traj_begin < diag_rows) ++n_diag;
  const int n_desc = n_diag + n_corr;
  // staged: the first[] of both launches, then their descriptors (16-byte aligned)
  const size_t first_bytes = ((size_t)n_desc * sizeof(int) + 15) & ~(size_t)15;
  const size_t bytes = first_bytes + (size_t)n_desc * sizeof(fo::DetailProb);
  fo::StageSlot* slot = nullptr;
  int rc = fo::stage_acquire(bytes, &slot);
  if (rc != FO_OK) return rc;
  int* first = reinterpret_cast<int*>(slot->host);
  fo::DetailProb* prob = reinterpret_cast<fo::DetailProb*>(slot->host + first_bytes);
  const unsigned char* arena = reinterpret_cast<const unsigned char*>(c.agent_table);
  long long pairs = 0;                           // sum of N_q A_q over the problems before p: the offset of p's blocks
  // problem p's descriptor; a stand-in has no agents and no detail blocks
  const auto fill = [&](fo::DetailProb& d, int p, bool stand_in) {
    const FoBatchProblem& q = b->problems[p];
    const int A = stand_in ? 0 : q.n_agents;
    const int Tp = A > 0 ? q.t_stride : 1;
    const fo::AgentTableView v = fo::agent_table_view(arena + (A > 0 ? q.table_offset : 0), A, Tp);
    d.t0 = v.t0; d.tv = v.tv; d.s0 = v.s0; d.s1 = v.s1; d.s2 = v.s2; d.prm = v.prm; d.orig = v.orig; d.tpsi = v.tpsi;
    d.pair = c.pair && !stand_in ? c.pair + (size_t)pairs * FO_PAIR_K : nullptr;
    d.step = c.step && !stand_in ? c.step + (size_t)pairs * Tm1 * FO_STEP_K : nullptr;
    d.row0 = (int)q.traj_begin; d.A = A; d.Tp = Tp; d.Ap = v.Ap;
    fo::fill_ego_const(vehicles ? vehicles[p] : c.vehicle, d.veh);
    d.s3_off = corr && corr[p] && A > 0 ? (uint32_t)(fo::agent_corr_offset(A, Tp) >> 4) : 0u;
  };
  int i = 0, ic = n_diag, nc = 0;                // next diagonal / correlated descriptor; trajectories of the latter
  for (int p = 0; p < P; ++p) {
    const FoBatchProblem& q = b->problems[p];
    if (q.n_traj == 0) continue;
    const bool qc = corr && corr[p];
    if (!qc || q.traj_begin < diag_rows) {
      fill(prob[i], p, qc);
      first[i++] = (int)q.traj_begin;
    }
    if (qc) {
      fill(prob[ic], p, false);
      first[ic++] = nc;
      nc += q.n_traj;
    }
    pairs += (long long)q.n_traj * q.n_agents;
  }
  cudaStream_t st = (cudaStream_t)stream;
  rc = fo::stage_upload(slot, bytes, st);
  if (rc != FO_OK) return rc;
  fo::MetricKArgs k;
  FoMetricArgs ca = c;
  ca.n_agents = 0;                           // per problem
  ca.agent_table = nullptr;
  ca.pair = ca.step = nullptr;
  fill_kargs(&ca, k);
  const int* first_dev = reinterpret_cast<const int*>(slot->dev);
  const fo::DetailProb* prob_dev = reinterpret_cast<const fo::DetailProb*>(slot->dev + first_bytes);
  if (n_diag > 0) {                          // first: the correlated launch overwrites its stand-ins' rows
    k.N = (int)diag_rows;
    rc = fo::launch_metric_batch_detail(k, num_sms, fo::DetailView{first_dev, prob_dev, n_diag}, st);
    if (rc != FO_OK) return rc;
  }
  if (n_corr > 0) {
    k.N = nc;
    k.corr = true;
    rc = fo::launch_metric_batch_detail(k, num_sms, fo::DetailView{first_dev + n_diag, prob_dev + n_diag, n_corr}, st);
    if (rc != FO_OK) return rc;
  }
  FO_CUDA_TRY(cudaEventRecord(slot->done, st));
  return FO_OK;
}

extern "C" int fo_metric_batch_detail(const FoMetricBatchArgs* b, void* stream) {
  return metric_batch_detail_impl("fo_metric_batch_detail", b, nullptr, nullptr, stream);
}

extern "C" int fo_metric_batch_detail_vehicles(const FoMetricBatchArgs* b, const FoVehicle* vehicles_host, void* stream) {
  const char* fn = "fo_metric_batch_detail_vehicles";
  if (b && b->n_problems > 0 && !vehicles_host) { fo::set_error("%s: vehicles_host must not be NULL", fn); return FO_ERR_INVALID_ARG; }
  return metric_batch_detail_impl(fn, b, nullptr, vehicles_host, stream);
}

// Correlated and diagonal problems in one batch: corr_host[p] != 0 = problem p's table is a correlated one.
static int check_corr_args(const char* fn, const FoMetricBatchArgs* b, const uint8_t* corr_host, const FoVehicle* vehicles_host) {
  if (b && b->n_problems > 0 && (!corr_host || !vehicles_host)) {
    fo::set_error("%s: corr_host and vehicles_host must not be NULL", fn);
    return FO_ERR_INVALID_ARG;
  }
  return FO_OK;
}

extern "C" int fo_metric_batch_corr(const FoMetricBatchArgs* b, const uint8_t* corr_host, const FoVehicle* vehicles_host,
                                    void* stream) {
  const char* fn = "fo_metric_batch_corr";
  const int rc = check_corr_args(fn, b, corr_host, vehicles_host);
  return rc != FO_OK ? rc : metric_batch_impl(fn, b, corr_host, vehicles_host, false, nullptr, stream);
}

extern "C" int fo_metric_batch_detail_corr(const FoMetricBatchArgs* b, const uint8_t* corr_host,
                                           const FoVehicle* vehicles_host, void* stream) {
  const char* fn = "fo_metric_batch_detail_corr";
  const int rc = check_corr_args(fn, b, corr_host, vehicles_host);
  return rc != FO_OK ? rc : metric_batch_detail_impl(fn, b, corr_host, vehicles_host, stream);
}

extern "C" int fo_metric_batch_select(const FoMetricBatchArgs* b, const uint8_t* corr_host, const FoVehicle* vehicles_host,
                                      int32_t* selected_dev, void* stream) {
  return metric_batch_impl("fo_metric_batch_select", b, corr_host, vehicles_host, true, selected_dev, stream);
}
