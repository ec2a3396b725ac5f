// Shared internals of libfo_b200.so (not part of the public ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "fo_b200.h"

namespace fo {

void set_error(const char* fmt, ...);
void count_launch(uint64_t n = 1);

// Host-side argument checks of the batch entry points (fo_metric.cu), before any device work; fn names the entry point
// in the messages.  check_batch: the metric calls (detail: fo_metric_batch_detail's outputs); on success *n_run = the
// problems with trajectories and *a_min = the fewest agents among them.  check_pack_batch: fo_agents_pack_batch; on
// success *n_packed = the problems with agents and *max_cells = the most table cells of one of them.  corr: NULL = every
// table is diagonal, else corr[p] != 0 = problem p's table is a correlated one (fo_agent_table_bytes_corr bytes).
int check_batch(const char* fn, const FoMetricBatchArgs* b, const uint8_t* corr, bool detail, int* n_run, int* a_min);
int check_pack_batch(const char* fn, const FoAgentsRaw* raw, int32_t n_problems, const FoBatchProblem* problems,
                     const uint8_t* corr, const void* arena_dev, size_t arena_bytes, int* n_packed, int* max_cells);

// fo_metric_batch_host's float64 -> float32 conversion of ego rows [row0, row0 + n_rows) of a batch ([rows, T, 5], src
// and dst point at row row0): first_dev[n_first] = the first rows of the problems with trajectories (strictly
// increasing, first_dev[0] = 0) and origin_dev[n_first] their origins.  One launch (fo_metric.cu).
int launch_ego_ingest(const double* src, float* dst, int row0, int n_rows, int T, const int* first_dev,
                      const double2* origin_dev, int n_first, cudaStream_t st);

#define FO_CUDA_TRY(expr)                                                                      \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess) {                                                                   \
      fo::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return FO_ERR_CUDA;                                                                      \
    }                                                                                          \
  } while (0)

// ---- packed agent table (written by fo_agents_pack, read by the metric kernels) ----------------
// Agents are stored in SLOT order: stable-sorted by harm model (unprotected first, then protected), so that a warp
// whose lanes are 32 consecutive slots runs ONE harm model (the LR4S impact-angle path costs an atan2f per state and
// would otherwise execute for every warp with a quarter of its lanes).  Per-trajectory results are order-independent
// reductions; the detail outputs are written at the ORIGINAL agent index through `orig`.
// [ float4 s0[A*Tp] | float4 s1[A*Tp] | AgentParams prm[A] | time-major copies ... | float2 s2[A*Tp] | tpsi | orig | slot ]
//   s0[i] = (px_i, py_i, cos yaw_i, sin yaw_i)
//   s1[i] = (yaw_i, v_i, px_{i-1}, py_{i-1})       previous position: CP pairs ego step i with agent
//                                                    position i-1 (collision_probability.py:52)
//   s2[i] = (1/(sqrt2 sigma_x), 1/(sqrt2 sigma_y)) of covariance i-1 (collision_probability.py:80)
struct __align__(16) AgentParams {
  int32_t n_states;
  int32_t model;   // 0 = unprotected (LR1S ego / pedestrian logit), 1 = protected (LR4S both), 2 = none (harm 1)
  float hl, hw;    // half extents of the unbuffered agent.shape  (DCE, BE)
  float hlb;       // half of the buffered prediction length     (CP front/back points)
  float ke, ko;    // m_o/(m_e+m_o), m_e/(m_e+m_o)               (harm_model.py:96-97)
  float pad;       // circumradius sqrt(hl^2 + hw^2)
};

// TIME-MAJOR copies for kernels whose lanes are agents (consecutive lanes read consecutive entries):
//   t0[i*Ap + a] = s0[a*Tp + i],  tv[i*Ap + a] = v_i,  tpsi[i*Ap + a] = yaw_i;  Ap = A rounded up to 32, padding zeroed
struct AgentTableView {
  const float4* s0;
  const float4* s1;
  const float2* s2;
  const AgentParams* prm;
  const float4* t0;
  const float* tv;
  const float4* aw;   // [n_windows][Ap] (x_lo, x_hi, y_lo, y_hi) of the positions at steps [8w-1, 8w+7] the agent has
  const float* avw;   // [n_windows][Ap] max speed over steps [8w, 8w+7]
  const float* tpsi;  // [Tp][Ap] yaw, time-major (impact-angle classes of the detail kernel)
  const int32_t* orig;  // [Ap] slot -> original agent index (-1 for padding slots)
  const int32_t* slot;  // [Ap] original agent index -> slot
  int Ap;
};

#ifndef FO_WIN_STEPS
#define FO_WIN_STEPS 8
#endif
constexpr int kWinSteps = FO_WIN_STEPS;   // steps per window of the summary kernel's window filter
__host__ __device__ inline int agent_windows(int Tp) { return (Tp + kWinSteps - 1) / kWinSteps; }

__host__ __device__ inline int agent_pad(int A) { return (A + 31) & ~31; }
__host__ __device__ inline size_t agent_table_bytes(int A, int Tp) {
  return (size_t)A * Tp * (2 * sizeof(float4) + sizeof(float2)) + (size_t)A * sizeof(AgentParams) +
         (size_t)agent_pad(A) * Tp * (sizeof(float4) + 2 * sizeof(float)) +
         (size_t)agent_pad(A) * agent_windows(Tp) * (sizeof(float4) + sizeof(float)) +
         (size_t)agent_pad(A) * 2 * sizeof(int32_t);
}
__host__ __device__ inline AgentTableView agent_table_view(const void* base, int A, int Tp) {
  AgentTableView v;
  v.s0 = reinterpret_cast<const float4*>(base);
  v.s1 = v.s0 + (size_t)A * Tp;
  v.prm = reinterpret_cast<const AgentParams*>(v.s1 + (size_t)A * Tp);
  v.t0 = reinterpret_cast<const float4*>(v.prm + A);
  v.Ap = agent_pad(A);
  v.tv = reinterpret_cast<const float*>(v.t0 + (size_t)v.Ap * Tp);
  v.aw = reinterpret_cast<const float4*>(v.tv + (size_t)v.Ap * Tp);
  v.avw = reinterpret_cast<const float*>(v.aw + (size_t)v.Ap * agent_windows(Tp));
  v.s2 = reinterpret_cast<const float2*>(v.avw + (size_t)v.Ap * agent_windows(Tp));
  v.tpsi = reinterpret_cast<const float*>(v.s2 + (size_t)A * Tp);
  v.orig = reinterpret_cast<const int32_t*>(v.tpsi + (size_t)v.Ap * Tp);
  v.slot = v.orig + v.Ap;
  return v;
}

// Correlated tables (fo_agents_pack_corr): the table above, then, 16-byte aligned, one more agent-major section
//   s3[i] = (1/sigma_x, 1/sigma_y, rho, 0) of covariance i-1, slot order (rho NaN when the covariance is not positive definite)
__host__ __device__ inline size_t agent_corr_offset(int A, int Tp) { return (agent_table_bytes(A, Tp) + 15) & ~(size_t)15; }
__host__ __device__ inline size_t agent_table_bytes_corr(int A, int Tp) {
  return agent_corr_offset(A, Tp) + (size_t)A * Tp * sizeof(float4);
}
__host__ __device__ inline const float4* agent_corr_view(const void* base, int A, int Tp) {
  return reinterpret_cast<const float4*>(reinterpret_cast<const unsigned char*>(base) + agent_corr_offset(A, Tp));
}

// sigma_x, sigma_y and rho of the covariance [[vx, c], [c, vy]] in float64, the all-zero matrix taken as 0.1 I
// (collision_probability.py:85-87); true when it is positive definite (|rho| < 1).  The one predicate of both places
// that look at it: fo_agents_corr_kernel writes rho = NaN where it is false, fo_metric_batch_host_corr rejects the call.
__host__ __device__ inline bool corr_terms(float vx, float vy, float c, double* sx, double* sy, double* rho) {
  if (vx == 0.0f && vy == 0.0f && c == 0.0f) { vx = 0.1f; vy = 0.1f; }
  *sx = sqrt((double)vx);
  *sy = sqrt((double)vy);
  *rho = (double)c / (*sx * *sy);
  return fabs(*rho) < 1.0;
}

}  // namespace fo
