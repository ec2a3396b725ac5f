// Stage 2: path-following vehicle rollout (Frenet quartic/quintic samples along a reference polyline).
// One warp per (agent, route) job; lanes = time steps.  Double arithmetic: the job count is tiny
// (<= a few dozen per planning cycle) and the float32 outputs should be the rounded image of a float64
// evaluation.  Restated from utils/frenetix_handler.py:66-125 and agent.py:364-426 (the C++ frenetix
// library itself is not available: parity unpinned, validated on invariants).
#include <math_constants.h>

#include "fo_common.cuh"

namespace fo {

constexpr int kMaxPathPts = 1024;
constexpr unsigned kFullMask = 0xffffffffu;
// a vertex closer than this to its predecessor is dropped: the heading of a (near-)zero chord is atan2 of rounding noise,
// and it would enter the curvature and yaw of the neighbouring samples (route paths end in such chords)
constexpr double kMinChord = 1e-3;

struct FrenetState { double s, sd, d, dd; };

// low_vel: frenetix' low-velocity mode (utils/frenetix_handler.py:91-95, v0 < 0.5 m/s): the lateral quintic runs over the
// covered ARC LENGTH instead of over time (a vehicle that barely moves cannot shift sideways), d' = dd/ds * ds/dt.
// Beyond the sampling horizon t1 (real agents: horizon 5 s > t1 = 3 s) the end speed and offset are kept.
__device__ __forceinline__ FrenetState frenet_at(double t, double t1, double s0, double v0, double sd1, double d0, double d1,
                                                 bool low_vel) {
  FrenetState f;
  // quartic: s(0)=s0, s'(0)=v0, s''(0)=0, s'(t1)=sd1, s''(t1)=0
  const double a3 = (sd1 - v0) / (t1 * t1), a4 = (v0 - sd1) / (2.0 * t1 * t1 * t1);
  const double s1 = s0 + v0 * t1 + a3 * t1 * t1 * t1 + a4 * t1 * t1 * t1 * t1;
  if (t < t1) {
    f.s = s0 + v0 * t + a3 * t * t * t + a4 * t * t * t * t;
    f.sd = v0 + 3.0 * a3 * t * t + 4.0 * a4 * t * t * t;
  } else {
    f.s = s1 + sd1 * (t - t1);
    f.sd = sd1;
  }
  if (t < t1 || low_vel) {
    // quintic: d(0)=d0, d'(0)=d''(0)=0, d(end)=d1, d'(end)=d''(end)=0 over time, or over arc length in low_vel mode
    // (there d follows the covered arc length at every t: an agent that has not moved has not shifted sideways)
    const double span = low_vel ? fmax(s1 - s0, 1e-9) : t1;
    const double tau = low_vel ? fmin(fmax((f.s - s0) / span, 0.0), 1.0) : t / t1;
    const double t2 = tau * tau, t3 = t2 * tau;
    f.d = d0 + (d1 - d0) * (10.0 * t3 - 15.0 * t3 * tau + 6.0 * t3 * t2);
    f.dd = (d1 - d0) / span * (30.0 * t2 - 60.0 * t3 + 30.0 * t2 * t2) * (low_vel ? f.sd : 1.0);
  } else {
    f.d = d1;
    f.dd = 0.0;
  }
  return f;
}

// polyline lookup: segment index for arc length s (clamped; extrapolates on the first / last segment)
__device__ __forceinline__ int seg_of(const double* cum, int np, double s) {
  int lo = 0, hi = np - 2;
  while (lo < hi) {
    int mid = (lo + hi + 1) >> 1;
    if (cum[mid] <= s) lo = mid; else hi = mid - 1;
  }
  return lo;
}

__global__ void __launch_bounds__(32) fo_rollout_path_kernel(const FoRolloutPathArgs k) {
  __shared__ double cum[kMaxPathPts];      // arc length at every vertex
  __shared__ float2 pts[kMaxPathPts];
  __shared__ double head[kMaxPathPts];     // heading of segment j (vertex j -> j + 1)
  const int job = blockIdx.x, lane = threadIdx.x;
  const int off = k.path_off[job], n_in = min(k.path_off[job + 1] - off, kMaxPathPts);
  const size_t row = (size_t)job * k.t_stride;
  int np = 0;
  {   // stage the polyline without vertices closer than kMinChord to their input predecessor: ballot + prefix per chunk
    const float2* src = reinterpret_cast<const float2*>(k.path_xy) + off;
    for (int j0 = 0; j0 < n_in; j0 += 32) {
      const int j = j0 + lane;
      bool keep = false;
      float2 p = make_float2(0.0f, 0.0f);
      if (j < n_in) {
        p = src[j];
        keep = j == 0;
        if (!keep) {
          const float2 q = src[j - 1];
          const double dx = (double)p.x - q.x, dy = (double)p.y - q.y;
          keep = !(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)) < kMinChord * kMinChord);
        }
      }
      const unsigned kept = __ballot_sync(kFullMask, keep);
      if (keep) pts[np + __popc(kept & ((1u << lane) - 1u))] = p;   // writes only at or below j: reads come from src
      np += __popc(kept);
    }
  }
  if (np < 2) {
    if (lane == 0) k.sample[job] = -1;
    for (int i = lane; i < k.t_stride; i += 32) { k.x[row + i] = 0; k.y[row + i] = 0; k.yaw[row + i] = 0; k.vel[row + i] = 0; k.var_x[row + i] = 0; k.var_y[row + i] = 0; }
    return;
  }
  __syncwarp();
  {   // arc length at every vertex: warp scan over chunks of 32 chords (a route path has up to 1024 vertices)
    double carry = 0.0;
    for (int j0 = 0; j0 < np; j0 += 32) {
      const int j = j0 + lane;
      double sc = (j >= 1 && j < np) ? hypot((double)pts[j].x - pts[j - 1].x, (double)pts[j].y - pts[j - 1].y) : 0.0;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const double t = __shfl_up_sync(kFullMask, sc, o);
        if (lane >= o) sc += t;
      }
      if (j < np) cum[j] = carry + sc;
      carry += __shfl_sync(kFullMask, sc, 31);
    }
  }
  for (int j = lane; j < np - 1; j += 32)
    head[j] = atan2((double)pts[j + 1].y - pts[j].y, (double)pts[j + 1].x - pts[j].x);
  __syncwarp();

  // ---- projection of the start position: closest point over all segments -> (s0, d0) -----------------
  const double px = k.x0[job], py = k.y0[job], v0 = k.v0[job];
  double best = CUDART_INF, bs = 0.0, bd = 0.0;
  for (int j = lane; j < np - 1; j += 32) {
    const double ax = pts[j].x, ay = pts[j].y, ex = pts[j + 1].x - ax, ey = pts[j + 1].y - ay;
    const double l2 = ex * ex + ey * ey;
    if (l2 <= 0.0) continue;
    double u = ((px - ax) * ex + (py - ay) * ey) / l2;
    const double uc = (j == 0 && u < 0.0) || (j == np - 2 && u > 1.0) ? u : fmin(fmax(u, 0.0), 1.0);   // open ends extrapolate
    const double qx = ax + uc * ex, qy = ay + uc * ey;
    const double dist = hypot(px - qx, py - qy);
    if (dist < best) {
      best = dist;
      const double l = sqrt(l2);
      bs = cum[j] + uc * l;
      bd = (ex * (py - ay) - ey * (px - ax)) / l;    // signed lateral offset, left of the path positive
    }
  }
  for (int o = 16; o > 0; o >>= 1) {
    const double ob = __shfl_xor_sync(kFullMask, best, o), os = __shfl_xor_sync(kFullMask, bs, o), od = __shfl_xor_sync(kFullMask, bd, o);
    if (ob < best || (ob == best && os < bs)) { best = ob; bs = os; bd = od; }
  }
  const double s0 = bs, d0 = bd;
  const bool low_vel = v0 < 0.5;                        // frenetix_handler.py:91-95

  // ---- 3 x 3 samples: variance of the Cartesian speed over the horizon -----------------------------------
  const int T = k.n_states;
  int best_k = 0;
  double best_var = CUDART_INF;
  for (int smp = 0; smp < 9; ++smp) {
    const double sd1 = v0 * (0.8 + 0.2 * (double)(smp / 3)), d1 = -0.5 + 0.5 * (double)(smp % 3);
    double sum = 0.0, sq = 0.0;
    for (int i = lane; i < T; i += 32) {
      const FrenetState f = frenet_at((double)i * k.dt, k.t1, s0, v0, sd1, d0, d1, low_vel);
      const int j = seg_of(cum, np, f.s);
      // curvature of the polyline at segment j: heading change to the next segment over the mean length
      double kap = 0.0;
      if (j + 2 < np) {
        double dh = head[j + 1] - head[j];
        dh -= 2.0 * CUDART_PI * rint(dh / (2.0 * CUDART_PI));
        kap = dh / (0.5 * (cum[j + 2] - cum[j]));
      }
      const double vl = f.sd * (1.0 - kap * f.d);
      const double v = sqrt(vl * vl + f.dd * f.dd);
      sum += v;
      sq += v * v;
    }
    for (int o = 16; o > 0; o >>= 1) { sum += __shfl_xor_sync(kFullMask, sum, o); sq += __shfl_xor_sync(kFullMask, sq, o); }
    const double mean = sum / T, var = fmax(sq / T - mean * mean, 0.0);   // np.var (population)
    if (var < best_var - 1e-15) { best_var = var; best_k = smp; }
  }
  if (lane == 0) k.sample[job] = best_k;

  // ---- write the selected sample -------------------------------------------------------------------------
  const double sd1 = v0 * (0.8 + 0.2 * (double)(best_k / 3)), d1 = -0.5 + 0.5 * (double)(best_k % 3);
  for (int i = lane; i < k.t_stride; i += 32) {
    float ox = 0, oy = 0, oyaw = 0, ov = 0, ovar = 0;
    if (i < T) {
      const FrenetState f = frenet_at((double)i * k.dt, k.t1, s0, v0, sd1, d0, d1, low_vel);
      const int j = seg_of(cum, np, f.s);
      const double ax = pts[j].x, ay = pts[j].y, ex = pts[j + 1].x - ax, ey = pts[j + 1].y - ay;
      const double l = fmax(cum[j + 1] - cum[j], 1e-12);
      const double u = (f.s - cum[j]) / l;
      const double tx = ex / l, ty = ey / l;
      double kap = 0.0;
      if (j + 2 < np) {
        double dh = head[j + 1] - head[j];
        dh -= 2.0 * CUDART_PI * rint(dh / (2.0 * CUDART_PI));
        kap = dh / (0.5 * (cum[j + 2] - cum[j]));
      }
      const double vl = f.sd * (1.0 - kap * f.d);
      ox = (float)(ax + u * ex - f.d * ty);
      oy = (float)(ay + u * ey + f.d * tx);
      oyaw = (float)(head[j] + atan2(f.dd, vl));
      ov = (float)sqrt(vl * vl + f.dd * f.dd);
      ovar = (float)(k.var0 * pow(k.var_factor, (double)i));
    }
    k.x[row + i] = ox; k.y[row + i] = oy; k.yaw[row + i] = oyaw; k.vel[row + i] = ov;
    k.var_x[row + i] = ovar; k.var_y[row + i] = ovar;
  }
}

}  // namespace fo

extern "C" int fo_rollout_path(const FoRolloutPathArgs* a, void* stream) {
  if (!a) { fo::set_error("fo_rollout_path: NULL args"); return FO_ERR_INVALID_ARG; }
  if (a->n_jobs < 0 || a->n_states < 0 || a->t_stride < a->n_states || !(a->t1 > 0.0)) {
    fo::set_error("fo_rollout_path: bad sizes");
    return FO_ERR_INVALID_ARG;
  }
  if (a->n_jobs == 0 || a->t_stride == 0) return FO_OK;
  if (!a->path_xy || !a->path_off || !a->x0 || !a->y0 || !a->v0 || !a->x || !a->y || !a->yaw || !a->vel ||
      !a->var_x || !a->var_y || !a->sample) {
    fo::set_error("fo_rollout_path: NULL array");
    return FO_ERR_INVALID_ARG;
  }
  fo::fo_rollout_path_kernel<<<a->n_jobs, 32, 0, (cudaStream_t)stream>>>(*a);
  fo::count_launch();
  FO_CUDA_TRY(cudaGetLastError());
  return FO_OK;
}
