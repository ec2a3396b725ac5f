// Stage 1: sensor visibility by ray casting, sm_100a.
//
// One CTA = 8 warps owns up to 16 fans of 256 consecutive rays of one frame (all 4096 rays of a frame when the call
// has enough frames to fill the GPU; fewer fans per CTA -- more CTAs per frame -- for the planner's single frame);
// one lane = one ray per fan.  Per CTA and tile of 1024 candidate edges (4 per obstacle rectangle + shared road-border
// segments), ONCE:
//   * transform into the ego frame, cull against the sensor disc, orient (cross(a, e) >= 0), compact into shared memory;
//   * per edge: a distance key (squared ego distance of its closest point) and its angular interval relative to ray 0;
//   * counting sort over 32 distance rings -> the staged edges in near-to-far order.
// Per fan: the staged edges whose angular interval meets the fan's are appended IN ORDER to a shared list (five
// compares per edge; round 2a recomputed three cross products per edge and fan).  Every warp walks that list (all
// lanes read the same word: broadcast) with a division-free ray/segment test, keeps the farthest current hit of its
// 32 rays, skips edges whose key lies beyond it and leaves the list at the first ring that lies wholly beyond it:
// in a cluttered scene the near occluders end the walk after a few edges.  Results are those of the plain loop over
// all edges (first hit = minimum; the skip margins are conservative).  Replaces the shapely clipping of
// sensor_model.py:103-193 (one polygon difference per border vertex / obstacle).
#include <math_constants.h>

#include "fo_common.cuh"

namespace fo {

constexpr int kVisThreads = 256;
constexpr int kVisTile = 1024;   // staged edges per tile: 1024 * (16 + 8 + 8 + 4 + 4) B = 40 KB
constexpr int kVisBins = 32;     // distance rings of the near-to-far ordering
constexpr int kVisFans = 16;     // fans one CTA owns at most (one ray per lane and fan)
constexpr int kVisTrCap = 512;   // listed transparent obstacles per frame (more: fall back to scanning all flags)

struct VisEdge {
  float4 g;   // a.x, a.y, e.x, e.y   (segment a -> a + e, ego frame)
};

// squared distance from the ego (origin) to the closest point of a segment: the sensor-disc cull and the distance key
__device__ __forceinline__ float edge_dist2(float ax, float ay, float bx, float by) {
  float ex = bx - ax, ey = by - ay;
  float l2 = fmaf(ex, ex, ey * ey);
  float t = l2 > 0.0f ? fminf(fmaxf(-(ax * ex + ay * ey) / l2, 0.0f), 1.0f) : 0.0f;
  float px = fmaf(t, ex, ax), py = fmaf(t, ey, ay);
  return fmaf(px, px, py * py);            // squared distance ego -> closest point of the segment
}
constexpr float TWO_PI = 6.28318530717958647692f;
constexpr float kVisPad = 2e-4f;   // angular padding of the per-fan cull (float32 atan2f / sincosf noise is ~1e-6)

// ring index (pre-shifted to its bit field) from which every edge lies beyond distance `wmax` with a 0.2 % margin
__device__ __forceinline__ uint32_t vis_ring_end(float wmax, float bin_scale) {
  return (uint32_t)min(kVisBins, (int)ceilf(fmaf(wmax * bin_scale, 1.002f, 1e-3f))) << 10;
}

__device__ __forceinline__ void ray_angle_params(const FoVisibilityArgs& k, float heading, float& a0, float& da) {
  const float PI_F = 3.14159265358979323846f;
  if (k.sensor_angle_deg >= 359.9f) {            // sensor_model.py:119-120
    a0 = heading - PI_F;
    da = 2.0f * PI_F / (float)k.n_rays;
  } else {
    const float fov = k.sensor_angle_deg * (PI_F / 180.0f);
    a0 = heading - 0.5f * fov;
    da = k.n_rays > 1 ? fov / (float)(k.n_rays - 1) : 0.0f;
  }
}

// COUNT: the instrumented twin behind fo_visibility_stats (work counters, never timed)
template <bool COUNT>
__global__ void __launch_bounds__(kVisThreads) fo_visibility_kernel(const FoVisibilityArgs k, const int fans_per_cta,
                                                                    unsigned long long* __restrict__ counters) {
  __shared__ float4 sg[kVisTile];       // a.x, a.y, e.x, e.y of the staged (disc-culled, oriented) edges
  __shared__ float2 st[kVisTile];       // (cross(a, e), owner as int bits)
  __shared__ float2 sphi[kVisTile];     // angular interval [lo, hi] of the edge relative to ray 0, lo in [0, 2 pi), padded
  __shared__ uint32_t s_sorted[kVisTile];  // staged edges near to far: (distance key, 17 bits) | ring << 10 | staged index
  __shared__ uint32_t s_list[kVisTile]; // the current fan's edges, same words, same order (during staging: unsorted words)
  __shared__ int s_bcount[kVisBins], s_boff[kVisBins];
  __shared__ __align__(16) int s_wcnt[2][kVisThreads / 32];
  __shared__ int s_count;
  __shared__ int s_ntr;                 // transparent (bicycle) obstacles of this frame
  __shared__ uint16_t s_tr[kVisTrCap];
  const int f = blockIdx.y;
  const int lane = threadIdx.x & 31;
  const float ex0 = k.ego[f * 3 + 0], ey0 = k.ego[f * 3 + 1], heading = k.ego[f * 3 + 2];
  float a0, da;
  ray_angle_params(k, heading, a0, da);
  const float R = k.sensor_radius, R2 = R * R;
  const float bin_scale = (float)kVisBins / R;
  const int fans_total = (k.n_rays + kVisThreads - 1) / kVisThreads;
  const int fan0 = blockIdx.x * fans_per_cta;
  const int n_fans = min(fans_per_cta, fans_total - fan0);

  unsigned long long n_test = 0, n_skip = 0;   // COUNT only

  // a ray's running first hit lives in its output slots between the tiles of a frame with more than kVisTile edges
  float* const range_f = k.range + (size_t)f * k.n_rays;
  int32_t* const hit_f = k.hit + (size_t)f * k.n_rays;

  const int n_rect_edges = k.n_obstacles * 4;
  const int n_cand = n_rect_edges + k.n_boundary;
  const float* rect = k.rect + (size_t)f * k.n_obstacles * 5;
  const uint8_t* flags = k.rect_flags + (size_t)f * k.n_obstacles;

  // transparent obstacles (type 'bicycle', sensor_model.py:177) cast no shadow but can be seen: list them once
  if (threadIdx.x == 0) s_ntr = 0;
  __syncthreads();
  if (k.visible) {
    for (int o = threadIdx.x; o < k.n_obstacles; o += kVisThreads) {
      const uint8_t fl = flags[o];
      if ((fl & FO_RECT_EXISTS) && (fl & FO_RECT_TRANSPARENT)) {
        const int p = atomicAdd(&s_ntr, 1);
        if (p < kVisTrCap) s_tr[p] = (uint16_t)o;
      }
    }
  }

  for (int base = 0; base < n_cand; base += kVisTile) {
    __syncthreads();                       // previous tile fully cast
    if (threadIdx.x == 0) s_count = 0;
    if (threadIdx.x < kVisBins) s_bcount[threadIdx.x] = 0;
    __syncthreads();
    // ---- stage ONCE per CTA: transform to the ego frame, cull against the sensor disc, orient, compact ----------
    for (int q0 = base; q0 < min(base + kVisTile, n_cand); q0 += kVisThreads) {
      const int q = q0 + threadIdx.x;
      bool keep = false;
      float ax = 0, ay = 0, bx = 0, by = 0, d2 = 0;
      int own = FO_HIT_NONE;
      if (q < min(base + kVisTile, n_cand)) {
        if (q < n_rect_edges) {
          const int o = q >> 2, e = q & 3;
          const uint8_t fl = flags[o];
          if ((fl & FO_RECT_EXISTS) && !(fl & FO_RECT_TRANSPARENT)) {
            const float cx = rect[o * 5 + 0] - ex0, cy = rect[o * 5 + 1] - ey0, yaw = rect[o * 5 + 2];
            const float hl = rect[o * 5 + 3], hw = rect[o * 5 + 4];
            float sn, cs;
            sincosf(yaw, &sn, &cs);
            // corner ring (-l,-w), (-l,+w), (+l,+w), (+l,-w)  (commonroad Rectangle vertex order)
            const float sx0 = (e == 0 || e == 1) ? -1.0f : 1.0f, sy0 = (e == 0 || e == 3) ? -1.0f : 1.0f;
            const float sx1 = (e == 0 || e == 3) ? -1.0f : 1.0f, sy1 = (e == 0 || e == 1) ? 1.0f : -1.0f;
            ax = cx + sx0 * hl * cs - sy0 * hw * sn; ay = cy + sx0 * hl * sn + sy0 * hw * cs;
            bx = cx + sx1 * hl * cs - sy1 * hw * sn; by = cy + sx1 * hl * sn + sy1 * hw * cs;
            own = o;
            d2 = edge_dist2(ax, ay, bx, by);
            keep = d2 <= R2;
          }
        } else {
          const float4 b = reinterpret_cast<const float4*>(k.boundary)[q - n_rect_edges];
          ax = b.x - ex0; ay = b.y - ey0; bx = b.z - ex0; by = b.w - ey0;
          own = FO_HIT_BOUNDARY;
          d2 = edge_dist2(ax, ay, bx, by);
          // a border segment whose line passes through the ego (cross(a, e) == 0) could only block at range 0, and
          // only the half-plane its listed direction faces: dropped, so the result does not depend on that direction
          keep = d2 <= R2 && ax * (by - ay) - ay * (bx - ax) != 0.0f;
        }
      }
      const unsigned m = __ballot_sync(0xffffffffu, keep);
      int pos = 0;
      if (lane == 0 && m) pos = atomicAdd(&s_count, __popc(m));
      pos = __shfl_sync(0xffffffffu, pos, 0);
      if (keep) {
        const int w = pos + __popc(m & ((1u << lane) - 1u));
        float exx = bx - ax, eyy = by - ay;
        float tn = ax * eyy - ay * exx;                      // cross(a, e)
        if (tn < 0.0f) {                                     // orient the edge so that cross(a, e) >= 0: a hit then
          ax = bx; ay = by; exx = -exx; eyy = -eyy; tn = -tn;  // needs cross(d, e) > 0 and the ray test loses its
        }                                                    // sign products and absolute values
        sg[w] = make_float4(ax, ay, exx, eyy);
        // +0, never -0 (an edge through the ego): a range of -0 would be the largest key of the cast's unsigned
        // warp maximum and end the walk of every ray of the warp
        st[w] = make_float2(fabsf(tn), __int_as_float(own));
        // distance key: squared ego distance of the closest point, shrunk by 0.2 % and truncated to 8 mantissa bits
        // (both conservative); ring = its distance bin
        const int b = min(kVisBins - 1, (int)(sqrtf(d2) * bin_scale));
        s_list[w] = (__float_as_uint(d2 * 0.998f) & 0xffff8000u) | ((uint32_t)b << 10) | (uint32_t)w;
        atomicAdd(&s_bcount[b], 1);
        // angular interval, counter-clockwise from a to a + e (cross(a, e) >= 0: at most 180 deg), relative to ray 0
        float ph = atan2f(ay, ax) - a0;
        ph -= TWO_PI * floorf(ph * (1.0f / TWO_PI));
        const float sp = atan2f(tn, fmaf(ax, ax + exx, ay * (ay + eyy)));
        float lo = ph - kVisPad, hi = ph + sp + kVisPad;
        if (lo < 0.0f) { lo += TWO_PI; hi += TWO_PI; }
        if (d2 < 1e-12f) { lo = 0.0f; hi = 3.0f * TWO_PI; }      // the ego stands on the edge: every fan lists it
        sphi[w] = make_float2(lo, hi);
      }
    }
    __syncthreads();
    const int cnt = s_count;
    if (COUNT && threadIdx.x == 0) atomicAdd(&counters[2], (unsigned long long)cnt);
    // near-to-far order of the staged edges (ring granularity): the cast then meets the close occluders first and skips
    // every edge that lies beyond the farthest current hit of its warp's 32 rays
    if (threadIdx.x < 32) {
      const int c0 = s_bcount[lane];
      int inc = c0;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const int o = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += o;
      }
      s_boff[lane] = inc - c0;
    }
    __syncthreads();
    for (int j = threadIdx.x; j < cnt; j += kVisThreads) {
      const uint32_t w = s_list[j];
      const int b = (w >> 10) & 31u;
      s_sorted[s_boff[b] + (atomicSub(&s_bcount[b], 1) - 1)] = w;
    }

    // ---- per fan: angular cull of the staged edges into an ordered list, then cast -------------------------------
#pragma unroll 1
    for (int q = 0; q < n_fans; ++q) {
      const int r_lo = (fan0 + q) * kVisThreads, r_hi = min(r_lo + kVisThreads, k.n_rays) - 1;
      const int r = r_lo + threadIdx.x;
      const float f_lo = da * (float)r_lo, f_hi = da * (float)r_hi;
      __syncthreads();                                 // s_sorted complete / previous fan's list fully consumed
      int nf = 0;
      for (int j0 = 0, par = 0; j0 < cnt; j0 += kVisThreads, par ^= 1) {
        const int p = j0 + threadIdx.x;
        bool keep = false;
        uint32_t w = 0;
        if (p < cnt) {
          w = s_sorted[p];
          const float2 ph = sphi[w & 1023u];
          keep = ((ph.x <= f_hi) & (ph.y >= f_lo)) | (ph.y - TWO_PI >= f_lo);
        }
        // ordered append (no atomics): the list keeps the near-to-far order of s_sorted
        const unsigned m = __ballot_sync(0xffffffffu, keep);
        if (lane == 0) s_wcnt[par][threadIdx.x >> 5] = __popc(m);
        __syncthreads();
        static_assert(kVisThreads == 256, "eight warp counts = two int4");
        const int4 c0 = *reinterpret_cast<const int4*>(&s_wcnt[par][0]), c1 = *reinterpret_cast<const int4*>(&s_wcnt[par][4]);
        const int wi = threadIdx.x >> 5;
        const int p1 = c0.x, p2 = p1 + c0.y, p3 = p2 + c0.z, p4 = p3 + c0.w, p5 = p4 + c1.x, p6 = p5 + c1.y, p7 = p6 + c1.z;
        const int total = p7 + c1.w;
        const int lo4 = wi & 2 ? (wi & 1 ? p3 : p2) : (wi & 1 ? p1 : 0), hi4 = wi & 2 ? (wi & 1 ? p7 : p6) : (wi & 1 ? p5 : p4);
        const int before = wi & 4 ? hi4 : lo4;
        if (keep) s_list[nf + before + __popc(m & ((1u << lane) - 1u))] = w;
        nf += total;
      }
      __syncthreads();
      if (COUNT && threadIdx.x == 0) atomicAdd(&counters[3], (unsigned long long)nf);
      if (r_lo + (int)(threadIdx.x & ~31u) < k.n_rays) {            // warp-uniform: the warp owns at least one ray
        const bool live = r < k.n_rays;
        float c, s;
        sincosf(a0 + da * (float)r, &s, &c);
        float bq = live ? R : 0.0f;
        int oq = FO_HIT_NONE;
        if (base > 0 && live) { bq = range_f[r]; oq = hit_f[r]; }
        // farthest current hit of the warp's rays, squared: an edge whose closest point is not nearer cannot improve any
        float wmax = __uint_as_float(__reduce_max_sync(0xffffffffu, __float_as_uint(bq)));
        float wmax2 = wmax * wmax;
        uint32_t ring_end = vis_ring_end(wmax, bin_scale);          // first ring that lies wholly beyond wmax
#pragma unroll 4
        for (int j = 0; j < nf; ++j) {
          const uint32_t w = s_list[j];
          if (__uint_as_float(w & 0xffff8000u) >= wmax2) {
            if ((w & 0x7c00u) >= ring_end) break;                   // ordered by ring: nothing nearer follows
            if (COUNT) ++n_skip;
            continue;
          }
          if (COUNT) ++n_test;
          const int e = w & 1023u;
          const float4 g = sg[e];
          const float2 t = st[e];
          const float D = c * g.w - s * g.z;           // cross(d, e)
          const float un = g.x * s - g.y * c;          // cross(a, d)
          // t = tn / D >= 0 with tn >= 0, u = un / D in [0, 1], t < best   (division-free, strict improvement only)
          const bool okk = (D > 0.0f) & (un >= 0.0f) & (un <= D) & (t.x < bq * D);
          if (__any_sync(0xffffffffu, okk)) {
            if (okk) {
              bq = t.x / D;
              oq = __float_as_int(t.y);
            }
            wmax = __uint_as_float(__reduce_max_sync(0xffffffffu, __float_as_uint(bq)));
            wmax2 = wmax * wmax;
            ring_end = vis_ring_end(wmax, bin_scale);
          }
        }
        if (live) {
          range_f[r] = bq;
          hit_f[r] = oq;
        }
      }
    }
  }
  __syncthreads();
  if (COUNT) {
    atomicAdd(&counters[0], n_test);                 // ray x edge tests executed (per lane)
    if (lane == 0) atomicAdd(&counters[1], n_skip);  // edges a warp skipped on the distance key
  }

#pragma unroll 1
  for (int q = 0; q < n_fans; ++q) {
    const int r = (fan0 + q) * kVisThreads + threadIdx.x;
    if (r >= k.n_rays) continue;
    float bq = R;
    int oq = FO_HIT_NONE;
    if (n_cand > 0) { bq = range_f[r]; oq = hit_f[r]; }
    else { range_f[r] = bq; hit_f[r] = oq; }            // no occluder at all: the tile loop never ran
    if (k.visible) {
      if (oq >= 0) k.visible[(size_t)f * k.n_obstacles + oq] = 1;
      // transparent obstacles (bicycles): visible when the ray crosses them before its first opaque hit
      const int ntr = s_ntr;
      const bool listed = ntr <= kVisTrCap && k.n_obstacles <= 65535;
      const int n_scan = listed ? ntr : k.n_obstacles;
      if (n_scan > 0) {
        float c, s;
        sincosf(a0 + da * (float)r, &s, &c);
        for (int qq = 0; qq < n_scan; ++qq) {
          const int o = listed ? (int)s_tr[qq] : qq;
          const uint8_t fl = flags[o];
          if ((fl & FO_RECT_EXISTS) && (fl & FO_RECT_TRANSPARENT)) {
            const float cx = rect[o * 5 + 0] - ex0, cy = rect[o * 5 + 1] - ey0;
            float sn, cs;
            sincosf(rect[o * 5 + 2], &sn, &cs);
            const float hl = rect[o * 5 + 3], hw = rect[o * 5 + 4];
            // ray vs box in the box frame (slab test)
            const float ox = -(cx * cs + cy * sn), oy = -(-cx * sn + cy * cs);
            const float dx = c * cs + s * sn, dy = -c * sn + s * cs;
            float t0 = 0.0f, t1 = bq;
            bool hitb = true;
            if (fabsf(dx) > 1e-12f) { float ta = (-hl - ox) / dx, tb = (hl - ox) / dx; t0 = fmaxf(t0, fminf(ta, tb)); t1 = fminf(t1, fmaxf(ta, tb)); }
            else if (fabsf(ox) > hl) hitb = false;
            if (fabsf(dy) > 1e-12f) { float ta = (-hw - oy) / dy, tb = (hw - oy) / dy; t0 = fmaxf(t0, fminf(ta, tb)); t1 = fminf(t1, fmaxf(ta, tb)); }
            else if (fabsf(oy) > hw) hitb = false;
            if (hitb && t0 <= t1) k.visible[(size_t)f * k.n_obstacles + o] = 1;
          }
        }
      }
    }
  }
}

// ---- stage 2: constant-velocity rollout (tiny; double arithmetic so the float32 table is the correctly
// rounded image of the reference's float64 numbers) ------------------------------------------------------
__global__ void fo_rollout_cv_kernel(const FoRolloutCvArgs k) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const int a = idx / k.t_stride, i = idx - a * k.t_stride;
  if (a >= k.n_agents) return;
  float x = 0, y = 0, yaw = 0, v = 0, var = 0;
  if (i < k.n_states) {
    const double phi = k.phi[a], sp = k.v[a];
    const double vx = rint(sp * cos(phi) * 1000.0) / 1000.0;   // round(v cos phi, 3), agent.py:492
    const double vy = rint(sp * sin(phi) * 1000.0) / 1000.0;   // agent.py:493
    const double t = (double)i * k.dt;                           // agent.py:499
    x = (float)(k.x0[a] + t * vx);
    y = (float)(k.y0[a] + t * vy);
    yaw = (float)phi;
    v = (float)sp;
    var = (float)(k.var0 * pow(k.var_factor, (double)i));        // agent.py:272
  }
  const size_t o = (size_t)a * k.t_stride + i;
  k.x[o] = x; k.y[o] = y; k.yaw[o] = yaw; k.vel[o] = v; k.var_x[o] = var; k.var_y[o] = var;
}

}  // namespace fo

static int visibility_launch(const FoVisibilityArgs* a, unsigned long long* counters, void* stream) {
  if (!a) { fo::set_error("fo_visibility_raycast: NULL args"); return FO_ERR_INVALID_ARG; }
  if (a->n_frames < 0 || a->n_rays < 0 || a->n_obstacles < 0 || a->n_boundary < 0) {
    fo::set_error("fo_visibility_raycast: negative size");
    return FO_ERR_INVALID_ARG;
  }
  if (a->n_frames == 0 || a->n_rays == 0) return FO_OK;
  if (!a->ego || !a->range || !a->hit || (a->n_obstacles > 0 && (!a->rect || !a->rect_flags)) ||
      (a->n_boundary > 0 && !a->boundary)) {
    fo::set_error("fo_visibility_raycast: NULL array");
    return FO_ERR_INVALID_ARG;
  }
  if (!(a->sensor_radius > 0.0f)) { fo::set_error("fo_visibility_raycast: sensor_radius must be positive"); return FO_ERR_INVALID_ARG; }
  if (a->n_frames > 65535) { fo::set_error("fo_visibility_raycast: at most 65535 frames per call"); return FO_ERR_UNSUPPORTED; }
  cudaStream_t st = (cudaStream_t)stream;
  if (a->visible && a->n_obstacles > 0)
    FO_CUDA_TRY(cudaMemsetAsync(a->visible, 0, (size_t)a->n_frames * a->n_obstacles, st));
  // fans per CTA: all of a frame's fans (staging done once per frame) when the frames alone fill the GPU, fewer --
  // more CTAs per frame -- for the planner's one or two frames
  const int fans_total = (a->n_rays + fo::kVisThreads - 1) / fo::kVisThreads;
  int dev = 0, sms = 148;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  int fpc = fo::kVisFans;
  while (fpc > 1 && (long long)a->n_frames * ((fans_total + fpc - 1) / fpc) < 4LL * sms) fpc >>= 1;
  if (fpc > fans_total) fpc = fans_total;
  dim3 grid((fans_total + fpc - 1) / fpc, a->n_frames);
  if (counters) fo::fo_visibility_kernel<true><<<grid, fo::kVisThreads, 0, st>>>(*a, fpc, counters);
  else fo::fo_visibility_kernel<false><<<grid, fo::kVisThreads, 0, st>>>(*a, fpc, nullptr);
  fo::count_launch();
  FO_CUDA_TRY(cudaGetLastError());
  return FO_OK;
}

extern "C" int fo_visibility_raycast(const FoVisibilityArgs* a, void* stream) { return visibility_launch(a, nullptr, stream); }

extern "C" int fo_visibility_stats(const FoVisibilityArgs* a, uint64_t* counters_dev, void* stream) {
  if (!counters_dev) { fo::set_error("fo_visibility_stats: NULL counters"); return FO_ERR_INVALID_ARG; }
  FO_CUDA_TRY(cudaMemsetAsync(counters_dev, 0, FO_VIS_STATS_K * sizeof(uint64_t), (cudaStream_t)stream));
  return visibility_launch(a, reinterpret_cast<unsigned long long*>(counters_dev), stream);
}

extern "C" int fo_rollout_cv(const FoRolloutCvArgs* a, void* stream) {
  if (!a) { fo::set_error("fo_rollout_cv: NULL args"); return FO_ERR_INVALID_ARG; }
  if (a->n_agents < 0 || a->n_states < 0 || a->t_stride < a->n_states) {
    fo::set_error("fo_rollout_cv: bad sizes");
    return FO_ERR_INVALID_ARG;
  }
  if (a->n_agents == 0 || a->t_stride == 0) return FO_OK;
  if (!a->x0 || !a->y0 || !a->v || !a->phi || !a->x || !a->y || !a->yaw || !a->vel || !a->var_x || !a->var_y) {
    fo::set_error("fo_rollout_cv: NULL array");
    return FO_ERR_INVALID_ARG;
  }
  const int total = a->n_agents * a->t_stride;
  fo::fo_rollout_cv_kernel<<<(total + 127) / 128, 128, 0, (cudaStream_t)stream>>>(*a);
  fo::count_launch();
  FO_CUDA_TRY(cudaGetLastError());
  return FO_OK;
}
