// Dense metric core of the Frenetix-Occlusion assessment path, sm_100a -- DETAIL kernel.
//
// Used when the caller wants the per-pair / per-step arrays of the reference result dict (drop-in
// Metric.evaluate_metrics, FOInterface.prefetch_assessments, assess_bundle(want_pair / want_step)); the
// throughput / latency path without those arrays is fo_metric_sweep.cu.  Per (trajectory n, prediction a, step i):
//   CP   metrics/utils/collision_probability.py:37-124   (Gaussian mass over three ego boxes, 5 m gate)
//   DCE  metrics/dce.py:52-99 + utils/convert_dynamic_obstacle.py  (oriented-box distance, round 1e-3)
//   TTC / TTCE / WTTC  metrics/ttc.py, ttce.py, wttc.py   (post-processing of DCE)
//   HR   metrics/utils/harm_model.py:58-105, logistic_regression.py, hr.py:76-114
//   BE   metrics/be.py:31-193                              (bisection on constant deceleration)
// followed by the threshold mask of metrics/metric.py:50-98.
//
// Mapping (same layout as the summary kernel: LANE = AGENT, time-major agent table):
//   * one WARP owns one trajectory at a time (its T ego states staged in the warp's own shared memory; warps never
//     synchronise with each other and claim trajectories from a device counter) and walks the agents in tiles of 32
//     consecutive SLOTS (slots are sorted by harm model in fo_agents_pack, so a tile runs one model); every lane walks
//     the T steps of its agent: per-pair reductions over time are register updates or shared-memory keys -- no shuffles;
//   * the step loop evaluates what every (agent, step) needs -- both harm values -- and only BOUNDS for the two
//     expensive parts: squared centre distance against an upper bound of the pair's minimum (a cheap pre-pass gives
//     min_i |centres|, the running exact minimum tightens it) and the 5 m gate of the collision probability.  Steps
//     that pass are pushed on two per-warp shared-memory queues and evaluated 32 at a time with all lanes busy: exact
//     oriented-box distance with np.round(d, 3) (float64 re-rounding next to a rounding boundary), 36-term Gaussian
//     box mass.  A collision probability joins its pair's maxima (risk = harm x cp, argmax cp) through shared-memory
//     atomics on order-preserving keys; its harm factors are read back from where the step loop stored them, so the
//     per-pair maxima are bit-for-bit the maxima of the per-step arrays that go to HBM;
//   * step[n, a, :, :] is a contiguous run of 12 (T-1) bytes per pair, but a lane = agent store pattern would touch
//     one 32-byte sector per lane and step: the (cp, ego_harm, obst_harm) triples of 16 steps are transposed through
//     a per-warp shared-memory tile and leave as 192-byte row segments (8-byte stores when T-1 is even);
//   * colliding pairs run the warp-cooperative BE bisection of the summary kernel (be_bisect, lanes = steps).
#include "fo_metric_dev.cuh"

namespace fo {

#ifndef FO_DT_MINB
#define FO_DT_MINB 5
#endif
#ifndef FO_DT_CHUNK
#define FO_DT_CHUNK 16
#endif
#ifndef FO_DT_WARPS
#define FO_DT_WARPS 4
#endif
constexpr int kDtChunk = FO_DT_CHUNK;        // steps per flush of the staging tile
constexpr int kDtRow = 3 * kDtChunk + 2;     // row stride in floats (even: rows stay 8-byte aligned)
constexpr int kDtQueue = 64;                 // <= 31 left over + 32 new items
constexpr int kDtWarps = FO_DT_WARPS;        // independent warps per CTA (no CTA-level synchronisation at all)
constexpr int kDtInvBytes = (kBeBuckets + 1 + 15) & ~15;

// per-warp shared memory: [ stage | ckey | okey | ekey | dkey | q_near | q_cp | q_tie | inv | egoA | egoB | dist ]
constexpr size_t kDtFixedBytes = 32 * kDtRow * 4 + 32 * (8 + 8 + 4 + 4) + 2 * kDtQueue * 4 + kDtQueue * 8 + kDtInvBytes;
__host__ __device__ inline size_t detail_warp_bytes(int T) {
  return (kDtFixedBytes + (size_t)T * (16 + 8) + (size_t)((T + 3) & ~3) * 4 + 15) & ~(size_t)15;
}

// MUFU forms without the denormal-scaling wrappers nvcc puts around rsqrtf / exp2f when -ftz is off (their arguments
// here are clamped or far from the denormal range)
__device__ __forceinline__ float fast_rsqrt(float x) { float r; asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float fast_ex2(float x) { float r; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float fast_rcp(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
// 1 / (1 + exp(-z))
__device__ __forceinline__ float dt_sigmoid(float z) { return fast_rcp(1.0f + fast_ex2(-1.4426950408889634f * z)); }

// LR4S impact-angle coefficients of ego and obstacle (logistic_regression.py:35-48, harm_model.py:81-105); one copy
// in the kernel (atan2f is ~100 instructions and the kernel sits next to a 32 kB instruction cache)
static __device__ __noinline__ float2 dt_lr4s_pair(float dyr, float dxr, float th, float psi, float side, float rear) {
  const float PI_F = 3.14159265358979323846f;
  const float rel = atan2f(dyr, dxr);
  return make_float2(lr4s_coef(rel - th, side, rear), lr4s_coef(PI_F + rel - psi, side, rear));
}

// per-agent logit coefficients: harm = sigmoid(ks * dv + kc (+ LR4S class coefficient)); harm_model.py:96-105,
// logistic_regression.py:45-48, 71-73
struct HarmLin { float kse, kce, kso, kco; };
__device__ __forceinline__ HarmLin harm_lin(const FoHarmCoeffs& hc, int model, float ke, float ko) {
  HarmLin h;
  const bool m0 = model == 0;
  h.kse = (m0 ? hc.ia_speed : hc.rs_speed) * ke;
  h.kso = (m0 ? hc.ped_speed : hc.rs_speed) * ko;
  h.kce = m0 ? hc.ia_const : hc.rs_const;
  h.kco = m0 ? -hc.ped_const : hc.rs_const;
  return h;
}
// exact harm of one (agent, state): harm_model.py:81-105
__device__ __forceinline__ void dt_harm(const FoHarmCoeffs& hc, int model, const HarmLin& h, float ve, float va, float c,
                                        float dxr, float dyr, float th, float psi, float& he, float& ho) {
  const float dv2 = fmaxf(fmaf(-2.0f * ve * va, c, fmaf(ve, ve, va * va)), 1e-30f);
  const float dv = dv2 * fast_rsqrt(dv2);
  float ze = fmaf(h.kse, dv, h.kce), zo = fmaf(h.kso, dv, h.kco);
  if (model == 1) {
    const float2 cls = dt_lr4s_pair(dyr, dxr, th, psi, hc.rs_side, hc.rs_rear);
    ze += cls.x;
    zo += cls.y;
  }
  he = dt_sigmoid(ze);
  ho = dt_sigmoid(zo);
  if (model == 2) { he = 1.0f; ho = 1.0f; }
}

// np.round(d, 3) next to a x.xxx5 boundary (dce.py:79): queued candidates are re-rounded from a float64 evaluation, up to
// 32 at a time and out of line.  A candidate matters only while its float32 rounding is within two units of its pair's
// running minimum (the float32 value is off by at most one unit); by the time the queue is drained most are not.
__device__ __forceinline__ void dt_drain_ties_body(const float4* t0, const AgentParams* prm, const float* tpsi, int Ap,
                                                   const EgoConst& veh, const float4* egoA, const float2* egoB,
                                                   uint32_t* dkey, const uint2* src, int cnt, int a0, int lane) {
  if (lane < cnt) {
    const uint2 it = src[lane];
    const int ial = (int)(it.x >> 8), ii = (int)(it.x & 0xffu);
    if (it.y <= (dkey[ial] >> 8) + 2u) {
      const int as = a0 + ial;
      const float4 s0 = __ldg(&t0[(size_t)ii * Ap + as]);
      const int4 pa = __ldg(reinterpret_cast<const int4*>(prm + as));
      const float4 EA = egoA[ii];
      const uint32_t r = obb_round_mm_f64(EA.x, EA.y, egoB[ii].x, veh.wb, veh.hEx, veh.hEy, s0.x, s0.y,
                                          __ldg(&tpsi[(size_t)ii * Ap + as]), __int_as_float(pa.z),
                                          __int_as_float(pa.w));
      atomicMin(&dkey[ial], (r << 8) | (uint32_t)ii);
    }
  }
  __syncwarp();
}
static __device__ __noinline__ void dt_drain_ties(const MetricKArgs& k, const float4* egoA, const float2* egoB,
                                                  uint32_t* dkey, const uint2* src, int cnt, int a0, int lane) {
  dt_drain_ties_body(k.tab.t0, k.tab.prm, k.tab.tpsi, k.tab.Ap, k.veh, egoA, egoB, dkey, src, cnt, a0, lane);
}
// batched kernel: the agent table and the ego box are the trajectory's problem's, passed in registers
static __device__ __noinline__ void dt_drain_ties_batch(const float4* t0, const AgentParams* prm, const float* tpsi, int Ap,
                                                        float wb, float hEx, float hEy, const float4* egoA,
                                                        const float2* egoB, uint32_t* dkey, const uint2* src, int cnt,
                                                        int a0, int lane) {
  EgoConst veh;
  veh.wb = wb; veh.hEx = hEx; veh.hEy = hEy;
  dt_drain_ties_body(t0, prm, tpsi, Ap, veh, egoA, egoB, dkey, src, cnt, a0, lane);
}

// MASK != 0: the activated metrics are a compile-time constant (all seven / the default six); 0 = read k.mmask.
// BATCH: every trajectory takes its agent table, agent count, pair / step blocks and ego vehicle from its problem (bv);
// otherwise from k, whose fields then stay kernel-parameter operands.
// CORR: correlated table (fo_metric_bundle_corr): every CP term is the float64 rectangle mass of the full covariance
// (cp_bvn_boxes, the table's s3 section).
template <uint32_t MASK, bool BATCH, bool CORR = false>
__device__ __forceinline__ void detail_body(const MetricKArgs& k, const DetailView& bv) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int T = k.T, Tm1 = T - 1, Apk = k.tab.Ap;
  // ---- shared memory of this warp -----------------------------------------------------------------------------
  unsigned char* const wbase = smem_raw + (size_t)wib * detail_warp_bytes(T);
  float* const stage = reinterpret_cast<float*>(wbase);                          // [32][kDtRow] (cp, ego_harm, obst_harm)
  unsigned long long* const ckey = reinterpret_cast<unsigned long long*>(stage + 32 * kDtRow);   // max cp, first index
  unsigned long long* const okey = ckey + 32;                                    // max obstacle risk, first index
  uint32_t* const ekey = reinterpret_cast<uint32_t*>(okey + 32);                 // max ego risk (bits, >= 0)
  uint32_t* const dkey = ekey + 32;                                              // (round(d * 1000) << 8 | step), min
  uint32_t* const q_near = dkey + 32;                                            // [kDtQueue] (agent lane << 8 | step)
  uint32_t* const q_cp = q_near + kDtQueue;
  uint2* const q_tie = reinterpret_cast<uint2*>(q_cp + kDtQueue);                // [kDtQueue] (item, float32 rounding)
  uint8_t* const inv = reinterpret_cast<uint8_t*>(q_tie + kDtQueue);             // arc-length bucket table (BE)
  float4* const egoA = reinterpret_cast<float4*>(inv + kDtInvBytes);             // [T] (x, y, cos theta, sin theta)
  float2* const egoB = reinterpret_cast<float2*>(egoA + T);                      // [T] (theta, v)
  float* const dist = reinterpret_cast<float*>(egoB + T);                        // [T] cumulative chord length (BE)
  const auto soff = [&](const void* q) { return (uint32_t)(reinterpret_cast<const unsigned char*>(q) - smem_raw); };
  const BeView bev{soff(egoA), soff(egoB), soff(dist), soff(inv), 0u};
  const BeConst bek = be_const(k);                // batched: the table and its stride are set per bisection
  // batched: the trajectory's problem's s3 section, set per trajectory
  const float4* s3 = (CORR && !BATCH) ? agent_corr_view(k.tab.s0, k.A, k.Tp) : nullptr;
  // batched: the warp's copy of its problem's descriptor, behind the per-warp regions (read where used, not held in
  // registers across the trajectory)
  DetailProb* const sdp = reinterpret_cast<DetailProb*>(smem_raw + kDtWarps * detail_warp_bytes(T)) + wib;

  const uint32_t mm = MASK ? MASK : k.mmask;
  const bool do_cp = mm & FO_M_CP, do_dce = mm & FO_M_DCE, do_hr = mm & FO_M_HR, do_be = mm & FO_M_BE,
             do_ttc = mm & FO_M_TTC;
  const unsigned lt_mask = (1u << lane) - 1u;
  float rE = sqrtf(k.veh.hEx * k.veh.hEx + k.veh.hEy * k.veh.hEy);   // batched: per trajectory
  bool rows8 = (Tm1 & 1) == 0 && (reinterpret_cast<uintptr_t>(k.step) & 7u) == 0;   // row segments 8-byte aligned
  size_t traj_step = (size_t)k.A * (size_t)Tm1 * FO_STEP_K;
  float* const srow_lane = stage + lane * kDtRow;

  // warp = trajectory: the first one by global warp index, every further one from the device counter.  A batch looks up
  // the problem of the next trajectory together with its claim.
  const int gw = blockIdx.x * kDtWarps + wib, n_gw = gridDim.x * kDtWarps;
  int p = BATCH ? find_problem(bv.first, bv.P, gw) : 0;
  for (int n = gw; n < k.N;) {
    int n_next = 0, p_next = 0;
    if (lane == 0) {
      n_next = k.claim ? (int)(n_gw + atomicAdd(k.claim, 1u)) : n + n_gw;
      if constexpr (BATCH) p_next = n_next < k.N ? find_problem(bv.first, bv.P, n_next) : 0;
    }
    int nb = n;                                        // the trajectory's index in its pair / step block
    int row = n;                                       // its row in ego / valid / summary / flags
    if constexpr (BATCH) {
      if (lane < (int)(sizeof(DetailProb) / 16))
        reinterpret_cast<int4*>(sdp)[lane] = __ldg(reinterpret_cast<const int4*>(bv.prob + p) + lane);
      __syncwarp();
      if constexpr (CORR) {                            // n numbers the trajectories of the launch's problems
        nb = n - __ldg(bv.first + p);
        row = sdp->row0 + nb;
        s3 = sdp->s0 + sdp->s3_off;
      } else {
        nb = n - sdp->row0;
      }
      rE = sqrtf(sdp->veh.hEx * sdp->veh.hEx + sdp->veh.hEy * sdp->veh.hEy);
      rows8 = (Tm1 & 1) == 0 && (reinterpret_cast<uintptr_t>(sdp->step) & 7u) == 0;
      traj_step = (size_t)sdp->A * (size_t)Tm1 * FO_STEP_K;
    }
    // references into the kernel parameters when not batched (their uses stay constant-bank operands), into the
    // descriptor's shared-memory copy when batched
    const auto& tab = [&]() -> const auto& { if constexpr (BATCH) return *sdp; else return k.tab; }();
    const int& A = BATCH ? sdp->A : k.A;
    const int& Tp = BATCH ? sdp->Tp : k.Tp;
    const int& Ap = BATCH ? sdp->Ap : Apk;
    float* const& pair = BATCH ? sdp->pair : k.pair;
    float* const& step = BATCH ? sdp->step : k.step;
    const EgoConst& veh = BATCH ? sdp->veh : k.veh;
    const auto drain_ties = [&](const uint2* src, int cnt, int a0) {
      if constexpr (BATCH)
        dt_drain_ties_batch(tab.t0, tab.prm, tab.tpsi, Ap, veh.wb, veh.hEx, veh.hEy, egoA, egoB, dkey, src, cnt, a0, lane);
      else
        dt_drain_ties(k, egoA, egoB, dkey, src, cnt, a0, lane);
    };
    // ---- stage the ego trajectory (this warp only) ---------------------------------------------------------------
    const float* eg = k.ego + (size_t)row * T * 5;
    float amin = 0.0f;
    for (int i = lane; i < T; i += 32) {
      const float x = __ldg(eg + i * 5 + 0), y = __ldg(eg + i * 5 + 1), th = __ldg(eg + i * 5 + 2);
      const float v = __ldg(eg + i * 5 + 3);
      amin = fminf(amin, __ldg(eg + i * 5 + 4));
      float sn, cs;
      sincosf(th, &sn, &cs);
      egoA[i] = make_float4(x, y, cs, sn);
      egoB[i] = make_float2(th, v);
    }
    __syncwarp();
    float be_lo0 = 0.0f;
    bool be_ready = false;                                                       // arc-length table built on first use
    if (do_be && do_ttc) {
      const float am = __uint_as_float(__reduce_max_sync(kFull, __float_as_uint(fabsf(amin))));   // |min(min a, 0)|, be.py:68 (amin <= 0)
      be_lo0 = rintf(am * 100.0f) / 100.0f;
    }
    float* const step_n = step ? step + (size_t)nb * traj_step : nullptr;

    // per-lane accumulators over the tiles (reduced once per trajectory)
    float acc_er = 0.0f, acc_or = 0.0f, acc_eh = 0.0f, acc_oh = 0.0f, acc_cp = 0.0f, acc_hwc = 0.0f;
    float acc_btn = 0.0f, acc_rcd = 0.0f;
    uint32_t acc_rmin = 0xffffffu, acc_col = 0xffffffffu, flags = 0u;

    for (int a0 = 0; a0 < A; a0 += 32) {
      const int a = a0 + lane;                           // slot (always inside the padded tables)
      const bool alive = a < A;
      AgentParams P;
      P.n_states = 0; P.model = 2; P.hl = P.hw = P.hlb = P.ke = P.ko = P.pad = 0.0f;
      int ao = 0;
      if (alive) { P = load_params(tab.prm + a); ao = __ldg(tab.orig + a); }
      const int nA = min(T, P.n_states);                 // DCE / CP range (dce.py:87-88, collision_probability.py:73)
      const int nH = min(Tm1, P.n_states);               // harm range (harm_model.py:67)
      const uint32_t rowoff = alive ? (uint32_t)ao * (uint32_t)(Tm1 * FO_STEP_K) : 0xffffffffu;
      const HarmLin hl = harm_lin(k.hc, P.model, P.ke, P.ko);

      // ---- pre-pass: min over time of the squared centre distance = upper bound of the pair's minimum distance --
      float U2 = CUDART_INF_F;
      int i_star = -1;                                   // step of the smallest centre distance
      if (do_dce) {
        const int nAmax = (int)__reduce_max_sync(kFull, (unsigned)nA);
        const float4* t0p = tab.t0 + a;
#pragma unroll 2
        for (int i = 0; i < nAmax; ++i, t0p += Ap) {
          if (i < nA) {
            const float4 s0 = __ldg(t0p);
            const float4 EA = egoA[i];
            const float dx = fmaf(-veh.wb, EA.z, s0.x - EA.x), dy = fmaf(-veh.wb, EA.w, s0.y - EA.y);
            const float c2 = fmaf(dx, dx, dy * dy);
            if (c2 < U2) { U2 = c2; i_star = i; }
          }
        }
      }
      // The exact distance of a step is needed only if its lower bound |centres| - rE - rO can still reach the pair's
      // minimum (+2 units of the 1 mm rounding grid: equal rounded values compete for the FIRST index).  dkey starts at
      // the pre-pass bound (step field 0xff = "no exact value yet"; the step that attains the minimum always passes
      // the bound, so a pair with states ends with a real key).
      const float lim0 = rE + P.pad;
      const uint32_t rU = (U2 < 6.0e7f) ? (uint32_t)(sqrtf(U2) * 1000.0f) + 2u : 0xffffffu;
      ckey[lane] = 0ull; okey[lane] = 0ull; ekey[lane] = 0u; dkey[lane] = (rU << 8) | 0xffu;
      __syncwarp();
      float lim2;
      auto upd_lim = [&]() {
        const float lim = lim0 + (float)((dkey[lane] >> 8) + 2u) * 0.001f;
        lim2 = lim * lim;
      };
      upd_lim();
      int c0 = 0;                                        // first step of the chunk currently staged

      // ---- drains ---------------------------------------------------------------------------------------------
      int qt = 0;
      auto drain_near = [&](const uint32_t* src, int cnt) {
        uint32_t item = 0, r32 = 0;
        bool tie = false;
        if (lane < cnt) item = src[lane];
        __syncwarp();
        if (lane < cnt) {
          const int ial = (int)(item >> 8), ii = (int)(item & 0xffu);
          const int as = a0 + ial;
          const float4 s0 = __ldg(&tab.t0[(size_t)ii * Ap + as]);
          const int4 pa = __ldg(reinterpret_cast<const int4*>(tab.prm + as));
          const float4 EA = egoA[ii];
          const float c = fmaf(EA.z, s0.z, EA.w * s0.w), s = fmaf(s0.w, EA.z, -s0.z * EA.w);
          const float dx = (s0.x - EA.x) - veh.wb * EA.z, dy = (s0.y - EA.y) - veh.wb * EA.w;
          const float rx = fmaf(dx, EA.z, dy * EA.w), ry = fmaf(dy, EA.z, -dx * EA.w);
          const float d = sqrtf(obb_d2(rx, ry, c, s, veh.hEx, veh.hEy, __int_as_float(pa.z), __int_as_float(pa.w)));
          uint32_t r = (uint32_t)__float2int_rn(fminf(d, 8000.0f) * 1000.0f);   // np.round(d, 3), dce.py:79
          // rounding ties: a candidate for the pair's minimum next to a x.xxx5 boundary is queued for a float64
          // re-rounding (the float32 value is off by at most one unit there); until then r + 1 bounds it from above
          tie = near_rounding_boundary(d) && r <= (dkey[ial] >> 8) + 2u;
          r32 = r;
          atomicMin(&dkey[ial], ((r + (tie ? 1u : 0u)) << 8) | (uint32_t)ii);
        }
        {
          const unsigned tb = __ballot_sync(kFull, tie);
          if (tb) {
            if (tie) q_tie[qt + __popc(tb & lt_mask)] = make_uint2(item, r32);
            qt += __popc(tb);
            __syncwarp();
            if (qt >= 32) { qt -= 32; drain_ties(q_tie + qt, 32, a0); }
          }
        }
        __syncwarp();
        upd_lim();
      };
      auto drain_cp = [&](const uint32_t* src, int cnt) {
        uint32_t item = 0;
        if (lane < cnt) item = src[lane];
        __syncwarp();
        const int ial = (int)(item >> 8), ii = (int)(item & 0xffu), t = ii - 1;
        const uint32_t ro = __shfl_sync(kFull, rowoff, ial);
        if (lane < cnt) {
          const int as = a0 + ial;
          const AgentParams Q = load_params(tab.prm + as);
          const size_t idx = (size_t)as * Tp + ii;
          const float4 s0i = __ldg(&tab.s0[idx]);
          const float4 s1i = __ldg(&tab.s1[idx]);
          const float4 Ei = egoA[ii];
          float cp;
          if constexpr (CORR) {
            cp = cp_bvn_boxes(s1i.z - Ei.x, s1i.w - Ei.y, Q.hlb * s0i.z, Q.hlb * s0i.w, veh.L3 * Ei.z, veh.L3 * Ei.w,
                              __ldg(&s3[idx]), veh.L6, veh.W2);
          } else {
            const float2 s2i = __ldg(&tab.s2[idx]);
            cp = cp_gauss_boxes<false>(s1i.z - Ei.x, s1i.w - Ei.y, Q.hlb * s0i.z, Q.hlb * s0i.w, veh.L3 * Ei.z,
                                       veh.L3 * Ei.w, s2i, veh.L6, veh.W2);
          }
          // where the step loop put state t: still in the staging tile, or already in HBM (L2)
          const bool staged = t >= c0;
          float* const srow = stage + ial * kDtRow + 3 * (t - c0);
          float* const grow = step_n ? step_n + ro + 3 * t : nullptr;
          if (step_n) { if (staged) srow[0] = cp; else grow[0] = cp; }
          const unsigned long long tkey = (unsigned long long)(0xffffu - (unsigned)t) << 16;
          if (cp > 0.0f) atomicMax(&ckey[ial], ((unsigned long long)__float_as_uint(cp) << 32) | tkey);
          if (do_hr && cp > 0.0f) {            // risk[t] = harm[t] * cp[t], cp[t] = CP of step t+1 (hr.py:78-79)
            float he, ho;
            if (step_n) {
              he = staged ? srow[1] : __ldcg(grow + 1);
              ho = staged ? srow[2] : __ldcg(grow + 2);
            } else {                           // no step array to read back from: same arithmetic as the step loop
              const float4 s0t = __ldg(&tab.s0[idx - 1]);
              const float4 s1t = __ldg(&tab.s1[idx - 1]);
              const float4 Et = egoA[t];
              const float2 EtB = egoB[t];
              dt_harm(k.hc, Q.model, harm_lin(k.hc, Q.model, Q.ke, Q.ko), EtB.y, s1t.y, fmaf(Et.z, s0t.z, Et.w * s0t.w),
                      s0t.x - Et.x, s0t.y - Et.y, EtB.x, s1t.x, he, ho);
            }
            atomicMax(&ekey[ial], __float_as_uint(he * cp));
            atomicMax(&okey[ial], ((unsigned long long)__float_as_uint(ho * cp) << 32) | tkey);
          }
        }
        __syncwarp();
      };
      // staged rows -> HBM: row r = agent lane r, 3 * cn floats starting at step c0
      auto flush = [&](int cn) {
        const int nf = 3 * cn;
        float* const gdst = step_n + 3 * c0;
        if (rows8) {
          const int j = 2 * lane;
          const float* src = stage + j;
#pragma unroll 4
          for (int r = 0; r < 32; ++r, src += kDtRow) {
            const uint32_t ro = __shfl_sync(kFull, rowoff, r);
            if (ro == 0xffffffffu) break;                       // dead lanes are the last ones of the tile
            if (j + 1 < nf) *reinterpret_cast<float2*>(gdst + ro + j) = *reinterpret_cast<const float2*>(src);
          }
        } else {
#pragma unroll 1
          for (int r = 0; r < 32; ++r) {
            const uint32_t ro = __shfl_sync(kFull, rowoff, r);
            if (ro == 0xffffffffu) break;
            for (int j = lane; j < nf; j += 32) gdst[ro + j] = stage[r * kDtRow + j];
          }
        }
      };

      // The step of the closest centres is queued FIRST: its exact distance is, or is close to, the pair's minimum, so
      // after the first drain (a full one for a full tile, at the top of the step loop) the bound is tight instead of
      // starting at the centre distance.
      int qn = 0;
      if (do_dce) {
        const bool has = i_star >= 0;
        const unsigned b = __ballot_sync(kFull, has);
        if (has) q_near[__popc(b & lt_mask)] = ((uint32_t)lane << 8) | (uint32_t)i_star;
        qn = __popc(b);
        __syncwarp();
      }

      // ---- the step loop: lane = agent, i = state index ----------------------------------------------------------
      float eh_m = 0.0f, oh_m = 0.0f;
      int qc = 0;
      float pxp = 0.0f, pyp = 0.0f;                      // position at i-1 (collision_probability.py:52)
      const float hlb2 = P.hlb * P.hlb, hlbm2 = -2.0f * P.hlb;
      const uint32_t item0 = (uint32_t)lane << 8;
      size_t toff = a;                                   // index into the time-major tables
      float* srow = srow_lane;
      // one extra iteration (i == T, no lane has work) drains what is left in the two queues through the same inlined
      // drain code -- a second inlined copy costs more in instruction-cache misses than the flag costs in the loop
#pragma unroll 1
      for (int i = 0; i <= T; ++i, toff += Ap) {
        const bool last = i == T;
        const bool liveA = i < nA;
        float4 s0 = make_float4(0.0f, 0.0f, 1.0f, 0.0f);
        float va = 0.0f;
        if (liveA) { s0 = __ldg(tab.t0 + toff); va = __ldg(tab.tv + toff); }
        const int ie = last ? Tm1 : i;
        const float4 EA = egoA[ie];
        const float2 EB = egoB[ie];
        const float dxr = s0.x - EA.x, dyr = s0.y - EA.y;
        const float c = fmaf(EA.z, s0.z, EA.w * s0.w);                                // cos(yaw - theta)
        if (do_dce) {
          const float dx = fmaf(-veh.wb, EA.z, dxr), dy = fmaf(-veh.wb, EA.w, dyr);   // centre to centre
          const bool need = liveA & (fmaf(dx, dx, dy * dy) < lim2) & (i != i_star);
          const unsigned b = __ballot_sync(kFull, need);
          if (b || last || qn >= 32) {
            if (need) q_near[qn + __popc(b & lt_mask)] = item0 | (uint32_t)i;
            qn += __popc(b);
            __syncwarp();
            if (qn >= 32 || (last && qn > 0)) { const int cn = min(qn, 32); qn -= cn; drain_near(q_near + qn, cn); }
          }
        }
        if (i < Tm1) {
          // harm at state t = i (same index both sides), harm_model.py:81-105; NaN where the agent has no state
          float he = CUDART_NAN_F, ho = CUDART_NAN_F;
          if (do_hr && i < nH) {
            const float psi = (P.model == 1) ? __ldg(tab.tpsi + toff) : 0.0f;
            dt_harm(k.hc, P.model, hl, EB.y, va, c, dxr, dyr, EB.x, psi, he, ho);
            eh_m = fmaxf(eh_m, he);
            oh_m = fmaxf(oh_m, ho);
          }
          if (step_n) { srow[0] = 0.0f; srow[1] = he; srow[2] = ho; srow += 3; }
        }
        if (do_cp) {                                                                  // 5 m gate, collision_probability.py:61-78
          // min over the points p, p +- h u of |. - e|^2  =  |m|^2 + min(0, h^2 - 2 h |m.u|),  m = p_{i-1} - e_i
          const float mx = pxp - EA.x, my = pyp - EA.y;
          const float mu = fmaf(mx, s0.z, my * s0.w);
          const float dmin = fmaf(mx, mx, my * my) + fminf(fmaf(hlbm2, fabsf(mu), hlb2), 0.0f);
          const bool ingate = liveA & (i >= 1) & (dmin <= 25.0f);
          const unsigned b = __ballot_sync(kFull, ingate);
          if (b || last) {
            if (ingate) q_cp[qc + __popc(b & lt_mask)] = item0 | (uint32_t)i;
            qc += __popc(b);
            __syncwarp();                    // also orders the staging-tile stores of state i-1 before the drain
            if (qc >= 32 || (last && qc > 0)) { const int cn = min(qc, 32); qc -= cn; drain_cp(q_cp + qc, cn); }
          }
        }
        pxp = s0.x; pyp = s0.y;
        if (step_n && i < Tm1 && (i - c0 == kDtChunk - 1 || i == Tm1 - 1)) {
          __syncwarp();
          flush(i - c0 + 1);
          __syncwarp();
          c0 = i + 1;
          srow = srow_lane;
        }
      }
      __syncwarp();
      while (qt > 0) { const int cn = min(qt, 32); qt -= cn; drain_ties(q_tie + qt, cn, a0); }

      // ---- per-pair results ---------------------------------------------------------------------------------------
      const unsigned long long ck = ckey[lane], ok = okey[lane];
      const float cpmax = __uint_as_float((uint32_t)(ck >> 32));
      const int cp_arg = ck ? (int)(0xffffu - (unsigned)((ck >> 16) & 0xffffu)) : 0;
      const float or_m = __uint_as_float((uint32_t)(ok >> 32));
      const int or_arg = ok ? (int)(0xffffu - (unsigned)((ok >> 16) & 0xffffu)) : 0;
      const float er_m = __uint_as_float(ekey[lane]);
      // harm_with_cp = obst_harm[argmax cp] if max cp > 0.01 (hr.py:81-84)
      float hwc = 0.0f;
      if (do_hr && cpmax > 0.01f) {
        if (step_n) {
          hwc = __ldcg(step_n + rowoff + 3 * cp_arg + 2);
        } else {
          const size_t idx = (size_t)a * Tp + cp_arg;
          const float4 s0t = __ldg(&tab.s0[idx]);
          const float4 s1t = __ldg(&tab.s1[idx]);
          const float4 Et = egoA[cp_arg];
          const float2 EtB = egoB[cp_arg];
          float he;
          dt_harm(k.hc, P.model, hl, EtB.y, s1t.y, fmaf(Et.z, s0t.z, Et.w * s0t.w), s0t.x - Et.x, s0t.y - Et.y, EtB.x,
                  s1t.x, he, hwc);
        }
      }
      const uint32_t kmin = dkey[lane];
      const bool has_d = do_dce && (kmin & 0xffu) != 0xffu;          // an exact distance exists (the agent has states)
      const bool collides = has_d && (kmin >> 8) == 0u;
      const int t_col = (int)(kmin & 0xffu);
      acc_er = fmaxf(acc_er, er_m); acc_or = fmaxf(acc_or, or_m);
      acc_eh = fmaxf(acc_eh, eh_m); acc_oh = fmaxf(acc_oh, oh_m);
      acc_cp = fmaxf(acc_cp, cpmax); acc_hwc = fmaxf(acc_hwc, hwc);
      if (has_d) acc_rmin = min(acc_rmin, kmin >> 8);
      if (collides && do_ttc) acc_col = min(acc_col, (uint32_t)t_col);

      // ---- BE for colliding pairs with ttc > 0 (be.py:49-56): warp-cooperative, one pair after the other ----------
      float rcd = 0.0f, btn = 0.0f;
      if (do_be && do_ttc) {
        unsigned todo = __ballot_sync(kFull, collides && t_col > 0);
        if (todo && !be_ready) { be_prepare<false>(bev, T, lane); be_ready = true; }    // arc length + bucket table, be.py:99
        while (todo) {
          const int src = __ffs(todo) - 1;
          todo &= todo - 1;
          const int ns_s = __shfl_sync(kFull, P.n_states, src);
          const float hl_s = __shfl_sync(kFull, P.hl, src), hw_s = __shfl_sync(kFull, P.hw, src);
          BeConst bk = bek;
          if constexpr (BATCH) {                         // the problem's agent-major states and ego box
            bk.s0 = tab.s0; bk.Tp = Tp; bk.wb = veh.wb; bk.hEx = veh.hEx; bk.hEy = veh.hEy;
          }
          const float r = be_bisect<false>(bk, bev, a0 + src, ns_s, hl_s, hw_s, be_lo0, lane, -1.0f).x;
          if (r != r) flags |= FO_F_BE_RANGE;            // NaN: the re-timed path overruns the planned one
          if (lane == src) { rcd = r; btn = __fdividef(r, veh.a_max); }
        }
        acc_rcd = fmaxf(acc_rcd, rcd);     // fmaxf ignores NaN
        acc_btn = fmaxf(acc_btn, btn);
      }
      if (pair && alive) {
        float4* pr = reinterpret_cast<float4*>(pair + ((size_t)nb * A + ao) * FO_PAIR_K);
        pr[0] = make_float4(has_d ? mm_to_m(kmin >> 8) : CUDART_INF_F, has_d ? (float)t_col : 0.0f, er_m, or_m);
        pr[1] = make_float4((float)or_arg, hwc, eh_m, oh_m);
        pr[2] = make_float4(cpmax, rcd, btn, (float)cp_arg);
      }
      __syncwarp();                                   // keys are re-initialised by the next tile
    }  // agent tiles

    // ---- per-trajectory reduction and threshold mask (metric.py:50-98) ----------------------------------------------
    {
      const float er = umaxf(acc_er), orr = umaxf(acc_or), eh = umaxf(acc_eh), oh = umaxf(acc_oh);
      const float cpm = umaxf(acc_cp), hwc_all = umaxf(acc_hwc), btn_all = umaxf(acc_btn), rcd_all = umaxf(acc_rcd);
      const uint32_t rmin = __reduce_min_sync(kFull, acc_rmin), col = __reduce_min_sync(kFull, acc_col);
      const uint32_t fl = __reduce_or_sync(kFull, flags);
      if (lane == 0) {
        const bool has_agents = A > 0 && mm != 0;
        const bool has_col = col != 0xffffffffu;
        bool ok = true;
        if (has_agents) {
          if (do_be && (k.tmask & FO_T_BE) && (double)btn_all > k.thr_be) ok = false;
          if (do_hr && (k.tmask & FO_T_HARM) && (double)hwc_all > k.thr_harm) ok = false;
          if (do_hr && (k.tmask & FO_T_RISK) && (double)orr > k.thr_risk) ok = false;
          if (do_hr && (k.tmask & FO_T_CP) && (double)cpm > k.thr_cp) ok = false;
          if (do_ttc && (k.tmask & FO_T_TTC) && has_col && col < k.thr_ttc_col) ok = false;
          if (do_dce && (k.tmask & FO_T_DCE) && rmin != 0xffffffu && rmin < k.thr_dce_mm) ok = false;
          if (fl & FO_F_BE_RANGE) ok = false;
        }
        k.valid[row] = ok ? 1 : 0;
        if (k.flags) k.flags[row] = fl;
        if (k.summary) {
          float* sm = k.summary + (size_t)row * FO_SUMMARY_K;
          sm[0] = er; sm[1] = orr; sm[2] = eh; sm[3] = oh; sm[4] = cpm; sm[5] = hwc_all;
          sm[6] = (rmin == 0xffffffu || !do_dce) ? CUDART_INF_F : mm_to_m(rmin);
          sm[7] = has_col ? step_to_s(col, k.dtd) : CUDART_INF_F;
          sm[8] = (fl & FO_F_BE_RANGE) ? CUDART_NAN_F : btn_all;
          sm[9] = (fl & FO_F_BE_RANGE) ? CUDART_NAN_F : rcd_all;
        }
      }
    }
    n = __shfl_sync(kFull, n_next, 0);
    if constexpr (BATCH) p = __shfl_sync(kFull, p_next, 0);
    __syncwarp();                                      // the ego arrays are rewritten by the next trajectory
  }
}

template <uint32_t MASK>
__global__ void __launch_bounds__(kDtWarps * 32, FO_DT_MINB) fo_metric_detail_kernel(const __grid_constant__ MetricKArgs k) {
  detail_body<MASK, false>(k, DetailView{});
}

// Correlated tables (fo_metric_bundle_corr), runtime metric mask.
__global__ void __launch_bounds__(kDtWarps * 32, FO_DT_MINB) fo_metric_detail_corr_kernel(const __grid_constant__ MetricKArgs k) {
  detail_body<0u, false, true>(k, DetailView{});
}

// A batch of independent problems (fo_metric_batch_detail): k.N = all rows of the batch, k.tab / k.A / k.Tp / k.pair /
// k.step / k.veh are unused -- every trajectory takes them from its problem.
template <uint32_t MASK>
__global__ void __launch_bounds__(kDtWarps * 32, FO_DT_MINB)
fo_metric_batch_detail_kernel(const __grid_constant__ MetricKArgs k, const __grid_constant__ DetailView bv) {
  detail_body<MASK, true>(k, bv);
}

// The correlated problems of a batch (fo_metric_batch_detail_corr), runtime metric mask: fo_metric_batch_detail_kernel with
// fo_metric_detail_corr_kernel's CP terms.  Its problems' rows need not be contiguous: bv.first numbers the trajectories
// of the launch (k.N = their count), and DetailProb::row0 places each problem's rows.
__global__ void __launch_bounds__(kDtWarps * 32, FO_DT_MINB)
fo_metric_batch_detail_corr_kernel(const __grid_constant__ MetricKArgs k, const __grid_constant__ DetailView bv) {
  detail_body<0u, true, true>(k, bv);
}

// Persistent launches: as many CTAs as fit on the device, their warps claiming trajectories independently.
int launch_metric_detail(const MetricKArgs& k, int num_sms, cudaStream_t st) {
  if (k.pair && (reinterpret_cast<uintptr_t>(k.pair) & 15u)) {
    set_error("fo_metric_bundle: pair must be 16-byte aligned");
    return FO_ERR_INVALID_ARG;
  }
  if (k.step && (reinterpret_cast<uintptr_t>(k.step) & 3u)) {
    set_error("fo_metric_bundle: step must be 4-byte aligned");
    return FO_ERR_INVALID_ARG;
  }
  const size_t smem = (size_t)kDtWarps * detail_warp_bytes(k.T);
  if (k.corr) return launch_persistent<fo_metric_detail_corr_kernel>(k, num_sms, kDtWarps * 32, kDtWarps, smem, false, st);
  return with_mask(k.mmask, [&](auto m) {
    return launch_persistent<fo_metric_detail_kernel<m>>(k, num_sms, kDtWarps * 32, kDtWarps, smem, false, st);
  });
}

// k.N = the batch's rows; the caller has validated the descriptors and the alignment of every pair / step block.  Each
// warp keeps a copy of its problem's descriptor behind the warps' own shared memory.
int launch_metric_batch_detail(const MetricKArgs& k, int num_sms, const DetailView& bv, cudaStream_t st) {
  const size_t smem = (size_t)kDtWarps * (detail_warp_bytes(k.T) + sizeof(DetailProb));
  if (k.corr)
    return launch_persistent<fo_metric_batch_detail_corr_kernel>(k, num_sms, kDtWarps * 32, kDtWarps, smem, false, st, bv);
  return with_mask(k.mmask, [&](auto m) {
    return launch_persistent<fo_metric_batch_detail_kernel<m>>(k, num_sms, kDtWarps * 32, kDtWarps, smem, false, st, bv);
  });
}

}  // namespace fo
