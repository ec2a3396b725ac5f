// Dense metric core, sm_100a -- the SUMMARY kernel (throughput sweeps and the per-planning-step latency case).
//
// Emits what the planner consumes per trajectory: the validity mask (metrics/metric.py:50-98), ten summary scalars
// and the flags.  Mapping (B200-first, not a translation of the reference's Python loops):
//
//   * one CTA = one TEAM of W warps owns one trajectory (persistent: teams claim trajectories from a per-launch device
//     counter, their cost varies several-fold); its T ego states are staged once in shared memory.  W = 1 for sweeps that oversubscribe the machine; W up to 8 when the whole
//     bundle fits in one wave, because then the latency of a bundle is the critical path of its slowest trajectory;
//   * LANE = (AGENT, TIME SLICE), the loop runs over the steps of the slice: with >= 32 agents a warp holds 32 agents
//     and one slice (the time index is warp-uniform, the ego state one broadcast LDS); with fewer agents the 32 lanes
//     are 32/A' slices x A' agents, so all lanes stay busy for the planner's usual handful of phantom agents.
//     Per-agent parameters stay in registers, consecutive lanes read consecutive entries of the TIME-MAJOR agent
//     table (coalesced), and the previous position the CP pairing needs (collision_probability.py:52) is simply last
//     iteration's register;
//   * the dense step per (trajectory, agent, step) is only *bounds*: squared centre distance vs. the running minimum
//     (oriented-box distance needed?), squared speed difference vs. the running maximum logits (impact-angle class
//     needed?), 5 m gate (collision probability needed?) -- about 50 instructions per 32 evaluations.  Everything
//     that passes a bound is pushed on one of two per-warp shared-memory queues and evaluated 32 items at a time with
//     all lanes active: the exact oriented-box distance (dce.py:75-79) and/or the LR4S impact-angle logit
//     (logistic_regression.py:35-48), and the 9-term Gaussian box mass (collision_probability.py:94-122).  What is
//     left in the queues at the end of an agent tile is pooled across the team and drained cooperatively;
//   * in the one-warp shape with >= 17 agents (UNI, the throughput case) a WINDOW FILTER runs in front of that loop:
//     lane = agent, one test per (agent, window of 8 steps) of the two paths' bounding boxes and top speeds against
//     the same bounds; surviving (agent, window) items are queued and the per-step loop runs with lane = item.  Four
//     out of five items never reach it;
//   * the running minimum distance and the running maximum logits are WARP-SHARED (REDUX after every drain), so a
//     near agent found by one lane prunes the work of all 32;
//   * colliding pairs are collected in a team list for the brake evaluation (BE, be.py:66-193): the one-warp shape walks
//     their common bisection tree (be_walk: one re-timed ego path per probe value instead of one per pair and probe),
//     the team shape deals one bisection per pair round-robin to its warps (be_bisect); per-trajectory results are
//     order-independent min/max reductions (lane -> warp REDUX -> team).
//
// All bounds are exact (a skipped evaluation cannot change a min / max / threshold decision); results equal the detail
// kernel's.  The kernel is instruction-issue- and instruction-cache-bound (DESIGN.md 6): code that exists twice after
// inlining costs more than a flag in a loop, hence the single call sites of the drains and the noinline helpers.  Reference semantics: SURVEY.md appendix A; citations on the helpers in fo_metric_dev.cuh.
#include <stdlib.h>

#include <mutex>

#include "fo_metric_dev.cuh"

namespace fo {

constexpr int kSwMaxWarps = 8;
#ifndef FO_SW_TILE
#define FO_SW_TILE 128
#endif
constexpr int kSwTile = FO_SW_TILE;   // agents per tile (<= 256: 8-bit agent-in-tile field of the window items); bounds the per-team pair arrays
static_assert(kSwTile <= 256, "agent-in-tile fields are 8 bits wide");
constexpr int kSwQueue = 64;
#ifndef FO_SW_MINB
#define FO_SW_MINB 4
#endif
#ifndef FO_SW_UNROLL
#define FO_SW_UNROLL 1
#endif
constexpr int kSwUnroll = FO_SW_UNROLL;
constexpr int kSwWinQueue = 64;   // <= 31 left over + 32 from one filter step
constexpr int kSwInvBytes = (kBeBuckets + 1 + 15) & ~15;   // arc-length bucket table, padded so that what follows stays 16-byte aligned

// The one-warp shape (uni) has no pooled leftovers; the rounding-tie queue exists only in the TIES variants.  At T = 51
// the throughput shape needs 5.6 kB: 32 one-warp CTAs per SM (the register file's limit) fit in shared memory.
__host__ __device__ inline size_t sweep_smem_bytes(int T, int W, bool uni, bool ties) {
  const size_t nW = (size_t)agent_windows(T);
  size_t b = (size_t)kSwTile * (8 + 4 + 2)       // pairkey, colfirst, BE pair list
             + 8 * 4 + kSwInvBytes               // scalars, arc-length bucket table
             + (size_t)kSwWinQueue * 2           // (agent, window) work items of the window filter
             + (size_t)W * (ties ? 3 : 2) * kSwQueue * 4   // per-warp near / cp / rounding-tie queues
             + (uni ? 0 : (size_t)W * 2 * 32 * 4)          // pooled leftovers
             + (size_t)W * 16 * 4                // per-warp partial results
             + nW * 16                           // ego window boxes
             + (size_t)T * (16 + 8 + 16)         // egoA, egoB, BE segment slopes
             + (size_t)((T + 3) & ~3) * 4        // dist
             + nW * 4;                           // ego window speeds
  return (b + 15) & ~(size_t)15;
}

struct SweepSmem {
  unsigned long long* pairkey;  // [kSwTile] (cp bits << 32 | (0xffff - t) << 16 | 1): argmax_t cp, first index on ties
  float4* egoA;                 // [T] (x, y, cos theta, sin theta)
  float2* egoB;                 // [T] (theta, v)
  float* dist;                  // [T] cumulative chord length (BE)
  float4* seg;                  // [T] BE segment slopes (BeView::seg)
  uint32_t* colfirst;           // [kSwTile] first step with rounded distance 0
  uint32_t* q_near;             // [W][kSwQueue] (need LR4S << 31 | need box distance << 30 | agent-in-tile << 8 | step)
  uint32_t* q_cp;               // [W][kSwQueue] (agent-in-tile << 8 | step)
  uint32_t* q_tie;              // [W][kSwQueue] (float32 rounding << 16 | agent-in-tile << 8 | step): distances to re-round in float64
  uint32_t* pool_near;          // [W * 32] leftovers of all warps
  uint32_t* pool_cp;            // [W * 32]
  float* red;                   // [W][16]
  uint32_t* scal;               // [8]: 0 |min(a, 0)| (float bits), 1 BE list length, 2 pooled near, 3 pooled cp
  uint16_t* be_list;            // [kSwTile]
  uint8_t* inv;                 // [kBeBuckets + 1]
  uint16_t* q_win;              // [kSwWinQueue] (agent-in-tile << 8 | window) items that passed the window filter
  float4* ew;                   // [windows] (x_lo, x_hi, y_lo, y_hi) of the ego reference point and centre over a window
  float* evw;                   // [windows] max |v| of the ego over a window
};

// Fixed-size arrays first, then the per-warp ones, then the T-sized ones: every hot array except egoB / dist sits at
// a compile-time offset when W is a constant (the one-warp throughput shape), so its address is an immediate.
__device__ __forceinline__ SweepSmem sweep_smem(unsigned char* base, int T, int W, bool uni, bool ties) {
  SweepSmem w;
  w.pairkey = reinterpret_cast<unsigned long long*>(base);
  w.colfirst = reinterpret_cast<uint32_t*>(w.pairkey + kSwTile);
  w.be_list = reinterpret_cast<uint16_t*>(w.colfirst + kSwTile);
  w.scal = reinterpret_cast<uint32_t*>(w.be_list + kSwTile);
  w.inv = reinterpret_cast<uint8_t*>(w.scal + 8);
  w.q_win = reinterpret_cast<uint16_t*>(w.inv + kSwInvBytes);
  w.q_near = reinterpret_cast<uint32_t*>(w.q_win + kSwWinQueue);
  w.q_cp = w.q_near + (size_t)W * kSwQueue;
  w.q_tie = w.q_cp + (size_t)W * kSwQueue;
  w.pool_near = w.q_tie + (ties ? (size_t)W * kSwQueue : 0);
  w.pool_cp = w.pool_near + (uni ? 0 : (size_t)W * 32);
  w.red = reinterpret_cast<float*>(w.pool_cp + (uni ? 0 : (size_t)W * 32));
  w.ew = reinterpret_cast<float4*>(w.red + (size_t)W * 16);
  w.egoA = w.ew + agent_windows(T);
  w.seg = w.egoA + T;
  w.egoB = reinterpret_cast<float2*>(w.seg + T);
  w.dist = reinterpret_cast<float*>(w.egoB + T);
  w.evw = w.dist + ((T + 3) & ~3);
  return w;
}

// order-preserving float <-> uint map (warp max of signed floats with one REDUX)
__device__ __forceinline__ uint32_t f2ord(float f) {
  uint32_t u = __float_as_uint(f);
  return u ^ ((u >> 31) ? 0xffffffffu : 0x80000000u);
}
__device__ __forceinline__ float ord2f(uint32_t u) {
  return __uint_as_float(u ^ ((u >> 31) ? 0x80000000u : 0xffffffffu));
}
__device__ __forceinline__ float warp_max_signed(float v) { return ord2f(__reduce_max_sync(kFull, f2ord(v))); }
// maximum of values >= 0 or NaN that keeps a NaN (bit order: every NaN above +inf); umaxf is its warp form
__device__ __forceinline__ float nan_maxf(float a, float b) { return __uint_as_float(max(__float_as_uint(a), __float_as_uint(b))); }

__device__ __forceinline__ float sw_sigmoid(float z) { return rcp_approx(1.0f + __expf(-z)); }   // 1 + exp >= 1: same bits as __fdividef(1, .)

// exact harm logits for one (agent, state) -- harm_model.py:81-105, logistic_regression.py:35-48,71-73
__device__ __forceinline__ void sw_harm_logits(const MetricKArgs& k, int model, float ke, float ko, float dv, float dxr,
                                               float dyr, float th, float psi, float& ze, float& zo) {
  if (model == 0) {
    ze = fmaf(k.hc.ia_speed * ke, dv, k.hc.ia_const);
    zo = fmaf(k.hc.ped_speed * ko, dv, -k.hc.ped_const);
  } else if (model == 1) {
    const float2 cls = lr4s_coefs(dyr, dxr, th, psi, k.hc.rs_side, k.hc.rs_rear);
    ze = fmaf(k.hc.rs_speed * ke, dv, k.hc.rs_const) + cls.x;
    zo = fmaf(k.hc.rs_speed * ko, dv, k.hc.rs_const) + cls.y;
  } else {
    ze = CUDART_INF_F;
    zo = CUDART_INF_F;
  }
}

// np.round(d, 3) next to a x.xxx5 boundary (dce.py:79): queued candidates for the minimum are re-rounded from a float64
// evaluation, 32 at a time with all lanes busy and out of line -- the float64 code (6 kB) and its call stay off the hot
// path of the drains.  Returns the minimum of the re-rounded values; steps that round to 0 enter colfirst.
// A queue entry carries the float32 rounding r of its distance ((r capped at 0xffff) << 16 | agent-in-tile << 8 | step).
// The float64 value is r - 1, r or r + 1, so by the time the queue is drained an entry still matters only if it can be a
// collision (r <= 1) or lie below the minimum found since (r <= rmin); when no lane holds such an entry the float64
// code is not entered at all -- in a dense sweep the minimum is 0 after the first collision and the 6 kB stay out of the
// instruction cache.
// K: anything with an EgoConst member veh.  The summary kernel passes its MetricKArgs, whose known 8-byte alignment
// lets adjacent fields be read with one load.
template <class K>
__device__ __forceinline__ uint32_t drain_ties_body(const K& kv, const AgentTableView& tab, const int& Tp,
                                                    const float4* egoA, const float2* egoB, uint32_t* colfirst,
                                                    const uint32_t* src, int cnt, int a0, int lane, uint32_t rmin) {
  uint32_t r = 0xffffffu;
  uint32_t item = 0u;
  bool keep = false;
  if (lane < cnt) {
    item = src[lane];
    const uint32_t rq = item >> 16;
    keep = rq <= 1u || rq <= rmin;
  }
  if (!__any_sync(kFull, keep)) return r;
  if (keep) {
    const int ial = (int)((item >> 8) & 0xffu), ii = (int)(item & 0xffu);
    const int a = a0 + ial;
    const float4 s0 = __ldg(&tab.t0[(size_t)ii * tab.Ap + a]);
    const int4 pa = __ldg(reinterpret_cast<const int4*>(tab.prm + a));
    const float4 EA = egoA[ii];
    r = obb_round_mm_f64(EA.x, EA.y, egoB[ii].x, kv.veh.wb, kv.veh.hEx, kv.veh.hEy, s0.x, s0.y,
                         __ldg(&tab.s1[(size_t)a * Tp + ii]).x, __int_as_float(pa.z), __int_as_float(pa.w));
    if (r == 0u) atomicMin(&colfirst[ial], (uint32_t)ii);
  }
  return __reduce_min_sync(kFull, r);
}
static __device__ __noinline__ uint32_t sw_drain_ties(const MetricKArgs& k, const float4* egoA, const float2* egoB,
                                                      uint32_t* colfirst, const uint32_t* src, int cnt, int a0, int lane,
                                                      uint32_t rmin) {
  return drain_ties_body(k, k.tab, k.Tp, egoA, egoB, colfirst, src, cnt, a0, lane, rmin);
}
// batched kernel: the agent table and the ego box are the trajectory's problem's, passed in registers
static __device__ __noinline__ uint32_t sw_drain_ties_batch(const float4* t0, const AgentParams* prm, const float4* s1,
                                                            int Ap, int Tp, float wb, float hEx, float hEy,
                                                            const float4* egoA, const float2* egoB, uint32_t* colfirst,
                                                            const uint32_t* src, int cnt, int a0, int lane, uint32_t rmin) {
  AgentTableView tab;
  tab.t0 = t0; tab.prm = prm; tab.s1 = s1; tab.Ap = Ap;
  struct { EgoConst veh; } kv;
  kv.veh.wb = wb; kv.veh.hEx = hEx; kv.veh.hEy = hEy;
  return drain_ties_body(kv, tab, Tp, egoA, egoB, colfirst, src, cnt, a0, lane, rmin);
}

// problem of trajectory n: the last p with first[p] <= n
__device__ __forceinline__ int batch_find(const BatchView& b, int n) { return find_problem(b.first, b.P, n); }

// claim n of a select launch -> (descriptor, rank): the segment of n (the last s with seg[s].x <= n), then rank-major
// within it over the segment's active descriptors
__device__ __forceinline__ int2 select_find(const SelectView& s, int n) {
  int lo = 0, hi = s.S - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (__ldg(&s.seg[mid].x) <= n) lo = mid; else hi = mid - 1;
  }
  const int4 g = __ldg(s.seg + lo);
  const int d = n - g.x;
  return make_int2(d % g.z, g.y + d / g.z);
}

// selected[p] as other teams' atomicMin left it: a relaxed load that does not stop in L1
__device__ __forceinline__ int ld_relaxed(const int32_t* p) {
  int v;
  asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}

struct SweepShape {
  int lg_agents;   // log2 of the agents held by one warp (0..5); a warp has 32 >> lg_agents time slices
};

// ---------------------------------------------------------------------------------------------
// UNI: one warp per trajectory and 32 agents per warp pass (the throughput shape): window filter + lane = (agent, window)
// items, no pooled leftovers (see the header comment).
// BATCH: every trajectory takes its agent table, agent count, lane grouping and ego vehicle from its problem (bv);
// otherwise from k.
// CORR: the table is a correlated one (fo_agents_pack_corr): the CP drain evaluates the nine rectangle masses of the
// full covariance (cp_bvn_boxes, the table's s3 section) instead of cp_gauss_boxes; a NaN CP (a covariance that is not
// positive definite) is carried into max_collision_probability_all.
// SELECT (with BATCH): claims map to (descriptor, rank) rank-major (sv, select_find), and a row whose rank exceeds its
// problem's sv.selected is not assessed -- checked when it is claimed, before each agent tile and before the BE walk --
// but written as valid = FO_VALID_SKIPPED.  A row that completes valid lowers selected to its rank.  Whether a row runs
// is all SELECT decides: a completed row equals the BATCH kernels' row.
// tid / block_dim are read in the __global__ function, where the compiler knows their range from the launch bounds.
template <uint32_t MASK, bool STATS, bool UNI, bool TIES, bool BATCH, bool CORR = false, bool SELECT = false>
__device__ __forceinline__ void sweep_body(const MetricKArgs& k, const SweepShape shape, const BatchView& bv,
                                           const int tid, const int block_dim, const SelectView& sv = SelectView{}) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  // the one-warp shape is launched with 32 threads: warp index, team size and lane are compile-time facts there (the
  // queue addresses become immediates instead of being re-derived from %tid wherever registers are short)
  const int nthr = UNI ? 32 : block_dim;
  const int lane = UNI ? tid : (tid & 31), wib = UNI ? 0 : (tid >> 5), W = UNI ? 1 : (nthr >> 5);
  const int T = k.T;
  const SweepSmem w = sweep_smem(smem_raw, T, UNI ? 1 : W, UNI, TIES);
  uint32_t* const q_near = w.q_near + wib * kSwQueue;
  uint32_t* const q_cp = w.q_cp + wib * kSwQueue;
  uint32_t* const q_tie = w.q_tie + wib * kSwQueue;
  const uint32_t mm = MASK ? MASK : k.mmask;
  const bool do_cp = mm & FO_M_CP, do_dce = mm & FO_M_DCE, do_hr = mm & FO_M_HR, do_be = mm & FO_M_BE,
             do_ttc = mm & FO_M_TTC;
  const unsigned lt_mask = (1u << lane) - 1u;
  float rE = sqrtf(k.veh.hEx * k.veh.hEx + k.veh.hEy * k.veh.hEy);   // ego circumradius (batched: per trajectory)
  const float cmax = fmaxf(0.0f, fmaxf(k.hc.rs_side, k.hc.rs_rear));
  int Ap = k.tab.Ap;
  const auto soff = [&](const void* q) { return (uint32_t)(reinterpret_cast<const unsigned char*>(q) - smem_raw); };
  const BeView bev{soff(w.egoA), soff(w.egoB), soff(w.dist), soff(w.inv), soff(w.seg)};
  // batched: the trajectory's problem's s3 section, set per trajectory
  const float4* s3 = (CORR && !BATCH) ? agent_corr_view(k.tab.s0, k.A, k.Tp) : nullptr;
  BeConst bek = be_const(k);                       // batched: the table and its stride are set per trajectory
  // lane -> (agent within the lane group, time slice); every (warp, slice) owns a contiguous range of steps
  const int lg = shape.lg_agents;
  const int group = 1 << lg;                      // agents per warp pass
  const int la = lane & (group - 1), ls = lane >> lg;
  const int n_slices = W * (32 >> lg);
  const int L = (T + n_slices - 1) / n_slices;    // steps per slice
  const int s_lo = (wib * (32 >> lg) + ls) * L;
  const int s_hi = min(T, s_lo + L);
  unsigned long long st_dense = 0, st_obb = 0, st_lr = 0, st_cp = 0, st_be = 0, st_probe = 0, st_win = 0, st_wkeep = 0;
  unsigned long long st_node = 0, st_path = 0;

  // Trajectories are claimed from a device counter (their cost varies several-fold with the number of near agents and
  // braking pairs); the claim for the next one is issued here and read at the bottom, so its latency is hidden.  A batch
  // looks up the problem of the claimed trajectory in the same place.
  // select: [2] the next claim's rank, [3] skip the claimed row, [4] stop the row in progress (a slot of its own: no
  // barrier separates the reads of [3] from the first write of [4])
  __shared__ int s_claim[BATCH ? (SELECT ? 5 : 2) : 1];   // next trajectory (and, batched, its problem)
  int& s_next = s_claim[0];
  // batched: the ego vehicle of the current trajectory's problem, read where used (held in registers it would spill)
  __shared__ EgoConst s_veh;
  const EgoConst& veh = BATCH ? s_veh : k.veh;
  int p = (BATCH && !SELECT) ? batch_find(bv, blockIdx.x) : 0;
  int rank = 0;
  if constexpr (SELECT) {
    const int2 q = select_find(sv, blockIdx.x);
    p = q.x; rank = q.y;
  }
  for (int n = blockIdx.x; n < k.N;) {
    AgentTableView btab;
    int row = n, bA = 0, bTp = 0, b_group = 1, b_la = 0, b_slo = 0, b_shi = 0;
    int32_t* sel = nullptr;                          // select: the problem's entry of sv.selected
    if constexpr (BATCH) {
      const BatchProb bp = bv.prob[p];
      row = bp.row0 + (SELECT ? rank : n - bp.first);
      if constexpr (SELECT) sel = sv.selected + __ldg(sv.out + p);
      bA = bp.A; bTp = bp.Tp;
      btab.t0 = bp.t0; btab.tv = bp.tv; btab.aw = bp.aw; btab.avw = bp.avw;
      btab.s0 = bp.s0; btab.s1 = bp.s1; btab.s2 = bp.s2; btab.prm = bp.prm;
      btab.Ap = Ap = bp.Ap;
      bek.s0 = bp.s0;                                // BE bisections read the agent-major states
      bek.Tp = bTp;
      b_group = 1 << bp.lg;                          // lane map of the problem's lane grouping, as above
      b_la = lane & (b_group - 1);
      const int bL = (T + W * (32 >> bp.lg) - 1) / (W * (32 >> bp.lg));
      b_slo = (wib * (32 >> bp.lg) + (lane >> bp.lg)) * bL;
      b_shi = min(T, b_slo + bL);
      if constexpr (CORR) s3 = bp.s3;
    }
    // references into the kernel parameters when not batched: their uses stay constant-bank operands
    const AgentTableView& tab = BATCH ? btab : k.tab;
    const int& A = BATCH ? bA : k.A;
    const int& Tp = BATCH ? bTp : k.Tp;
    const auto drain_ties = [&](const uint32_t* src, int cnt, int a0, int lane, uint32_t rmin) {
      if constexpr (BATCH)
        return sw_drain_ties_batch(tab.t0, tab.prm, tab.s1, Ap, Tp, veh.wb, veh.hEx, veh.hEy, w.egoA, w.egoB, w.colfirst,
                                   src, cnt, a0, lane, rmin);
      else
        return sw_drain_ties(k, w.egoA, w.egoB, w.colfirst, src, cnt, a0, lane, rmin);
    };
    // ---- stage the ego trajectory (whole team) ---------------------------------------------------
    const float* eg = k.ego + (size_t)row * T * 5;
    __syncthreads();                                   // previous trajectory fully consumed
    if (tid < 8) w.scal[tid] = 0u;
    if constexpr (BATCH) {
      if (tid < (int)(sizeof(EgoConst) / 4))
        reinterpret_cast<float*>(&s_veh)[tid] = __ldg(reinterpret_cast<const float*>(&bv.prob[p].veh) + tid);
    }
    if (tid == 0) {
      s_next = k.claim ? (int)(gridDim.x + atomicAdd(k.claim, 1u)) : n + (int)gridDim.x;
      if constexpr (SELECT) {
        if (s_next < k.N) {
          const int2 q = select_find(sv, s_next);
          s_claim[1] = q.x; s_claim[2] = q.y;
        }
        s_claim[3] = ld_relaxed(sel) < rank;
        s_claim[4] = 0;
      } else if constexpr (BATCH) {
        s_claim[1] = s_next < k.N ? batch_find(bv, s_next) : 0;
      }
    }
    __syncthreads();
    // select: a row ranked after its problem's valid row so far is written as skipped, not staged
    const auto skip_row = [&]() {
      if (tid == 0) k.valid[row] = FO_VALID_SKIPPED;
      n = s_next;
      p = s_claim[1];
      rank = s_claim[2];
    };
    if constexpr (SELECT) {
      if (s_claim[3]) { skip_row(); continue; }
    }
    if constexpr (BATCH) rE = sqrtf(veh.hEx * veh.hEx + veh.hEy * veh.hEy);
    {
      float amin = 0.0f;
      for (int i = tid; i < T; i += nthr) {
        float x = __ldg(eg + i * 5 + 0), y = __ldg(eg + i * 5 + 1), th = __ldg(eg + i * 5 + 2);
        float v = __ldg(eg + i * 5 + 3);
        amin = fminf(amin, __ldg(eg + i * 5 + 4));
        float sn, cs;
        sincosf(th, &sn, &cs);
        w.egoA[i] = make_float4(x, y, cs, sn);
        w.egoB[i] = make_float2(th, v);
      }
      if (do_be && amin < 0.0f) atomicMax(&w.scal[0], __float_as_uint(-amin));   // |min(min a, 0)|, be.py:68
    }
    if (UNI) {                                         // boxes of the ego over windows of kWinSteps steps
      __syncthreads();
      if (tid * kWinSteps < T) {
        float xl = 1e30f, xh = -1e30f, yl = 1e30f, yh = -1e30f, vm = 0.0f;
#pragma unroll 1
        for (int i = tid * kWinSteps; i < min(T, (tid + 1) * kWinSteps); ++i) {
          const float4 EA = w.egoA[i];
          const float cx = fmaf(veh.wb, EA.z, EA.x), cy = fmaf(veh.wb, EA.w, EA.y); // box centre (dce.py:57-60)
          xl = fminf(xl, fminf(EA.x, cx)); xh = fmaxf(xh, fmaxf(EA.x, cx));
          yl = fminf(yl, fminf(EA.y, cy)); yh = fmaxf(yh, fmaxf(EA.y, cy));
          vm = fmaxf(vm, fabsf(w.egoB[i].y));
        }
        w.ew[tid] = make_float4(xl, xh, yl, yh);
        w.evw[tid] = vm;
      }
    }

    uint32_t rmin = 0xffffffu;                       // warp-uniform running min of round(d * 1000)
    float zb_e = -CUDART_INF_F, zb_o = -CUDART_INF_F; // warp-uniform running maxima of the harm logits
    uint32_t acc_col = 0xffffffffu;
    float acc_ze = -CUDART_INF_F, acc_zo = -CUDART_INF_F;
    float acc_er = 0.0f, acc_or = 0.0f, acc_cp = 0.0f, acc_hwc = 0.0f;
    float btn_all = 0.0f, rcd_all = 0.0f;
    uint32_t flags = 0;
    bool be_ready = false;

    for (int a0 = 0; a0 < A; a0 += kSwTile) {
      const int nAt = min(kSwTile, A - a0);
      for (int j = tid; j < nAt; j += nthr) { w.pairkey[j] = 0ull; w.colfirst[j] = 0xffffffffu; }
      if constexpr (SELECT) {                          // before the tile's sweep and queued drains
        if (tid == 0) s_claim[4] = ld_relaxed(sel) < rank;
      }
      __syncthreads();                                 // ego staged, pair arrays cleared
      if constexpr (SELECT) {
        if (s_claim[4]) break;
      }
      int qn = 0, qc = 0, qt = 0;
      // per-lane bound state of the current lane group (refreshed after every drain)
      float lim0 = 0.0f, lim2 = 0.0f, thr2 = CUDART_INF_F;
      HarmLin hl{};
      bool is_m1 = false;

      // distance >= |centres| - rE - rO: the exact box distance is needed only while that bound can still lower
      // the running minimum (+2 units of the 1 mm rounding grid)
      auto upd_lim = [&]() {
        const float lim = lim0 + (float)(rmin + 2u) * 0.001f;
        lim2 = lim * lim;
      };
      // LR4S logit <= ks dv + kc + cmax: the impact-angle class is needed only while that can still raise a
      // running maximum, i.e. dv^2 > thr2 (slightly lowered so float rounding can only add work)
      auto upd_thr = [&]() {
        float t2 = CUDART_INF_F;
        if (is_m1) {
          const float ze_m = fmaxf(zb_e, acc_ze), zo_m = fmaxf(zb_o, acc_zo);
          const float te = (hl.kse > 1e-30f) ? (ze_m - cmax - hl.kce) * rcp_approx(hl.kse)
                                             : ((hl.kce + cmax > ze_m) ? -1.0f : CUDART_INF_F);
          const float to = (hl.kso > 1e-30f) ? (zo_m - cmax - hl.kco) * rcp_approx(hl.kso)
                                             : ((hl.kco + cmax > zo_m) ? -1.0f : CUDART_INF_F);
          const float tm = fminf(te, to);
          t2 = (tm > 0.0f) ? tm * tm * 0.99999f : -1.0f;
        }
        thr2 = t2;
      };

      // ---- drains: up to 32 queued items at a time ------------------------------------------------------
      auto drain_near = [&](const uint32_t* src, int cnt) {
        uint32_t item = 0;
        if (lane < cnt) item = src[lane];
        __syncwarp();
        uint32_t r = 0xffffffu;
        bool tie = false;
        if (lane < cnt) {
          const int ial = (int)((item >> 8) & 0xffffu), ii = (int)(item & 0xffu);
          const int a = a0 + ial;
          const float4 s0 = __ldg(&tab.t0[(size_t)ii * Ap + a]);
          const float4 EA = w.egoA[ii];
          const float c = fmaf(EA.z, s0.z, EA.w * s0.w), s = fmaf(s0.w, EA.z, -s0.z * EA.w);
          const float dxr = s0.x - EA.x, dyr = s0.y - EA.y;
          if (item & 0x40000000u) {            // exact oriented-box distance, np.round(d, 3) (dce.py:75-79)
            const int4 pa = __ldg(reinterpret_cast<const int4*>(tab.prm + a));
            const float d = ego_box_dist(dxr, dyr, EA, c, s, veh, __int_as_float(pa.z), __int_as_float(pa.w));
            r = (uint32_t)__float2int_rn(fminf(d, 8000.0f) * 1000.0f);
            // np.round(d, 3) next to a x.xxx5 boundary: a candidate for the minimum is queued for a float64
            // re-rounding (rmin only falls, so "r <= rmin + 2" is a superset of the candidates of the final minimum);
            // until then it bounds the minimum from above with r + 1 -- min_dce, wttc and the dce / ttc threshold
            // clauses are then the float64 reference's except for distances within 1e-12 of a boundary
            if (TIES) {
              tie = near_rounding_boundary(d) && r <= rmin + 2u;
              if (tie) ++r;
            }
            if (r == 0u && !tie) atomicMin(&w.colfirst[ial], (uint32_t)ii);
            if (STATS) ++st_obb;
          }
          if (item & 0x80000000u) {            // LR4S logits with the impact-angle class (protected agents)
            const int4 pb = __ldg(reinterpret_cast<const int4*>(tab.prm + a) + 1);
            const float4 s1 = __ldg(&tab.s1[(size_t)a * Tp + ii]);
            const float2 EB = w.egoB[ii];
            const float dv2 = fmaxf(fmaf(EB.y, EB.y, s1.y * s1.y) - 2.0f * EB.y * s1.y * c, 0.0f);
            const float dv = dv2 * rsqrtf(fmaxf(dv2, 1e-30f));
            float ze, zo;
            sw_harm_logits(k, 1, __int_as_float(pb.y), __int_as_float(pb.z), dv, dxr, dyr, EB.x, s1.x, ze, zo);
            acc_ze = fmaxf(acc_ze, ze);
            acc_zo = fmaxf(acc_zo, zo);
            if (STATS) ++st_lr;
          }
        }
        rmin = min(rmin, __reduce_min_sync(kFull, r));
        if (TIES) {
          const unsigned tb = __ballot_sync(kFull, tie);
          if (tb) {
            if (tie) q_tie[qt + __popc(tb & lt_mask)] = (item & 0xffffu) | (min(r - 1u, 0xffffu) << 16);   // r was bumped above
            qt += __popc(tb);
            __syncwarp();
            if (qt >= 32) { qt -= 32; rmin = min(rmin, drain_ties(q_tie + qt, 32, a0, lane, rmin)); }
          }
        }
        zb_e = fmaxf(zb_e, warp_max_signed(acc_ze));
        zb_o = fmaxf(zb_o, warp_max_signed(acc_zo));
        upd_lim();
        upd_thr();
      };
      auto drain_cp = [&](const uint32_t* src, int cnt) {
        uint32_t item = 0;
        if (lane < cnt) item = src[lane];
        __syncwarp();
        if (lane < cnt) {
          const int ial = (int)(item >> 8), ii = (int)(item & 0xffu), t = ii - 1;
          const int a = a0 + ial;
          const AgentParams P = load_params(tab.prm + a);
          const size_t idx = (size_t)a * Tp + ii;
          const float4 s0i = __ldg(&tab.s0[idx]);
          const float4 s1i = __ldg(&tab.s1[idx]);
          const float4 Ei = w.egoA[ii];
          float cp;
          if constexpr (CORR) {
            cp = cp_bvn_boxes(s1i.z - Ei.x, s1i.w - Ei.y, P.hlb * s0i.z, P.hlb * s0i.w, veh.L3 * Ei.z, veh.L3 * Ei.w,
                              __ldg(&s3[idx]), veh.L6, veh.W2);
            acc_cp = nan_maxf(acc_cp, cp);
          } else {
            const float2 s2i = __ldg(&tab.s2[idx]);
            cp = cp_gauss_boxes(s1i.z - Ei.x, s1i.w - Ei.y, P.hlb * s0i.z, P.hlb * s0i.w, veh.L3 * Ei.z, veh.L3 * Ei.w,
                                s2i, veh.L6, veh.W2);
            acc_cp = fmaxf(acc_cp, cp);
          }
          if (do_hr) {                       // risk[t] = harm[t] * cp[t], cp[t] = CP of step t+1 (hr.py:78-79)
            const float4 s0t = __ldg(&tab.s0[idx - 1]);
            const float4 s1t = __ldg(&tab.s1[idx - 1]);
            const float4 Et = w.egoA[t];
            const float2 EtB = w.egoB[t];
            const float ct = fmaf(Et.z, s0t.z, Et.w * s0t.w);
            const float dv = sqrtf(fmaxf(fmaf(EtB.y, EtB.y, s1t.y * s1t.y) - 2.0f * EtB.y * s1t.y * ct, 0.0f));
            float ze, zo;
            sw_harm_logits(k, P.model, P.ke, P.ko, dv, s0t.x - Et.x, s0t.y - Et.y, EtB.x, s1t.x, ze, zo);
            acc_er = fmaxf(acc_er, sw_sigmoid(ze) * cp);
            acc_or = fmaxf(acc_or, sw_sigmoid(zo) * cp);
            if (cp > 0.01f)                  // candidates for obst_harm[argmax cp] (hr.py:81-84)
              atomicMax(&w.pairkey[ial], ((unsigned long long)__float_as_uint(cp) << 32) |
                                             ((unsigned long long)(0xffffu - (unsigned)t) << 16) | 1ull);
          }
          if (STATS) ++st_cp;
        }
        __syncwarp();
      };

      // ---- dense sweep: lane groups of `group` agents x the steps of this lane's slice ------------------
      // flush (warp-uniform): no lane has work; drain what is left in the two queues through the same inlined drains
      auto run_group = [&](const int al, const bool alive, const int i_lo, const int i_hi, const bool flush) {
        const int a = a0 + al;
        AgentParams P;
        P.n_states = 0; P.model = 2; P.hl = P.hw = P.hlb = P.ke = P.ko = P.pad = 0.0f;
        if (alive) P = load_params(tab.prm + a);
        const int nS = min(P.n_states, i_hi);             // this lane evaluates steps [i_lo, nS)
        const int nH = min(nS, T - 1);                    // harm is evaluated at steps < min(T-1, n_states)
        const int n_it = flush ? 1 : (int)__reduce_max_sync(kFull, (unsigned)max(nS - i_lo, 0));
        const bool is_m0 = P.model == 0;
        is_m1 = P.model == 1;
        hl = harm_lin(k.hc, P.model, P.ke, P.ko);
        if (do_hr && alive && P.model == 2 && nH > i_lo) { acc_ze = CUDART_INF_F; acc_zo = CUDART_INF_F; }
        lim0 = rE + P.pad;
        upd_lim();
        upd_thr();
        const float hlb2 = P.hlb * P.hlb, hlbm2 = -2.0f * P.hlb;
        const uint32_t item0 = (uint32_t)al << 8;
        // time-major table, agents padded to a multiple of 32: the agent index is always in bounds; rows are only
        // read for steps the agent has (i < n_states <= t_stride)
        // one 32-bit element offset into both time-major arrays (base pointers are kernel arguments: uniform registers)
        uint32_t toff = (uint32_t)(i_lo * Ap + a);
        float pxp = 0.0f, pyp = 0.0f;                      // position at i-1 (collision_probability.py:52)
        if (do_cp && i_lo >= 1 && i_lo < nS) { const float4 sp = __ldg(tab.t0 + (toff - (uint32_t)Ap)); pxp = sp.x; pyp = sp.y; }
        float acc_dv2 = -1.0f;                             // unprotected agents: max_t logit = ks sqrt(max_t dv^2) + kc
        int i = i_lo;
#pragma unroll kSwUnroll
        for (int r = 0; r < n_it; ++r, ++i, toff += (uint32_t)Ap) {
          const bool live = i < nS;
          float4 s0 = make_float4(0.0f, 0.0f, 1.0f, 0.0f);
          float va = 0.0f;
          if (live) { s0 = __ldg(tab.t0 + toff); va = __ldg(tab.tv + toff); }
          const int ie = min(i, T - 1);
          const float4 EA = w.egoA[ie];
          const float ve = w.egoB[ie].y;
          bool need_obb = false, need_lr = false, ingate = false;
          if (do_dce) {
            const float2 d = fma2(f2(-veh.wb), make_float2(EA.z, EA.w),
                                  add2(make_float2(s0.x, s0.y), make_float2(-EA.x, -EA.y)));   // centre to centre
            need_obb = live & (fmaf(d.x, d.x, d.y * d.y) < lim2);
          }
          if (do_hr) {
            const float c = fmaf(EA.z, s0.z, EA.w * s0.w);                            // cos(yaw - theta)
            const float dv2 = fmaxf(fmaf(-2.0f * ve * va, c, fmaf(ve, ve, va * va)), 0.0f);
            const bool live_h = i < nH;
            if (live_h) acc_dv2 = fmaxf(acc_dv2, dv2);
            need_lr = live_h & (dv2 > thr2);
          }
          if (do_cp) {                                                                // 5 m gate, collision_probability.py:61-78
            // min over the points p, p +- h u of |. - e|^2  =  |m|^2 + min(0, h^2 - 2 h |m.u|),  m = p_{i-1} - e_i
            const float2 m = add2(make_float2(pxp, pyp), make_float2(-EA.x, -EA.y));
            const float mx = m.x, my = m.y;
            const float mu = fmaf(mx, s0.z, my * s0.w);
            const float dmin = fmaf(mx, mx, my * my) + fminf(fmaf(hlbm2, fabsf(mu), hlb2), 0.0f);
            ingate = live & (i >= 1) & (dmin <= 25.0f);
          }
          pxp = s0.x; pyp = s0.y;
          const bool near = need_obb | need_lr;
          unsigned b = __ballot_sync(kFull, near);
          if (b || flush) {
            if (near) q_near[qn + __popc(b & lt_mask)] = item0 | (uint32_t)i | (need_obb ? 0x40000000u : 0u) |
                                                       (need_lr ? 0x80000000u : 0u);
            qn += __popc(b);
            __syncwarp();
            if (qn >= 32 || (flush && qn > 0)) { const int c = min(qn, 32); qn -= c; drain_near(q_near + qn, c); }
          }
          b = __ballot_sync(kFull, ingate);
          if (b || flush) {
            if (ingate) q_cp[qc + __popc(b & lt_mask)] = item0 | (uint32_t)i;
            qc += __popc(b);
            __syncwarp();
            if (qc >= 32 || (flush && qc > 0)) { const int c = min(qc, 32); qc -= c; drain_cp(q_cp + qc, c); }
          }
          if (STATS) st_dense += live;
        }
        if (do_hr && is_m0 && acc_dv2 >= 0.0f) {
          const float dvm = acc_dv2 * rsqrtf(fmaxf(acc_dv2, 1e-30f));
          acc_ze = fmaxf(acc_ze, fmaf(hl.kse, dvm, hl.kce));
          acc_zo = fmaxf(acc_zo, fmaf(hl.kso, dvm, hl.kco));
        }
        if (do_hr) {
          zb_e = fmaxf(zb_e, warp_max_signed(acc_ze));
          zb_o = fmaxf(zb_o, warp_max_signed(acc_zo));
        }
      };

      if (UNI) {
        // Window filter (one warp, >= 32 agents per pass).  lane = agent: every window of kWinSteps steps is tested with
        // the boxes of the two paths over that window -- gap between the boxes against the reach of the distance and
        // 5 m-gate bounds, sum of the top speeds against the logit bound -- and only the (agent, window) items that can
        // still change a result are queued; full warps of items then run the per-step loop, lane = item.
        int sub = 0, wi = 0, qw = 0, f_nS = 0, f_nH = 0, f_nW = 0;
        float f_reach2 = 0.0f, f_thr2 = -1.0f;
        // cursors into the window tables; re-derived whenever the per-agent state is (they do not live across run_group)
        const float4* awp = tab.aw;
        const float* avp = tab.avw;
        const float4* ewp = w.ew;
        const float* evp = w.evw;
        bool more = nAt > 0, stale = true, flushed = false;
        for (;;) {
          while (more && qw < 32) {
            const int al = sub + lane;
            if (stale) {
              AgentParams P;
              P.n_states = 0; P.model = 2; P.hl = P.hw = P.hlb = P.ke = P.ko = P.pad = 0.0f;
              if (al < nAt) P = load_params(tab.prm + a0 + al);
              f_nS = min(P.n_states, T);
              f_nH = min(f_nS, T - 1);
              f_nW = (int)__reduce_max_sync(kFull, (unsigned)((f_nS + kWinSteps - 1) / kWinSteps));
              // reach of the per-step distance bounds (+1 mm: the per-step code rounds its differences differently)
              const float lim = do_dce ? rE + P.pad + (float)(rmin + 2u) * 0.001f + 0.001f : 0.0f;
              const float gate = do_cp ? 5.001f + P.hlb : 0.0f;
              const float reach = fmaxf(lim, gate);
              f_reach2 = reach * reach;
              float t2 = CUDART_INF_F;                      // harm logit <= ks (|v_e| + |v_a|) + kc (+ cmax)
              if (do_hr && P.model != 2) {
                const float cm = P.model == 0 ? 0.0f : cmax;
                const HarmLin h = harm_lin(k.hc, P.model, P.ke, P.ko);
                const float fce = h.kce + cm, fco = h.kco + cm;
                const float ze_m = fmaxf(zb_e, acc_ze), zo_m = fmaxf(zb_o, acc_zo);
                const float te = (h.kse > 1e-30f) ? (ze_m - fce) * rcp_approx(h.kse) : ((fce > ze_m) ? -1.0f : CUDART_INF_F);
                const float to = (h.kso > 1e-30f) ? (zo_m - fco) * rcp_approx(h.kso) : ((fco > zo_m) ? -1.0f : CUDART_INF_F);
                const float tm = fminf(te, to);
                t2 = (tm > 0.0f) ? tm * tm * 0.99999f : -1.0f;
              }
              f_thr2 = t2;
              awp = tab.aw + (size_t)wi * Ap + a0 + al;
              avp = tab.avw + (size_t)wi * Ap + a0 + al;
              ewp = w.ew + wi;
              evp = w.evw + wi;
              stale = false;
            }
            if (wi < f_nW) {
              const float4 B = __ldg(awp);
              const float av = __ldg(avp);
              const float4 E = *ewp;
              const float dvu = *evp + av;
              awp += Ap; avp += Ap; ++ewp; ++evp;
              const float gx = fmaxf(fmaxf(B.x - E.y, E.x - B.y), 0.0f), gy = fmaxf(fmaxf(B.z - E.w, E.z - B.w), 0.0f);
              const int i0 = wi * kWinSteps;
              const bool keep = (i0 < f_nS) & ((fmaf(gx, gx, gy * gy) < f_reach2) | ((i0 < f_nH) & (dvu * dvu > f_thr2)));
              const unsigned b = __ballot_sync(kFull, keep);
              if (keep) w.q_win[qw + __popc(b & lt_mask)] = (uint16_t)((al << 8) | wi);
              qw += __popc(b);
              if (STATS) { st_win += (i0 < f_nS); st_wkeep += keep; }
            }
            if (++wi >= f_nW) { wi = 0; sub += 32; more = sub < nAt; stale = true; }
          }
          bool flush = false;
          if (qw == 0) {                                // all items done: one more pass drains the two queues
            if (flushed) break;
            flushed = flush = true;
          }
          const int cnt = min(qw, 32);
          qw -= cnt;
          __syncwarp();
          const uint32_t it = (lane < cnt) ? (uint32_t)w.q_win[qw + lane] : 0u;
          __syncwarp();
          const int i0 = (int)(it & 0xffu) * kWinSteps;
          run_group((int)(it >> 8), lane < cnt, i0, min(T, i0 + kWinSteps), flush);
          stale = true;
        }
      } else {
        if constexpr (BATCH) {
          for (int sub = 0; sub < nAt; sub += b_group) run_group(sub + b_la, sub + b_la < nAt, b_slo, b_shi, false);
        } else {
          for (int sub = 0; sub < nAt; sub += group) run_group(sub + la, sub + la < nAt, s_lo, s_hi, false);
        }
      }
      // ---- pool what is left in the per-warp queues across the team and drain it cooperatively --------------
      is_m1 = false;
      if (TIES && UNI && qt > 0) { rmin = min(rmin, drain_ties(q_tie, qt, a0, lane, rmin)); qt = 0; }
      if (!UNI) {
        unsigned base_n = 0, base_c = 0;
        if (lane == 0) {
          if (qn > 0) base_n = atomicAdd(&w.scal[2], (unsigned)qn);
          if (qc > 0) base_c = atomicAdd(&w.scal[3], (unsigned)qc);
        }
        base_n = __shfl_sync(kFull, base_n, 0);
        base_c = __shfl_sync(kFull, base_c, 0);
        if (lane < qn) w.pool_near[base_n + lane] = q_near[lane];
        if (lane < qc) w.pool_cp[base_c + lane] = q_cp[lane];
        __syncthreads();
        const int tot_n = (int)w.scal[2], tot_c = (int)w.scal[3];
        for (int c = wib * 32; c < tot_n; c += 32 * W) drain_near(w.pool_near + c, min(32, tot_n - c));
        for (int c = wib * 32; c < tot_c; c += 32 * W) drain_cp(w.pool_cp + c, min(32, tot_c - c));
        while (TIES && qt > 0) { const int c = min(qt, 32); qt -= c; rmin = min(rmin, drain_ties(q_tie + qt, c, a0, lane, rmin)); }
      }
      __syncthreads();                                 // pairkey / colfirst of the tile complete
      if (tid == 0) { w.scal[2] = 0u; w.scal[3] = 0u; }

      // ---- tile epilogue: harm_with_cp, wttc, BE list -----------------------------------------------------------
      for (int j = tid; j < nAt; j += nthr) {
        const unsigned long long key = w.pairkey[j];
        const uint32_t cf = w.colfirst[j];
        if (key != 0ull) {
          const int t = (int)(0xffffu - (unsigned)((key >> 16) & 0xffffu));
          const int a = a0 + j;
          const AgentParams P = load_params(tab.prm + a);
          const size_t idx = (size_t)a * Tp + t;
          const float4 s0t = __ldg(&tab.s0[idx]);
          const float4 s1t = __ldg(&tab.s1[idx]);
          const float4 Et = w.egoA[t];
          const float2 EtB = w.egoB[t];
          const float ct = fmaf(Et.z, s0t.z, Et.w * s0t.w);
          const float dv = sqrtf(fmaxf(fmaf(EtB.y, EtB.y, s1t.y * s1t.y) - 2.0f * EtB.y * s1t.y * ct, 0.0f));
          float ze, zo;
          sw_harm_logits(k, P.model, P.ke, P.ko, dv, s0t.x - Et.x, s0t.y - Et.y, EtB.x, s1t.x, ze, zo);
          acc_hwc = fmaxf(acc_hwc, sw_sigmoid(zo));
        }
        if (do_ttc) acc_col = min(acc_col, cf);
        if (do_be && do_ttc && cf != 0xffffffffu && cf > 0u)           // be.py:49-50
          w.be_list[atomicAdd(&w.scal[1], 1u)] = (uint16_t)j;
      }
      if (do_be && do_ttc) {
        if constexpr (SELECT) {                        // before the BE walk
          if (tid == 0) s_claim[4] = ld_relaxed(sel) < rank;
        }
        __syncthreads();                               // BE list complete
        if constexpr (SELECT) {
          if (s_claim[4]) break;
        }
        const int n_be = (int)w.scal[1];
        if (n_be > 0) {
          if (!be_ready) {
            if (wib == 0) be_prepare<true>(bev, T, lane);
            __syncthreads();
            be_ready = true;
          }
          const float be_lo0 = rintf(__uint_as_float(w.scal[0]) * 100.0f) / 100.0f;   // be.py:68
          BeConst bk = bek;
          if constexpr (BATCH) { bk.wb = veh.wb; bk.hEx = veh.hEx; bk.hEy = veh.hEy; }
          if constexpr (UNI) {
            // one walk over the bisection tree of the tile's pairs (be_walk); only the maximum over the pairs is kept,
            // and after a range error no further pair matters (the outputs are NaN, the trajectory invalid)
            if (!(flags & FO_F_BE_RANGE)) {
              bk.s0 += (size_t)a0 * bk.Tp;               // the tile's first agent
              const BeWalk be = be_walk<STATS>(bk, tab.prm + a0, bev, soff(w.be_list), n_be, be_lo0, rcd_all, lane);
              if (be.range) flags |= FO_F_BE_RANGE;
              rcd_all = be.rcd;
              btn_all = fmaxf(btn_all, rcd_all / veh.a_max);   // division is monotone: the maximum of the quotients
              if (STATS && lane == 0) { st_be += n_be; st_probe += be.tests; st_node += be.nodes; st_path += be.chunks; }
            }
          } else {
            // team shape: bisections dealt round-robin to the warps; a bisection stops as soon as its bracket lies
            // below the running maximum (be_bisect), and a range error makes every further one moot
            for (int q = wib; q < n_be && !(flags & FO_F_BE_RANGE); q += W) {
              const int a = a0 + (int)w.be_list[q];
              const int4 pa = __ldg(reinterpret_cast<const int4*>(tab.prm + a));
              const float2 be = be_bisect<true>(bk, bev, a, pa.x, __int_as_float(pa.z), __int_as_float(pa.w), be_lo0,
                                                lane, rcd_all);
              const float rcd = be.x;
              if (rcd != rcd) flags |= FO_F_BE_RANGE;    // NaN: the re-timed path overruns the planned one
              rcd_all = fmaxf(rcd_all, rcd);
              btn_all = fmaxf(btn_all, rcd / veh.a_max);
              if (STATS && lane == 0) { st_be += 1; st_probe += (unsigned)__float_as_int(be.y); }
            }
          }
        }
        __syncthreads();                               // list consumed before the next tile refills it
        if (tid == 0) w.scal[1] = 0u;
      }
    }  // agent tiles
    if constexpr (SELECT) {
      if (s_claim[4]) { skip_row(); continue; }
    }

    // ---- per-trajectory reduction (warp, then team) and threshold mask (metric.py:50-98) --------------------
    {
      const float er = umaxf(acc_er), orr = umaxf(acc_or), cpm = umaxf(acc_cp), hwc = umaxf(acc_hwc);
      const float ze = warp_max_signed(acc_ze), zo = warp_max_signed(acc_zo);
      const uint32_t col = __reduce_min_sync(kFull, acc_col);
      const uint32_t fl = __reduce_or_sync(kFull, flags);
      if (lane == 0) {
        float* r = w.red + wib * 16;
        r[0] = er; r[1] = orr; r[2] = cpm; r[3] = hwc; r[4] = ze; r[5] = zo;
        r[6] = __uint_as_float(rmin); r[7] = __uint_as_float(col); r[8] = __uint_as_float(fl);
        r[9] = btn_all; r[10] = rcd_all;
      }
    }
    __syncthreads();
    if (tid == 0) {
      float er = 0.0f, orr = 0.0f, cpm = 0.0f, hwc_all = 0.0f, ze = -CUDART_INF_F, zo = -CUDART_INF_F, btn = 0.0f, rcd = 0.0f;
      uint32_t rmin_t = 0xffffffu, col = 0xffffffffu, fl = 0u;
      for (int q = 0; q < W; ++q) {
        const float* r = w.red + q * 16;
        er = fmaxf(er, r[0]); orr = fmaxf(orr, r[1]); cpm = CORR ? nan_maxf(cpm, r[2]) : fmaxf(cpm, r[2]);
        hwc_all = fmaxf(hwc_all, r[3]);
        ze = fmaxf(ze, r[4]); zo = fmaxf(zo, r[5]);
        rmin_t = min(rmin_t, __float_as_uint(r[6])); col = min(col, __float_as_uint(r[7])); fl |= __float_as_uint(r[8]);
        btn = fmaxf(btn, r[9]); rcd = fmaxf(rcd, r[10]);
      }
      const float eh = sw_sigmoid(ze), oh = sw_sigmoid(zo);   // logistic is monotone: max harm = logistic(max logit)
      const bool has_agents = A > 0 && mm != 0;
      const bool has_col = col != 0xffffffffu;
      bool ok = true;
      if (has_agents) {
        if (do_be && (k.tmask & FO_T_BE) && (double)btn > k.thr_be) ok = false;
        if (do_hr && (k.tmask & FO_T_HARM) && (double)hwc_all > k.thr_harm) ok = false;
        if (do_hr && (k.tmask & FO_T_RISK) && (double)orr > k.thr_risk) ok = false;
        if (do_hr && (k.tmask & FO_T_CP) && (double)cpm > k.thr_cp) ok = false;
        if (do_ttc && (k.tmask & FO_T_TTC) && has_col && col < k.thr_ttc_col) ok = false;
        if (do_dce && (k.tmask & FO_T_DCE) && rmin_t != 0xffffffu && rmin_t < k.thr_dce_mm) ok = false;
        if (fl & FO_F_BE_RANGE) ok = false;
      }
      const float o6 = (rmin_t == 0xffffffu || !do_dce) ? CUDART_INF_F : mm_to_m(rmin_t);
      const float o7 = has_col ? step_to_s(col, k.dtd) : CUDART_INF_F;
      const float o8 = (fl & FO_F_BE_RANGE) ? CUDART_NAN_F : btn, o9 = (fl & FO_F_BE_RANGE) ? CUDART_NAN_F : rcd;
      // Fused result exchange of a sharded sweep: the same stores go to this rank's slice of every peer's gather buffer
      // (peer-mapped device memory, NVLink); p = -1 is the local copy.  Rows are 40 bytes: five 8-byte stores.
#pragma unroll 1
      for (int p = -1; p < k.n_peers; ++p) {
        const long long dl = p < 0 ? 0ll : k.peer_delta[p];
        reinterpret_cast<uint8_t*>(reinterpret_cast<char*>(k.valid) + dl)[row] = ok ? 1 : 0;
        if (k.flags) reinterpret_cast<uint32_t*>(reinterpret_cast<char*>(k.flags) + dl)[row] = fl;
        if (k.summary) {
          float2* sm = reinterpret_cast<float2*>(reinterpret_cast<char*>(k.summary) + dl) + (size_t)row * (FO_SUMMARY_K / 2);
          sm[0] = make_float2(er, orr);
          sm[1] = make_float2(do_hr ? eh : 0.0f, do_hr ? oh : 0.0f);
          sm[2] = make_float2(cpm, hwc_all);
          sm[3] = make_float2(o6, o7);
          sm[4] = make_float2(o8, o9);
        }
      }
      if constexpr (SELECT) {
        if (ok) atomicMin(sel, rank);
      }
    }
    n = s_next;
    if constexpr (BATCH) p = s_claim[1];
    if constexpr (SELECT) rank = s_claim[2];
  }
  if (STATS && k.stats) {
    auto wsum = [&](unsigned long long v) {
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
      return v;
    };
    const unsigned long long s6 = wsum(st_win), s7 = wsum(st_wkeep);
    const unsigned long long s0 = wsum(st_dense), s1 = wsum(st_obb), s2 = wsum(st_lr), s3 = wsum(st_cp);
    st_be = wsum(st_be); st_probe = wsum(st_probe); st_node = wsum(st_node); st_path = wsum(st_path);
    if (lane == 0) {
      atomicAdd(&k.stats[0], s0); atomicAdd(&k.stats[1], s1); atomicAdd(&k.stats[2], s2); atomicAdd(&k.stats[3], s3);
      atomicAdd(&k.stats[4], st_be); atomicAdd(&k.stats[5], st_probe);
      atomicAdd(&k.stats[6], s6); atomicAdd(&k.stats[7], s7);
      atomicAdd(&k.stats[8], st_node); atomicAdd(&k.stats[9], st_path);
    }
  }
}

template <uint32_t MASK, bool STATS, bool UNI, bool TIES>
__global__ void __launch_bounds__(kSwMaxWarps * 32, FO_SW_MINB)
fo_metric_sweep_kernel(const __grid_constant__ MetricKArgs k, const SweepShape shape) {
  sweep_body<MASK, STATS, UNI, TIES, false>(k, shape, BatchView{}, threadIdx.x, blockDim.x);
}

// Correlated tables (fo_metric_bundle_corr): the runtime metric mask, both shapes, with and without the tie path.
template <bool UNI, bool TIES>
__global__ void __launch_bounds__(kSwMaxWarps * 32, FO_SW_MINB)
fo_metric_sweep_corr_kernel(const __grid_constant__ MetricKArgs k, const SweepShape shape) {
  sweep_body<0u, false, UNI, TIES, false, true>(k, shape, BatchView{}, threadIdx.x, blockDim.x);
}

// Work counters on correlated tables (fo_metric_stats_corr): fo_metric_sweep_corr_kernel with the counters of
// fo_metric_sweep_kernel<0, true>.  They count geometric work and queue items only, so on the same geometry they equal
// the diagonal table's (DESIGN.md 5.13: where the team shape's warp order makes some of them vary, on both tables).
template <bool UNI, bool TIES>
__global__ void __launch_bounds__(kSwMaxWarps * 32, FO_SW_MINB)
fo_metric_sweep_corr_stats_kernel(const __grid_constant__ MetricKArgs k, const SweepShape shape) {
  sweep_body<0u, true, UNI, TIES, false, true>(k, shape, BatchView{}, threadIdx.x, blockDim.x);
}

// One shape class of a batch of independent problems (fo_metric_batch): k.N is the class's trajectory count, k.tab / k.A
// / k.Tp / k.veh and shape.lg_agents are unused -- every trajectory takes them from its problem.
template <uint32_t MASK, bool UNI, bool TIES>
__global__ void __launch_bounds__(kSwMaxWarps * 32, FO_SW_MINB)
fo_metric_batch_kernel(const __grid_constant__ MetricKArgs k, const SweepShape shape, const __grid_constant__ BatchView bv) {
  sweep_body<MASK, false, UNI, TIES, true>(k, shape, bv, threadIdx.x, blockDim.x);
}

// One shape class of the correlated problems of a batch (fo_metric_batch_corr): fo_metric_batch_kernel's problem lookup
// with fo_metric_sweep_corr_kernel's CP drain; every trajectory reads its problem's s3 section (BatchProb::s3).
template <bool UNI, bool TIES>
__global__ void __launch_bounds__(kSwMaxWarps * 32, FO_SW_MINB)
fo_metric_batch_corr_kernel(const __grid_constant__ MetricKArgs k, const SweepShape shape, const __grid_constant__ BatchView bv) {
  sweep_body<0u, false, UNI, TIES, true, true>(k, shape, bv, threadIdx.x, blockDim.x);
}

// One shape class of a batch for its problems' first valid rows (fo_metric_batch_select): fo_metric_batch_kernel<0> /
// fo_metric_batch_corr_kernel with rank-major claims and early exit.
template <bool UNI, bool TIES, bool CORR>
__global__ void __launch_bounds__(kSwMaxWarps * 32, FO_SW_MINB)
fo_metric_batch_select_kernel(const __grid_constant__ MetricKArgs k, const SweepShape shape,
                              const __grid_constant__ BatchView bv, const __grid_constant__ SelectView sv) {
  sweep_body<0u, false, UNI, TIES, true, CORR, true>(k, shape, bv, threadIdx.x, blockDim.x, sv);
}

// Team shape.  lg_agents: a warp holds min(32, next power of two >= A) agents, the remaining lanes are time slices.
// W: as many warps per trajectory as keeps the whole bundle resident in one wave (the latency of a bundle is its
// slowest trajectory), as long as every (warp, slice) still owns at least 4 steps.
int lane_group_log2(int A) {
  int lg = 0;
  while ((1 << lg) < A && lg < 5) ++lg;
  return lg;
}

// A batch takes N = its total trajectory count and A = the fewest agents of any problem (the most time slices per warp).
int pick_team_warps(int N, int T, int A, int num_sms) {
  const int slices_per_warp = 32 >> lane_group_log2(A);
  const int warp_slots = num_sms * 8 * FO_SW_MINB;               // registers per thread are capped for FO_SW_MINB 256-thread CTAs per SM
  int w = warp_slots / (N > 0 ? N : 1);
  const int max_w = T / (4 * slices_per_warp);
  if (w > max_w) w = max_w;
  if (w > kSwMaxWarps) w = kSwMaxWarps;
  if (w < 1) w = 1;
  const char* forced = getenv("FO_TEAM_WARPS");                  // measurement / test switch (DESIGN.md)
  if (forced) { int f = atoi(forced); if (f >= 1 && f <= kSwMaxWarps) w = f; }
  return w;
}

// Teams of W warps resident at once: the warp slots pick_team_warps shares out.
int resident_teams(int W, int num_sms) { return num_sms * 8 * FO_SW_MINB / (W > 0 ? W : 1); }

// Claim counters: one 4-byte slot per launch, zeroed in-stream before the kernel.  Eager launches rotate through a ring
// (a slot is reused kClaimRing launches later); a launch recorded into a CUDA graph keeps a slot of its own for the
// life of the process, because the graph may be replayed while later eager launches are in flight.  When the graph
// slots run out the kernel falls back to static striding (claim == NULL).
constexpr int kClaimRing = 1024, kClaimGraph = 3072;
unsigned int* claim_slot(cudaStream_t st) {
  static std::mutex mu;
  static unsigned int* pool[kMaxDev] = {};
  static int ring_next[kMaxDev] = {}, graph_next[kMaxDev] = {};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDev) return nullptr;
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(st, &cap) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  std::lock_guard<std::mutex> g(mu);
  if (!pool[dev]) {
    if (cap != cudaStreamCaptureStatusNone) return nullptr;        // no allocation while a capture is open
    if (cudaMalloc(&pool[dev], (kClaimRing + kClaimGraph) * sizeof(unsigned int)) != cudaSuccess) {
      cudaGetLastError();
      pool[dev] = nullptr;
      return nullptr;
    }
  }
  if (cap != cudaStreamCaptureStatusNone) {
    if (graph_next[dev] >= kClaimGraph) return nullptr;
    return pool[dev] + kClaimRing + graph_next[dev]++;
  }
  const int s = ring_next[dev];
  ring_next[dev] = (s + 1) % kClaimRing;
  return pool[dev] + s;
}

// Float64 re-rounding of np.round(d, 3) ties is compiled into the variants that run when a clause of the validity mask
// hangs on a rounded distance (dce / ttc / be thresholds armed, or the caller asked for it): there the mask is the
// float64 reference's.  With those thresholds null (the deployment default, occlusion.yaml:20-28) only the last
// digit of the reported min_dce could differ, and the kernel without the tie path is a quarter faster (DESIGN.md 5.1).
static bool needs_ties(const MetricKArgs& k) { return (k.tmask & (FO_T_DCE | FO_T_TTC | FO_T_BE)) != 0 || k.exact_dce; }

// FO_STATIC_STRIDE=1: teams stride over the trajectories instead of claiming them (A/B switch, summary kernels only)
static bool static_stride() {
  const char* fixed = getenv("FO_STATIC_STRIDE");
  return fixed && fixed[0] == '1';
}

// f(UNI, TIES) as std::bool_constants: the shape and tie-path variant of a summary-kernel family
template <class F>
static int with_shape(bool uni, bool ties, F&& f) {
  if (uni) return ties ? f(std::true_type{}, std::true_type{}) : f(std::true_type{}, std::false_type{});
  return ties ? f(std::false_type{}, std::true_type{}) : f(std::false_type{}, std::false_type{});
}

// One team of W warps per trajectory (persistent: as many teams as fit on the device, claiming trajectories).
int launch_metric_sweep(const MetricKArgs& k, int num_sms, cudaStream_t st) {
  const SweepShape shape{lane_group_log2(k.A)};
  const int W = pick_team_warps(k.N, k.T, k.A, num_sms);
  const bool uni = W == 1 && shape.lg_agents == 5, ties = needs_ties(k);
  const size_t smem = sweep_smem_bytes(k.T, W, uni, ties);
  const bool fixed = static_stride();
  return with_shape(uni, ties, [&](auto u, auto t) {
    if (k.corr && k.stats)
      return launch_persistent<fo_metric_sweep_corr_stats_kernel<u, t>>(k, num_sms, W * 32, 1, smem, fixed, st, shape);
    if (k.corr) return launch_persistent<fo_metric_sweep_corr_kernel<u, t>>(k, num_sms, W * 32, 1, smem, fixed, st, shape);
    if (k.stats)
      return launch_persistent<fo_metric_sweep_kernel<0u, true, u, t>>(k, num_sms, W * 32, 1, smem, fixed, st, shape);
    return with_mask(k.mmask, [&](auto m) {
      return launch_persistent<fo_metric_sweep_kernel<m, false, u, t>>(k, num_sms, W * 32, 1, smem, fixed, st, shape);
    });
  });
}

int launch_metric_batch(const MetricKArgs& k, int num_sms, int W, bool uni, const BatchView& bv, const SelectView& sv,
                        cudaStream_t st) {
  const SweepShape shape{0};
  const bool ties = needs_ties(k);
  const size_t smem = sweep_smem_bytes(k.T, W, uni, ties);
  const bool fixed = static_stride();
  return with_shape(uni, ties, [&](auto u, auto t) {
    if (sv.selected && k.corr)
      return launch_persistent<fo_metric_batch_select_kernel<u, t, true>>(k, num_sms, W * 32, 1, smem, fixed, st, shape, bv, sv);
    if (sv.selected)
      return launch_persistent<fo_metric_batch_select_kernel<u, t, false>>(k, num_sms, W * 32, 1, smem, fixed, st, shape, bv, sv);
    if (k.corr) return launch_persistent<fo_metric_batch_corr_kernel<u, t>>(k, num_sms, W * 32, 1, smem, fixed, st, shape, bv);
    return with_mask(k.mmask, [&](auto m) {
      return launch_persistent<fo_metric_batch_kernel<m, u, t>>(k, num_sms, W * 32, 1, smem, fixed, st, shape, bv);
    });
  });
}

}  // namespace fo
