/*
 * fo_b200.h -- C ABI of the B200-native Frenetix-Occlusion assessment hot path (libfo_b200.so).
 *
 * Plain C: device/host pointers and sizes only, no torch / C++ types.  Every entry point returns
 * FO_OK (0) or a negative FoStatus; nothing throws across the boundary; fo_last_error() gives the
 * thread-local message of the last failure.  "dev" pointers are CUDA device pointers owned by the
 * caller (they must stay alive until the stream work has completed); all device entry points are
 * asynchronous on the given stream (a cudaStream_t passed as void*; NULL = legacy default stream).
 *
 * The reference is pure Python and has no FFI; each entry point names the reference interface it
 * replaces (paths relative to the reference repository root).  The Python host
 * (frenetix_occlusion_b200/) binds these with ctypes, see INTEGRATION.md.
 */
#ifndef FO_B200_H
#define FO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FO_ABI_VERSION 1

typedef enum FoStatus {
  FO_OK = 0,
  FO_ERR_INVALID_ARG = -1,   /* NULL pointer, negative size, unsupported shape */
  FO_ERR_UNSUPPORTED = -2,   /* e.g. T > FO_MAX_STATES */
  FO_ERR_CUDA = -3,          /* a CUDA runtime call failed (message in fo_last_error) */
  FO_ERR_NO_DEVICE = -4
} FoStatus;

#define FO_MAX_STATES 128    /* states per trajectory / prediction (reference uses 31 and 51) */

/* ---- metric activation bits: names of frenetix_occlusion/metrics/metric.py:109-117 ------------ */
enum {
  FO_M_CP = 1u << 0, FO_M_DCE = 1u << 1, FO_M_TTC = 1u << 2, FO_M_HR = 1u << 3,
  FO_M_BE = 1u << 4, FO_M_TTCE = 1u << 5, FO_M_WTTC = 1u << 6
};
/* ---- armed-threshold bits: metric_thresholds of configurations/simulation/occlusion.yaml:20-28;
 *      only these six are ever checked by the reference (metric.py:55-98) ---------------------- */
enum {
  FO_T_HARM = 1u << 0, FO_T_RISK = 1u << 1, FO_T_BE = 1u << 2, FO_T_CP = 1u << 3,
  FO_T_TTC = 1u << 4, FO_T_DCE = 1u << 5
};
/* ---- agent kinds (commonroad ObstacleType values the reference can produce, agent.py:74-120,
 *      harm_model.py:15-32,158-190) ------------------------------------------------------------- */
enum {
  FO_KIND_PEDESTRIAN = 0, FO_KIND_BICYCLE = 1, FO_KIND_CAR = 2, FO_KIND_TRUCK = 3,
  FO_KIND_BUS = 4, FO_KIND_MOTORCYCLE = 5, FO_KIND_PRIORITY_VEHICLE = 6, FO_KIND_PARKED_VEHICLE = 7,
  FO_KIND_TAXI = 8, FO_KIND_TRAIN = 9, FO_KIND_UNKNOWN = 10
};

/* per-trajectory flag bits written to FoMetricArgs.flags */
enum {
  FO_F_BE_RANGE = 1u << 0    /* reference raises ValueError here: re-timed path overruns the original
                                (scipy interp1d bounds_error, metrics/be.py:117-124) */
};

/* Ego vehicle parameters: vehicle_params.{length,width,mass,wb_rear_axle,a_max}
 * (collision_probability.py:35, harm_model.py:96-97, convert_dynamic_obstacle.py:60,78, be.py:56). */
typedef struct FoVehicle {
  float length, width, mass, wb_rear_axle, a_max;
} FoVehicle;

/* Logistic harm coefficients: frenetix_occlusion/config/harm_params.json keys
 * log_reg.reduced_sym_angle_areas.{const,speed,side,rear}, log_reg.ignore_angle.{const,speed},
 * pedestrian.{const,speed} (logistic_regression.py:35-48,71-73; harm_model.py:137-146). */
typedef struct FoHarmCoeffs {
  float rs_const, rs_speed, rs_side, rs_rear;
  float ia_const, ia_speed;
  float ped_const, ped_speed;
} FoHarmCoeffs;

/* Raw phantom-agent predictions, SoA, padded to t_stride states per agent: what
 * FOAgentManager.predictions holds per prediction id (agent.py:420-424, 530-534) plus the owning
 * agent's type and unbuffered shape (agent.py:213-217).  All pointers are device pointers. */
typedef struct FoAgentsRaw {
  int32_t n_agents;
  int32_t t_stride;            /* padded row length (>= max n_states) */
  const float *x, *y;          /* [A, t_stride] pos_list */
  const float *yaw;            /* [A, t_stride] orientation_list */
  const float *v;              /* [A, t_stride] v_list */
  const float *var_x, *var_y;  /* [A, t_stride] diag(cov_list); both 0 -> 0.1 (collision_probability.py:85-87) */
  const int32_t *n_states;     /* [A] len(pos_list) */
  const int32_t *kind;         /* [A] FO_KIND_* */
  const float *length, *width; /* [A] agent.shape (unbuffered) -> DCE / BE rectangles */
  const float *buf_length, *buf_width; /* [A] prediction['shape'] (buffered) -> CP points, mass */
} FoAgentsRaw;

/* Number of bytes of device memory fo_agents_pack() needs for its packed table. */
size_t fo_agent_table_bytes(int32_t n_agents, int32_t t_stride);

/* Stage 2 -> stage 3 hand-over: derive per-state (cos,sin yaw, 1/(sqrt2 sigma)) and per-agent
 * (protection class, mass split m_o/(m_e+m_o), half extents) quantities once per planning cycle.
 * Replaces the per-trajectory re-derivation in harm_model.py:58-79 and
 * convert_dynamic_obstacle.py:17-49. */
int fo_agents_pack(const FoAgentsRaw *raw, const FoVehicle *vehicle, void *table_dev, size_t table_bytes,
                   void *stream);

#define FO_MAX_PEERS 8
#define FO_SUMMARY_K 10
/* summary[n, :] = { max_ego_risk_all, max_obst_risk_all, max_ego_harm_all, max_obst_harm_all,
 *                   max_collision_probability_all, max_obst_harm_with_cp_all   (hr.py:108-114),
 *                   min over agents of dce [m]            (dce.py:52-99; +inf without agents),
 *                   wttc [s]                              (wttc.py:32-42; +inf = no collision),
 *                   max over agents of break_threat_number (be.py:56),
 *                   max over agents of required_constant_deceleration (be.py:53) } */
#define FO_PAIR_K 12
/* pair[n, a, :] = { dce, time_dce, max_ego_risk, max_obst_risk, max_obst_risk_index,
 *                   max_obst_harm_with_cp, max_ego_harm, max_obst_harm, max_collision_probability,
 *                   required_constant_deceleration, break_threat_number, argmax_cp_index } */
#define FO_STEP_K 3
/* step[n, a, j, :] = { collision_probability[j] (CP of ego step j+1), ego_harm[j], obst_harm[j] },
 *                    j in [0, T-1); harm entries are NaN for j >= min(T-1, n_states[a]). */

typedef struct FoMetricArgs {
  /* ---- inputs --------------------------------------------------------------------------------- */
  const float *ego;        /* dev [N, T, 5] (x, y, theta, v, a): trajectory.cartesian.* of every sampled
                              trajectory, rear-axle reference point (SURVEY.md 8a) */
  int32_t n_traj;          /* N */
  int32_t n_states;        /* T = len(trajectory.cartesian.x) */
  const void *agent_table; /* dev, written by fo_agents_pack */
  int32_t n_agents;        /* A (0 -> every trajectory valid, metric.py:44-45) */
  int32_t t_stride;
  FoVehicle vehicle;
  FoHarmCoeffs harm;
  double dt;               /* agent_manager.dt */
  uint32_t metric_mask;    /* FO_M_* after dependency resolution (metric.py:125-147) */
  uint32_t threshold_mask; /* FO_T_* for thresholds that are not null */
  double thr_harm, thr_risk, thr_be, thr_cp, thr_ttc, thr_dce;  /* strict > / < as metric.py:55-98 */
  /* ---- outputs (device; optional ones may be NULL) --------------------------------------------- */
  uint8_t *valid;          /* [N] safety_check of Metric.evaluate_metrics */
  float *summary;          /* [N, FO_SUMMARY_K], 8-byte aligned */
  uint32_t *flags;         /* [N] FO_F_* */
  float *pair;             /* [N, A, FO_PAIR_K] or NULL; 16-byte aligned */
  float *step;             /* [N, A, T-1, FO_STEP_K] or NULL */
  /* ---- fused result exchange of a trajectory-sharded sweep (summary path only) ------------------- */
  int32_t n_peers;         /* 0 = none.  Otherwise the kernel's epilogue stores valid / summary / flags of every trajectory
                              ALSO at the same addresses shifted by peer_delta[p] bytes: the mapped buffers of the other
                              ranks (fo_peer_open), reached over NVLink.  This rank's slice of every rank's gather buffer
                              is complete when the launch has finished; no all-gather follows (SURVEY.md 8e). */
  int32_t reserved_;
  int64_t peer_delta[FO_MAX_PEERS];
} FoMetricArgs;

/* Stage 3, the dense core: every trajectory x every phantom prediction x every step.
 * Replaces Metric.evaluate_metrics (metrics/metric.py:35-100) and everything it dispatches to
 * (cp.py, dce.py, ttc.py, ttce.py, wttc.py, hr.py, be.py, metrics/utils/ helpers) for a whole bundle. */
int fo_metric_bundle(const FoMetricArgs *args, void *stream);

/* Work counters of one pass of the summary path over the bundle (same arguments as fo_metric_bundle, pair and
 * step must be NULL): how much of the algorithmic work survives the exact bounds.  bench.py uses them for the
 * flop model behind roofline.achieved.  counters_dev[FO_STATS_K] (device, zeroed by the call) =
 * { (trajectory, agent, step) evaluations visited, exact oriented-box distances, LR4S impact-angle logits,
 *   collision-probability evaluations (inside the 5 m gate), BE pairs, BE pair tests (the probes of one bisection
 *   per pair), (agent, 8-step window) items tested by the window filter, items it kept, BE tree nodes walked, BE
 *   re-timed ego-path chunks of 32 steps computed }  -- the window and tree counters are 0 when the bundle is small
 *   enough for the multi-warp team shape, which has no window filter and bisects one BE pair at a time. */
#define FO_STATS_K 10
int fo_metric_stats(const FoMetricArgs *args, uint64_t *counters_dev, void *stream);

/* Predictions with full 2x2 covariances [[var_x, cov_xy], [cov_xy, var_y]] (a learned predictor's correlated ones):
 * the collision probability of each gated step is the mass of N(mu, Sigma) with the full Sigma of covariance i-1 over
 * each of the three ego boxes, per obstacle point, / 3 -- the reference's mvnun (collision_probability.py:94-122).
 * Everything else (5 m gate, index offsets, ego boxes, the all-zero matrix -> 0.1 I rule) is as on the diagonal path.
 *
 * fo_agent_table_bytes_corr: fo_agent_table_bytes plus one appended per-(agent, state) section; the layout of the
 * diagonal table in front of it is unchanged.
 * fo_agents_pack_corr: `cov_xy` is a device array [A, t_stride] aligned with raw->var_x / var_y.  Writes what
 * fo_agents_pack writes, byte for byte, plus the correlation section.  PRECONDITION: every covariance of a state the
 * agent has is symmetric positive definite (or all zero); the device data is not inspected by the host, and a state
 * that violates it (|rho| >= 1, a zero variance with a non-zero covariance) gets NaN collision probabilities.
 * fo_metric_bundle_corr: fo_metric_bundle on a table written by fo_agents_pack_corr, with its outputs, checks and
 * CUDA-graph capture behaviour.  Each CP term is a float64 bivariate-normal rectangle mass.  n_peers > 0 returns
 * FO_ERR_UNSUPPORTED; fo_metric_bundle_corr_peers (below) takes peer stores.  fo_metric_stats_corr (below) gives the work
 * counters of a correlated table.  Batches take correlated tables through their *_corr forms (fo_agents_pack_batch_corr,
 * below), and so do batches from host memory (fo_metric_batch_host_corr, below); fo_metric_bundle_host,
 * fo_metric_batch_host and fo_metric_stats take diagonal tables only. */
size_t fo_agent_table_bytes_corr(int32_t n_agents, int32_t t_stride);
int fo_agents_pack_corr(const FoAgentsRaw *raw, const float *cov_xy, const FoVehicle *vehicle, void *table_dev,
                        size_t table_bytes, void *stream);
int fo_metric_bundle_corr(const FoMetricArgs *args, void *stream);

/* fo_metric_bundle_corr with the fused result exchange of a trajectory-sharded sweep: n_peers / peer_delta are honoured
 * on the summary path as fo_metric_bundle honours them.  n_peers outside [0, FO_MAX_PEERS] is FO_ERR_INVALID_ARG and
 * n_peers > 0 with pair / step is FO_ERR_UNSUPPORTED, both checked before any device query; with n_peers = 0 it is
 * fo_metric_bundle_corr. */
int fo_metric_bundle_corr_peers(const FoMetricArgs *args, void *stream);

/* fo_metric_stats on a table written by fo_agents_pack_corr: the same checks, zeroed counters, summary outputs only and
 * no peers.  The FO_STATS_K counters do not depend on the covariances (gate, window filter, BE pairs, probes and tree
 * walk, drained CP items), so they equal fo_metric_stats' on the diagonal table of the same agents.  (With a team of
 * W > 1 warps the box-distance, LR4S, BE-pair and BE-probe counts depend on the order in which the warps pool their
 * work, and vary from run to run on either table; the others do not.)  Costs one pass of the correlated summary path. */
int fo_metric_stats_corr(const FoMetricArgs *args, uint64_t *counters_dev, void *stream);

/* Same computation driven from HOST buffers (pinned or pageable): copies ego / agents to the
 * device, runs fo_agents_pack + fo_metric_bundle, copies valid/summary/flags back and synchronises.
 * This is the call a non-torch embedder of the reference would make; device workspace is owned by
 * the library and grown on demand (per calling thread). `agents` holds HOST pointers here;
 * `out_pair` / `out_step` may be NULL.  When `params->valid`, `->summary` and `->flags` are all non-NULL (and no detail
 * output is requested) they are DEVICE buffers of n_traj rows in which the results are left as well -- a rank's slice of
 * a gather buffer -- and `params->n_peers` / `peer_delta` apply as in fo_metric_bundle; otherwise they are ignored. */
int fo_metric_bundle_host(const float *ego_host, int32_t n_traj, int32_t n_states, const FoAgentsRaw *agents_host,
                          const FoMetricArgs *params /* vehicle, harm, dt, masks, thresholds; optional device outputs */,
                          uint8_t *out_valid, float *out_summary, uint32_t *out_flags, float *out_pair,
                          float *out_step);

/* ---- batches of independent planning problems --------------------------------------------------------
 * P problems (one ego each: the vehicles of a multi-agent simulation, the scenes of a re-simulation) assessed by
 * ONE pack call and ONE metric call.  Replaces a loop of Metric.evaluate_metrics / assess_bundle calls, one
 * set_agents + fo_metric_bundle per problem.  Problem p has its own phantom agents (A_p may be 0) and trajectories
 * (N_p may be 0); T, dt, metrics, thresholds and harm coefficients are shared.  The ego vehicle is shared by the entry
 * points below, and per problem with their *_vehicles forms (the vehicles of a mixed fleet).  Problem p's results
 * equal those fo_metric_bundle gives for it alone under FO_TEAM_WARPS set to the batch's team size. */
typedef struct FoBatchProblem {
  int64_t traj_begin;      /* first row of the problem in ego / valid / summary / flags: rows are contiguous, in problem
                              order, and the problems together cover [0, n_traj) */
  int32_t n_traj;          /* N_p */
  int32_t n_agents;        /* A_p */
  int32_t t_stride;        /* stride of the problem's packed table (>= its longest prediction, <= FO_MAX_STATES) */
  int32_t reserved_;
  int64_t table_offset;    /* byte offset of the problem's packed table in the arena (16-byte aligned) */
} FoBatchProblem;

/* Arena layout of P packed tables: table_offset_host[p] receives the offset of problem p's table, every table starts
 * 16-byte aligned and takes fo_agent_table_bytes(A_p, t_stride_p) bytes, problems without agents take none.  Returns
 * the arena size (0 and an error message for malformed input).  Host only. */
size_t fo_agent_batch_layout(int32_t n_problems, const int32_t *n_agents_host, const int32_t *t_stride_host,
                             int64_t *table_offset_host);

/* fo_agents_pack for P problems in two launches: `raw` (device arrays) holds the agents of all problems concatenated in
 * problem order -- raw->n_agents = sum A_p, row stride raw->t_stride >= every t_stride_p.  Problem p's table is
 * byte-identical to what fo_agents_pack writes for its agents alone with t_stride_p.  `problems_host`: n_agents,
 * t_stride and table_offset are read (HOST memory). */
int fo_agents_pack_batch(const FoAgentsRaw *raw, int32_t n_problems, const FoBatchProblem *problems_host,
                         const FoVehicle *vehicle, void *arena_dev, size_t arena_bytes, void *stream);

typedef struct FoMetricBatchArgs {
  FoMetricArgs common;     /* ego [n_traj, T, 5] of all problems, n_traj = sum N_p; agent_table = the arena;
                              n_agents / t_stride are ignored (per problem); n_peers 0; pair / step must be NULL for
                              fo_metric_batch (see fo_metric_batch_detail) */
  int32_t n_problems;
  int32_t reserved_;
  const FoBatchProblem *problems;   /* HOST [n_problems]: validated before any device work */
  size_t arena_bytes;
} FoMetricBatchArgs;

/* fo_metric_bundle's summary path over a batch: valid / summary / flags of every row.  One team size W for the batch,
 * chosen as fo_metric_bundle chooses it for n_traj trajectories and the problem with the fewest agents; with W = 1 the
 * problems with >= 17 agents run the one-warp window-filter shape (one launch) and the others the team shape (a second
 * launch).  The per-problem descriptors are staged through library-owned page-locked and device buffers (per calling
 * thread and device).  Not capturable in a CUDA graph. */
int fo_metric_batch(const FoMetricBatchArgs *args, void *stream);

/* fo_metric_bundle's detail path over a batch, in one launch: valid / summary / flags of every row and the pair / step
 * arrays of every problem.  Same arguments as fo_metric_batch, except that common.pair and / or common.step must be
 * non-NULL (both NULL: FO_ERR_INVALID_ARG) and n_peers must be 0 (else FO_ERR_UNSUPPORTED).  Problem p's blocks sit back
 * to back, in problem order:
 *   pair: [N_p, A_p, FO_PAIR_K]          at float offset  FO_PAIR_K * sum_{q<p} N_q A_q
 *   step: [N_p, A_p, T-1, FO_STEP_K]     at float offset  FO_STEP_K * (T-1) * sum_{q<p} N_q A_q
 * pair must be 16-byte aligned (then so is every block) and step 4-byte aligned (every block is 8-byte aligned when T-1
 * is even and step is).  Problem p's five outputs equal, bit for bit, what fo_metric_bundle gives for it alone with the
 * same detail buffers requested; a problem without agents gets what fo_metric_bundle gives it without detail buffers.
 * The descriptors are validated and staged as in fo_metric_batch.  Not capturable in a CUDA graph. */
int fo_metric_batch_detail(const FoMetricBatchArgs *args, void *stream);

/* The three batch calls with one ego vehicle per problem: vehicles_host is a HOST array of n_problems entries (read
 * before the call returns), and problem p is assessed with vehicles_host[p] wherever the calls above use the shared
 * vehicle (pack: its mass enters the harm mass split; metrics: args->common.vehicle is ignored).  Problem p's table
 * and outputs equal, bit for bit, what fo_agents_pack + fo_metric_bundle give for it alone with
 * FoMetricArgs.vehicle = vehicles_host[p].  A NULL vehicles_host with n_problems > 0 is FO_ERR_INVALID_ARG, checked
 * before any device work; otherwise the arguments are validated as in the shared-vehicle calls, which are the case
 * vehicles_host[p] = the shared vehicle for every p. */
int fo_agents_pack_batch_vehicles(const FoAgentsRaw *raw, int32_t n_problems, const FoBatchProblem *problems_host,
                                  const FoVehicle *vehicles_host, void *arena_dev, size_t arena_bytes, void *stream);
int fo_metric_batch_vehicles(const FoMetricBatchArgs *args, const FoVehicle *vehicles_host, void *stream);
int fo_metric_batch_detail_vehicles(const FoMetricBatchArgs *args, const FoVehicle *vehicles_host, void *stream);

/* Correlated and diagonal problems in one batch (predictions with full 2x2 covariances, fo_agents_pack_corr).
 * corr_host is a HOST array of n_problems flags: nonzero = problem p's table is a correlated one; vehicles_host is as in
 * the *_vehicles calls.  Problem p's table and outputs equal, bit for bit, what fo_agents_pack_corr +
 * fo_metric_bundle_corr (flagged) or fo_agents_pack + fo_metric_bundle (not flagged) give for it alone with its vehicle
 * and FO_TEAM_WARPS set to the batch's team size W, chosen as in fo_metric_batch from all problems.  A NULL corr_host or
 * vehicles_host with n_problems > 0 is FO_ERR_INVALID_ARG; every argument is validated before any device work, as in
 * the calls above, with a flagged table checked against fo_agent_table_bytes_corr.
 *
 * fo_agent_batch_layout_corr: fo_agent_batch_layout, except that a flagged problem with agents takes
 * fo_agent_table_bytes_corr bytes (rounded up to 16); with every flag 0 the same offsets and size.
 * fo_agents_pack_batch_corr: fo_agents_pack_batch_vehicles plus one launch that writes the correlation sections of
 * all flagged problems.  cov_xy is a device array [raw->n_agents, raw->t_stride] aligned with raw->var_x / var_y; it
 * may be NULL when no flagged problem has agents.  The positive-definiteness precondition of fo_agents_pack_corr holds.
 * fo_metric_batch_corr / fo_metric_batch_detail_corr: fo_metric_batch_vehicles / fo_metric_batch_detail_vehicles over
 * such an arena, with their outputs, layout and checks.  The summary call makes one launch per non-empty class of
 * problems (diagonal or correlated x window-filter or team shape), the detail call one per non-empty class (diagonal,
 * correlated).  n_peers != 0 is FO_ERR_UNSUPPORTED; not capturable in a CUDA graph. */
size_t fo_agent_batch_layout_corr(int32_t n_problems, const int32_t *n_agents_host, const int32_t *t_stride_host,
                                  const uint8_t *corr_host, int64_t *table_offset_host);
int fo_agents_pack_batch_corr(const FoAgentsRaw *raw, const float *cov_xy, int32_t n_problems,
                              const FoBatchProblem *problems_host, const uint8_t *corr_host,
                              const FoVehicle *vehicles_host, void *arena_dev, size_t arena_bytes, void *stream);
int fo_metric_batch_corr(const FoMetricBatchArgs *args, const uint8_t *corr_host, const FoVehicle *vehicles_host,
                         void *stream);
int fo_metric_batch_detail_corr(const FoMetricBatchArgs *args, const uint8_t *corr_host, const FoVehicle *vehicles_host,
                                void *stream);

/* A batch driven from HOST buffers (pinned or pageable), for embedders without a CUDA runtime of their own: the
 * planner's float64 ego rows in the caller's world frame and one float64 origin per problem in, results in host arrays
 * out, synchronised.  The library shifts every row by its problem's origin on the device, in float64, and only then
 * rounds to float32: (float)(x - origin_p.x), (float)(y - origin_p.y), (float)theta, (float)v, (float)a -- what
 * MetricEngine.assess_batch stages on the host.  It then packs the agents into a library-owned arena and makes the
 * batch call, so the results equal, bit for bit, fo_agents_pack_batch[_vehicles] + fo_metric_batch[_vehicles] on that
 * bundle, or fo_metric_batch_detail[_vehicles] when out_pair or out_step is non-NULL and there is a pair / step block
 * to write (some problem has trajectories and agents; for step also T > 1) -- otherwise the summary path runs and the
 * detail outputs are not touched.  out_pair / out_step are laid out as in fo_metric_batch_detail and need no alignment;
 * out_summary / out_flags may be NULL.
 *   ego_host      [n_traj, T, 5] (x, y, theta, v, a), rows of the problems contiguous in problem order
 *   origins_host  [n_problems, 2] problem p's origin
 *   agents_host   HOST pointers: the agents of all problems concatenated in problem order, positions already relative
 *                 to their problem's origin, row stride t_stride >= every problem's t_stride (as fo_agents_pack_batch)
 *   problems_host traj_begin, n_traj, n_agents, t_stride; table_offset is ignored (the library places the tables)
 *   vehicles_host [n_problems] or NULL: params->vehicle for every problem
 *   params        vehicle, harm, dt, metric / threshold masks and thresholds; its device pointers (ego, agent_table,
 *                 valid, summary, flags, pair, step) and sizes are ignored; n_peers != 0 is FO_ERR_UNSUPPORTED
 * Every argument is validated before any device work, with the checks and messages of the device batch calls; NULL
 * problems_host, origins_host or agents_host with n_problems > 0, and NULL ego_host or out_valid with n_traj > 0, are
 * FO_ERR_INVALID_ARG.  The float64 rows cross PCIe in chunks (FO_HOST_CHUNK_MB, as fo_metric_bundle_host), each
 * converted while the next one is copied; the metric call follows the last chunk.  Device workspace as
 * fo_metric_bundle_host's (per calling thread, grown on demand). */
int fo_metric_batch_host(const double *ego_host, int32_t n_traj, int32_t n_states, const double *origins_host,
                         const FoAgentsRaw *agents_host, int32_t n_problems, const FoBatchProblem *problems_host,
                         const FoVehicle *vehicles_host, const FoMetricArgs *params, uint8_t *out_valid,
                         float *out_summary, uint32_t *out_flags, float *out_pair, float *out_step);

/* fo_metric_batch_host with correlated predictions (full 2x2 covariances), for host-memory embedders: the arguments,
 * outputs, float64 ingest, workspace and checks of fo_metric_batch_host, plus
 *   cov_xy_host   [agents_host->n_agents, agents_host->t_stride] float32, the off-diagonal term of every covariance,
 *                 aligned with var_x / var_y (cov_list[..., 0, 1] of the reference); may be NULL when no flagged problem
 *                 has agents
 *   corr_host     [n_problems]: nonzero = problem p is correlated (no effect on a problem without agents); NULL with
 *                 n_problems > 0 is FO_ERR_INVALID_ARG
 * Tables are placed as fo_agent_batch_layout_corr places them and packed by fo_agents_pack_batch_corr; the metric call is
 * fo_metric_batch_corr, or fo_metric_batch_detail_corr under fo_metric_batch_host's rule for the detail path, with
 * vehicles_host or, when it is NULL, params->vehicle for every problem.  The results equal, bit for bit, those calls on
 * the bundle fo_metric_batch_host's ingest produces.  One correlated planner is the case n_problems = 1: its team size is
 * the one fo_metric_bundle_corr picks, so it gets fo_agents_pack_corr + fo_metric_bundle_corr bit for bit.
 * The covariances are checked on the host before any device work: every covariance the correlation pack reads (covariance
 * i-1 of every state i < min(n_states[a], t_stride_p) of a flagged problem's agents; state 0 reads covariance 0) must be
 * positive definite by the predicate under which fo_agents_pack_corr writes NaN -- the all-zero matrix is 0.1 I, and
 * otherwise |cov_xy / sqrt(var_x var_y)| < 1 in float64 -- else FO_ERR_INVALID_ARG names the problem, the agent within it
 * and the covariance index.  This rejects a state with one zero variance and zero covariance, which the reference's
 * diagonal rule accepts but which gives NaN collision probabilities on the correlated path.  Covariances the pack never
 * reads (index n_states - 1, the padding up to t_stride) are not checked.  n_peers != 0 is FO_ERR_UNSUPPORTED. */
int fo_metric_batch_host_corr(const double *ego_host, int32_t n_traj, int32_t n_states, const double *origins_host,
                              const FoAgentsRaw *agents_host, const float *cov_xy_host, int32_t n_problems,
                              const FoBatchProblem *problems_host, const uint8_t *corr_host,
                              const FoVehicle *vehicles_host, const FoMetricArgs *params, uint8_t *out_valid,
                              float *out_summary, uint32_t *out_flags, float *out_pair, float *out_step);


/* ---- stage 1: sensor visibility by ray casting ----------------------------------------------------
 * Replaces SensorModel.calc_visible_and_occluded_area (sensor_model.py:41-193): the reference clips
 * road ∩ sensor-sector with one "shadow" quad per road-border edge (sensor_model.py:137-155) and per
 * non-bicycle obstacle (sensor_model.py:174-191, helper_functions.py:139-176).  A point lies in such a
 * shadow exactly when the segment ego->point crosses the occluding edge, so the same region is
 * described by the first-hit range of every ray of a fan over the field of view.  F independent
 * frames per call (frame = one ego pose + obstacle set); rays are uniform over
 * [heading - fov/2, heading + fov/2] (fov >= 359.9 deg: full circle, angle_r = heading - pi + 2 pi r / R). */
#define FO_HIT_NONE (-1)      /* ray reaches the sensor radius unobstructed */
#define FO_HIT_BOUNDARY (-2)  /* first hit is a road-border segment */
enum { FO_RECT_EXISTS = 1u << 0,        /* obstacle has a state at this time step (fo_obstacle.py:79-116) */
       FO_RECT_TRANSPARENT = 1u << 1 }; /* obstacle type 'bicycle': seen but casts no shadow (sensor_model.py:177) */

typedef struct FoVisibilityArgs {
  int32_t n_frames, n_rays, n_obstacles, n_boundary;
  const float *ego;            /* dev [F, 3] (x, y, heading) */
  const float *rect;           /* dev [F, O, 5] (cx, cy, yaw, half_length, half_width): corner points as
                                  helper_functions.py:99-112 */
  const uint8_t *rect_flags;   /* dev [F, O] FO_RECT_* */
  const float *boundary;       /* dev [B, 4] (x1, y1, x2, y2) opaque road-border segments, world frame,
                                  shared by all frames; may be NULL when n_boundary == 0 */
  float sensor_radius;         /* occlusion.yaml:36 */
  float sensor_angle_deg;      /* occlusion.yaml:37 */
  float *range;                /* dev [F, R] first-hit distance, <= sensor_radius */
  int32_t *hit;                /* dev [F, R] obstacle index | FO_HIT_NONE | FO_HIT_BOUNDARY */
  uint8_t *visible;            /* dev [F, O] 1 = some ray sees the obstacle (visible_objects_timestep,
                                  sensor_model.py:64-76); may be NULL */
} FoVisibilityArgs;

int fo_visibility_raycast(const FoVisibilityArgs *args, void *stream);

/* Work counters of one fo_visibility_raycast pass (same arguments; the outputs are written as well): what survives
 * the culls.  counters_dev[FO_VIS_STATS_K] (device, zeroed by the call) = { ray x edge tests executed, (warp, edge)
 * pairs skipped because the edge lies beyond the farthest current hit of the warp's rays, edges staged after the
 * sensor-disc cull (summed over CTAs), edges listed by the per-fan sector cull (summed over fans) }.
 * bench.py uses them for the executed-work roofline of the stage. */
#define FO_VIS_STATS_K 4
int fo_visibility_stats(const FoVisibilityArgs *args, uint64_t *counters_dev, void *stream);

/* ---- stage 1 -> spawn locator: exact visibility / occlusion / road membership of query points -----
 * Replaces the shapely predicates SpawnLocator evaluates against SensorModel's products
 * (spawn_locator.py:263-275, 298, 406-444, 521, 552): `within` / `intersects` of points, lines and discs
 * with visible_area (sensor_model.py:79), occluded_area (sensor_model.py:85-93), road_polygon
 * (sensor_model.py:195-199) and obstacle_occlusions[id] (sensor_model.py:182-183).  The host samples the
 * geometry it is interested in (lines, disc rims, raster windows) and this kernel classifies every sample
 * with the reference's own construction evaluated point-wise: a point is shadowed iff the segment
 * ego -> point crosses an opaque edge (border edge of road ∩ sector, sensor_model.py:137-155; non-bicycle
 * obstacle, sensor_model.py:174-191) or lies inside an opaque obstacle.  One frame per call. */
enum {
  FO_PT_IN_SENSOR = 1u << 0,    /* inside the sensor sector: radius and field of view (sensor_model.py:114-125) */
  FO_PT_ON_ROAD = 1u << 1,      /* inside at least one lanelet polygon (road_polygon) */
  FO_PT_SHADOWED = 1u << 2,     /* segment ego -> point crosses an opaque edge */
  FO_PT_IN_OBSTACLE = 1u << 3,  /* inside an existing, opaque obstacle rectangle */
  FO_PT_VISIBLE = 1u << 4,      /* IN_SENSOR & ON_ROAD & !SHADOWED & !IN_OBSTACLE  == within visible_area */
  FO_PT_OCCLUDED = 1u << 5,     /* ON_ROAD & within +-90 deg of the heading & closer than occluded_radius
                                   & !VISIBLE                                       == within occluded_area */
  FO_PT_FOCUS_SHADOW = 1u << 6, /* behind (not inside) obstacle `focus_obstacle` as seen from the ego
                                                                  == within obstacle_occlusions[id] */
  FO_PT_FOCUS_NEAR = 1u << 7    /* closer than `focus_margin` to obstacle `focus_obstacle` (0 inside)
                                   == within current_polygon.buffer(focus_margin), spawn_locator.py:275 */
};

typedef struct FoPointQueryArgs {
  int32_t n_points, n_obstacles, n_boundary, n_polygons;
  const float *ego;            /* dev [3] (x, y, heading) */
  const float *points;         /* dev [M, 2] query points, same frame as ego / rect / boundary */
  const float *rect;           /* dev [O, 5] as FoVisibilityArgs.rect (one frame) */
  const uint8_t *rect_flags;   /* dev [O] FO_RECT_* */
  const float *boundary;       /* dev [B, 4] opaque road-border segments */
  const float *poly_xy;        /* dev [V, 2] lanelet polygon rings (lanelet.polygon), concatenated, open rings */
  const int32_t *poly_off;     /* dev [n_polygons + 1] offsets into poly_xy */
  float sensor_radius, sensor_angle_deg;
  float occluded_radius;       /* 1.5 * sensor_radius (sensor_model.py:88) */
  int32_t focus_obstacle;      /* obstacle index for FO_PT_FOCUS_SHADOW / FO_PT_FOCUS_NEAR, or -1 */
  float focus_margin;          /* buffer distance of FO_PT_FOCUS_NEAR [m] */
  uint32_t *flags;             /* dev [M] FO_PT_* */
  int32_t *blocker;            /* dev [M] first opaque thing the segment ego -> point meets: obstacle index |
                                  FO_HIT_BOUNDARY | FO_HIT_NONE; may be NULL */
  uint64_t *lanelets;          /* dev [M] bit i set = point inside polygon i (i < 64); may be NULL */
} FoPointQueryArgs;

int fo_visibility_points(const FoPointQueryArgs *args, void *stream);

/* Which obstacles are seen ON THE ROAD: the reference intersects every obstacle polygon with the road-clipped visible
 * area (sensor_model.py:59-76); here an obstacle counts when some ray of a finished fo_visibility_raycast pass ends on
 * it at a point inside a lanelet polygon.  Ray end points: ego + (range - 1e-3f) (cos a, sin a), a = angle0 + dangle r
 * in float64, shifted by the frame origin, rounded to float32 and tested like fo_visibility_points' FO_PT_ON_ROAD. */
typedef struct FoHitsOnRoadArgs {
  int32_t n_rays, n_obstacles, n_polygons;
  const float *range;          /* dev [R] of one frame */
  const int32_t *hit;          /* dev [R] */
  const float *ego;            /* dev [3] frame ego (relative to the frame origin), as FoPointQueryArgs.ego */
  const float *poly_xy;        /* dev [V, 2] lanelet polygon rings relative to the frame origin */
  const int32_t *poly_off;     /* dev [n_polygons + 1] */
  double ego_x, ego_y;         /* ego position, caller's world frame */
  double angle0, dangle;       /* ray r points along angle0 + dangle * r */
  double org_x, org_y;         /* frame origin */
  uint8_t *on_road;            /* dev [O] out (zeroed by the call) */
} FoHitsOnRoadArgs;

int fo_visibility_hits_on_road(const FoHitsOnRoadArgs *args, void *stream);

/* ---- spawn locator, behind-dynamic-obstacle finder on the device --------------------------------------
 * Replaces the shapely chain of SpawnLocator._find_spawn_point_behind_dynamic_obstacle (spawn_locator.py:254-287:
 * possible_polygon ∩ (obstacle shadow | occluded area) ∩ disc − obstacle.buffer(1), largest part of the result, its
 * area / centroid / `contains`) and of _find_matching_rectangle (spawn_locator.py:695-726: clip a candidate box with
 * that part, area and centroid of the remainder, outline for the minimum rotated rectangle) by rasters that are
 * generated, classified (same predicate code as fo_visibility_points), labelled and reduced on the device; the host
 * reads back one small result record per raster.
 *
 * A raster is a grid of cell centres  P(i, j) = C + gx (cs, sn) + gy (-sn, cs),  gx = (i + 0.5) cell - hx,
 * gy = (j + 0.5) cell - hy, i < nx, j < ny, evaluated in float64 exactly as written (no contraction), then shifted by
 * the frame origin and rounded to float32 for the classification.  Linear cell index = i * ny + j. */
typedef struct FoRasterSpec {
  double cx, cy;               /* C, caller's world frame */
  double cs, sn;               /* direction of the first axis */
  double hx, hy;               /* half extents */
  double cell;
  double org_x, org_y;         /* frame origin: FoPointQueryArgs geometry is given relative to it */
  int32_t nx, ny;
} FoRasterSpec;

typedef struct FoRegionPredicate {
  uint64_t lanelet_mask;       /* a cell must lie in one of these lanelet polygons (bits as FoPointQueryArgs.lanelets) */
  uint32_t want_flags;         /* ... carry one of these FO_PT_* flags (FO_PT_FOCUS_SHADOW or FO_PT_OCCLUDED) */
  uint32_t reject_flags;       /* ... and none of these (FO_PT_FOCUS_NEAR) */
  double disc_x, disc_y, disc_r;   /* ... within disc_r of this point (world frame, float64 hypot) */
} FoRegionPredicate;

typedef struct FoRasterResult {
  double sum_x, sum_y;         /* sums of the selected cell centres (world frame): centroid = sum / count */
  int32_t count;               /* selected cells (area = count * cell^2) */
  int32_t contains;            /* region: 1 = the probe point lies in a selected cell */
  int32_t n_outline;           /* rect: selected cells with a missing 4-neighbour (may exceed the outline capacity) */
  int32_t n_components;        /* region: connected parts found */
} FoRasterResult;

typedef struct FoSpawnRegionArgs {
  FoPointQueryArgs frame;      /* geometry, sensor and focus_obstacle / focus_margin; points, flags, blocker, lanelets and
                                  n_points are ignored */
  FoRasterSpec raster;         /* nx * ny <= 2^30 */
  FoRegionPredicate pred;
  double probe_x, probe_y;     /* point of FoRasterResult.contains */
  int32_t *label;              /* dev [nx * ny] workspace; on return the component label of every cell (-1 = outside) */
  int32_t *size;               /* dev [nx * ny] workspace */
  unsigned long long *best;    /* dev [1] workspace */
  uint8_t *mask_dilated;       /* dev [nx * ny] out: largest 4-connected part (first in raster order on ties, as
                                  scipy.ndimage.label + argmax), dilated by one cell (4-neighbourhood) */
  FoRasterResult *result;      /* dev [1] out */
} FoSpawnRegionArgs;

int fo_spawn_region(const FoSpawnRegionArgs *args, void *stream);

typedef struct FoSpawnRectArgs {
  FoPointQueryArgs frame;
  FoRasterSpec raster;
  FoRegionPredicate pred;
  const FoRasterResult *centre_from;  /* dev, optional: when its count >= 3 the raster centre C is its centroid (the
                                         bicycle box is centred on what is left of the car box, spawn_locator.py:702-704) */
  const uint8_t *region_mask;  /* dev [region_n * region_n] FoSpawnRegionArgs.mask_dilated of the selected part */
  double region_ox, region_oy, region_cell;   /* lower-left corner and cell of that raster */
  int32_t region_n;
  int32_t outline_cap;
  uint8_t *mask;               /* dev [nx * ny] workspace */
  double *outline;             /* dev [outline_cap, 2] out: centres of the outline cells (any order) */
  FoRasterResult *result;      /* dev [1] out */
} FoSpawnRectArgs;

int fo_spawn_rect(const FoSpawnRectArgs *args, void *stream);

/* ---- peer-mapped result buffers (multi-GPU sweeps, one process per GPU) --------------------------------
 * The single exchange step of the sharded path (SURVEY.md 8e: one all-gather of valid / summary / flags) fused into the
 * metric kernel: every rank allocates its gather buffer with fo_peer_alloc, passes the handle to the other ranks (any
 * host channel; the Python host uses torch.distributed.all_gather_object), maps theirs with fo_peer_open and hands the
 * address differences to fo_metric_bundle as FoMetricArgs.peer_delta.  Buffers are plain device memory for every other
 * purpose.  CUDA IPC underneath: one process per GPU on one node, peer access over NVLink / NVSwitch. */
typedef struct FoPeerHandle { uint8_t bytes[64]; } FoPeerHandle;
int fo_peer_alloc(size_t bytes, void **dev_ptr, FoPeerHandle *handle);   /* zero-filled */
int fo_peer_open(const FoPeerHandle *handle, void **dev_ptr);            /* another process's buffer, mapped here */
int fo_peer_close(void *dev_ptr);                                        /* unmap (fo_peer_open) */
int fo_peer_free(void *dev_ptr);                                         /* release (fo_peer_alloc) */

/* ---- stage 2: phantom-agent rollouts ---------------------------------------------------------------
 * Constant-velocity pedestrian prediction: OAPPedestrianAgent._create_ped_trajectory (agent.py:451-505)
 * + _create_cr_predictions (agent.py:520-536) + create_cov_matrix (agent.py:260-280), written straight
 * into the SoA layout FoAgentsRaw expects.  Per agent: start (x0, y0) [double, origin-shifted by the
 * caller], speed v and heading phi; vx = round(v cos phi, 3), vy = round(v sin phi, 3) (agent.py:492-493);
 * pos[k] = p0 + k dt (vx, vy), yaw[k] = phi, v[k] = v, var[k] = var0 * factor^k. */
typedef struct FoRolloutCvArgs {
  int32_t n_agents;
  int32_t n_states;            /* int(horizon / dt) + 1 (agent.py:496) */
  int32_t t_stride;            /* row stride of the outputs (>= n_states) */
  double dt;
  double var0, var_factor;     /* 0.1 and agent_manager.prediction.variance_factor (occlusion.yaml:91) */
  const double *x0, *y0, *v, *phi;   /* dev [A] */
  float *x, *y, *yaw, *vel, *var_x, *var_y;   /* dev [A, t_stride] */
} FoRolloutCvArgs;

int fo_rollout_cv(const FoRolloutCvArgs *args, void *stream);

/* Path-following vehicle prediction (Car / Bicycle / Truck phantoms and configured real agents):
 * replaces OAPVehicleAgent (agent.py:283-426) + FrenetixHandler.create_trajectories
 * (utils/frenetix_handler.py:66-125), whose arithmetic lives in the un-vendored C++ `frenetix` library
 * (PARITY UNPINNED, DESIGN.md 2).  One job per (agent, route reference path).  Per job the 3 x 3 Frenet
 * samples of the reference are rolled out -- longitudinal quartic from (s0, v0, 0) to speed
 * {0.8, 1.0, 1.2} * v0 with zero end acceleration at t1, lateral quintic from (d0, 0, 0) to offset
 * {-0.5, 0, +0.5} m at t1 (frenetix_handler.py:80-105) -- mapped to Cartesian along the polyline, and the
 * sample with the smallest variance of the Cartesian speed is kept (agent.py:364-375). */
typedef struct FoRolloutPathArgs {
  int32_t n_jobs;
  int32_t n_states;            /* int(horizon / dt) + 1 */
  int32_t t_stride;
  double dt, t1;               /* t1 = 3.0 (frenetix_handler.py:80) */
  double var0, var_factor;
  const float *path_xy;        /* dev [P_total, 2] reference polylines of all jobs, concatenated */
  const int32_t *path_off;     /* dev [n_jobs + 1] offsets into path_xy (each path: 2..1024 points) */
  const double *x0, *y0, *v0;  /* dev [n_jobs] initial position and speed */
  float *x, *y, *yaw, *vel, *var_x, *var_y;   /* dev [n_jobs, t_stride] */
  int32_t *sample;             /* dev [n_jobs] selected sample 0..8 (speed-major), -1 = no valid projection */
} FoRolloutPathArgs;

int fo_rollout_path(const FoRolloutPathArgs *args, void *stream);

/* FP32 FMA-pipe probe used by bench.py to measure the roofline denominator on the box it runs on:
 * runs `iters` dependent-chain FFMAs on every lane of a full-occupancy grid and returns elapsed
 * milliseconds (CUDA events) in *ms and the flop count in *flops. */
int fo_probe_fp32_peak(int32_t iters, float *ms, double *flops, void *stream);

/* Number of kernel launches issued by this library since load (bench.py's gpu_launches). */
uint64_t fo_launch_count(void);

int fo_version(void);
const char *fo_last_error(void);

#ifdef __cplusplus
}
#endif
#endif /* FO_B200_H */
