// Device-side helpers shared by the metric kernels (detail kernel: fo_metric_detail.cu,
// summary kernel: fo_metric_sweep.cu).
#pragma once
#include <math_constants.h>

#include <atomic>
#include <type_traits>

#include "fo_common.cuh"

namespace fo {

constexpr unsigned kFull = 0xffffffffu;

// Constants of the ego vehicle in the units the kernels use (fill_ego_const in fo_metric.cu).  A batch of independent
// problems carries one per problem (BatchProb / DetailProb::veh).
struct EgoConst {
  float hEx, hEy;      // ego half extents
  float wb, a_max;
  float L3, L6, W2;    // L/3, L/6, W/2 (CP boxes)
};

struct MetricKArgs {
  const float* ego;
  int N, T, A, Tp;
  AgentTableView tab;
  EgoConst veh;
  FoHarmCoeffs hc;
  float dt;
  double dtd;
  uint32_t mmask, tmask;
  double thr_harm, thr_risk, thr_be, thr_cp, thr_ttc, thr_dce;
  // the two discrete threshold clauses in the units the kernels hold (host-computed, exact in float64):
  //   dce < thr_dce   <=>  round(d * 1000) < thr_dce_mm        (np.round(d, 3) = r / 1000.0, dce.py:79, metric.py:92-98)
  //   ttc < thr_ttc   <=>  first colliding step < thr_ttc_col  (np.round(step * dt, 3), ttc.py:43, metric.py:85-89)
  uint32_t thr_dce_mm, thr_ttc_col;
  bool exact_dce;      // summary kernel: re-round np.round(d, 3) ties in float64 even when no threshold needs it (FO_EXACT_DCE=1)
  bool corr;           // the table is a correlated one (fo_metric_bundle_corr): the CORR kernels read its s3 section
                       // (agent_corr_view).  Sits in padding: MetricKArgs and every parameter offset keep their size / place.
  uint8_t* valid;
  float* summary;
  uint32_t* flags;
  float* pair;
  float* step;
  unsigned long long* stats;   // optional [FO_STATS_K] work counters (see fo_metric_stats), NULL in production launches
  unsigned int* claim;         // zeroed per launch: next-trajectory counter of the summary kernel (NULL = static striding)
  int n_peers;                 // summary kernel: results are also stored at these byte offsets (peer-mapped gather buffers)
  long long peer_delta[FO_MAX_PEERS];
};

// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ AgentParams load_params(const AgentParams* p) {   // two 16-byte loads
  const int4* q = reinterpret_cast<const int4*>(p);
  int4 a = __ldg(q), b = __ldg(q + 1);
  AgentParams r;
  r.n_states = a.x; r.model = a.y; r.hl = __int_as_float(a.z); r.hw = __int_as_float(a.w);
  r.hlb = __int_as_float(b.x); r.ke = __int_as_float(b.y); r.ko = __int_as_float(b.z); r.pad = __int_as_float(b.w);
  return r;
}

// r / 1000 as the float the outputs carry (r = round(d * 1000) is exact in float32; correctly rounded division)
__device__ __forceinline__ float mm_to_m(uint32_t r) { return __fdiv_rn((float)r, 1000.0f); }
// np.round(step * dt, 3) as a float (ttc.py:43)
__device__ __forceinline__ float step_to_s(uint32_t step, double dt) { return (float)(rint((double)step * dt * 1000.0) * 0.001); }

__device__ __forceinline__ float umaxf(float v) {  // warp max of non-negative floats (bit order == value order)
  return __uint_as_float(__reduce_max_sync(kFull, __float_as_uint(v)));
}

__device__ __forceinline__ float pt_box_d2(float px, float py, float hx, float hy) {
  float dx = fmaxf(fabsf(px) - hx, 0.0f);
  float dy = fmaxf(fabsf(py) - hy, 0.0f);
  return fmaf(dx, dx, dy * dy);
}

// Oriented-box test in the frame of box E (half extents hEx,hEy): box O centred at (rx, ry) in that
// frame, rotated by the angle whose cos/sin are (c, s), half extents (hl, hw).
// Returns squared distance (0 when the closed boxes intersect).  dce.py:75-79 / be.py:181.
__device__ __forceinline__ float obb_d2(float rx, float ry, float c, float s, float hEx, float hEy, float hl, float hw) {
  float ac = fabsf(c), as = fabsf(s);
  // centre of E in O's frame is -(rox, roy)
  float rox = fmaf(rx, c, ry * s);
  float roy = fmaf(ry, c, -rx * s);
  bool sep = (fabsf(rx) > hEx + fmaf(hl, ac, hw * as)) | (fabsf(ry) > hEy + fmaf(hl, as, hw * ac)) |
             (fabsf(rox) > hl + fmaf(hEx, ac, hEy * as)) | (fabsf(roy) > hw + fmaf(hEx, as, hEy * ac));
  if (!sep) return 0.0f;
  // corners of O in E's frame: r +- hl*(c,s) +- hw*(-s,c)
  float ux = hl * c, uy = hl * s, wx = -hw * s, wy = hw * c;
  float d2 = pt_box_d2(rx + ux + wx, ry + uy + wy, hEx, hEy);
  d2 = fminf(d2, pt_box_d2(rx + ux - wx, ry + uy - wy, hEx, hEy));
  d2 = fminf(d2, pt_box_d2(rx - ux + wx, ry - uy + wy, hEx, hEy));
  d2 = fminf(d2, pt_box_d2(rx - ux - wx, ry - uy - wy, hEx, hEy));
  // corners of E in O's frame: -ro +- hEx*(c,-s) +- hEy*(s,c)
  ux = hEx * c; uy = -hEx * s; wx = hEy * s; wy = hEy * c;
  d2 = fminf(d2, pt_box_d2(-rox + ux + wx, -roy + uy + wy, hl, hw));
  d2 = fminf(d2, pt_box_d2(-rox + ux - wx, -roy + uy - wy, hl, hw));
  d2 = fminf(d2, pt_box_d2(-rox - ux + wx, -roy - uy + wy, hl, hw));
  d2 = fminf(d2, pt_box_d2(-rox - ux - wx, -roy - uy - wy, hl, hw));
  return d2;
}

// Exact distance between the ego box and an agent box (half extents hl, hw) of one state (dce.py:75-79): (dxr, dyr) =
// agent position minus ego reference point, EA = (x, y, cos theta, sin theta) of the ego, (c, s) = cos / sin of the
// agent's heading relative to the ego's.
__device__ __forceinline__ float ego_box_dist(float dxr, float dyr, float4 EA, float c, float s, const EgoConst& veh,
                                              float hl, float hw) {
  const float dx = dxr - veh.wb * EA.z, dy = dyr - veh.wb * EA.w;
  const float rx = fmaf(dx, EA.z, dy * EA.w), ry = fmaf(dy, EA.z, -dx * EA.w);
  return sqrtf(obb_d2(rx, ry, c, s, veh.hEx, veh.hEy, hl, hw));
}

// ---- rounding-tie refinement of np.round(d, 3) (dce.py:79) ---------------------------------------------------------
// The float32 distance carries an error of a few 1e-5 m; when d * 1000 lies within kTieBand of a rounding boundary
// (x.5) the float64 reference may round the other way.  Such candidates are re-evaluated here in double from the
// same float32 inputs (the formulation of oracle/geometry.py: SAT, then the 8 corner-to-box distances), so dce,
// time_dce and the first-collision step agree with the float64 reference except when the exact distance itself sits
// within 1e-12 of a boundary.  Rare path (a few per cent of the exact distance evaluations), kept out of line.
constexpr float kTieBand = 0.08f;

__device__ __forceinline__ bool near_rounding_boundary(float d) {
  const float t = d * 1000.0f;
  return fabsf(t - floorf(t) - 0.5f) < kTieBand;
}

__device__ __forceinline__ double pt_box_d2_f64(double px, double py, double hx, double hy) {
  const double dx = fmax(fabs(px) - hx, 0.0), dy = fmax(fabs(py) - hy, 0.0);
  return dx * dx + dy * dy;
}

// sin / cos in float64 of a float32 angle.  CUDA's sincos(double) drags an 8 kB Payne-Hanek slow path into every
// kernel that calls it (the metric kernels live next to a 32 kB instruction cache); headings are float32 values of
// moderate size, so a two-term Cody-Waite reduction by pi/2 plus the fdlibm kernel polynomials (|r| <= pi/4, error
// below 1e-16) is exact enough for a tie-break that only matters within 1e-12 of a rounding boundary.
static __device__ __noinline__ void sincos_f64_of_f32(float af, double* sn, double* cs) {
  const double a = (double)af;
  const double q = rint(a * 0.63661977236758134308);                 // 2 / pi
  double r = fma(-q, 1.57079632679489655800e+00, a);                 // pi/2 high part
  r = fma(-q, 6.12323399573676603587e-17, r);                        // pi/2 low part
  const double z = r * r;
  double ps = 1.58969099521155010221e-10;
  ps = fma(ps, z, -2.50507602534068634195e-08);
  ps = fma(ps, z, 2.75573137070700676789e-06);
  ps = fma(ps, z, -1.98412698298579493134e-04);
  ps = fma(ps, z, 8.33333333332248946124e-03);
  ps = fma(ps, z, -1.66666666666666324348e-01);
  const double s = fma(r * z, ps, r);
  double pc = -1.13596475577881948265e-11;
  pc = fma(pc, z, 2.08757232129817482790e-09);
  pc = fma(pc, z, -2.75573143513906633035e-07);
  pc = fma(pc, z, 2.48015872894767294178e-05);
  pc = fma(pc, z, -1.38888888888741095749e-03);
  pc = fma(pc, z, 4.16666666666666019037e-02);
  const double c = fma(z * z, pc, fma(-0.5, z, 1.0));
  const int n = (int)(long long)q & 3;
  *sn = (n == 0) ? s : (n == 1) ? c : (n == 2) ? -s : -c;
  *cs = (n == 0) ? c : (n == 1) ? -s : (n == 2) ? -c : s;
}

// ego reference point (ex, ey, eth), rectangle centre wb ahead; agent rectangle (ax, ay, ayaw); returns round(d * 1000)
static __device__ __noinline__ uint32_t obb_round_mm_f64(float ex, float ey, float eth, float wb, float hEx, float hEy,
                                                         float ax, float ay, float ayaw, float hl, float hw) {
  double se, ce, sa, ca;
  sincos_f64_of_f32(eth, &se, &ce);
  sincos_f64_of_f32(ayaw, &sa, &ca);
  const double cx = (double)ex + (double)wb * ce, cy = (double)ey + (double)wb * se;
  const double rx = (double)ax - cx, ry = (double)ay - cy;
  const double HEx = hEx, HEy = hEy, HL = hl, HW = hw;
  const double rax = rx * ce + ry * se, ray = -rx * se + ry * ce;     // agent centre in the ego frame
  const double rbx = rx * ca + ry * sa, rby = -rx * sa + ry * ca;     // the same offset in the agent frame
  const double c = fabs(ce * ca + se * sa), s = fabs(sa * ce - ca * se);
  const bool sep = (fabs(rax) > HEx + HL * c + HW * s) | (fabs(ray) > HEy + HL * s + HW * c) |
                   (fabs(rbx) > HL + HEx * c + HEy * s) | (fabs(rby) > HW + HEx * s + HEy * c);
  if (!sep) return 0u;
  double best = 1.0e300;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const double sx = (q & 1) ? 1.0 : -1.0, sy = (q & 2) ? 1.0 : -1.0;
    double wx = rx + sx * HL * ca - sy * HW * sa, wy = ry + sx * HL * sa + sy * HW * ca;     // agent corner vs ego box
    best = fmin(best, pt_box_d2_f64(wx * ce + wy * se, -wx * se + wy * ce, HEx, HEy));
    wx = -rx + sx * HEx * ce - sy * HEy * se; wy = -ry + sx * HEx * se + sy * HEy * ce;      // ego corner vs agent box
    best = fmin(best, pt_box_d2_f64(wx * ca + wy * sa, -wx * sa + wy * ca, HL, HW));
  }
  return (uint32_t)llrint(fmin(sqrt(best), 8000.0) * 1000.0);
}

__device__ __forceinline__ bool obb_hit(float rx, float ry, float c, float s, float hEx, float hEy, float hl, float hw) {
  float ac = fabsf(c), as = fabsf(s);
  float rox = fmaf(rx, c, ry * s);
  float roy = fmaf(ry, c, -rx * s);
  bool sep = (fabsf(rx) > hEx + fmaf(hl, ac, hw * as)) | (fabsf(ry) > hEy + fmaf(hl, as, hw * ac)) |
             (fabsf(rox) > hl + fmaf(hEx, ac, hEy * as)) | (fabsf(roy) > hw + fmaf(hEx, as, hEy * ac));
  return !sep;
}

// Single MUFU forms.  __fdividef / __expf wrap the same MUFU.RCP / MUFU.EX2 in range guards (denormal divisor, result
// below 2^-126: 4 and 3 more instructions per call) that cannot fire for the arguments used here; inside the guards'
// dead range the results are bit-identical.
__device__ __forceinline__ float rcp_approx(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float ex2_approx(float x) {
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

// erfc(z), z >= 0, fractional error < 1.2e-7 in exact arithmetic (Chebyshev fit of Numerical Recipes' erfcc:
// t = 1/(1 + z/2), erfc = t exp(-z^2 + P9(t))); about 4e-6 relative in float32 because of the exponent's
// magnitude -- two orders below the 1e-4 parity tolerance.  17 instructions instead of erfcf's ~45.  This form (guarded
// __expf) serves the detail kernel; the summary kernel evaluates the same chain two at a time (erf_span2).
__device__ __forceinline__ float erfc_pos_fast(float z) {
  const float t = rcp_approx(fmaf(0.5f, z, 1.0f));      // 1 + z/2 >= 1: same bits as __fdividef(1, .)
  float p = 0.17087277f;
  p = fmaf(p, t, -0.82215223f);
  p = fmaf(p, t, 1.48851587f);
  p = fmaf(p, t, -1.13520398f);
  p = fmaf(p, t, 0.27886807f);
  p = fmaf(p, t, -0.18628806f);
  p = fmaf(p, t, 0.09678418f);
  p = fmaf(p, t, 0.37409196f);
  p = fmaf(p, t, 1.00002368f);
  p = fmaf(p, t, -1.26551223f);
  const float a = fmaf(-z, z, p);
  return t * __expf(a);
}

// Packed float32 (sm_100 FFMA2 / FADD2 / FMUL2): two IEEE operations in one issue slot, each lane bit-identical to the
// scalar FFMA / FADD / FMUL.  ptxas does not form them itself.  A scalar operand is broadcast without a move (f2).
__device__ __forceinline__ float2 f2(float v) { return make_float2(v, v); }
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ float2 add2(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 mul2(float2 a, float2 b) { return __fmul2_rn(a, b); }

// erf(b) - erf(a), a < b, from erfc(|a|) and erfc(|b|) of erfc_pos_fast's chain, the two chains packed into one.
// exp is one FMUL + MUFU.EX2 (flushes results below 2^-126 to zero): the summary kernel's cut-off keeps one end of every
// evaluated interval within 4.7, so a flushed far end (< 1e-38 against >= 3e-11) cannot change a bit of the factor.
// The last products are formed as the scalar chains' contractions formed them, so the result keeps their bits:
// erfc(|b|) = t.y * e.y rounded once, erfc(|a|) = t.x * e.x fused into both combinations.  A packed product of the two
// would round erfc(|a|) as well.
__device__ __forceinline__ float erf_span2(float a, float b) {
  const float2 z = make_float2(fabsf(a), fabsf(b));
  const float2 d = fma2(f2(0.5f), z, f2(1.0f));
  const float2 t = make_float2(rcp_approx(d.x), rcp_approx(d.y));
  float2 p = fma2(f2(0.17087277f), t, f2(-0.82215223f));
  p = fma2(p, t, f2(1.48851587f));
  p = fma2(p, t, f2(-1.13520398f));
  p = fma2(p, t, f2(0.27886807f));
  p = fma2(p, t, f2(-0.18628806f));
  p = fma2(p, t, f2(0.09678418f));
  p = fma2(p, t, f2(0.37409196f));
  p = fma2(p, t, f2(1.00002368f));
  p = fma2(p, t, f2(-1.26551223f));
  const float2 x = mul2(fma2(make_float2(-z.x, -z.y), z, p), f2(1.4426950216293334961f));
  const float2 e = make_float2(ex2_approx(x.x), ex2_approx(x.y));
  const float eb = __fmul_rn(t.y, e.y);
  return ((a > 0.0f) == (b > 0.0f)) ? fabsf(fmaf(t.x, e.x, -eb)) : __fsub_rn(fmaf(-t.x, e.x, 2.0f), eb);
}

// Collision probability of one gated step (collision_probability.py:94-122): Gaussian mass of the 3 obstacle
// points over the 3 axis-aligned ego boxes, divided by 3.  (mx, my) = obstacle position i-1 minus ego position i,
// (hx, hy) = half buffered length along yaw_i, (bx, by) = (L/3)(cos, sin theta_i), s2 = 1/(sqrt2 sigma_{x,y}).
// CUT (summary kernel): a factor whose standardised interval lies beyond 4.7 (erfc < 3e-11) contributes less than the
// 1e-10 that the comparison floor of 2e-7 can resolve and is skipped before any erfc is evaluated.  The detail kernel
// evaluates all nine terms: its per-step values feed first-index decisions of the reference's result dict
// (max_obst_risk_index = first maximum of harm x cp, hr.py:87-98), where a 1e-12 must not become an exact zero.
template <bool CUT = true>
__device__ __forceinline__ float cp_gauss_boxes(float mx, float my, float hx, float hy, float bx, float by, float2 s2,
                                                float L6, float W2) {
  constexpr float kFar = 4.7f;
  float prob = 0.0f;
  float fm = 0.0f;                 // obstacle point: centre, front, back
#pragma unroll 1
  for (int m = 0; m < 3; ++m) {
    const float uy = fmaf(fm, hy, my), ux = fmaf(fm, hx, mx);
    float fb = 0.0f;               // ego box: middle, front, rear
#pragma unroll 1
    for (int bb = 0; bb < 3; ++bb) {
      const float f = fb;
      fb = (bb == 0) ? 1.0f : -1.0f;
      if constexpr (CUT) {
        // both ends of an interval as one packed pair: (f b -+ half) - u, times s2 (the scalar code's contraction)
        const float2 y = mul2(add2(fma2(f2(f), f2(by), make_float2(-W2, W2)), f2(-uy)), f2(s2.y));   // y.x < y.y
        if (y.x > kFar || y.y < -kFar) continue;
        const float2 x = mul2(add2(fma2(f2(f), f2(bx), make_float2(-L6, L6)), f2(-ux)), f2(s2.x));
        if (x.x > kFar || x.y < -kFar) continue;
        const float py = erf_span2(y.x, y.y);
        const float px = erf_span2(x.x, x.y);
        prob = fmaf(0.25f * px, py, prob);
      } else {
        const float cyb = f * by, cxb = f * bx;
        const float ya = (cyb - W2 - uy) * s2.y, yb = (cyb + W2 - uy) * s2.y;     // ya < yb
        const float xa = (cxb - L6 - ux) * s2.x, xb = (cxb + L6 - ux) * s2.x;
        const float eya = erfc_pos_fast(fabsf(ya)), eyb = erfc_pos_fast(fabsf(yb));
        const float py = ((ya > 0.0f) == (yb > 0.0f)) ? fabsf(eya - eyb) : (2.0f - eya - eyb);
        const float exa = erfc_pos_fast(fabsf(xa)), exb = erfc_pos_fast(fabsf(xb));
        const float px = ((xa > 0.0f) == (xb > 0.0f)) ? fabsf(exa - exb) : (2.0f - exa - exb);
        prob = fmaf(0.25f * px, py, prob);
      }
    }
    fm = (m == 0) ? 1.0f : -1.0f;
  }
  return prob * (1.0f / 3.0f);
}

// ---- collision probability with a full 2x2 covariance (fo_metric_bundle_corr) ---------------------------------------
// Gauss-Legendre nodes (negative half) and weights of orders 6, 12 and 20, at offsets 0, 3 and 9.
static __constant__ double kBvnX[19] = {
    -0.9324695142031519, -0.6612093864662645, -0.2386191860831969,
    -0.9815606342467192, -0.9041172563704748, -0.7699026741943047, -0.5873179542866175, -0.3678314989981802,
    -0.1252334085114689,
    -0.993128599185095, -0.9639719272779138, -0.912234428251326, -0.8391169718222188, -0.7463319064601508,
    -0.636053680726515, -0.5108670019508271, -0.37370608871541955, -0.22778585114164507, -0.07652652113349734};
static __constant__ double kBvnW[19] = {
    0.17132449237917027, 0.3607615730481387, 0.46791393457269104,
    0.04717533638651141, 0.10693932599531907, 0.16007832854334642, 0.20316742672306573, 0.2334925365383546,
    0.2491470458134027,
    0.017614007139150893, 0.040601429800386446, 0.06267204833410879, 0.08327674157670471, 0.1019301198172407,
    0.1181945319615186, 0.1316886384491769, 0.1420961093183824, 0.14917298647260424, 0.15275338713072628};

// One out-of-line copy each of the float64 normal CDF and exp: bvn_upper evaluates them at seven and five sites.
static __device__ __noinline__ double bvn_phi(double x) { return normcdf(x); }
static __device__ __noinline__ double bvn_exp(double x) { return exp(x); }

// P(X > h, Y > k) of a standard bivariate normal with correlation r, |r| < 1: Genz's BVNU (Drezner-Wesolowsky with
// 6 / 12 / 20-point Gauss-Legendre by |r|, and the expansion around |r| = 1 above 0.925), float64.
__device__ __forceinline__ double bvn_upper(double h, double k, double r) {
  constexpr double kTwoPi = 6.283185307179586;
  const double ar = fabs(r);
  const int g0 = ar < 0.3 ? 0 : (ar < 0.75 ? 3 : 9), lg = ar < 0.3 ? 3 : (ar < 0.75 ? 6 : 10);
  double hk = h * k, bvn = 0.0;
  if (ar < 0.925) {
    // sinpi: the argument is at most pi/2, so sin's Payne-Hanek reduction (8 kB of code) is not needed
    const double hs = 0.5 * (h * h + k * k), asr = asin(r), asr_pi = asr * (0.5 / CUDART_PI);
#pragma unroll 1
    for (int i = 0; i < 2 * lg; ++i) {
      const double x = (i & 1) ? -kBvnX[g0 + (i >> 1)] : kBvnX[g0 + (i >> 1)];
      const double sn = sinpi(asr_pi * (x + 1.0));
      bvn += kBvnW[g0 + (i >> 1)] * bvn_exp((sn * hk - hs) / (1.0 - sn * sn));
    }
    return bvn * asr / (2.0 * kTwoPi) + bvn_phi(-h) * bvn_phi(-k);
  }
  if (r < 0.0) { k = -k; hk = -hk; }
  const double as = (1.0 - r) * (1.0 + r);
  double a = sqrt(as);
  const double bs = (h - k) * (h - k), c = (4.0 - hk) / 8.0, d = (12.0 - hk) / 16.0;
  bvn = a * bvn_exp(-0.5 * (bs / as + hk)) * (1.0 - c * (bs - as) * (1.0 - d * bs / 5.0) / 3.0 + c * d * as * as / 5.0);
  if (hk > -160.0) {
    const double b = sqrt(bs);
    bvn -= bvn_exp(-0.5 * hk) * sqrt(kTwoPi) * bvn_phi(-b / a) * b * (1.0 - c * bs * (1.0 - d * bs / 5.0) / 3.0);
  }
  a *= 0.5;
#pragma unroll 1
  for (int i = 0; i < 2 * lg; ++i) {
    const double x = (i & 1) ? -kBvnX[g0 + (i >> 1)] : kBvnX[g0 + (i >> 1)];
    const double xs = (a * (x + 1.0)) * (a * (x + 1.0)), rs = sqrt(1.0 - xs);
    bvn += a * kBvnW[g0 + (i >> 1)] *
           (bvn_exp(-bs / (2.0 * xs) - hk / (1.0 + rs)) / rs - bvn_exp(-0.5 * (bs / xs + hk)) * (1.0 + c * xs * (1.0 + d * xs)));
  }
  bvn = -bvn / kTwoPi;
  if (r > 0.0) return bvn + bvn_phi(-fmax(h, k));
  bvn = -bvn;
  if (k > h) bvn += h < 0.0 ? bvn_phi(k) - bvn_phi(h) : bvn_phi(-h) - bvn_phi(-k);
  return bvn;
}

// Mass of a standard bivariate normal with correlation r over [a1, b1] x [a2, b2] (a < b), float64.  The four corners
// are combined on the tails: a coordinate whose interval lies mostly below the mean is reflected (r changes sign), so a
// box far from the mean is a difference of small upper-orthant masses and keeps its relative accuracy.  NaN unless
// |r| < 1 (a covariance that is not positive definite).
static __device__ __noinline__ double bvn_rect(double a1, double b1, double a2, double b2, double r) {
  if (!(fabs(r) < 1.0)) return CUDART_NAN;
  if (a1 + b1 < 0.0) { const double t = a1; a1 = -b1; b1 = -t; r = -r; }
  if (a2 + b2 < 0.0) { const double t = a2; a2 = -b2; b2 = -t; r = -r; }
  double p = 0.0;
#pragma unroll 1
  for (int q = 0; q < 4; ++q) {
    const double u = bvn_upper((q & 1) ? b1 : a1, (q & 2) ? b2 : a2, r);
    p += (q == 0 || q == 3) ? u : -u;
  }
  return p;
}

// cp_gauss_boxes with the correlated covariance s3 = (1/sigma_x, 1/sigma_y, rho, 0) of the state (fo_agents_pack_corr):
// the same nine box x point terms and the same float32 box limits, each term the float64 rectangle mass.  No cut-off:
// the 4.7-sigma rule of the diagonal path bounds each axis factor of a product, which a correlated mass is not.
__device__ __forceinline__ float cp_bvn_boxes(float mx, float my, float hx, float hy, float bx, float by, float4 s3,
                                              float L6, float W2) {
  const double isx = s3.x, isy = s3.y;
  double prob = 0.0;
  float fm = 0.0f;                 // obstacle point: centre, front, back
#pragma unroll 1
  for (int m = 0; m < 3; ++m) {
    const float uy = fmaf(fm, hy, my), ux = fmaf(fm, hx, mx);
    float fb = 0.0f;               // ego box: middle, front, rear
#pragma unroll 1
    for (int bb = 0; bb < 3; ++bb) {
      const float cyb = fb * by, cxb = fb * bx;
      fb = (bb == 0) ? 1.0f : -1.0f;
      prob += bvn_rect((double)(cxb - L6 - ux) * isx, (double)(cxb + L6 - ux) * isx, (double)(cyb - W2 - uy) * isy,
                       (double)(cyb + W2 - uy) * isy, (double)s3.z);
    }
    fm = (m == 0) ? 1.0f : -1.0f;
  }
  // the inclusion-exclusion can leave -1e-20 where the mass is 0: the result is +0 there (the summary kernel's maximum
  // compares bit patterns), and a NaN (not positive definite) stays NaN
  return (float)(prob > 0.0 ? prob / 3.0 : (prob == prob ? 0.0 : prob));
}

// LR4S angle coefficient, logistic_regression.py:35-42 (angles are NOT wrapped)
__device__ __forceinline__ float lr4s_coef(float ang, float side, float rear) {
  const float ta = 0.78539816339744830962f, tb = 2.35619449019234492885f;
  float c = rear;
  if ((ang >= ta && ang < tb) || (ang <= -ta && ang > -tb)) c = side;
  if (ang > -ta && ang < ta) c = 0.0f;
  return c;
}

// LR4S impact-angle coefficients of ego and obstacle (logistic_regression.py:35-48, harm_model.py:81-105); one copy per
// kernel (atan2f is ~100-150 instructions, the harm logits are needed at several inlined sites, and the kernels sit next
// to a 32 kB instruction cache: they are instruction-cache-bound, not call-bound).  ptxas lays a kernel's out-of-line
// helpers out in the order of their mangled names, so a rename can move this one and every call offset with it.
static __device__ __noinline__ float2 lr4s_coefs(float dyr, float dxr, float th, float psi, float side, float rear) {
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

// ---- BE (be.py:66-193) shared by the summary kernels: warp-cooperative bisection on a re-timed ego path -----
// The helpers are out of line (one copy per kernel).  Their view of the staged ego trajectory is a set of BYTE OFFSETS
// into the kernel's dynamic shared memory, and the few kernel arguments they need travel by value: pointers and a
// `const MetricKArgs&` would reach a noinline function as generic addresses (LD.E plus a uniform-register pair per access
// instead of LDS / a register).
#ifndef FO_BE_BUCKETS
#define FO_BE_BUCKETS 64
#endif
constexpr int kBeBuckets = FO_BE_BUCKETS;   // arc-length -> state-index lookup used by the interpolation
struct BeView {
  uint32_t egoA;   // float4 [T] (x, y, cos theta, sin theta)
  uint32_t egoB;   // float2 [T] (theta, v)
  uint32_t dist;   // float [T] cumulative chord length (be.py:99)
  uint32_t inv;    // uint8 [kBeBuckets + 1] last state index with dist <= b * dmax / kBeBuckets
  uint32_t seg;    // float4 [T] (SEG variants only): per segment j -> j + 1 the slopes ((x1-x0) inv, (y1-y0) inv, (th1-th0) inv, 0),
                   // inv = 1 / (dist[j+1] - dist[j]) -- the products be_bisect would form per lane and probe, formed once
};
struct BeConst {
  const float4* s0;   // agent-major states of the table
  int T, Tp;
  float dt, wb, hEx, hEy;
};
__device__ __forceinline__ BeConst be_const(const MetricKArgs& k) {
  return BeConst{k.tab.s0, k.T, k.Tp, k.dt, k.veh.wb, k.veh.hEx, k.veh.hEy};
}

template <bool SEG>
static __device__ __noinline__ void be_prepare(const BeView v, int T, int lane) {
  extern __shared__ __align__(16) unsigned char fo_dyn_smem[];
  const float4* const egoA = reinterpret_cast<const float4*>(fo_dyn_smem + v.egoA);
  const float2* const egoB = reinterpret_cast<const float2*>(fo_dyn_smem + v.egoB);
  float4* const seg = reinterpret_cast<float4*>(fo_dyn_smem + v.seg);
  float* const dist = reinterpret_cast<float*>(fo_dyn_smem + v.dist);
  uint8_t* const inv = fo_dyn_smem + v.inv;
  float carry = 0.0f;
#pragma unroll 1
  for (int i0 = 0; i0 < T; i0 += 32) {
    const int i = i0 + lane;
    float seg = 0.0f;
    if (i >= 1 && i < T) {
      float4 p = egoA[i], q = egoA[i - 1];
      seg = sqrtf((p.x - q.x) * (p.x - q.x) + (p.y - q.y) * (p.y - q.y));
    }
    float sc = seg;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      float t = __shfl_up_sync(kFull, sc, o);
      if (lane >= o) sc += t;
    }
    if (i < T) dist[i] = carry + sc;
    carry += __shfl_sync(kFull, sc, 31);
  }
  __syncwarp();
  if (SEG) {
#pragma unroll 1
    for (int j = lane; j < T - 1; j += 32) {
      const float4 A0 = egoA[j], A1 = egoA[j + 1];
      const float inv = 1.0f / (dist[j + 1] - dist[j]);     // a zero-length segment is never selected by the lookup
      seg[j] = make_float4((A1.x - A0.x) * inv, (A1.y - A0.y) * inv, (egoB[j + 1].x - egoB[j].x) * inv, 0.0f);
    }
  }
  const float bw = dist[T - 1] / (float)kBeBuckets;
#pragma unroll 1
  for (int b = lane; b <= kBeBuckets; b += 32) {
    const float q = (b == kBeBuckets) ? CUDART_INF_F : (float)b * bw;
    int lo_j = 0, hi_j = T - 1;
    while (lo_j < hi_j) {
      const int mid = (lo_j + hi_j + 1) >> 1;
      if (dist[mid] <= q) lo_j = mid; else hi_j = mid - 1;
    }
    inv[b] = (uint8_t)lo_j;
  }
  __syncwarp();
}

// lanes = time steps.  v_new[0] = v0, v_new[k+1] = max(v1 - d k dt, 0) (be.py:109); dist_new[i] = dt sum_{k<i} v_new[k]
// (be.py:113) in closed form: the clipped arithmetic series has floor(v1 / (d dt)) + 1 positive terms.  dist_new is
// non-decreasing in i, so scipy interp1d's bounds_error (be.py:117-124) fires iff its LAST element overruns.
__device__ __forceinline__ float be_arclen(float dt, float v0, float v1, float step, float mpos, int i) {
  const float m = fminf((float)(i - 1), mpos);
  return (i == 0) ? 0.0f : dt * (v0 + fmaf(m, v1, -0.5f * step * m * (m - 1.0f)));
}

// number of positive terms of the clipped series at the probe step = deceleration * dt; step in [4e-4, 0.5]:
// v1 * rcp == __fdividef(v1, step) bit for bit
__device__ __forceinline__ float be_mpos(float v1, float step) {
  return (step > 0.0f) ? fmaxf(floorf(v1 * rcp_approx(step)) + 1.0f, 0.0f) : 1.0e9f;
}

// Re-timed ego reference point (x, y) and heading (sin, cos) of step i at the probe (step, mpos) (be.py:109-130).
struct BePose {
  float x, y, s, c;
};
template <bool SEG>
__device__ __forceinline__ BePose be_pose(const BeView& v, int T, float dt, float v0, float v1, float inv_w, float step,
                                          float mpos, int i) {
  extern __shared__ __align__(16) unsigned char fo_dyn_smem[];
  const float4* const egoA = reinterpret_cast<const float4*>(fo_dyn_smem + v.egoA);
  const float2* const egoB = reinterpret_cast<const float2*>(fo_dyn_smem + v.egoB);
  const float* const dist = reinterpret_cast<const float*>(fo_dyn_smem + v.dist);
  const uint8_t* const inv_tab = fo_dyn_smem + v.inv;
  const float4* const seg = reinterpret_cast<const float4*>(fo_dyn_smem + v.seg);
  const float q = be_arclen(dt, v0, v1, step, mpos, i);
  // numpy.interp: j = last index with dist[j] <= q.  The bucket of q brackets it: j0 = inv[b] (stepped one bucket
  // down when float32 rounding of the bucket index put it too high), j1 = inv[b + 1]; a bisection of [j0, j1] --
  // most buckets hold at most one state -- and a final upward check for a q that rounded across the bucket's end
  int b = min(__float2int_rd(q * inv_w), kBeBuckets - 1);
  int j = inv_tab[b];
  if (dist[j] > q) { b = max(b - 1, 0); j = inv_tab[b]; }
  int jh = inv_tab[b + 1];
  while (j < jh) {
    const int mid = (j + jh + 1) >> 1;
    if (dist[mid] <= q) j = mid; else jh = mid - 1;
  }
  while (j < T - 1 && dist[j + 1] <= q) ++j;
  const float dj = dist[j];
  const float4 A0 = egoA[j];
  float xn = A0.x, yn = A0.y, tn = egoB[j].x;
  if (j != T - 1 && dj != q) {
    const float wq = q - dj;
    if (SEG) {
      const float4 sl = seg[j];
      xn = fmaf(sl.x, wq, A0.x);
      yn = fmaf(sl.y, wq, A0.y);
      tn = fmaf(sl.z, wq, tn);
    } else {
      const float4 A1 = egoA[j + 1];
      const float inv = 1.0f / (dist[j + 1] - dj);
      xn = fmaf((A1.x - A0.x) * inv, wq, A0.x);
      yn = fmaf((A1.y - A0.y) * inv, wq, A0.y);
      tn = fmaf((egoB[j + 1].x - tn) * inv, wq, tn);
    }
  }
  BePose p;
  p.x = xn;
  p.y = yn;
  __sincosf(tn, &p.s, &p.c);
  return p;
}

// the agent's state s0 at that step against the ego box at the re-timed pose (be.py:181)
__device__ __forceinline__ bool be_hit(const BeConst& k, const BePose& p, const float4 s0, float hl, float hw) {
  const float dx = (s0.x - p.x) - k.wb * p.c;
  const float dy = (s0.y - p.y) - k.wb * p.s;
  const float rx = fmaf(dx, p.c, dy * p.s), ry = fmaf(dy, p.c, -dx * p.s);
  const float c = fmaf(p.c, s0.z, p.s * s0.w), s = fmaf(s0.w, p.c, -s0.z * p.s);
  return obb_hit(rx, ry, c, s, k.hEx, k.hEy, hl, hw);
}

// BE of one pair: returns (required constant deceleration, number of probes as int bits); the deceleration is NaN
// when the re-timed path overruns the planned one (the reference raises, be.py:117-124).
// floor_rcd (team shape of the summary kernel; negative = off): the caller keeps only the MAXIMUM over a trajectory's
// pairs.  The bracket [lo, hi] only shrinks and the result is its last midpoint, so once hi <= floor_rcd this pair
// cannot raise the maximum and the bisection stops -- provided no later probe could overrun the planned path:
// dist_new[T-1] falls with the deceleration, the smallest deceleration the rest of the bisection can probe is the end
// of its all-miss branch, and that one is checked (with a margin for the float32 closed form; inside the margin the
// bisection simply runs on).
template <bool SEG>
static __device__ __noinline__ float2 be_bisect(const BeConst k, const BeView v, int a, int n_states, float hl, float hw,
                                                float lo0, int lane, float floor_rcd) {
  extern __shared__ __align__(16) unsigned char fo_dyn_smem[];
  const float2* const egoB = reinterpret_cast<const float2*>(fo_dyn_smem + v.egoB);
  const float* const dist = reinterpret_cast<const float*>(fo_dyn_smem + v.dist);
  const int T = k.T;
  const int nA = min(T, n_states);
  const float v0 = egoB[0].y, v1 = egoB[T > 1 ? 1 : 0].y;
  const float dmax = dist[T - 1];
  const float inv_w = dmax > 0.0f ? (float)kBeBuckets / dmax : 0.0f;
  // the agent's states do not depend on the probe: the first two 32-step chunks stay in registers for the whole
  // bisection (covers T <= 64, i.e. every horizon the reference uses), later chunks are re-read per probe
  const float4* sa = k.s0 + (size_t)a * k.Tp;
  const float4 pre0 = (lane < nA) ? __ldg(sa + lane) : make_float4(0, 0, 1, 0);
  const float4 pre1 = (32 + lane < nA) ? __ldg(sa + 32 + lane) : make_float4(0, 0, 1, 0);
  float lo = lo0, hi = 5.0f, cur = 0.0f;
  int probes = 0;
#pragma unroll 1
  for (int it = 0; it < 10; ++it) {
    cur = 0.5f * (lo + hi);
    ++probes;
    const float step = cur * k.dt;
    const float mpos = be_mpos(v1, step);
    if (be_arclen(k.dt, v0, v1, step, mpos, T - 1) > dmax) return make_float2(CUDART_NAN_F, __int_as_float(probes));
    bool any_hit = false;
#pragma unroll 1
    for (int i0 = 0; i0 < nA && !any_hit; i0 += 32) {
      const int i = i0 + lane;
      bool hit = false;
      if (i < nA) {
        const BePose p = be_pose<SEG>(v, T, k.dt, v0, v1, inv_w, step, mpos, i);
        hit = be_hit(k, p, (i0 == 0) ? pre0 : ((i0 == 32) ? pre1 : __ldg(sa + i)), hl, hw);
      }
      any_hit = __any_sync(kFull, hit);
    }
    if (nA > 0 && !any_hit) hi = cur; else lo = cur;   // be.py:74-77 (an agent that never exists counts as a hit)
    if (hi - lo < 0.1f) break;                         // be.py:79
    if (hi <= floor_rcd) {
      float h = hi, c = cur;
      for (int j = it + 1; j < 10; ++j) {              // the all-miss branch of what is left, same arithmetic
        c = 0.5f * (lo + h);
        h = c;
        if (h - lo < 0.1f) break;
      }
      const float st = c * k.dt;
      if (be_arclen(k.dt, v0, v1, st, be_mpos(v1, st), T - 1) < dmax * 0.99999f) break;
    }
  }
  return make_float2(cur, __int_as_float(probes));
}

// ---- BE of the summary kernels: the maximum over a trajectory's colliding pairs, one walk over one bisection tree ---
// Every pair starts from the bracket [lo0, 5] and follows the same midpoint and stop rules, so all probes of a
// trajectory are nodes of one binary tree, and each pair's bisection is one root-to-leaf path through it.  be_walk
// visits that tree depth first.  The re-timed ego path of a node is computed once, 32 steps at a time (lane = step),
// and every pair that reaches the node is tested against it, with the per-chunk early exit of be_bisect: the pairs
// that hit move to the right child (cur, hi), the others to the left child (lo, cur).  A pair sees the probes of its
// own bisection and decides each from the same operations on the same inputs (be_pose, be_hit), so it ends in the
// same leaf; only the maximum over the leaves leaves the kernel.
// Floor: the maximum so far.  A pending node whose bracket lies at or below it cannot raise it (a result is the last
// midpoint, inside the bracket) and is dropped -- provided no probe below it could overrun the planned path:
// dist_new[T-1] falls with the deceleration, the smallest deceleration below the node is the end of its all-miss
// branch, and that one is checked with a margin for the float32 closed form (inside the margin the walk goes on).
// The hit child is visited first: high decelerations raise the floor soonest.  A range error ends the walk (the
// outputs are NaN, the trajectory invalid).
// k.s0 / prm: the tile's first agent; list: byte offset of the tile's pair list (agent-in-tile indices, reordered in
// place).  Pending nodes sit one per lane (at most one per depth, depth <= 10): no local memory.
// Used by the one-warp throughput shape.  The team (latency) shape keeps one be_bisect per pair: there a warp holds one
// or two pairs, and the walk's per-node loads of the pair parameters and states lengthen the critical path (DESIGN.md 5.1).
struct BeWalk {
  float rcd;                       // maximum of the floor and the leaves' decelerations
  bool range;                      // a probe overran the planned path (be.py:117-124)
  unsigned tests, nodes, chunks;   // STATS: pair tests (probes of be_bisect), nodes visited, ego-path chunks computed
};
template <bool STATS>
static __device__ __noinline__ BeWalk be_walk(const BeConst k, const AgentParams* prm, const BeView v, uint32_t list, int n,
                                              float lo0, float rcd, int lane) {
  extern __shared__ __align__(16) unsigned char fo_dyn_smem[];
  uint16_t* const lst = reinterpret_cast<uint16_t*>(fo_dyn_smem + list);
  const float2* const egoB = reinterpret_cast<const float2*>(fo_dyn_smem + v.egoB);
  const float* const dist = reinterpret_cast<const float*>(fo_dyn_smem + v.dist);
  const int T = k.T;
  const float v0 = egoB[0].y, v1 = egoB[T > 1 ? 1 : 0].y;
  const float dmax = dist[T - 1];
  const float inv_w = dmax > 0.0f ? (float)kBeBuckets / dmax : 0.0f;
  BeWalk r;
  r.range = false;
  if (STATS) r.tests = r.nodes = r.chunks = 0u;
  float lo = lo0, hi = 5.0f;
  int b = 0, e = n, d = 0;               // node: bracket, its pairs lst[b, e), probes above it
  float st_lo = 0.0f, st_hi = 0.0f;      // lane j: pending node j
  int st_n = 0, sp = 0;
  bool below = false;                    // the node lies at or below the floor: is it safe to drop?
  for (;;) {
    // the probe of the node, or (below) the end of its all-miss branch; one closed-form path length serves both tests
    float cur = 0.5f * (lo + hi);
    if (below)
      for (int j = d + 1; j < 10 && !(cur - lo < 0.1f); ++j) cur = 0.5f * (lo + cur);
    const float step = cur * k.dt;
    const float mpos = be_mpos(v1, step);
    const float len = be_arclen(k.dt, v0, v1, step, mpos, T - 1);
    bool pop = true;
    if (below) {
      below = false;
      pop = len < dmax * 0.99999f;       // dropped; otherwise visited next time round
    } else {
      if (len > dmax) { r.range = true; break; }
      if (STATS) { ++r.nodes; r.tests += (unsigned)(e - b); }
      int m = e;                         // lst[b, m): no hit so far
#pragma unroll 1
      for (int i0 = 0; m > b; i0 += 32) {
        const int i = i0 + lane;
        const BePose p = be_pose<true>(v, T, k.dt, v0, v1, inv_w, step, mpos, i);
        if (STATS) ++r.chunks;
        bool more = false;               // a pair without a hit has steps after this chunk
#pragma unroll 1
        for (int s = b; s < m;) {
          const int al = lst[s];
          const int4 pa = __ldg(reinterpret_cast<const int4*>(prm + al));
          const int nA = min(T, pa.x);
          bool hit = nA == 0;            // be.py:74-77 (an agent that never exists counts as a hit)
          if (i < nA) hit = be_hit(k, p, __ldg(k.s0 + al * k.Tp + i), __int_as_float(pa.z), __int_as_float(pa.w));
          if (__any_sync(kFull, hit)) {  // to the hit end of the node's pairs
            --m;
            if (lane == 0) { lst[s] = lst[m]; lst[m] = (uint16_t)al; }
            __syncwarp();
          } else {
            more |= nA > i0 + 32;
            ++s;
          }
        }
        if (!more) break;
      }
      // children: misses lst[b, m) with (lo, cur), hits lst[m, e) with (cur, hi).  A child at the stop rule (be.py:79)
      // or after the tenth probe is a leaf: its pairs' result is cur.  Pushed left first: the hit child is popped first.
      ++d;
#pragma unroll 1
      for (int h = 0; h < 2; ++h) {
        const float cl = h ? cur : lo, ch = h ? hi : cur;
        const int cb = h ? m : b, ce = h ? e : m;
        if (cb < ce) {
          if (ch - cl < 0.1f || d == 10) {
            rcd = fmaxf(rcd, cur);
          } else {
            if (lane == sp) { st_lo = cl; st_hi = ch; st_n = cb | ce << 9 | d << 18; }
            ++sp;
          }
        }
      }
    }
    if (pop) {
      if (sp == 0) break;
      --sp;
      lo = __shfl_sync(kFull, st_lo, sp);
      hi = __shfl_sync(kFull, st_hi, sp);
      const int nd = __shfl_sync(kFull, st_n, sp);
      b = nd & 0x1ff; e = (nd >> 9) & 0x1ff; d = nd >> 18;
      below = hi <= rcd;
    }
  }
  r.rcd = rcd;
  return r;
}

// one zeroed-per-launch device counter (trajectory claims of the persistent kernels), see fo_metric_sweep.cu
unsigned int* claim_slot(cudaStream_t st);

// The metric sets with instantiations of their own; any other set is read from MetricKArgs::mmask at run time (MASK 0).
constexpr uint32_t kAllMetrics = FO_M_CP | FO_M_DCE | FO_M_TTC | FO_M_HR | FO_M_BE | FO_M_TTCE | FO_M_WTTC;
constexpr uint32_t kDefaultMetrics = kAllMetrics & ~FO_M_BE;   // occlusion.yaml:12-18

// f(std::integral_constant<uint32_t, MASK>) with the MASK the kernels are instantiated for when mmask is asked for
template <class F>
int with_mask(uint32_t mmask, F&& f) {
  if (mmask == kAllMetrics) return f(std::integral_constant<uint32_t, kAllMetrics>{});
  if (mmask == kDefaultMetrics) return f(std::integral_constant<uint32_t, kDefaultMetrics>{});
  return f(std::integral_constant<uint32_t, 0u>{});
}

constexpr int kMaxDev = 64;   // devices with per-device host state (claim slots, function attributes)

// Persistent launch of one metric-kernel instantiation: as many CTAs of `threads` threads as fit on the device, each
// owning traj_per_cta trajectories at a time.  When one wave does not cover k.N, the trajectories are claimed from a
// device counter (their cost varies several-fold), unless static_stride: then the CTAs stride over them.
template <auto KERNEL, class... Extra>
int launch_persistent(const MetricKArgs& k, int num_sms, int threads, int traj_per_cta, size_t smem, bool static_stride,
                      cudaStream_t st, const Extra&... extra) {
  // the opt-in shared-memory size is a per-device function attribute: remember what each device has been given
  static std::atomic<size_t> configured[kMaxDev];
  int dev = 0;
  FO_CUDA_TRY(cudaGetDevice(&dev));
  const bool tracked = dev >= 0 && dev < kMaxDev;
  if (!tracked || smem > configured[dev].load(std::memory_order_acquire)) {
    FO_CUDA_TRY(cudaFuncSetAttribute(KERNEL, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (tracked) configured[dev].store(smem, std::memory_order_release);
  }
  int per_sm = 1;
  FO_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, KERNEL, threads, smem));
  if (per_sm < 1) per_sm = 1;
  const int full = num_sms * per_sm;
  const int need = (k.N + traj_per_cta - 1) / traj_per_cta;
  const int grid = need < full ? need : full;
  MetricKArgs kk = k;
  kk.claim = (k.N > grid * traj_per_cta && !static_stride) ? claim_slot(st) : nullptr;
  if (kk.claim) FO_CUDA_TRY(cudaMemsetAsync(kk.claim, 0, sizeof(unsigned int), st));
  KERNEL<<<grid, threads, smem, st>>>(kk, extra...);
  count_launch();
  FO_CUDA_TRY(cudaGetLastError());
  return FO_OK;
}

int launch_metric_detail(const MetricKArgs& k, int num_sms, cudaStream_t st);
int launch_metric_sweep(const MetricKArgs& k, int num_sms, cudaStream_t st);
// Batch of independent problems (fo_metric_batch): the trajectories of one launch belong to problems with their own
// agent tables and ego vehicles.  A launch sees the problems of one shape class; `first` numbers their trajectories consecutively.  The
// table pointers are resolved on the host (agent_table_view of the problem's table in the arena): the kernel loads them
// and does no address arithmetic of its own per trajectory.
struct __align__(16) BatchProb {
  const float4* t0;
  const float* tv;
  const float4* aw;
  const float* avw;
  const float4* s0;
  const float4* s1;
  const float2* s2;
  const AgentParams* prm;
  int first;            // index of the problem's first trajectory within the launch
  int row0;             // its row in ego / valid / summary / flags
  int A, Tp, Ap;        // agents, table stride, agents padded to 32
  int lg;               // log2 of the agents held by one warp (team shape)
  EgoConst veh;         // the problem's ego vehicle
  const float4* s3;     // correlated tables (fo_metric_batch_corr): the s3 section (agent_corr_view); NULL otherwise
};
static_assert(sizeof(BatchProb) == 128, "eight 16-byte loads");
struct BatchView {
  const int* first;     // [P] BatchProb::first, strictly increasing (problems without trajectories are left out)
  const BatchProb* prob;
  int P;
};
// the last p in [0, P) with first[p] <= n (first strictly increasing, first[0] <= n)
__device__ __forceinline__ int find_problem(const int* first, int P, int n) {
  int lo = 0, hi = P - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (__ldg(first + mid) <= n) lo = mid; else hi = mid - 1;
  }
  return lo;
}
// Batch of independent problems with detail outputs (fo_metric_batch_detail): one launch over all rows [0, n_traj).
// Besides the table pointers the detail kernel and its helpers read, a descriptor holds the base of the problem's pair /
// step block (NULL when that output is not requested); all resolved on the host.
struct __align__(16) DetailProb {
  const float4* t0;
  const float* tv;
  const float4* s0;
  const float4* s1;
  const float2* s2;
  const AgentParams* prm;
  const int32_t* orig;
  const float* tpsi;
  float* pair;          // [N_p, A_p, FO_PAIR_K]
  float* step;          // [N_p, A_p, T-1, FO_STEP_K]
  int row0;             // the problem's first row in ego / valid / summary / flags
  int A, Tp, Ap;        // agents, table stride, agents padded to 32
  EgoConst veh;         // the problem's ego vehicle
  uint32_t s3_off;      // correlated tables (fo_metric_batch_detail_corr): s3 = s0 + s3_off (float4 units); 0 otherwise
};
static_assert(sizeof(DetailProb) == 128, "eight 16-byte loads");
struct DetailView {
  const int* first;     // [P] DetailProb::row0, strictly increasing (problems without trajectories are left out); the
                        // correlated kernel numbers its trajectories within the launch instead, as BatchView::first
  const DetailProb* prob;
  int P;
};
int launch_metric_batch_detail(const MetricKArgs& k, int num_sms, const DetailView& bv, cudaStream_t st);
// First valid row per problem (fo_metric_batch_select): one launch's state besides its BatchView.  The launch's
// descriptors are sorted by N_p in descending order, so the problems with a row of rank j are a prefix of them; claims
// run rank-major, and the ranks split into segments over which that prefix is the same.
struct SelectView {
  const int4* seg;      // [S] (first claim, first rank, active descriptors, 0) of each segment, in rank order
  const int* out;       // [descriptors] the problem index of each descriptor (its entry of selected)
  int32_t* selected;    // [n_problems] smallest rank whose row completed valid; initialised to N_p
  int S;
};
// summary kernel over one shape class of a batch (uni: the one-warp window-filter shape, W == 1); k.N = the class's
// trajectory count.  k.corr: the class's tables are correlated ones.  sv.selected != NULL: the select launch
// (fo_metric_batch_select_kernel), else fo_metric_batch[_corr]_kernel.
int launch_metric_batch(const MetricKArgs& k, int num_sms, int W, bool uni, const BatchView& bv, const SelectView& sv,
                        cudaStream_t st);
int lane_group_log2(int A);                                  // team shape: a warp holds 1 << lg agents
int pick_team_warps(int N, int T, int A, int num_sms);       // team size W (FO_TEAM_WARPS overrides)
int resident_teams(int W, int num_sms);                      // teams of W warps resident on the device at once

}  // namespace fo
