// b747_model_mx.cuh -- throughput ("f32") path of the B747 model step: one environment per thread,
// K fused RK4 substeps per launch with the state held in registers.
//
// Same block diagram as b747_model_f64.cuh (model_simple_step dll@0x16d0, SURVEY.md Appendix B),
// re-formulated for the FP32 issue rate of an SM (ncu r1a: the kernel is instruction-issue bound,
// 561 warp instructions per diagram pass, half of them compare/select/move work of the table
// searches and libm calls):
//  * aerodynamics, atmosphere, trigonometry, table look-ups, actuator and PIDs in float32;
//  * the attitude is carried as the pitch angle itself (theta' = wz) instead of the quaternion the
//    DLL integrates and re-normalises: for a pitch-only rotation the two are the same ODE
//    (q = (cos th/2, 0, 0, sin th/2)), and RK4 on either differs by O((wz h)^5) ~ 1e-20;
//  * the pitch-error chain -- theta, dvartheta = ref - theta, its integral, ITSE and the two
//    finite-difference Derivative blocks -- is kept in float64 (the observation and the CLASSIC reward
//    difference it over 5..10 ms, SURVEY.md 7 hard part 3); B200 issues DFMA at half the FFMA rate,
//    so these ~10 operations per pass are nearly free;
//  * every integrator state is accumulated in float64 across steps (y += h/6 * sum), the stage
//    values inside a step are float32;
//  * look-ups: the five tables are re-sampled on merged, sentinel-extended axes (b747_tables.h: one Mach,
//    one alpha, one altitude and one CYa axis instead of the DLL's eight breakpoint sets -- exact for a
//    bilinear interpolant) and stored as polynomial coefficients in the offsets from the interval's lower
//    breakpoint.  The current interval {bp, width} of every axis and the coefficients of the current cells
//    live in REGISTERS (TabCache); a pass validates them with one unsigned compare per axis and evaluates
//    the tables with packed FFMA2 (CYa + mz as coefficient pairs, the inner terms of CXa / dCm as pairs).  Shared
//    memory is touched only when an operand crossed a breakpoint (about once per model step and warp: CYa and
//    alpha cross their 0.1 / 0.6-deg intervals): the CYa walk is inline, the alpha-only and the full refill are
//    out-of-line functions (ncu r1d: the per-pass LDS.128 validation of the previous design drew 40 % of
//    the kernel's stall samples and 72 % of the shared-memory wavefront peak);
//  * sin/cos(theta), atan(wb/ub) and the ISA density power are short float32 polynomials
//    (b747_poly.h, generated + validated by tools/gen_poly.py) with libm fall-backs outside their
//    fitted ranges, evaluated at the major pass only: the three RK stages advance sin/cos by a rotation
//    and alpha by the asin of the normalised cross product of the body-velocity vectors (TrigMx), the
//    atmosphere by its derivative in h (AtmoMx); sin(alpha), cos(alpha) come from the body-axis velocity
//    components;
//  * the RK4 bookkeeping runs on register pairs with packed FFMA2, the weights as broadcast scalars;
//  * the transport delay (0.03 s = 3 steps), the Derivative and rate-limiter stamps are resolved
//    from the integer tick, so no time-stamp arithmetic is left in floating point;
//  * states that no observation/reward reads (ITAE, IAE, ISE; x and the altitude-loop PID unless the
//    configuration needs them) are not integrated.
#pragma once
#include <math.h>

#include "b747_common.cuh"
#include "b747_poly.h"
#include "b747_tables.h"

namespace b747 {

// packed FP32 FMA on a register pair (one FFMA2)
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }

__host__ __device__ constexpr double Pc(int i) {
  constexpr double a[kNP] = B747_P_INIT;
  return a[i];
}
template <int I>
struct PF { static constexpr float v = (float)Pc(I); };
#define PCF(i) (PF<(i)>::v)

// the ISA temperature ratio is clamped by the troposphere limits, so the density polynomial's
// fitted range always covers it
static_assert((Pc(16) - Pc(17) * Pc(19)) * Pc(127) > 0.70 && (Pc(16) - Pc(18) * Pc(19)) * Pc(127) < 1.01,
              "ISA temperature ratio leaves the range of the density polynomial (tools/gen_poly.py)");

// Look-up tables: re-gridded on merged axes by the host (b747_tables.h), staged in shared memory.
constexpr int kFastCells = ft::CELLS;

// Register-resident table state of one environment: current interval of each axis and current cells.
struct TabCache {
  float bM, wM, bA, wA, bH, wH, bC, wC;  // lower breakpoint and width of the current interval (alpha in radians)
  float k0, k1;                          // K_alpha = k0 + k1 dA on the current alpha interval
  // cells as coefficient PAIRS for packed FFMA2 evaluation, y = (c0 + c1 dM) + (c2 + c3 dM) d1 with d1 = dA / dC / dH:
  float2 pCM[4];                         // (CYa, mz) coefficient pairs k = 0..3 (the two tables share both operands)
  float2 cxA, cxB, dcA, dcB;             // CXa and dCm cells as (c3, c1) and (c2, c0): inner terms by one FFMA2
  uint32_t ix;                           // interval indices iM | iA << 5 | iH << 10 | iC << 13, kIxEmpty = none (read by the
                                         // refill only; persisted between launches in the spare bits of the tick word)
};

// float copies of the uniform tunables + folded constants (built on the host, b747_kernels_f32.cu)
// Manual switches of the diagram, resolved on the host against their thresholds (P148, P9, P149)
enum { SW_RL = 1, SW_SS = 2, SW_RP = 4, SW_SS_ON = 8 };
struct MP32 {
  float PID_SS[4];
  float P_m, g, kS_m, half_Sc_over_Iz;  // thrust / m0, g, P134 S / m0, P135 S c / Iz
  int sw;
};

struct RegsMx {
  double h, th, Vx, Vy, wz, ssi, ssf, dvi, itse;  // integrator states, accumulated in float64
  double csi, csf, x;                              // GEN only
  double d1_u;                                     // dvartheta at the last major step
  double vref, href, ep_return;
  double vartheta;                                 // current pitch reference (the DLL's `vartheta` param); registers only
  float df_x, df_y, rl_prev, deltaz, uh[4], sig_upid, d2_u, sig_vzh, tf_tp;
  float sumA[5];                                   // 1 + aero_err[k]
  double oscA[3], oscf[3];
  int tick, flags;
  uint32_t ep_idx;
  TabCache tc;                                     // look-up state (registers only; invalid at load: widths 0)
};

struct PassMx {
  double dv;
  double thd;  // folded pitch in float64 (trace only)
  float dvf;
  float th, V, alpha, Mach, CXa, CYa, mz, K_alpha, dCm, U_com, U_com_PID, deltaz_RP, vartheta_zh, td, rl_out;
  bool and_ss, and_cs;
};

// stage-4 (predictor) state values = what the DLL's `state`/integral signals show after a step
struct Stage4Mx { float h, Vx, Vy, wz, x; double dvi, itse; };

__device__ __forceinline__ float satf(float u, float lo, float hi) { return fminf(fmaxf(u, lo), hi); }
// single-instruction MUFU forms (operands here are far from the denormal range)
__device__ __forceinline__ float rsqrt_fast(float x) {
  float y;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float rcp_fast(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float ex2_fast(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ int sgnf(float x) { return (x > 0.f) - (x < 0.f); }

// ---- rare paths, kept out of line so that the pass loop stays small in the instruction cache ----
__device__ __noinline__ float atan2_far(float y, float x) { return atan2f(y, x); }

// alpha = -atan2(wb, ub) = atan(-wb/ub) for ub > 0
__device__ __forceinline__ float alpha_of(float wb, float ub) {
  const float q = -wb * rcp_fast(ub);
  if (ub > 0.f && fabsf(q) <= poly::ATAN_MAX) {
    const float z = q * q;
    float p = fmaf(poly::ATAN6, z, poly::ATAN5); p = fmaf(p, z, poly::ATAN4); p = fmaf(p, z, poly::ATAN3);
    p = fmaf(p, z, poly::ATAN2); p = fmaf(p, z, poly::ATAN1); p = fmaf(p, z, poly::ATAN0);
    return fmaf(q * z, p, q);
  }
  return atan2_far(-wb, ub);
}

// 0 <= d < w as ONE unsigned compare: a negative d has its sign bit set, NaN compares above every finite width
__device__ __forceinline__ bool axis_miss(float d, float w) { return __float_as_uint(d) >= __float_as_uint(w); }

// Walk from interval i to the one that holds u (or to the end of the axis; NaN stops at once); returns its record.
template <int OFF, int N>
__device__ __forceinline__ float4 axis_seek(const float4* __restrict__ sT, float u, int& i) {
  float4 q = sT[OFF + i];
  if (u < q.x) {
    while (i > 0) { --i; q = sT[OFF + i]; if (!(u < q.x)) break; }
  } else {
    while (u - q.x >= q.y && i < N - 1) { ++i; q = sT[OFF + i]; }
  }
  return q;
}
// first search of a launch: coarse index map of axis k (b747_tables.h), `lo`/`inv` = range the map resolves
template <int K>
__device__ __forceinline__ int axis_guess(const float4* __restrict__ sT, float u, float lo, float inv) {
  const int b = min(max((int)((u - lo) * inv), 0), ft::LUT_N - 1);
  return ((const unsigned char*)(sT + ft::LUT))[K * ft::LUT_N + b];
}

__device__ __forceinline__ float bilinear(const float4 c, float d0, float d1) {
  return fmaf(fmaf(c.w, d0, c.z), d1, fmaf(c.y, d0, c.x));
}
// two tables at once: three FFMA2 (sm_100 packed FP32; the scalar offsets ride as broadcast operands)
__device__ __forceinline__ float2 bilinear2(const float2 p[4], float d0, float2 d1) {
  const float2 d00 = make_float2(d0, d0);
  return fma2(fma2(p[3], d00, p[2]), d1, fma2(p[1], d00, p[0]));
}

// Cold paths.  An operand left its cached interval (or nothing is cached yet); interval indices move incrementally (an
// operand crosses into a NEIGHBOUR interval).  The cached record of an axis is always the one `ix` names, so cells and
// offsets stay consistent.
//  * Mach / alpha / h miss: their records and the three cells they address are reloaded.  ONE out-of-line copy, result
//    through memory, so that the four unrolled stage copies of the pass stay small in the instruction cache (ncu r1f:
//    the fully inlined form doubled the loop to 26 KB and tripled the no_instruction stalls).
//  * CYa miss -- the common case, CYa crosses its 0.1-wide intervals with every degree of alpha: a few inline
//    instructions move the interval and reload the CXa cell.
constexpr uint32_t kIxEmpty = 0xffffffffu;
struct TabMAH { float bM, wM, bA, wA, bH, wH, k0, k1; float4 cm0, cm1, cDC; uint32_t ix; };

__device__ __noinline__ void tab_refill_mah(const float4* __restrict__ sT, float Mach, float alpha, float h, float cy_gain,
                                            uint32_t ix, TabMAH* __restrict__ out) {
  int iM = ix & 31, iA = (ix >> 5) & 31, iH = (ix >> 10) & 7, iC = (ix >> 13) & 15;
  const bool empty = ix == kIxEmpty;
  // indices restored from HBM are only hints (the state may have been edited): keep them on their axes
  iM = min(iM, ft::NM - 1); iA = min(iA, ft::NA - 1); iH = min(iH, ft::NH - 1); iC = min(iC, ft::NC - 1);
  constexpr float rad = (float)Pc(21);
  if (empty) {
    iM = axis_guess<0>(sT, Mach, (float)ft::LUT_M_LO, (float)(ft::LUT_N / (ft::LUT_M_HI - ft::LUT_M_LO)));
    iA = axis_guess<1>(sT, alpha, (float)(ft::LUT_A_LO / rad), (float)(ft::LUT_N * rad / (ft::LUT_A_HI - ft::LUT_A_LO)));
    iH = axis_guess<2>(sT, h, (float)ft::LUT_H_LO, (float)(ft::LUT_N / (ft::LUT_H_HI - ft::LUT_H_LO)));
  }
  TabMAH t;
  const float4 qM = axis_seek<ft::AXM, ft::NM>(sT, Mach, iM);
  const float4 qA = axis_seek<ft::AXA, ft::NA>(sT, alpha, iA);
  const float4 qH = axis_seek<ft::AXH, ft::NH>(sT, h, iH);
  t.bM = qM.x; t.wM = qM.y; t.bA = qA.x; t.wA = qA.y; t.k0 = qA.z; t.k1 = qA.w; t.bH = qH.x; t.wH = qH.y;
  const float4* cMA = sT + ft::T_MA + 2 * (iA * ft::NM + iM);
  t.cm0 = cMA[0]; t.cm1 = cMA[1];
  t.cDC = sT[ft::T_HM + iM * ft::NH + iH];
  if (empty) {
    const float CYa = bilinear(make_float4(t.cm0.x, t.cm0.z, t.cm1.x, t.cm1.z), Mach - t.bM, alpha - t.bA) * cy_gain;
    iC = axis_guess<3>(sT, CYa, (float)ft::LUT_C_LO, (float)(ft::LUT_N / (ft::LUT_C_HI - ft::LUT_C_LO)));
  }
  t.ix = (uint32_t)iM | (uint32_t)iA << 5 | (uint32_t)iH << 10 | (uint32_t)iC << 13;
  *out = t;
}

// The common Mach / alpha / h miss: alpha alone crossed a breakpoint of its finely broken axis (0.6 deg intervals around
// the cruise incidence).  Only the alpha record and the (CYa, mz) cell change -- 13 words instead of the 21 of the full
// refill, one walk instead of three.  Out of line like the full refill (one copy for the four stage copies of the pass).
struct TabA { float bA, wA, k0, k1; float4 cm0, cm1; uint32_t ix; };

__device__ __noinline__ void tab_refill_alpha(const float4* __restrict__ sT, float alpha, uint32_t ix, TabA* __restrict__ out) {
  int iA = min((int)((ix >> 5) & 31), ft::NA - 1);
  const float4 qA = axis_seek<ft::AXA, ft::NA>(sT, alpha, iA);
  const float4* cMA = sT + ft::T_MA + 2 * (iA * ft::NM + (int)(ix & 31));
  TabA t;
  t.bA = qA.x; t.wA = qA.y; t.k0 = qA.z; t.k1 = qA.w;
  t.cm0 = cMA[0]; t.cm1 = cMA[1];
  t.ix = (ix & ~(31u << 5)) | (uint32_t)iA << 5;
  *out = t;
}

__device__ __forceinline__ void tab_update(const float4* __restrict__ sT, float Mach, float alpha, float h, float cy_gain,
                                           bool missMAH, TabCache& t, float& dM, float& dA, float& dH, float2& cm, float& dC) {
  if (missMAH) {
    if (!(axis_miss(dM, t.wM) | axis_miss(dH, t.wH)) && t.wA != 0.f) {
      TabA m;
      tab_refill_alpha(sT, alpha, t.ix, &m);
      t.bA = m.bA; t.wA = m.wA; t.k0 = m.k0; t.k1 = m.k1;
      t.pCM[0] = make_float2(m.cm0.x, m.cm0.y); t.pCM[1] = make_float2(m.cm0.z, m.cm0.w);
      t.pCM[2] = make_float2(m.cm1.x, m.cm1.y); t.pCM[3] = make_float2(m.cm1.z, m.cm1.w);
      t.ix = m.ix;
      dA = alpha - t.bA;
    } else {
      TabMAH m;
      tab_refill_mah(sT, Mach, alpha, h, cy_gain, t.ix, &m);
      t.bM = m.bM; t.wM = m.wM; t.bA = m.bA; t.wA = m.wA; t.bH = m.bH; t.wH = m.wH; t.k0 = m.k0; t.k1 = m.k1;
      t.pCM[0] = make_float2(m.cm0.x, m.cm0.y); t.pCM[1] = make_float2(m.cm0.z, m.cm0.w);
      t.pCM[2] = make_float2(m.cm1.x, m.cm1.y); t.pCM[3] = make_float2(m.cm1.z, m.cm1.w);
      t.dcA = make_float2(m.cDC.x, m.cDC.y); t.dcB = make_float2(m.cDC.z, m.cDC.w);
      t.ix = m.ix;
      dM = Mach - t.bM; dA = alpha - t.bA; dH = h - t.bH;
    }
    cm = bilinear2(t.pCM, dM, make_float2(dA, dA));
    cm.x *= cy_gain;
  }
  int iC = (t.ix >> 13) & 15;
  const float4 qC = axis_seek<ft::AXC, ft::NC>(sT, cm.x, iC);
  t.bC = qC.x; t.wC = qC.y;
  const float4 cx = sT[ft::T_MC + iC * ft::NM + (t.ix & 31)];
  t.cxA = make_float2(cx.x, cx.y); t.cxB = make_float2(cx.z, cx.w);
  dC = cm.x - t.bC;
  t.ix = (t.ix & 0x1fffu) | (uint32_t)iC << 13;
}

// Atmosphere of one model step: evaluated in full at the major pass, carried to the three minor passes by its first
// derivative in h.  Within a step the altitude moves by |Vy| h < 1 m against a density scale height of ~8 km, so the
// neglected second-order term is ~1e-9 relative (float32 rounds at 6e-8); only the step that crosses the ISA kinks
// (0 m, 11 km) sees a one-off slope error of ~1e-5 relative, on a force that acts for 10 ms.
struct AtmoMx { float h0, rho0, ia0, s_rho, s_ia; };

// Trigonometry of one model step: sin/cos of the (folded) pitch and the angle of attack are evaluated in full at the major
// pass and carried to the three minor passes by their exact increments -- the pitch moves by delta = wz h (<= a few 1e-2
// rad even for a tumbling airframe), so sin/cos follow by a rotation with short series for sin/cos(delta), and alpha by
// the angle between the body-velocity vectors of the two passes (asin of their normalised cross product).  Both are
// more accurate than re-evaluating the float32 polynomials (no argument rounding), and need no range checks.
struct TrigMx { float2 sc, cn; float thf, sgn, ub, wb, rV, alpha; double thd; };  // sc = (sin, cos), cn = (cos, -sin) of the major pass

// One pass over the diagram at a stage state.  stage: 0 major, 1/2 half steps, 3 full step.
// Passes 0 and 3 -- the ones whose pitch error is differenced by the Derivative blocks, observed and rewarded -- carry
// the pitch angle and the pitch error in float64 (th_d); the half-step passes only feed float32 RK4 sums and use th_f.
// TIER 0: canonical (LEAN) model; 1: + aero-disturbance gains (general layout, no altitude loop); 2: + the altitude loop (СУ PID)
// SW >= 0: the diagram's manual switches as a compile-time constant (the canonical env: SW_RP only); -1: read mp.sw
template <int TIER, int SW = -1>
__device__ __forceinline__ void pass32(const float4* __restrict__ sT, const MP32& mp, const DevCfg& c, int stage, int n,
                                       double th_d, float dth, TrigMx& tg, float vref_f, float t_f, float h, double h_d, float Vx,
                                       float Vy, float wz, float ssi, float ssf, double csi, double csf, RegsMx& r,
                                       AtmoMx& at, bool& memout_ss, bool& memout_cs, PassMx& o, float& f_h, float& f_Vx,
                                       float& f_Vy, float& f_wz, float& f_ssi, float& f_ssf, double& f_csi, double& f_csf,
                                       float& f_itse) {
  constexpr bool GEN = TIER >= 1, CS = TIER >= 2;
  const bool major = stage == 0;
  const bool dbl = stage == 0 || stage == 3;
  // attitude.  Beyond +-90 deg the DLL's pitch asin(sin(theta)) folds back: with k = round(theta/pi) and
  // r = theta - k*pi (two-constant Cody-Waite reduction) asin(sin(theta)) = (-1)^k r, and the DLL's sin/cos of the
  // folded pitch are sin(theta) and |cos(theta)| = cos(r).  Rare, cheap, and the polynomial covers the folded range.
  // The folded pitch is continuous in theta with slope sgn = (-1)^k, which is what the minor passes advance it with.
  float thf, sn, cs;
  double th_fold = th_d;
  static_assert(poly::SINCOS_MAX >= 1.57079632679f, "sin/cos polynomial must cover the unfolded pitch range");
  if (dbl) {
    thf = __double2float_rn(th_d);
    float sgn = 1.0f;
    if (fabsf(thf) > 1.57079632679f) {
      const double k = rint(th_d * 0.318309886183790671538);
      double rr = fma(-k, 3.141592653589793116, th_d);
      rr = fma(-k, 1.2246467991473532e-16, rr);
      const bool odd = ((int)k) & 1;
      th_fold = odd ? -rr : rr;
      sgn = odd ? -1.0f : 1.0f;
      thf = __double2float_rn(th_fold);
    }
    if (major) tg.sgn = sgn;
  }
  if (major) {
    const float z = thf * thf;
    float ps = fmaf(poly::SIN4, z, poly::SIN3); ps = fmaf(ps, z, poly::SIN2); ps = fmaf(ps, z, poly::SIN1); ps = fmaf(ps, z, poly::SIN0);
    float pc = fmaf(poly::COS4, z, poly::COS3); pc = fmaf(pc, z, poly::COS2); pc = fmaf(pc, z, poly::COS1); pc = fmaf(pc, z, poly::COS0);
    sn = fmaf(thf * z, ps, thf);
    cs = fmaf(z, pc, 1.0f);
    tg.sc = make_float2(sn, cs); tg.cn = make_float2(cs, -sn); tg.thf = thf; tg.thd = th_fold;
  } else {
    // increment of the folded pitch since the major pass: exact difference at the full step (the fold is continuous),
    // sgn * wz * h/2 at the half steps
    const float dl = dbl ? __double2float_rn(th_fold - tg.thd) : tg.sgn * dth;
    if (!dbl) {
      // a half step may cross the fold: asin(sin x) = max(min(x, pi - x), -pi - x) for |x| < pi.  The pitch error feeds
      // the derivative filter of the SS PID (gain Kd N ~ 390), so a kink missed for one pass would show in U_com_PID
      const float x = tg.thf + dl;
      thf = fmaxf(fminf(x, 3.14159274f - x), -3.14159274f - x);
    }
    const float d2 = dl * dl;
    const float sd = fmaf(dl * d2, fmaf(d2, 8.33333333e-3f, -0.166666667f), dl);
    const float cd = fmaf(d2, fmaf(d2, 4.16666667e-2f, -0.5f), 1.0f);
    // (sin, cos)(theta0 + dl) = (sin, cos) cd + (cos, -sin) sd: one packed multiply and one packed FMA
    const float2 cdd = make_float2(cd, cd), sdd = make_float2(sd, sd);
    const float2 t = __fmul2_rn(tg.cn, sdd);
    const float2 rot = fma2(tg.sc, cdd, t);
    sn = rot.x;
    cs = fabsf(rot.y);  // the folded pitch stays within +-90 deg: cos >= 0 (a half step may cross the fold)
  }
  o.th = thf;
  o.thd = th_fold;
  const float ub = fmaf(cs, Vx, sn * Vy);
  const float wb = fmaf(cs, Vy, -sn * Vx);
  const float V2 = fmaf(ub, ub, wb * wb);
  const float rV = rsqrt_fast(V2);
  const float V = V2 * rV;
  float alpha;
  if (major) {
    alpha = alpha_of(wb, ub);
    tg.ub = ub; tg.wb = wb; tg.rV = rV; tg.alpha = alpha;
  } else {
    // alpha = angle of (ub, -wb): sin(alpha - alpha0) = (wb0 ub - ub0 wb) / (V0 V), asin by its series (|x| <~ 0.1)
    const float x = fmaf(tg.wb, ub, -(tg.ub * wb)) * (tg.rV * rV);
    const float x2 = x * x;
    alpha = tg.alpha + fmaf(x * x2, fmaf(x2, 0.075f, 0.166666667f), x);
  }
  o.V = V; o.alpha = alpha;
  // ISA atmosphere: density rho0 (T/T0)^(g/(LR)-1) [* exp(g/R sat(11000-h)/T) above the tropopause] and 1/a
  float rho, ia;
  if (major) {
    const float hs = fminf(fmaxf(h, PCF(18)), PCF(17));
    const float T = fmaf(-hs, PCF(19), PCF(16));
    const float rT = rcp_fast(T);
    ia = rsqrt_fast(T * PCF(20));
    const float u = fmaf(T, PCF(127), -poly::RHO_CENTER);
    float pr = fmaf(poly::RHO6, u, poly::RHO5); pr = fmaf(pr, u, poly::RHO4); pr = fmaf(pr, u, poly::RHO3);
    pr = fmaf(pr, u, poly::RHO2); pr = fmaf(pr, u, poly::RHO1); pr = fmaf(pr, u, poly::RHO0);
    const float dh = PCF(130) - h;
    // the saturation makes the exponential exactly 1 below the tropopause: evaluated unconditionally (a third of the
    // environments start within 3 km of 11 km, a branch would diverge in most warps)
    rho = PCF(129) * pr * ex2_fast(fminf(fmaxf(dh, PCF(132)), PCF(131)) * (PCF(133) * 1.4426950408889634f) * rT);
    // d/dh: troposphere (T not clamped): rho' = -rho (g/(LR)-1) L / T, (1/a)' = (1/a) L / (2T);
    //       stratosphere (exponent not clamped): rho' = -rho (g/R) / T
    const bool tropo = (h > PCF(18)) & (h < PCF(17));
    const bool strato = (dh < PCF(131)) & (dh > PCF(132));
    const float kr = (tropo ? (PCF(128) - 1.0f) * PCF(19) : 0.f) + (strato ? PCF(133) : 0.f);
    at.h0 = h; at.rho0 = rho; at.ia0 = ia;
    at.s_rho = -rho * rT * kr;
    at.s_ia = tropo ? ia * rT * (0.5f * PCF(19)) : 0.f;
  } else {
    const float dlt = h - at.h0;
    rho = fmaf(at.s_rho, dlt, at.rho0);
    ia = fmaf(at.s_ia, dlt, at.ia0);
  }
  const float Mach = V * ia;
  o.Mach = Mach;
  // look-ups on the merged axes (b747_tables.h) from the register cache.  The cache is validated with the offsets
  // themselves (the CYa axis speculatively, from the cached CYa cell); the refill is rare and out of line.
  // The alpha axis is stored in radians (breakpoints / P21), so no conversion to degrees is needed.
  TabCache& tc = r.tc;
  const float cy_gain = GEN ? r.sumA[1] : 1.0f;
  float dM = Mach - tc.bM, dA = alpha - tc.bA, dH = h - tc.bH;
  float2 cm = bilinear2(tc.pCM, dM, make_float2(dA, dA));  // (CYa, mz)
  if (GEN) cm.x *= cy_gain;
  float dC = cm.x - tc.bC;
  const bool missMAH = axis_miss(dM, tc.wM) | axis_miss(dA, tc.wA) | axis_miss(dH, tc.wH);
  if (__builtin_expect(missMAH | axis_miss(dC, tc.wC), 0))
    tab_update(sT, Mach, alpha, h, cy_gain, missMAH, tc, dM, dA, dH, cm, dC);
  const float2 dMM = make_float2(dM, dM);
  const float2 ix = fma2(tc.cxA, dMM, tc.cxB), id = fma2(tc.dcA, dMM, tc.dcB);  // inner terms (c3 dM + c2, c1 dM + c0)
  const float CYa = cm.x;
  // cx = P126 CXa and dcm = P217 P150 dCm: the cells carry the diagram's gains (b747_tables.h)
  float mz = cm.y, cx = fmaf(ix.x, dC, ix.y), dcm = fmaf(id.x, dH, id.y);
  if (GEN) cx *= r.sumA[0];
  float Ka = fmaf(tc.k1, dA, tc.k0);
  if (GEN) { dcm *= r.sumA[3]; Ka *= r.sumA[4]; mz *= r.sumA[2]; }
  o.CYa = CYa; o.K_alpha = Ka; o.mz = mz;
  if (GEN) {  // the signals themselves are only read by observation layouts / exports of the general tiers
    o.CXa = cx * (float)(1.0 / Pc(126));
    o.dCm = dcm * (float)(1.0 / (Pc(217) * Pc(150)));
  }
  // aerodynamic + thrust acceleration in body axes, straight from the body velocity components:
  // drag/lift rotated by alpha with sin(alpha) = -wb/V, cos(alpha) = ub/V gives
  //   Fx = q S (c_x ub - CYa wb)/V + P,  Fy = q S (CYa ub + c_x wb)/V,  q S / V = rho V S / 2,  c_x = P126 CXa
  const float rV2 = rho * V2;
  const float kq = rV2 * (rV * mp.kS_m);
  const float Fx = fmaf(kq, fmaf(-CYa, wb, cx * ub), mp.P_m);
  const float Fy = kq * fmaf(cx, wb, CYa * ub);
  // actuator: transport delay (3 steps) -> discrete filter (every 5th tick) -> rate limiter -> saturation
  float td;
  if (stage == 0) td = n > 3 ? r.uh[1] : PCF(137);
  else if (stage == 3) td = n >= 3 ? r.uh[2] : PCF(137);
  else td = n >= 3 ? 0.5f * (r.uh[1] + r.uh[2]) : PCF(137);
  o.td = td;
  if (major && (n % 5) == 0) r.df_y = fmaf(r.df_x, PCF(140), PCF(141) * td);
  if (stage != 2) {  // the second half-step pass sees the same filter output, memory and dT as the first: o keeps its values
    float yv = r.df_y;
    if (!(major && n == 0)) {
      const float dT = stage == 1 ? 0.005f : 0.01f;
      yv = r.rl_prev + fminf(fmaxf(yv - r.rl_prev, dT * PCF(143)), dT * PCF(142));
    }
    o.rl_out = yv;
    o.deltaz_RP = satf(yv, PCF(145), PCF(144));
  }
  // СУ PID (altitude loop) -- only integrated when the configuration can close it.  Its output is the
  // pitch reference, which the СС PID differentiates with a gain of Kd*N ~ 390, so the whole
  // altitude-error chain is float64 (a float32 altitude quantises it at ~1e-5 rad).
  bool use_cs = false;
  double cs_pre = 0.0, cs_d = 0.0, e_h = 0.0, vzh_d = 0.0;
  if (CS) {
    use_cs = (r.flags & FL_USE_CTRL) && (1.f >= PCF(146));
    e_h = r.href - h_d;  // h_zh - h
    cs_d = (e_h * c.mp.PID_CS[2] - csf) * c.mp.PID_CS[3];
    cs_pre = e_h * c.mp.PID_CS[0] + csi + cs_d;
    vzh_d = fmin(fmax(cs_pre, Pc(4)), Pc(6));
    o.vartheta_zh = __double2float_rn(vzh_d);
  } else {
    o.vartheta_zh = 0.f;
  }
  // pitch error
  float dv;
  if (dbl) {
    const double dv_d = ((CS && use_cs) ? vzh_d : r.vartheta) - th_fold;
    o.dv = dv_d;
    dv = __double2float_rn(dv_d);
  } else {
    dv = ((CS && use_cs) ? o.vartheta_zh : vref_f) - thf;
  }
  o.dvf = dv;
  // СС PID
  const float ss_d = (dv * mp.PID_SS[2] - ssf) * mp.PID_SS[3];
  const float ss_pre = fmaf(dv, mp.PID_SS[0], ssi) + ss_d;
  o.U_com_PID = satf(ss_pre, PCF(5), PCF(7));
  const int sw = SW >= 0 ? SW : mp.sw;
  if (sw & SW_RL) o.U_com = PCF(147) > fabsf(o.U_com_PID) ? 0.f : o.U_com_PID;
  else o.U_com = (sw & SW_SS) ? o.U_com_PID : r.deltaz;
  const float ax = fmaf(Fx, cs, -sn * Fy);
  const float ay = fmaf(Fy, cs, fmaf(Fx, sn, -mp.g));
  const float dze = (sw & SW_RP) ? o.deltaz_RP : o.U_com;
  const float Cm = fmaf(dcm * Ka, dze, mz);
  const float wzd = Cm * (rV2 * mp.half_Sc_over_Iz);
  // clamping anti-windup (СС)
  const float dz = ss_pre - o.U_com_PID;
  float ss_i = mp.PID_SS[1] * dv;
  if (PCF(291) == 0.f)  // ZeroGain: ss_pre*0 != dz  <=>  dz != 0 (finite ss_pre); sign(dz)==sign(ss_i) via the sign bits
    o.and_ss = (dz != 0.f) & (ss_i != 0.f) & ((__float_as_int(dz) ^ __float_as_int(ss_i)) >= 0);
  else
    o.and_ss = (ss_pre * PCF(291) != dz) && (sgnf(dz) == sgnf(ss_i));
  if (major) memout_ss = (r.flags & FL_MEM_SS) != 0;
  if (memout_ss) ss_i = PCF(10);
  f_h = Vy; f_Vx = ax; f_Vy = ay; f_wz = wzd; f_ssi = ss_i; f_ssf = ss_d;
  f_itse = dv * dv * t_f;
  if (CS) {
    const double dzc = cs_pre - vzh_d;
    double cs_i = e_h * c.mp.PID_CS[1];
    o.and_cs = (cs_pre * Pc(292) != dzc) && (((dzc > 0.0) - (dzc < 0.0)) == ((cs_i > 0.0) - (cs_i < 0.0)));
    if (major) memout_cs = (r.flags & FL_MEM_CS) != 0;
    if (memout_cs) cs_i = Pc(11);
    f_csi = cs_i; f_csf = cs_d;
  } else {
    o.and_cs = false; f_csi = 0.0; f_csf = 0.0;
  }
}

// model_simple_step in the mixed formulation.  On return r holds the post-update state, `o` the
// stage-4 pass and s4 the stage-4 (predictor) state values.
template <int TIER, int SW = -1>
__device__ __forceinline__ void model_step32(const float4* __restrict__ sT, const MP32& mp, const DevCfg& c, RegsMx& r,
                                             PassMx& o, Stage4Mx& s4, bool want_x) {
  constexpr bool CS = TIER >= 2;
  const int n = r.tick;
  const float hh = (float)kH, hhalf = 0.5f * (float)kH;
  const float t0f = (float)n * hh;
  // float32 copies of the accumulated state for the stage evaluations
  const float y_h = __double2float_rn(r.h), y_Vx = __double2float_rn(r.Vx), y_Vy = __double2float_rn(r.Vy),
              y_wz = __double2float_rn(r.wz), y_ssi = __double2float_rn(r.ssi), y_ssf = __double2float_rn(r.ssf),
              y_th = __double2float_rn(r.th);
  const float vref_f = __double2float_rn(r.vartheta);
  // RK4 bookkeeping in register PAIRS (packed FFMA2, the weights ride as broadcast scalars): the stage state pair
  // (Vy, wz) is at the same time the derivative of (h, theta); (Vx, ssi) and (ssf, int dvartheta) pair up likewise.
  const float2 yVW = make_float2(y_Vy, y_wz), yXI = make_float2(y_Vx, y_ssi);
  float2 XVW = yVW, XXI = yXI;  // (X_Vy, X_wz), (X_Vx, X_ssi)
  float X_h = y_h, X_ssf = y_ssf, d_th = 0.f;
  double X_th = r.th, Xd_h = r.h, X_csi = r.csi, X_csf = r.csf;
  float2 aHT = make_float2(0.f, 0.f), aVW = aHT, aXI = aHT, aFD = aHT;  // sums for (h, th) (Vy, wz) (Vx, ssi) (ssf, dvi)
  float a_x = 0, a_itse = 0;
  double a_csi = 0, a_csf = 0;
  bool memout_ss = false, memout_cs = false;
  float u_n = 0.f;
  AtmoMx at;
  TrigMx tg;
#pragma unroll
  for (int s = 0; s < 4; s++) {
    const bool ends = (s == 0 || s == 3);
    const float t_f = s == 0 ? t0f : (s == 3 ? t0f + hh : t0f + hhalf);
    float f_h, f_Vx, f_Vy, f_wz, f_ssi, f_ssf, f_itse;
    double f_csi, f_csf;
    pass32<TIER, SW>(sT, mp, c, s, n, X_th, d_th, tg, vref_f, t_f, X_h, Xd_h, XXI.x, XVW.x, XVW.y, XXI.y, X_ssf, X_csi, X_csf, r, at,
                memout_ss, memout_cs, o, f_h, f_Vx, f_Vy, f_wz, f_ssi, f_ssf, f_csi, f_csf, f_itse);
    if (s == 0) {
      // update(): discrete filter, rate-limiter memory, Memory blocks, Derivative history, delay push
      if ((n % 5) == 0) r.df_x = fmaf(PCF(138), r.df_x, PCF(139) * o.td);
      r.rl_prev = o.rl_out;
      r.flags = (r.flags & ~(FL_MEM_SS | FL_MEM_CS)) | (o.and_ss ? FL_MEM_SS : 0) | (o.and_cs ? FL_MEM_CS : 0);
      const double dvdt_major = n >= 1 ? (o.dv - r.d1_u) * 100.0 : 0.0;
      r.d1_u = o.dv;
      r.d2_u = __double2float_rn(dvdt_major);
      u_n = o.U_com;
    }
    const float2 fVW = make_float2(f_Vy, f_wz), fXI = make_float2(f_Vx, f_ssi), fFD = make_float2(f_ssf, o.dvf);
    const double wd = ends ? 1.0 : 2.0;
    if (s == 0) {  // first term of the sums: plain copies
      aHT = XVW; aVW = fVW; aXI = fXI; aFD = fFD; a_itse = f_itse;
      if (want_x) a_x = XXI.x;
    } else {
      const float w = ends ? 1.f : 2.f;
      const float2 ww = make_float2(w, w);
      aHT = fma2(ww, XVW, aHT); aVW = fma2(ww, fVW, aVW); aXI = fma2(ww, fXI, aXI);
      aFD = fma2(ww, fFD, aFD);
      a_itse = fmaf(w, f_itse, a_itse);
      if (want_x) a_x = fmaf(w, XXI.x, a_x);
    }
    if (CS) { a_csi = fma(wd, f_csi, a_csi); a_csf = fma(wd, f_csf, a_csf); }
    if (s < 3) {
      const float cf = (s == 2) ? hh : hhalf;
      const double cfd = (s == 2) ? kH : 0.5 * kH;
      if (s == 2) {  // integral / position signals at stage 4 = y + h*f2
        s4.dvi = r.dvi + (double)(hh * o.dvf);
        s4.itse = r.itse + (double)(hh * f_itse);
        s4.x = want_x ? (float)r.x + hh * XXI.x : 0.f;
        X_th = fma(kH, (double)XVW.y, r.th);  // theta' = wz: the full-step pass needs the float64 pitch
      } else {
        d_th = cf * XVW.y;                   // half-step passes: float32 pitch increment since the major pass
      }
      const float2 cc = make_float2(cf, cf);
      X_h = fmaf(cf, f_h, y_h);
      XVW = fma2(cc, fVW, yVW); XXI = fma2(cc, fXI, yXI);
      X_ssf = fmaf(cf, f_ssf, y_ssf);
      if (CS) {
        X_csi = fma(cfd, f_csi, r.csi); X_csf = fma(cfd, f_csf, r.csf);
        Xd_h = fma(cfd, (double)f_h, r.h);
      }
    }
  }
  const float X_Vx = XXI.x, X_Vy = XVW.x, X_wz = XVW.y;
  const float a_h = aHT.x, a_th = aHT.y, a_Vy = aVW.x, a_wz = aVW.y, a_Vx = aXI.x, a_ssi = aXI.y, a_ssf = aFD.x, a_dvi = aFD.y;
  s4.h = X_h; s4.Vx = X_Vx; s4.Vy = X_Vy; s4.wz = X_wz;
  // y += h/6 * sum, accumulated in float64: one conversion and one DFMA per state
  const double h6d = kH / 6.0;
  r.h = fma((double)a_h, h6d, r.h); r.Vx = fma((double)a_Vx, h6d, r.Vx); r.Vy = fma((double)a_Vy, h6d, r.Vy);
  r.wz = fma((double)a_wz, h6d, r.wz); r.ssi = fma((double)a_ssi, h6d, r.ssi); r.ssf = fma((double)a_ssf, h6d, r.ssf);
  r.th = fma((double)a_th, h6d, r.th);
  if (CS) { r.csi = fma(h6d, a_csi, r.csi); r.csf = fma(h6d, a_csf, r.csf); }
  if (want_x) r.x = fma((double)a_x, h6d, r.x);
  r.dvi = fma((double)a_dvi, h6d, r.dvi);
  r.itse = fma((double)a_itse, h6d, r.itse);
  r.uh[0] = r.uh[1]; r.uh[1] = r.uh[2]; r.uh[2] = r.uh[3]; r.uh[3] = u_n;
  r.tick = n + 1;
}

// model_simple_initialize + Model.initialize (core/model.py:238-244)
__device__ __forceinline__ void model_init32(const double s0[6], RegsMx& r) {
  r.x = s0[0]; r.h = s0[1]; r.th = s0[4]; r.Vx = s0[2]; r.Vy = s0[3]; r.wz = s0[5];
  r.csi = Pc(2); r.csf = Pc(0); r.ssi = Pc(3); r.ssf = Pc(1);
  r.dvi = Pc(293); r.itse = Pc(297);
  r.df_x = PCF(8); r.df_y = 0.f; r.rl_prev = 0.f;
  r.uh[0] = r.uh[1] = r.uh[2] = r.uh[3] = 0.f;
  r.d1_u = 0.0; r.d2_u = 0.f;
  r.tick = 0;
  r.flags &= ~(FL_MEM_SS | FL_MEM_CS);
  r.sig_upid = 0.f; r.sig_vzh = 0.f;
  r.deltaz = 0.f;
}

}  // namespace b747
