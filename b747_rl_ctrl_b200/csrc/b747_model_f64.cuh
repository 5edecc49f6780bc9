// b747_model_f64.cuh -- float64 parity path: one environment per thread, every block of the
// Simulink diagram evaluated in the DLL's operation order (model_simple_step dll@0x16d0,
// rt_ertODEUpdateContinuousStates/ode4 dll@0x2c60, look2_binlx dll@0x1000,
// rt_TDelayInterpolate dll@0x29e0; SURVEY.md Appendix B).
//
// Differences from a literal transcription, all exact (documented in DESIGN.md):
//  * X[3]=X[4] (q1,q2) are identically zero for the pitch-only attitude, so they are not carried;
//  * the 1024-entry transport-delay ring is replaced by the last four U_com samples: with h=0.01 and
//    a 0.03 s delay the interpolation only ever touches samples n-4..n-1, and the buffered time
//    stamps are fl(k*0.01), recomputed from the tick;
//  * Derivative / rate-limiter time stamps are recomputed from the tick the same way;
//  * the extra minor-mode output pass of the very first step (dll@0x28fb) reproduces the major
//    pass bit for bit (nothing it reads has changed value), so it is skipped.
#pragma once
#include <math.h>

#include "b747_common.cuh"

namespace b747 {

struct Regs64 {
  // continuous states (true post-update values)
  double X[16];  // x h q0 q3 Vx Vy wz cs_int cs_flt ss_int ss_flt dv_int itae iae ise itse
  double df_x, df_y, rl_prev, uh[4], d1_u, d2_u;
  double deltaz, vartheta, h_zh, aerr[5];
  double sig_upid, sig_vzh;
  double vref, href, oscA[3], oscf[3];
  double ep_return, tf_tp;
  int tick, flags;
  uint32_t ep_idx;
  double use_PID_CS;  // per env (HYBRID toggles it per episode); derived from flags
  unsigned long long lut = 0;  // last interval of the nine prelookups, 4 bits each (registers only; always re-validated)
};

enum { IX_x = 0, IX_h, IX_q0, IX_q3, IX_Vx, IX_Vy, IX_wz, IX_csi, IX_csf, IX_ssi, IX_ssf, IX_dvi, IX_itae, IX_iae, IX_ise, IX_itse };

// Values of one pass over the diagram (the DLL's exported signals + what update() consumes).
struct Pass64 {
  double th, V, alpha, Mach, CXa, CYa, mz, K_alpha, dCm, U_com, U_com_PID, deltaz_RP, vartheta_zh;
  double dv, dv_dt, dv_dt_dt, SE, TSE, AE, TAE, td, rl_out;
  double CXa_tab, CYa_tab, mz_tab, dCm_tab;  // table outputs before the aero-error gains (legacy signal taps)
  bool and_ss, and_cs;
};

// Values held between major steps (Simulink "held" block outputs).
struct Held64 {
  double sumA[5];
  bool memout_ss, memout_cs;
};

__device__ __forceinline__ double sat64(double u, double lo, double hi) { return u > hi ? hi : (u >= lo ? u : lo); }
__device__ __forceinline__ int sgn8(double x) { return x < 0.0 ? -1 : (x > 0.0 ? 1 : 0); }

// look2_binlx prelookup: binary search, linear extrapolation at both ends (dll@0x1000)
__device__ __forceinline__ unsigned prelookup64(double u, const double* bp, unsigned maxIndex, double& frac) {
  unsigned iLeft;
  if (u <= bp[0]) {
    iLeft = 0;
    frac = (u - bp[0]) / (bp[1] - bp[0]);
  } else if (u < bp[maxIndex]) {
    unsigned bpIdx = maxIndex >> 1, iRght = maxIndex;
    iLeft = 0;
    while (iRght - iLeft > 1) {
      if (u < bp[bpIdx]) iRght = bpIdx; else iLeft = bpIdx;
      bpIdx = (iRght + iLeft) >> 1;
    }
    frac = (u - bp[iLeft]) / (bp[iLeft + 1] - bp[iLeft]);
  } else {
    iLeft = maxIndex - 1;
    frac = (u - bp[maxIndex - 1]) / (bp[maxIndex] - bp[maxIndex - 1]);
  }
  return iLeft;
}

// The same prelookup with the previous interval as a hint: the operands move by a small fraction of an interval per
// pass, so the DLL's binary search almost always lands where it landed last time.  The hint is checked against the
// search's own postcondition (u <= bp[0] -> 0; u >= bp[max] -> max-1; else bp[i] <= u < bp[i+1]) and the fraction uses
// the same expression, so index and fraction are bit-identical to prelookup64 -- only the search is skipped.
template <int SLOT>
__device__ __forceinline__ unsigned prelookup64c(double u, const double* bp, unsigned maxIndex, double& frac,
                                                 unsigned long long& lut) {
  unsigned i = (unsigned)(lut >> (4 * SLOT)) & 15u;
  if (i > maxIndex - 1) i = maxIndex - 1;
  const double lo = bp[i], hi = bp[i + 1];
  if ((i == 0 || u >= lo) && (i == maxIndex - 1 || u < hi)) {
    frac = (u - lo) / (hi - lo);
    return i;
  }
  i = prelookup64(u, bp, maxIndex, frac);
  lut = (lut & ~(15ull << (4 * SLOT))) | ((unsigned long long)i << (4 * SLOT));
  return i;
}

template <int SLOT>
__device__ __forceinline__ double look2_64(double u0, double u1, const double* bp0, const double* bp1, const double* tab,
                                           unsigned max0, unsigned max1, unsigned stride, unsigned long long& lut) {
  double f0, f1;
  unsigned i0 = prelookup64c<SLOT>(u0, bp0, max0, f0, lut);
  unsigned i1 = prelookup64c<SLOT + 1>(u1, bp1, max1, f1, lut);
  unsigned o = i1 * stride + i0;
  double yL = (tab[o + 1] - tab[o]) * f0 + tab[o];
  o += stride;
  double yR = (tab[o + 1] - tab[o]) * f0 + tab[o];
  return (yR - yL) * f1 + yL;
}

__device__ __forceinline__ double rt_atan2_64(double u0, double u1) {  // rt_atan2d_snf
  if (isnan(u0) || isnan(u1)) return nan("");
  if (isinf(u0) && isinf(u1)) return atan2(u0 > 0 ? 1.0 : -1.0, u1 > 0 ? 1.0 : -1.0);
  if (u1 == 0.0) return u0 > 0.0 ? kPi / 2.0 : (u0 < 0.0 ? -(kPi / 2.0) : 0.0);
  return atan2(u0, u1);
}

__device__ __forceinline__ double rt_pow_64(double u0, double u1) {  // rt_powd_snf, dll@0x3530
  if (isnan(u0) || isnan(u1)) return nan("");
  double a0 = fabs(u0), a1 = fabs(u1);
  if (isinf(u1)) {
    if (a0 == 1.0) return 1.0;
    if (a0 > 1.0) return u1 > 0.0 ? INFINITY : 0.0;
    return u1 > 0.0 ? 0.0 : INFINITY;
  }
  if (a1 == 0.0) return 1.0;
  if (a1 == 1.0) return u1 > 0.0 ? u0 : 1.0 / u0;
  if (u1 == 2.0) return u0 * u0;
  if (u1 == 0.5 && u0 >= 0.0) return sqrt(u0);
  if (u0 < 0.0 && u1 > floor(u1)) return nan("");
  return pow(u0, u1);
}

// rt_TDelayInterpolate (dll@0x29e0) over the compact history: uh[j] = U_com sampled at major tick
// n-4+j; buffered stamps are fl(k*0.01).  n = tick of the step being integrated.
__device__ __forceinline__ double tdelay64(double t, int n, const double uh[4], const double* P) {
  double tmd = t - P[136];
  if (tmd <= 0.0) return P[137];
  int k = -1;
#pragma unroll
  for (int c = -3; c <= -1; c++) {
    int kc = n + c;
    if (k < 0 && kc >= 1 && (double)kc * kH >= tmd) k = kc;
  }
  if (k < 0) k = n - 1;  // not reachable for a 3-step delay; mirrors the forward-search break
  int j = k - (n - 4);   // 1..3
  double u2 = j == 1 ? uh[1] : (j == 2 ? uh[2] : uh[3]);
  double u1 = j == 1 ? uh[0] : (j == 2 ? uh[1] : uh[2]);
  double t2 = (double)k * kH, t1 = (double)(k - 1) * kH;
  if (t2 == t1) return tmd >= t2 ? u2 : u1;
  double f1 = (t2 - tmd) / (t2 - t1);
  double f2 = 1.0 - f1;
  return f1 * u1 + f2 * u2;
}

// One pass over the block diagram.  Xs = stage state, t = stage time, t_last = time stamp of the
// most recent update() (valid if have_last), n = tick of the step being integrated.
__device__ __forceinline__ void pass64(const double* __restrict__ P, const ModelParams& mp, const double Xs[16], double t,
                                    double t_last, bool have_last, bool major, int n, Regs64& r, Held64& hd, Pass64& o,
                                    double dX[16]) {
  // quaternion normalisation (q1=q2=0) and pitch angle
  double nq = sqrt(Xs[IX_q0] * Xs[IX_q0] + 0.0 + 0.0 + Xs[IX_q3] * Xs[IX_q3]);
  double q3 = Xs[IX_q3] / nq, q0 = Xs[IX_q0] / nq;
  double th = asin((0.0 + q3 * q0) * 2.0);
  o.th = th;
  double sn, cs;
  sincos(th, &sn, &cs);  // one argument reduction for both (same values as sin / cos)
  double Vx = Xs[IX_Vx], Vy = Xs[IX_Vy];
  double ub = cs * Vx + sn * Vy;
  double wb = cs * Vy - sn * Vx;
  // MATLAB scaled 2-norm
  double scale = 3.3121686421112381E-170, y, a;
  a = fabs(ub);
  if (a > scale) { y = 1.0; scale = a; } else { double q = a / scale; y = q * q; }
  a = fabs(wb);
  if (a > scale) { double q = scale / a; y = y * q * q + 1.0; scale = a; } else { double q = a / scale; y += q * q; }
  double V = scale * sqrt(y);
  double alpha = -rt_atan2_64(wb, ub);
  o.V = V; o.alpha = alpha;
  // ISA atmosphere
  double h = Xs[IX_h];
  double hs = h > P[17] ? P[17] : (h >= P[18] ? h : P[18]);
  double T = P[16] - hs * P[19];
  double asnd = sqrt(T * P[20]);
  double ad = alpha * P[21];
  double Mach = V / asnd;
  o.Mach = Mach;
  if (major) { hd.sumA[1] = r.aerr[1] + P[51]; hd.sumA[0] = r.aerr[0] + P[51]; }
  o.CYa_tab = look2_64<0>(Mach, ad, P + 42, P + 46, P + 22, 3, 4, 4, r.lut);
  double CYa = o.CYa_tab * hd.sumA[1];
  o.CXa_tab = look2_64<2>(Mach, CYa, P + 108, P + 112, P + 52, 3, 13, 4, r.lut);
  double CXa = o.CXa_tab * hd.sumA[0];
  o.CYa = CYa; o.CXa = CXa;
  double Tr = T * P[127];
  double pw = (Tr < 0.0 && P[128] > floor(P[128])) ? -rt_pow_64(-Tr, P[128]) : rt_pow_64(Tr, P[128]);
  double dh = P[130] - h;
  double xs = dh > P[131] ? P[131] : (dh >= P[132] ? dh : P[132]);
  double rho = pw / Tr * P[129] * exp(xs * P[133] * (1.0 / T));
  double rV2 = rho * (V * V);
  double qS = rV2 * P[134] * mp.S;
  double sa, ca;
  sincos(alpha, &sa, &ca);
  double mD = P[126] * CXa * qS;
  double Lf = qS * CYa;
  double Fx = mD * ca + sa * Lf + mp.P;
  double Fy = ca * Lf - mD * sa + 0.0;
  // actuator: transport delay -> discrete filter -> rate limiter -> saturation
  double td = tdelay64(t, n, r.uh, P);
  o.td = td;
  if (major && (n % 5) == 0) r.df_y = r.df_x * P[140] + P[141] * td;
  double yv = r.df_y;
  if (have_last) {
    double dT = t - t_last, rate = yv - r.rl_prev;
    if (rate > dT * P[142]) yv = dT * P[142] + r.rl_prev;
    else if (dT * P[143] > rate) yv = dT * P[143] + r.rl_prev;
  }
  o.rl_out = yv;
  o.deltaz_RP = sat64(yv, P[145], P[144]);
  // СУ PID (altitude -> pitch reference)
  double e_h = r.h_zh - h;
  double cs_d = (e_h * mp.PID_CS[2] - Xs[IX_csf]) * mp.PID_CS[3];
  double cs_pre = e_h * mp.PID_CS[0] + Xs[IX_csi] + cs_d;
  o.vartheta_zh = sat64(cs_pre, P[4], P[6]);
  double vref = r.use_PID_CS >= P[146] ? o.vartheta_zh : r.vartheta;
  double dv = vref - th;
  o.dv = dv;
  // СС PID (pitch error -> elevator command)
  double ss_d = (dv * mp.PID_SS[2] - Xs[IX_ssf]) * mp.PID_SS[3];
  double ss_pre = dv * mp.PID_SS[0] + Xs[IX_ssi] + ss_d;
  o.U_com_PID = sat64(ss_pre, P[5], P[7]);
  if (mp.use_RL >= P[148]) o.U_com = P[147] > fabs(0.0 - o.U_com_PID) ? 0.0 : o.U_com_PID;
  else o.U_com = mp.use_PID_SS >= P[9] ? o.U_com_PID : r.deltaz;
  if (major) { hd.sumA[3] = r.aerr[3] + P[216]; hd.sumA[4] = r.aerr[4] + P[216]; }
  o.dCm_tab = look2_64<4>(h, Mach, P + 201, P + 206, P + 151, 4, 9, 5, r.lut);
  o.dCm = o.dCm_tab * hd.sumA[3];
  {
    double f;
    unsigned i = prelookup64c<6>(ad, P + 225, 6, f, r.lut);
    o.K_alpha = ((P[218 + i + 1] - P[218 + i]) * f + P[218 + i]) * hd.sumA[4];
  }
  if (major) hd.sumA[2] = r.aerr[2] + P[216];
  o.mz_tab = look2_64<7>(Mach, ad, P + 276, P + 280, P + 232, 3, 10, 4, r.lut);
  o.mz = o.mz_tab * hd.sumA[2];
  double ax = (Fx * cs - sn * Fy) / mp.m0;
  double ay = (Fy * cs + Fx * sn) / mp.m0 - mp.g;
  double dze = mp.use_RP >= P[149] ? o.deltaz_RP : o.U_com;
  double Cm = P[217] * o.dCm * o.K_alpha * (dze * P[150]) + o.mz;
  double wzd = Cm * (rV2 * P[135] * mp.S * mp.c_) / mp.Iz;
  double wz = Xs[IX_wz];
  double dq0 = (-wz) * q3 * 0.5, dq3 = q0 * wz * 0.5;
  // clamping anti-windup (СС)
  double dz = ss_pre > P[7] ? ss_pre - P[7] : (ss_pre >= P[5] ? 0.0 : ss_pre - P[5]);
  double ss_i = mp.PID_SS[1] * dv;
  o.and_ss = (ss_pre * P[291] != dz) && (sgn8(dz) == sgn8(ss_i));
  if (major) hd.memout_ss = (r.flags & FL_MEM_SS) != 0;
  if (hd.memout_ss) ss_i = P[10];
  // Derivative blocks
  o.dv_dt = have_last ? (dv - r.d1_u) / (t - t_last) : 0.0;
  o.dv_dt_dt = have_last ? (o.dv_dt - r.d2_u) / (t - t_last) : 0.0;
  o.SE = dv * dv; o.TSE = o.SE * t; o.AE = fabs(dv); o.TAE = o.AE * t;
  dz = cs_pre > P[6] ? cs_pre - P[6] : (cs_pre >= P[4] ? 0.0 : cs_pre - P[4]);
  double cs_i = e_h * mp.PID_CS[1];
  o.and_cs = (cs_pre * P[292] != dz) && (sgn8(dz) == sgn8(cs_i));
  if (major) hd.memout_cs = (r.flags & FL_MEM_CS) != 0;
  if (hd.memout_cs) cs_i = P[11];
  dX[IX_x] = Vx; dX[IX_h] = Vy; dX[IX_q0] = dq0; dX[IX_q3] = dq3; dX[IX_Vx] = ax; dX[IX_Vy] = ay; dX[IX_wz] = wzd;
  dX[IX_csi] = cs_i; dX[IX_csf] = cs_d; dX[IX_ssi] = ss_i; dX[IX_ssf] = ss_d; dX[IX_dvi] = dv;
  dX[IX_itae] = o.TAE; dX[IX_iae] = o.AE; dX[IX_ise] = o.SE; dX[IX_itse] = o.TSE;
}

// model_simple_step: major pass + update + ode4.  On return r.X holds the post-update states,
// `o` and Xs4 the stage-4 pass (= what the DLL's exported signals show, SURVEY.md 0.4).
__device__ __forceinline__ void model_step64(const double* __restrict__ P, const ModelParams& mp, Regs64& r, Pass64& o,
                                             double Xs4[16]) {
  const int n = r.tick;
  const double t0 = (double)n * kH, tnew = (double)(n + 1) * kH;
  const double t_prev = (double)(n - 1) * kH;
  Held64 hd;
  double f[16];
  double acc[16], y[16];
#pragma unroll
  for (int i = 0; i < 16; i++) { y[i] = r.X[i]; Xs4[i] = r.X[i]; }
  const double hh = kH, temp = 0.5 * hh;
  const double th = t0 + temp;
  double u_n = 0.0;
  // One copy of the diagram code, four passes: major (+update) and the three ode4 stages.
#pragma unroll 1
  for (int s = 0; s < 4; s++) {
    const bool major = (s == 0);
    const double t = major ? t0 : (s == 3 ? tnew : th);
    pass64(P, mp, Xs4, t, major ? t_prev : t0, major ? (n >= 1) : true, major, n, r, hd, o, f);
    if (major) {
      // update (dll@0x271a): delay ring push, discrete filter, rate-limiter memory, Memory blocks, Derivative history
      if ((n % 5) == 0) r.df_x = P[138] * r.df_x + P[139] * o.td;
      r.rl_prev = o.rl_out;
      r.flags = (r.flags & ~(FL_MEM_SS | FL_MEM_CS)) | (o.and_ss ? FL_MEM_SS : 0) | (o.and_cs ? FL_MEM_CS : 0);
      r.d1_u = o.dv; r.d2_u = o.dv_dt;
      u_n = o.U_com;  // pushed into the ring; first needed as uh[3] of the NEXT step
#pragma unroll
      for (int i = 0; i < 16; i++) acc[i] = f[i];
    } else if (s < 3) {
#pragma unroll
      for (int i = 0; i < 16; i++) acc[i] = acc[i] + 2.0 * f[i];
    }
    if (s < 3) {
      const double c = (s == 2) ? hh : temp;
#pragma unroll
      for (int i = 0; i < 16; i++) Xs4[i] = y[i] + c * f[i];
    }
  }
  const double h6 = hh / 6.0;
#pragma unroll
  for (int i = 0; i < 16; i++) r.X[i] = y[i] + h6 * (acc[i] + f[i]);
  r.uh[0] = r.uh[1]; r.uh[1] = r.uh[2]; r.uh[2] = r.uh[3]; r.uh[3] = u_n;
  r.tick = n + 1;
}

// model_simple_initialize (dll@0x12a0) + Model.initialize's Python part (core/model.py:238-244).
__device__ __forceinline__ void model_init64(const double* __restrict__ P, const double s0[6], Regs64& r) {
  r.X[IX_x] = s0[0]; r.X[IX_h] = s0[1];
  r.X[IX_q0] = cos(s0[4] / 2.0); r.X[IX_q3] = sin(s0[4] / 2.0);
  r.X[IX_Vx] = s0[2]; r.X[IX_Vy] = s0[3]; r.X[IX_wz] = s0[5];
  r.X[IX_csi] = P[2]; r.X[IX_csf] = P[0]; r.X[IX_ssi] = P[3]; r.X[IX_ssf] = P[1];
#pragma unroll
  for (int i = 0; i < 5; i++) r.X[IX_dvi + i] = P[293 + i];
  r.df_x = P[8]; r.df_y = 0.0; r.rl_prev = 0.0;
  r.uh[0] = r.uh[1] = r.uh[2] = r.uh[3] = 0.0;
  r.d1_u = r.d2_u = 0.0;
  r.tick = 0;
  r.flags &= ~(FL_MEM_SS | FL_MEM_CS);
  r.sig_upid = 0.0; r.sig_vzh = 0.0;  // every exported signal is zeroed
  r.deltaz = 0.0; r.vartheta = 0.0;   // Model.initialize: self.deltaz = 0; self.vartheta_zh = 0
}

}  // namespace b747
