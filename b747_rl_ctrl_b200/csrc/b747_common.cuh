// b747_common.cuh -- shared device-side definitions for the B747 env-step kernels (sm_100a).
//
// Reference being replaced: the Simulink-Coder model in core/model_simple_win64.dll
// (model_simple_step dll@0x16d0, ode4 dll@0x2c60; SURVEY.md Appendix B) and the Python layers
// core/controller.py:134-264 and env/ctrl_env.py:109-278.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/b747.h"
#include "../../include/b747_params.h"

namespace b747 {

constexpr int kNP = B747_NP;            // block parameters (model_simple_P)
constexpr double kH = 0.01;             // fixed integrator step (core/model.py:121)
constexpr double kPi = 3.141592653589793238462643383279502884;

// ---------------------------------------------------------------------------------------------
// Persistent per-environment state in HBM: structure of arrays, field-major.
//   f64 handle: double  slot[NSLOT_F64][n_pad]   (+ int32 tick/flags/episode arrays)
//   f32 handle: see b747_model_mx.cuh
// Consecutive threads own consecutive envs, so every field access of a warp is one fully
// coalesced 256-byte (f64) / 128-byte (f32) segment; pairs of fields are fetched as 128-bit
// vectors where the layout groups them (f32 path).
// ---------------------------------------------------------------------------------------------
#define B747_F64_SLOTS(X)                                                                          \
  /* 16 continuous states (X[3]=X[4]=0 identically for a pitch-only attitude, so q1,q2 are not stored) */ \
  X(x) X(h) X(q0) X(q3) X(Vx) X(Vy) X(wz) X(cs_int) X(cs_flt) X(ss_int) X(ss_flt) X(dv_int) X(itae) X(iae) X(ise) X(itse) \
  /* discrete / hidden block state */                                                               \
  X(df_x) X(df_y) X(rl_prev) X(uh0) X(uh1) X(uh2) X(uh3) X(d1_u) X(d2_u)                            \
  /* per-env tunables the Python layer writes every step / every reset */                            \
  X(deltaz) X(vartheta) X(h_zh) X(aerr0) X(aerr1) X(aerr2) X(aerr3) X(aerr4)                        \
  /* stage-4 signals the next env step reads (Controller.step / vartheta_ref) */                    \
  X(sig_upid) X(sig_vzh)                                                                            \
  /* episode reference */                                                                            \
  X(vref) X(href) X(oscA0) X(oscA1) X(oscA2) X(oscf0) X(oscf1) X(oscf2)                              \
  /* env bookkeeping */                                                                              \
  X(ep_return) X(tf_tp)

enum F64Slot {
#define X(n) S_##n,
  B747_F64_SLOTS(X)
#undef X
      NSLOT_F64
};

// flag bits (int32 flags array)
enum { FL_MEM_SS = 1, FL_MEM_CS = 2, FL_USE_CTRL = 4, FL_OSC = 8 };

// Stage-4 signal export (optional, [NSIG][n_pad] in the handle dtype): the DLL's exported signals.
#define B747_SIGNALS(X)                                                                             \
  X(state_x) X(state_y) X(state_Vx) X(state_Vy) X(state_vartheta) X(state_wz) X(sim_time) X(vartheta_zh) \
  X(U_com_PID) X(CXa) X(CYa) X(mz) X(K_alpha) X(dCm_ddeltaz) X(U_com) X(deltaz_RP) X(dvartheta)      \
  X(dvartheta_int) X(dvartheta_dt) X(dvartheta_dt_dt) X(TAE) X(ITAE) X(TSE) X(ITSE) X(AE) X(IAE)     \
  X(SE) X(ISE) X(alpha) X(V) X(Mach)                                                                \
  /* table outputs BEFORE the (1 + aero_err) gains: what the legacy model_win64.dll exports as CXa / CYa / mz / dCm */ \
  X(CXa_tab) X(CYa_tab) X(mz_tab) X(dCm_tab)

enum Signal {
#define X(n) SIG_##n,
  B747_SIGNALS(X)
#undef X
      NSIG
};

// Uniform (whole-batch) model tunables: exported DLL globals that the Python layer never varies
// per environment (core/model.py:154-164 binds PID_SS/PID_CS/P/use_RP; Iz,S,c_,g,m0,use_RL unbound).
struct ModelParams {
  double PID_SS[4], PID_CS[4];
  double P, Iz, S, c_, g, m0;
  double use_RP, use_RL, use_PID_SS;
};

// Kernel-side configuration (copied by value into the launch).
struct DevCfg {
  int32_t n_envs, n_pad;
  int32_t env_lo, env_hi;  // env range of this launch of the step kernels ([0, n_envs) except in b747_step_host's pipeline)
  int32_t obs_type, obs_dim, rew_type, ctrl_type, ctrl_mode, reset_ref_mode, disturbance_mode;
  int32_t norm_obs, norm_act, use_limiter, substeps, auto_reset, env_layer, has_fixed_aero_err;
  int32_t force_full;  // explicit episodes / edited flags: the f32 launch must take the full kernel tier
  int64_t done_tick, env_id_offset;
  uint64_t seed;
  double tk, action_max, vartheta_max, sample_time;
  double rew[8];
  double fixed_aero_err[5];
  ModelParams mp;
};

// ---------------------------------------------------------------------------------------------
// Philox4x32-10 (counter-based; identical definition in oracle/b747_env_ref.c).
// ---------------------------------------------------------------------------------------------
__host__ __device__ inline void philox4x32(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
  uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3], k0 = key[0], k1 = key[1];
#pragma unroll
  for (int r = 0; r < 10; r++) {
    uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
    uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1;
    uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// 53-bit uniform in [0,1): draw j of (seed, env, episode) -- same construction as CPython's random()
__host__ __device__ inline double uniform53(uint64_t seed, uint64_t env, uint32_t episode, uint32_t draw) {
  uint32_t ctr[4] = {(uint32_t)env, (uint32_t)(env >> 32), episode, draw >> 1};
  uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)}, w[4];
  philox4x32(ctr, key, w);
  uint32_t a = w[2 * (draw & 1)] >> 5, b = w[2 * (draw & 1) + 1] >> 6;
  return ((double)a * 67108864.0 + (double)b) * (1.0 / 9007199254740992.0);
}

// Per-episode reference / initial condition in registers (Controller.reset's decisions).
struct Episode {
  double s0[6];
  double vref, href, oscA[3], oscf[3], aerr[5];
  int use_ctrl, osc;
};

// An explicit episode of the C ABI (b747_reset_to) in the kernels' form.
__device__ inline void episode_from_abi(const b747_episode& e, Episode& ep) {
  for (int k = 0; k < 6; k++) ep.s0[k] = e.state0[k];
  ep.vref = e.vref_const; ep.href = e.h_ref; ep.use_ctrl = e.use_ctrl; ep.osc = e.oscillating;
  for (int k = 0; k < 3; k++) { ep.oscA[k] = e.osc_A[k]; ep.oscf[k] = e.osc_f[k]; }
  for (int k = 0; k < 5; k++) ep.aerr[k] = e.aero_err[k];
}

// Controller.reset random part (core/controller.py:144-193): distributions and draw order are the
// reference's; the stream is Philox keyed by (seed, global env id, episode index).
__device__ inline void draw_episode(const DevCfg& c, uint64_t env, uint32_t epi, Episode& ep) {
  const uint64_t sd = c.seed;
  auto uni = [&](uint32_t j, double a, double b) { return a + (b - a) * uniform53(sd, env, epi, j); };
  ep.use_ctrl = (c.ctrl_type == B747_CTRL_SEMI_MANUAL || c.ctrl_type == B747_CTRL_FULL_AUTO);
  ep.osc = 0;
  ep.vref = 0.0; ep.href = 11000.0;
  for (int i = 0; i < 3; i++) { ep.oscA[i] = 0.0; ep.oscf[i] = 0.0; }
  for (int i = 0; i < 5; i++) ep.aerr[i] = 0.0;
  double h0 = uni(0, 1000, 11000);
  double Vx = uni(1, 100, 265);
  double Vy = uni(2, -20, 20);
  double wz0 = uni(3, -0.001, 0.001);
  if (c.reset_ref_mode == B747_RESET_CONST) {
    double v = uni(4, -c.vartheta_max, -1 * kPi / 180);
    v *= (uniform53(sd, env, epi, 5) < 0.5) ? 1.0 : -1.0;
    ep.vref = v;
  } else if (c.reset_ref_mode == B747_RESET_OSCILLATING) {
    double A1 = uni(4, 0, c.vartheta_max);
    double A2 = uni(5, 0, c.vartheta_max - A1);
    double A3 = uni(6, 0, c.vartheta_max - A1 - A2);
    ep.oscA[0] = A1; ep.oscA[1] = A2; ep.oscA[2] = A3;
    for (int i = 0; i < 3; i++) ep.oscf[i] = uni(7 + i, 0.01, 0.5);
    ep.osc = 1;
  } else if (c.reset_ref_mode == B747_RESET_HYBRID) {
    ep.use_ctrl = uniform53(sd, env, epi, 4) < 0.5;
    if (ep.use_ctrl) ep.href = h0 + uni(5, -1000, 1000);
    else ep.vref = uni(5, -c.vartheta_max, c.vartheta_max);
  }
  ep.s0[0] = 0; ep.s0[1] = h0; ep.s0[2] = Vx; ep.s0[3] = Vy; ep.s0[4] = 0; ep.s0[5] = wz0;
  if (c.disturbance_mode == B747_DIST_AERO) {
    const double mean[5] = {-0.1, 0.1, -0.1, -0.1, 0.1};
    for (int i = 0; i < 5; i++) {
      if (c.has_fixed_aero_err) { ep.aerr[i] = c.fixed_aero_err[i]; continue; }
      double u1 = 1.0 - uniform53(sd, env, epi, 10 + 2 * i);
      double u2 = uniform53(sd, env, epi, 11 + 2 * i);
      double z = sqrt(-2.0 * log(u1)) * cos(2.0 * kPi * u2);
      ep.aerr[i] = mean[i] + 0.5 * z;  // np.random.normal(mean, 0.5)
    }
  }
}

// Block-level episode statistics: done lanes are found with a warp ballot, their (count, return,
// length, return^2) are reduced with shuffles, one shared-memory partial per warp, and one set of
// atomics per block -- the only cross-environment traffic on the step path.
struct EpStatsSmem { double v[4][32]; };

__device__ inline void block_episode_stats(EpStatsSmem& sm, bool done, double ep_ret, double ep_len, double* g_stats) {
  const unsigned full = 0xffffffffu;
  unsigned ballot = __ballot_sync(full, done);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = (blockDim.x + 31) >> 5;
  double v0 = 0, v1 = 0, v2 = 0, v3 = 0;
  if (ballot) {  // warp-uniform
    v0 = done ? 1.0 : 0.0; v1 = done ? ep_ret : 0.0; v2 = done ? ep_len : 0.0; v3 = done ? ep_ret * ep_ret : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      v0 += __shfl_xor_sync(full, v0, o); v1 += __shfl_xor_sync(full, v1, o);
      v2 += __shfl_xor_sync(full, v2, o); v3 += __shfl_xor_sync(full, v3, o);
    }
  }
  if (lane == 0) { sm.v[0][warp] = v0; sm.v[1][warp] = v1; sm.v[2][warp] = v2; sm.v[3][warp] = v3; }
  __syncthreads();
  if (warp == 0) {
    double a0 = lane < nwarp ? sm.v[0][lane] : 0.0, a1 = lane < nwarp ? sm.v[1][lane] : 0.0;
    double a2 = lane < nwarp ? sm.v[2][lane] : 0.0, a3 = lane < nwarp ? sm.v[3][lane] : 0.0;
    if (__ballot_sync(full, a0 != 0.0)) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        a0 += __shfl_xor_sync(full, a0, o); a1 += __shfl_xor_sync(full, a1, o);
        a2 += __shfl_xor_sync(full, a2, o); a3 += __shfl_xor_sync(full, a3, o);
      }
      if (lane == 0) {
        atomicAdd(g_stats + 0, a0); atomicAdd(g_stats + 1, a1); atomicAdd(g_stats + 2, a2); atomicAdd(g_stats + 3, a3);
      }
    }
  }
}

// Warp-level form for persistent kernels: no block barrier per tile; done lanes are found with a ballot, reduced with
// shuffles and added to the block's shared-memory partials (flushed to HBM once, when the block has finished).
__device__ inline void warp_episode_stats(double* s_stats, bool done, double ep_ret, double ep_len) {
  const unsigned full = 0xffffffffu;
  if (!__ballot_sync(full, done)) return;  // warp-uniform
  double v0 = done ? 1.0 : 0.0, v1 = done ? ep_ret : 0.0, v2 = done ? ep_len : 0.0, v3 = done ? ep_ret * ep_ret : 0.0;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    v0 += __shfl_xor_sync(full, v0, o); v1 += __shfl_xor_sync(full, v1, o);
    v2 += __shfl_xor_sync(full, v2, o); v3 += __shfl_xor_sync(full, v3, o);
  }
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(s_stats + 0, v0); atomicAdd(s_stats + 1, v1); atomicAdd(s_stats + 2, v2); atomicAdd(s_stats + 3, v3);
  }
}

__device__ inline double nan_to_num(double x) {  // np.nan_to_num (core/model.py:167-168)
  if (x != x) return 0.0;
  if (isinf(x)) return x > 0 ? 1.7976931348623157e308 : -1.7976931348623157e308;
  return x;
}


// ---------------------------------------------------------------------------------------------
// Trace: the reference's `Storage` recorder and `calc_stepinfo` (tools/general.py:46-61,315-329), hooked where
// Controller._post_step records -- after EVERY model step (core/controller.py:209-228).
//   recorder: rec[step][REC field][env] (float64), step = model step of the running episode (0-based), up to
//             rec_cap steps; the recorded names and unit conversions are Controller._post_step's.
//   tracker : calc_stepinfo evaluated online, O(1) state per env and signal -- first sample, extrema, last
//             sample, index of the first sample inside the 5 % band (rise) and of the last one outside it
//             (settling).  Slot 0 tracks the pitch angle against vartheta_ref (Controller.stepinfo_SS), slot 1
//             the altitude against hzh (stepinfo_CS).  calc_stepinfo normalises every sample with the LAST
//             reference value; the online form uses the current one, identical for the constant references
//             the reference's evaluation harness uses (neural/callbacks.py:61-100, neural/agent.py:235-266).
//   At `done` the tracker (+ Controller.quality) is copied to `snap` before the auto-reset clears it.
// Evaluation feature: state sits in HBM and is read-modify-written per model step; a handle without it pays nothing.
// ---------------------------------------------------------------------------------------------
enum RecField { REC_t = 0, REC_U_com, REC_U_PID, REC_deltaz, REC_hzh, REC_vartheta_ref, REC_U_RL, REC_x, REC_y, REC_Vx,
                REC_Vy, REC_vartheta, REC_wz, NREC };
enum TrkField { TRK_y0 = 0, TRK_ymax, TRK_ymin, TRK_ylast, TRK_irise, TRK_iout, TRK_n, TRK_ybase, TRK_quality, NTRK };
struct TraceState {
  double* trk = nullptr;   // [2][NTRK][n_pad]
  double* snap = nullptr;  // [2][NTRK][n_pad]
  double* rec = nullptr;   // [rec_cap][NREC][rec_stride]
  int rec_cap = 0;
  int rec_stride = 0;      // = n_envs (no padding: a single-env facade records 2000 x 13 doubles, not x 128)
};
struct TraceSample {  // what Controller._post_step reads after one model step (stage-4 signals), SI units / radians
  double t, U_com, U_PID, deltaz_RP, hzh, vref, U_RL, x, y, Vx, Vy, th, wz;
};

__device__ inline void trk_update(double* __restrict__ T, size_t np, int i, double y, double ybase) {
#define TK(f) T[(size_t)(f) * np + i]
  const double n = TK(TRK_n);
  double y0 = TK(TRK_y0), ymax = TK(TRK_ymax), ymin = TK(TRK_ymin), irise = TK(TRK_irise), iout = TK(TRK_iout);
  if (n == 0.0) { y0 = y; ymax = y; ymin = y; irise = -1.0; iout = -1.0; }
  ymax = y > ymax ? y : ymax;
  ymin = y < ymin ? y : ymin;
  const double band = 0.05, ratio = (y - y0) / (ybase - y0);
  if (irise < 0.0 && ratio >= (1 - band)) irise = n;
  if (ratio <= 1 - band || ratio >= 1 + band) iout = n;
  TK(TRK_y0) = y0; TK(TRK_ymax) = ymax; TK(TRK_ymin) = ymin; TK(TRK_ylast) = y; TK(TRK_irise) = irise;
  TK(TRK_iout) = iout; TK(TRK_n) = n + 1.0; TK(TRK_ybase) = ybase;
#undef TK
}

// after one model step; `step` = 0-based model step of the episode (tick after the step - 1)
__device__ inline void trace_model_step(const TraceState& tr, size_t np, int i, int step, const TraceSample& s) {
  const double vartheta_deg = nan_to_num(s.th) * (180 / kPi);  // `v *= 180/pi` on state_dict['vartheta']
  const double vref_deg = s.vref * 180 / kPi;                  // self.vartheta_ref*180/pi
  if (tr.rec && step < tr.rec_cap) {
    const size_t rs = (size_t)tr.rec_stride;
    double* R = tr.rec + ((size_t)step * NREC) * rs + i;
    R[REC_t * rs] = s.t; R[REC_U_com * rs] = s.U_com; R[REC_U_PID * rs] = s.U_PID;
    R[REC_deltaz * rs] = s.deltaz_RP * 180 / kPi; R[REC_hzh * rs] = s.hzh; R[REC_vartheta_ref * rs] = vref_deg;
    R[REC_U_RL * rs] = s.U_RL; R[REC_x * rs] = nan_to_num(s.x); R[REC_y * rs] = nan_to_num(s.y);
    R[REC_Vx * rs] = nan_to_num(s.Vx); R[REC_Vy * rs] = nan_to_num(s.Vy); R[REC_vartheta * rs] = vartheta_deg;
    R[REC_wz * rs] = nan_to_num(s.wz);
  }
  if (tr.trk) {
    trk_update(tr.trk, np, i, vartheta_deg, vref_deg);
    trk_update(tr.trk + (size_t)NTRK * np, np, i, nan_to_num(s.y), s.hzh);
  }
}

// at done: freeze the finished episode's tracker (+ Controller.quality, core/controller.py:334-336)
__device__ inline void trace_snapshot(const TraceState& tr, size_t np, int i, double quality) {
  if (!tr.trk) return;
  for (int w = 0; w < 2; w++)
    for (int f = 0; f < NTRK; f++) {
      const size_t k = ((size_t)w * NTRK + f) * np + i;
      tr.snap[k] = f == TRK_quality ? quality : tr.trk[k];
    }
}
__device__ inline void trace_clear(const TraceState& tr, size_t np, int i) {
  if (!tr.trk) return;
  tr.trk[(size_t)TRK_n * np + i] = 0.0;
  tr.trk[((size_t)NTRK + TRK_n) * np + i] = 0.0;
}

__host__ __device__ inline int obs_dim_of(int obs_type) {
  switch (obs_type) {
    case B747_OBS_PID_LIKE: return 3;
    case B747_OBS_SPEED_MODE: return 5;
    case B747_OBS_PID_AERO: return 8;
    case B747_OBS_PID_SPEED_AERO: return 10;
    case B747_OBS_MODEL_STATE: return 7;
  }
  return -1;
}

}  // namespace b747
