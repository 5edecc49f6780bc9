// b747_kernels_f64.cu -- float64 parity kernels (compiled with -fmad=false: the reference DLL is
// SSE2 code without fused multiply-add, so products and sums are rounded separately here too).
//
// One environment per thread; the whole env step -- Controller.step's action law
// (core/controller.py:231-251), K model steps (model_simple_step dll@0x16d0), observation
// (env/ctrl_env.py:200-247), reward (env/ctrl_env.py:109-192), done (env/ctrl_env.py:255-257) and the
// VecEnv auto-reset (Controller.reset, core/controller.py:134-201) -- is one launch.
#include "b747_kernels.h"
#include "b747_model_f64.cuh"

namespace b747 {

__device__ __forceinline__ void load_regs64(const double* __restrict__ sl, const int* __restrict__ tick,
                                            const int* __restrict__ flags, const uint32_t* __restrict__ epi, size_t np,
                                            int i, Regs64& r) {
#define LD(slot) sl[(size_t)(slot) * np + i]
#pragma unroll
  for (int k = 0; k < 16; k++) r.X[k] = LD(S_x + k);
  r.df_x = LD(S_df_x); r.df_y = LD(S_df_y); r.rl_prev = LD(S_rl_prev);
#pragma unroll
  for (int k = 0; k < 4; k++) r.uh[k] = LD(S_uh0 + k);
  r.d1_u = LD(S_d1_u); r.d2_u = LD(S_d2_u);
  r.deltaz = LD(S_deltaz); r.vartheta = LD(S_vartheta); r.h_zh = LD(S_h_zh);
#pragma unroll
  for (int k = 0; k < 5; k++) r.aerr[k] = LD(S_aerr0 + k);
  r.sig_upid = LD(S_sig_upid); r.sig_vzh = LD(S_sig_vzh);
  r.vref = LD(S_vref); r.href = LD(S_href);
#pragma unroll
  for (int k = 0; k < 3; k++) { r.oscA[k] = LD(S_oscA0 + k); r.oscf[k] = LD(S_oscf0 + k); }
  r.ep_return = LD(S_ep_return); r.tf_tp = LD(S_tf_tp);
#undef LD
  r.tick = tick[i]; r.flags = flags[i]; r.ep_idx = epi[i];
  r.use_PID_CS = (r.flags & FL_USE_CTRL) ? 1.0 : 0.0;
}

__device__ __forceinline__ void store_regs64(double* __restrict__ sl, int* __restrict__ tick, int* __restrict__ flags,
                                             uint32_t* __restrict__ epi, size_t np, int i, const Regs64& r) {
#define ST(slot, v) sl[(size_t)(slot) * np + i] = (v)
#pragma unroll
  for (int k = 0; k < 16; k++) ST(S_x + k, r.X[k]);
  ST(S_df_x, r.df_x); ST(S_df_y, r.df_y); ST(S_rl_prev, r.rl_prev);
#pragma unroll
  for (int k = 0; k < 4; k++) ST(S_uh0 + k, r.uh[k]);
  ST(S_d1_u, r.d1_u); ST(S_d2_u, r.d2_u);
  ST(S_deltaz, r.deltaz); ST(S_vartheta, r.vartheta); ST(S_h_zh, r.h_zh);
#pragma unroll
  for (int k = 0; k < 5; k++) ST(S_aerr0 + k, r.aerr[k]);
  ST(S_sig_upid, r.sig_upid); ST(S_sig_vzh, r.sig_vzh);
  ST(S_vref, r.vref); ST(S_href, r.href);
#pragma unroll
  for (int k = 0; k < 3; k++) { ST(S_oscA0 + k, r.oscA[k]); ST(S_oscf0 + k, r.oscf[k]); }
  ST(S_ep_return, r.ep_return); ST(S_tf_tp, r.tf_tp);
#undef ST
  tick[i] = r.tick; flags[i] = r.flags; epi[i] = r.ep_idx;
}

// Controller.reset (model side) + Model.initialize for one env.
__device__ __forceinline__ void env_reset64(const DevCfg& c, const double* __restrict__ P, const Episode& ep, Regs64& r,
                                            double* __restrict__ sl, size_t np, int i) {
  int use_ctrl = (c.ctrl_type == B747_CTRL_SEMI_MANUAL || c.ctrl_type == B747_CTRL_FULL_AUTO);
  if (c.reset_ref_mode == B747_RESET_HYBRID) {
    // Controller._init_model re-creates the Model: altitude set-point and aero errors back to the DLL defaults.  The
    // handle's and the env's tunables (PID_SS, PID_CS, P, ...) are configuration and survive (b747.h, b747_set_param)
    use_ctrl = ep.use_ctrl;
    r.h_zh = B747_DEF_H_ZH;
#pragma unroll
    for (int k = 0; k < 5; k++) r.aerr[k] = 0.0;
  }
  r.flags = (use_ctrl ? FL_USE_CTRL : 0) | (ep.osc ? FL_OSC : 0);
  r.use_PID_CS = use_ctrl ? 1.0 : 0.0;
  if (c.disturbance_mode == B747_DIST_AERO) {
#pragma unroll
    for (int k = 0; k < 5; k++) r.aerr[k] = ep.aerr[k];
  }
  model_init64(P, ep.s0, r);
  r.vref = ep.vref; r.href = ep.href;
#pragma unroll
  for (int k = 0; k < 3; k++) { r.oscA[k] = ep.oscA[k]; r.oscf[k] = ep.oscf[k]; }
  r.ep_return = 0.0;
#pragma unroll
  for (int k = 0; k < 6; k++) sl[(size_t)(NSLOT_F64 + k) * np + i] = ep.s0[k];  // the DLL's `state0` param
}

__device__ __forceinline__ void episode_from_slots(const double* __restrict__ sl, size_t np, int i, const Regs64& r,
                                                   Episode& ep) {
#pragma unroll
  for (int k = 0; k < 6; k++) ep.s0[k] = sl[(size_t)(NSLOT_F64 + k) * np + i];
  ep.vref = r.vref; ep.href = r.href;
#pragma unroll
  for (int k = 0; k < 3; k++) { ep.oscA[k] = r.oscA[k]; ep.oscf[k] = r.oscf[k]; }
#pragma unroll
  for (int k = 0; k < 5; k++) ep.aerr[k] = r.aerr[k];
  ep.use_ctrl = (r.flags & FL_USE_CTRL) != 0;
  ep.osc = (r.flags & FL_OSC) != 0;
}

// Controller.vartheta_ref (core/controller.py:267-270)
__device__ __forceinline__ double vartheta_ref64(const Regs64& r) { return r.use_PID_CS != 0.0 ? r.sig_vzh : r.vartheta; }

// ControllerEnv._get_obs (env/ctrl_env.py:200-247) from the stage-4 pass
__device__ __forceinline__ void get_obs64(const DevCfg& c, const Regs64& r, const Pass64& o, const double Xs4[16],
                                          double obs[10]) {
  double mx[10];
  int n;
  if (c.obs_type == B747_OBS_MODEL_STATE) {
    obs[0] = vartheta_ref64(r);
    obs[1] = nan_to_num(Xs4[IX_x]); obs[2] = nan_to_num(Xs4[IX_h]); obs[3] = nan_to_num(Xs4[IX_Vx]);
    obs[4] = nan_to_num(Xs4[IX_Vy]); obs[5] = nan_to_num(o.th); obs[6] = nan_to_num(Xs4[IX_wz]);
    mx[0] = 10 * kPi / 180; mx[1] = 12000; mx[2] = 15000; mx[3] = 500; mx[4] = 100; mx[5] = kPi; mx[6] = kPi;
    n = 7;
  } else {
    obs[0] = Xs4[IX_dvi]; obs[1] = o.dv; obs[2] = o.dv_dt;
    mx[0] = 60 * kPi; mx[1] = kPi; mx[2] = kPi;
    n = 3;
    if (c.obs_type == B747_OBS_SPEED_MODE || c.obs_type == B747_OBS_PID_SPEED_AERO) {
      obs[n] = nan_to_num(Xs4[IX_Vx]); mx[n++] = 500;
      obs[n] = nan_to_num(Xs4[IX_Vy]); mx[n++] = 100;
    }
    if (c.obs_type == B747_OBS_PID_AERO || c.obs_type == B747_OBS_PID_SPEED_AERO) {
      obs[n] = o.CXa; mx[n++] = 0.5;
      obs[n] = o.CYa; mx[n++] = 2;
      obs[n] = o.mz; mx[n++] = 0.6;
      obs[n] = o.dCm; mx[n++] = 0.05;
      obs[n] = o.K_alpha; mx[n++] = 1.;
    }
  }
  if (c.norm_obs)
    for (int k = 0; k < n; k++) obs[k] /= mx[k];
}

// ControllerEnv.get_reward (env/ctrl_env.py:109-192); all inputs are stage-4 signals.
__device__ __forceinline__ double get_reward64(const DevCfg& c, Regs64& r, const Pass64& o, double itse, double time) {
  const double* k = c.rew;
  double vr = vartheta_ref64(r);
  double vf = vr != 0.0 ? vr : c.vartheta_max;
  double dv = o.dv;
  switch (c.rew_type) {
    case B747_REW_CLASSIC: {
      double r1 = 0.50 * exp(-k[3] * (k[0] * fabs(dv) + k[1] * 1 * fabs(o.dv_dt) + k[2] * fabs(o.dv_dt_dt)) / fabs(vf));
      double r2 = (vr * dv < 0) ? 0.20 * exp(-k[7] * fabs(dv / vf)) : 0.20;
      double r3 = (fabs(dv / vf) > 0.05) ? 0.20 * exp(-k[6] * time) : 0.20;
      double r4 = 0.1 * exp(-k[4] * itse / (vf * vf));
      double rf = 0;
      if (c.ctrl_mode == B747_MODE_DIRECT) rf = -k[5] * fabs(dv / (2 * vf)) * (fabs(r.deltaz - o.U_com_PID)) / (34 * kPi / 180);
      return r1 + r2 + r3 + r4 + rf;
    }
    case B747_REW_PID_LIKE:
      return exp(-k[0] * fabs(o.U_com - o.U_com_PID) / (34 * kPi / 180));
    case B747_REW_QUALITY:
    case B747_REW_MINIMAL:
      return exp(-60 * 0.1 * itse / (c.tk * (vr * vr)));  // Controller.quality, core/controller.py:334-336
    case B747_REW_TF_REFERENCE: {
      double overshoot = fabs(dv / vf) * 100;
      if (overshoot > 5) r.tf_tp = time;
      return exp(-k[2] * fabs(overshoot - k[0]) * fabs(k[1] - r.tf_tp));
    }
  }
  return 0.0;
}

__device__ __forceinline__ void export_signals64(double* __restrict__ sig, size_t np, int i, const Regs64& r,
                                                 const Pass64& o, const double Xs4[16], double time) {
#define SG(name, v) sig[(size_t)SIG_##name * np + i] = (v)
  SG(state_x, Xs4[IX_x]); SG(state_y, Xs4[IX_h]); SG(state_Vx, Xs4[IX_Vx]); SG(state_Vy, Xs4[IX_Vy]);
  SG(state_vartheta, o.th); SG(state_wz, Xs4[IX_wz]); SG(sim_time, time); SG(vartheta_zh, o.vartheta_zh);
  SG(U_com_PID, o.U_com_PID); SG(CXa, o.CXa); SG(CYa, o.CYa); SG(mz, o.mz); SG(K_alpha, o.K_alpha);
  SG(dCm_ddeltaz, o.dCm); SG(U_com, o.U_com); SG(deltaz_RP, o.deltaz_RP); SG(dvartheta, o.dv);
  SG(dvartheta_int, Xs4[IX_dvi]); SG(dvartheta_dt, o.dv_dt); SG(dvartheta_dt_dt, o.dv_dt_dt);
  SG(TAE, o.TAE); SG(ITAE, Xs4[IX_itae]); SG(TSE, o.TSE); SG(ITSE, Xs4[IX_itse]); SG(AE, o.AE);
  SG(IAE, Xs4[IX_iae]); SG(SE, o.SE); SG(ISE, Xs4[IX_ise]); SG(alpha, o.alpha); SG(V, o.V); SG(Mach, o.Mach);
  SG(CXa_tab, o.CXa_tab); SG(CYa_tab, o.CYa_tab); SG(mz_tab, o.mz_tab); SG(dCm_tab, o.dCm_tab);
#undef SG
}

__device__ __forceinline__ void load_tables64(double* sP) {
  static const __device__ double gP[kNP] = B747_P_INIT;
  for (int k = threadIdx.x; k < kNP; k += blockDim.x) sP[k] = gP[k];
  __syncthreads();
}

// per-env twins (PE): the launch's tunables with this env's rows in place of the per-env names
__device__ __forceinline__ void env_params64(const EnvParams& pe, const ModelParams& batch, size_t np, int i, ModelParams& mp) {
  mp = batch;
  const double* R = pe.rows;
#define EPV(k) R[(size_t)(k) * np + i]
  mp.m0 = EPV(EP_m0); mp.Iz = EPV(EP_Iz); mp.P = EPV(EP_P); mp.S = EPV(EP_S); mp.c_ = EPV(EP_c);
#pragma unroll
  for (int k = 0; k < 4; k++) { mp.PID_SS[k] = EPV(EP_PID_SS + k); mp.PID_CS[k] = EPV(EP_PID_CS + k); }
#undef EPV
}

// ------------------------------------------------------------------------------------------
// ControllerEnv.step for every env of the handle.  PE: the per-env twin, which reads the tunables from the env's rows
// in `pe` and redraws the ranged ones at an auto-reset.
// ------------------------------------------------------------------------------------------
constexpr int kF64MinBlocks = 2;  // measured: beats 3 / 4 blocks at 168 / 128 registers (1.783 vs 2.04-2.22 ms: spills)
template <bool PE>
__global__ void __launch_bounds__(128, kF64MinBlocks) k_env_step64(DevCfg c, StateF64 st, const double* __restrict__ actions,
                                                    double* __restrict__ obs_out, double* __restrict__ rew_out,
                                                    uint8_t* __restrict__ done_out, double* __restrict__ term_obs,
                                                    const __grid_constant__ EnvParams pe) {
  __shared__ double sP[kNP];
  __shared__ EpStatsSmem sst;
  load_tables64(sP);
  const int i = c.env_lo + blockIdx.x * blockDim.x + threadIdx.x;
  const bool live = i < c.env_hi;
  const size_t np = (size_t)c.n_pad;
  bool done = false;
  double ep_ret = 0.0, ep_len = 0.0;
  if (live) {
    Regs64 r;
    load_regs64(st.slots, st.tick, st.flags, st.ep_idx, np, i, r);
    ModelParams mpe;
    if (PE) env_params64(pe, c.mp, np, i, mpe);
    const ModelParams& mp = PE ? mpe : c.mp;
    Pass64 o;
    double Xs4[16];
    double a = actions[i];
    if (c.norm_act) a *= c.action_max;  // env/ctrl_env.py:262-264
    // Controller.step (core/controller.py:233-251): reference, then the action law
    const double time0 = (double)r.tick * kH;  // model.time == exported sim_time
    if (!(r.flags & FL_USE_CTRL)) {
      if (r.flags & FL_OSC)
        r.vartheta = r.oscA[0] * sin(2 * kPi * r.oscf[0] * time0) + r.oscA[1] * sin(2 * kPi * r.oscf[1] * time0) +
                     r.oscA[2] * sin(2 * kPi * r.oscf[2] * time0);
      else
        r.vartheta = r.vref;
    } else {
      r.h_zh = r.href;
    }
    if (!(c.mp.use_PID_SS != 0.0)) {
      const double lim = 17 * kPi / 180;
      double dz;
      switch (c.ctrl_mode) {
        case B747_MODE_ADD_PROC: dz = (1 + a) * r.sig_upid; dz = dz < -lim ? -lim : (dz > lim ? lim : dz); break;
        case B747_MODE_ADD_DIRECT: dz = a + r.sig_upid; dz = dz < -lim ? -lim : (dz > lim ? lim : dz); break;
        case B747_MODE_ANG_VEL: dz = r.deltaz + a * c.sample_time; dz = dz < -lim ? -lim : (dz > lim ? lim : dz); break;
        default: dz = a; break;
      }
      r.deltaz = dz;
    }
    const bool tracing = st.trace.trk || st.trace.rec;
#pragma unroll 1
    for (int k = 0; k < c.substeps; k++) {
      model_step64(sP, mp, r, o, Xs4);
      if (tracing) {  // Controller._post_step (core/controller.py:209-228)
        TraceSample ts;
        ts.t = (double)r.tick * kH; ts.U_com = o.U_com; ts.U_PID = o.U_com_PID; ts.deltaz_RP = o.deltaz_RP;
        ts.hzh = r.h_zh; ts.vref = r.use_PID_CS != 0.0 ? o.vartheta_zh : r.vartheta; ts.U_RL = a;
        ts.x = Xs4[IX_x]; ts.y = Xs4[IX_h]; ts.Vx = Xs4[IX_Vx]; ts.Vy = Xs4[IX_Vy]; ts.th = o.th; ts.wz = Xs4[IX_wz];
        trace_model_step(st.trace, np, i, r.tick - 1, ts);
      }
    }
    r.sig_upid = o.U_com_PID; r.sig_vzh = o.vartheta_zh;
    const double time = (double)r.tick * kH;
    if (st.trace.trk) {  // Controller.quality of the running episode
      const double vr = vartheta_ref64(r);
      const double q = exp(-60 * 0.1 * Xs4[IX_itse] / (c.tk * (vr * vr)));
      st.trace.trk[(size_t)TRK_quality * np + i] = q;
      st.trace.trk[((size_t)NTRK + TRK_quality) * np + i] = q;
    }
    double obs[10];
    get_obs64(c, r, o, Xs4, obs);
    double rew = get_reward64(c, r, o, Xs4[IX_itse], time);
    r.ep_return += rew;
    done = (int64_t)r.tick >= c.done_tick;  // Controller.is_done with time == fl(tick*0.01)
    if (c.use_limiter && (fabs(nan_to_num(o.th)) > 5 * kPi / 180 + c.vartheta_max || r.deltaz > c.action_max)) done = true;
    if (st.sig) export_signals64(st.sig, np, i, r, o, Xs4, time);
    rew_out[i] = rew;
    done_out[i] = done ? 1 : 0;
    const int od = c.obs_dim;
    if (term_obs)
      for (int k = 0; k < od; k++) term_obs[(size_t)i * od + k] = obs[k];
    if (done) {
      ep_ret = r.ep_return; ep_len = (double)(r.tick / c.substeps);
      st.last_ret[i] = ep_ret; st.last_len[i] = r.tick / c.substeps;
      if (st.trace.trk) trace_snapshot(st.trace, np, i, st.trace.trk[(size_t)TRK_quality * np + i]);
      if (c.auto_reset) {
        trace_clear(st.trace, np, i);
        Episode ep;
        if (c.reset_ref_mode == B747_RESET_NONE) episode_from_slots(st.slots, np, i, r, ep);
        else {
          draw_episode(c, (uint64_t)(c.env_id_offset + i), r.ep_idx, ep);
          if (PE) draw_env_params(pe, c.seed, (uint64_t)(c.env_id_offset + i), r.ep_idx, np, i);
          r.ep_idx++;
        }
        env_reset64(c, sP, ep, r, st.slots, np, i);
        for (int k = 0; k < od; k++) obs[k] = 0.0;  // every exported signal is zero after initialize
        if (st.sig) for (int k = 0; k < NSIG; k++) st.sig[(size_t)k * np + i] = 0.0;
      }
    }
    for (int k = 0; k < od; k++) obs_out[(size_t)i * od + k] = obs[k];
    store_regs64(st.slots, st.tick, st.flags, st.ep_idx, np, i, r);
  }
  block_episode_stats(sst, done, ep_ret, ep_len, st.stats);
}

// Model.step x n_steps (core/model.py:247-250): no action law, no reward.  PE: per-env twin.
template <bool PE>
__global__ void __launch_bounds__(128) k_model_step64(DevCfg c, StateF64 st, int n_steps, const __grid_constant__ EnvParams pe) {
  __shared__ double sP[kNP];
  load_tables64(sP);
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= c.n_envs) return;
  const size_t np = (size_t)c.n_pad;
  Regs64 r;
  load_regs64(st.slots, st.tick, st.flags, st.ep_idx, np, i, r);
  ModelParams mpe;
  if (PE) env_params64(pe, c.mp, np, i, mpe);
  const ModelParams& mp = PE ? mpe : c.mp;
  Pass64 o;
  double Xs4[16];
#pragma unroll 1
  for (int k = 0; k < n_steps; k++) model_step64(sP, mp, r, o, Xs4);
  r.sig_upid = o.U_com_PID; r.sig_vzh = o.vartheta_zh;
  if (st.sig) export_signals64(st.sig, np, i, r, o, Xs4, (double)r.tick * kH);
  store_regs64(st.slots, st.tick, st.flags, st.ep_idx, np, i, r);
}

// b747_reset of a handle with parameter ranges: the ranged rows of the envs about to draw a new episode, with the episode
// index k_reset64 is about to use (launched just before it)
__global__ void __launch_bounds__(128) k_env_param_draw64(DevCfg c, StateF64 st, const __grid_constant__ EnvParams pe,
                                                          const uint8_t* __restrict__ mask) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= c.n_envs || (mask && !mask[i])) return;
  draw_env_params(pe, c.seed, (uint64_t)(c.env_id_offset + i), st.ep_idx[i], (size_t)c.n_pad, i);
}

// Controller.reset + ControllerEnv.reset: random draws (eps==nullptr) or explicit episodes.
__global__ void __launch_bounds__(128) k_reset64(DevCfg c, StateF64 st, const uint8_t* __restrict__ mask,
                                                 const b747_episode* __restrict__ eps, double* __restrict__ obs_out) {
  __shared__ double sP[kNP];
  load_tables64(sP);
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= c.n_envs) return;
  if (mask && !mask[i]) return;
  const size_t np = (size_t)c.n_pad;
  Regs64 r;
  load_regs64(st.slots, st.tick, st.flags, st.ep_idx, np, i, r);
  Episode ep;
  if (eps) {
    episode_from_abi(eps[i], ep);
  } else if (c.reset_ref_mode == B747_RESET_NONE) {
    episode_from_slots(st.slots, np, i, r, ep);
  } else {
    draw_episode(c, (uint64_t)(c.env_id_offset + i), r.ep_idx, ep);
    r.ep_idx++;
  }
  env_reset64(c, sP, ep, r, st.slots, np, i);
  trace_clear(st.trace, np, i);
  if (obs_out)
    for (int k = 0; k < c.obs_dim; k++) obs_out[(size_t)i * c.obs_dim + k] = 0.0;
  if (st.sig) for (int k = 0; k < NSIG; k++) st.sig[(size_t)k * np + i] = 0.0;
  store_regs64(st.slots, st.tick, st.flags, st.ep_idx, np, i, r);
}

// Fresh handle: DLL .data defaults for the per-env tunables, then initialize with the default state0.
__global__ void __launch_bounds__(128) k_defaults64(DevCfg c, StateF64 st) {
  __shared__ double sP[kNP];
  load_tables64(sP);
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= c.n_pad) return;
  const size_t np = (size_t)c.n_pad;
  Regs64 r;
  const double s0[6] = B747_DEF_STATE0;
  r.flags = (c.ctrl_type == B747_CTRL_SEMI_MANUAL || c.ctrl_type == B747_CTRL_FULL_AUTO) ? FL_USE_CTRL : 0;
  r.ep_idx = 0;
  r.h_zh = B747_DEF_H_ZH;
  for (int k = 0; k < 5; k++) r.aerr[k] = 0.0;
  model_init64(sP, s0, r);
  r.vartheta = 0.0; r.deltaz = 0.0;
  r.vref = 0.0; r.href = B747_DEF_H_ZH;
  for (int k = 0; k < 3; k++) { r.oscA[k] = 0.0; r.oscf[k] = 0.0; }
  r.ep_return = 0.0; r.tf_tp = 0.0;
  for (int k = 0; k < 6; k++) st.slots[(size_t)(NSLOT_F64 + k) * np + i] = s0[k];
  if (st.sig) for (int k = 0; k < NSIG; k++) st.sig[(size_t)k * np + i] = 0.0;
  st.last_ret[i] = 0.0; st.last_len[i] = 0;
  store_regs64(st.slots, st.tick, st.flags, st.ep_idx, np, i, r);
}

// Model.initialize for envs of a raw-model handle: re-read state0, zero signals/time, deltaz = vartheta = 0.
__global__ void __launch_bounds__(128) k_model_init64(DevCfg c, StateF64 st) {
  __shared__ double sP[kNP];
  load_tables64(sP);
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= c.n_envs) return;
  const size_t np = (size_t)c.n_pad;
  Regs64 r;
  load_regs64(st.slots, st.tick, st.flags, st.ep_idx, np, i, r);
  double s0[6];
  for (int k = 0; k < 6; k++) s0[k] = st.slots[(size_t)(NSLOT_F64 + k) * np + i];
  model_init64(sP, s0, r);
  if (st.sig) for (int k = 0; k < NSIG; k++) st.sig[(size_t)k * np + i] = 0.0;
  store_regs64(st.slots, st.tick, st.flags, st.ep_idx, np, i, r);
}

// calc_stepinfo's final arithmetic (tools/general.py:46-61) + Controller.quality for every env.
// ts[j] = fl((j+1)*0.01) is model.time after model step j, so ts[j]-ts[0] reproduces the reference's floats.
__global__ void __launch_bounds__(128) k_transfer_metrics(int n_envs, size_t np, const double* __restrict__ T,
                                                          double* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_envs) return;
#define TK(f) T[(size_t)(f) * np + i]
  const double qnan = nan("");
  const double n = TK(TRK_n), ybase = TK(TRK_ybase), irise = TK(TRK_irise), iout = TK(TRK_iout);
  double* o = out + (size_t)i * 5;
  if (!(n > 0.0)) { o[0] = o[1] = o[2] = o[3] = qnan; o[4] = TK(TRK_quality); return; }
  const double t0 = 1.0 * kH;
  o[0] = ybase != 0.0 ? ((ybase > 0.0 ? TK(TRK_ymax) : TK(TRK_ymin)) - ybase) / ybase * 100 : qnan;
  o[1] = (irise >= 0.0 && irise <= n - 2.0) ? (irise + 1.0) * kH - t0 : qnan;  // range(0, len-1) skips the last sample
  o[2] = iout >= 0.0 ? (iout + 1.0) * kH - t0 : qnan;
  o[3] = fabs(TK(TRK_ylast) - ybase);
  o[4] = TK(TRK_quality);
#undef TK
}

static inline int grid_for(int n, int block) { return (n + block - 1) / block; }

void launch_transfer_metrics(const DevCfg& c, const TraceState& tr, int which, int snapshot, double* out_dev,
                             cudaStream_t s) {
  const double* T = (snapshot ? tr.snap : tr.trk) + (size_t)(which ? 1 : 0) * NTRK * (size_t)c.n_pad;
  k_transfer_metrics<<<grid_for(c.n_envs, 128), 128, 0, s>>>(c.n_envs, (size_t)c.n_pad, T, out_dev);
}

void launch_env_step64(const DevCfg& c, const StateF64& st, const double* actions, double* obs, double* rew,
                       uint8_t* done, double* term_obs, cudaStream_t s, const EnvParams* pe) {
  const int n = c.env_hi - c.env_lo;
  if (n <= 0) return;
  if (pe) k_env_step64<true><<<grid_for(n, 128), 128, 0, s>>>(c, st, actions, obs, rew, done, term_obs, *pe);
  else k_env_step64<false><<<grid_for(n, 128), 128, 0, s>>>(c, st, actions, obs, rew, done, term_obs, EnvParams{});
}
void launch_model_step64(const DevCfg& c, const StateF64& st, int n_steps, cudaStream_t s, const EnvParams* pe) {
  if (pe) k_model_step64<true><<<grid_for(c.n_envs, 128), 128, 0, s>>>(c, st, n_steps, *pe);
  else k_model_step64<false><<<grid_for(c.n_envs, 128), 128, 0, s>>>(c, st, n_steps, EnvParams{});
}
void launch_reset64(const DevCfg& c, const StateF64& st, const uint8_t* mask, const b747_episode* eps, double* obs,
                    cudaStream_t s, const EnvParams* pe) {
  if (pe && pe->ranged && !eps && c.reset_ref_mode != B747_RESET_NONE)
    k_env_param_draw64<<<grid_for(c.n_envs, 128), 128, 0, s>>>(c, st, *pe, mask);
  k_reset64<<<grid_for(c.n_envs, 128), 128, 0, s>>>(c, st, mask, eps, obs);
}
void launch_defaults64(const DevCfg& c, const StateF64& st, cudaStream_t s) {
  k_defaults64<<<grid_for(c.n_pad, 128), 128, 0, s>>>(c, st);
}
void launch_model_init64(const DevCfg& c, const StateF64& st, cudaStream_t s) {
  k_model_init64<<<grid_for(c.n_envs, 128), 128, 0, s>>>(c, st);
}

}  // namespace b747
