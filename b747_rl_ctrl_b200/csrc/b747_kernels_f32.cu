// b747_kernels_f32.cu -- throughput kernels ("f32" handles): ControllerEnv.step for every env in one
// launch, one env per thread, K fused RK4 substeps with the state in registers
// (replaces env/ctrl_env.py:260-270 -> core/controller.py:231-264 -> model_simple_step dll@0x16d0 xK).
//
// HBM layout (per handle): field groups of 16 bytes per env, group-major --
//   D[g][env] : double2   g = 0:(h,th) 1:(Vx,Vy) 2:(wz,ssi) 3:(ssf,dvi) 4:(itse,d1_u) 5:(vref,ep_return)
//                             6:(csi,csf) 7:(x,href) 8..10: oscillating-reference (A0,A1)(A2,f0)(f1,f2)
//                             11..13: state0
//   F[g][env] : float4    g = 0:(df_x,df_y,rl_prev,deltaz) 1:(uh0..uh3) 2:(sig_upid,d2_u,tick|look-up hints,flags|episode<<8)
//                             3:(sumA0..3) 4:(sumA4,tf_tp,sig_vzh,-)
// so each thread moves its state with 128-bit loads/stores and a warp touches one contiguous 512-byte
// segment per group.  The canonical configuration (LEAN) reads and writes groups D0-5 and F0-2 only:
// 144 B in + 144 B out per env step, plus action (4) obs (12) reward (4) done (1) = 309 B/env-step,
// independent of K.
//
// Instantiations of the step kernel (launch_env_step32 picks one per handle): tier 0 the canonical family on the LEAN
// layout, tier 1 the general layout without the altitude loop, tier 2 with it, tier 3 with recorder / tracker / signal
// export as well (each feature left out of a tier is left out of its instruction footprint).  All are persistent-warp kernels: grid = SMs x resident blocks, tables staged once per block.
#include <string.h>

#include <atomic>
#include <vector>

#include "b747_kernels.h"
#include "b747_model_mx.cuh"

namespace b747 {

enum { DG_h_th = 0, DG_V, DG_wz_ssi, DG_ssf_dvi, DG_itse_d1, DG_vref_ret, DG_cs, DG_x_href, DG_osc0, DG_osc1, DG_osc2,
       DG_s0a, DG_s0b, DG_s0c, ND_GROUPS };
enum { FG_act = 0, FG_uh, FG_misc, FG_sumA, FG_misc2, NF_GROUPS };
static_assert(DG_vref_ret == 5 && FG_misc == 2, "stage_issue copies D groups 0-5 and F groups 0-2");

// The tick word of F[FG_misc] also carries the look-up interval indices between launches (no extra HBM bytes): bit 31
// set = {tick in bits 0-13, indices in bits 14-30}; bit 31 clear = plain tick (episodes beyond 16383 ticks), no indices.
__host__ __device__ __forceinline__ void unpack_tick(uint32_t w, int& tick, uint32_t& ix) {
  if (w & 0x80000000u) { tick = (int)(w & 0x3fffu); ix = (w >> 14) & 0x1ffffu; }
  else { tick = (int)w; ix = kIxEmpty; }
}
__device__ __forceinline__ uint32_t pack_tick(int tick, uint32_t ix) {
  return ((unsigned)tick < 0x4000u && ix != kIxEmpty) ? (0x80000000u | (ix & 0x1ffffu) << 14 | (uint32_t)tick) : (uint32_t)tick;
}

// CSF = false (step kernel, tier 1): the altitude-loop states and h_zh are neither read nor integrated, so they are not
// carried through the step at all (8 registers); a reset inside the step writes their fresh values (store_mx, full).
// D, F: the group arrays with `np` envs per group -- the handle's state in HBM, or a warp's staged tile (np = 32).
template <bool GEN, bool CSF = true>
__device__ __forceinline__ void load_mx(const double2* __restrict__ D, const float4* __restrict__ F, size_t np, int i,
                                        RegsMx& r) {
  double2 d;
  d = D[DG_h_th * np + i]; r.h = d.x; r.th = d.y;
  d = D[DG_V * np + i]; r.Vx = d.x; r.Vy = d.y;
  d = D[DG_wz_ssi * np + i]; r.wz = d.x; r.ssi = d.y;
  d = D[DG_ssf_dvi * np + i]; r.ssf = d.x; r.dvi = d.y;
  d = D[DG_itse_d1 * np + i]; r.itse = d.x; r.d1_u = d.y;
  d = D[DG_vref_ret * np + i]; r.vref = d.x; r.ep_return = d.y;
  float4 f;
  f = F[FG_act * np + i]; r.df_x = f.x; r.df_y = f.y; r.rl_prev = f.z; r.deltaz = f.w;
  f = F[FG_uh * np + i]; r.uh[0] = f.x; r.uh[1] = f.y; r.uh[2] = f.z; r.uh[3] = f.w;
  f = F[FG_misc * np + i]; r.sig_upid = f.x; r.d2_u = f.y;
  uint32_t ix_hint;
  unpack_tick(__float_as_uint(f.z), r.tick, ix_hint);
  const unsigned fw = __float_as_uint(f.w);
  r.flags = (int)(fw & 0xffu); r.ep_idx = fw >> 8;
  if (GEN) {
    if (CSF) {
      d = D[DG_cs * np + i]; r.csi = d.x; r.csf = d.y;
      d = D[DG_x_href * np + i]; r.x = d.x; r.href = d.y;
    } else {
      r.csi = r.csf = 0.0; r.href = 0.0;
      r.x = ((const double*)(D + DG_x_href * np + i))[0];
    }
    d = D[DG_osc0 * np + i]; r.oscA[0] = d.x; r.oscA[1] = d.y;
    d = D[DG_osc1 * np + i]; r.oscA[2] = d.x; r.oscf[0] = d.y;
    d = D[DG_osc2 * np + i]; r.oscf[1] = d.x; r.oscf[2] = d.y;
    f = F[FG_sumA * np + i]; r.sumA[0] = f.x; r.sumA[1] = f.y; r.sumA[2] = f.z; r.sumA[3] = f.w;
    f = F[FG_misc2 * np + i]; r.sumA[4] = f.x; r.tf_tp = f.y; r.sig_vzh = f.z;
  } else {
    r.csi = r.csf = r.x = 0.0; r.href = B747_DEF_H_ZH;
#pragma unroll
    for (int k = 0; k < 3; k++) { r.oscA[k] = 0.0; r.oscf[k] = 0.0; }
#pragma unroll
    for (int k = 0; k < 5; k++) r.sumA[k] = 1.0f;
    r.tf_tp = 0.f; r.sig_vzh = 0.f;
  }
  r.vartheta = 0.0;
  r.tc = TabCache{};  // look-up cache: zero widths = nothing cached, refilled on first use (from the persisted indices)
  r.tc.ix = ix_hint;
}

// ---- TMA staging of the canonical (LEAN) state: each warp owns a 4.5 KB shared-memory buffer; one elected lane issues
// nine 512-byte bulk copies (one per 16-byte field group of the warp's 32 environments) that complete on the warp's
// mbarrier.  The copy of tile k+1 is issued as soon as tile k has been read into registers, so the HBM latency of the
// next tile hides behind the K model steps of the current one and the memory system always has every warp's next
// tile in flight (ncu r1e: at K = 1 the step was latency-bound at 58 % of the HBM roof with plain loads).
// Selected per launch (launch_env_step32): on for K <= kStagedMaxK substeps, where the step is HBM-latency bound
// (measured round 1, 1 Mi envs: K=1 0.0737 -> 0.0715 ms), off above (K=2 0.090 vs 0.091 ms, K=10 0.283 vs 0.289 ms: the extra
// shared-memory round trip costs issue slots the compute-bound regime does not have).
constexpr int kStagedMaxK = 1;
constexpr int kStageGroups = 9, kStageBytes = kStageGroups * 512;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  do {
    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                 : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  } while (!ok);
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
// one lane: queue the nine field groups of the 32 environments starting at env i0
__device__ __forceinline__ void stage_issue(const StateF32& st, size_t np, int i0, uint32_t buf, uint32_t bar) {
  mbar_expect_tx(bar, kStageBytes);
#pragma unroll
  for (int g = 0; g < 6; g++) bulk_g2s(buf + g * 512, st.D + (size_t)g * np + i0, 512, bar);
#pragma unroll
  for (int g = 0; g < 3; g++) bulk_g2s(buf + (6 + g) * 512, st.F + (size_t)g * np + i0, 512, bar);
}

// `full`: also the groups a step never changes (reference, aero sums, state0) -- reset paths only.
template <bool GEN, bool CSF = true>
__device__ __forceinline__ void store_mx(const StateF32& st, size_t np, int i, const RegsMx& r, bool full) {
  double2* __restrict__ D = st.D;
  float4* __restrict__ F = st.F;
  D[DG_h_th * np + i] = make_double2(r.h, r.th);
  D[DG_V * np + i] = make_double2(r.Vx, r.Vy);
  D[DG_wz_ssi * np + i] = make_double2(r.wz, r.ssi);
  D[DG_ssf_dvi * np + i] = make_double2(r.ssf, r.dvi);
  D[DG_itse_d1 * np + i] = make_double2(r.itse, r.d1_u);
  D[DG_vref_ret * np + i] = make_double2(r.vref, r.ep_return);
  F[FG_act * np + i] = make_float4(r.df_x, r.df_y, r.rl_prev, r.deltaz);
  F[FG_uh * np + i] = make_float4(r.uh[0], r.uh[1], r.uh[2], r.uh[3]);
  F[FG_misc * np + i] = make_float4(r.sig_upid, r.d2_u, __uint_as_float(pack_tick(r.tick, r.tc.ix)),
                                    __uint_as_float(((unsigned)r.flags & 0xffu) | (r.ep_idx << 8)));
  if (GEN) {
    if (CSF || full) {
      D[DG_cs * np + i] = make_double2(r.csi, r.csf);
      D[DG_x_href * np + i] = make_double2(r.x, r.href);
    } else {
      ((double*)(D + DG_x_href * np + i))[0] = r.x;
    }
    F[FG_misc2 * np + i] = make_float4(r.sumA[4], r.tf_tp, r.sig_vzh, 0.f);
    if (full) {
      D[DG_osc0 * np + i] = make_double2(r.oscA[0], r.oscA[1]);
      D[DG_osc1 * np + i] = make_double2(r.oscA[2], r.oscf[0]);
      D[DG_osc2 * np + i] = make_double2(r.oscf[1], r.oscf[2]);
      F[FG_sumA * np + i] = make_float4(r.sumA[0], r.sumA[1], r.sumA[2], r.sumA[3]);
    }
  }
}

__device__ __forceinline__ void store_state0_mx(const StateF32& st, size_t np, int i, const double s0[6]) {
  st.D[DG_s0a * np + i] = make_double2(s0[0], s0[1]);
  st.D[DG_s0b * np + i] = make_double2(s0[2], s0[3]);
  st.D[DG_s0c * np + i] = make_double2(s0[4], s0[5]);
}

template <bool GEN>
__device__ __forceinline__ void env_reset_mx(const DevCfg& c, const Episode& ep, RegsMx& r, const StateF32& st, size_t np,
                                             int i) {
  int use_ctrl = (c.ctrl_type == B747_CTRL_SEMI_MANUAL || c.ctrl_type == B747_CTRL_FULL_AUTO);
  if (c.reset_ref_mode == B747_RESET_HYBRID) {
    use_ctrl = ep.use_ctrl;
#pragma unroll
    for (int k = 0; k < 5; k++) r.sumA[k] = 1.0f;
  }
  r.flags = (use_ctrl ? FL_USE_CTRL : 0) | (ep.osc ? FL_OSC : 0);
  if (c.disturbance_mode == B747_DIST_AERO) {
#pragma unroll
    for (int k = 0; k < 5; k++) r.sumA[k] = (float)(ep.aerr[k] + 1.0);
  }
  model_init32(ep.s0, r);
  r.vref = ep.vref; r.href = ep.href;
#pragma unroll
  for (int k = 0; k < 3; k++) { r.oscA[k] = ep.oscA[k]; r.oscf[k] = ep.oscf[k]; }
  r.ep_return = 0.0;
  r.vartheta = 0.0;
  if (GEN) store_state0_mx(st, np, i, ep.s0);
}

__device__ __forceinline__ void episode_from_state_mx(const StateF32& st, size_t np, int i, const RegsMx& r, Episode& ep) {
  double2 d;
  d = st.D[DG_s0a * np + i]; ep.s0[0] = d.x; ep.s0[1] = d.y;
  d = st.D[DG_s0b * np + i]; ep.s0[2] = d.x; ep.s0[3] = d.y;
  d = st.D[DG_s0c * np + i]; ep.s0[4] = d.x; ep.s0[5] = d.y;
  ep.vref = r.vref; ep.href = r.href;
#pragma unroll
  for (int k = 0; k < 3; k++) { ep.oscA[k] = r.oscA[k]; ep.oscf[k] = r.oscf[k]; }
#pragma unroll
  for (int k = 0; k < 5; k++) ep.aerr[k] = (double)r.sumA[k] - 1.0;
  ep.use_ctrl = (r.flags & FL_USE_CTRL) != 0;
  ep.osc = (r.flags & FL_OSC) != 0;
}

// exp for the reward terms: one multiply and one MUFU.EX2 (2 ulp; the rewards carry a 2e-3 bound).  Arguments are <= 0
// except for non-finite states, where ex2 returns +inf / NaN like expf.
__device__ __forceinline__ float exp_fast(float x) { return ex2_fast(x * 1.4426950408889634f); }

__device__ __forceinline__ float nan_to_num_f(float x) {
  if (x != x) return 0.f;
  if (isinf(x)) return x > 0 ? 3.402823466e38f : -3.402823466e38f;
  return x;
}

// look-up tables in the fast path's layout (b747_tables.h; built on the host at handle creation): HBM/L2 -> shared
__device__ __forceinline__ void load_tables32(float4* sT, const float4* __restrict__ g) {
  for (int k = threadIdx.x; k < kFastCells; k += blockDim.x) sT[k] = g[k];
  __syncthreads();
}

// ------------------------------------------------------------------------------------------
constexpr int kStepThreads = 128, kStepWarps = kStepThreads / 32;  // threads per block of every step kernel tier
constexpr int kF32MinBlocks = 4;  // measured: 4 x 128 threads at 126 registers, no spills, beats every other occupancy point
constexpr int kExtMinBlocks = 3;
constexpr int kGenMinBlocks = 3;  // measured: 168 registers x 12 warps beats 242 x 8 (0.66 -> 0.52 ms per 1 Mi-env K=10 step)
// TIER 0: canonical family (LEAN layout); 1: general layout without the altitude loop (other observation layouts,
// oscillating references, aero disturbance, TF reward); 2: + the altitude loop (СУ PID); 3: + recorder, tracker, signal export.
// PFA: the next tile's actions are fetched while the current tile is stepped (host-mapped action buffers: a PCIe read
// has ~2 us of latency, a tile at K = 10 takes ~20 us).
template <int TIER, int SW = -1, bool STG = false, bool PFA = false>
__global__ void __launch_bounds__(kStepThreads, TIER >= 2 ? kGenMinBlocks : (TIER == 1 ? kExtMinBlocks : kF32MinBlocks))
k_env_step32(DevCfg c, MP32 mp, StateF32 st, const float* __restrict__ actions, float* __restrict__ obs_out,
             float* __restrict__ rew_out, uint8_t* __restrict__ done_out, float* __restrict__ term_obs,
             float4* __restrict__ out4, uint32_t* __restrict__ done_bits, unsigned int* __restrict__ tile_ctr) {
  // Persistent warps: the launch fills the GPU once (blocks = SMs x resident blocks per SM), the tables are staged into
  // shared memory once per block, and every warp then walks its own stride of 32-env tiles with no block-level
  // synchronisation until the episode statistics are flushed at the very end.
  constexpr bool GEN = TIER >= 1, CS = TIER >= 2, TRACE = TIER >= 3;
  constexpr bool STAGED = !GEN && STG;
  __shared__ float4 sT[kFastCells];
  __shared__ double s_stats[4];
  __shared__ __align__(128) unsigned char sStage[STAGED ? kStepWarps : 1][STAGED ? kStageBytes : 16];
  __shared__ __align__(8) unsigned long long sBar[kStepWarps];
  const size_t np = (size_t)c.n_pad;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps_per_block = blockDim.x >> 5;
  const int n_tiles = (c.env_hi - c.env_lo + 31) >> 5;
  const int wt0 = blockIdx.x * warps_per_block + warp, wstride = gridDim.x * warps_per_block;
  const uint32_t bar = smem_u32(&sBar[warp]), buf = smem_u32(&sStage[STAGED ? warp : 0][0]);
  if (threadIdx.x < 4) s_stats[threadIdx.x] = 0.0;
  if (STAGED && lane == 0) {
    mbar_init(bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    if (wt0 < n_tiles) stage_issue(st, np, c.env_lo + wt0 * 32, buf, bar);  // first tile: flies while the tables load
  }
  load_tables32(sT, st.tables);
  uint32_t phase = 0;
  float a_next = 0.f;
  if ((STAGED || PFA) && wt0 < n_tiles && c.env_lo + wt0 * 32 + lane < c.env_hi) a_next = actions[c.env_lo + wt0 * 32 + lane];
  // Tiles: the first one of every warp is fixed (wt0); the following ones are handed out by a global counter (tile_ctr)
  // in completion order, so a warp whose envs took slow paths (table re-searches, libm fall-backs of tumbling airframes)
  // does not hold a fixed share of the remaining work -- the static stride left the block barrier at the end of the
  // kernel with 8 % of all stall samples (ncu r2g).  STAGED keeps the static stride (its next tile is already in flight).
  const bool dyn = !STAGED && tile_ctr != nullptr;
#pragma unroll 1
  for (int wt = wt0; wt < n_tiles;) {
  int wn = wt + wstride;
  if (dyn) {
    unsigned nx = 0;
    if (lane == 0) nx = atomicAdd(tile_ctr, 1u);
    wn = wstride + (int)__shfl_sync(0xffffffffu, nx, 0);
  }
  const int i = c.env_lo + wt * 32 + lane;
  const bool live = i < c.env_hi;
  bool done = false;
  double ep_ret = 0.0, ep_len = 0.0;
  RegsMx r;
  float a = a_next;
  if (STAGED) {
    mbar_wait(bar, phase);
    phase ^= 1;
    const unsigned char* tile = &sStage[STAGED ? warp : 0][0];
    load_mx<false>((const double2*)tile, (const float4*)(tile + 6 * 512), 32, lane, r);
    __syncwarp();  // every lane has read its slots: the buffer can take the next tile
    if (wn < n_tiles) {
      if (lane == 0) stage_issue(st, np, c.env_lo + wn * 32, buf, bar);
      if (c.env_lo + wn * 32 + lane < c.env_hi) a_next = actions[c.env_lo + wn * 32 + lane];
    }
  }
  if (PFA && !STAGED) {
    const int in = c.env_lo + wn * 32 + lane;
    if (wn < n_tiles && in < c.env_hi) a_next = actions[in];
  }
  if (live) {
    if (!STAGED) {
      load_mx<GEN, CS>(st.D, st.F, np, i, r);
      if (!PFA) a = actions[i];
    }
    if (c.norm_act) a *= (float)c.action_max;
    const bool use_ctrl = CS && (r.flags & FL_USE_CTRL);
    // Controller.step: reference, then the action law (core/controller.py:233-251)
    if (!use_ctrl) {
      if (GEN && (r.flags & FL_OSC)) {
        const double time0 = (double)r.tick * kH;
        r.vartheta = r.oscA[0] * sin(2 * kPi * r.oscf[0] * time0) + r.oscA[1] * sin(2 * kPi * r.oscf[1] * time0) +
                     r.oscA[2] * sin(2 * kPi * r.oscf[2] * time0);
      } else {
        r.vartheta = r.vref;
      }
    }
    if (!((SW >= 0 ? SW : mp.sw) & SW_SS_ON)) {
      const float lim = (float)(17 * kPi / 180);
      float dz;
      switch (c.ctrl_mode) {
        case B747_MODE_ADD_PROC: dz = satf((1.f + a) * r.sig_upid, -lim, lim); break;
        case B747_MODE_ADD_DIRECT: dz = satf(a + r.sig_upid, -lim, lim); break;
        case B747_MODE_ANG_VEL: dz = satf(fmaf(a, (float)c.sample_time, r.deltaz), -lim, lim); break;
        default: dz = a; break;
      }
      r.deltaz = dz;
    }
    PassMx o;
    Stage4Mx s4;
    const bool tracing = TRACE && (st.trace.trk || st.trace.rec);  // recorder / tracker / signal export: tier 3 only
    const bool want_x = GEN && (c.obs_type == B747_OBS_MODEL_STATE || tracing);
#pragma unroll 1
    for (int k = 0; k < c.substeps; k++) {
      model_step32<TIER, SW>(sT, mp, c, r, o, s4, want_x);
      if (TRACE && tracing) {  // Controller._post_step (core/controller.py:209-228)
        TraceSample ts;
        ts.t = (double)r.tick * kH; ts.U_com = o.U_com; ts.U_PID = o.U_com_PID; ts.deltaz_RP = o.deltaz_RP;
        ts.hzh = r.href; ts.vref = use_ctrl ? (double)o.vartheta_zh : r.vartheta; ts.U_RL = a;
        ts.x = s4.x; ts.y = s4.h; ts.Vx = s4.Vx; ts.Vy = s4.Vy; ts.th = o.thd; ts.wz = s4.wz;
        trace_model_step(st.trace, np, i, r.tick - 1, ts);
      }
    }
    r.sig_upid = o.U_com_PID; r.sig_vzh = o.vartheta_zh;
    // stage-4 Derivative-block signals (float64 differences of the pitch error)
    const double dv_dt = (o.dv - r.d1_u) * 100.0;
    const float dv_dt_f = (float)dv_dt;
    const float dv_dt_dt = (dv_dt_f - r.d2_u) * 100.0f;
    const float dv = (float)o.dv;
    const float time = (float)r.tick * (float)kH;  // float32 product: 6e-8 relative, read by exp(-kt t) and the T?E signals only
    // Controller.vartheta_ref (core/controller.py:267-270)
    const float vr = use_ctrl ? r.sig_vzh : (float)r.vartheta;
    // observation (env/ctrl_env.py:200-247)
    float obs[GEN ? 10 : 3];
    const int od = GEN ? c.obs_dim : 3;
    if (!GEN) {  // canonical layout (PID_LIKE): three scalars, no indexed array
      obs[0] = (float)s4.dvi; obs[1] = dv; obs[2] = dv_dt_f;
      if (c.norm_obs) { obs[0] *= (float)(1.0 / (60 * kPi)); obs[1] *= (float)(1.0 / kPi); obs[2] *= (float)(1.0 / kPi); }
    } else {
      const float pi = (float)kPi;
      if (c.obs_type == B747_OBS_MODEL_STATE) {
        obs[0] = vr; obs[1] = nan_to_num_f(s4.x); obs[2] = nan_to_num_f(s4.h); obs[3] = nan_to_num_f(s4.Vx);
        obs[4] = nan_to_num_f(s4.Vy); obs[5] = nan_to_num_f(o.th); obs[6] = nan_to_num_f(s4.wz);
        if (c.norm_obs) {
          obs[0] /= (float)(10 * kPi / 180); obs[1] /= 12000.f; obs[2] /= 15000.f; obs[3] /= 500.f; obs[4] /= 100.f;
          obs[5] /= pi; obs[6] /= pi;
        }
      } else {
        float mx[10];
        int n = 3;
        obs[0] = (float)s4.dvi; obs[1] = dv; obs[2] = dv_dt_f;
        mx[0] = (float)(60 * kPi); mx[1] = pi; mx[2] = pi;
        if (c.obs_type == B747_OBS_SPEED_MODE || c.obs_type == B747_OBS_PID_SPEED_AERO) {
          obs[n] = nan_to_num_f(s4.Vx); mx[n++] = 500.f;
          obs[n] = nan_to_num_f(s4.Vy); mx[n++] = 100.f;
        }
        if (c.obs_type == B747_OBS_PID_AERO || c.obs_type == B747_OBS_PID_SPEED_AERO) {
          obs[n] = o.CXa; mx[n++] = 0.5f; obs[n] = o.CYa; mx[n++] = 2.f; obs[n] = o.mz; mx[n++] = 0.6f;
          obs[n] = o.dCm; mx[n++] = 0.05f; obs[n] = o.K_alpha; mx[n++] = 1.f;
        }
        if (c.norm_obs)
          for (int k = 0; k < n; k++) obs[k] /= mx[k];
      }
    }
    if (TRACE && st.trace.trk) {  // Controller.quality of the running episode
      const double q = exp(-60 * 0.1 * s4.itse / (c.tk * ((double)vr * (double)vr)));
      st.trace.trk[(size_t)TRK_quality * np + i] = q;
      st.trace.trk[((size_t)NTRK + TRK_quality) * np + i] = q;
    }
    // reward (env/ctrl_env.py:109-192)
    float rew = 0.f;
    {
      const float vf = vr != 0.f ? vr : (float)c.vartheta_max;
      const float itse = (float)s4.itse;
      switch (c.rew_type) {
        case B747_REW_CLASSIC: {
          const float k1 = (float)c.rew[0], k2 = (float)c.rew[1], k3 = (float)c.rew[2], k0 = (float)c.rew[3],
                      kI = (float)c.rew[4], kf = (float)c.rew[5], kt = (float)c.rew[6], ko = (float)c.rew[7];
          const float inv_vf = 1.0f / vf;
          const float rel = fabsf(dv * inv_vf);
          float r1 = 0.5f * exp_fast(-k0 * (k1 * fabsf(dv) + k2 * fabsf(dv_dt_f) + k3 * fabsf(dv_dt_dt)) * fabsf(inv_vf));
          float r2 = (vr * dv < 0.f) ? 0.2f * exp_fast(-ko * rel) : 0.2f;
          float r3 = (rel > 0.05f) ? 0.2f * exp_fast(-kt * time) : 0.2f;
          float r4 = 0.1f * exp_fast(-kI * itse * inv_vf * inv_vf);
          float rf = 0.f;
          if (c.ctrl_mode == B747_MODE_DIRECT)
            rf = -kf * (0.5f * rel) * fabsf(r.deltaz - o.U_com_PID) * (float)(1.0 / (34 * kPi / 180));
          rew = r1 + r2 + r3 + r4 + rf;
          break;
        }
        case B747_REW_PID_LIKE:
          rew = expf(-(float)c.rew[0] * fabsf(o.U_com - o.U_com_PID) * (float)(1.0 / (34 * kPi / 180)));
          break;
        case B747_REW_QUALITY:
        case B747_REW_MINIMAL:
          rew = expf(-6.0f * itse / ((float)c.tk * (vr * vr)));
          break;
        case B747_REW_TF_REFERENCE: {
          float overshoot = fabsf(dv / vf) * 100.f;
          if (overshoot > 5.f) r.tf_tp = time;
          rew = expf(-(float)c.rew[2] * fabsf(overshoot - (float)c.rew[0]) * fabsf((float)c.rew[1] - r.tf_tp));
          break;
        }
      }
    }
    r.ep_return += (double)rew;
    done = (int64_t)r.tick >= c.done_tick;
    if (c.use_limiter && (fabsf(nan_to_num_f(o.th)) > (float)(5 * kPi / 180 + c.vartheta_max) || r.deltaz > (float)c.action_max))
      done = true;
    if (TRACE && st.sig) {  // signal export: full tier only (launch_env_step32)
      float* sg = st.sig;
#define SG(name, v) sg[(size_t)SIG_##name * np + i] = (v)
      const float qn = nanf("");
      SG(state_x, s4.x); SG(state_y, s4.h); SG(state_Vx, s4.Vx); SG(state_Vy, s4.Vy); SG(state_vartheta, o.th);
      SG(state_wz, s4.wz); SG(sim_time, time); SG(vartheta_zh, o.vartheta_zh); SG(U_com_PID, o.U_com_PID);
      SG(CXa, o.CXa); SG(CYa, o.CYa); SG(mz, o.mz); SG(K_alpha, o.K_alpha); SG(dCm_ddeltaz, o.dCm); SG(U_com, o.U_com);
      SG(deltaz_RP, o.deltaz_RP); SG(dvartheta, dv); SG(dvartheta_int, (float)s4.dvi); SG(dvartheta_dt, dv_dt_f);
      SG(dvartheta_dt_dt, dv_dt_dt); SG(TAE, fabsf(dv) * time); SG(ITAE, qn); SG(TSE, dv * dv * time);
      SG(ITSE, (float)s4.itse); SG(AE, fabsf(dv)); SG(IAE, qn); SG(SE, dv * dv); SG(ISE, qn); SG(alpha, o.alpha);
      SG(V, o.V); SG(Mach, o.Mach);
      SG(CXa_tab, qn); SG(CYa_tab, qn); SG(mz_tab, qn); SG(dCm_tab, qn);  // float64 handles only (legacy boundary)
#undef SG
    }
    // Outputs.  Packed form (b747_step*_packed): one record of 4 * ceil((obs_dim + 1) / 4) floats per env --
    // (obs before any auto-reset, reward, zero padding), a single 128-bit store for the 3-scalar layouts -- and the done
    // flags as one ballot word per warp (below); the observation after an auto-reset is all zeros (ControllerEnv.reset), so
    // the caller derives it from the done bit.
    const bool packed = out4 != nullptr;
    if (packed) {
      if (!GEN) {
        out4[i] = make_float4(obs[0], obs[1], obs[2], rew);
      } else {
        const int rec4 = (od + 4) >> 2;  // float4s per record
        float rec[12];
#pragma unroll
        for (int k = 0; k < 12; k++) rec[k] = k < od ? obs[k < 10 ? k : 9] : (k == od ? rew : 0.f);
        float4* q = out4 + (size_t)i * rec4;
        for (int k = 0; k < rec4; k++) q[k] = make_float4(rec[4 * k], rec[4 * k + 1], rec[4 * k + 2], rec[4 * k + 3]);
      }
    } else {
      rew_out[i] = rew;
      done_out[i] = done ? 1 : 0;
      if (term_obs)
        for (int k = 0; k < od; k++) term_obs[(size_t)i * od + k] = obs[k];
    }
    bool full_store = false;
    if (done) {
      ep_ret = r.ep_return; ep_len = (double)(r.tick / c.substeps);
      st.last_ret[i] = ep_ret; st.last_len[i] = r.tick / c.substeps;
      if (TRACE && st.trace.trk) trace_snapshot(st.trace, np, i, st.trace.trk[(size_t)TRK_quality * np + i]);
      if (c.auto_reset) {
        if (TRACE) trace_clear(st.trace, np, i);
        Episode ep;
        if (c.reset_ref_mode == B747_RESET_NONE) episode_from_state_mx(st, np, i, r, ep);
        else { draw_episode(c, (uint64_t)(c.env_id_offset + i), r.ep_idx, ep); r.ep_idx++; }
        env_reset_mx<GEN>(c, ep, r, st, np, i);
        full_store = true;
        for (int k = 0; k < od; k++) obs[k] = 0.f;
        if (TRACE && st.sig) for (int k = 0; k < NSIG; k++) st.sig[(size_t)k * np + i] = 0.f;
      }
    }
    if (!packed) {
      if (od == 3) {  // canonical layout: three contiguous floats per env
        float* q = obs_out + (size_t)i * 3;
        q[0] = obs[0]; q[1] = obs[1]; q[2] = obs[2];
      } else {
        for (int k = 0; k < od; k++) obs_out[(size_t)i * od + k] = obs[k];
      }
    }
    store_mx<GEN, CS>(st, np, i, r, full_store);
  }
  if (done_bits) {  // done flags of the tile as one word (env_lo is a multiple of 32: launch_env_step32)
    const unsigned b = __ballot_sync(0xffffffffu, done);
    if (lane == 0) done_bits[(c.env_lo >> 5) + wt] = b;
  }
  warp_episode_stats(s_stats, done, ep_ret, ep_len);
  wt = wn;
  }
  __syncthreads();
  if (threadIdx.x < 4 && s_stats[threadIdx.x] != 0.0) atomicAdd(st.stats + threadIdx.x, s_stats[threadIdx.x]);
}

template <bool GEN>
__global__ void __launch_bounds__(128) k_reset32(DevCfg c, StateF32 st, const uint8_t* __restrict__ mask,
                                                 const b747_episode* __restrict__ eps, float* __restrict__ obs_out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= c.n_envs) return;
  if (mask && !mask[i]) return;
  const size_t np = (size_t)c.n_pad;
  RegsMx r;
  load_mx<GEN>(st.D, st.F, np, i, r);
  Episode ep;
  if (eps) {
    episode_from_abi(eps[i], ep);
  } else if (c.reset_ref_mode == B747_RESET_NONE) {
    episode_from_state_mx(st, np, i, r, ep);
  } else {
    draw_episode(c, (uint64_t)(c.env_id_offset + i), r.ep_idx, ep);
    r.ep_idx++;
  }
  env_reset_mx<GEN>(c, ep, r, st, np, i);
  trace_clear(st.trace, np, i);
  if (obs_out)
    for (int k = 0; k < c.obs_dim; k++) obs_out[(size_t)i * c.obs_dim + k] = 0.f;
  if (st.sig) for (int k = 0; k < NSIG; k++) st.sig[(size_t)k * np + i] = 0.f;
  store_mx<GEN>(st, np, i, r, true);
}

__global__ void __launch_bounds__(128) k_defaults32(DevCfg c, StateF32 st) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= c.n_pad) return;
  const size_t np = (size_t)c.n_pad;
  RegsMx r;
  const double s0[6] = B747_DEF_STATE0;
  r.flags = (c.ctrl_type == B747_CTRL_SEMI_MANUAL || c.ctrl_type == B747_CTRL_FULL_AUTO) ? FL_USE_CTRL : 0;
  r.ep_idx = 0;
  r.tc.ix = kIxEmpty;
  for (int k = 0; k < 5; k++) r.sumA[k] = 1.0f;
  model_init32(s0, r);
  r.vref = 0.0; r.href = B747_DEF_H_ZH; r.vartheta = 0.0;
  for (int k = 0; k < 3; k++) { r.oscA[k] = 0.0; r.oscf[k] = 0.0; }
  r.ep_return = 0.0; r.tf_tp = 0.f;
  store_state0_mx(st, np, i, s0);
  if (st.sig) for (int k = 0; k < NSIG; k++) st.sig[(size_t)k * np + i] = 0.f;
  st.last_ret[i] = 0.0; st.last_len[i] = 0;
  store_mx<true>(st, np, i, r, true);
}

// ---- host side --------------------------------------------------------------------------------
bool f32_is_lean(const DevCfg& c) {
  return c.ctrl_type == B747_CTRL_MANUAL && c.reset_ref_mode == B747_RESET_CONST && c.disturbance_mode == B747_DIST_NONE &&
         c.rew_type != B747_REW_TF_REFERENCE && c.obs_type == B747_OBS_PID_LIKE;
}

// can the altitude loop be closed (FL_USE_CTRL set by a reset)?  Explicit episodes (b747_reset_to) and flag edits set
// DevCfg::force_full instead.
bool f32_needs_cs(const DevCfg& c) {
  return c.ctrl_type != B747_CTRL_MANUAL || c.reset_ref_mode == B747_RESET_HYBRID || c.reset_ref_mode == B747_RESET_NONE;
}

static MP32 make_mp32(const ModelParams& m) {
  MP32 p;
  for (int k = 0; k < 4; k++) p.PID_SS[k] = (float)m.PID_SS[k];
  p.P_m = (float)(m.P / m.m0); p.g = (float)m.g;
  p.kS_m = (float)(Pc(134) * m.S / m.m0);
  p.half_Sc_over_Iz = (float)(Pc(135) * m.S * m.c_ / m.Iz);
  p.sw = (m.use_RL >= Pc(148) ? SW_RL : 0) | (m.use_PID_SS >= Pc(9) ? SW_SS : 0) | (m.use_RP >= Pc(149) ? SW_RP : 0) |
         (m.use_PID_SS != 0.0 ? SW_SS_ON : 0);
  return p;
}

int f32_alloc(const DevCfg& c, StateF32& s, bool export_signals, cudaStream_t stream) {
  const size_t np = (size_t)c.n_pad;
  const ft::Fast F = ft::build();
  if (!F.ok) return -2;  // model_simple_P does not fit the compiled table layout (checked before anything is allocated)
  bool ok = cudaMalloc(&s.D, sizeof(double2) * np * ND_GROUPS) == cudaSuccess &&
            cudaMalloc(&s.F, sizeof(float4) * np * NF_GROUPS) == cudaSuccess &&
            (!export_signals || cudaMalloc(&s.sig, sizeof(float) * np * NSIG) == cudaSuccess) &&
            cudaMalloc(&s.stats, sizeof(double) * 4) == cudaSuccess &&
            cudaMalloc(&s.last_ret, sizeof(double) * np) == cudaSuccess &&
            cudaMalloc(&s.last_len, sizeof(int) * np) == cudaSuccess &&
            cudaMalloc(&s.tables, sizeof(float4) * ft::CELLS) == cudaSuccess &&
            cudaMalloc(&s.tile_ctr, sizeof(unsigned int) * 64) == cudaSuccess &&
            cudaMemcpy(s.tables, F.v.data(), sizeof(float4) * ft::CELLS, cudaMemcpyHostToDevice) == cudaSuccess;
  if (!ok) {  // release whatever was allocated: a retry with fewer envs must find the HBM free (the CUDA error stays
    f32_free(s);  // readable for the caller's message)
    return -1;
  }
  cudaMemsetAsync(s.D, 0, sizeof(double2) * np * ND_GROUPS, stream);
  cudaMemsetAsync(s.F, 0, sizeof(float4) * np * NF_GROUPS, stream);
  cudaMemsetAsync(s.stats, 0, sizeof(double) * 4, stream);
  return 0;
}

void f32_state_blocks(size_t np, bool export_signals, const StateF32* s, StateTable& t) {
  t.add(s ? s->D : nullptr, sizeof(double2), sizeof(double2) * np, ND_GROUPS);
  t.add(s ? s->F : nullptr, sizeof(float4), sizeof(float4) * np, NF_GROUPS);
  t.add(s ? s->last_ret : nullptr, sizeof(double), 0, 1);
  t.add(s ? s->last_len : nullptr, sizeof(int), 0, 1);
  if (export_signals) t.add(s ? s->sig : nullptr, sizeof(float), sizeof(float) * np, NSIG);
}

void f32_free(StateF32& s) {
  cudaFree(s.D); cudaFree(s.F); cudaFree(s.sig); cudaFree(s.stats); cudaFree(s.last_ret); cudaFree(s.last_len); cudaFree(s.tables); cudaFree(s.tile_ctr);
  s = StateF32{};
}

static inline int grid_for(int n, int block) { return (n + block - 1) / block; }

constexpr int kTileCtrSlots = 64;
// grid of the step kernel: enough blocks to fill every SM at the occupancy of the instantiation that is launched,
// never more than the tiles need
template <int TIER, int SW = -1, bool STG = false, bool PFA = false>
static int step_grid(int n) {
  const int need = grid_for(n, kStepThreads);
  static int resident[64] = {0};  // per device: SMs x blocks per SM
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) return need;
  if (!resident[dev]) {
    int sms = 0, per_sm = 0;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_env_step32<TIER, SW, STG, PFA>, kStepThreads, 0);
    resident[dev] = sms > 0 && per_sm > 0 ? sms * per_sm : need;
  }
  return need < resident[dev] ? need : resident[dev];
}

// resolve the persistent grids once, outside any stream capture (b747_create)
void f32_warm_launch() {
  const int big = 1 << 30;
  step_grid<0, SW_RP, false, true>(big); step_grid<0, SW_RP, true>(big); step_grid<0, SW_RP>(big); step_grid<0>(big);
  step_grid<1, SW_RP>(big); step_grid<1>(big); step_grid<2>(big); step_grid<3>(big);
}

void launch_env_step32(const DevCfg& c, const StateF32& st, const float* actions, float* obs, float* rew, uint8_t* done,
                       float* term_obs, cudaStream_t s, float4* out4, uint32_t* done_bits, bool prefetch_actions) {
  const MP32 mp = make_mp32(c.mp);
  const int n = c.env_hi - c.env_lo;
  if (n <= 0) return;
  const bool plain = !st.trace.trk && !st.trace.rec && !st.sig && !c.force_full;
  const bool lean = plain && f32_is_lean(c);
  const bool lean_rp = lean && mp.sw == SW_RP;  // the canonical switch setting (use_RP only) as a compile-time constant
  const bool staged = lean_rp && !prefetch_actions && c.substeps <= kStagedMaxK;  // HBM-bound regime: TMA-staged state
  // tile counter of this launch: one of kTileCtrSlots words, zeroed on the launch stream (launches of one handle may
  // overlap on different streams -- b747_step_host's chunk pipeline -- so consecutive launches take different slots)
  unsigned int* ctr = nullptr;
  if (st.tile_ctr && !staged) {
    static std::atomic<unsigned> seq{0};
    ctr = st.tile_ctr + (seq.fetch_add(1) % kTileCtrSlots);
    cudaMemsetAsync(ctr, 0, sizeof(unsigned int), s);
  }
#define B747_LAUNCH(TIER, ...) \
  k_env_step32<TIER, ##__VA_ARGS__><<<step_grid<TIER, ##__VA_ARGS__>(n), kStepThreads, 0, s>>>( \
      c, mp, st, actions, obs, rew, done, term_obs, out4, done_bits, ctr)
  if (lean_rp && prefetch_actions)  // host-mapped action buffer (b747_step_host_packed)
    B747_LAUNCH(0, SW_RP, false, true);
  else if (staged)
    B747_LAUNCH(0, SW_RP, true);
  else if (lean_rp)
    B747_LAUNCH(0, SW_RP);
  else if (lean)
    B747_LAUNCH(0);
  else if (plain && !f32_needs_cs(c) && mp.sw == SW_RP)
    B747_LAUNCH(1, SW_RP);
  else if (plain && !f32_needs_cs(c))
    B747_LAUNCH(1);
  else if (plain)
    B747_LAUNCH(2);
  else
    B747_LAUNCH(3);
#undef B747_LAUNCH
}
void launch_reset32(const DevCfg& c, const StateF32& st, const uint8_t* mask, const b747_episode* eps, float* obs,
                    cudaStream_t s) {
  // resets always go through the general layout so that every group is initialised
  k_reset32<true><<<grid_for(c.n_envs, 128), 128, 0, s>>>(c, st, mask, eps, obs);
}
void launch_defaults32(const DevCfg& c, const StateF32& st, cudaStream_t s) {
  k_defaults32<<<grid_for(c.n_pad, 128), 128, 0, s>>>(c, st);
}

// Per-env fields of an f32 handle: (group, lane) lookup by name; returns non-zero if unavailable.
namespace {
struct MxField { const char* name; int is_f; int group; int lane; };
const MxField kMxFields[] = {
    {"h", 0, DG_h_th, 0}, {"th", 0, DG_h_th, 1}, {"Vx", 0, DG_V, 0}, {"Vy", 0, DG_V, 1}, {"wz", 0, DG_wz_ssi, 0},
    {"ss_int", 0, DG_wz_ssi, 1}, {"ss_flt", 0, DG_ssf_dvi, 0}, {"dv_int", 0, DG_ssf_dvi, 1}, {"itse", 0, DG_itse_d1, 0},
    {"d1_u", 0, DG_itse_d1, 1}, {"vref", 0, DG_vref_ret, 0}, {"ep_return", 0, DG_vref_ret, 1}, {"cs_int", 0, DG_cs, 0},
    {"cs_flt", 0, DG_cs, 1}, {"x", 0, DG_x_href, 0}, {"href", 0, DG_x_href, 1},
    {"df_x", 1, FG_act, 0}, {"df_y", 1, FG_act, 1}, {"rl_prev", 1, FG_act, 2}, {"deltaz", 1, FG_act, 3},
    {"uh0", 1, FG_uh, 0}, {"uh1", 1, FG_uh, 1}, {"uh2", 1, FG_uh, 2}, {"uh3", 1, FG_uh, 3},
    {"sig_upid", 1, FG_misc, 0}, {"d2_u", 1, FG_misc, 1}, {"tf_tp", 1, FG_misc2, 1}, {"sig_vzh", 1, FG_misc2, 2},
};
}  // namespace

int f32_field_io(const DevCfg& c, StateF32& s, FieldKind kind, int row, const char* name, double* out, const double* in,
                 cudaStream_t stream) {
  const size_t n = (size_t)c.n_envs, np = (size_t)c.n_pad;
  if (kind == FK_SIG) {
    if (!s.sig || in) return -1;
    std::vector<float> tmp(n);
    if (cudaMemcpy(tmp.data(), s.sig + (size_t)row * np, sizeof(float) * n, cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
    for (size_t i = 0; i < n; i++) out[i] = tmp[i];
    return 0;
  }
  if (kind == FK_LASTRET) {
    if (in) return -1;
    return cudaMemcpy(out, s.last_ret, sizeof(double) * n, cudaMemcpyDeviceToHost) != cudaSuccess;
  }
  if (kind == FK_LASTLEN) {
    if (in) return -1;
    std::vector<int> tmp(n);
    if (cudaMemcpy(tmp.data(), s.last_len, sizeof(int) * n, cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
    for (size_t i = 0; i < n; i++) out[i] = tmp[i];
    return 0;
  }
  if (kind == FK_TICK || kind == FK_FLAGS || kind == FK_EPIDX) {
    std::vector<float4> tmp(n);
    float4* dev = s.F + (size_t)FG_misc * np;
    if (cudaMemcpy(tmp.data(), dev, sizeof(float4) * n, cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
    for (size_t i = 0; i < n; i++) {
      uint32_t tz, fw, ix;
      memcpy(&tz, &tmp[i].z, 4); memcpy(&fw, &tmp[i].w, 4);
      int tick;
      unpack_tick(tz, tick, ix);
      if (out) out[i] = kind == FK_TICK ? (double)tick : (kind == FK_FLAGS ? (double)(fw & 0xffu) : (double)(fw >> 8));
      else {
        if (kind == FK_TICK) tz = (uint32_t)(int)in[i] & 0x7fffffffu;  // plain tick: the interval hints are dropped
        else if (kind == FK_FLAGS) fw = (fw & ~0xffu) | ((uint32_t)in[i] & 0xffu);
        else fw = (fw & 0xffu) | ((uint32_t)in[i] << 8);
        memcpy(&tmp[i].z, &tz, 4); memcpy(&tmp[i].w, &fw, 4);
      }
    }
    if (in && cudaMemcpy(dev, tmp.data(), sizeof(float4) * n, cudaMemcpyHostToDevice) != cudaSuccess) return -1;
    return 0;
  }
  for (const MxField& f : kMxFields) {
    if (strcmp(f.name, name)) continue;
    if (f.is_f) {
      std::vector<float4> tmp(n);
      float4* dev = s.F + (size_t)f.group * np;
      if (cudaMemcpy(tmp.data(), dev, sizeof(float4) * n, cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
      for (size_t i = 0; i < n; i++) {
        float* p = &tmp[i].x + f.lane;
        if (out) out[i] = *p; else *p = (float)in[i];
      }
      if (in && cudaMemcpy(dev, tmp.data(), sizeof(float4) * n, cudaMemcpyHostToDevice) != cudaSuccess) return -1;
    } else {
      std::vector<double2> tmp(n);
      double2* dev = s.D + (size_t)f.group * np;
      if (cudaMemcpy(tmp.data(), dev, sizeof(double2) * n, cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
      for (size_t i = 0; i < n; i++) {
        double* p = &tmp[i].x + f.lane;
        if (out) out[i] = *p; else *p = in[i];
      }
      if (in && cudaMemcpy(dev, tmp.data(), sizeof(double2) * n, cudaMemcpyHostToDevice) != cudaSuccess) return -1;
    }
    return 0;
  }
  return -1;
}

}  // namespace b747
