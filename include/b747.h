/*
 * b747.h -- C ABI of libb747_b200.so: the B200-native replacement for the model library
 * that the reference loads with ctypes (core/model.py:104-164) and for the per-step
 * Python work above it (core/controller.py:231-264, env/ctrl_env.py:237-270).
 *
 * Two surfaces:
 *  (1) the reference's own scalar boundary, bit-for-bit the same names and meaning
 *      (declared in b747_scalar.h): model_simple_initialize/step/terminate + the named
 *      `double` globals -- an unchanged Model-style wrapper binds to it;
 *  (2) the batched boundary below: N independent environments resident in HBM, one
 *      launch per env step (K fused RK4 substeps, observation, reward, done, auto-reset).
 *
 * Plain C: pointers and sizes only, no torch types.  All compute runs as sm_100a CUDA
 * kernels; there is no CPU fallback -- every entry point returns B747_ERR_CUDA (and
 * b747_last_error() says why) when no device is usable.
 *
 * Threading: calls on one handle are ordered on the handle's stream (or the stream passed
 * to the *_async entry points); different handles are independent.  Ownership: the handle
 * owns the environment state; I/O buffers belong to the caller.
 */
#ifndef B747_H
#define B747_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B747_ABI_VERSION 2

/* Return codes */
enum { B747_OK = 0, B747_ERR_ARG = -1, B747_ERR_CUDA = -2, B747_ERR_ALLOC = -3, B747_ERR_STATE = -4 };

/* Arithmetic mode of a handle.
 * B747_F64: every operation in float64 in the DLL's evaluation order (parity mode; the
 *           reference's real_T is double, core/rtwtypes.py:27).  I/O buffers are double.
 * B747_F32: throughput mode.  Aerodynamics / atmosphere / trigonometry / table look-ups in
 *           float32; integrator state, pitch-error chain and finite-difference blocks are
 *           accumulated in float64 (DESIGN.md "fp32 mode").  I/O buffers are float. */
enum { B747_F64 = 0, B747_F32 = 1 };

/* Enum values equal the reference's Enum values. */
enum { B747_CTRL_FULL_AUTO = 0, B747_CTRL_AUTO = 1, B747_CTRL_SEMI_MANUAL = 2, B747_CTRL_MANUAL = 3 }; /* core/controller.py:14-19 */
enum { B747_MODE_DIRECT = 0, B747_MODE_ADD_PROC = 1, B747_MODE_ANG_VEL = 2, B747_MODE_ADD_DIRECT = 3 }; /* core/controller.py:21-26 */
/* ctrl_mode=None of the reference (allowed with CtrlType.AUTO / FULL_AUTO, core/controller.py:103; what ControllerAgent.test
 * sets on its PID env, neural/agent.py:301): the action law falls through to deltaz = action like DIRECT_CONTROL
 * (core/controller.py:241), but the CLASSIC reward's shaping term rf is 0 because the mode is not DIRECT_CONTROL
 * (env/ctrl_env.py:141). */
enum { B747_MODE_NONE = -1 };
enum { B747_RESET_NONE = -1, B747_RESET_CONST = 0, B747_RESET_OSCILLATING = 1, B747_RESET_HYBRID = 2 }; /* core/controller.py:28-32 */
enum { B747_DIST_NONE = -1, B747_DIST_AERO = 0 };                                                    /* core/controller.py:34-36 */
enum { B747_OBS_PID_LIKE = 0, B747_OBS_SPEED_MODE = 1, B747_OBS_PID_AERO = 2, B747_OBS_PID_SPEED_AERO = 3, B747_OBS_MODEL_STATE = 4 }; /* env/ctrl_env.py:16-22 */
enum { B747_REW_CLASSIC = 0, B747_REW_PID_LIKE = 1, B747_REW_QUALITY = 2, B747_REW_MINIMAL = 3, B747_REW_TF_REFERENCE = 4 };          /* env/ctrl_env.py:24-30 */

/* Environment configuration == the ControllerEnv(...)/Controller(...) constructor arguments
 * (env/ctrl_env.py:65-74, core/controller.py:72-89). */
typedef struct b747_cfg {
  int32_t abi_version;     /* B747_ABI_VERSION */
  int32_t device;          /* CUDA device ordinal */
  int32_t dtype;           /* B747_F64 / B747_F32 */
  int32_t n_envs;
  int32_t obs_type, rew_type, ctrl_type, ctrl_mode, reset_ref_mode, disturbance_mode;
  int32_t norm_obs, norm_act, use_limiter;
  int32_t substeps;        /* K = round(sample_time/dt) model steps per env step (core/controller.py:261) */
  int32_t auto_reset;      /* 1: done envs are reset in-kernel and return the reset observation (SB3 VecEnv contract) */
  int32_t env_layer;       /* 1: full env step; 0: raw model stepping only (Model.step), obs/rew/done untouched */
  int64_t done_tick;       /* smallest tick with fl(tick*0.01) >= tk (Controller.is_done, core/controller.py:316-319) */
  int64_t env_id_offset;   /* global id of env 0 of this handle (sharding across GPUs keeps streams identical) */
  uint64_t seed;           /* Philox key */
  double tk, action_max, vartheta_max, sample_time;
  double rew[8];           /* reward constants, layout in DESIGN.md (CLASSIC: k1,k2,k3,k0,kITSE,kf,kt,ko) */
  double fixed_aero_err[5];
  int32_t has_fixed_aero_err;
  int32_t export_signals;  /* 1: every step also writes the DLL's exported signals (stage-4 values) per env */
  int32_t track_transfer;  /* 1: calc_stepinfo (tools/general.py:46-61) evaluated online after every MODEL step, for the
                              pitch angle vs vartheta_ref (Controller.stepinfo_SS) and the altitude vs hzh (stepinfo_CS) */
  int32_t record_capacity; /* > 0: Controller(use_storage=True) -- record what Controller._post_step records
                              (core/controller.py:209-228) for the first record_capacity model steps of the running episode */
} b747_cfg;

/* Per-episode initial condition and reference (what Controller.reset decides, core/controller.py:134-201). */
typedef struct b747_episode {
  double state0[6];        /* x, y, Vx, Vy, vartheta, wz  (core/model.py:226) */
  int32_t use_ctrl;        /* altitude loop (СУ PID) closed; only honoured with B747_RESET_HYBRID (else ctrl_type decides) */
  int32_t oscillating;
  double vref_const;
  double osc_A[3], osc_f[3];
  double h_ref;
  double aero_err[5];
} b747_episode;

typedef struct b747_handle b747_handle;

const char *b747_last_error(void);
/* which: 0 -> ABI version, 1 -> sizeof(b747_cfg), 2 -> sizeof(b747_episode) (binding self-check) */
int b747_abi_info(int which);
int b747_obs_dim(int obs_type);
int64_t b747_done_tick(double tk);

int b747_create(const b747_cfg *cfg, b747_handle **out);
int b747_destroy(b747_handle *h);
/* CUDA stream (cudaStream_t) the handle launches on; set_stream adopts a caller stream. */
void *b747_stream(b747_handle *h);
int b747_set_stream(b747_handle *h, void *cuda_stream);

/* Controller.reset + ControllerEnv.reset for every env (mask==NULL) or the envs with mask[i]!=0.
 * Random draws: Philox4x32-10 keyed by cfg.seed, counter (global env id, episode index, draw).
 * obs (device, [n_envs][obs_dim], handle dtype) may be NULL. */
int b747_reset(b747_handle *h, const uint8_t *mask_dev, void *obs_dev);
/* Deterministic reset: episodes is a HOST array of n_envs descriptors (Controller.reset(state0) with
 * an explicit reference, as neural/callbacks.py:61-100 does). */
int b747_reset_to(b747_handle *h, const b747_episode *episodes_host, void *obs_dev);
/* Same, for the envs with mask_dev[i] != 0 only (mask on the device like b747_reset's; NULL = all): what
 * `vec_env.env_method("reset", state0, indices=[i])` of the SB3 contract needs.  obs rows of other envs are untouched. */
int b747_reset_to_masked(b747_handle *h, const b747_episode *episodes_host, const uint8_t *mask_dev, void *obs_dev);

/* ControllerEnv.step for all envs: device buffers of the handle dtype.
 *   actions [n_envs]; obs [n_envs][obs_dim]; rew [n_envs]; done [n_envs] (uint8);
 *   terminal_obs [n_envs][obs_dim] or NULL (observation before auto-reset, SB3's
 *   infos[i]["terminal_observation"]).  Asynchronous on the handle's stream. */
int b747_step(b747_handle *h, const void *actions_dev, void *obs_dev, void *rew_dev, uint8_t *done_dev,
              void *terminal_obs_dev);
/* Same call with HOST buffers (pinned or pageable): H2D of actions, the step, D2H of obs/rew/done,
 * synchronised on return.  This is the call a ctypes/gym user makes.  Batches of >= 128 Ki envs are
 * pipelined over env chunks (copy-in, step and copy-out of neighbouring chunks overlap; pinned buffers
 * are needed for the overlap, pageable ones still work); results are identical to the one-launch form. */
int b747_step_host(b747_handle *h, const void *actions, void *obs, void *rew, uint8_t *done, void *terminal_obs);
/* Number of chunks of the host-step pipeline of b747_step_host and of b747_step_host_packed's staged copies (mode 0,
 * pinned buffers): 0 = automatic (4 from 128 Ki envs, else 1), 1 = no pipeline. */
int b747_set_host_chunks(b747_handle *h, int n_chunks);

/* Packed outputs (f32 handles): per env ONE record of R = b747_packed_record_floats(obs_type) = 4 * ceil((obs_dim + 1) / 4)
 * floats (4 for PID_LIKE, 8 for SPEED_MODE and MODEL_STATE, 12 for PID_AERO and PID_SPEED_AERO):
 *   out[i * R + k]       = obs[k], k < obs_dim  -- the observation BEFORE any auto-reset, i.e. SB3's
 *                                                  infos[i]["terminal_observation"] where the env finished;
 *   out[i * R + obs_dim] = reward; the rest of the record is zero padding;
 *   bit (i & 31) of done_bits[i >> 5] = done flag  -- done_bits holds (n_envs + 31) / 32 words.
 * The observation after an auto-reset is all zeros (every exported signal is zero after Model.initialize,
 * env/ctrl_env.py:273-278), so a caller derives the returned observation as done ? 0 : record.obs.
 * b747_step_packed: device buffers, asynchronous on the handle's stream.
 * b747_step_host_packed: HOST buffers, synchronised on return.  With page-locked (cudaHostAlloc / cudaHostRegister)
 * buffers the kernel reads the actions from and stores the records into the caller's memory directly (posted PCIe
 * writes of whole 128-bit words that overlap the stepping of the other envs); pageable buffers are staged. */
int b747_packed_record_floats(int obs_type);
int b747_step_packed(b747_handle *h, const float *actions_dev, float *out4_dev, uint32_t *done_bits_dev);
int b747_step_host_packed(b747_handle *h, const float *actions, float *out4, uint32_t *done_bits);
/* Host path of b747_step_host_packed with page-locked buffers: 0 staged copies (the chunk pipeline of b747_step_host;
 * b747_set_host_chunks applies), 1 actions copied / records stored zero-copy, 2 actions and records zero-copy,
 * -1 automatic (default): the first ten calls alternate between 2 and 0 and are timed, the faster path is kept
 * (zero-copy when the GPU has the host link to itself, staged copies when many GPUs share it).  Results are identical
 * in every mode. */
int b747_set_host_mode(b747_handle *h, int mode);
/* env.seed(s) of the gym / SB3 API (neural/agent.py:80): re-keys the Philox stream used by every later random reset. */
int b747_set_seed(b747_handle *h, uint64_t seed);

/* Raw model stepping (Model.step xN, core/model.py:247-250): no action law, no reward (f64 handles).
 * b747_model_initialize == Model.initialize (core/model.py:238-244): re-reads state0_*, zeroes time,
 * signals and hidden state, sets deltaz = vartheta = 0. */
int b747_model_step(b747_handle *h, int32_t n_steps);
int b747_model_initialize(b747_handle *h);

/* Whole-batch model tunables (the DLL globals the Python layer never varies per env):
 * "PID_SS"[4], "PID_CS"[4], "P", "Iz", "S", "c_", "g", "m0", "use_RP", "use_RL", "use_PID_SS". */
int b747_set_param(b747_handle *h, const char *name, const double *v, int n);
int b747_get_param(b747_handle *h, const char *name, double *v, int n);

/* Named per-env fields (state, parameters, stage-4 signals) as float64 host arrays [n_envs].
 * Names: the DLL's exported globals ("state" is 6 names state_x..state_wz) plus internal
 * state listed by b747_field_name(). */
int b747_n_fields(void);
const char *b747_field_name(int field);
int b747_field_index(const char *name);
int b747_get_field(b747_handle *h, int field, double *out_host);
int b747_set_field(b747_handle *h, int field, const double *in_host);
/* f32 handles integrate only what their configuration's kernel tier needs: "x", "cs_int", "cs_flt" (canonical and
 * general tiers without the altitude loop) and "sig_vzh" (canonical tier) keep their reset values there.  Writing
 * "flags" (closing the altitude loop of single envs by hand) moves the handle to the full tier for good; the extra
 * states then start from those reset values, so reset the affected envs (b747_reset / b747_reset_to_masked) after such
 * an edit.  float64 handles integrate everything always. */

/* Episode statistics accumulated in-kernel since the last call (then zeroed):
 * out[0]=episodes finished, out[1]=sum of episode returns, out[2]=sum of episode lengths (env steps),
 * out[3]=sum of squared returns.  This is the only quantity that crosses GPUs (summed by the caller). */
int b747_episode_stats(b747_handle *h, double out_host[4]);
/* Per-env return/length of the most recently finished episode (VecMonitor's infos[i]["episode"]). */
int b747_last_episode(b747_handle *h, double *ret_host, int32_t *len_host);
/* The same for n_idx chosen envs (idx_host[k] in [0, n_envs)): ret_host[k], len_host[k] of env idx_host[k]. */
int b747_last_episode_of(b747_handle *h, const int32_t *idx_host, int32_t n_idx, double *ret_host, int32_t *len_host);

/* Step-response metrics (handles created with track_transfer): out_host[n_envs][5] = overshoot [%], rise time [s],
 * settling time [s], static error, Controller.quality() -- calc_stepinfo's definitions (5 % band, times relative to
 * the first recorded sample); NaN where the reference returns None.  which: 0 = pitch (stepinfo_SS), 1 = altitude
 * (stepinfo_CS).  finished: 0 = the running episode so far, 1 = the most recently finished episode. */
int b747_transfer_metrics(b747_handle *h, int which, int finished, double *out_host);
/* Recorder (handles created with record_capacity > 0): the running episode of one env, field-major:
 * out_host[b747_recorder_n_fields()][record_capacity]; *n_steps = recorded model steps. Field names are the
 * reference Storage's: t, U_com, U_PID, deltaz [deg], hzh, vartheta_ref [deg], U_RL, x, y, Vx, Vy, vartheta [deg], wz. */
int b747_recorder_n_fields(void);
const char *b747_recorder_field_name(int field);
int b747_recorder_read(b747_handle *h, int env, double *out_host, int32_t *n_steps);

/* Save, restore and fork per-env state.  A state blob is device memory: a 64-byte header (magic, format version,
 * dtype, n, flags, a 64-bit key of every b747_cfg field except n_envs, device, seed and env_id_offset) followed by n
 * entries of every per-env array the handle allocates, byte for byte -- f32 handles: the double2 and float4 state
 * groups (tick word with its look-up hints, episode index), last_ret, last_len; f64 handles: every slot including
 * state0, tick, flags, ep_idx, last_ret, last_len; both: the exported signals, the transfer tracker and its snapshot,
 * and the recorder rows when the handle has them.  Not in a blob: b747_set_param tunables, the seed, the
 * b747_episode_stats accumulators and the handle's scratch.  After a load, later random resets of env j are drawn
 * from the loading handle's seed, its env_id_offset + j and the episode index that came from the blob.
 * The blob must be 16-byte aligned (cudaMalloc and torch allocations are; a slice at another offset is not), index
 * arrays are int32 device arrays; a misaligned pointer is B747_ERR_ARG and nothing is launched.  An index entry outside
 * [0, n_envs) or outside [0, blob n) skips that k (nothing is written).  Duplicate env_idx entries in a load give an
 * unspecified result without a fault: that env's rows may come from different ones of its entries.
 *
 * b747_state_bytes: bytes of a blob holding n envs of a handle created with *cfg (no GPU needed); < 0 on a bad argument.
 * b747_save_state: blob entry k <- env env_idx_dev[k] for k < n (env_idx_dev NULL: env k, n <= n_envs).
 *   Asynchronous on the handle's stream.
 * b747_load_state: env env_idx_dev[k] <- blob entry blob_idx_dev[k] for k < n (NULL: identity; env_idx_dev NULL needs
 *   n <= n_envs).  Reads the header first and returns B747_ERR_STATE, writing nothing, on a wrong magic or version,
 *   another dtype or another configuration key.  A blob saved by a handle that ran the full f32 kernel tier moves this
 *   handle there too (like b747_reset_to with a closed altitude loop).  Synchronised on return. */
int64_t b747_state_bytes(const b747_cfg *cfg, int32_t n);
int b747_save_state(b747_handle *h, const int32_t *env_idx_dev, int32_t n, void *blob_dev);
int b747_load_state(b747_handle *h, const void *blob_dev, const int32_t *blob_idx_dev, const int32_t *env_idx_dev,
                    int32_t n);

/* Number of kernel launches issued through this handle so far (bench.py's gpu_launches). */
int64_t b747_launch_count(b747_handle *h);
int b747_synchronize(b747_handle *h);

/* Host-side self-test of the merged-axis look-up tables the f32 kernels read (b747_tables.h): re-samples
 * model_simple_P, then compares the re-gridded interpolation with look2_binlx / look1 semantics
 * (dll@0x1000) on n_points pseudo-random operands in float64.  extrapolate != 0 also draws operands far
 * outside the breakpoint ranges.  out_max_rel_err: CYa, CXa, dCm_ddeltaz, mz, K_alpha.  No GPU needed. */
int b747_selftest_tables(int n_points, int extrapolate, double out_max_rel_err[5]);

/* Philox4x32-10 as used for resets (exposed for known-answer tests). */
void b747_philox4x32(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);

#ifdef __cplusplus
}
#endif
#endif /* B747_H */
