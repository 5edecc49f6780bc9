// b747_capi.cu -- the C ABI of libb747_b200.so (include/b747.h).  Host-side glue only: device
// memory, streams, launches.  There is no CPU implementation behind any entry point.
#include <math.h>
#include <algorithm>
#include <stdio.h>
#include <string.h>

#include <chrono>
#include <mutex>
#include <string>
#include <vector>

#include "b747_kernels.h"
#include "b747_tables.h"

using namespace b747;

static thread_local std::string g_err;
static int fail(int code, const std::string& msg) { g_err = msg; return code; }
#define CU(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess)                                                                         \
      return fail(B747_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));              \
  } while (0)

struct b747_handle {
  b747_cfg cfg;
  DevCfg dc;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  StateF64 s64{};
  StateF32 s32{};
  // staging for b747_step_host
  void *d_act = nullptr, *d_obs = nullptr, *d_rew = nullptr, *d_term = nullptr;
  uint8_t* d_done = nullptr;
  float4* d_out4 = nullptr;      // packed outputs of b747_step_host_packed (pageable / copy modes), allocated on first use
  uint32_t* d_bits = nullptr;    // done flags, one bit per env
  int host_mode = -1;            // b747_step_host_packed: -1 automatic, 0 copy pipeline, 1 zero-copy outputs, 2 zero-copy both ways
  // automatic mode: the first calls alternate between zero-copy (2) and staged copies (0) and are timed; the faster one is
  // kept.  Alone on the host link zero-copy wins (2.7e9 against 2.2e9 env-steps/s at 1 Mi envs); with eight GPUs sharing
  // it the copy engines hold the link better (7.3e9 against 6.8e9, profiles/r2_hostlink_probe.md).  Results are identical.
  int auto_calls = 0, auto_choice = -1;
  double auto_sec[2] = {0.0, 0.0};
  // host-step pipeline (issue_pipeline): copy-in / second compute / copy-out streams and per-chunk events
  cudaStream_t s_in = nullptr, s_aux = nullptr, s_out = nullptr, s_cap = nullptr;
  std::vector<cudaEvent_t> ev_in, ev_k;
  cudaEvent_t ev_start = nullptr, ev_done = nullptr;
  int host_chunks = 0;  // 0 = choose from n_envs
  // the pipeline as an instantiated CUDA graph per set of (pinned) host buffers: one launch call per env step
  struct HostGraph { const void* act; void *obs, *rew, *done, *term; int chunks; uint64_t epoch; cudaGraphExec_t exec; };
  std::vector<HostGraph> graphs;
  uint64_t epoch = 0;     // bumped by everything that changes launch arguments (b747_set_param)
  bool use_graphs = true;
  b747_episode* d_eps = nullptr;
  double* d_metrics = nullptr;  // [n_pad][5] staging for b747_transfer_metrics
  TraceState trace;
  int64_t launches = 0;
  size_t elem() const { return cfg.dtype == B747_F64 ? 8 : 4; }
};

extern "C" const char* b747_last_error(void) { return g_err.c_str(); }
extern "C" int b747_obs_dim(int obs_type) { return obs_dim_of(obs_type); }

extern "C" int64_t b747_done_tick(double tk) {
  if (!(tk == tk) || isinf(tk)) return tk < 0 ? 0 : INT64_MAX;
  if (tk <= 0) return 0;
  int64_t n = (int64_t)floor(tk / 0.01) - 2;
  if (n < 0) n = 0;
  while (!((double)n * 0.01 >= tk)) n++;
  return n;
}

extern "C" int b747_abi_info(int which) {
  switch (which) {
    case 0: return B747_ABI_VERSION;
    case 1: return (int)sizeof(b747_cfg);
    case 2: return (int)sizeof(b747_episode);
  }
  return -1;
}

extern "C" void b747_philox4x32(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
  philox4x32(ctr, key, out);
}

// ---- field table -----------------------------------------------------------------------------
namespace {
struct FieldDesc { const char* name; FieldKind kind; int row; };
const std::vector<FieldDesc>& fields() {
  static std::vector<FieldDesc> f;
  static std::once_flag once;
  std::call_once(once, [] {
#define X(n) f.push_back({#n, FK_SLOT, S_##n});
    B747_F64_SLOTS(X)
#undef X
    static const char* s0n[6] = {"state0_x", "state0_y", "state0_Vx", "state0_Vy", "state0_vartheta", "state0_wz"};
    for (int k = 0; k < 6; k++) f.push_back({s0n[k], FK_STATE0, k});
#define X(n) f.push_back({"sig_" #n, FK_SIG, SIG_##n});
    B747_SIGNALS(X)
#undef X
    f.push_back({"tick", FK_TICK, 0});
    f.push_back({"flags", FK_FLAGS, 0});
    f.push_back({"ep_idx", FK_EPIDX, 0});
    f.push_back({"last_ret", FK_LASTRET, 0});
    f.push_back({"last_len", FK_LASTLEN, 0});
    f.push_back({"th", FK_MXONLY, 0});  // f32 handles carry the pitch angle itself instead of (q0, q3)
  });
  return f;
}
}  // namespace

extern "C" int b747_selftest_tables(int n_points, int extrapolate, double out[5]) {
  const b747::ft::Fast F = b747::ft::build();
  if (!F.ok || !out) return fail(B747_ERR_STATE, "model_simple_P does not fit the compiled table layout");
  const b747::ft::Orig O;
  const b747::ft::FastEval E{F};
  const double scale[5] = {1.0, 0.1, 0.02, 0.3, 1.0};
  for (int j = 0; j < 5; j++) out[j] = 0.0;
  uint32_t key[2] = {0x747u, 0u};
  for (int k = 0; k < n_points; k++) {
    uint32_t ctr[4] = {(uint32_t)k, 0u, 0u, 0u}, w[4];
    b747::philox4x32(ctr, key, w);
    const double u0 = w[0] / 4294967296.0, u1 = w[1] / 4294967296.0, u2 = w[2] / 4294967296.0;
    const double M = extrapolate ? -0.1 + 1.4 * u0 : 0.1 + 0.95 * u0;
    const double a = extrapolate ? -40.0 + 100.0 * u1 : -10.0 + 45.0 * u1;
    const double h = extrapolate ? -2000.0 + 18000.0 * u2 : 12500.0 * u2;
    double o[5];
    E.eval(M, a, h, o);
    const double cy = O.CYa(M, a);
    const double r[5] = {cy, O.CXa(M, cy), O.dCm(h, M), O.mz(M, a), O.Ka(a)};
    for (int j = 0; j < 5; j++) out[j] = fmax(out[j], fabs(o[j] - r[j]) / (fabs(r[j]) + scale[j]));
  }
  return B747_OK;
}

extern "C" int b747_n_fields(void) { return (int)fields().size(); }
extern "C" const char* b747_field_name(int i) { return (i >= 0 && i < (int)fields().size()) ? fields()[i].name : nullptr; }
extern "C" int b747_field_index(const char* name) {
  const auto& f = fields();
  for (size_t i = 0; i < f.size(); i++)
    if (!strcmp(f[i].name, name)) return (int)i;
  return -1;
}

// ---- lifecycle -------------------------------------------------------------------------------
static int fill_devcfg(const b747_cfg& c, DevCfg& d) {
  memset(&d, 0, sizeof d);
  d.n_envs = c.n_envs;
  d.n_pad = (c.n_envs + 127) / 128 * 128;
  d.env_lo = 0; d.env_hi = c.n_envs;
  d.obs_type = c.obs_type; d.obs_dim = obs_dim_of(c.obs_type); d.rew_type = c.rew_type;
  d.ctrl_type = c.ctrl_type; d.ctrl_mode = c.ctrl_mode; d.reset_ref_mode = c.reset_ref_mode;
  d.disturbance_mode = c.disturbance_mode; d.norm_obs = c.norm_obs; d.norm_act = c.norm_act;
  d.use_limiter = c.use_limiter; d.substeps = c.substeps; d.auto_reset = c.auto_reset; d.env_layer = c.env_layer;
  d.has_fixed_aero_err = c.has_fixed_aero_err; d.done_tick = c.done_tick; d.env_id_offset = c.env_id_offset;
  d.seed = c.seed; d.tk = c.tk; d.action_max = c.action_max; d.vartheta_max = c.vartheta_max;
  d.sample_time = c.sample_time;
  memcpy(d.rew, c.rew, sizeof d.rew);
  memcpy(d.fixed_aero_err, c.fixed_aero_err, sizeof d.fixed_aero_err);
  const double pid_cs[4] = B747_DEF_PID_CS, pid_ss[4] = B747_DEF_PID_SS;
  memcpy(d.mp.PID_CS, pid_cs, sizeof pid_cs); memcpy(d.mp.PID_SS, pid_ss, sizeof pid_ss);
  d.mp.P = B747_DEF_P; d.mp.Iz = B747_DEF_IZ; d.mp.S = B747_DEF_S; d.mp.c_ = B747_DEF_C; d.mp.g = B747_DEF_G;
  d.mp.m0 = B747_DEF_M0; d.mp.use_RP = 1.0; d.mp.use_RL = B747_DEF_USE_RL;
  // Controller._init_model (core/controller.py:128-131): use_PID_SS = not manual_stab
  bool manual = c.ctrl_type == B747_CTRL_MANUAL || c.ctrl_type == B747_CTRL_SEMI_MANUAL;
  d.mp.use_PID_SS = manual ? 0.0 : 1.0;
  return 0;
}

static int create_body(b747_handle* h, const b747_cfg* cfg);

extern "C" int b747_create(const b747_cfg* cfg, b747_handle** out) {
  if (!cfg || !out) return fail(B747_ERR_ARG, "null argument");
  if (cfg->abi_version != B747_ABI_VERSION) return fail(B747_ERR_ARG, "abi_version mismatch");
  if (cfg->n_envs <= 0) return fail(B747_ERR_ARG, "n_envs must be > 0");
  if (cfg->dtype != B747_F64 && cfg->dtype != B747_F32) return fail(B747_ERR_ARG, "dtype must be B747_F64 or B747_F32");
  if (obs_dim_of(cfg->obs_type) < 0) return fail(B747_ERR_ARG, "unknown obs_type");
  if (cfg->rew_type < 0 || cfg->rew_type > 4) return fail(B747_ERR_ARG, "unknown rew_type");
  if (cfg->ctrl_type < 0 || cfg->ctrl_type > 3) return fail(B747_ERR_ARG, "unknown ctrl_type");
  if (cfg->ctrl_mode < B747_MODE_NONE || cfg->ctrl_mode > 3) return fail(B747_ERR_ARG, "unknown ctrl_mode");
  // the reference asserts this in Controller.__init__ (core/controller.py:103)
  if (cfg->ctrl_mode == B747_MODE_NONE && cfg->env_layer &&
      (cfg->ctrl_type == B747_CTRL_MANUAL || cfg->ctrl_type == B747_CTRL_SEMI_MANUAL))
    return fail(B747_ERR_ARG, "ctrl_mode None needs the СС PID in the loop (CtrlType.AUTO / FULL_AUTO)");
  if (cfg->reset_ref_mode < -1 || cfg->reset_ref_mode > 2) return fail(B747_ERR_ARG, "unknown reset_ref_mode");
  if (cfg->substeps < 1) return fail(B747_ERR_ARG, "substeps must be >= 1");
  if (cfg->dtype == B747_F32 && !cfg->env_layer)
    return fail(B747_ERR_ARG, "env_layer=0 (raw Model stepping) needs dtype B747_F64");
  // the reference asserts this in Controller.reset (core/controller.py:145)
  if (cfg->reset_ref_mode != B747_RESET_NONE && cfg->env_layer &&
      !(cfg->ctrl_type == B747_CTRL_SEMI_MANUAL || cfg->ctrl_type == B747_CTRL_MANUAL))
    return fail(B747_ERR_ARG, "random reset needs the NN in the stabilisation loop (MANUAL / SEMI_MANUAL)");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(B747_ERR_CUDA, std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "count=0") +
                                   " (libb747_b200 has no CPU path)");
  if (cfg->device < 0 || cfg->device >= ndev) return fail(B747_ERR_ARG, "device ordinal out of range");
  CU(cudaSetDevice(cfg->device));
  if (cfg->record_capacity > 0 &&
      sizeof(double) * (size_t)cfg->record_capacity * NREC * (size_t)cfg->n_envs > ((size_t)8 << 30))
    return fail(B747_ERR_ALLOC, "recorder larger than 8 GiB: lower record_capacity or n_envs");
  b747_handle* h = new b747_handle();
  h->cfg = *cfg;
  fill_devcfg(*cfg, h->dc);
  // every failure below releases the handle and whatever it allocated so far (a retry with fewer envs finds the HBM free)
  const int rc = create_body(h, cfg);
  if (rc != B747_OK) {
    const std::string msg = g_err;
    b747_destroy(h);
    return fail(rc, msg);
  }
  *out = h;
  return B747_OK;
}

static int create_body(b747_handle* h, const b747_cfg* cfg) {
  CU(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  h->own_stream = true;
  const size_t np = (size_t)h->dc.n_pad;
  const int od = h->dc.obs_dim;
  if (cfg->track_transfer) {
    CU(cudaMalloc(&h->trace.trk, sizeof(double) * 2 * NTRK * np));
    CU(cudaMalloc(&h->trace.snap, sizeof(double) * 2 * NTRK * np));
    CU(cudaMemsetAsync(h->trace.trk, 0, sizeof(double) * 2 * NTRK * np, h->stream));
    CU(cudaMemsetAsync(h->trace.snap, 0, sizeof(double) * 2 * NTRK * np, h->stream));
    CU(cudaMalloc(&h->d_metrics, sizeof(double) * 5 * np));
  }
  if (cfg->record_capacity > 0) {
    const size_t bytes = sizeof(double) * (size_t)cfg->record_capacity * NREC * (size_t)cfg->n_envs;
    CU(cudaMalloc(&h->trace.rec, bytes));
    CU(cudaMemsetAsync(h->trace.rec, 0, bytes, h->stream));
    h->trace.rec_cap = cfg->record_capacity;
    h->trace.rec_stride = cfg->n_envs;
  }
  h->s64.trace = h->trace;
  h->s32.trace = h->trace;
  if (cfg->dtype == B747_F64) {
    StateF64& s = h->s64;
    CU(cudaMalloc(&s.slots, sizeof(double) * np * (NSLOT_F64 + 6)));
    CU(cudaMalloc(&s.tick, sizeof(int) * np));
    CU(cudaMalloc(&s.flags, sizeof(int) * np));
    CU(cudaMalloc(&s.ep_idx, sizeof(uint32_t) * np));
    if (cfg->export_signals) CU(cudaMalloc(&s.sig, sizeof(double) * np * NSIG));
    CU(cudaMalloc(&s.stats, sizeof(double) * 4));
    CU(cudaMalloc(&s.last_ret, sizeof(double) * np));
    CU(cudaMalloc(&s.last_len, sizeof(int) * np));
    CU(cudaMemsetAsync(s.slots, 0, sizeof(double) * np * (NSLOT_F64 + 6), h->stream));
    CU(cudaMemsetAsync(s.stats, 0, sizeof(double) * 4, h->stream));
    launch_defaults64(h->dc, s, h->stream);
    h->launches++;
  } else {
    int rc = f32_alloc(h->dc, h->s32, cfg->export_signals != 0, h->stream);
    if (rc) return fail(B747_ERR_CUDA, std::string("f32 state allocation: ") + cudaGetErrorString(cudaGetLastError()));
    launch_defaults32(h->dc, h->s32, h->stream);
    h->launches++;
    f32_warm_launch();
  }
  CU(cudaMalloc(&h->d_act, h->elem() * np));
  CU(cudaMalloc(&h->d_obs, h->elem() * np * od));
  CU(cudaMalloc(&h->d_rew, h->elem() * np));
  CU(cudaMalloc(&h->d_term, h->elem() * np * od));
  CU(cudaMalloc(&h->d_done, np));
  CU(cudaMalloc(&h->d_eps, sizeof(b747_episode) * np));
  CU(cudaGetLastError());
  CU(cudaStreamSynchronize(h->stream));
  return B747_OK;
}

extern "C" int b747_destroy(b747_handle* h) {
  if (!h) return B747_OK;
  cudaSetDevice(h->cfg.device);
  if (h->stream || !h->own_stream) cudaStreamSynchronize(h->stream);
  cudaFree(h->d_out4); cudaFree(h->d_bits);
  cudaFree(h->trace.trk); cudaFree(h->trace.snap); cudaFree(h->trace.rec); cudaFree(h->d_metrics);
  StateF64& s = h->s64;
  cudaFree(s.slots); cudaFree(s.tick); cudaFree(s.flags); cudaFree(s.ep_idx); cudaFree(s.sig); cudaFree(s.stats);
  cudaFree(s.last_ret); cudaFree(s.last_len);
  f32_free(h->s32);
  cudaFree(h->d_act); cudaFree(h->d_obs); cudaFree(h->d_rew); cudaFree(h->d_term); cudaFree(h->d_done); cudaFree(h->d_eps);
  if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
  for (cudaEvent_t e : h->ev_in) cudaEventDestroy(e);
  for (cudaEvent_t e : h->ev_k) cudaEventDestroy(e);
  if (h->ev_start) cudaEventDestroy(h->ev_start);
  if (h->ev_done) cudaEventDestroy(h->ev_done);
  for (auto& g : h->graphs) cudaGraphExecDestroy(g.exec);
  if (h->s_in) cudaStreamDestroy(h->s_in);
  if (h->s_aux) cudaStreamDestroy(h->s_aux);
  if (h->s_out) cudaStreamDestroy(h->s_out);
  if (h->s_cap) cudaStreamDestroy(h->s_cap);
  delete h;
  return B747_OK;
}

extern "C" void* b747_stream(b747_handle* h) { return h ? (void*)h->stream : nullptr; }
extern "C" int b747_set_stream(b747_handle* h, void* s) {
  if (!h) return fail(B747_ERR_ARG, "null handle");
  cudaStreamSynchronize(h->stream);
  if (h->own_stream) cudaStreamDestroy(h->stream);
  h->stream = (cudaStream_t)s;
  h->own_stream = false;
  return B747_OK;
}
extern "C" int64_t b747_launch_count(b747_handle* h) { return h ? h->launches : 0; }

// ---- trace: step-response metrics and recorder ---------------------------------------------------
extern "C" int b747_transfer_metrics(b747_handle* h, int which, int finished, double* out) {
  if (!h || !out) return fail(B747_ERR_ARG, "null argument");
  if (!h->trace.trk) return fail(B747_ERR_STATE, "handle was created without track_transfer");
  CU(cudaSetDevice(h->cfg.device));
  launch_transfer_metrics(h->dc, h->trace, which, finished, h->d_metrics, h->stream);
  h->launches++;
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(out, h->d_metrics, sizeof(double) * 5 * h->cfg.n_envs, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return B747_OK;
}
static const char* kRecNames[NREC] = {"t", "U_com", "U_PID", "deltaz", "hzh", "vartheta_ref", "U_RL", "x", "y", "Vx", "Vy",
                                      "vartheta", "wz"};
extern "C" int b747_recorder_n_fields(void) { return NREC; }
extern "C" const char* b747_recorder_field_name(int f) { return (f >= 0 && f < NREC) ? kRecNames[f] : nullptr; }
extern "C" int b747_recorder_read(b747_handle* h, int env, double* out, int32_t* n_steps) {
  if (!h || !out || !n_steps) return fail(B747_ERR_ARG, "null argument");
  if (!h->trace.rec) return fail(B747_ERR_STATE, "handle was created with record_capacity = 0");
  if (env < 0 || env >= h->cfg.n_envs) return fail(B747_ERR_ARG, "env out of range");
  CU(cudaSetDevice(h->cfg.device));
  CU(cudaStreamSynchronize(h->stream));
  const int tick_field = b747_field_index("tick");
  std::vector<double> ticks(h->cfg.n_envs);
  int rc = b747_get_field(h, tick_field, ticks.data());
  if (rc) return rc;
  const int cap = h->trace.rec_cap, n = std::min(cap, (int)ticks[env]);
  const size_t rs = (size_t)h->trace.rec_stride;
  // rec[step][field][env]: one strided 2-D copy (one double per (step, field) row)
  std::vector<double> tmp((size_t)cap * NREC);
  CU(cudaMemcpy2D(tmp.data(), sizeof(double), h->trace.rec + env, sizeof(double) * rs, sizeof(double), (size_t)cap * NREC,
                  cudaMemcpyDeviceToHost));
  for (int f = 0; f < NREC; f++)
    for (int k = 0; k < cap; k++) out[(size_t)f * cap + k] = k < n ? tmp[(size_t)k * NREC + f] : 0.0;
  *n_steps = n;
  return B747_OK;
}
extern "C" int b747_synchronize(b747_handle* h) {
  if (!h) return fail(B747_ERR_ARG, "null handle");
  CU(cudaStreamSynchronize(h->stream));
  return B747_OK;
}

// ---- reset / step ----------------------------------------------------------------------------
extern "C" int b747_reset(b747_handle* h, const uint8_t* mask_dev, void* obs_dev) {
  if (!h) return fail(B747_ERR_ARG, "null handle");
  CU(cudaSetDevice(h->cfg.device));
  if (h->cfg.dtype == B747_F64) launch_reset64(h->dc, h->s64, mask_dev, nullptr, (double*)obs_dev, h->stream);
  else launch_reset32(h->dc, h->s32, mask_dev, nullptr, (float*)obs_dev, h->stream);
  h->launches++;
  CU(cudaGetLastError());
  return B747_OK;
}

extern "C" int b747_reset_to_masked(b747_handle* h, const b747_episode* eps, const uint8_t* mask_dev, void* obs_dev) {
  if (!h || !eps) return fail(B747_ERR_ARG, "null argument");
  CU(cudaSetDevice(h->cfg.device));
  // explicit episodes can ask for what the handle's configuration family never produces (closed altitude loop,
  // oscillating reference, aero errors): from then on the f32 launch takes the full kernel tier
  for (int i = 0; i < h->cfg.n_envs && !h->dc.force_full; i++) {
    const b747_episode& e = eps[i];
    bool special = e.use_ctrl || e.oscillating;
    for (int k = 0; k < 5; k++) special = special || e.aero_err[k] != 0.0;
    if (special) { h->dc.force_full = 1; h->epoch++; }
  }
  CU(cudaMemcpyAsync(h->d_eps, eps, sizeof(b747_episode) * h->cfg.n_envs, cudaMemcpyHostToDevice, h->stream));
  if (h->cfg.dtype == B747_F64) launch_reset64(h->dc, h->s64, mask_dev, h->d_eps, (double*)obs_dev, h->stream);
  else launch_reset32(h->dc, h->s32, mask_dev, h->d_eps, (float*)obs_dev, h->stream);
  h->launches++;
  CU(cudaGetLastError());
  CU(cudaStreamSynchronize(h->stream));  // eps is caller memory
  return B747_OK;
}

extern "C" int b747_reset_to(b747_handle* h, const b747_episode* eps, void* obs_dev) {
  return b747_reset_to_masked(h, eps, nullptr, obs_dev);
}

// One env step of envs [lo, hi) on stream s with the step kernel of the handle's dtype.
static void step_range(b747_handle* h, int lo, int hi, const void* act, void* obs, void* rew, uint8_t* done, void* term,
                       cudaStream_t s) {
  DevCfg dc = h->dc;
  dc.env_lo = lo; dc.env_hi = hi;
  if (h->cfg.dtype == B747_F64)
    launch_env_step64(dc, h->s64, (const double*)act, (double*)obs, (double*)rew, done, (double*)term, s);
  else
    launch_env_step32(dc, h->s32, (const float*)act, (float*)obs, (float*)rew, done, (float*)term, s);
  h->launches++;
}

extern "C" int b747_step(b747_handle* h, const void* act, void* obs, void* rew, uint8_t* done, void* term) {
  if (!h || !act || !obs || !rew || !done) return fail(B747_ERR_ARG, "null argument");
  if (!h->cfg.env_layer) return fail(B747_ERR_STATE, "handle was created with env_layer=0; use b747_model_step");
  CU(cudaSetDevice(h->cfg.device));
  step_range(h, 0, h->cfg.n_envs, act, obs, rew, done, term, h->stream);
  CU(cudaGetLastError());
  return B747_OK;
}

extern "C" int b747_set_host_chunks(b747_handle* h, int n_chunks) {
  if (!h || n_chunks < 0 || n_chunks > 64) return fail(B747_ERR_ARG, "n_chunks must be in 0..64 (0 = automatic)");
  h->host_chunks = n_chunks;
  return B747_OK;
}

// Number of chunks of a host step, `per` envs each (whole thread blocks; the last chunk is ragged).  Without
// can_pipeline the step is one chunk.
static int plan_chunks(const b747_handle* h, bool can_pipeline, size_t& per) {
  const size_t n = (size_t)h->cfg.n_envs;
  int chunks = 1;
  if (can_pipeline) chunks = h->host_chunks ? h->host_chunks : (n >= ((size_t)1 << 17) ? 4 : 1);  // measured: 4 beats 8 and 2
  per = ((n + chunks - 1) / chunks + 127) / 128 * 128;
  return (int)((n + per - 1) / per);  // whole-block rounding can empty the last chunks
}

// The pipeline's copy-in / second compute / copy-out streams, the capture stream, the fork / join events and one pair of
// events per chunk, created on first use (b747_destroy releases them).
static int pipeline_resources(b747_handle* h, int chunks) {
  if (chunks < 2) return B747_OK;
  if (!h->s_in) {
    CU(cudaStreamCreateWithFlags(&h->s_in, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&h->s_aux, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&h->s_out, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&h->s_cap, cudaStreamNonBlocking));
    CU(cudaEventCreateWithFlags(&h->ev_start, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&h->ev_done, cudaEventDisableTiming));
  }
  while ((int)h->ev_in.size() < chunks) {
    cudaEvent_t a, b;
    CU(cudaEventCreateWithFlags(&a, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&b, cudaEventDisableTiming));
    h->ev_in.push_back(a); h->ev_k.push_back(b);
  }
  return B747_OK;
}

// A copy between a caller's host buffer and its device staging: unit_bytes per envs_per_unit envs (1 for per-env
// arrays, 32 for done bits; chunks start at whole thread blocks, so at whole units).
struct HostXfer {
  void* host;
  void* dev;
  size_t unit_bytes, envs_per_unit;
  size_t off(size_t lo) const { return lo / envs_per_unit * unit_bytes; }
  size_t len(size_t lo, size_t hi) const { return (hi - lo + envs_per_unit - 1) / envs_per_unit * unit_bytes; }
};

// Enqueue one env step with HOST buffers (b747_step_host, and b747_step_host_packed in copy mode): per chunk [lo, hi)
// the copy-in, launch(lo, hi, stream) and the copy-outs in list order.  One chunk runs on `origin` alone.  More chunks
// run as a pipeline -- actions of chunk c+1 go up and results of chunk c-1 come down (PCIe is full duplex, the copy
// engines run beside the SMs) while chunk c is stepped; chunks alternate between two compute streams so that the tail
// wave of one overlaps the head of the next.  The pipeline forks from `origin` and joins back into it, so the whole step
// is ordered like a single operation on that stream -- and can be stream-captured.  Environments are independent, so
// chunking cannot change any result.
template <class Launch>
static int issue_pipeline(b747_handle* h, cudaStream_t origin, const HostXfer& in, const HostXfer* outs, int n_outs,
                          int chunks, size_t per, Launch launch) {
  const size_t n = (size_t)h->cfg.n_envs;
  const bool fork = chunks > 1;
  const cudaStream_t s_in = fork ? h->s_in : origin, s_out = fork ? h->s_out : origin;
  if (fork) {  // everything queued on the origin stream so far (resets, device-side steps) comes first
    CU(cudaEventRecord(h->ev_start, origin));
    CU(cudaStreamWaitEvent(h->s_in, h->ev_start, 0));
    CU(cudaStreamWaitEvent(h->s_aux, h->ev_start, 0));
  }
  for (int c = 0; c < chunks; c++) {
    const size_t lo = (size_t)c * per, hi = std::min(n, lo + per);
    CU(cudaMemcpyAsync((char*)in.dev + in.off(lo), (char*)in.host + in.off(lo), in.len(lo, hi), cudaMemcpyHostToDevice, s_in));
    const cudaStream_t sc = (c & 1) ? h->s_aux : origin;
    if (fork) {
      CU(cudaEventRecord(h->ev_in[c], s_in));
      CU(cudaStreamWaitEvent(sc, h->ev_in[c], 0));
    }
    launch((int)lo, (int)hi, sc);
    CU(cudaGetLastError());
    if (fork) {
      CU(cudaEventRecord(h->ev_k[c], sc));
      CU(cudaStreamWaitEvent(s_out, h->ev_k[c], 0));
    }
    for (const HostXfer* o = outs; o < outs + n_outs; o++)
      CU(cudaMemcpyAsync((char*)o->host + o->off(lo), (char*)o->dev + o->off(lo), o->len(lo, hi), cudaMemcpyDeviceToHost, s_out));
  }
  if (fork) {  // join: the copy-out stream has seen every chunk's kernel (and through them every copy-in)
    CU(cudaEventRecord(h->ev_done, s_out));
    CU(cudaStreamWaitEvent(origin, h->ev_done, 0));
  }
  return B747_OK;
}

static bool is_pinned(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeHost;
}

extern "C" int b747_step_host(b747_handle* h, const void* act, void* obs, void* rew, uint8_t* done, void* term) {
  if (!h || !act || !obs || !rew || !done) return fail(B747_ERR_ARG, "null argument");
  if (!h->cfg.env_layer) return fail(B747_ERR_STATE, "handle was created with env_layer=0; use b747_model_step");
  CU(cudaSetDevice(h->cfg.device));
  const size_t es = h->elem(), od = (size_t)h->dc.obs_dim;
  size_t per;
  const int chunks = plan_chunks(h, true, per);
  int rc = pipeline_resources(h, chunks);
  if (rc != B747_OK) return rc;
  const HostXfer in{(void*)act, h->d_act, es, 1};
  const HostXfer outs[4] = {{obs, h->d_obs, es * od, 1}, {rew, h->d_rew, es, 1}, {done, h->d_done, 1, 1},
                            {term, h->d_term, es * od, 1}};
  const int n_outs = term ? 4 : 3;
  void* d_term = term ? h->d_term : nullptr;
  auto launch = [&](int lo, int hi, cudaStream_t s) { step_range(h, lo, hi, h->d_act, h->d_obs, h->d_rew, h->d_done, d_term, s); };
  // Pinned buffers: the ~70 stream operations of the pipeline are captured once per buffer set into a CUDA graph and
  // replayed with one launch call per step (the host-side issue time of the eager form is a third of the step).
  if (chunks > 1 && h->use_graphs && is_pinned(act) && is_pinned(obs) && is_pinned(rew) && is_pinned(done) &&
      (!term || is_pinned(term))) {
    cudaGraphExec_t exec = nullptr;
    for (auto& g : h->graphs)
      if (g.act == act && g.obs == obs && g.rew == rew && g.done == done && g.term == term && g.chunks == chunks &&
          g.epoch == h->epoch) { exec = g.exec; break; }
    if (!exec) {
      cudaGraph_t graph = nullptr;
      // captured on an internal stream (the handle's stream may be the legacy default stream, which cannot capture)
      CU(cudaStreamBeginCapture(h->s_cap, cudaStreamCaptureModeThreadLocal));
      const int64_t launches0 = h->launches;
      rc = issue_pipeline(h, h->s_cap, in, outs, n_outs, chunks, per, launch);
      h->launches = launches0;
      const cudaError_t ce = cudaStreamEndCapture(h->s_cap, &graph);
      if (rc != B747_OK || ce != cudaSuccess || !graph) {
        if (graph) cudaGraphDestroy(graph);
        cudaGetLastError();
        h->use_graphs = false;  // capture is not available here: eager pipeline from now on
      } else {
        const cudaError_t ie = cudaGraphInstantiate(&exec, graph, 0);
        cudaGraphDestroy(graph);
        if (ie != cudaSuccess) { cudaGetLastError(); exec = nullptr; h->use_graphs = false; }
        else {
          if (h->graphs.size() >= 8) { cudaGraphExecDestroy(h->graphs.front().exec); h->graphs.erase(h->graphs.begin()); }
          h->graphs.push_back({act, obs, rew, (void*)done, term, chunks, h->epoch, exec});
        }
      }
    }
    if (exec) {
      CU(cudaGraphLaunch(exec, h->stream));
      h->launches += chunks;
      CU(cudaStreamSynchronize(h->stream));
      return B747_OK;
    }
  }
  rc = issue_pipeline(h, h->stream, in, outs, n_outs, chunks, per, launch);
  if (rc != B747_OK) return rc;
  CU(cudaStreamSynchronize(h->stream));
  return B747_OK;
}

// ---- packed outputs ------------------------------------------------------------------------------
// One record per env (obs before any auto-reset, reward, padded to whole float4s) + one done bit per env: what the
// SB3-facing VecEnv needs from a step; ONE 128-bit store per thread for the 3-scalar layouts, 2-3 for the wider ones.
static int packed_ok(b747_handle* h) {
  if (h->cfg.dtype != B747_F32) return fail(B747_ERR_STATE, "packed outputs need an f32 handle");
  if (!h->cfg.env_layer) return fail(B747_ERR_STATE, "handle was created with env_layer=0; use b747_model_step");
  return B747_OK;
}
extern "C" int b747_packed_record_floats(int obs_type) {
  const int od = obs_dim_of(obs_type);
  return od < 0 ? -1 : 4 * ((od + 4) / 4);
}

extern "C" int b747_step_packed(b747_handle* h, const float* act_dev, float* out4_dev, uint32_t* done_bits_dev) {
  if (!h || !act_dev || !out4_dev || !done_bits_dev) return fail(B747_ERR_ARG, "null argument");
  const int rc = packed_ok(h);
  if (rc) return rc;
  CU(cudaSetDevice(h->cfg.device));
  launch_env_step32(h->dc, h->s32, act_dev, nullptr, nullptr, nullptr, nullptr, h->stream, (float4*)out4_dev, done_bits_dev);
  h->launches++;
  CU(cudaGetLastError());
  return B747_OK;
}

extern "C" int b747_set_host_mode(b747_handle* h, int mode) {
  if (!h || mode < -1 || mode > 2) return fail(B747_ERR_ARG, "mode must be -1 (automatic), 0, 1 or 2");
  h->host_mode = mode;
  h->auto_calls = 0; h->auto_choice = -1; h->auto_sec[0] = h->auto_sec[1] = 0.0;
  return B747_OK;
}

// device alias of a pinned (mapped) host pointer; nullptr if the memory is not pinned or not device-accessible
static void* mapped_ptr(const void* p, bool pinned) {
  void* d = nullptr;
  if (pinned && cudaHostGetDevicePointer(&d, (void*)p, 0) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  return d;
}

extern "C" int b747_step_host_packed(b747_handle* h, const float* act, float* out4, uint32_t* done_bits) {
  if (!h || !act || !out4 || !done_bits) return fail(B747_ERR_ARG, "null argument");
  int rc = packed_ok(h);
  if (rc) return rc;
  CU(cudaSetDevice(h->cfg.device));
  const size_t n = (size_t)h->cfg.n_envs, np = (size_t)h->dc.n_pad, nw = (n + 31) / 32;
  const size_t rec4 = ((size_t)h->dc.obs_dim + 4) / 4;  // float4s per record
  if (!h->d_bits) CU(cudaMalloc(&h->d_bits, sizeof(uint32_t) * (np / 32)));
  const bool pin_act = is_pinned(act), pin_out = is_pinned(out4), pin_bits = is_pinned(done_bits);
  float* m_act = (float*)mapped_ptr(act, pin_act);
  float4* m_out = (float4*)mapped_ptr(out4, pin_out);
  int mode = h->host_mode;
  const bool can_map = m_out && m_act && pin_bits;
  bool calibrating = false;
  if (mode < 0) {
    mode = 2;
    if (can_map && n >= ((size_t)1 << 17)) {  // small batches: launch-bound either way, zero-copy has fewer operations
      if (h->auto_choice >= 0) mode = h->auto_choice;
      else { calibrating = true; mode = (h->auto_calls & 1) ? 0 : 2; }
    }
  }
  if (!m_out || !pin_bits) mode = 0;
  if (mode == 2 && !m_act) mode = 1;
  const auto t_begin = std::chrono::steady_clock::now();
  struct Calib {  // on every return path: book the call's time and decide after 4 + 4 calls (the first pair is warm-up)
    b747_handle* h; bool on; int mode; std::chrono::steady_clock::time_point t0;
    ~Calib() {
      if (!on) return;
      const double dt = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
      if (h->auto_calls >= 2) h->auto_sec[mode == 0 ? 1 : 0] += dt;
      if (++h->auto_calls >= 10) h->auto_choice = h->auto_sec[1] < 0.95 * h->auto_sec[0] ? 0 : 2;
    }
  } calib{h, calibrating, mode, t_begin};
  if (mode >= 1) {
    // Zero-copy: the kernel stores each env's float4 straight into the caller's pinned buffer -- 512 contiguous bytes per
    // warp, posted PCIe writes that overlap the stepping of the other tiles -- and (mode 2) fetches the actions from the
    // pinned buffer one tile ahead.  No chunk pipeline, no fill / drain: one launch and one 4-byte-per-warp copy of the
    // done words.
    const float* a_dev = m_act;
    if (mode == 1) {
      CU(cudaMemcpyAsync(h->d_act, act, sizeof(float) * n, cudaMemcpyHostToDevice, h->stream));
      a_dev = (const float*)h->d_act;
    }
    launch_env_step32(h->dc, h->s32, a_dev, nullptr, nullptr, nullptr, nullptr, h->stream, m_out, h->d_bits, mode == 2);
    h->launches++;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(done_bits, h->d_bits, sizeof(uint32_t) * nw, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return B747_OK;
  }
  // copy mode (pageable buffers, or asked for): the host-step pipeline of b747_step_host with records and done words;
  // chunked only when all three buffers are pinned
  if (!h->d_out4) CU(cudaMalloc(&h->d_out4, sizeof(float4) * rec4 * np));
  size_t per;
  const int chunks = plan_chunks(h, pin_act && pin_out && pin_bits, per);
  rc = pipeline_resources(h, chunks);
  if (rc != B747_OK) return rc;
  const HostXfer in{(void*)act, h->d_act, sizeof(float), 1};
  const HostXfer outs[2] = {{out4, h->d_out4, sizeof(float4) * rec4, 1}, {done_bits, h->d_bits, sizeof(uint32_t), 32}};
  rc = issue_pipeline(h, h->stream, in, outs, 2, chunks, per, [&](int lo, int hi, cudaStream_t s) {
    DevCfg dc = h->dc;
    dc.env_lo = lo; dc.env_hi = hi;
    launch_env_step32(dc, h->s32, (const float*)h->d_act, nullptr, nullptr, nullptr, nullptr, s, h->d_out4, h->d_bits);
    h->launches++;
  });
  if (rc != B747_OK) return rc;
  CU(cudaStreamSynchronize(h->stream));
  return B747_OK;
}

// SB3's env.seed(s) (neural/agent.py:80): re-keys the Philox stream of every later random reset.
extern "C" int b747_set_seed(b747_handle* h, uint64_t seed) {
  if (!h) return fail(B747_ERR_ARG, "null handle");
  h->cfg.seed = seed;
  h->dc.seed = seed;
  h->epoch++;
  return B747_OK;
}

extern "C" int b747_model_step(b747_handle* h, int32_t n_steps) {
  if (!h || n_steps < 0) return fail(B747_ERR_ARG, "bad argument");
  CU(cudaSetDevice(h->cfg.device));
  if (h->cfg.dtype != B747_F64) return fail(B747_ERR_STATE, "raw model stepping needs an f64 handle (the reference's real_T is double)");
  launch_model_step64(h->dc, h->s64, n_steps, h->stream);
  h->launches++;
  CU(cudaGetLastError());
  return B747_OK;
}

extern "C" int b747_model_initialize(b747_handle* h) {
  if (!h) return fail(B747_ERR_ARG, "null handle");
  CU(cudaSetDevice(h->cfg.device));
  if (h->cfg.dtype != B747_F64) return fail(B747_ERR_STATE, "raw model stepping needs an f64 handle (the reference's real_T is double)");
  launch_model_init64(h->dc, h->s64, h->stream);
  h->launches++;
  CU(cudaGetLastError());
  return B747_OK;
}

// ---- uniform model parameters ----------------------------------------------------------------
static double* param_ptr(ModelParams& mp, const char* name, int& n) {
  n = 1;
  if (!strcmp(name, "PID_SS")) { n = 4; return mp.PID_SS; }
  if (!strcmp(name, "PID_CS")) { n = 4; return mp.PID_CS; }
  if (!strcmp(name, "P")) return &mp.P;
  if (!strcmp(name, "Iz")) return &mp.Iz;
  if (!strcmp(name, "S")) return &mp.S;
  if (!strcmp(name, "c_")) return &mp.c_;
  if (!strcmp(name, "g")) return &mp.g;
  if (!strcmp(name, "m0")) return &mp.m0;
  if (!strcmp(name, "use_RP")) return &mp.use_RP;
  if (!strcmp(name, "use_RL")) return &mp.use_RL;
  if (!strcmp(name, "use_PID_SS")) return &mp.use_PID_SS;
  return nullptr;
}
extern "C" int b747_set_param(b747_handle* h, const char* name, const double* v, int n) {
  if (!h || !name || !v) return fail(B747_ERR_ARG, "null argument");
  int len;
  double* p = param_ptr(h->dc.mp, name, len);
  if (!p || n != len) return fail(B747_ERR_ARG, std::string("unknown parameter or wrong length: ") + name);
  memcpy(p, v, sizeof(double) * len);
  h->epoch++;  // launch arguments changed: captured pipelines are stale
  return B747_OK;
}
extern "C" int b747_get_param(b747_handle* h, const char* name, double* v, int n) {
  if (!h || !name || !v) return fail(B747_ERR_ARG, "null argument");
  int len;
  double* p = param_ptr(h->dc.mp, name, len);
  if (!p || n != len) return fail(B747_ERR_ARG, std::string("unknown parameter or wrong length: ") + name);
  memcpy(v, p, sizeof(double) * len);
  return B747_OK;
}

// ---- per-env fields ---------------------------------------------------------------------------
static int field_io(b747_handle* h, int field, double* out, const double* in) {
  if (!h || field < 0 || field >= (int)fields().size()) return fail(B747_ERR_ARG, "bad field");
  CU(cudaSetDevice(h->cfg.device));
  CU(cudaStreamSynchronize(h->stream));
  const FieldDesc& f = fields()[field];
  const size_t n = (size_t)h->cfg.n_envs, np = (size_t)h->dc.n_pad;
  if (h->cfg.dtype == B747_F32) return f32_field_io(h->dc, h->s32, f.kind, f.row, f.name, out, in, h->stream) ? fail(B747_ERR_ARG, std::string("field not available on an f32 handle: ") + f.name) : B747_OK;
  StateF64& s = h->s64;
  std::vector<int> tmp;
  auto io_double = [&](double* dev) -> int {
    if (out) CU(cudaMemcpy(out, dev, sizeof(double) * n, cudaMemcpyDeviceToHost));
    else CU(cudaMemcpy(dev, in, sizeof(double) * n, cudaMemcpyHostToDevice));
    return B747_OK;
  };
  auto io_int = [&](int* dev) -> int {
    tmp.resize(n);
    if (out) {
      CU(cudaMemcpy(tmp.data(), dev, sizeof(int) * n, cudaMemcpyDeviceToHost));
      for (size_t i = 0; i < n; i++) out[i] = (double)tmp[i];
    } else {
      for (size_t i = 0; i < n; i++) tmp[i] = (int)in[i];
      CU(cudaMemcpy(dev, tmp.data(), sizeof(int) * n, cudaMemcpyHostToDevice));
    }
    return B747_OK;
  };
  switch (f.kind) {
    case FK_SLOT: return io_double(s.slots + (size_t)f.row * np);
    case FK_STATE0: return io_double(s.slots + (size_t)(NSLOT_F64 + f.row) * np);
    case FK_SIG:
      if (!s.sig) return fail(B747_ERR_STATE, "handle was created without export_signals");
      return io_double(s.sig + (size_t)f.row * np);
    case FK_TICK: return io_int(s.tick);
    case FK_FLAGS: return io_int(s.flags);
    case FK_EPIDX: return io_int((int*)s.ep_idx);
    case FK_LASTRET: return io_double(s.last_ret);
    case FK_LASTLEN: return io_int(s.last_len);
    case FK_MXONLY: return fail(B747_ERR_ARG, std::string("field only exists on f32 handles: ") + f.name);
  }
  return fail(B747_ERR_ARG, "bad field kind");
}
extern "C" int b747_get_field(b747_handle* h, int field, double* out) {
  if (!out) return fail(B747_ERR_ARG, "null argument");
  return field_io(h, field, out, nullptr);
}
extern "C" int b747_set_field(b747_handle* h, int field, const double* in) {
  if (!in) return fail(B747_ERR_ARG, "null argument");
  if (h && field == b747_field_index("flags") && !h->dc.force_full) { h->dc.force_full = 1; h->epoch++; }
  return field_io(h, field, nullptr, in);
}

// ---- state save / load (row table and copy kernel in b747_state.cu) -----------------------------------
static bool dtype_ok(int dtype) { return dtype == B747_F64 || dtype == B747_F32; }

extern "C" int64_t b747_state_bytes(const b747_cfg* cfg, int32_t n) {
  if (!cfg || n < 0 || !dtype_ok(cfg->dtype)) return fail(B747_ERR_ARG, "bad argument");
  return (int64_t)state_blob_bytes(state_table(*cfg, 0, nullptr, nullptr, nullptr), n);
}

static StateTable handle_state(const b747_handle* h) {
  return state_table(h->cfg, (size_t)h->dc.n_pad, &h->s32, &h->s64, &h->trace);
}

// the copy kernel moves 16-byte rows with 128-bit accesses at 16-byte offsets from the blob and reads int32 indices: a
// misaligned pointer would fault the context, so it is refused before anything is launched
static int state_ptrs_ok(const void* blob, const int32_t* a, const int32_t* b) {
  if ((uintptr_t)blob & 15) return fail(B747_ERR_ARG, "state blob must be 16-byte aligned");
  if (((uintptr_t)a | (uintptr_t)b) & 3) return fail(B747_ERR_ARG, "index arrays must be 4-byte aligned");
  return B747_OK;
}

extern "C" int b747_save_state(b747_handle* h, const int32_t* env_idx, int32_t n, void* blob) {
  if (!h || !blob || n < 0) return fail(B747_ERR_ARG, "bad argument");
  if (!env_idx && n > h->cfg.n_envs) return fail(B747_ERR_ARG, "n > n_envs without an index array");
  if (const int rc = state_ptrs_ok(blob, env_idx, nullptr)) return rc;
  CU(cudaSetDevice(h->cfg.device));
  const StateHeader hd = state_header(h->cfg, n, h->dc.force_full != 0);
  launch_state_copy(handle_state(h), (char*)blob, n, env_idx, nullptr, n, h->cfg.n_envs, true, hd, h->stream);
  h->launches++;
  CU(cudaGetLastError());
  return B747_OK;
}

extern "C" int b747_load_state(b747_handle* h, const void* blob, const int32_t* blob_idx, const int32_t* env_idx,
                               int32_t n) {
  if (!h || !blob || n < 0) return fail(B747_ERR_ARG, "bad argument");
  if (!env_idx && n > h->cfg.n_envs) return fail(B747_ERR_ARG, "n > n_envs without an index array");
  if (const int rc = state_ptrs_ok(blob, env_idx, blob_idx)) return rc;
  CU(cudaSetDevice(h->cfg.device));
  StateHeader hd;
  CU(cudaMemcpyAsync(&hd, blob, sizeof hd, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  const StateHeader want = state_header(h->cfg, hd.n, false);
  if (hd.magic != want.magic || hd.version != want.version || hd.n < 0)
    return fail(B747_ERR_STATE, "not a state blob of this format version");
  if (hd.dtype != want.dtype) return fail(B747_ERR_STATE, "state blob was saved from a handle of the other dtype");
  if (hd.key != want.key) return fail(B747_ERR_STATE, "state blob was saved from a handle with another configuration");
  // a restored closed altitude loop (or oscillating reference, aero errors) needs the full f32 kernel tier
  if ((hd.flags & kStateForceFull) && !h->dc.force_full) { h->dc.force_full = 1; h->epoch++; }
  launch_state_copy(handle_state(h), (char*)blob, hd.n, env_idx, blob_idx, n, h->cfg.n_envs, false, hd, h->stream);
  h->launches++;
  CU(cudaGetLastError());
  CU(cudaStreamSynchronize(h->stream));
  return B747_OK;
}

// ---- episode statistics -----------------------------------------------------------------------
extern "C" int b747_episode_stats(b747_handle* h, double out[4]) {
  if (!h || !out) return fail(B747_ERR_ARG, "null argument");
  CU(cudaSetDevice(h->cfg.device));
  double* st = h->cfg.dtype == B747_F64 ? h->s64.stats : h->s32.stats;
  CU(cudaMemcpyAsync(out, st, sizeof(double) * 4, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaMemsetAsync(st, 0, sizeof(double) * 4, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return B747_OK;
}

// Return / length of the most recently finished episode of SOME envs (the ones that just reported done): the
// VecMonitor record of a step costs a few kilobytes instead of two whole-batch copies.
__global__ void k_gather_last_episode(const double* __restrict__ ret, const int* __restrict__ len,
                                      const int32_t* __restrict__ idx, int n_idx, double* __restrict__ out_ret,
                                      int32_t* __restrict__ out_len) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_idx) return;
  out_ret[k] = ret[idx[k]];
  out_len[k] = len[idx[k]];
}

extern "C" int b747_last_episode_of(b747_handle* h, const int32_t* idx, int32_t n_idx, double* ret, int32_t* len) {
  if (!h || !idx || !ret || !len || n_idx < 0) return fail(B747_ERR_ARG, "bad argument");
  if (n_idx == 0) return B747_OK;
  if (n_idx > h->cfg.n_envs) return fail(B747_ERR_ARG, "more indices than environments");
  for (int32_t k = 0; k < n_idx; k++)
    if (idx[k] < 0 || idx[k] >= h->cfg.n_envs) return fail(B747_ERR_ARG, "env index out of range");
  CU(cudaSetDevice(h->cfg.device));
  // staging: the handle's per-env scratch (d_eps holds n_pad episode descriptors of 152 bytes: room for idx, ret and len)
  char* scratch = (char*)h->d_eps;
  int32_t* d_idx = (int32_t*)scratch;
  double* d_ret = (double*)(scratch + sizeof(double) * (size_t)h->dc.n_pad);
  int32_t* d_len = (int32_t*)(scratch + 2 * sizeof(double) * (size_t)h->dc.n_pad);
  CU(cudaMemcpyAsync(d_idx, idx, sizeof(int32_t) * n_idx, cudaMemcpyHostToDevice, h->stream));
  const double* lr = h->cfg.dtype == B747_F64 ? h->s64.last_ret : h->s32.last_ret;
  const int* ll = h->cfg.dtype == B747_F64 ? h->s64.last_len : h->s32.last_len;
  k_gather_last_episode<<<(n_idx + 255) / 256, 256, 0, h->stream>>>(lr, ll, d_idx, n_idx, d_ret, d_len);
  h->launches++;
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(ret, d_ret, sizeof(double) * n_idx, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaMemcpyAsync(len, d_len, sizeof(int32_t) * n_idx, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return B747_OK;
}

extern "C" int b747_last_episode(b747_handle* h, double* ret, int32_t* len) {
  if (!h || !ret || !len) return fail(B747_ERR_ARG, "null argument");
  CU(cudaSetDevice(h->cfg.device));
  CU(cudaStreamSynchronize(h->stream));
  const size_t n = (size_t)h->cfg.n_envs;
  if (h->cfg.dtype == B747_F64) {
    CU(cudaMemcpy(ret, h->s64.last_ret, sizeof(double) * n, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(len, h->s64.last_len, sizeof(int) * n, cudaMemcpyDeviceToHost));
  } else {
    CU(cudaMemcpy(ret, h->s32.last_ret, sizeof(double) * n, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(len, h->s32.last_len, sizeof(int) * n, cudaMemcpyDeviceToHost));
  }
  return B747_OK;
}
