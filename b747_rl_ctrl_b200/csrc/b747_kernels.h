// b747_kernels.h -- host-visible launchers of the env-step kernels (internal to libb747_b200.so).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "b747_common.cuh"

namespace b747 {

// Device pointers of a float64 handle.  slots: [NSLOT_F64 + 6][n_pad] doubles (the last six rows are
// the DLL's `state0` parameter); sig: [NSIG][n_pad] stage-4 signal export or nullptr.
struct StateF64 {
  double* slots;
  int* tick;
  int* flags;
  uint32_t* ep_idx;
  double* sig;
  double* stats;     // [4] episodes, sum return, sum length, sum return^2
  double* last_ret;  // [n_pad] return of the most recently finished episode
  int* last_len;     // [n_pad] its length in env steps
  TraceState trace;  // recorder / step-response tracker (optional)
};

// Device pointers of an f32 (throughput) handle; layout in b747_kernels_f32.cu.
struct StateF32 {
  double2* D = nullptr;
  float4* F = nullptr;
  float* sig = nullptr;
  double* stats = nullptr;
  double* last_ret = nullptr;
  int* last_len = nullptr;
  TraceState trace;  // recorder / step-response tracker (optional; routes the launch to the general kernel)
  float4* tables = nullptr;  // merged-axis look-up tables (b747_tables.h), ft::CELLS float4
  unsigned int* tile_ctr = nullptr;  // 64 tile counters of the persistent step kernel (one per launch in flight)
};

// A handle's per-env storage as row blocks for b747_save_state / b747_load_state: n_rows rows of elem bytes per env
// (4, 8 or 16), row r of env i at base + r * stride + i * elem.  The blob stores each row as its entries padded to
// 16 bytes (state_blob_bytes); a table built without a handle (null bases) still gives every size.
struct StateBlock {
  char* base;
  size_t stride;  // bytes between rows
  int32_t elem, n_rows;
};
constexpr int kMaxStateBlocks = 12;
struct StateTable {
  StateBlock b[kMaxStateBlocks];
  int n_blocks = 0, n_rows = 0;
  void add(const void* base, int elem, size_t stride, int n_rows_) {
    b[n_blocks++] = {(char*)base, stride, elem, n_rows_};
    n_rows += n_rows_;
  }
};
// Leading 64 bytes of a blob.  key: hash of every b747_cfg field that fixes the layout or meaning of the state
// (all but n_envs, device, seed, env_id_offset).
struct StateHeader {
  uint32_t magic, version;
  int32_t dtype, n;
  uint32_t flags;  // kStateForceFull
  uint32_t reserved0;
  uint64_t key;
  uint64_t reserved[4];
};
static_assert(sizeof(StateHeader) == 64, "blob rows start 16-byte aligned");
constexpr uint32_t kStateMagic = 0x53373437u;  // "747S"
constexpr uint32_t kStateVersion = 1;
constexpr uint32_t kStateForceFull = 1;        // the saving handle ran the full f32 kernel tier (DevCfg::force_full)

// np: the handle's n_pad; s32 / s64 / trace may be null (sizes only).
StateTable state_table(const b747_cfg& cfg, size_t np, const StateF32* s32, const StateF64* s64,
                       const TraceState* trace);
size_t state_blob_bytes(const StateTable& t, int n);
StateHeader state_header(const b747_cfg& cfg, int n, bool force_full);
// save: blob entry k <- env env_idx[k] (+ the header); load: env env_idx[k] <- blob entry blob_idx[k] of a blob of
// blob_n entries.  Null index arrays are the identity; out-of-range entries skip k.
void launch_state_copy(const StateTable& t, char* blob, int blob_n, const int32_t* env_idx, const int32_t* blob_idx,
                       int n, int n_envs, bool save, const StateHeader& hdr, cudaStream_t s);

int f32_alloc(const DevCfg& c, StateF32& s, bool export_signals, cudaStream_t stream);
void f32_free(StateF32& s);
// the row blocks of what f32_alloc allocates per env (s may be null)
void f32_state_blocks(size_t np, bool export_signals, const StateF32* s, StateTable& t);
bool f32_is_lean(const DevCfg& c);
bool f32_needs_cs(const DevCfg& c);
void f32_warm_launch();
// out4 != nullptr: packed outputs (one float4 = obs[3] + reward per env, done flags as one bit per env in done_bits);
// obs / rew / done / term_obs are then unused.  prefetch_actions: `actions` is host-mapped memory.
// pe: the handle's per-env tunables (b747_set_env_param), nullptr outside per-env mode.
void launch_env_step32(const DevCfg& c, const StateF32& st, const float* actions, float* obs, float* rew, uint8_t* done,
                       float* term_obs, cudaStream_t s, float4* out4 = nullptr, uint32_t* done_bits = nullptr,
                       bool prefetch_actions = false, const EnvParams* pe = nullptr);
// random resets (eps == nullptr) of a handle with parameter ranges also draw the ranged rows of pe
void launch_reset32(const DevCfg& c, const StateF32& st, const uint8_t* mask, const b747_episode* eps, float* obs,
                    cudaStream_t s, const EnvParams* pe = nullptr);
// the float rows of envs env_idx[k] (nullptr: k) for k < n, recomputed from their double rows
void launch_env_param_derive32(const EnvParams& pe, size_t np, const int32_t* env_idx, int n, int n_envs, cudaStream_t s);
void launch_defaults32(const DevCfg& c, const StateF32& st, cudaStream_t s);
// Storage kind of a per-env field of b747_get_field / b747_set_field (field table in b747_capi.cu).
enum FieldKind { FK_SLOT, FK_STATE0, FK_SIG, FK_TICK, FK_FLAGS, FK_EPIDX, FK_LASTRET, FK_LASTLEN, FK_MXONLY };
int f32_field_io(const DevCfg& c, StateF32& s, FieldKind kind, int row, const char* name, double* out, const double* in,
                 cudaStream_t stream);

void launch_env_step64(const DevCfg& c, const StateF64& st, const double* actions, double* obs, double* rew,
                       uint8_t* done, double* term_obs, cudaStream_t s, const EnvParams* pe = nullptr);
void launch_model_step64(const DevCfg& c, const StateF64& st, int n_steps, cudaStream_t s, const EnvParams* pe = nullptr);
void launch_reset64(const DevCfg& c, const StateF64& st, const uint8_t* mask, const b747_episode* eps, double* obs,
                    cudaStream_t s, const EnvParams* pe = nullptr);
// b747_set_env_param / b747_get_env_param: rows [row0, row0 + n_comp) of envs env_idx[k] (nullptr: k) <-> vals[k][n_comp]
// (out-of-range entries skip k).  Outside per-env mode (pe.rows == nullptr) a get returns `batch`.
void launch_env_param_io(const EnvParams& pe, size_t np, int row0, int n_comp, const int32_t* env_idx, int n, int n_envs,
                         double* vals, bool set, const double batch[4], cudaStream_t s);
// every env's rows [row0, row0 + n_comp) <- v (entering per-env mode, b747_set_param in per-env mode)
void launch_env_param_fill(const EnvParams& pe, int n_envs, size_t np, int row0, int n_comp, const double v[4],
                           cudaStream_t s);
void launch_defaults64(const DevCfg& c, const StateF64& st, cudaStream_t s);
void launch_model_init64(const DevCfg& c, const StateF64& st, cudaStream_t s);
// calc_stepinfo's final arithmetic on the tracker (snapshot != 0: the last finished episode): out[env][5] =
// overshoot %, rise time, settling time, static error, Controller.quality (NaN where the reference returns None)
void launch_transfer_metrics(const DevCfg& c, const TraceState& tr, int which, int snapshot, double* out_dev,
                             cudaStream_t s);

}  // namespace b747
