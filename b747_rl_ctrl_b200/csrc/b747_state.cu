// b747_state.cu -- save / restore / fork of per-env state (b747_save_state, b747_load_state).
//
// A handle's per-env arrays are described by one table of row blocks (state_table); the blob is a 64-byte header
// followed by every row of every block, each row holding the n saved envs' entries padded to 16 bytes.  One kernel
// gathers (save) or scatters (load) (row, k) elements between the two in either direction; b747_state_bytes and the
// kernel both size the blob from the same table.
#include <string.h>

#include <algorithm>

#include "b747_kernels.h"

namespace b747 {

StateTable state_table(const b747_cfg& c, size_t np, const StateF32* s32, const StateF64* s64, const TraceState* tr) {
  StateTable t;
  if (c.dtype == B747_F32) {
    f32_state_blocks(np, c.export_signals != 0, s32, t);
  } else {
    t.add(s64 ? s64->slots : nullptr, sizeof(double), sizeof(double) * np, NSLOT_F64 + 6);  // + the six state0 rows
    t.add(s64 ? s64->tick : nullptr, sizeof(int), 0, 1);
    t.add(s64 ? s64->flags : nullptr, sizeof(int), 0, 1);
    t.add(s64 ? s64->ep_idx : nullptr, sizeof(uint32_t), 0, 1);
    t.add(s64 ? s64->last_ret : nullptr, sizeof(double), 0, 1);
    t.add(s64 ? s64->last_len : nullptr, sizeof(int), 0, 1);
    if (c.export_signals) t.add(s64 ? s64->sig : nullptr, sizeof(double), sizeof(double) * np, NSIG);
  }
  if (c.track_transfer) {
    t.add(tr ? tr->trk : nullptr, sizeof(double), sizeof(double) * np, 2 * NTRK);
    t.add(tr ? tr->snap : nullptr, sizeof(double), sizeof(double) * np, 2 * NTRK);
  }
  if (c.record_capacity > 0)  // rec[step][field][env], rows of n_envs (not n_pad) doubles
    t.add(tr ? tr->rec : nullptr, sizeof(double), sizeof(double) * (size_t)c.n_envs, c.record_capacity * NREC);
  return t;
}

__host__ __device__ inline size_t blob_row_bytes(size_t n, int elem) { return (n * (size_t)elem + 15) / 16 * 16; }

size_t state_blob_bytes(const StateTable& t, int n) {
  size_t bytes = sizeof(StateHeader);
  for (int j = 0; j < t.n_blocks; j++) bytes += (size_t)t.b[j].n_rows * blob_row_bytes((size_t)n, t.b[j].elem);
  return bytes;
}

// FNV-1a over the fields of b747_cfg that fix the layout or the meaning of the saved state
StateHeader state_header(const b747_cfg& c, int n, bool force_full) {
  uint64_t k = 0xcbf29ce484222325ull;
  auto mix = [&k](const void* p, size_t len) {
    for (size_t i = 0; i < len; i++) { k ^= ((const unsigned char*)p)[i]; k *= 0x100000001b3ull; }
  };
#define M(f) mix(&c.f, sizeof c.f);
  M(abi_version) M(dtype) M(obs_type) M(rew_type) M(ctrl_type) M(ctrl_mode) M(reset_ref_mode) M(disturbance_mode)
  M(norm_obs) M(norm_act) M(use_limiter) M(substeps) M(auto_reset) M(env_layer) M(done_tick) M(tk) M(action_max)
  M(vartheta_max) M(sample_time) M(rew) M(fixed_aero_err) M(has_fixed_aero_err) M(export_signals) M(track_transfer)
  M(record_capacity)
#undef M
  StateHeader h;
  memset(&h, 0, sizeof h);
  h.magic = kStateMagic; h.version = kStateVersion; h.dtype = c.dtype; h.n = n;
  h.flags = force_full ? kStateForceFull : 0u;
  h.key = k;
  return h;
}

// Thread (blockIdx.x, threadIdx.x) owns kStateEntries entries of the copy, kStateThreads apart, and walks rows
// blockIdx.y, + gridDim.y, ...: in each row it issues the loads of all its entries before their stores, so a thread keeps
// up to 64 bytes in flight, and a warp's access to one entry slot of a row is one contiguous (identity) or gathered
// segment.  16-byte rows move as 128-bit words.
constexpr int kStateThreads = 256, kStateEntries = 4;

template <class W>
__device__ __forceinline__ void copy_row(char* __restrict__ hrow, char* __restrict__ brow, const int* env, const int* e,
                                         const bool* ok, bool save) {
  W v[kStateEntries];
#pragma unroll
  for (int i = 0; i < kStateEntries; i++)
    if (ok[i]) v[i] = *(const W*)(save ? hrow + (size_t)env[i] * sizeof(W) : brow + (size_t)e[i] * sizeof(W));
#pragma unroll
  for (int i = 0; i < kStateEntries; i++)
    if (ok[i]) *(W*)(save ? brow + (size_t)e[i] * sizeof(W) : hrow + (size_t)env[i] * sizeof(W)) = v[i];
}

__global__ void __launch_bounds__(kStateThreads) k_state_copy(const StateTable t, char* __restrict__ blob, int blob_n,
                                                             const int32_t* __restrict__ env_idx,
                                                             const int32_t* __restrict__ blob_idx, int n, int n_envs,
                                                             bool save, const StateHeader hdr) {
  if (save && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) *(StateHeader*)blob = hdr;
  int env[kStateEntries], e[kStateEntries];
  bool ok[kStateEntries], any = false;
#pragma unroll
  for (int i = 0; i < kStateEntries; i++) {
    const int k = (blockIdx.x * kStateEntries + i) * kStateThreads + threadIdx.x;
    env[i] = k < n ? (env_idx ? env_idx[k] : k) : -1;
    e[i] = k < n ? (save ? k : (blob_idx ? blob_idx[k] : k)) : -1;
    ok[i] = env[i] >= 0 && env[i] < n_envs && e[i] >= 0 && e[i] < blob_n;
    any = any || ok[i];
  }
  if (!any) return;
  for (int r = blockIdx.y; r < t.n_rows; r += gridDim.y) {
    size_t off = sizeof(StateHeader);
    int j = 0, row = r;
    for (; row >= t.b[j].n_rows; j++) {
      off += (size_t)t.b[j].n_rows * blob_row_bytes((size_t)blob_n, t.b[j].elem);
      row -= t.b[j].n_rows;
    }
    const StateBlock& b = t.b[j];
    char* hrow = b.base + (size_t)row * b.stride;
    char* brow = blob + off + (size_t)row * blob_row_bytes((size_t)blob_n, b.elem);
    if (b.elem == 16) copy_row<uint4>(hrow, brow, env, e, ok, save);
    else if (b.elem == 8) copy_row<uint64_t>(hrow, brow, env, e, ok, save);
    else copy_row<uint32_t>(hrow, brow, env, e, ok, save);
  }
}

void launch_state_copy(const StateTable& t, char* blob, int blob_n, const int32_t* env_idx, const int32_t* blob_idx,
                       int n, int n_envs, bool save, const StateHeader& hdr, cudaStream_t s) {
  const int per_block = kStateThreads * kStateEntries;
  const dim3 grid((unsigned)std::max(1, (n + per_block - 1) / per_block), (unsigned)std::min(t.n_rows, 65535));
  k_state_copy<<<grid, kStateThreads, 0, s>>>(t, blob, blob_n, env_idx, blob_idx, n, n_envs, save, hdr);
}

}  // namespace b747
