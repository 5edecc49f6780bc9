// b747_env_params.cu -- per-env model tunables (b747_set_env_param / b747_get_env_param): scatter, gather and fill of a
// handle's double rows [NEP][n_pad] (EnvParams, b747_common.cuh).  The float rows of f32 handles are recomputed from the
// double rows by launch_env_param_derive32 (b747_kernels_f32.cu) after every write.
#include "b747_kernels.h"

namespace b747 {

// entry k: env env_idx[k] (k without an index array); an entry outside [0, n_envs) skips k
__global__ void __launch_bounds__(128) k_env_param_io(EnvParams pe, size_t np, int row0, int n_comp,
                                                      const int32_t* __restrict__ env_idx, int n, int n_envs,
                                                      double* __restrict__ vals, bool set, double b0, double b1, double b2,
                                                      double b3) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int i = env_idx ? env_idx[k] : k;
  if (i < 0 || i >= n_envs) return;
  const double batch[4] = {b0, b1, b2, b3};
  for (int j = 0; j < n_comp; j++) {
    double* row = pe.rows ? pe.rows + (size_t)(row0 + j) * np + i : nullptr;
    double* v = vals + (size_t)k * n_comp + j;
    if (set) *row = *v;
    else *v = row ? *row : batch[j];
  }
}

__global__ void __launch_bounds__(128) k_env_param_fill(EnvParams pe, int n_envs, size_t np, int row0, int n_comp,
                                                        double v0, double v1, double v2, double v3) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_envs) return;
  const double v[4] = {v0, v1, v2, v3};
  for (int j = 0; j < n_comp; j++) pe.rows[(size_t)(row0 + j) * np + i] = v[j];
}

void launch_env_param_io(const EnvParams& pe, size_t np, int row0, int n_comp, const int32_t* env_idx, int n, int n_envs,
                         double* vals, bool set, const double batch[4], cudaStream_t s) {
  if (n <= 0) return;
  k_env_param_io<<<(n + 127) / 128, 128, 0, s>>>(pe, np, row0, n_comp, env_idx, n, n_envs, vals, set, batch[0], batch[1],
                                                 batch[2], batch[3]);
}

void launch_env_param_fill(const EnvParams& pe, int n_envs, size_t np, int row0, int n_comp, const double v[4],
                           cudaStream_t s) {
  k_env_param_fill<<<(n_envs + 127) / 128, 128, 0, s>>>(pe, n_envs, np, row0, n_comp, v[0], v[1], v[2], v[3]);
}

}  // namespace b747
