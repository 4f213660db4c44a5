// odg_mppi.cu — MPPI sampling, cost accumulation and the on-device softmin reduction (include/odg_mppi.h).
#include <cuda_runtime.h>

#include <string>

#include "../../include/odg.h"
#include "../../include/odg_mppi.h"
#include "odg_sim_internal.h"

namespace {
using odg_internal::set_error;
#define CUDA_TRY(expr)                                                                         \
  do { cudaError_t e_ = (expr);                                                                \
       if (e_ != cudaSuccess) return set_error(ODG_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_)); } while (0)

__global__ void k_mppi_sample(const float* __restrict__ mean, float sigma, int N, int A, uint32_t seed_lo, uint32_t seed_hi,
                              uint32_t iteration, uint32_t t, float* __restrict__ action) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n < N) odg::mppi_sample_row(mean, sigma, n, A, seed_lo, seed_hi, iteration, t, action);
}

__global__ void k_mppi_accum(const float* __restrict__ reward, const unsigned char* __restrict__ term, int N, float term_cost,
                             float* __restrict__ cost, unsigned char* __restrict__ alive) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N || !alive[n]) return;
  float c = cost[n] - reward[n];
  if (term[n]) { c += term_cost; alive[n] = 0; }
  cost[n] = c;
}

constexpr int kRedThreads = 1024;
// One block per group of S samples (block g reads samples [g S, (g + 1) S) of the [T][N][A] action tensor and writes
// mean_out[g] and stats[g]); a group's arithmetic is that of a single-group call on a contiguous copy of its samples.
__global__ void __launch_bounds__(kRedThreads) k_mppi_reduce(const float* __restrict__ cost, const float* __restrict__ actions, int T,
                                                             int S, int N, int A, float lambda, float* __restrict__ mean_out,
                                                             float* __restrict__ stats) {
  extern __shared__ float s_w[];                 // [S] weights
  const int g = blockIdx.x;
  cost += (size_t)g * S; actions += (size_t)g * S * A; mean_out += (size_t)g * T * A;
  if (stats) stats += 4 * g;
  __shared__ float s_red[kRedThreads]; __shared__ int s_idx[kRedThreads];
  const int tid = threadIdx.x;
  // min cost (and its index), fixed tree
  float m = 3.4e38f; int mi = 0; float sum_c = 0.f;
  for (int n = tid; n < S; n += kRedThreads) { const float c = cost[n]; sum_c += c; if (c < m) { m = c; mi = n; } }
  s_red[tid] = m; s_idx[tid] = mi;
  __syncthreads();
  for (int d = kRedThreads / 2; d > 0; d >>= 1) {
    if (tid < d) {
      const float o = s_red[tid + d]; const int oi = s_idx[tid + d];
      if (o < s_red[tid] || (o == s_red[tid] && oi < s_idx[tid])) { s_red[tid] = o; s_idx[tid] = oi; }
    }
    __syncthreads();
  }
  const float cmin = s_red[0]; const int imin = s_idx[0];
  __syncthreads();
  // weights and their sum
  float ws = 0.f;
  for (int n = tid; n < S; n += kRedThreads) { const float w = expf(-(cost[n] - cmin) / lambda); s_w[n] = w; ws += w; }
  s_red[tid] = ws;
  __syncthreads();
  for (int d = kRedThreads / 2; d > 0; d >>= 1) { if (tid < d) s_red[tid] += s_red[tid + d]; __syncthreads(); }
  const float wsum = s_red[0];
  __syncthreads();
  s_red[tid] = sum_c;
  __syncthreads();
  for (int d = kRedThreads / 2; d > 0; d >>= 1) { if (tid < d) s_red[tid] += s_red[tid + d]; __syncthreads(); }
  if (tid == 0 && stats) { stats[0] = cmin; stats[1] = s_red[0] / (float)S; stats[2] = wsum; stats[3] = (float)imin; }
  // weighted mean per (t, a): thread per output element, samples summed in index order
  for (int o = tid; o < T * A; o += kRedThreads) {
    const int t = o / A, a = o % A;
    const float* p = actions + (size_t)t * N * A + a;
    float acc = 0.f;
    for (int n = 0; n < S; n++) acc += s_w[n] * p[(size_t)n * A];
    mean_out[o] = acc / wsum;
  }
}
}  // namespace

extern "C" {

int odg_mppi_sample(const float* mean_dev, float sigma, int n_samples, int act_dim, uint64_t seed, uint32_t iteration,
                    uint32_t t, float* action_dev, void* stream) {
  if (!mean_dev || !action_dev || n_samples < 1 || act_dim < 1 || act_dim > 16)
    return set_error(ODG_ERR_INVALID, "odg_mppi_sample: bad arguments");
  k_mppi_sample<<<(n_samples + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      mean_dev, sigma, n_samples, act_dim, (uint32_t)seed, (uint32_t)(seed >> 32), iteration, t, action_dev);
  CUDA_TRY(cudaGetLastError());
  return ODG_OK;
}

int odg_mppi_accumulate(const float* reward_dev, const uint8_t* terminated_dev, int n_samples, float termination_cost,
                        float* cost_dev, uint8_t* alive_dev, void* stream) {
  if (!reward_dev || !terminated_dev || !cost_dev || !alive_dev || n_samples < 1)
    return set_error(ODG_ERR_INVALID, "odg_mppi_accumulate: bad arguments");
  k_mppi_accum<<<(n_samples + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(reward_dev, terminated_dev, n_samples,
                                                                                        termination_cost, cost_dev, alive_dev);
  CUDA_TRY(cudaGetLastError());
  return ODG_OK;
}

int odg_mppi_reduce(const float* cost_dev, const float* actions_dev, int horizon, int n_samples, int act_dim, float lambda,
                    float* mean_out_dev, float* stats_dev, void* stream) {
  if (!cost_dev || !actions_dev || !mean_out_dev || horizon < 1 || n_samples < 1 || n_samples > 12000 || act_dim < 1 || !(lambda > 0.f))
    return set_error(ODG_ERR_INVALID, "odg_mppi_reduce: bad arguments (n_samples <= 12000)");
  return odg_mppi_reduce_groups(cost_dev, actions_dev, horizon, 1, n_samples, act_dim, lambda, mean_out_dev, stats_dev, stream);
}

int odg_mppi_reduce_groups(const float* cost_dev, const float* actions_dev, int horizon, int groups, int samples_per_group,
                           int act_dim, float lambda, float* mean_out_dev, float* stats_dev, void* stream) {
  if (!cost_dev || !actions_dev || !mean_out_dev || horizon < 1 || groups < 1 || samples_per_group < 1 ||
      samples_per_group > 12000 || act_dim < 1 || !(lambda > 0.f) || (long long)groups * samples_per_group > 0x7fffffff)
    return set_error(ODG_ERR_INVALID, "odg_mppi_reduce_groups: bad arguments (samples_per_group <= 12000)");
  // [S] weights in dynamic shared memory next to 8 KB of static reduction rows: above 48 KB in total the kernel
  // needs the opt-in limit (S > ~10000)
  const size_t smem = (size_t)samples_per_group * sizeof(float);
  CUDA_TRY(cudaFuncSetAttribute(k_mppi_reduce, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_mppi_reduce<<<groups, kRedThreads, smem, static_cast<cudaStream_t>(stream)>>>(
      cost_dev, actions_dev, horizon, samples_per_group, groups * samples_per_group, act_dim, lambda, mean_out_dev, stats_dev);
  CUDA_TRY(cudaGetLastError());
  return ODG_OK;
}

}  // extern "C"
