// odg_sim.cu — libodgsim: kernels + the C ABI declared in include/odg.h.  sm_100a only.
//
// Kernel map
//   k_step<NJL>   the fused environment step (odg_core.cuh: env_step). 4 lanes per environment,
//                 8 environments per warp. Model constants arrive as a __grid_constant__ kernel
//                 parameter (constant bank), per-leg constants and hull vertices are staged ONCE per
//                 persistent block into shared memory; per-env state is SoA in HBM and is read and
//                 written exactly once per env-step (all frame_skip substeps stay in registers).
//   k_reset<NJL>  reset_model for masked environments.
//   k_init        construction-time state.
//   k_*_state     layout transposes between the caller's [N][dim] tensors and the SoA state.
//
// There is no CPU path in this library: without a CUDA device odg_create fails with ODG_ERR_NO_DEVICE.
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <new>
#include <string>

#include "../../include/odg_mppi.h"
#include "odg_sim_internal.h"

namespace {

thread_local std::string g_err;
int fail(int code, const std::string& msg) { g_err = msg; return code; }
#define CUDA_TRY(expr)                                                                         \
  do { cudaError_t e_ = (expr);                                                                \
       if (e_ != cudaSuccess) return fail(ODG_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_)); } while (0)

using odg::DevConst; using odg::SimPtrs; using odg::StepArgs;
}  // namespace
namespace odg_internal { int set_error(int code, const std::string& msg) { return fail(code, msg); } }   // for odg_policy.cu
namespace {


#ifndef ODG_MIN_BLOCKS
#define ODG_MIN_BLOCKS 1
#endif
#ifndef ODG_MAX_BLOCK
#define ODG_MAX_BLOCK 128
#endif
template <int NJL, bool FAT>
__global__ void __launch_bounds__(ODG_MAX_BLOCK, ODG_MIN_BLOCKS) k_step(const __grid_constant__ DevConst C, const SimPtrs P, const StepArgs A,
                                              const __grid_constant__ odg::MppiArgs M,
                                              const float* __restrict__ g_lc, const float* __restrict__ g_gc,
                                              const float* __restrict__ g_vert, SmemLayout L, int lanes) {
  extern __shared__ __align__(16) float smem[];
  const float4* s_vert; const float* s_lc; const float* s_gc;
  stage_constants(smem, g_lc, g_gc, g_vert, L, &s_vert, &s_lc, &s_gc);
  // `lanes` = active lanes per warp (32, 16 or 8 -> 8, 4 or 2 environments per warp). Small batches leave most of
  // the GPU empty, so they run with fewer environments per warp: less divergence between the environments that
  // share a warp, and more warps to interleave per scheduler.
  const int leg = threadIdx.x & 3;
  const int lane = threadIdx.x & 31;
  // per-group reduction rows (odg_core.cuh: grp_sum28) follow the staged constants
  float* s_red = smem + L.vert_floats + L.lc_floats + L.gc_floats + (threadIdx.x >> 2) * odg::kRedGroup;
  if (lane >= lanes) return;
  const unsigned gm = 0xFu << (lane & 28);
  const int envs_per_warp = lanes >> 2;
  const int envs_per_block = (blockDim.x >> 5) * envs_per_warp;
  // Ordinary step: one env-step per environment. MPPI rollout (M.T > 0; odg_mppi_rollout): the SAME code walks a whole
  // horizon per environment — draw the step's action row, take the env-step, add minus the unclipped reward to the
  // sample's cost — so between the steps of a sample nothing waits on any other sample (no launch boundary, no grid-wide
  // barrier), and a rollout is bit-identical to the same action rows stepped one launch at a time (one call site of
  // env_step = one copy of its arithmetic). A sample that terminates pays once and only keeps drawing its action rows.
  const int horizon = M.T > 0 ? M.T : 1;
  const uint32_t iteration = (M.T > 0 && M.iteration_dev) ? *M.iteration_dev : M.iteration;
  for (int base = blockIdx.x * envs_per_block; base < P.N; base += gridDim.x * envs_per_block) {
    const int env = base + (threadIdx.x >> 5) * envs_per_warp + (lane >> 2);
    if (env >= P.N) continue;
    // MPPI groups, once per sample: env = g * S + s. Padding environments (env >= n) take the last group, so no mean
    // pointer goes past it; they draw no rows.
    const int g = M.T > 0 ? min(env, P.n - 1) / M.S : 0, s = env - g * M.S;
    float cost = 0.f;
    bool alive = true;
    for (int t = 0; t < horizon; t++) {
      const float* action = A.action;
      if (M.T > 0) {
        float* row = M.actions + (size_t)t * P.n * C.nu;
        if (leg == 0 && env < P.n) {
          const uint64_t key = ((((uint64_t)M.seed_hi) << 32) | M.seed_lo) + (uint64_t)g;
          odg::mppi_sample_row(M.mean + (size_t)g * M.mean_stride + (size_t)t * C.nu, M.sigma, s, C.nu, (uint32_t)key,
                               (uint32_t)(key >> 32), iteration, (uint32_t)t, row + (size_t)(env - s) * C.nu);
        }
        __syncwarp(gm);                            // the group's other lanes read the row lane 0 just wrote
        action = row;
      }
      if (alive) {
        const odg::StepResult r = odg::env_step<NJL, FAT>(C, s_lc, s_gc, s_vert, P, A, action, env, leg, gm, s_red);
        cost -= r.reward_unclipped;
        if (r.terminated && M.T > 0) { cost += M.term_cost; alive = false; }
      }
    }
    if (M.T > 0 && leg == 0 && env < P.n) M.cost[env] = cost;
  }
}

template <int NJL>
__global__ void __launch_bounds__(128) k_reset(const __grid_constant__ DevConst C, const SimPtrs P,
                                               const unsigned char* __restrict__ mask, float* obs,
                                               const float* __restrict__ g_lc) {
  extern __shared__ __align__(16) float smem[];
  for (int i = threadIdx.x; i < NJL * odg::LC_COUNT * 4; i += blockDim.x) smem[i] = g_lc[i];
  __syncthreads();
  const int leg = threadIdx.x & 3;
  const unsigned gm = 0xFu << (threadIdx.x & 28);
  const int env = blockIdx.x * (blockDim.x >> 2) + (threadIdx.x >> 2);
  if (env >= P.N) return;
  if (mask && env < P.n && !mask[env]) return;
  odg::env_reset<NJL>(C, smem, P, obs, env, leg, gm);
}

__global__ void k_init(const __grid_constant__ DevConst C, const SimPtrs P) {
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env < P.N) odg::env_init(C, P, env);
}

// dst[env][k] = src[k][env] (to_soa = false) or the reverse
__global__ void k_transpose(float* aos, float* soa, int n, int stride, int dim, bool to_soa) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)n * dim) return;
  const int env = (int)(i / dim), k = (int)(i % dim);
  if (to_soa) soa[(size_t)k * stride + env] = aos[i]; else aos[i] = soa[(size_t)k * stride + env];
}
__global__ void k_fill(float* p, long long n, float v) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}
template <typename T>
__global__ void k_copy(T* dst, const T* src, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = src[i];
}

// odg_mppi_broadcast: sample n of D <- robot first + n / S of R, every per-environment field env_step reads (SoA to SoA)
__global__ void k_mppi_broadcast(const SimPtrs D, const SimPtrs R, int first, int S, int nq, int nv, int nu) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= D.n) return;
  const int r = first + n / S;
  for (int k = 0; k < nq; k++) D.qpos[(size_t)k * D.N + n] = R.qpos[(size_t)k * R.N + r];
  for (int k = 0; k < nv; k++) {
    D.qvel[(size_t)k * D.N + n] = R.qvel[(size_t)k * R.N + r];
    D.warm[(size_t)k * D.N + n] = R.warm[(size_t)k * R.N + r];
  }
  for (int k = 0; k < nu; k++) D.last_action[(size_t)k * D.N + n] = R.last_action[(size_t)k * R.N + r];
  for (int k = 0; k < 3; k++) D.desvel[(size_t)k * D.N + n] = R.desvel[(size_t)k * R.N + r];
  D.step[n] = R.step[r]; D.gait_idx[n] = R.gait_idx[r]; D.gait_cnt[n] = R.gait_cnt[r]; D.fresh[n] = R.fresh[r];
}

}  // namespace


namespace {

typedef void (*StepKernel)(const DevConst, const SimPtrs, const StepArgs, const odg::MppiArgs, const float*, const float*, const float*, SmemLayout, int);
// `fat` = the instantiation that keeps more per-contact data in local memory (odg_core.cuh: substep<NJL, FAT>): chosen,
// like lockstep, from the batch size; results are bit-identical either way
StepKernel step_kernel_fn(const DevConst& C, bool fat) {
  if (C.njl == 2) return fat ? k_step<2, true> : k_step<2, false>;
  return fat ? k_step<3, true> : k_step<3, false>;
}
const void* step_kernel(const DevConst& C, bool fat) { return (const void*)step_kernel_fn(C, fat); }

int choose_launch(OdgSim* s) {
  // 4 lanes per env, persistent blocks (constants staged once per block). Shared memory per block = the staged constants
  // + one reduction area per 4-lane group of THIS block size: how much shared memory the resident blocks of an SM take
  // decides the carve-out and with it how much L1 is left for the kernel's local-memory traffic (per-contact records) —
  // at 65536 envs one carve-out step (32 KB of L1) is worth 25 % of the throughput.
  const void* kern = step_kernel(s->prep.C, false);
  auto smem_for = [&](int block) { return s->smem_const + (size_t)(block / 4) * odg::kRedGroup * sizeof(float); };
  CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_for(ODG_MAX_BLOCK)));
  CUDA_TRY(cudaFuncSetAttribute(step_kernel(s->prep.C, true), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_for(ODG_MAX_BLOCK)));
  // Measured on B200 (tools/tune_launch_shape.sh, tools/tune_4096.sh, tools/tune_fat.sh): 8 environments per warp; fewer
  // environments per warp or one-warp blocks lose more to instruction fetch than they gain in divergence.
  int lanes = 32;
  // tiny batches (MPPI: 1024 samples) leave most schedulers empty: 2 environments per warp, so 4x the warps share the
  // work and fewer environments wait on the slowest one of their warp (40.5 vs 46.6 ms per 1024 x 64 plan)
  if (s->P.N / 8 < s->num_sms) lanes = 8;
  if (s->cfg_lanes) lanes = s->cfg_lanes;
  const long long warps = ((long long)s->P.N * 4 + lanes - 1) / lanes;
  auto occupancy = [&](int block, int* occ) -> cudaError_t {
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(occ, kern, block, smem_for(block));
    if (*occ < 1) *occ = 1;
    return e;
  };
  // is the batch more than half a wave of two-warp blocks? (measured: lockstep and the lean instantiation pay from ~8192 envs up)
  int occ64 = 1;
  CUDA_TRY(occupancy(64, &occ64));
  const bool deep = 2 * ((warps + 1) / 2) > (long long)s->num_sms * occ64;
  int block = 64;
  // a small batch that 64-thread blocks would spread unevenly (more blocks than SMs, fewer than two per SM) but 128-thread
  // blocks place one per SM — one warp per scheduler everywhere — takes the larger block: 4096 envs = 128 blocks, +1.5 %
  if (lanes == 32 && (warps + 1) / 2 > s->num_sms && (warps + 3) / 4 <= s->num_sms) block = 128;
  // lockstep: 0 = free-running warps, 1 = all warps of a block take Newton iterations together, 2 = PAIRS of warps inside
  // 128-thread blocks (named barriers): the fastest pairing with the constants staged once for two pairs. Deep batches
  // get 2, shallow ones 0.
  int lockstep = deep ? (lanes == 32 ? 2 : 1) : 0;
  // 3-joint legs (Go1: 17 k instructions, instruction fetch is its top stall even at one warp per scheduler): pairs whenever
  // warps are whole (measured, tools/tune_go1.sh: +11 % at 4096 envs, +10 % at 16384, +12 % at 65536 together with FAT)
  if (s->prep.C.njl == 3 && lanes == 32) lockstep = 2;
  if (s->cfg_lockstep >= 0) lockstep = s->cfg_lockstep;
  if (lockstep == 2 && !s->cfg_block) block = 128;
  if (s->cfg_block) block = s->cfg_block;
  if (lockstep == 2 && (block != 128 || lanes != 32)) lockstep = 1;      // pairs need whole warps in 128-thread blocks
  int occ = 1;
  CUDA_TRY(occupancy(block, &occ));
  const long long wpb = block / 32, need = (warps + wpb - 1) / wpb, cap = (long long)s->num_sms * occ;
  s->step_lanes = lanes; s->step_block = block; s->smem_step = smem_for(block);
  s->prep.C.lockstep = lockstep;
  // The instantiation that keeps per-contact Jacobian columns and line-search coefficients in local memory: at every batch
  // size. Mid-round it lost 18 % at 65536 envs (its per-contact words did not fit the L1 of 8 resident warps); with 16-byte
  // records, the cone constants in their spare words and shared memory sized per block it wins there too (measured at the
  // end of round 2, tools/tune_fat2.sh, with lockstep pairs: +12 % at 8192 / 32768 envs, +11 % at 16384, +10 % at 65536).
  // The lean instantiation stays selectable (OdgEnvConfig::launch_fat = 0): the GPU suite holds both to the same bits.
  s->step_fat = 1;
  if (s->cfg_fat >= 0) s->step_fat = s->cfg_fat ? 1 : 0;
  s->step_grid = (int)(need < cap ? need : cap);
  return ODG_OK;
}

int launch_step(OdgSim* s, const StepArgs& A, cudaStream_t st) {
  odg::MppiArgs M;
  std::memset(&M, 0, sizeof(M));
  step_kernel_fn(s->prep.C, s->step_fat != 0)<<<s->step_grid, s->step_block, s->smem_step, st>>>(s->prep.C, s->P, A, M, s->d_lc, s->d_gc, s->d_vert, s->L, s->step_lanes);
  s->launches++;
  CUDA_TRY(cudaGetLastError());
  return ODG_OK;
}

void fill_args(StepArgs* A, const float* action, float* obs, float* reward, uint8_t* term, uint8_t* trunc,
               const OdgInfoPtrs* info, int mode) {
  std::memset(A, 0, sizeof(*A));
  A->action = action; A->obs = obs; A->reward = reward; A->terminated = term; A->truncated = trunc; A->mode = mode;
  if (info) {
    A->want_info = 1;
    A->x_position = info->x_position; A->y_position = info->y_position; A->distance = info->distance_from_origin;
    A->paw_forces = info->paw_contact_forces; A->patterns_matches = info->patterns_matches;
    A->lin_vel_reward = info->linear_vel_tracking_reward; A->reward_ctrl = info->reward_ctrl;
    A->terminal_obs = info->terminal_obs; A->paws_in_ground = info->paws_in_ground; A->gait_reward = info->gait_reward;
    A->qacc = info->qacc; A->ncon = info->ncon; A->fn_sum = info->contact_normal_force; A->solver_iters = info->solver_iters; A->ls_evals = info->ls_evals;
    A->reward_raw = info->reward_unclipped;
    A->cfrc_ext = info->cfrc_ext; A->task_terms = info->task_terms;
  }
}

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

// odg_mppi_rollout (groups = 1) and odg_mppi_rollout_groups: one launch of the step kernel in MPPI mode
int mppi_rollout(OdgSim* s, int groups, const float* mean_dev, float sigma, int horizon, uint64_t seed, uint32_t iteration,
                 const uint32_t* iteration_dev, float termination_cost, float* actions_dev, float* cost_dev, cudaStream_t st,
                 const char* who) {
  if (!s || !mean_dev || !actions_dev || !cost_dev || horizon < 1 || !(sigma >= 0.f) || groups < 1)
    return fail(ODG_ERR_INVALID, std::string(who) + ": bad arguments");
  if (s->P.n % groups) return fail(ODG_ERR_INVALID, std::string(who) + ": the handle's environments are not a whole number of groups");
  if (s->prep.C.auto_reset) return fail(ODG_ERR_INVALID, std::string(who) + ": the handle must be created with auto_reset = 0");
  DeviceGuard guard(s->device);
  DevConst C = s->prep.C;
  C.lockstep = 0;                                  // samples leave the horizon loop at different times: no block barriers
  odg::MppiArgs M;
  M.T = horizon; M.S = s->P.n / groups; M.mean_stride = horizon * C.nu; M.sigma = sigma; M.term_cost = termination_cost;
  M.seed_lo = (uint32_t)seed; M.seed_hi = (uint32_t)(seed >> 32); M.iteration = iteration; M.iteration_dev = iteration_dev;
  M.mean = mean_dev; M.actions = actions_dev; M.cost = cost_dev;
  StepArgs A;
  fill_args(&A, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 0);
  // every sample gets its own 4-lane group for the whole horizon: one tile per block, never a second wave
  const int epb = (s->step_block / 32) * (s->step_lanes / 4);
  const int grid = (s->P.N + epb - 1) / epb;
  step_kernel_fn(C, s->step_fat != 0)<<<grid, s->step_block, s->smem_step, st>>>(C, s->P, A, M, s->d_lc, s->d_gc, s->d_vert, s->L, s->step_lanes);
  s->launches++;
  CUDA_TRY(cudaGetLastError());
  return ODG_OK;
}

}  // namespace

extern "C" {

void odg_default_config(OdgEnvConfig* cfg) { if (cfg) odg::default_config(cfg); }
const char* odg_last_error(void) { return g_err.c_str(); }
const char* odg_version(void) { return "odgsim 0.1 sm_100a"; }

int odg_create(const OdgModel* model, const OdgEnvConfig* cfg_in, int num_envs, int device, uint64_t seed, OdgSim** out) {
  if (!model || !out || num_envs < 1) return fail(ODG_ERR_INVALID, "odg_create: bad arguments");
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(ODG_ERR_NO_DEVICE, "no CUDA device: libodgsim has no CPU fallback");
  if (device < 0 || device >= ndev) return fail(ODG_ERR_INVALID, "odg_create: device out of range");
  OdgEnvConfig cfg;
  if (cfg_in) cfg = *cfg_in; else odg::default_config(&cfg);
  OdgSim* s = new (std::nothrow) OdgSim();
  if (!s) return fail(ODG_ERR_ALLOC, "out of host memory");
  std::string why = odg::prepare(*model, cfg, seed, &s->prep);
  if (!why.empty()) { delete s; return fail(ODG_ERR_INVALID, "odg_create: " + why); }
  DeviceGuard guard(device);
  s->device = device; s->N = num_envs;
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  s->num_sms = prop.multiProcessorCount;
  const DevConst& C = s->prep.C;
  const size_t N = ((size_t)num_envs + 63) / 64 * 64;      // stride: whole blocks of up to 64 environments
  // one slab: qpos, qvel, warm, last_action, desvel (float) | step, gait_idx, gait_cnt, episode (i32) | fresh (u8)
  const size_t nfloat = (size_t)(C.nq + 2 * C.nv + C.nu + 3) * N, nint = 5 * N;
  const size_t bytes = nfloat * 4 + nint * 4 + N;
  if (cudaMalloc(&s->d_state, bytes) != cudaSuccess) { delete s; return fail(ODG_ERR_ALLOC, "cudaMalloc(state) failed"); }
  float* f = static_cast<float*>(s->d_state);
  s->P.N = (int)N; s->P.n = num_envs;
  s->P.qpos = f; f += (size_t)C.nq * N;
  s->P.qvel = f; f += (size_t)C.nv * N;
  s->P.warm = f; f += (size_t)C.nv * N;
  s->P.last_action = f; f += (size_t)C.nu * N;
  s->P.desvel = f; f += 3 * N;
  int* ip = reinterpret_cast<int*>(f);
  s->P.step = ip; s->P.gait_idx = ip + N; s->P.gait_cnt = ip + 2 * N; s->P.episode = reinterpret_cast<unsigned*>(ip + 3 * N);
  s->P.work = ip + 4 * N;
  s->P.fresh = reinterpret_cast<unsigned char*>(ip + 5 * N);
  auto upload = [&](float** dst, const std::vector<float>& v) -> cudaError_t {
    cudaError_t e = cudaMalloc(dst, v.size() * sizeof(float));
    if (e != cudaSuccess) return e;
    return cudaMemcpy(*dst, v.data(), v.size() * sizeof(float), cudaMemcpyHostToDevice);
  };
  if (upload(&s->d_lc, s->prep.lc) != cudaSuccess || upload(&s->d_gc, s->prep.gc) != cudaSuccess ||
      upload(&s->d_vert, s->prep.vert) != cudaSuccess) { odg_destroy(s); return fail(ODG_ERR_ALLOC, "constant upload failed"); }
  s->L.lc_floats = (int)s->prep.lc.size(); s->L.gc_floats = (int)s->prep.gc.size(); s->L.vert_floats = (int)s->prep.vert.size();
  s->smem_const = (size_t)(s->L.lc_floats + s->L.gc_floats + s->L.vert_floats) * sizeof(float);
  if ((cfg.launch_lanes != 0 && cfg.launch_lanes != 4 && cfg.launch_lanes != 8 && cfg.launch_lanes != 16 && cfg.launch_lanes != 32) ||
      (cfg.launch_block != 0 && cfg.launch_block != 32 && cfg.launch_block != 64 && cfg.launch_block != 128 &&
       !(cfg.launch_block == 256 && ODG_MAX_BLOCK >= 256)) || cfg.launch_lockstep < -1 || cfg.launch_lockstep > 2 ||
      cfg.launch_fat < -1 || cfg.launch_fat > 1) {
    odg_destroy(s); return fail(ODG_ERR_INVALID, "odg_create: bad launch_lanes / launch_block / launch_lockstep / launch_fat");
  }
  s->cfg_lanes = cfg.launch_lanes; s->cfg_block = cfg.launch_block; s->cfg_lockstep = cfg.launch_lockstep; s->cfg_fat = cfg.launch_fat;
  CUDA_TRY(cudaMemset(s->P.work, 0, N * sizeof(int)));
  int rc = choose_launch(s);
  if (rc != ODG_OK) { odg_destroy(s); return rc; }
  k_init<<<(unsigned)((N + 127) / 128), 128>>>(C, s->P);
  s->launches++;
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) { odg_destroy(s); return fail(ODG_ERR_CUDA, std::string("k_init: ") + cudaGetErrorString(e)); }
  *out = s;
  return ODG_OK;
}

void odg_destroy(OdgSim* s) {
  if (!s) return;
  DeviceGuard guard(s->device);
  cudaFree(s->d_state); cudaFree(s->d_lc); cudaFree(s->d_gc); cudaFree(s->d_vert);
  delete s;
}

int odg_num_envs(const OdgSim* s) { return s ? s->N : 0; }
int odg_obs_dim(const OdgSim* s) { return s ? s->prep.C.obs_dim : 0; }
int odg_act_dim(const OdgSim* s) { return s ? s->prep.C.nu : 0; }
int odg_nq(const OdgSim* s) { return s ? s->prep.C.nq : 0; }
int odg_nv(const OdgSim* s) { return s ? s->prep.C.nv : 0; }
long long odg_launch_count(const OdgSim* s) { return s ? s->launches : 0; }
int odg_set_frame_skip(OdgSim* s, int frame_skip) {
  if (!s || frame_skip < 1) return fail(ODG_ERR_INVALID, "odg_set_frame_skip: bad arguments");
  s->prep.C.frame_skip = frame_skip;
  return ODG_OK;
}

int odg_reset(OdgSim* s, const uint8_t* mask_dev, float* obs_dev, void* stream) {
  if (!s) return fail(ODG_ERR_INVALID, "odg_reset: null handle");
  DeviceGuard guard(s->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int block = 128, grid = (s->P.N * 4 + block - 1) / block;
  const size_t smem = (size_t)s->prep.C.njl * odg::LC_COUNT * 4 * sizeof(float);
  if (s->prep.C.njl == 2) k_reset<2><<<grid, block, smem, st>>>(s->prep.C, s->P, mask_dev, obs_dev, s->d_lc);
  else k_reset<3><<<grid, block, smem, st>>>(s->prep.C, s->P, mask_dev, obs_dev, s->d_lc);
  s->launches++;
  CUDA_TRY(cudaGetLastError());
  return ODG_OK;
}

int odg_step(OdgSim* s, const float* action_dev, float* obs_dev, float* reward_dev, uint8_t* terminated_dev,
             uint8_t* truncated_dev, const OdgInfoPtrs* info, void* stream) {
  if (!s || !action_dev) return fail(ODG_ERR_INVALID, "odg_step: null handle or action");
  DeviceGuard guard(s->device);
  StepArgs A;
  fill_args(&A, action_dev, obs_dev, reward_dev, terminated_dev, truncated_dev, info, 0);
  return launch_step(s, A, static_cast<cudaStream_t>(stream));
}

int odg_step_host(OdgSim* s, const float* action_host, float* action_pinned, float* action_dev, float* obs_dev,
                  float* reward_dev, uint8_t* terminated_dev, uint8_t* truncated_dev, const OdgInfoPtrs* info,
                  const void* out_dev, void* out_host, size_t out_bytes, void* stream) {
  if (!s || !action_host || !action_dev) return fail(ODG_ERR_INVALID, "odg_step_host: null handle or action");
  if ((out_dev == nullptr) != (out_host == nullptr)) return fail(ODG_ERR_INVALID, "odg_step_host: out_dev and out_host go together");
  DeviceGuard guard(s->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t abytes = (size_t)s->N * s->prep.C.nu * sizeof(float);
  const float* src = action_host;
  if (action_pinned && action_pinned != action_host) { std::memcpy(action_pinned, action_host, abytes); src = action_pinned; }
  // action_dev == the page-locked source: the kernel reads the actions in place over PCIe (unified addressing: page-locked
  // memory has the same address on the device), which takes the copy engine's launch latency off the step's critical path
  if (action_dev != src) CUDA_TRY(cudaMemcpyAsync(action_dev, src, abytes, cudaMemcpyHostToDevice, st));
  StepArgs A;
  fill_args(&A, action_dev, obs_dev, reward_dev, terminated_dev, truncated_dev, info, 0);
  int rc = launch_step(s, A, st);
  if (rc != ODG_OK) return rc;
  if (out_dev && out_bytes) CUDA_TRY(cudaMemcpyAsync(out_host, out_dev, out_bytes, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  return ODG_OK;
}

int odg_mppi_rollout(OdgSim* s, const float* mean_dev, float sigma, int horizon, uint64_t seed, uint32_t iteration,
                     const uint32_t* iteration_dev, float termination_cost, float* actions_dev, float* cost_dev, void* stream) {
  return mppi_rollout(s, 1, mean_dev, sigma, horizon, seed, iteration, iteration_dev, termination_cost, actions_dev, cost_dev,
                      static_cast<cudaStream_t>(stream), "odg_mppi_rollout");
}

int odg_mppi_rollout_groups(OdgSim* s, int groups, const float* mean_dev, float sigma, int horizon, uint64_t seed,
                            uint32_t iteration, const uint32_t* iteration_dev, float termination_cost, float* actions_dev,
                            float* cost_dev, void* stream) {
  return mppi_rollout(s, groups, mean_dev, sigma, horizon, seed, iteration, iteration_dev, termination_cost, actions_dev,
                      cost_dev, static_cast<cudaStream_t>(stream), "odg_mppi_rollout_groups");
}

int odg_mppi_broadcast(OdgSim* samples, const OdgSim* robots, int first_robot, int groups, void* stream) {
  if (!samples || !robots) return fail(ODG_ERR_INVALID, "odg_mppi_broadcast: null handle");
  const DevConst& D = samples->prep.C; const DevConst& R = robots->prep.C;
  if (samples->device != robots->device) return fail(ODG_ERR_INVALID, "odg_mppi_broadcast: the handles are on different devices");
  if (D.nq != R.nq || D.nv != R.nv || D.nu != R.nu || D.task != R.task)
    return fail(ODG_ERR_INVALID, "odg_mppi_broadcast: the handles differ in nq / nv / nu / task");
  if (groups < 1 || first_robot < 0 || first_robot > robots->P.n - groups)
    return fail(ODG_ERR_INVALID, "odg_mppi_broadcast: robots [first_robot, first_robot + groups) out of range");
  if (samples->P.n % groups) return fail(ODG_ERR_INVALID, "odg_mppi_broadcast: the samples are not a whole number of groups");
  if (D.auto_reset) return fail(ODG_ERR_INVALID, "odg_mppi_broadcast: the samples handle must be created with auto_reset = 0");
  DeviceGuard guard(samples->device);
  k_mppi_broadcast<<<(samples->P.n + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      samples->P, robots->P, first_robot, samples->P.n / groups, D.nq, D.nv, D.nu);
  samples->launches++;
  CUDA_TRY(cudaGetLastError());
  return ODG_OK;
}

int odg_evaluate(OdgSim* s, const float* ctrl_dev, float* obs_dev, float* reward_dev, uint8_t* terminated_dev,
                 uint8_t* truncated_dev, const OdgInfoPtrs* info, void* stream) {
  if (!s || !ctrl_dev) return fail(ODG_ERR_INVALID, "odg_evaluate: null handle or ctrl");
  DeviceGuard guard(s->device);
  StepArgs A;
  fill_args(&A, ctrl_dev, obs_dev, reward_dev, terminated_dev, truncated_dev, info, 1);
  return launch_step(s, A, static_cast<cudaStream_t>(stream));
}

static int transpose(OdgSim* s, float* aos, float* soa, int dim, bool to_soa, cudaStream_t st) {
  const long long n = (long long)s->N * dim;
  k_transpose<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(aos, soa, s->N, s->P.N, dim, to_soa);
  s->launches++;
  CUDA_TRY(cudaGetLastError());
  return ODG_OK;
}

int odg_get_state(OdgSim* s, float* qpos_dev, float* qvel_dev, void* stream) {
  if (!s) return fail(ODG_ERR_INVALID, "odg_get_state: null handle");
  DeviceGuard guard(s->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int rc = ODG_OK;
  if (qpos_dev) rc = transpose(s, qpos_dev, s->P.qpos, s->prep.C.nq, false, st);
  if (rc == ODG_OK && qvel_dev) rc = transpose(s, qvel_dev, s->P.qvel, s->prep.C.nv, false, st);
  return rc;
}

int odg_set_state(OdgSim* s, const float* qpos_dev, const float* qvel_dev, const float* warm_dev, void* stream) {
  if (!s) return fail(ODG_ERR_INVALID, "odg_set_state: null handle");
  DeviceGuard guard(s->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int rc = ODG_OK;
  if (qpos_dev) rc = transpose(s, const_cast<float*>(qpos_dev), s->P.qpos, s->prep.C.nq, true, st);
  if (rc == ODG_OK && qvel_dev) rc = transpose(s, const_cast<float*>(qvel_dev), s->P.qvel, s->prep.C.nv, true, st);
  if (rc != ODG_OK) return rc;
  if (warm_dev) return transpose(s, const_cast<float*>(warm_dev), s->P.warm, s->prep.C.nv, true, st);
  const long long n = (long long)s->P.N * s->prep.C.nv;
  k_fill<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(s->P.warm, n, 0.f);
  s->launches++;
  CUDA_TRY(cudaGetLastError());
  return ODG_OK;
}

int odg_get_env_state(OdgSim* s, int32_t* step, int32_t* gidx, int32_t* gcnt, float* last_action, float* desvel,
                      uint8_t* fresh, void* stream) {
  if (!s) return fail(ODG_ERR_INVALID, "odg_get_env_state: null handle");
  DeviceGuard guard(s->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t N = (size_t)s->N;
  if (step) CUDA_TRY(cudaMemcpyAsync(step, s->P.step, N * 4, cudaMemcpyDeviceToDevice, st));
  if (gidx) CUDA_TRY(cudaMemcpyAsync(gidx, s->P.gait_idx, N * 4, cudaMemcpyDeviceToDevice, st));
  if (gcnt) CUDA_TRY(cudaMemcpyAsync(gcnt, s->P.gait_cnt, N * 4, cudaMemcpyDeviceToDevice, st));
  if (fresh) CUDA_TRY(cudaMemcpyAsync(fresh, s->P.fresh, N, cudaMemcpyDeviceToDevice, st));
  int rc = ODG_OK;
  if (last_action) rc = transpose(s, last_action, s->P.last_action, s->prep.C.nu, false, st);
  if (rc == ODG_OK && desvel) rc = transpose(s, desvel, s->P.desvel, 3, false, st);
  return rc;
}

int odg_set_env_state(OdgSim* s, const int32_t* step, const int32_t* gidx, const int32_t* gcnt, const float* last_action,
                      const float* desvel, const uint8_t* fresh, void* stream) {
  if (!s) return fail(ODG_ERR_INVALID, "odg_set_env_state: null handle");
  DeviceGuard guard(s->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t N = (size_t)s->N;
  if (step) CUDA_TRY(cudaMemcpyAsync(s->P.step, step, N * 4, cudaMemcpyDeviceToDevice, st));
  if (gidx) CUDA_TRY(cudaMemcpyAsync(s->P.gait_idx, gidx, N * 4, cudaMemcpyDeviceToDevice, st));
  if (gcnt) CUDA_TRY(cudaMemcpyAsync(s->P.gait_cnt, gcnt, N * 4, cudaMemcpyDeviceToDevice, st));
  if (fresh) CUDA_TRY(cudaMemcpyAsync(s->P.fresh, fresh, N, cudaMemcpyDeviceToDevice, st));
  int rc = ODG_OK;
  if (last_action) rc = transpose(s, const_cast<float*>(last_action), s->P.last_action, s->prep.C.nu, true, st);
  if (rc == ODG_OK && desvel) rc = transpose(s, const_cast<float*>(desvel), s->P.desvel, 3, true, st);
  return rc;
}

}  // extern "C"
