// odg_policy.cu — the rollout side of libodgsim (C ABI: include/odg_policy.h).  sm_100a only.
//
//   k_mlp        ActorCritic forward for 128 environments per CTA on the 5th-generation tensor cores:
//                obs -> Linear(S,512)-tanh -> Linear(512,256)-tanh -> Linear(256,A)-tanh   (actor)
//                    -> Linear(S,512)-tanh -> Linear(512,256)-tanh -> Linear(256,1)        (critic)
//                (reference: sim2real/train.py:132-149) fused with Normal sampling and log-prob (:542-543).
//                bf16 operands in shared memory (canonical K-major core-matrix layout, no swizzle), fp32
//                accumulators in TMEM (tcgen05.mma issued by one thread), weights streamed chunk by chunk with
//                1-D bulk async copies (TMA engine, mbarrier complete_tx) double-buffered against the MMAs,
//                activations never leave the SM: the 512- and 256-wide hidden layers go TMEM -> registers
//                (tcgen05.ld) -> bias+tanh -> bf16 -> shared memory as the next layer's A operand.
//   k_pack       fp32 torch state_dict weights -> bf16 operand chunks in that canonical layout.
//   k_gae*       GAE scan + deterministic advantage statistics; k_adv_norm: normalisation.
#include <cuda_runtime.h>
#include <cuda_bf16.h>

#include <cstdio>
#include <cstring>
#include <new>
#include <string>

#include "../../include/odg.h"
#include "../../include/odg_policy.h"
#include "odg_core.cuh"      // philox4x32 / u01 (same counter-based RNG as the step kernel and the oracle)

namespace odg_internal { int set_error(int code, const std::string& msg); }

namespace {

using odg_internal::set_error;
#define CUDA_TRY(expr)                                                                         \
  do { cudaError_t e_ = (expr);                                                                \
       if (e_ != cudaSuccess) return set_error(ODG_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_)); } while (0)

constexpr int kH1 = ODG_POLICY_H1, kH2 = ODG_POLICY_H2;
constexpr int kM = 128;                  // environments (rows) per CTA = UMMA M
constexpr int kNOut = 16;                // output layer padded to the smallest UMMA N
constexpr int kK2Chunk = 32;             // columns of W2 streamed per chunk (2 MMAs of K = 16)
constexpr int kL1Rows = 128;             // rows of W1 per chunk (a quarter of the layer: N = 128 per MMA)
constexpr int kL1Chunks = kH1 / kL1Rows, kL2Chunks = kH1 / kK2Chunk;
constexpr int kRingChunks = kL1Chunks + kL2Chunks;      // chunks of a network that stream through the stage ring (W1, W2)
constexpr int kNumChunks = kRingChunks + 1;             // + W3  (= 21 packed chunks per network)
constexpr int kStages = 4;               // weight stages in flight (16 KB each)
constexpr int kCluster = 2;              // CTAs per cluster: every weight chunk is fetched from L2 once per cluster and multicast
constexpr uint32_t kStreamSample = 0x53414d50u;      // Philox stream id "SAMP"
// thread roles: warps 0-7 = two epilogue warpgroups (TMEM lane quarter = warp & 3, column half = warp >> 2),
// warp 8 = MMA issuer (one elected thread), warp 9 = weight producer (one elected thread, bulk async copies)
constexpr int kEpiThreads = 256, kThreads = kEpiThreads + 64;
constexpr int kIssuerTid = kEpiThreads, kProducerTid = kEpiThreads + 32;

// ---- shared memory map (bytes)
constexpr int kA0Bytes = kM * ODG_POLICY_MAX_STATE * 2;       // 16 KB  obs tile
constexpr int kA1Bytes = kM * kH1 * 2;                         // 128 KB hidden 1 (hidden 2 aliases its first half)
constexpr int kWBufBytes = 16384;                              // one weight stage: 128 x 64 (W1), 256 x 32 (W2), 16 x 256 (W3)
constexpr int kW3Bytes = kNOut * kH2 * 2;                      // 8 KB  output-layer weights: their own buffer, outside the ring
constexpr int kOffA0 = 0, kOffA1 = kOffA0 + kA0Bytes, kOffW = kOffA1 + kA1Bytes, kOffW3 = kOffW + kStages * kWBufBytes;
constexpr int kOffBar = kOffW3 + kW3Bytes;
constexpr int kBiasFloats = kH1 + kH2 + kNOut;                  // per network: b1 | b2 | b3
constexpr int kOffBias = kOffBar + 256;
constexpr int kSmemBytes = kOffBias + 2 * kBiasFloats * 4;

// byte offset of element (r, k) of an operand tile with kc columns in the canonical K-major no-swizzle layout:
// 8x8 core matrices (8 rows x 16 bytes, contiguous 128 B); K-adjacent core matrices are 128 B apart (LBO),
// 8-row groups are (kc/8)*128 B apart (SBO).
__host__ __device__ inline int canon_off(int r, int k, int kc) {
  return (r >> 3) * ((kc >> 3) * 128) + (k >> 3) * 128 + (r & 7) * 16 + (k & 7) * 2;
}

struct ChunkDesc { int rows, kc; int layer, row0, k0; };      // layer 0..2; rows x kc block of W_layer at (row0, k0)
__host__ __device__ inline ChunkDesc chunk_desc(int c, int K0p) {
  ChunkDesc d;
  if (c < kL1Chunks) { d.rows = kL1Rows; d.kc = K0p; d.layer = 0; d.row0 = c * kL1Rows; d.k0 = 0; }
  else if (c < kL1Chunks + kL2Chunks) { d.rows = 256; d.kc = kK2Chunk; d.layer = 1; d.row0 = 0; d.k0 = (c - kL1Chunks) * kK2Chunk; }
  else { d.rows = kNOut; d.kc = kH2; d.layer = 2; d.row0 = 0; d.k0 = 0; }
  return d;
}
__host__ __device__ inline int chunk_bytes(int c, int K0p) { ChunkDesc d = chunk_desc(c, K0p); return d.rows * d.kc * 2; }
__host__ __device__ inline int chunk_offset(int c, int K0p) { int o = 0; for (int i = 0; i < c; i++) o += chunk_bytes(i, K0p); return o; }

// ---------------------------------------------------------------------------------------------- PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* b, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(b)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* b, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* b) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_u32(b)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* b, uint32_t parity) {
  uint32_t ok;
  asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
               : "=r"(ok) : "r"(smem_u32(b)), "r"(parity) : "memory");
  return ok != 0;
}
// bounded wait: a barrier that never completes is a bug; trap (kernel error) instead of hanging the GPU
__device__ __forceinline__ void mbar_wait(uint64_t* b, uint32_t parity) {
  const long long t0 = clock64();
  while (!mbar_try_wait(b, parity)) if (clock64() - t0 > 4000000000ll) __trap();
}
// the same copy delivered to the same shared-memory offset (data and mbarrier) of every CTA of the cluster in `mask`
__device__ __forceinline__ void bulk_g2s_multicast(void* dst, const void* src, uint32_t bytes, uint64_t* bar, uint16_t mask) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1], %2, [%3], %4;"
               :: "r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)), "h"(mask) : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  // tcgen05 shared-memory matrix descriptor: start>>4 [0,14), LBO>>4 [16,30), SBO>>4 [32,46), version=1 [46,48),
  // base_offset 0, layout_type SWIZZLE_NONE (0) [61,64)
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | ((uint64_t)1 << 46);
}
__host__ __device__ constexpr uint32_t make_idesc(int M, int N) {
  // kind::f16 instruction descriptor: D = F32 [4,6)=1, A = BF16 [7,10)=1, B = BF16 [10,13)=1, A and B K-major,
  // N>>3 [17,23), M>>4 [24,29)
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile("{\n .reg .pred p;\n setp.ne.b32 p, %4, 0;\n tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}\n"
               :: "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(smem_u32(bar)) : "memory");
}
// arrive on the mbarrier at the same offset in every CTA of the cluster in `mask` once the MMAs issued so far retire
__device__ __forceinline__ void umma_commit_multicast(uint64_t* bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               :: "r"(smem_u32(bar)), "h"(mask) : "memory");
}
__device__ __forceinline__ void tmem_ld32_nowait(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
               "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
               "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                 "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
                 "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
                 "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
               : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 "
               "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                 "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
               : "r"(taddr) : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ float tanh_fast(float x) { float y; asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}

#ifdef ODG_MLP_TIMING            // clock64 stamps of CTA 0 (tools/mlp_time.py): [0,16) epilogue thread 0, [16,32) issuer, [32,40) producer
__device__ long long g_mlp_t[64];
#define MLP_STAMP(i) do { if (blockIdx.x == 0) g_mlp_t[i] = clock64(); } while (0)
#else
#define MLP_STAMP(i) do { } while (0)
#endif

struct MlpParams {
  const float* obs; int n, S, A, K0p;
  const uint8_t* wpack[2];     // actor / critic operand chunks (bf16, canonical layout, chunk after chunk)
  const float* bias[2];        // b1[512] | b2[256] | b3[16]
  const float* log_std;
  float* mean; float* value; float* action; float* logp;
  uint32_t seed_lo, seed_hi, step; const uint32_t* step_base; int first_row;
};

// obs tile -> bf16 A0 (rows past the batch and columns past S are zero): the 256 epilogue threads, two per row
__device__ __forceinline__ void load_obs_tile(const MlpParams& P, int K0p, uint8_t* sA0, int tid) {
  if (tid >= kEpiThreads) return;
  const int r = tid & (kM - 1), g = blockIdx.x * kM + r;
  const float* o = P.obs + (size_t)g * P.S;
  for (int k8 = (tid >> 7) * 8; k8 < K0p; k8 += 16) {
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
      const int k = k8 + 2 * i;
      float x0 = (g < P.n && k < P.S) ? o[k] : 0.f;
      float x1 = (g < P.n && k + 1 < P.S) ? o[k + 1] : 0.f;
      w[i] = pack_bf16(x0, x1);
    }
    *reinterpret_cast<uint4*>(sA0 + canon_off(r, k8, K0p)) = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

// Normal(mean, exp(log_std)) of row `grow`: sample + summed log-prob (sim2real/train.py:542-543). Philox4x32-10 keyed by
// (seed, first_row + grow, step + *step_base, block of 4 action dims, "SAMP"), Box-Muller; shared by both forward kernels,
// so that the same key draws the same noise whatever the hidden widths.
__device__ __forceinline__ void sample_row(const MlpParams& P, int grow, const float (&outv)[kNOut]) {
  const uint32_t step_ctr = P.step + (P.step_base ? __ldg(P.step_base) : 0u);
  float lp = 0.f;
#pragma unroll
  for (int blk = 0; blk < kNOut / 4; blk++) {
    if (blk * 4 >= P.A) break;
    uint32_t r[4];
    odg::philox4x32(P.seed_lo, P.seed_hi, (uint32_t)(P.first_row + grow), step_ctr, (uint32_t)blk, kStreamSample, r);
#pragma unroll
    for (int pr = 0; pr < 2; pr++) {                                  // Box-Muller: 2 uniforms -> 2 normals
      const float u1 = ((float)(r[2 * pr] >> 8) + 1.0f) * 5.9604644775390625e-08f;     // (0, 1]
      const float u2 = odg::u01(r[2 * pr + 1]);
      const float rad = sqrtf(-2.0f * logf(u1));
      float sn, cs; sincosf(6.283185307179586f * u2, &sn, &cs);
      const float e[2] = { rad * cs, rad * sn };
#pragma unroll
      for (int q = 0; q < 2; q++) {
        const int a = blk * 4 + pr * 2 + q;
        if (a < P.A) {
          const float ls = __ldg(P.log_std + a);
          if (P.mean) P.mean[(size_t)grow * P.A + a] = outv[a];
          if (P.action) P.action[(size_t)grow * P.A + a] = outv[a] + expf(ls) * e[q];
          lp += -0.5f * e[q] * e[q] - ls - 0.9189385332046727f;
        }
      }
    }
  }
  if (P.logp) P.logp[grow] = lp;
}

// hidden-layer epilogue of one thread: D[row][c0 .. c0 + ncols) (TMEM, fp32) + bias -> tanh -> bf16 -> A operand tile
// with `kc_out` columns, written at columns [kofs + c0, ...). Two 32-column TMEM loads are in flight at a time.
__device__ __forceinline__ void epilogue_hidden(uint32_t taddr_row, int c0, int ncols, const float* __restrict__ bias,
                                                uint8_t* a_out, int kc_out, int kofs, int row) {
  for (int cb = c0; cb < c0 + ncols; cb += 64) {
    uint32_t va[32], vb[32];
    tmem_ld32_nowait(taddr_row + cb, va);
    tmem_ld32_nowait(taddr_row + cb + 32, vb);
    tmem_ld_wait();
#pragma unroll
    for (int half = 0; half < 2; half++) {
#pragma unroll
      for (int g = 0; g < 4; g++) {
        uint32_t w[4];
#pragma unroll
        for (int i = 0; i < 4; i++) {
          const int col = cb + half * 32 + g * 8 + i * 2;
          const uint32_t r0 = half ? vb[g * 8 + i * 2] : va[g * 8 + i * 2], r1 = half ? vb[g * 8 + i * 2 + 1] : va[g * 8 + i * 2 + 1];
          w[i] = pack_bf16(tanh_fast(__uint_as_float(r0) + bias[col]), tanh_fast(__uint_as_float(r1) + bias[col + 1]));
        }
        *reinterpret_cast<uint4*>(a_out + canon_off(row, kofs + cb + half * 32 + g * 8, kc_out)) = make_uint4(w[0], w[1], w[2], w[3]);
      }
    }
  }
}

// Warp-specialised forward. Per network the work is four accumulator stages, alternating between the two halves of
// the 512 TMEM columns, so the MMAs of stage i+1 run while the epilogue warps drain stage i:
//   stage 0  layer 1, outputs   0..255  -> region 0     stage 2  layer 2 (16 K-chunks)   -> region 0
//   stage 1  layer 1, outputs 256..511  -> region 1     stage 3  layer 3 (N = 16)        -> region 1
// Barriers (all single-CTA mbarriers):
//   w3_full / w3_free       the output layer's weights have their own 8 KB buffer (in the ring they would hold a stage
//                           from the end of layer 2's stream until layer 3 is issued and stall the next network's stream)
//   w_full[s] / w_free[s]   weight stage s landed (bulk copy multicast by the cluster CTA that owns the chunk) / the MMAs
//                           that read it have retired in BOTH CTAs of the cluster (multicast commits, count 2)
//   acc_full[r]             the MMAs of the stage that accumulates into TMEM region r retired
//   acc_free[r]             the 256 epilogue threads have drained region r (tcgen05.ld done)
//   a_ready[0..2]           hidden-1 columns 0..255 / 256..511 / hidden-2 written to shared memory (the A operand of the
//                           next layer); layer 2's first 8 K-chunks only need the first half of hidden 1
__global__ void __cluster_dims__(kCluster, 1, 1) __launch_bounds__(kThreads, 1) k_mlp(const MlpParams P) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sA0 = smem + kOffA0; uint8_t* sA1 = smem + kOffA1;
  uint8_t* sW = smem + kOffW;
  uint64_t* w_full = reinterpret_cast<uint64_t*>(smem + kOffBar);      // [kStages]
  uint64_t* w_free = w_full + kStages;                                  // [kStages]
  uint64_t* acc_full = w_free + kStages;                                // [2]
  uint64_t* acc_free = acc_full + 2;                                    // [2]
  uint64_t* a_ready = acc_free + 2;                                     // [3]
  uint64_t* w3_full = a_ready + 3;
  uint64_t* w3_free = w3_full + 1;
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(w3_free + 1);
  uint8_t* sW3 = smem + kOffW3;
  float* s_bias = reinterpret_cast<float*>(smem + kOffBias);            // both networks' biases (epilogue broadcasts)
  const int tid = threadIdx.x, warp = tid >> 5;
  const int K0p = P.K0p;
  const int total_chunks = 2 * kRingChunks;

  if (tid == 0) {
    for (int i = 0; i < kStages; i++) { mbar_init(&w_full[i], 1); mbar_init(&w_free[i], kCluster); }
    for (int i = 0; i < 2; i++) { mbar_init(&acc_full[i], 1); mbar_init(&acc_free[i], kEpiThreads); }
    for (int i = 0; i < 3; i++) mbar_init(&a_ready[i], kEpiThreads);
    mbar_init(w3_full, 1); mbar_init(w3_free, kCluster);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(s_tmem)), "r"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  __syncthreads();
  cluster_sync_all();                                  // the peer's barriers are initialised before anything arrives on them
  constexpr uint16_t kAllCtas = (uint16_t)((1u << kCluster) - 1);
  const uint32_t crank = cluster_ctarank();
  // one weight chunk: every CTA arms its own barrier, the chunk's owner fetches it once and multicasts it to the cluster
  auto send = [&](uint8_t* dst, uint64_t* bar, int net, int packed_chunk, bool owner) {
    const uint32_t bytes = (uint32_t)chunk_bytes(packed_chunk, K0p);
    mbar_expect_tx(bar, bytes);
    if (owner) bulk_g2s_multicast(dst, P.wpack[net] + chunk_offset(packed_chunk, K0p), bytes, bar, kAllCtas);
  };
  if (tid == kProducerTid) {                           // the first stages fill while the other warps stage biases and observations
    MLP_STAMP(32);
    for (int c = 0; c < kStages; c++) send(sW + c * kWBufBytes, &w_full[c], 0, c, (uint32_t)(c % kCluster) == crank);
    send(sW3, w3_full, 0, kRingChunks, crank == 0);
  }
  for (int i = tid; i < 2 * kBiasFloats; i += kThreads) s_bias[i] = P.bias[i / kBiasFloats][i % kBiasFloats];
  load_obs_tile(P, K0p, sA0, tid);
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *s_tmem;

  if (tid == kProducerTid) {
    // ---- weight producer: the flat ring sequence (actor W1 + W2 chunks, then the critic's) through kStages buffers
    for (int c = kStages; c < total_chunks; c++) {
      if (c == kL1Chunks) MLP_STAMP(33);
      if (c == kRingChunks) MLP_STAMP(34);
      if (c == kRingChunks + kL1Chunks) MLP_STAMP(35);
      const int st = c % kStages;
      mbar_wait(&w_free[st], (uint32_t)((c / kStages - 1) & 1));          // freed by every CTA of the cluster
      send(sW + st * kWBufBytes, &w_full[st], c / kRingChunks, c % kRingChunks, (uint32_t)(c % kCluster) == crank);
      if (c == total_chunks - kStages) {               // the critic's W3, long after the actor's layer 3 has retired
        mbar_wait(w3_free, 0u);
        send(sW3, w3_full, 1, kRingChunks, crank == 0);
      }
    }
    MLP_STAMP(36);
  } else if (tid == kIssuerTid) {
    // ---- MMA issuer
    int c = 0;
    uint32_t ph_free[2] = { 0, 0 }, ph_ready[3] = { 0, 0, 0 };
    auto mma_chunk = [&](uint32_t a_saddr, uint32_t a_sbo, int ksteps, uint32_t dcol, int ncols, bool accumulate) {
      const int st = c % kStages;
      mbar_wait(&w_full[st], (uint32_t)((c / kStages) & 1));
      tc_fence_after();
      const ChunkDesc d = chunk_desc(c % kRingChunks, K0p);
      const uint32_t b_saddr = smem_u32(sW + st * kWBufBytes), b_sbo = (uint32_t)(d.kc >> 3) * 128u;
      const uint32_t idesc = make_idesc(kM, ncols);
      for (int k = 0; k < ksteps; k++)
        umma_bf16(tmem + dcol, make_desc(a_saddr + k * 256, 128, a_sbo), make_desc(b_saddr + k * 256, 128, b_sbo), idesc,
                  (accumulate || k > 0) ? 1u : 0u);
      umma_commit_multicast(&w_free[st], kAllCtas);
      c++;
    };
    for (int net = 0; net < 2; net++) {
      for (int h = 0; h < 2; h++) {                                      // stages 0, 1: layer 1 halves -> regions 0, 1
        if (net > 0) { mbar_wait(&acc_free[h], ph_free[h]); ph_free[h] ^= 1; tc_fence_after(); }
        for (int q = 0; q < 2; q++)
          mma_chunk(smem_u32(sA0), (uint32_t)(K0p >> 3) * 128u, K0p / 16, (uint32_t)(h * 256 + q * kL1Rows), kL1Rows, false);
        umma_commit(&acc_full[h]);
        MLP_STAMP(16 + net * 8 + h);
      }
      mbar_wait(&acc_free[0], ph_free[0]); ph_free[0] ^= 1;               // stage 2: layer 2 -> region 0
      for (int kc = 0; kc < kL2Chunks; kc++) {
        if (kc == 0) { mbar_wait(&a_ready[0], ph_ready[0]); ph_ready[0] ^= 1; tc_fence_after(); }
        if (kc == kL2Chunks / 2) { MLP_STAMP(16 + net * 8 + 2); mbar_wait(&a_ready[1], ph_ready[1]); ph_ready[1] ^= 1; tc_fence_after(); }
        mma_chunk(smem_u32(sA1) + kc * (kK2Chunk / 8) * 128, (uint32_t)(kH1 >> 3) * 128u, kK2Chunk / 16, 0u, 256, kc > 0);
      }
      umma_commit(&acc_full[0]);
      MLP_STAMP(16 + net * 8 + 3);
      mbar_wait(&acc_free[1], ph_free[1]); ph_free[1] ^= 1;               // stage 3: layer 3 -> region 1
      mbar_wait(&a_ready[2], ph_ready[2]); ph_ready[2] ^= 1; tc_fence_after();
      mbar_wait(w3_full, (uint32_t)net);
      tc_fence_after();
      for (int k = 0; k < kH2 / 16; k++)
        umma_bf16(tmem + 256u, make_desc(smem_u32(sA1) + k * 256, 128, (uint32_t)(kH2 >> 3) * 128u),
                  make_desc(smem_u32(sW3) + k * 256, 128, (uint32_t)(kH2 >> 3) * 128u), make_idesc(kM, kNOut), k > 0 ? 1u : 0u);
      umma_commit_multicast(w3_free, kAllCtas);
      umma_commit(&acc_full[1]);
      MLP_STAMP(16 + net * 8 + 4);
    }
  } else if (tid < kEpiThreads) {
    // ---- epilogue warpgroups: thread = (row, column half)
    const int row = tid & (kM - 1), ch = tid >> 7;
    const int grow = blockIdx.x * kM + row;
    const uint32_t tmem_row = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    uint32_t ph_full[2] = { 0, 0 };
    auto wait_full = [&](int r) { mbar_wait(&acc_full[r], ph_full[r]); ph_full[r] ^= 1; tc_fence_after(); };
    // region drained (+ A operand written and visible to the async proxy): let the issuer go on
    auto release = [&](int r, int ready) {
      tc_fence_before();
      if (ready >= 0) { fence_async_smem(); mbar_arrive(&a_ready[ready]); }
      mbar_arrive(&acc_free[r]);
    };
    float outv[kNOut];
    // the actor's sample + log-prob: runs in the epilogue warps' idle time while the critic's layer-2 weights stream in
    auto sample_actor = [&]() { if (ch == 0 && grow < P.n) sample_row(P, grow, outv); };
    if (tid == 0) MLP_STAMP(0);
    for (int net = 0; net < 2; net++) {
      const float* b1 = s_bias + net * kBiasFloats; const float* b2 = b1 + kH1; const float* b3 = b2 + kH2;
      for (int h = 0; h < 2; h++) {
        wait_full(h);
        if (tid == 0) MLP_STAMP(1 + net * 7 + h * 2);
        epilogue_hidden(tmem_row + h * 256, ch * 128, 128, b1 + h * 256, sA1, kH1, h * 256, row);
        release(h, h);
        if (tid == 0) MLP_STAMP(2 + net * 7 + h * 2);
        if (net == 1 && h == 1) sample_actor();
      }
      wait_full(0);                                                      // every layer-2 MMA retired: hidden 2 may overwrite hidden 1
      if (tid == 0) MLP_STAMP(5 + net * 7);
      epilogue_hidden(tmem_row, ch * 128, 128, b2, sA1, kH2, 0, row);
      release(0, 2);
      if (tid == 0) MLP_STAMP(6 + net * 7);
      wait_full(1);
      if (tid == 0) MLP_STAMP(7 + net * 7);
      if (ch == 0) {
        uint32_t v[16];
        tmem_ld16(tmem_row + 256, v);
        if (net == 0) {
#pragma unroll
          for (int a = 0; a < kNOut; a++) outv[a] = tanhf(__uint_as_float(v[a]) + b3[a]);   // actor: Tanh head
        } else if (grow < P.n && P.value) {
          P.value[grow] = __uint_as_float(v[0]) + b3[0];
        }
      }
      release(1, -1);
    }
    if (tid == 0) MLP_STAMP(15);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "r"(512) : "memory");
  }
  cluster_sync_all();                                  // no CTA leaves while its peer may still signal its barriers
}

// ---------------------------------------------------------------------------------------------- k_mlp_wide
// The terrain trainer's ActorCritic (sim2real/train2.py:149-157): Linear(S,1024)-tanh -> Linear(1024,512)-tanh -> head,
// with k_mlp's contract (bf16 operands, fp32 accumulation in TMEM, tanh.approx on the hidden layers, tanhf on the actor
// head, sample_row). A 128 x 1024 bf16 hidden-1 tile (256 KB) does not fit shared memory, so hidden 1 is never stored
// whole. Layer 2 runs as two N = 256 halves, each accumulating in TMEM columns 0-255; for each half hidden 1 is recomputed
// in 128-column chunks (layer 1 has K = K0p <= 64: K0p / (K0p + 512) more FLOPs, 3 % at the terrain trainer's S = 12, 11 % at S = 64) into TMEM columns 256-383 / 384-511 (ping-pong), and the
// epilogue drains each chunk into one of two 32 KB bf16 buffers, the A operand of that chunk's layer-2 MMAs. The head
// (K = 512; A or 1 outputs) runs on CUDA cores inside the hidden-2 epilogue: bf16-rounded hidden 2 times bf16 W3, fp32
// sums, so no 128 KB hidden-2 tile either. Work unit U = (network, half, chunk), 32 per CTA; the MMA issue order is
// L1(0), L1(1), L2(0), L1(2), L2(1), ... so that the epilogue drains chunk U + 1 while the layer-2 MMAs of chunk U run.
constexpr int kWH1 = 1024, kWH2 = 512;
constexpr int kWChunkCols = 128;                                 // hidden-1 columns per recomputed chunk (N of layer 1)
constexpr int kWChunks = kWH1 / kWChunkCols;                     // 8 chunks per layer-2 half
constexpr int kWHalves = kWH2 / 256;                             // 2 layer-2 halves of N = 256
constexpr int kWUnitsPerNet = kWHalves * kWChunks, kWUnits = 2 * kWUnitsPerNet;
constexpr int kWL2PerUnit = kWChunkCols / kK2Chunk;              // 4 W2 stages (256 x 32) per unit
constexpr int kWW2Chunks = kWHalves * (kWH1 / kK2Chunk);         // 64 packed W2 chunks per network
constexpr int kWNumChunks = kWChunks + kWW2Chunks + 1;           // + W3 = 73 packed chunks per network
constexpr int kWW3Bytes = kWH2 * kNOut * 2;                      // 16 KB: W3 as [512][16] bf16 (a hidden-2 unit's head weights)
constexpr int kWH1Bytes = kM * kWChunkCols * 2;                  // 32 KB hidden-1 chunk
constexpr int kWOffA0 = 0, kWOffH1 = kWOffA0 + kA0Bytes, kWOffW = kWOffH1 + 2 * kWH1Bytes;
constexpr int kWOffW3 = kWOffW + kStages * kWBufBytes;          // both networks' W3, loaded once
constexpr int kWOffX = kWOffW3 + 2 * kWW3Bytes;                 // head partial sums of the second column half, [2][128][16] f32
constexpr int kWOffBar = kWOffX + 2 * kM * kNOut * 4;
constexpr int kWBiasFloats = kWH1 + kWH2 + kNOut;               // per network: b1 | b2 | b3
constexpr int kWOffBias = kWOffBar + 256;
constexpr int kWSmemBytes = kWOffBias + 2 * kWBiasFloats * 4;
static_assert(kWSmemBytes <= 227 * 1024, "k_mlp_wide: shared memory over the 227 KB a block may use");

// packed chunks of one network: W1 [0, 8) (128 x K0p), W2 [8, 72) (256 x 32: half h, K-chunk k at 8 + 32 h + k), W3 72
__host__ __device__ inline int wide_chunk_bytes(int c, int K0p) { return c < kWChunks ? kWChunkCols * K0p * 2 : kWBufBytes; }
__host__ __device__ inline int wide_chunk_offset(int c, int K0p) {
  return c <= kWChunks ? c * kWChunkCols * K0p * 2 : kWChunks * kWChunkCols * K0p * 2 + (c - kWChunks) * kWBufBytes;
}

// hidden-2 epilogue of one thread with the head folded in: for the 128 columns [c0, c0 + 128) of a layer-2 half,
// h = bf16(tanh(D + b2)) (the value the next layer's bf16 operand would hold), acc[a] += h * W3[a][col] for a < NO
template <int NO>
__device__ __forceinline__ void epilogue_head(uint32_t taddr_row, int c0, const float* __restrict__ bias, const uint8_t* w3,
                                              float (&acc)[kNOut]) {
  for (int cb = c0; cb < c0 + 128; cb += 32) {
    uint32_t v[32];
    tmem_ld32_nowait(taddr_row + cb, v);
    tmem_ld_wait();
#pragma unroll
    for (int i = 0; i < 32; i++) {
      const int col = cb + i;
      const float h = __bfloat162float(__float2bfloat16_rn(tanh_fast(__uint_as_float(v[i]) + bias[col])));
      const __nv_bfloat162* w = reinterpret_cast<const __nv_bfloat162*>(w3 + col * kNOut * 2);
#pragma unroll
      for (int a = 0; a < NO; a += 2) {
        const float2 wf = __bfloat1622float2(w[a / 2]);
        acc[a] = fmaf(h, wf.x, acc[a]);
        if (a + 1 < NO) acc[a + 1] = fmaf(h, wf.y, acc[a + 1]);
      }
    }
  }
}

// Barriers (single-CTA mbarriers unless noted):
//   w_full[s] / w_free[s]   weight stage s landed / its MMAs retired in BOTH CTAs of the cluster (as in k_mlp)
//   w3_full                 both networks' W3 landed (one multicast copy per network)
//   l1_full[b]              layer-1 MMAs of a chunk into TMEM region 256 + 128 b retired
//   h1_ready[b]             the epilogue drained region b and wrote hidden-1 buffer b (256 arrivals)
//   h1_free[b]              the layer-2 MMAs reading hidden-1 buffer b retired
//   acc2_full / acc2_free   a layer-2 half in TMEM columns 0-255 is complete / drained by the epilogue
__global__ void __cluster_dims__(kCluster, 1, 1) __launch_bounds__(kThreads, 1) k_mlp_wide(const MlpParams P) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sA0 = smem + kWOffA0; uint8_t* sH1 = smem + kWOffH1; uint8_t* sW = smem + kWOffW; uint8_t* sW3 = smem + kWOffW3;
  float* sX = reinterpret_cast<float*>(smem + kWOffX);
  uint64_t* w_full = reinterpret_cast<uint64_t*>(smem + kWOffBar);      // [kStages]
  uint64_t* w_free = w_full + kStages;                                  // [kStages]
  uint64_t* l1_full = w_free + kStages;                                 // [2]
  uint64_t* h1_ready = l1_full + 2;                                     // [2]
  uint64_t* h1_free = h1_ready + 2;                                     // [2]
  uint64_t* acc2_full = h1_free + 2;
  uint64_t* acc2_free = acc2_full + 1;
  uint64_t* w3_full = acc2_free + 1;
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(w3_full + 1);
  float* s_bias = reinterpret_cast<float*>(smem + kWOffBias);
  const int tid = threadIdx.x, warp = tid >> 5;
  const int K0p = P.K0p;

  if (tid == 0) {
    for (int i = 0; i < kStages; i++) { mbar_init(&w_full[i], 1); mbar_init(&w_free[i], kCluster); }
    for (int i = 0; i < 2; i++) { mbar_init(&l1_full[i], 1); mbar_init(&h1_ready[i], kEpiThreads); mbar_init(&h1_free[i], 1); }
    mbar_init(acc2_full, 1); mbar_init(acc2_free, kEpiThreads); mbar_init(w3_full, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(s_tmem)), "r"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  __syncthreads();
  cluster_sync_all();
  constexpr uint16_t kAllCtas = (uint16_t)((1u << kCluster) - 1);
  const uint32_t crank = cluster_ctarank();
  for (int i = tid; i < 2 * kWBiasFloats; i += kThreads) s_bias[i] = P.bias[i / kWBiasFloats][i % kWBiasFloats];
  load_obs_tile(P, K0p, sA0, tid);
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *s_tmem;

  if (tid == kProducerTid) {
    // ---- weight producer: both W3 once, then the ring in the issuer's order (W1 of unit U + 1 before the W2 of unit U)
    mbar_expect_tx(w3_full, 2u * kWW3Bytes);
    for (int net = 0; net < 2; net++)
      if ((uint32_t)(net % kCluster) == crank)
        bulk_g2s_multicast(sW3 + net * kWW3Bytes, P.wpack[net] + wide_chunk_offset(kWNumChunks - 1, K0p), kWW3Bytes, w3_full, kAllCtas);
    int c = 0;
    auto push = [&](int net, int packed) {
      const int st = c % kStages;
      if (c >= kStages) mbar_wait(&w_free[st], (uint32_t)((c / kStages - 1) & 1));       // freed by every CTA of the cluster
      const uint32_t bytes = (uint32_t)wide_chunk_bytes(packed, K0p);
      mbar_expect_tx(&w_full[st], bytes);
      if ((uint32_t)(c % kCluster) == crank)
        bulk_g2s_multicast(sW + st * kWBufBytes, P.wpack[net] + wide_chunk_offset(packed, K0p), bytes, &w_full[st], kAllCtas);
      c++;
    };
    push(0, 0);
    for (int U = 0; U < kWUnits; U++) {
      if (U + 1 < kWUnits) push((U + 1) / kWUnitsPerNet, (U + 1) % kWChunks);
      const int net = U / kWUnitsPerNet, nh = (U / kWChunks) % kWHalves, j = U % kWChunks;
      for (int q = 0; q < kWL2PerUnit; q++) push(net, kWChunks + nh * (kWH1 / kK2Chunk) + j * kWL2PerUnit + q);
    }
  } else if (tid == kIssuerTid) {
    // ---- MMA issuer
    int c = 0;
    uint32_t ph_ready[2] = { 0, 0 }, ph_acc2_free = 0;
    auto mma_stage = [&](uint32_t a_saddr, uint32_t a_sbo, int ksteps, uint32_t b_sbo, uint32_t dcol, int ncols, bool accumulate) {
      const int st = c % kStages;
      mbar_wait(&w_full[st], (uint32_t)((c / kStages) & 1));
      tc_fence_after();
      const uint32_t b_saddr = smem_u32(sW + st * kWBufBytes), idesc = make_idesc(kM, ncols);
      for (int k = 0; k < ksteps; k++)
        umma_bf16(tmem + dcol, make_desc(a_saddr + k * 256, 128, a_sbo), make_desc(b_saddr + k * 256, 128, b_sbo), idesc,
                  (accumulate || k > 0) ? 1u : 0u);
      umma_commit_multicast(&w_free[st], kAllCtas);
      c++;
    };
    // layer 1 of unit U -> TMEM region U & 1. Its previous user, unit U - 2, was drained: the issuer waited for h1_ready of
    // U - 2 before issuing L2(U - 2), which precedes this call
    auto layer1 = [&](int U) {
      const uint32_t sbo = (uint32_t)(K0p >> 3) * 128u;
      mma_stage(smem_u32(sA0), sbo, K0p / 16, sbo, 256u + (uint32_t)(U & 1) * kWChunkCols, kWChunkCols, false);
      umma_commit(&l1_full[U & 1]);
    };
    layer1(0);
    for (int U = 0; U < kWUnits; U++) {
      if (U + 1 < kWUnits) layer1(U + 1);
      const int b = U & 1, j = U % kWChunks;
      mbar_wait(&h1_ready[b], ph_ready[b]); ph_ready[b] ^= 1;
      if (j == 0 && U > 0) { mbar_wait(acc2_free, ph_acc2_free); ph_acc2_free ^= 1; }
      tc_fence_after();
      for (int q = 0; q < kWL2PerUnit; q++)
        mma_stage(smem_u32(sH1 + b * kWH1Bytes) + q * (kK2Chunk / 8) * 128, (uint32_t)(kWChunkCols >> 3) * 128u, kK2Chunk / 16,
                  (uint32_t)(kK2Chunk >> 3) * 128u, 0u, 256, j > 0 || q > 0);
      umma_commit(&h1_free[b]);
      if (j == kWChunks - 1) umma_commit(acc2_full);
    }
  } else if (tid < kEpiThreads) {
    // ---- epilogue warpgroups: thread = (row, column half)
    const int row = tid & (kM - 1), ch = tid >> 7;
    const int grow = blockIdx.x * kM + row;
    const uint32_t tmem_row = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    uint32_t ph_l1[2] = { 0, 0 }, ph_free[2] = { 0, 0 }, ph_acc2 = 0;
    float acc[kNOut], outv[kNOut];
    for (int U = 0; U < kWUnits; U++) {
      const int net = U / kWUnitsPerNet, nh = (U / kWChunks) % kWHalves, j = U % kWChunks, b = U & 1;
      const float* b1 = s_bias + net * kWBiasFloats; const float* b2 = b1 + kWH1; const float* b3 = b2 + kWH2;
      if (U % kWUnitsPerNet == 0) {
#pragma unroll
        for (int a = 0; a < kNOut; a++) acc[a] = 0.f;
      }
      mbar_wait(&l1_full[b], ph_l1[b]); ph_l1[b] ^= 1;
      if (U >= 2) { mbar_wait(&h1_free[b], ph_free[b]); ph_free[b] ^= 1; }          // L2(U - 2) no longer reads buffer b
      tc_fence_after();
      epilogue_hidden(tmem_row + 256 + b * kWChunkCols, ch * 64, 64, b1 + j * kWChunkCols, sH1 + b * kWH1Bytes, kWChunkCols, 0, row);
      tc_fence_before();
      fence_async_smem();
      mbar_arrive(&h1_ready[b]);
      if (j != kWChunks - 1) continue;
      // ---- a layer-2 half is complete: hidden 2 + head partial sums
      mbar_wait(acc2_full, ph_acc2); ph_acc2 ^= 1;
      tc_fence_after();
      if (U == kWChunks - 1) mbar_wait(w3_full, 0u);
      const uint8_t* w3 = sW3 + net * kWW3Bytes + nh * 256 * kNOut * 2;
      if (net == 1) epilogue_head<1>(tmem_row, ch * 128, b2 + nh * 256, w3, acc);
      else if (P.A <= 8) epilogue_head<8>(tmem_row, ch * 128, b2 + nh * 256, w3, acc);
      else epilogue_head<16>(tmem_row, ch * 128, b2 + nh * 256, w3, acc);
      tc_fence_before();
      mbar_arrive(acc2_free);
      if (nh != kWHalves - 1) continue;
      // ---- the network is complete: add the two column halves' partial sums (fixed order), head bias, output
      float* x = sX + (net * kM + row) * kNOut;
      if (ch == 1) {
#pragma unroll
        for (int a = 0; a < kNOut; a++) x[a] = acc[a];
      }
      asm volatile("bar.sync 1, %0;" :: "r"(kEpiThreads) : "memory");     // the 256 epilogue threads only
      if (ch == 0) {
        if (net == 0) {
#pragma unroll
          for (int a = 0; a < kNOut; a++) outv[a] = tanhf(acc[a] + x[a] + b3[a]);          // actor: Tanh head
          if (grow < P.n) sample_row(P, grow, outv);
        } else if (grow < P.n && P.value) {
          P.value[grow] = acc[0] + x[0] + b3[0];
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "r"(512) : "memory");
  }
  cluster_sync_all();                                  // no CTA leaves while its peer may still signal its barriers
}

// fp32 [out][in] weights -> bf16 chunks. One thread per destination element pair.
__global__ void k_pack(const float* __restrict__ w0, const float* __restrict__ w1, const float* __restrict__ w2,
                       int S, int nout, int K0p, uint8_t* __restrict__ dst) {
  const int c = blockIdx.y;
  const ChunkDesc d = chunk_desc(c, K0p);
  const int e = blockIdx.x * blockDim.x + threadIdx.x;                  // element index r * kc + k
  if (e >= d.rows * d.kc) return;
  const int r = e / d.kc, k = e % d.kc;
  float v = 0.f;
  if (d.layer == 0) { if (k < S) v = w0[(size_t)(d.row0 + r) * S + k]; }
  else if (d.layer == 1) v = w1[(size_t)r * kH1 + d.k0 + k];
  else { if (r < nout) v = w2[(size_t)r * kH2 + k]; }
  *reinterpret_cast<__nv_bfloat16*>(dst + chunk_offset(c, K0p) + canon_off(r, k, d.kc)) = __float2bfloat16_rn(v);
}
// the same for k_mlp_wide's chunks (wide_chunk_offset); W3 goes to [512][16] for the CUDA-core head
__global__ void k_pack_wide(const float* __restrict__ w0, const float* __restrict__ w1, const float* __restrict__ w2,
                            int S, int nout, int K0p, uint8_t* __restrict__ dst) {
  const int c = blockIdx.y;
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  float v = 0.f;
  int off;
  if (c < kWChunks) {                                                   // W1 rows [128 c, 128 c + 128)
    if (e >= kWChunkCols * K0p) return;
    const int r = e / K0p, k = e % K0p;
    if (k < S) v = w0[(size_t)(c * kWChunkCols + r) * S + k];
    off = canon_off(r, k, K0p);
  } else if (c < kWChunks + kWW2Chunks) {                               // W2 rows of half h, K-chunk kq
    if (e >= 256 * kK2Chunk) return;
    const int q = c - kWChunks, h = q / (kWH1 / kK2Chunk), kq = q % (kWH1 / kK2Chunk);
    const int r = e / kK2Chunk, k = e % kK2Chunk;
    v = w1[(size_t)(h * 256 + r) * kWH1 + kq * kK2Chunk + k];
    off = canon_off(r, k, kK2Chunk);
  } else {                                                              // W3 transposed: [hidden-2 unit][output]
    if (e >= kWH2 * kNOut) return;
    const int k = e / kNOut, a = e % kNOut;
    if (a < nout) v = w2[(size_t)a * kWH2 + k];
    off = e * 2;
  }
  *reinterpret_cast<__nv_bfloat16*>(dst + wide_chunk_offset(c, K0p) + off) = __float2bfloat16_rn(v);
}
// b1 [h1] | b2 [h2] | b3 [nout] zero-padded to 16
__global__ void k_pack_bias(const float* b0, const float* b1, const float* b2, int h1, int h2, int nout, float* dst) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < h1) dst[i] = b0[i];
  else if (i < h1 + h2) dst[i] = b1[i - h1];
  else if (i < h1 + h2 + kNOut) { const int a = i - h1 - h2; dst[i] = a < nout ? b2[a] : 0.f; }
}

// ---------------------------------------------------------------------------------------------- GAE
constexpr int kGaeBlock = 256;
// one thread per environment: reverse scan over T steps; block-level fixed-order sum of adv and adv^2
__global__ void k_gae(const float* __restrict__ rew, const float* __restrict__ val, const uint8_t* __restrict__ done,
                      int T, int n, float gamma, float lam, float* __restrict__ adv, float* __restrict__ ret,
                      double* __restrict__ partial) {
  __shared__ double s_sum[kGaeBlock], s_sq[kGaeBlock];
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  double sum = 0.0, sq = 0.0;
  if (e < n) {
    float a = 0.f, vnext = val[(size_t)T * n + e];
    for (int t = T - 1; t >= 0; t--) {
      const size_t i = (size_t)t * n + e;
      const float m = done[i] ? 0.f : 1.f, v = val[i];
      const float delta = rew[i] + gamma * vnext * m - v;
      a = delta + gamma * lam * m * a;
      adv[i] = a; if (ret) ret[i] = a + v;
      sum += (double)a; sq += (double)a * (double)a;
      vnext = v;
    }
  }
  s_sum[threadIdx.x] = sum; s_sq[threadIdx.x] = sq;
  __syncthreads();
  for (int d = kGaeBlock / 2; d > 0; d >>= 1) {
    if (threadIdx.x < d) { s_sum[threadIdx.x] += s_sum[threadIdx.x + d]; s_sq[threadIdx.x] += s_sq[threadIdx.x + d]; }
    __syncthreads();
  }
  if (threadIdx.x == 0) { partial[2 * blockIdx.x] = s_sum[0]; partial[2 * blockIdx.x + 1] = s_sq[0]; }
}
__global__ void k_gae_finish(const double* __restrict__ partial, int nblocks, long long count, double* __restrict__ stats) {
  __shared__ double s_sum[kGaeBlock], s_sq[kGaeBlock];
  double sum = 0.0, sq = 0.0;
  for (int i = threadIdx.x; i < nblocks; i += kGaeBlock) { sum += partial[2 * i]; sq += partial[2 * i + 1]; }
  s_sum[threadIdx.x] = sum; s_sq[threadIdx.x] = sq;
  __syncthreads();
  for (int d = kGaeBlock / 2; d > 0; d >>= 1) {
    if (threadIdx.x < d) { s_sum[threadIdx.x] += s_sum[threadIdx.x + d]; s_sq[threadIdx.x] += s_sq[threadIdx.x + d]; }
    __syncthreads();
  }
  if (threadIdx.x == 0) { stats[0] = s_sum[0]; stats[1] = s_sq[0]; stats[2] = (double)count; }
}
__global__ void k_adv_norm(float* __restrict__ adv, long long count, const double* __restrict__ stats) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const double n = stats[2], mean = stats[0] / n;
  const double var = n > 1.0 ? fmax(0.0, (stats[1] - n * mean * mean) / (n - 1.0)) : 0.0;   // torch.std: unbiased
  adv[i] = (float)(((double)adv[i] - mean) / (sqrt(var) + 1e-8));
}

// ---- PPO update phase: the backward of a hidden layer's tanh fused with the bias gradient of its Linear ----------------
// g = gy * (1 - y*y) (bf16 in, fp32 arithmetic, bf16 out: torch's tanh_backward) and, in the same pass, the column sums of
// the ROUNDED g (what grad_output.sum(0) of the Linear's backward adds up) as per-block fp32 partials in a fixed order.
// torch runs these as two passes over the [rows, cols] gradient, the second one a bf16 column reduction at ~2 TB/s: 17 % of
// a PPO epoch at 65536 envs x 24 (tools/prof_ppo2.py).
constexpr int kTbGrid = 592;                        // 148 SMs x 4 blocks; also the row count of the partial-sum scratch
constexpr int kTbBlock = 256;
__device__ __forceinline__ void tb_unpack(const uint4& v, float (&f)[8]) {
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
  for (int k = 0; k < 4; k++) { const float2 t = __bfloat1622float2(h[k]); f[2 * k] = t.x; f[2 * k + 1] = t.y; }
}
__global__ void __launch_bounds__(kTbBlock) k_tanh_bwd_bias(const uint4* __restrict__ gy, const uint4* __restrict__ y,
                                                            uint4* __restrict__ g, float* __restrict__ partial,
                                                            long long rows, int cols) {
  __shared__ float s_acc[kTbBlock * 8];
  const int groups = cols >> 3;                     // 16-byte column groups per row (a power of two <= 256)
  const int cg = threadIdx.x & (groups - 1), rl = threadIdx.x / groups, rp = kTbBlock / groups;
  long long chunk = (rows + gridDim.x - 1) / gridDim.x;
  chunk = (chunk + rp - 1) / rp * rp;
  const long long r0 = (long long)blockIdx.x * chunk, r1 = r0 + chunk < rows ? r0 + chunk : rows;
  float acc[8];
#pragma unroll
  for (int k = 0; k < 8; k++) acc[k] = 0.f;
  auto one = [&](const uint4& a, const uint4& b, long long r) {
    float fa[8], fb[8];
    tb_unpack(a, fa); tb_unpack(b, fb);
    uint4 o; __nv_bfloat162* oh = reinterpret_cast<__nv_bfloat162*>(&o);
#pragma unroll
    for (int k = 0; k < 4; k++) {
      const float g0 = fa[2 * k] * (1.f - fb[2 * k] * fb[2 * k]), g1 = fa[2 * k + 1] * (1.f - fb[2 * k + 1] * fb[2 * k + 1]);
      oh[k] = __floats2bfloat162_rn(g0, g1);
      const float2 q = __bfloat1622float2(oh[k]);
      acc[2 * k] += q.x; acc[2 * k + 1] += q.y;
    }
    g[r * groups + cg] = o;
  };
  long long r = r0 + rl;
  for (; r + 3LL * rp < r1; r += 4LL * rp) {        // four rows in flight per thread (8 x 16-byte loads)
    uint4 a[4], b[4];
#pragma unroll
    for (int u = 0; u < 4; u++) { a[u] = __ldcs(gy + (r + (long long)u * rp) * groups + cg); b[u] = __ldcs(y + (r + (long long)u * rp) * groups + cg); }
#pragma unroll
    for (int u = 0; u < 4; u++) one(a[u], b[u], r + (long long)u * rp);
  }
  for (; r < r1; r += rp) one(__ldcs(gy + r * groups + cg), __ldcs(y + r * groups + cg), r);
  // the block's column sums: row lanes added in lane order
#pragma unroll
  for (int k = 0; k < 8; k++) s_acc[rl * cols + cg * 8 + k] = acc[k];
  __syncthreads();
  for (int c = threadIdx.x; c < cols; c += kTbBlock) {
    float t = 0.f;
    for (int q = 0; q < rp; q++) t += s_acc[q * cols + c];
    partial[(size_t)blockIdx.x * cols + c] = t;
  }
}
// 32 columns per block, 8 threads per column: each adds every 8th block's partial, the 8 sums are added in slice order
__global__ void __launch_bounds__(256) k_colsum_finish(const float* __restrict__ partial, int nblocks, int cols,
                                                       float* __restrict__ out) {
  __shared__ float s_t[8][32];
  const int cl = threadIdx.x & 31, sl = threadIdx.x >> 5, c = blockIdx.x * 32 + cl;
  float t = 0.f;
  if (c < cols) for (int b = sl; b < nblocks; b += 8) t += partial[(size_t)b * cols + c];
  s_t[sl][cl] = t;
  __syncthreads();
  if (sl == 0 && c < cols) {
    float u = 0.f;
#pragma unroll
    for (int q = 0; q < 8; q++) u += s_t[q][cl];
    out[c] = u;
  }
}

// ---- PPO update phase: the clipped-surrogate loss of one minibatch and its gradients in one pass ----------------------
// (SB3's PPO objective with the hyper-parameters of train/train.py:117-130; sim2real/train.py:566-569 is its special case
// clip = +inf, logp_old = logp: Normal log-prob, probability ratio, clipped surrogate, value MSE, entropy bonus). torch evaluates this as ~170 element-wise / reduction launches per minibatch over [B, A] tensors
// (1.5 ms of an 11.8 ms epoch at 65536 envs x 24); here one thread per sample computes its loss terms AND
// d loss / d mean, d loss / d value, and its share of d loss / d log_std; block partials are added in a fixed order.
constexpr int kPlBlock = 256, kPlMaxGrid = 1184, kPlCols = 32, kPlMaxA = 16;
__global__ void __launch_bounds__(kPlBlock) k_ppo_loss(const float* __restrict__ mean, const float* __restrict__ value,
                                                       const float* __restrict__ log_std, const float* __restrict__ action,
                                                       const float* __restrict__ logp_old, const float* __restrict__ adv,
                                                       const float* __restrict__ ret, long long B, int A, float clip,
                                                       float vf_coef, float* __restrict__ g_mean, float* __restrict__ g_value,
                                                       float* __restrict__ partial) {
  __shared__ float s_w[kPlBlock / 32][kPlCols];
  float ls[kPlMaxA], inv_sig[kPlMaxA], acc[2 + kPlMaxA];
#pragma unroll
  for (int k = 0; k < kPlMaxA; k++) { ls[k] = k < A ? log_std[k] : 0.f; inv_sig[k] = expf(-ls[k]); }
#pragma unroll
  for (int k = 0; k < 2 + kPlMaxA; k++) acc[k] = 0.f;
  const float invB = 1.f / (float)B;
  for (long long i = (long long)blockIdx.x * kPlBlock + threadIdx.x; i < B; i += (long long)gridDim.x * kPlBlock) {
    float z[kPlMaxA], logp = 0.f;
#pragma unroll
    for (int k = 0; k < kPlMaxA; k++) if (k < A) {
      z[k] = (action[i * A + k] - mean[i * A + k]) * inv_sig[k];
      logp += -0.5f * z[k] * z[k] - ls[k] - 0.9189385332046727f;
    }
    const float ratio = expf(logp - logp_old[i]), a = adv[i];
    const float s1 = ratio * a, s2 = fminf(fmaxf(ratio, 1.f - clip), 1.f + clip) * a;
    const bool inside = ratio >= 1.f - clip && ratio <= 1.f + clip;
    // d min(s1, s2) / d ratio with torch's conventions: the smaller argument takes the gradient, a tie splits it evenly;
    // clamp passes the gradient inside [1 - clip, 1 + clip], ends included
    const float w1 = s1 < s2 ? 1.f : (s1 > s2 ? 0.f : 0.5f), w2 = 1.f - w1;
    const float dmin = w1 * a + (inside ? w2 * a : 0.f);
    const float dlogp = -dmin * ratio * invB;       // d (mean of -min) / d logp_i
    acc[0] += -fminf(s1, s2);
    const float dv = value[i] - ret[i];
    acc[1] += dv * dv;
    g_value[i] = vf_coef * 2.f * dv * invB;
#pragma unroll
    for (int k = 0; k < kPlMaxA; k++) if (k < A) {
      g_mean[i * A + k] = dlogp * z[k] * inv_sig[k];
      acc[2 + k] += dlogp * (z[k] * z[k] - 1.f);
    }
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < 2 + kPlMaxA; k++) {
    float t = acc[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (lane == 0) s_w[warp][k] = t;
  }
  __syncthreads();
  if (threadIdx.x < kPlCols) {
    float t = 0.f;
    if (threadIdx.x < 2 + kPlMaxA) for (int w = 0; w < kPlBlock / 32; w++) t += s_w[w][threadIdx.x];
    partial[(size_t)blockIdx.x * kPlCols + threadIdx.x] = t;
  }
}
__global__ void __launch_bounds__(256) k_ppo_finish(const float* __restrict__ partial, int nblocks, int A,
                                                    const float* __restrict__ log_std, float invB, float vf_coef,
                                                    float ent_coef, float* __restrict__ loss, float* __restrict__ terms,
                                                    float* __restrict__ g_log_std) {
  __shared__ float s_t[8][kPlCols];
  __shared__ float s_sum[kPlCols];
  const int cl = threadIdx.x & 31, sl = threadIdx.x >> 5;
  float t = 0.f;
  for (int b = sl; b < nblocks; b += 8) t += partial[(size_t)b * kPlCols + cl];
  s_t[sl][cl] = t;
  __syncthreads();
  if (sl == 0) {
    float u = 0.f;
#pragma unroll
    for (int q = 0; q < 8; q++) u += s_t[q][cl];
    s_sum[cl] = u;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const float pg = s_sum[0] * invB, vf = s_sum[1] * invB;
    float ent = 0.f;
    for (int k = 0; k < A; k++) ent += 1.4189385332046727f + log_std[k];       // 0.5 + 0.5 log(2 pi) + log sigma
    terms[0] = pg + vf_coef * vf - ent_coef * ent; terms[1] = pg; terms[2] = vf; terms[3] = ent;
    loss[0] = terms[0];
  }
  if (threadIdx.x < A) g_log_std[threadIdx.x] = s_sum[2 + threadIdx.x] - ent_coef;
}

// tanh of a bf16 activation tensor in place (the update-phase forward): MUFU tanh.approx — the same function the rollout
// kernel's epilogue applies, so the update-time policy is the rollout-time policy — at HBM speed (torch's tanhf-based
// kernel is instruction-bound at ~4.8 TB/s for bf16)
__device__ __forceinline__ float tanh_approx(float x) { float y; asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__global__ void __launch_bounds__(256) k_tanh_bf16(const uint4* x, uint4* y, long long n16) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  auto one = [](uint4 v) {
    __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&v);
#pragma unroll
    for (int k = 0; k < 4; k++) { const float2 t = __bfloat1622float2(h[k]); h[k] = __floats2bfloat162_rn(tanh_approx(t.x), tanh_approx(t.y)); }
    return v;
  };
  for (; i + 3 * stride < n16; i += 4 * stride) {
    uint4 v[4];
#pragma unroll
    for (int u = 0; u < 4; u++) v[u] = __ldcs(x + i + u * stride);
#pragma unroll
    for (int u = 0; u < 4; u++) y[i + u * stride] = one(v[u]);
  }
  for (; i < n16; i += stride) y[i] = one(__ldcs(x + i));
}

}  // namespace

struct OdgPolicy {
  int device = 0, S = 0, A = 0, K0p = 0;
  bool wide = false;                     // hidden 1024 / 512 (k_mlp_wide) instead of 512 / 256 (k_mlp)
  uint8_t* d_wpack[2] = { nullptr, nullptr };
  float* d_bias[2] = { nullptr, nullptr };
  float* d_log_std = nullptr;
  double* d_partial = nullptr; int partial_cap = 0;
  size_t wpack_bytes = 0;
  long long launches = 0;
};

namespace {
struct DevGuard {
  int prev = -1;
  explicit DevGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
  ~DevGuard() { if (prev >= 0) cudaSetDevice(prev); }
};
// device that owns a caller buffer (entry points without a handle run where their tensors live)
int device_of(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess || a.type != cudaMemoryTypeDevice) { cudaGetLastError(); return -1; }
  return a.device;
}
bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }
}  // namespace

extern "C" {

int odg_policy_create(int state_dim, int action_dim, int device, OdgPolicy** out) {
  return odg_policy_create_hidden(state_dim, action_dim, kH1, kH2, device, out);
}

int odg_policy_create_hidden(int state_dim, int action_dim, int h1, int h2, int device, OdgPolicy** out) {
  if (!out || state_dim < 1 || state_dim > ODG_POLICY_MAX_STATE || action_dim < 1 || action_dim > ODG_POLICY_MAX_ACTION)
    return set_error(ODG_ERR_INVALID, "odg_policy_create: state_dim must be in [1,64], action_dim in [1,16]");
  const bool wide = h1 == kWH1 && h2 == kWH2;
  if (!wide && !(h1 == kH1 && h2 == kH2))
    return set_error(ODG_ERR_INVALID, "odg_policy_create_hidden: hidden widths must be (512, 256) or (1024, 512)");
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return set_error(ODG_ERR_NO_DEVICE, "no CUDA device: libodgsim has no CPU fallback");
  if (device < 0 || device >= ndev) return set_error(ODG_ERR_INVALID, "odg_policy_create: device out of range");
  DevGuard guard(device);
  OdgPolicy* p = new (std::nothrow) OdgPolicy();
  if (!p) return set_error(ODG_ERR_ALLOC, "out of host memory");
  p->device = device; p->S = state_dim; p->A = action_dim; p->K0p = (state_dim + 15) / 16 * 16; p->wide = wide;
  p->wpack_bytes = (size_t)(wide ? wide_chunk_offset(kWNumChunks, p->K0p) : chunk_offset(kNumChunks, p->K0p));
  const size_t bias_floats = wide ? kWBiasFloats : kBiasFloats;
  for (int net = 0; net < 2; net++) {
    if (cudaMalloc(&p->d_wpack[net], p->wpack_bytes) != cudaSuccess ||
        cudaMalloc(&p->d_bias[net], bias_floats * sizeof(float)) != cudaSuccess) {
      odg_policy_destroy(p); return set_error(ODG_ERR_ALLOC, "cudaMalloc(policy) failed");
    }
  }
  if (cudaMalloc(&p->d_log_std, ODG_POLICY_MAX_ACTION * sizeof(float)) != cudaSuccess) {
    odg_policy_destroy(p); return set_error(ODG_ERR_ALLOC, "cudaMalloc(policy) failed");
  }
  CUDA_TRY(cudaMemset(p->d_log_std, 0, ODG_POLICY_MAX_ACTION * sizeof(float)));
  if (wide) CUDA_TRY(cudaFuncSetAttribute(k_mlp_wide, cudaFuncAttributeMaxDynamicSharedMemorySize, kWSmemBytes));
  else CUDA_TRY(cudaFuncSetAttribute(k_mlp, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
  *out = p;
  return ODG_OK;
}

void odg_policy_destroy(OdgPolicy* p) {
  if (!p) return;
  DevGuard guard(p->device);
  for (int net = 0; net < 2; net++) { cudaFree(p->d_wpack[net]); cudaFree(p->d_bias[net]); }
  cudaFree(p->d_log_std);
  delete p;
}

int odg_policy_load(OdgPolicy* p, const OdgPolicyWeights* w, void* stream) {
  if (!p || !w) return set_error(ODG_ERR_INVALID, "odg_policy_load: null argument");
  DevGuard guard(p->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  for (int net = 0; net < 2; net++) {
    const float* const* W = net == 0 ? w->actor_w : w->critic_w;
    const float* const* B = net == 0 ? w->actor_b : w->critic_b;
    for (int i = 0; i < 3; i++) if (!W[i] || !B[i]) return set_error(ODG_ERR_INVALID, "odg_policy_load: missing weight pointer");
    const int nout = net == 0 ? p->A : 1;
    const int max_elems = kWBufBytes / 2;                            // elements of the largest chunk
    const int h1 = p->wide ? kWH1 : kH1, h2 = p->wide ? kWH2 : kH2;
    if (p->wide) k_pack_wide<<<dim3((max_elems + 255) / 256, kWNumChunks), 256, 0, st>>>(W[0], W[1], W[2], p->S, nout, p->K0p, p->d_wpack[net]);
    else k_pack<<<dim3((max_elems + 255) / 256, kNumChunks), 256, 0, st>>>(W[0], W[1], W[2], p->S, nout, p->K0p, p->d_wpack[net]);
    k_pack_bias<<<(h1 + h2 + kNOut + 255) / 256, 256, 0, st>>>(B[0], B[1], B[2], h1, h2, nout, p->d_bias[net]);
    p->launches += 2;
  }
  if (w->action_log_std)
    CUDA_TRY(cudaMemcpyAsync(p->d_log_std, w->action_log_std, p->A * sizeof(float), cudaMemcpyDeviceToDevice, st));
  CUDA_TRY(cudaGetLastError());
  return ODG_OK;
}

int odg_policy_forward(OdgPolicy* p, const float* obs_dev, int n, float* mean_dev, float* value_dev, float* action_dev,
                       float* logp_dev, uint64_t seed, uint32_t step, const uint32_t* step_base_dev,
                       int first_row_id, void* stream) {
  if (!p || !obs_dev || n < 1) return set_error(ODG_ERR_INVALID, "odg_policy_forward: bad arguments");
  DevGuard guard(p->device);
  MlpParams P;
  P.obs = obs_dev; P.n = n; P.S = p->S; P.A = p->A; P.K0p = p->K0p;
  P.wpack[0] = p->d_wpack[0]; P.wpack[1] = p->d_wpack[1]; P.bias[0] = p->d_bias[0]; P.bias[1] = p->d_bias[1];
  P.log_std = p->d_log_std; P.mean = mean_dev; P.value = value_dev; P.action = action_dev; P.logp = logp_dev;
  P.seed_lo = (uint32_t)seed; P.seed_hi = (uint32_t)(seed >> 32); P.step = step; P.step_base = step_base_dev; P.first_row = first_row_id;
  const int ctas = ((n + kM - 1) / kM + kCluster - 1) / kCluster * kCluster;       // whole clusters; surplus rows are masked
  if (p->wide) k_mlp_wide<<<ctas, kThreads, kWSmemBytes, static_cast<cudaStream_t>(stream)>>>(P);
  else k_mlp<<<ctas, kThreads, kSmemBytes, static_cast<cudaStream_t>(stream)>>>(P);
  p->launches++;
  CUDA_TRY(cudaGetLastError());
  return ODG_OK;
}

int odg_gae(const float* reward_dev, const float* value_dev, const uint8_t* done_dev, int T, int n, float gamma,
            float lambda, float* adv_dev, float* ret_dev, double* stats_dev, void* stream) {
  if (!reward_dev || !value_dev || !done_dev || !adv_dev || T < 1 || n < 1)
    return set_error(ODG_ERR_INVALID, "odg_gae: bad arguments");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int nblocks = (n + kGaeBlock - 1) / kGaeBlock;
  const int dev = device_of(reward_dev);
  if (dev < 0) return set_error(ODG_ERR_INVALID, "odg_gae: reward_dev is not device memory");
  DevGuard guard(dev);
  // per-block partial sums: a stream-ordered allocation that lives for this call only (no state shared between
  // streams, threads or devices)
  double* partial = nullptr;
  CUDA_TRY(cudaMallocAsync(&partial, (size_t)2 * nblocks * sizeof(double), st));
  k_gae<<<nblocks, kGaeBlock, 0, st>>>(reward_dev, value_dev, done_dev, T, n, gamma, lambda, adv_dev, ret_dev, partial);
  if (stats_dev) k_gae_finish<<<1, kGaeBlock, 0, st>>>(partial, nblocks, (long long)T * n, stats_dev);
  cudaError_t e = cudaGetLastError();
  cudaFreeAsync(partial, st);
  if (e != cudaSuccess) return set_error(ODG_ERR_CUDA, std::string("odg_gae: ") + cudaGetErrorString(e));
  return ODG_OK;
}

int odg_normalize_advantages(float* adv_dev, long long count, const double* stats_dev, void* stream) {
  if (!adv_dev || !stats_dev || count < 1) return set_error(ODG_ERR_INVALID, "odg_normalize_advantages: bad arguments");
  const int dev = device_of(adv_dev);
  if (dev < 0) return set_error(ODG_ERR_INVALID, "odg_normalize_advantages: adv_dev is not device memory");
  DevGuard guard(dev);
  k_adv_norm<<<(unsigned)((count + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(adv_dev, count, stats_dev);
  CUDA_TRY(cudaGetLastError());
  return ODG_OK;
}

int odg_tanh_backward_bias_scratch_floats(int cols) { return cols > 0 ? kTbGrid * cols : 0; }

int odg_tanh_backward_bias(const void* grad_y_bf16, const void* y_bf16, void* grad_x_bf16, float* bias_grad_dev,
                           float* scratch_dev, long long rows, int cols, void* stream) {
  const int groups = cols >> 3;
  if (!grad_y_bf16 || !y_bf16 || !grad_x_bf16 || !bias_grad_dev || !scratch_dev || rows < 1 || cols < 8 || (cols & 7) ||
      groups > kTbBlock || (groups & (groups - 1)))
    return set_error(ODG_ERR_INVALID, "odg_tanh_backward_bias: bad arguments (cols must be 8 x a power of two, <= 2048)");
  if (!aligned16(grad_y_bf16) || !aligned16(y_bf16) || !aligned16(grad_x_bf16))       // the kernel moves 16-byte vectors
    return set_error(ODG_ERR_INVALID, "odg_tanh_backward_bias: grad_y, y and grad_x must be 16-byte aligned");
  const int dev = device_of(grad_y_bf16);
  if (dev < 0) return set_error(ODG_ERR_INVALID, "odg_tanh_backward_bias: grad_y is not device memory");
  DevGuard guard(dev);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  k_tanh_bwd_bias<<<kTbGrid, kTbBlock, 0, st>>>(static_cast<const uint4*>(grad_y_bf16), static_cast<const uint4*>(y_bf16),
                                                static_cast<uint4*>(grad_x_bf16), scratch_dev, rows, cols);
  k_colsum_finish<<<(cols + 31) / 32, 256, 0, st>>>(scratch_dev, kTbGrid, cols, bias_grad_dev);
  CUDA_TRY(cudaGetLastError());
  return ODG_OK;
}

int odg_ppo_loss_scratch_floats(void) { return kPlMaxGrid * kPlCols; }

int odg_ppo_loss(const float* mean_dev, const float* value_dev, const float* log_std_dev, const float* action_dev,
                 const float* logp_old_dev, const float* adv_dev, const float* ret_dev, long long B, int A, float clip,
                 float vf_coef, float ent_coef, float* loss_dev, float* terms_dev, float* grad_mean_dev,
                 float* grad_value_dev, float* grad_log_std_dev, float* scratch_dev, void* stream) {
  if (!mean_dev || !value_dev || !log_std_dev || !action_dev || !logp_old_dev || !adv_dev || !ret_dev || !loss_dev ||
      !terms_dev || !grad_mean_dev || !grad_value_dev || !grad_log_std_dev || !scratch_dev || B < 1 || A < 1 || A > kPlMaxA)
    return set_error(ODG_ERR_INVALID, "odg_ppo_loss: bad arguments (1 <= act_dim <= 16)");
  const int dev = device_of(mean_dev);
  if (dev < 0) return set_error(ODG_ERR_INVALID, "odg_ppo_loss: mean_dev is not device memory");
  DevGuard guard(dev);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long want = (B + kPlBlock - 1) / kPlBlock;
  const int grid = (int)(want < kPlMaxGrid ? want : kPlMaxGrid);
  k_ppo_loss<<<grid, kPlBlock, 0, st>>>(mean_dev, value_dev, log_std_dev, action_dev, logp_old_dev, adv_dev, ret_dev, B, A,
                                        clip, vf_coef, grad_mean_dev, grad_value_dev, scratch_dev);
  k_ppo_finish<<<1, 256, 0, st>>>(scratch_dev, grid, A, log_std_dev, 1.f / (float)B, vf_coef, ent_coef, loss_dev, terms_dev,
                                  grad_log_std_dev);
  CUDA_TRY(cudaGetLastError());
  return ODG_OK;
}

int odg_tanh_bf16(const void* x_bf16, void* y_bf16, long long count, void* stream) {
  if (!x_bf16 || !y_bf16 || count < 8 || (count & 7)) return set_error(ODG_ERR_INVALID, "odg_tanh_bf16: bad arguments (count must be a multiple of 8)");
  if (!aligned16(x_bf16) || !aligned16(y_bf16))                                       // the kernel moves 16-byte vectors
    return set_error(ODG_ERR_INVALID, "odg_tanh_bf16: x and y must be 16-byte aligned");
  const int dev = device_of(x_bf16);
  if (dev < 0) return set_error(ODG_ERR_INVALID, "odg_tanh_bf16: x is not device memory");
  DevGuard guard(dev);
  const long long n16 = count >> 3, want = (n16 + 255) / 256;
  k_tanh_bf16<<<(unsigned)(want < 148 * 8 ? want : 148 * 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const uint4*>(x_bf16), static_cast<uint4*>(y_bf16), n16);
  CUDA_TRY(cudaGetLastError());
  return ODG_OK;
}

long long odg_policy_launch_count(const OdgPolicy* p) { return p ? p->launches : 0; }
#ifdef ODG_MLP_TIMING
int odg_mlp_timing(long long* out) { return cudaMemcpyFromSymbol(out, g_mlp_t, sizeof(long long) * 64) == cudaSuccess ? 0 : -1; }
#endif

}  // extern "C"
