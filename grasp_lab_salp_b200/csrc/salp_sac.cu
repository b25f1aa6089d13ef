// salp_sac.cu -- the rollout-side SAC actor (stable-baselines3 SACPolicy, net_arch [256, 256]) in one kernel.
//
// For N envs, between two salp_step calls:
//   latent = ReLU(W2 ReLU(W1 obs + b1) + b2)                  hidden 256
//   mu = Wmu latent + bmu,  log_std = clamp(Wls latent + bls, -20, 2)
//   u = mu + exp(log_std) noise   (noise == NULL: u = mu, SB3's predict(deterministic=True))
//   a = tanh(u)                                              the scaled action the replay stores
//   env_action = low + (a + 1) / 2 (high - low)              what salp_step gets
//
// salp_sac_act_kernel: persistent CTAs (at most one per SM: ~203 KB of shared memory), each taking a
// contiguous range of 128-env tiles.  W2, packed once per weight update as a bf16 K-major image with the
// 128-byte swizzle (salp_sac_pack_weights), is copied into shared memory when a CTA starts on an agent.
// One launch serves K agents (salp_sac_act_grouped; salp_sac_act is K = 1): agent k owns env rows
// [k n, (k + 1) n) and packed image k, a tile never spans two agents, and the (agent, tile) list is
// agent-major, so a CTA's range changes agent at most a few times.  Per tile:
//   layer 1   SIMT fp32, two threads per env row (128 hidden units each): K is only obs_dim, no tile
//             for a tensor core.  W1 is read through L1 (warp-uniform addresses: broadcasts).  ReLU'd h1
//             goes to shared memory as bf16 in the swizzled A layout, then fence.proxy.async so the
//             tensor cores see it.
//   layer 2   one thread issues 16 tcgen05.mma.kind::f16 (M 128 x N 256 x K 16) into 256 TMEM columns.
//   epilogue  eight warps read TMEM back with tcgen05.ld (warp w: lanes 32 (w % 4).., columns
//             128 (w / 4)..), add b2, ReLU, and accumulate the six head dot products in fp32 against
//             Wmu / Wls in shared memory; the two column halves meet in shared memory, then clamp,
//             sample, tanh, scale.
// Layer 1 is an fmaf chain in input order starting from b1, so a test can reproduce h1 exactly.
// Only layer 2's operands are bf16.  Every mbarrier wait is bounded (~1 s): a broken descriptor shows as
// SALP_ERR_CUDA from salp_sac_check(), never as a hung GPU.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/salp_b200.h"
#include "salp_tcgen05.cuh"

#define SAC_H 256                         // hidden units of both layers
#define SAC_A 3                           // action dimension
#define SAC_MAX_D 64                      // obs_dim limit (the env gives 6 + 2 num_obstacles <= 22)
#define SAC_BM 128                        // envs per tile (UMMA M)
#define SAC_BK 64                         // bf16 per 128-byte swizzle row
#define SAC_NKB (SAC_H / SAC_BK)          // 4 K blocks
#define SAC_UK 16                         // K of one tcgen05.mma.kind::f16
#define SAC_THREADS 256
#define SAC_W2_BYTES (SAC_NKB * SAC_H * 128)    // 128 KB: 4 K blocks x 256 rows x 128 bytes
#define SAC_A_BYTES (SAC_NKB * SAC_BM * 128)    // 64 KB
#define SAC_HEADS (2 * SAC_A)                   // mu rows, then log_std rows
// fp32 part of the packed weights, after the W2 image: W1 [256, D], b1 [256], b2 [256], Wh [6, 256], bh [6]
#define SAC_F32_FLOATS(D) (SAC_H * (D) + 2 * SAC_H + SAC_HEADS * SAC_H + SAC_HEADS)
#define SAC_SMEM (SAC_W2_BYTES + SAC_A_BYTES + (SAC_HEADS * SAC_H + SAC_H + SAC_BM * SAC_HEADS + 8) * 4 + 1024)
#define SAC_TMEM_COLS 256
#define SAC_MAX_AGENTS 65535                    // grid.y of the pack kernel

__device__ int salp_sac_status_word = 0;

struct SacBox {
  float lo[SAC_A], hi[SAC_A];
};

// one thread per element of W2 (into the swizzled bf16 image) or of the fp32 part of agent blockIdx.y's image
// (parameters stacked [K, ...], images `image_bytes` apart)
__global__ void salp_sac_pack_kernel(const float* __restrict__ w1, const float* __restrict__ b1, const float* __restrict__ w2,
                                     const float* __restrict__ b2, const float* __restrict__ w_mu, const float* __restrict__ b_mu,
                                     const float* __restrict__ w_ls, const float* __restrict__ b_ls, int D, int64_t image_bytes,
                                     uint8_t* __restrict__ packed) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t ag = blockIdx.y;
  packed += ag * image_bytes;
  if (idx < SAC_H * SAC_H) {
    const int r = idx / SAC_H, k = idx % SAC_H;    // torch weight [out = r, in = k]: K-major already
    const uint32_t off = (uint32_t)(k / SAC_BK) * (SAC_H * 128) + sw128_offset(r, k % SAC_BK);
    *reinterpret_cast<__nv_bfloat16*>(packed + off) = __float2bfloat16_rn(w2[ag * SAC_H * SAC_H + idx]);
    return;
  }
  int i = idx - SAC_H * SAC_H;
  if (i >= SAC_F32_FLOATS(D)) return;
  float* f = reinterpret_cast<float*>(packed + SAC_W2_BYTES);
  const int j = i;
  float x;
  if (i < SAC_H * D) x = w1[ag * SAC_H * D + i];
  else if ((i -= SAC_H * D) < SAC_H) x = b1[ag * SAC_H + i];
  else if ((i -= SAC_H) < SAC_H) x = b2[ag * SAC_H + i];
  else if ((i -= SAC_H) < SAC_A * SAC_H) x = w_mu[ag * SAC_A * SAC_H + i];
  else if ((i -= SAC_A * SAC_H) < SAC_A * SAC_H) x = w_ls[ag * SAC_A * SAC_H + i];
  else if ((i -= SAC_A * SAC_H) < SAC_A) x = b_mu[ag * SAC_A + i];
  else x = b_ls[ag * SAC_A + i - SAC_A];
  f[j] = x;
}

__global__ void __launch_bounds__(SAC_THREADS, 1)
salp_sac_act_kernel(const uint8_t* __restrict__ packed, int64_t image_bytes, int num_agents, int D, const float* __restrict__ obs,
                    const float* __restrict__ noise, int64_t n, SacBox box, float* __restrict__ env_action,
                    float* __restrict__ scaled_action) {
  extern __shared__ uint8_t sac_smem_raw[];
  __shared__ __align__(8) uint64_t bar_acc;
  __shared__ uint32_t tmem_base_slot;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q = warp & 3, half = warp >> 2;        // TMEM lane quarter (env rows), column half
  const int row = q * 32 + lane;
  const uint32_t base = (smem_u32(sac_smem_raw) + 1023u) & ~1023u;   // swizzle atoms want 1024-byte alignment
  uint8_t* smem = sac_smem_raw + (base - smem_u32(sac_smem_raw));
  const uint32_t s_w2 = base, s_a = base + SAC_W2_BYTES;
  float* wh_s = reinterpret_cast<float*>(smem + SAC_W2_BYTES + SAC_A_BYTES);   // [6][256], then bh [6]
  float* bh_s = wh_s + SAC_HEADS * SAC_H;
  float* b2_s = bh_s + 8;
  float* part_s = b2_s + SAC_H;                                                 // [128][6]

  if (threadIdx.x == 0) {
    mbar_init(smem_u32(&bar_acc), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_slot)),
                 "r"((uint32_t)SAC_TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_slot;
  const uint32_t t_row = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(half * (SAC_H / 2));
  // this CTA's contiguous range of the agent-major (agent, tile) list
  const int64_t tiles = (n + SAC_BM - 1) / SAC_BM, total = tiles * num_agents;
  const int64_t t_begin = total * blockIdx.x / gridDim.x, t_end = total * (blockIdx.x + 1) / gridDim.x;
  const float* w1 = nullptr;
  const float* b1 = nullptr;
  int64_t agent = -1;
  bool ok = true;

  uint32_t it = 0;
  for (int64_t t = t_begin; t < t_end; t++, it++) {
    const int64_t ag = t / tiles, tile = t - ag * tiles;
    if (ag != agent) {                           // this agent's W2, b2 and heads into shared memory
      agent = ag;
      const uint8_t* img = packed + ag * image_bytes;
      w1 = reinterpret_cast<const float*>(img + SAC_W2_BYTES);
      b1 = w1 + SAC_H * D;
      __syncthreads();                           // the previous tile's epilogue is done with wh_s / b2_s
      const uint4* src = reinterpret_cast<const uint4*>(img);
      uint4* dst = reinterpret_cast<uint4*>(smem);
      for (int i = threadIdx.x; i < SAC_W2_BYTES / 16; i += SAC_THREADS) dst[i] = __ldg(src + i);
      const float* b2 = b1 + SAC_H;
      const float* wh = b2 + SAC_H;
      for (int i = threadIdx.x; i < SAC_HEADS * SAC_H; i += SAC_THREADS) wh_s[i] = wh[i];
      if (threadIdx.x < SAC_HEADS) bh_s[threadIdx.x] = wh[SAC_HEADS * SAC_H + threadIdx.x];
      b2_s[threadIdx.x] = b2[threadIdx.x];
      fence_proxy_async_smem();                  // W2 was written through the generic proxy
      __syncthreads();
    }
    const int64_t el = tile * SAC_BM + row;      // env row within the agent
    const bool live = el < n;
    const int64_t e = ag * n + el;
    // ---- layer 1: this thread's env row, hidden units 128 half .. + 127 -> bf16 A tile
    float x[SAC_MAX_D];
#pragma unroll
    for (int d = 0; d < SAC_MAX_D; d++) x[d] = (live && d < D) ? __ldg(obs + e * D + d) : 0.f;
#pragma unroll 1
    for (int j0 = half * (SAC_H / 2); j0 < (half + 1) * (SAC_H / 2); j0 += 8) {
      float acc[8];
#pragma unroll
      for (int u = 0; u < 8; u++) acc[u] = __ldg(b1 + j0 + u);
#pragma unroll
      for (int d = 0; d < SAC_MAX_D; d++) {
        if (d >= D) break;
#pragma unroll
        for (int u = 0; u < 8; u++) acc[u] = fmaf(__ldg(w1 + (j0 + u) * D + d), x[d], acc[u]);
      }
      __align__(16) __nv_bfloat162 o[4];
#pragma unroll
      for (int u = 0; u < 4; u++) o[u] = __floats2bfloat162_rn(fmaxf(acc[2 * u], 0.f), fmaxf(acc[2 * u + 1], 0.f));
      const uint32_t off = (uint32_t)(j0 / SAC_BK) * (SAC_BM * 128) + sw128_offset(row, j0 % SAC_BK);
      *reinterpret_cast<uint4*>(smem + SAC_W2_BYTES + off) = *reinterpret_cast<const uint4*>(o);
    }
    fence_proxy_async_smem();                    // h1 was written through the generic proxy
    tc_fence_before();                           // (and the previous tile's TMEM reads are done)
    __syncthreads();
    // ---- layer 2 on the tensor cores
    if (threadIdx.x == 0) {
      tc_fence_after();
      const uint32_t idesc = umma_idesc_bf16(SAC_BM, SAC_H);
#pragma unroll
      for (int kb = 0; kb < SAC_NKB; kb++) {
#pragma unroll
        for (int k = 0; k < SAC_BK / SAC_UK; k++) {
          const uint64_t da = umma_desc_sw128(s_a + kb * (SAC_BM * 128) + k * SAC_UK * 2);
          const uint64_t db = umma_desc_sw128(s_w2 + kb * (SAC_H * 128) + k * SAC_UK * 2);
          umma_bf16(tmem, da, db, idesc, (kb | k) != 0 ? 1u : 0u);
        }
      }
      umma_commit(smem_u32(&bar_acc));           // arrives when every MMA above has completed
    }
    __syncwarp();
    if (!mbar_wait(smem_u32(&bar_acc), it & 1u)) ok = false;
    tc_fence_after();
    // ---- epilogue: latent = ReLU(acc + b2) over this warp's 128 columns, six partial head sums
    float p[SAC_HEADS] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll 2
    for (int j = 0; j < SAC_H / 2; j += 8) {
      float v[8];
      tmem_ld8(t_row + j, v);
      tmem_ld_wait();
      const int c0 = half * (SAC_H / 2) + j;
#pragma unroll
      for (int u = 0; u < 8; u++) {
        const float l = fmaxf(v[u] + b2_s[c0 + u], 0.f);
#pragma unroll
        for (int h = 0; h < SAC_HEADS; h++) p[h] = fmaf(wh_s[h * SAC_H + c0 + u], l, p[h]);
      }
    }
    if (half == 1) {
#pragma unroll
      for (int h = 0; h < SAC_HEADS; h++) part_s[row * SAC_HEADS + h] = p[h];
    }
    __syncthreads();
    if (half == 0 && live) {
#pragma unroll
      for (int i = 0; i < SAC_A; i++) {
        const float mu = p[i] + part_s[row * SAC_HEADS + i] + bh_s[i];
        float u = mu;
        if (noise) {
          const float ls = fminf(fmaxf(p[SAC_A + i] + part_s[row * SAC_HEADS + SAC_A + i] + bh_s[SAC_A + i], -20.f), 2.f);
          u = fmaf(expf(ls), __ldg(noise + e * SAC_A + i), mu);
        }
        const float a = tanhf(u);
        scaled_action[e * SAC_A + i] = a;
        env_action[e * SAC_A + i] = box.lo[i] + (a + 1.f) * 0.5f * (box.hi[i] - box.lo[i]);
      }
    }
  }
  if (!ok && lane == 0) atomicExch(&salp_sac_status_word, 1);
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"((uint32_t)SAC_TMEM_COLS) : "memory");
  }
}

// the entry points run on the device that owns `ptr`, whatever device is current
namespace {
struct DeviceOf {
  int prev = -1, dev = -1;
  explicit DeviceOf(const void* ptr) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, ptr) != cudaSuccess || a.type != cudaMemoryTypeDevice) return;
    if (cudaGetDevice(&prev) != cudaSuccess) return;
    if (prev != a.device && cudaSetDevice(a.device) != cudaSuccess) return;
    dev = a.device;
  }
  ~DeviceOf() {
    if (dev >= 0 && prev != dev) cudaSetDevice(prev);
  }
};
}  // namespace

extern "C" {

int64_t salp_sac_weight_bytes(int32_t obs_dim) {
  if (obs_dim < 1 || obs_dim > SAC_MAX_D) return SALP_ERR_INVALID;
  return ((int64_t)SAC_W2_BYTES + 4 * (int64_t)SAC_F32_FLOATS(obs_dim) + 15) / 16 * 16;
}

int salp_sac_pack_weights_grouped(const float* w1, const float* b1, const float* w2, const float* b2, const float* w_mu,
                                  const float* b_mu, const float* w_log_std, const float* b_log_std, int32_t num_agents,
                                  int32_t obs_dim, void* packed_dev, void* stream) {
  if (!w1 || !b1 || !w2 || !b2 || !w_mu || !b_mu || !w_log_std || !b_log_std || !packed_dev) return SALP_ERR_INVALID;
  if (num_agents < 1 || num_agents > SAC_MAX_AGENTS) return SALP_ERR_INVALID;
  if (obs_dim < 1 || obs_dim > SAC_MAX_D || ((uintptr_t)packed_dev & 15)) return SALP_ERR_INVALID;
  DeviceOf guard(packed_dev);
  if (guard.dev < 0) return SALP_ERR_INVALID;
  const int total = SAC_H * SAC_H + SAC_F32_FLOATS(obs_dim);
  salp_sac_pack_kernel<<<dim3((total + 255) / 256, num_agents), 256, 0, (cudaStream_t)stream>>>(
      w1, b1, w2, b2, w_mu, b_mu, w_log_std, b_log_std, obs_dim, salp_sac_weight_bytes(obs_dim),
      reinterpret_cast<uint8_t*>(packed_dev));
  return cudaPeekAtLastError() == cudaSuccess ? SALP_OK : SALP_ERR_CUDA;
}

int salp_sac_pack_weights(const float* w1, const float* b1, const float* w2, const float* b2, const float* w_mu,
                          const float* b_mu, const float* w_log_std, const float* b_log_std, int32_t obs_dim,
                          void* packed_dev, void* stream) {
  return salp_sac_pack_weights_grouped(w1, b1, w2, b2, w_mu, b_mu, w_log_std, b_log_std, 1, obs_dim, packed_dev, stream);
}

int salp_sac_act_grouped(const void* packed_dev, int32_t num_agents, int32_t obs_dim, const float* obs_dev,
                         const float* noise_dev, int64_t envs_per_agent, const float* action_low, const float* action_high,
                         float* env_action_dev, float* scaled_action_dev, void* stream) {
  const int64_t n = envs_per_agent;
  if (!packed_dev || !obs_dev || !action_low || !action_high || !env_action_dev || !scaled_action_dev || n <= 0)
    return SALP_ERR_INVALID;
  if (num_agents < 1 || num_agents > SAC_MAX_AGENTS) return SALP_ERR_INVALID;
  if (obs_dim < 1 || obs_dim > SAC_MAX_D || ((uintptr_t)packed_dev & 15)) return SALP_ERR_INVALID;
  DeviceOf guard(packed_dev);
  if (guard.dev < 0 || guard.dev >= 64) return SALP_ERR_INVALID;
  static int sms[64] = {};                       // per device: SM count, and the shared-memory attribute is set
  if (!sms[guard.dev]) {
    int c = 0;
    if (cudaDeviceGetAttribute(&c, cudaDevAttrMultiProcessorCount, guard.dev) != cudaSuccess || c <= 0) return SALP_ERR_CUDA;
    if (cudaFuncSetAttribute(salp_sac_act_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SAC_SMEM) != cudaSuccess)
      return SALP_ERR_CUDA;
    sms[guard.dev] = c;
  }
  SacBox box;
  for (int i = 0; i < SAC_A; i++) {
    box.lo[i] = action_low[i];
    box.hi[i] = action_high[i];
  }
  const int64_t tiles = (n + SAC_BM - 1) / SAC_BM * num_agents;
  const unsigned grid = (unsigned)(tiles < sms[guard.dev] ? tiles : sms[guard.dev]);
  salp_sac_act_kernel<<<grid, SAC_THREADS, SAC_SMEM, (cudaStream_t)stream>>>(
      reinterpret_cast<const uint8_t*>(packed_dev), salp_sac_weight_bytes(obs_dim), num_agents, obs_dim, obs_dev, noise_dev,
      n, box, env_action_dev, scaled_action_dev);
  return cudaPeekAtLastError() == cudaSuccess ? SALP_OK : SALP_ERR_CUDA;
}

int salp_sac_act(const void* packed_dev, int32_t obs_dim, const float* obs_dev, const float* noise_dev, int64_t n,
                 const float* action_low, const float* action_high, float* env_action_dev, float* scaled_action_dev,
                 void* stream) {
  return salp_sac_act_grouped(packed_dev, 1, obs_dim, obs_dev, noise_dev, n, action_low, action_high, env_action_dev,
                              scaled_action_dev, stream);
}

/* synchronises the current device; SALP_ERR_CUDA if a kernel since the last call gave up on a barrier */
int salp_sac_check(void) {
  int w = 0;
  if (cudaDeviceSynchronize() != cudaSuccess) return SALP_ERR_CUDA;
  if (cudaMemcpyFromSymbol(&w, salp_sac_status_word, sizeof(int)) != cudaSuccess) return SALP_ERR_CUDA;
  if (w != 0) {
    const int zero = 0;
    cudaMemcpyToSymbol(salp_sac_status_word, &zero, sizeof(int));
    return SALP_ERR_CUDA;
  }
  return SALP_OK;
}

}  // extern "C"
