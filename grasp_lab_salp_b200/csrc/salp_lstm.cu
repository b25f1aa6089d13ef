// salp_lstm.cu -- the rollout-side LSTM cell of RecurrentPPO on the 5th-generation tensor cores.
//
// SURVEY 2a / north_star: tensor cores "only where the batched policy MLP/LSTM forward really is a
// dense GEMM".  The MlpLstmPolicy the reference trains (src/train_robot_recurrent_ppo.py:100-105:
// lstm_hidden_size = 256, separate actor / critic LSTMs on the flattened observation) spends every
// rollout step in  gates[N, 1024] = [h * keep | obs] [N, 266] x [W_hh | W_ih]^T [266, 1024]  -- the one
// dense GEMM on the path -- followed by the element-wise cell update.  Here that is ONE kernel:
//
//   salp_lstm_pack_a_kernel   [h * keep | obs | 0] -> bf16 rows of 320 (the episode-start reset of
//                             sb3_contrib's _process_sequence is the `keep` factor)
//   salp_lstm_cell_kernel     per CTA a 128-env x (4 gates x 32 units) tile: TMA (128-byte swizzle)
//                             brings the five 64-wide K blocks of A and W through a two-stage ring of
//                             shared memory, one thread issues 20 tcgen05.mma (bf16 x bf16 -> fp32,
//                             M 128 x N 128 x K 16) into a 128-column TMEM accumulator, four warps read
//                             it back with tcgen05.ld and apply  i, f, o = sigmoid, g = tanh,
//                             c' = f c + i g, h' = o tanh(c')  in fp32 -- the gate pre-activations never
//                             reach HBM.  Three CTAs per SM (64 KB of operands, 128 TMEM columns each), so
//                             one tile's epilogue overlaps its neighbours' loads and MMAs; h' and c' are
//                             staged in the freed operand memory and leave as full 128-byte lines.
//
// The weight rows are permuted once per rollout (salp_lstm_pack_weights) so that the four gates of a
// hidden unit fall into the SAME accumulator tile: packed row t * 128 + g * 32 + u = torch row
// g * 256 + t * 32 + u (torch gate order i, f, g, o).  Operands are bf16 (weights and h rounded once,
// products exact, fp32 accumulation): |h' - fp32 torch| ~ 2-5e-3 with 1.5x-scaled default weights;
// tests/test_ppo.py states that tolerance and also compares against a float64 cell fed the same
// bf16-rounded operands (measured 3e-7, bar 2e-5).
// Measured (profiles/README.md): 18.8 us per 8192-env cell + 4.6 us for the pack, against 160 us for
// nn.LSTMCell in fp32 and 75-81 us with TF32 / bf16-autocast cuBLAS.
// Every mbarrier wait is bounded (~1 s): a broken descriptor shows as SALP_ERR_CUDA from
// salp_lstm_check(), never as a hung GPU.
#include <cuda.h>           // CUtensorMap and its enums (types only: the encoder is fetched through the runtime)
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/salp_b200.h"
#include "salp_tcgen05.cuh"

#define LSTM_H 256                       // hidden units
#define LSTM_G (4 * LSTM_H)              // gate rows
#define LSTM_KP 320                      // padded K: 256 (h) + 64 (obs, zero-padded)
#define LSTM_BM 128                      // envs per tile (UMMA M)
#define LSTM_BN 128                      // gate columns per tile (UMMA N): 4 gates x 32 units
#define LSTM_UNITS (LSTM_BN / 4)
#define LSTM_BK 64                       // bf16 per 128-byte swizzle row
#define LSTM_NKB (LSTM_KP / LSTM_BK)     // 5 K blocks through a ring of LSTM_STAGES shared-memory stages
#define LSTM_STAGES 2                    // 2 x 32 KB: three CTAs per SM, so one tile's epilogue overlaps the
                                         // loads and MMAs of its neighbours (TMEM: 3 x 128 of 512 columns)
#define LSTM_UK 16                       // K of one tcgen05.mma.kind::f16
#define LSTM_STAGE_A (LSTM_BM * LSTM_BK * 2)
#define LSTM_STAGE_B (LSTM_BN * LSTM_BK * 2)
#define LSTM_SMEM (LSTM_STAGES * (LSTM_STAGE_A + LSTM_STAGE_B) + 1024)
#define LSTM_THREADS 192                 // warp 0 TMA, warp 1 TMEM + MMA, warps 2-5 epilogue
#define LSTM_TMEM_COLS 128

__device__ int salp_lstm_status_word = 0;

// ------------------------------------------------------------------------------------------------
// packing kernels
// ------------------------------------------------------------------------------------------------
__global__ void salp_lstm_pack_weights_kernel(const float* __restrict__ w_ih, const float* __restrict__ w_hh,
                                              const float* __restrict__ b_ih, const float* __restrict__ b_hh, int D,
                                              __nv_bfloat16* __restrict__ wp, float* __restrict__ bias_p) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= LSTM_G * LSTM_KP) return;
  const int r = idx / LSTM_KP, k = idx - r * LSTM_KP;
  const int t = r / LSTM_BN, g = (r % LSTM_BN) / LSTM_UNITS, u = r % LSTM_UNITS;
  const int src = g * LSTM_H + t * LSTM_UNITS + u;
  float x = 0.f;
  if (k < LSTM_H) x = w_hh[(size_t)src * LSTM_H + k];
  else if (k - LSTM_H < D) x = w_ih[(size_t)src * D + (k - LSTM_H)];
  wp[idx] = __float2bfloat16_rn(x);
  if (k == 0) bias_p[r] = b_ih[src] + b_hh[src];
}

// one thread per 8 consecutive K entries of one (padded) env row
__global__ void salp_lstm_pack_a_kernel(const float* __restrict__ h, const float* __restrict__ obs,
                                        const uint8_t* __restrict__ starts, int64_t n, int64_t n_pad, int D,
                                        __nv_bfloat16* __restrict__ a) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  constexpr int PER_ROW = LSTM_KP / 8;
  if (idx >= n_pad * PER_ROW) return;
  const int64_t row = idx / PER_ROW;
  const int k0 = (int)(idx - row * PER_ROW) * 8;
  float x[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (row < n) {
    if (k0 < LSTM_H) {
      const float keep = (starts && starts[row]) ? 0.f : 1.f;
      const float4 p = *reinterpret_cast<const float4*>(h + row * LSTM_H + k0);
      const float4 q = *reinterpret_cast<const float4*>(h + row * LSTM_H + k0 + 4);
      x[0] = p.x * keep; x[1] = p.y * keep; x[2] = p.z * keep; x[3] = p.w * keep;
      x[4] = q.x * keep; x[5] = q.y * keep; x[6] = q.z * keep; x[7] = q.w * keep;
    } else {
#pragma unroll
      for (int j = 0; j < 8; j++) {
        const int d = k0 - LSTM_H + j;
        if (d < D) x[j] = obs[row * D + d];
      }
    }
  }
  __align__(16) __nv_bfloat162 o[4];
#pragma unroll
  for (int j = 0; j < 4; j++) o[j] = __floats2bfloat162_rn(x[2 * j], x[2 * j + 1]);
  *reinterpret_cast<uint4*>(a + row * LSTM_KP + k0) = *reinterpret_cast<const uint4*>(o);
}

// MUFU.EX2 + MUFU.RCP forms, 4-5 instructions each (ex2.approx 2 ulp, rcp.approx 1 ulp; absolute error
// of the activations ~2e-7; +-inf saturate correctly).  The libm expf / tanhf paths made the epilogue ~200
// instructions per hidden unit, __expf / __fdividef with their range fix-ups 56; this is ~30, and the
// ten MUFU per unit are then what bounds the epilogue (XU pipe).
__device__ __forceinline__ float ex2_(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float rcp_(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float sigmoidf_(float x) { return rcp_(1.f + ex2_(-1.4426950408889634f * x)); }
__device__ __forceinline__ float tanhf_(float x) { return fmaf(-2.f, rcp_(ex2_(2.8853900817779268f * x) + 1.f), 1.f); }

// ------------------------------------------------------------------------------------------------
// the cell: gates = A W^T (tcgen05), then the element-wise update from TMEM
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(LSTM_THREADS, 3)
salp_lstm_cell_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_w,
                      const float* __restrict__ bias_p, const uint8_t* __restrict__ starts,
                      const float* c_in, float* h_out, float* c_out, int64_t n) {   // (c_out may alias c_in)
  extern __shared__ uint8_t lstm_smem_raw[];
  __shared__ __align__(8) uint64_t bar_full[LSTM_STAGES];
  __shared__ __align__(8) uint64_t bar_empty[LSTM_STAGES];
  __shared__ __align__(8) uint64_t bar_acc;
  __shared__ uint32_t tmem_base_slot;
  __shared__ float bias_s[LSTM_BN];

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m0 = blockIdx.x * LSTM_BM;           // first env of the tile
  const int tile_n = blockIdx.y;                 // 32 hidden units x 4 gates
  const uint32_t smem0 = (smem_u32(lstm_smem_raw) + 1023u) & ~1023u;   // swizzle atoms want 1024-byte alignment
  const uint32_t smem_a = smem0, smem_b = smem0 + LSTM_STAGES * LSTM_STAGE_A;

  if (threadIdx.x == 0) {
    for (int s = 0; s < LSTM_STAGES; s++) {
      mbar_init(smem_u32(&bar_full[s]), 1);
      mbar_init(smem_u32(&bar_empty[s]), 1);
    }
    mbar_init(smem_u32(&bar_acc), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_slot)),
                 "r"((uint32_t)LSTM_TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (threadIdx.x >= 64) bias_s[threadIdx.x - 64] = bias_p[tile_n * LSTM_BN + (threadIdx.x - 64)];
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_slot;

  if (warp == 0) {
    if (lane == 0) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&map_a)) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&map_w)) : "memory");
      // K block kb goes to stage kb % STAGES; a stage is refilled once the MMAs that read it have
      // completed (tcgen05.commit on bar_empty).  Phase of the n-th use of a barrier: n & 1.
      for (int kb = 0; kb < LSTM_NKB; kb++) {
        const int s = kb % LSTM_STAGES;
        if (kb >= LSTM_STAGES && !mbar_wait(smem_u32(&bar_empty[s]), (uint32_t)(kb / LSTM_STAGES - 1) & 1u)) {
          atomicExch(&salp_lstm_status_word, 3);
          break;
        }
        const uint32_t bar = smem_u32(&bar_full[s]);
        mbar_expect_tx(bar, LSTM_STAGE_A + LSTM_STAGE_B);
        tma_load_2d(smem_a + s * LSTM_STAGE_A, &map_a, bar, kb * LSTM_BK, m0);
        tma_load_2d(smem_b + s * LSTM_STAGE_B, &map_w, bar, kb * LSTM_BK, tile_n * LSTM_BN);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc = umma_idesc_bf16(LSTM_BM, LSTM_BN);
      bool ok = true;
      for (int kb = 0; kb < LSTM_NKB; kb++) {
        const int s = kb % LSTM_STAGES;
        ok = mbar_wait(smem_u32(&bar_full[s]), (uint32_t)(kb / LSTM_STAGES) & 1u);
        if (!ok) break;
        tc_fence_after();
#pragma unroll
        for (int k = 0; k < LSTM_BK / LSTM_UK; k++) {
          const uint64_t da = umma_desc_sw128(smem_a + s * LSTM_STAGE_A + k * LSTM_UK * 2);
          const uint64_t db = umma_desc_sw128(smem_b + s * LSTM_STAGE_B + k * LSTM_UK * 2);
          umma_bf16(tmem, da, db, idesc, (kb | k) != 0 ? 1u : 0u);
        }
        if (kb + LSTM_STAGES < LSTM_NKB) umma_commit(smem_u32(&bar_empty[s]));   // stage s may be refilled
      }
      if (!ok) atomicExch(&salp_lstm_status_word, 1);
      umma_commit(smem_u32(&bar_acc));           // arrives when every MMA above has completed
    }
    __syncwarp();
  } else {
    // epilogue: warp w reads TMEM lanes 32 (w % 4) .. + 31 = env rows of the tile; a thread owns one env
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const int64_t e = (int64_t)m0 + row;
    const bool live = e < n;
    // the env's 32 cell states of this tile (one 128-byte line), requested BEFORE the wait for the MMAs
    const size_t off = (size_t)(live ? e : 0) * LSTM_H + (size_t)tile_n * LSTM_UNITS;
    float4 cprev[LSTM_UNITS / 4];
#pragma unroll
    for (int k = 0; k < LSTM_UNITS / 4; k++)
      cprev[k] = live ? *(reinterpret_cast<const float4*>(c_in + off) + k) : make_float4(0.f, 0.f, 0.f, 0.f);
    const float keep = (live && starts && starts[e]) ? 0.f : 1.f;
    if (!mbar_wait(smem_u32(&bar_acc), 0)) atomicExch(&salp_lstm_status_word, 2);
    tc_fence_after();
    // Every MMA has completed, so the operand stages are free: each warp stages its 32 x 32 tiles of
    // h' and c' there ([row][16-byte chunk ^ (row & 7)]: conflict-free both ways) and writes them out
    // with consecutive lanes on consecutive 16 bytes -- four full 128-byte lines per store instruction
    // instead of 32 scattered 16-byte pieces.
    float4* st_h = reinterpret_cast<float4*>(lstm_smem_raw + (smem0 - smem_u32(lstm_smem_raw))) + q * 512;
    float4* st_c = st_h + 256;
    const uint32_t t_row = tmem + ((uint32_t)(q * 32) << 16);
#pragma unroll
    for (int j = 0; j < LSTM_UNITS; j += 8) {
      float gi[8], gf[8], gg[8], go[8];
      tmem_ld8(t_row + 0 * LSTM_UNITS + j, gi);
      tmem_ld8(t_row + 1 * LSTM_UNITS + j, gf);
      tmem_ld8(t_row + 2 * LSTM_UNITS + j, gg);
      tmem_ld8(t_row + 3 * LSTM_UNITS + j, go);
      tmem_ld_wait();
      const float cp[8] = {cprev[j / 4].x,     cprev[j / 4].y,     cprev[j / 4].z,     cprev[j / 4].w,
                           cprev[j / 4 + 1].x, cprev[j / 4 + 1].y, cprev[j / 4 + 1].z, cprev[j / 4 + 1].w};
      float hn[8], cn[8];
#pragma unroll
      for (int u = 0; u < 8; u++) {
        const float i_ = sigmoidf_(gi[u] + bias_s[0 * LSTM_UNITS + j + u]);
        const float f_ = sigmoidf_(gf[u] + bias_s[1 * LSTM_UNITS + j + u]);
        const float g_ = tanhf_(gg[u] + bias_s[2 * LSTM_UNITS + j + u]);
        const float o_ = sigmoidf_(go[u] + bias_s[3 * LSTM_UNITS + j + u]);
        cn[u] = fmaf(f_, cp[u] * keep, i_ * g_);
        hn[u] = o_ * tanhf_(cn[u]);
      }
      const int ch = j / 4, sw = lane & 7;
      st_c[lane * 8 + (ch ^ sw)] = make_float4(cn[0], cn[1], cn[2], cn[3]);
      st_c[lane * 8 + ((ch + 1) ^ sw)] = make_float4(cn[4], cn[5], cn[6], cn[7]);
      st_h[lane * 8 + (ch ^ sw)] = make_float4(hn[0], hn[1], hn[2], hn[3]);
      st_h[lane * 8 + ((ch + 1) ^ sw)] = make_float4(hn[4], hn[5], hn[6], hn[7]);
    }
    __syncwarp();
#pragma unroll
    for (int it = 0; it < 8; it++) {
      const int r = it * 4 + (lane >> 3), ch = lane & 7;
      const int64_t er = (int64_t)m0 + q * 32 + r;
      if (er < n) {
        const size_t o = (size_t)er * LSTM_H + (size_t)tile_n * LSTM_UNITS + ch * 4;
        *reinterpret_cast<float4*>(h_out + o) = st_h[r * 8 + (ch ^ (r & 7))];
        *reinterpret_cast<float4*>(c_out + o) = st_c[r * 8 + (ch ^ (r & 7))];
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"((uint32_t)LSTM_TMEM_COLS) : "memory");
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
typedef CUresult (*SalpEncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static SalpEncodeTiled lstm_encoder() {
  static SalpEncodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<SalpEncodeTiled>(p);
  }
  return fn;
}
// bf16 matrix [rows, LSTM_KP] row-major, boxes of 64 (K) x 128 (rows), 128-byte swizzle
static bool lstm_make_map(CUtensorMap* map, const void* base, uint64_t rows) {
  SalpEncodeTiled enc = lstm_encoder();
  if (!enc) return false;
  const cuuint64_t dims[2] = {LSTM_KP, rows};
  const cuuint64_t strides[1] = {LSTM_KP * 2};
  const cuuint32_t box[2] = {LSTM_BK, LSTM_BM};
  const cuuint32_t estr[2] = {1, 1};
  return enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
static_assert(LSTM_BM == LSTM_BN, "one box shape serves both operands");

extern "C" {

int64_t salp_lstm_weight_bytes(void) { return (int64_t)LSTM_G * LSTM_KP * 2; }
int64_t salp_lstm_scratch_bytes(int64_t n) { return n <= 0 ? 0 : (n + LSTM_BM - 1) / LSTM_BM * LSTM_BM * LSTM_KP * 2; }

int salp_lstm_pack_weights(const float* w_ih_dev, const float* w_hh_dev, const float* b_ih_dev, const float* b_hh_dev,
                           int32_t obs_dim, int32_t hidden, void* packed_dev, float* bias_dev, void* stream) {
  if (!w_ih_dev || !w_hh_dev || !b_ih_dev || !b_hh_dev || !packed_dev || !bias_dev) return SALP_ERR_INVALID;
  if (hidden != LSTM_H || obs_dim < 1 || obs_dim > LSTM_KP - LSTM_H) return SALP_ERR_INVALID;
  const int total = LSTM_G * LSTM_KP;
  salp_lstm_pack_weights_kernel<<<(total + 255) / 256, 256, 0, (cudaStream_t)stream>>>(
      w_ih_dev, w_hh_dev, b_ih_dev, b_hh_dev, obs_dim, reinterpret_cast<__nv_bfloat16*>(packed_dev), bias_dev);
  return cudaPeekAtLastError() == cudaSuccess ? SALP_OK : SALP_ERR_CUDA;
}

int salp_lstm_cell(const void* packed_dev, const float* bias_dev, const float* obs_dev, const uint8_t* starts_dev,
                   const float* h_in_dev, const float* c_in_dev, float* h_out_dev, float* c_out_dev, void* scratch_dev,
                   int64_t n, int32_t obs_dim, int32_t hidden, void* stream) {
  if (!packed_dev || !bias_dev || !obs_dev || !h_in_dev || !c_in_dev || !h_out_dev || !c_out_dev || !scratch_dev || n <= 0)
    return SALP_ERR_INVALID;
  if (hidden != LSTM_H || obs_dim < 1 || obs_dim > LSTM_KP - LSTM_H) return SALP_ERR_INVALID;
  if (((uintptr_t)packed_dev | (uintptr_t)scratch_dev | (uintptr_t)h_in_dev | (uintptr_t)c_in_dev | (uintptr_t)h_out_dev |
       (uintptr_t)c_out_dev) & 15)
    return SALP_ERR_INVALID;
  const int64_t n_pad = (n + LSTM_BM - 1) / LSTM_BM * LSTM_BM;
  if (n_pad / LSTM_BM > 0x7fffffff) return SALP_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  static bool attr_set[64] = {};                  // (the attribute is per device)
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return SALP_ERR_CUDA;
  if (dev < 0 || dev >= 64 || !attr_set[dev]) {
    if (cudaFuncSetAttribute(salp_lstm_cell_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, LSTM_SMEM) != cudaSuccess)
      return SALP_ERR_CUDA;
    if (dev >= 0 && dev < 64) attr_set[dev] = true;
  }
  CUtensorMap map_a, map_w;
  if (!lstm_make_map(&map_a, scratch_dev, (uint64_t)n_pad) || !lstm_make_map(&map_w, packed_dev, LSTM_G)) return SALP_ERR_CUDA;
  const int64_t items = n_pad * (LSTM_KP / 8);
  salp_lstm_pack_a_kernel<<<(unsigned)((items + 255) / 256), 256, 0, s>>>(h_in_dev, obs_dev, starts_dev, n, n_pad, obs_dim,
                                                                          reinterpret_cast<__nv_bfloat16*>(scratch_dev));
  const dim3 grid((unsigned)(n_pad / LSTM_BM), LSTM_G / LSTM_BN);
  salp_lstm_cell_kernel<<<grid, LSTM_THREADS, LSTM_SMEM, s>>>(map_a, map_w, bias_dev, starts_dev, c_in_dev, h_out_dev, c_out_dev, n);
  return cudaPeekAtLastError() == cudaSuccess ? SALP_OK : SALP_ERR_CUDA;
}

/* synchronises the device; SALP_ERR_CUDA if a kernel since the last call gave up on a barrier */
int salp_lstm_check(void) {
  int w = 0;
  if (cudaDeviceSynchronize() != cudaSuccess) return SALP_ERR_CUDA;
  if (cudaMemcpyFromSymbol(&w, salp_lstm_status_word, sizeof(int)) != cudaSuccess) return SALP_ERR_CUDA;
  if (w != 0) {
    const int zero = 0;
    cudaMemcpyToSymbol(salp_lstm_status_word, &zero, sizeof(int));
    return SALP_ERR_CUDA;
  }
  return SALP_OK;
}

}  // extern "C"
