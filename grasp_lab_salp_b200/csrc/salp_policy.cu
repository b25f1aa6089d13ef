// salp_policy.cu -- the rollout-side forward of the PPO MlpPolicy as ONE kernel (SURVEY 2a: "policy
// forward inside rollout: MLP 10 -> 64 -> 64 -> {3, 1}, FP32 SIMT; too small for tensor cores").
//
// Replaces, per env-step of a rollout, the ~20 launches of the torch forward (two 3-layer MLPs, four
// tanh, noise scaling, log-prob, clip): actor and critic weights are staged in shared memory once
// per block, one thread owns one env, both hidden layers live in registers.  Semantics follow
// stable-baselines3's MlpPolicy as ppo.MlpPolicy restates it (separate actor / critic 64-64 tanh
// networks, state-independent log_std, diagonal Gaussian; actions clipped to the Box only for the
// env):  mean = actor(obs); a = mean + noise * exp(log_std);  logp = sum(-z^2/2 - log_std - log(2 pi)/2);
// value = critic(obs).  The standard-normal `noise` is an input (the caller's torch generator keeps
// the stream reproducible and CUDA-graph capturable).
//
// Deterministic mode (SB3 predict(deterministic=True)): noise == NULL gives action = mean exactly and
// clipped = the Box clip of the mean; logp may then be NULL (not written).  value == NULL skips the
// critic (its weights are not even staged), so an evaluation pass does half the work.  With noise
// given, logp and value are mandatory and the stochastic path is the one above, unchanged.
//
// Weights arrive as ONE packed float array (ppo.MlpPolicy.packed()):
//   actor : W1 [H, D] b1 [H]  W2 [H, H] b2 [H]  W3 [A, H] b3 [A]
//   critic: W1 [H, D] b1 [H]  W2 [H, H] b2 [H]  W3 [1, H] b3 [1]
//   log_std [A]                                   (H = 64, A = 3, row-major like nn.Linear.weight)
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/salp_b200.h"

#define MLP_H 64
#define MLP_A 3

struct MlpOffsets {
  int aW1, ab1, aW2, ab2, aW3, ab3, cW1, cb1, cW2, cb2, cW3, cb3, log_std, total;
};
// PAD = 1: the packed global layout; PAD = 4: the shared-memory copy, every segment starting on a
// 16-byte boundary (the 64 x 64 layers are read with 128-bit loads)
static __host__ __device__ MlpOffsets mlp_offsets(int D, int PAD = 1) {
  MlpOffsets o;
  int p = 0;
  auto seg = [&](int& field, int count) { field = p; p += (count + PAD - 1) / PAD * PAD; };
  seg(o.aW1, MLP_H * D); seg(o.ab1, MLP_H); seg(o.aW2, MLP_H * MLP_H); seg(o.ab2, MLP_H);
  seg(o.aW3, MLP_A * MLP_H); seg(o.ab3, MLP_A);
  seg(o.cW1, MLP_H * D); seg(o.cb1, MLP_H); seg(o.cW2, MLP_H * MLP_H); seg(o.cb2, MLP_H);
  seg(o.cW3, MLP_H); seg(o.cb3, 1);
  seg(o.log_std, MLP_A);
  o.total = p;
  return o;
}
__device__ __forceinline__ void stage_segment(float* sw, const float* __restrict__ w, int dst, int src, int count) {
  for (int k = threadIdx.x; k < count; k += blockDim.x) sw[dst + k] = w[src + k];
}

// y = tanh(W2 tanh(W1 x + b1) + b2) for one thread's x; weights broadcast from shared memory
template <int MAXD>
__device__ __forceinline__ void mlp_trunk(const float* __restrict__ sw, int W1, int b1, int W2, int b2, int D,
                                          const float (&x)[MAXD], float (&h2)[MLP_H]) {
  float h1[MLP_H];
#pragma unroll
  for (int j = 0; j < MLP_H; j++) {
    float acc = sw[b1 + j];
    for (int k = 0; k < D; k++) acc = fmaf(sw[W1 + j * D + k], x[k], acc);
    h1[j] = tanhf(acc);
  }
#pragma unroll 4
  for (int j = 0; j < MLP_H; j++) {
    float acc = sw[b2 + j];
    const float4* row = reinterpret_cast<const float4*>(sw + W2 + j * MLP_H);
#pragma unroll
    for (int k = 0; k < MLP_H / 4; k++) {
      const float4 w = row[k];
      acc = fmaf(w.x, h1[4 * k], acc); acc = fmaf(w.y, h1[4 * k + 1], acc);
      acc = fmaf(w.z, h1[4 * k + 2], acc); acc = fmaf(w.w, h1[4 * k + 3], acc);
    }
    h2[j] = tanhf(acc);
  }
}

template <int MAXD>
__global__ void __launch_bounds__(128)
salp_mlp_act_kernel(const float* __restrict__ weights, const float* __restrict__ obs, const float* __restrict__ noise,
                    int64_t n, int D, float lo0, float lo1, float lo2, float hi0, float hi1, float hi2,
                    float* __restrict__ action, float* __restrict__ clipped, float* __restrict__ logp,
                    float* __restrict__ value) {
  extern __shared__ __align__(16) float sw[];
  const MlpOffsets g = mlp_offsets(D, 1), o = mlp_offsets(D, 4);
  stage_segment(sw, weights, o.aW1, g.aW1, MLP_H * D); stage_segment(sw, weights, o.ab1, g.ab1, MLP_H);
  stage_segment(sw, weights, o.aW2, g.aW2, MLP_H * MLP_H); stage_segment(sw, weights, o.ab2, g.ab2, MLP_H);
  stage_segment(sw, weights, o.aW3, g.aW3, MLP_A * MLP_H); stage_segment(sw, weights, o.ab3, g.ab3, MLP_A);
  if (value) {
    stage_segment(sw, weights, o.cW1, g.cW1, MLP_H * D); stage_segment(sw, weights, o.cb1, g.cb1, MLP_H);
    stage_segment(sw, weights, o.cW2, g.cW2, MLP_H * MLP_H); stage_segment(sw, weights, o.cb2, g.cb2, MLP_H);
    stage_segment(sw, weights, o.cW3, g.cW3, MLP_H); stage_segment(sw, weights, o.cb3, g.cb3, 1);
  }
  stage_segment(sw, weights, o.log_std, g.log_std, MLP_A);
  __syncthreads();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float x[MAXD];
#pragma unroll
  for (int k = 0; k < MAXD; k++) x[k] = k < D ? obs[i * D + k] : 0.f;
  float h[MLP_H];
  // actor
  mlp_trunk<MAXD>(sw, o.aW1, o.ab1, o.aW2, o.ab2, D, x, h);
  const float lo[3] = {lo0, lo1, lo2}, hi[3] = {hi0, hi1, hi2};
  float lp = 0.f;
#pragma unroll
  for (int a = 0; a < MLP_A; a++) {
    float m = sw[o.ab3 + a];
#pragma unroll
    for (int k = 0; k < MLP_H; k++) m = fmaf(sw[o.aW3 + a * MLP_H + k], h[k], m);
    float act = m;                                         // deterministic: the mean itself
    if (noise) {
      const float ls = sw[o.log_std + a];
      const float z = noise[i * MLP_A + a];
      act = fmaf(z, expf(ls), m);
      lp += -0.5f * z * z - ls - 0.918938533204672742f;    // log(2 pi) / 2
    }
    action[i * MLP_A + a] = act;
    clipped[i * MLP_A + a] = fminf(fmaxf(act, lo[a]), hi[a]);
  }
  if (logp) logp[i] = lp;
  if (!value) return;
  // critic
  mlp_trunk<MAXD>(sw, o.cW1, o.cb1, o.cW2, o.cb2, D, x, h);
  float v = sw[o.cb3];
#pragma unroll
  for (int k = 0; k < MLP_H; k++) v = fmaf(sw[o.cW3 + k], h[k], v);
  value[i] = v;
}

extern "C" {

int64_t salp_mlp_packed_size(int32_t obs_dim) { return mlp_offsets(obs_dim).total; }

int salp_mlp_act(const float* weights_dev, int32_t obs_dim, const float* obs_dev, const float* noise_dev, int64_t n,
                 const float* action_low, const float* action_high, float* action_dev, float* clipped_dev,
                 float* logp_dev, float* value_dev, void* stream) {
  if (!weights_dev || !obs_dev || !action_dev || !clipped_dev || n <= 0 || !action_low || !action_high)
    return SALP_ERR_INVALID;
  if (noise_dev && (!logp_dev || !value_dev)) return SALP_ERR_INVALID;    // the rollout needs both
  if (obs_dim < 1 || obs_dim > SALP_OBS_BASE + 2 * SALP_MAX_OBSTACLES) return SALP_ERR_INVALID;
  const MlpOffsets o = mlp_offsets(obs_dim, 4);
  const size_t smem = sizeof(float) * (size_t)o.total;
  const unsigned grid = (unsigned)((n + 127) / 128);
  cudaStream_t s = (cudaStream_t)stream;
  if (obs_dim <= 10) {
    if (smem > 48 * 1024 &&
        cudaFuncSetAttribute(salp_mlp_act_kernel<10>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
      return SALP_ERR_CUDA;
    salp_mlp_act_kernel<10><<<grid, 128, smem, s>>>(weights_dev, obs_dev, noise_dev, n, obs_dim, action_low[0], action_low[1],
                                                     action_low[2], action_high[0], action_high[1], action_high[2], action_dev,
                                                     clipped_dev, logp_dev, value_dev);
  } else {
    if (smem > 48 * 1024 &&
        cudaFuncSetAttribute(salp_mlp_act_kernel<22>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
      return SALP_ERR_CUDA;
    salp_mlp_act_kernel<22><<<grid, 128, smem, s>>>(weights_dev, obs_dev, noise_dev, n, obs_dim, action_low[0], action_low[1],
                                                     action_low[2], action_high[0], action_high[1], action_high[2], action_dev,
                                                     clipped_dev, logp_dev, value_dev);
  }
  return cudaPeekAtLastError() == cudaSuccess ? SALP_OK : SALP_ERR_CUDA;
}

}  // extern "C"
