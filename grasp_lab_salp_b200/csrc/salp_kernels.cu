// salp_kernels.cu -- __global__ kernels and their launchers (sm_100a).
//
// One thread per environment, state columns in HBM (SoA, coalesced), the whole breathing cycle
// of an env in registers.  Kernel arguments (SalpParams, SalpView, SalpStepIO) are
// __grid_constant__: they sit in the constant bank and every access is a uniform c[][] operand.
#include "salp_step_kernel.cuh"
#include "salp_pipe4_kernel.cuh"

__global__ void salp_init_kernel(const __grid_constant__ SalpParams p, const __grid_constant__ SalpView v) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < v.n) env_init(p, v, i);
}

__global__ void salp_reset_kernel(const __grid_constant__ SalpParams p, const __grid_constant__ SalpView v,
                                  const uint8_t* __restrict__ mask, float* __restrict__ obs) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= v.n) return;
  if (mask && !mask[i]) return;
  const int D = SALP_OBS_BASE + 2 * p.num_obstacles;
  env_reset(p, v, i, obs ? obs + i * D : nullptr);
}

__global__ void salp_trace_kernel(const __grid_constant__ SalpParams p, const __grid_constant__ SalpView v, int64_t env,
                                  float a0, float a1, float a2, double* trace, int capacity, int32_t* K_out) {
  if (threadIdx.x == 0 && blockIdx.x == 0) *K_out = env_trace_cycle(p, v, env, a0, a1, a2, trace, capacity);
}

// ---- K-sort: balance warps by substep count (SURVEY.md hard part 3) ----------------------------
// salp_plan_kernel recomputes the cycle plan of every env (cheap: one inverse-kinematics solve)
// and histograms the sort key (K bucket, end of shape motion); salp_scan_kernel turns the histogram into descending-K offsets;
// salp_scatter_kernel writes the env permutation.  The step kernel then walks `order`.
__global__ void salp_plan_kernel(const __grid_constant__ SalpParams p, const __grid_constant__ SalpView v,
                                 const float* __restrict__ actions, int32_t* __restrict__ Kout,
                                 int32_t* __restrict__ hist) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= v.n) return;
  Cols c{v, i};
  CyclePlan plan = make_cycle_plan(p, actions[3 * i], actions[3 * i + 1], actions[3 * i + 2],
                                   c.d(SALP_F_NOZZLE_ANGLE1), c.d(SALP_F_NOZZLE_ANGLE2));
  int K = plan_substeps(plan, v.time_table);
  K = K < 0 ? SALP_MAX_SUBSTEPS : K;
  const int key = sort_key(K, make_phase_plan(plan, v.time_table, 1.0 / p.dt));
  Kout[i] = key;
  atomicAdd(&hist[key], 1);
}

// one block of 1024 threads; bins 0..SALP_SORT_BINS-1; offsets for DESCENDING key (long cycles first)
__global__ void salp_scan_kernel(int32_t* __restrict__ hist) {
  __shared__ int32_t part[1024];
  constexpr int NB = SALP_SORT_BINS;
  constexpr int PER = (NB + 1023) / 1024;
  int tid = threadIdx.x;
  int32_t local[PER];
  int32_t sum = 0;
#pragma unroll
  for (int j = 0; j < PER; j++) {
    int bin = NB - 1 - (tid * PER + j);          // reversed: thread 0 owns the largest K
    int32_t h = bin >= 0 ? hist[bin] : 0;
    local[j] = sum;
    sum += h;
  }
  part[tid] = sum;
  __syncthreads();
  for (int off = 1; off < 1024; off <<= 1) {
    int32_t x = tid >= off ? part[tid - off] : 0;
    __syncthreads();
    part[tid] += x;
    __syncthreads();
  }
  int32_t base = tid ? part[tid - 1] : 0;
#pragma unroll
  for (int j = 0; j < PER; j++) {
    int bin = NB - 1 - (tid * PER + j);
    if (bin >= 0) hist[bin] = base + local[j];
  }
}

__global__ void salp_scatter_kernel(int64_t n, const int32_t* __restrict__ K, int32_t* __restrict__ offsets,
                                    int32_t* __restrict__ order) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int32_t slot = atomicAdd(&offsets[K[i]], 1);
  order[slot] = (int32_t)i;
}

#define SALP_LAUNCH_CHECK()                                  \
  do {                                                       \
    if (cudaPeekAtLastError() != cudaSuccess) return SALP_ERR_CUDA; \
  } while (0)

int salp_launch_init(const SalpParams& p, const SalpView& v, cudaStream_t stream) {
  salp_init_kernel<<<grid_for(v.n, 128), 128, 0, stream>>>(p, v);
  SALP_LAUNCH_CHECK();
  return 1;
}

int salp_launch_reset(const SalpParams& p, const SalpView& v, const uint8_t* mask, float* obs,
                      cudaStream_t stream) {
  salp_reset_kernel<<<grid_for(v.n, 128), 128, 0, stream>>>(p, v, mask, obs);
  SALP_LAUNCH_CHECK();
  return 1;
}

int salp_launch_trace(const SalpParams& p, const SalpView& v, int64_t env, const float action[3], double* trace,
                      int capacity, int32_t* K_out, cudaStream_t stream) {
  salp_trace_kernel<<<1, 32, 0, stream>>>(p, v, env, action[0], action[1], action[2], trace, capacity, K_out);
  SALP_LAUNCH_CHECK();
  return 1;
}

int salp_launch_step(const SalpParams& p, const SalpView& v, const SalpStepIO& io, uint32_t flags,
                     const SalpScratch& scratch, cudaStream_t stream, const char** kernel_name) {
  int launches = 0;
  const char* dummy;
  const char*& name = kernel_name ? *kernel_name : dummy;
  const int32_t* order = nullptr;
  SalpDerived dv = make_derived(p);
  if (flags & SALP_STEP_GENERIC) dv.axisym = 0;      // the general form of the loop even for axisymmetric coefficient sets
  if (flags & SALP_STEP_SORT_BY_K) {
    if (cudaMemsetAsync(scratch.hist, 0, sizeof(int32_t) * SALP_SORT_BINS, stream) != cudaSuccess)
      return SALP_ERR_CUDA;
    salp_plan_kernel<<<grid_for(v.n, 128), 128, 0, stream>>>(p, v, io.actions, scratch.K, scratch.hist);
    salp_scan_kernel<<<1, 1024, 0, stream>>>(scratch.hist);
    salp_scatter_kernel<<<grid_for(v.n, 256), 256, 0, stream>>>(v.n, scratch.K, scratch.hist, scratch.order);
    SALP_LAUNCH_CHECK();
    launches += 3;
    order = scratch.order;
  }
  const int block = block_for(v.n);
  // Small batches: the warp-specialised pipeline kernel (salp_pipe4_kernel.cuh), natural or K-sorted
  // order, unless SALP_STEP_FUSED asks for the one-warp kernel.  Up to one 32-env block per SM (4736
  // envs) it is 1.39x faster than the fused kernel (131.5 vs 182.8 us per uniform-random step, L2 warm);
  // with two co-resident blocks per SM, the second one with rotated warp roles, still 1.20x at 6144,
  // 1.16x at 8192 and 1.06x at 9472 envs (the producers of the two blocks share sub-partitions while the
  // shape moves): used up to two full blocks per SM, 64 envs.  A third block does not fit the register
  // file.  SALP_PIPE_BLOCKS_PER_SM=1 restores the one-block limit, SALP_PIPE_ENVS_PER_SM moves the upper
  // one (experiment switches).
  const int sms = v.sm_count > 0 ? v.sm_count : 148;
  const bool pipe_ok = p.precision == SALP_PRECISION_MIXED && p.randomization == 0 && !(flags & SALP_STEP_FUSED);
  static const int pipe_blocks_per_sm = [] { const char* e = getenv("SALP_PIPE_BLOCKS_PER_SM"); return e ? atoi(e) : 2; }();
  static const int pipe_envs_per_sm = [] { const char* e = getenv("SALP_PIPE_ENVS_PER_SM"); return e ? atoi(e) : 64; }();
  const int64_t pipe_max_envs = (int64_t)sms * (pipe_blocks_per_sm >= 2 ? pipe_envs_per_sm : 32);
  if (pipe_ok && v.n <= pipe_max_envs) {
    static bool configured4[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64 || !configured4[dev]) {
      SalpParams widest = p;
      widest.num_obstacles = SALP_MAX_OBSTACLES;
      const int bytes = (int)pipe4_smem_bytes(widest, false, false);
      const int bytes_wide = (int)pipe4_smem_bytes(widest, false, true);
      if (cudaFuncSetAttribute(salp_step_kernel_pipe4<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes) != cudaSuccess ||
          cudaFuncSetAttribute(salp_step_kernel_pipe4<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes) != cudaSuccess ||
          cudaFuncSetAttribute(salp_step_kernel_pipe4<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes_wide) != cudaSuccess ||
          cudaFuncSetAttribute(salp_step_kernel_pipe4<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes_wide) != cudaSuccess)
        return SALP_ERR_CUDA;
      if (dev >= 0 && dev < 64) configured4[dev] = true;
    }
    // One block per SM (<= #SMs blocks): the 8-warp form, whose four producer warps hand the dyn warp
    // whole coefficient sets (salp_pipe4_kernel.cuh).  SALP_PIPE_WIDE=0 forces the 4-warp form there
    // (experiment switch; read at every launch so that one process can compare the two).
    const bool shared_sm = grid_for(v.n, 32) > sms;
    const char* wide_env = getenv("SALP_PIPE_WIDE");
    const bool wide = !shared_sm && !(wide_env && atoi(wide_env) == 0);
    const uint32_t pflags = (flags & 0x3fffffffu) | (shared_sm ? SALP_P4_FLAG_SHARED_SM : 0u);
    const dim3 grid((unsigned)grid_for(v.n, 32));
    const size_t smem = pipe4_smem_bytes(p, dv.axisym != 0, wide);
    const bool check = (flags & SALP_STEP_CHECK_HANDOFF) != 0;   // (a separate kernel: the production one keeps its register allocation)
    if (wide && check)
      salp_step_kernel_pipe4<true, true><<<grid, SALP_P4W_THREADS, smem, stream>>>(p, dv, v, io, pflags, order);
    else if (wide)
      salp_step_kernel_pipe4<false, true><<<grid, SALP_P4W_THREADS, smem, stream>>>(p, dv, v, io, pflags, order);
    else if (check)
      salp_step_kernel_pipe4<true, false><<<grid, SALP_P4_THREADS, smem, stream>>>(p, dv, v, io, pflags, order);
    else
      salp_step_kernel_pipe4<false, false><<<grid, SALP_P4_THREADS, smem, stream>>>(p, dv, v, io, pflags, order);
    name = "salp_step_kernel_pipe4";
    SALP_LAUNCH_CHECK();
    return launches + 1;
  }
  if (p.precision == SALP_PRECISION_F64) {
    salp_launch_step_f64(p, v, io, flags, order, stream);     // salp_step_f64.cu (compiled with -fmad=false)
    name = "salp_step_kernel<F64>";
  } else if (p.randomization != 0) {   // default-off robustness switches: separate instantiation
    salp_step_kernel_lat<SALP_PRECISION_MIXED_RANDOMIZED><<<grid_for(v.n, 32), 32, lat_tile_bytes(p), stream>>>(p, dv, v, io, flags, order);
    name = "salp_step_kernel_lat<MIXED_RANDOMIZED>";
  } else if (block == 32) {
    salp_step_kernel_lat<SALP_PRECISION_MIXED><<<grid_for(v.n, 32), 32, lat_tile_bytes(p), stream>>>(p, dv, v, io, flags, order);
    name = "salp_step_kernel_lat<MIXED>";
  } else {
    salp_step_kernel<SALP_PRECISION_MIXED><<<grid_for(v.n, block), block, 0, stream>>>(p, dv, v, io, flags, order);
    name = "salp_step_kernel<MIXED>";
  }
  SALP_LAUNCH_CHECK();
  return launches + 1;
}

// ---- FP32 pipe probe (roofline denominator; SURVEY.md 8d) -------------------------------------
__global__ void __launch_bounds__(256) salp_ffma_probe_kernel(float* out, int iters, float a, float b) {
  float x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
  for (int i = 0; i < iters; i++) {
#pragma unroll
    for (int u = 0; u < 16; u++) {
      x0 = fmaf(x0, a, b); x1 = fmaf(x1, a, b); x2 = fmaf(x2, a, b); x3 = fmaf(x3, a, b);
      x4 = fmaf(x4, a, b); x5 = fmaf(x5, a, b); x6 = fmaf(x6, a, b); x7 = fmaf(x7, a, b);
    }
  }
  float s = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
  if (s == 12345.678f) out[0] = s;     // never true; keeps the chains alive
}

int salp_launch_ffma_probe(float* scratch, int blocks, int iters, cudaStream_t stream) {
  salp_ffma_probe_kernel<<<blocks, 256, 0, stream>>>(scratch, iters, 0.999f, 0.001f);
  SALP_LAUNCH_CHECK();
  return 1;
}

// Diagnostic (tools/diag_stamps.py): the clock64() stamps block 0's dyn warp took in the last pipeline
// step launched with flag bit 29 (salp_pipe4_kernel.cuh: P4_STAMP), plus K_max and W of that block.
extern "C" int salp_debug_p4_stamps(long long* out16) {
  if (!out16) return SALP_ERR_INVALID;
  if (cudaDeviceSynchronize() != cudaSuccess) return SALP_ERR_CUDA;
  return cudaMemcpyFromSymbol(out16, salp_p4_stamps, sizeof(long long) * 16) == cudaSuccess ? SALP_OK : SALP_ERR_CUDA;
}
