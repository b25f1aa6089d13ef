// salp_pipe4_kernel.cuh -- the small-batch step kernel: four warps per 32 envs.
//
// With a few thousand envs the GPU is almost empty and one env-step costs K_max (~1340 substeps of
// the slowest env) x the time ONE warp needs per substep -- and a lone warp issues well below one
// instruction per cycle on this code (measured: 150-160 cycles for the 129 instructions of a coast
// substep, ~400 while the shape moves).  So the substep is cut along its feed-forward structure
// (salp_pipe_kernel.cuh) into four instruction streams, one warp each, each warp on its own SM
// sub-partition:
//
//   warp 3 (front)   fp64 shape chain + backward differences of substep j               -> ring 1
//   warp 2 (coefs R) rotational half of the fp32 coefficient set from ring 1           -> ring 2
//   warp 0 (dyn)     the ONLY recurrence that feeds back: (v, w, a, alpha) of substep j.  It computes
//                    the translational half of the coefficient set itself, from ring 1 -- stateless
//                    work that fills the latency shadows of the recurrence -- takes the rotational
//                    half from ring 2, and also carries the body-frame integrals (kin_body: they only
//                    need v, w).                                                        -> ring 3
//   warp 1 (kin)     Euler angles and world position from the (v, w) stream (kin_world); nothing
//                    flows back to the dynamics, so this warp simply trails the dyn warp.
//
// Measured stage costs for a lone warp (tools/ubench_substep.cu, cycles per substep): front 135-165,
// the whole coefficient set 210 (hence its split), dyn 77-100, kin 82.  (A fifth warp for half of
// the coefficient set was measured slower, 300-350 vs 250 cycles per shape-moving substep: two busy
// warps on one sub-partition cost more than the sum of their lone times.)
// Hand-off is chunk-granular (8 substeps) on named barriers with 3 / 2 / 2 chunks in flight on rings
// 1 / 2 / 3 (14 of the 16 hardware barriers).  The warps execute the functions of run_cycle_mixed
// with the same fixed 32-substep grouping of the fp32 chunk sums, and every operation is explicitly
// rounded: bit-identical with the fused kernel (tests/test_gpu_parity.py).
//
// The 32 lanes of a block end their cycles at different substeps (K is anything in 0..1348).  The
// consumer warps never test for that inside the loops: a finished lane rides along, its state having
// been put aside by predicated shared-memory stores at its last substep (p4_run_chunk below).
//
// "warp r" above is a ROLE; which hardware warp takes it is decided at the top of the body (two
// co-resident blocks per SM interleave their roles over the sub-partitions).
//
// Envs may be visited through a permutation (`order`, the K-sort).
//
// With one block per SM (<= #SMs x 32 envs) the launcher runs the 8-warp form (WIDE): four producer warps
// compute whole coefficient sets for every fourth chunk, side by side in time, and the dyn warp only loads
// them (see the producer branch below; DESIGN.md 3.2).
#pragma once
#include <type_traits>

#include "salp_pipe_kernel.cuh"

#define SALP_P4_CHUNK 8
#define SALP_P4_NBUF1 3
#define SALP_P4_NBUF2 2
#define SALP_P4_NBUF3 2
#define SALP_P4_SLOTS1 (SALP_P4_CHUNK * SALP_P4_NBUF1)
#define SALP_P4_SLOTS2 (SALP_P4_CHUNK * SALP_P4_NBUF2)
#define SALP_P4_SLOTS3 (SALP_P4_CHUNK * SALP_P4_NBUF3)
#define SALP_P4_THREADS 128
#define SALP_P4_MERGE 16

#define P4_FULL1(b) (1 + (b))
#define P4_EMPTY1(b) (1 + SALP_P4_NBUF1 + (b))
#define P4_FULL2(b) (1 + 2 * SALP_P4_NBUF1 + (b))
#define P4_EMPTY2(b) (1 + 2 * SALP_P4_NBUF1 + SALP_P4_NBUF2 + (b))
#define P4_FULL3(b) (1 + 2 * SALP_P4_NBUF1 + 2 * SALP_P4_NBUF2 + (b))
#define P4_EMPTY3(b) (1 + 2 * SALP_P4_NBUF1 + 2 * SALP_P4_NBUF2 + SALP_P4_NBUF3 + (b))

// dynamic shared memory.  Rings are stored as planes of quads, [slot][quad][lane] float4, so that the
// 32 lanes of a 128-bit access touch 512 consecutive bytes (no bank conflicts).
template <bool AXI>
struct P4Layout {
  static constexpr int Q2 = AXI ? 2 : 4;                                                       // quads per ring-2 row (rotational half)
  static constexpr size_t ring2 = 0;                                                           // [SLOTS2][Q2][32] float4
  static constexpr size_t ring1 = ring2 + sizeof(float4) * SALP_P4_SLOTS2 * Q2 * 32;           // [SLOTS1][2][32] float4
  static constexpr size_t ring3a = ring1 + sizeof(float4) * SALP_P4_SLOTS1 * 2 * 32;           // [SLOTS3][32] float4 (v0 v1 v2 w0)
  static constexpr size_t ring3b = ring3a + sizeof(float4) * SALP_P4_SLOTS3 * 32;              // [SLOTS3][32] float2 (w1 w2)
  static constexpr size_t merge = ring3b + sizeof(float2) * SALP_P4_SLOTS3 * 32;               // [MERGE][32] double
  static constexpr size_t snap = merge + sizeof(double) * SALP_P4_MERGE * 32;                  // end-of-cycle snapshots: [2 warps][5][32] float4 + [2 warps][3][32] double2
  static constexpr size_t tags = snap + 2 * (sizeof(float4) * 5 * 32 + sizeof(double2) * 3 * 32);   // [SLOTS1 + SLOTS2 + SLOTS3][32] int (checked mode)
  static constexpr size_t tile = tags + sizeof(int) * (SALP_P4_SLOTS1 + SALP_P4_SLOTS2 + SALP_P4_SLOTS3) * 32;   // [2][32][D] float
};

// The wide form (one block per SM, 8 warps): the four producer warps each compute WHOLE coefficient
// sets (shape_front + make_coefs) for every fourth chunk, into ring C: one slot of 8 rows per
// producer, rows of five quads (axisymmetric form) or seven, stored as planes of quads.  Rings 1 and
// 2 do not exist in this form, so ring C's full / empty barriers take their ids (1..8); ring 3 keeps
// its own (11..14).
#define SALP_P4W_THREADS 256
#define SALP_P4W_PRODUCERS 4
#define SALP_P4W_SLOTSC (SALP_P4_CHUNK * SALP_P4W_PRODUCERS)
#define P4W_FULLC(b) (1 + (b))
#define P4W_EMPTYC(b) (1 + SALP_P4W_PRODUCERS + (b))
static_assert(P4W_EMPTYC(SALP_P4W_PRODUCERS - 1) < P4_FULL3(0), "ring C's barriers must not reach ring 3's");
template <bool AXI>
struct P4WLayout {
  static constexpr int QC = AXI ? 5 : 7;                                                       // quads per ring-C row (whole Coef32)
  static constexpr size_t ringC = 0;                                                           // [SLOTSC][QC][32] float4
  static constexpr size_t ring3a = ringC + sizeof(float4) * SALP_P4W_SLOTSC * QC * 32;
  static constexpr size_t ring3b = ring3a + sizeof(float4) * SALP_P4_SLOTS3 * 32;
  static constexpr size_t merge = ring3b + sizeof(float2) * SALP_P4_SLOTS3 * 32;
  static constexpr size_t snap = merge + sizeof(double) * SALP_P4_MERGE * 32;
  static constexpr size_t tags = snap + 2 * (sizeof(float4) * 5 * 32 + sizeof(double2) * 3 * 32);   // [SLOTSC + SLOTS3][32] int (checked mode)
  static constexpr size_t tile = tags + sizeof(int) * (SALP_P4W_SLOTSC + SALP_P4_SLOTS3) * 32;
};
static inline size_t pipe4_smem_bytes(const SalpParams& p, bool axi, bool wide) {
  const size_t tile = sizeof(float) * 2 * 32 * (SALP_OBS_BASE + 2 * p.num_obstacles);
  if (wide) return (axi ? P4WLayout<true>::tile : P4WLayout<false>::tile) + tile;
  return (axi ? P4Layout<true>::tile : P4Layout<false>::tile) + tile;
}
// whole coefficient set of one substep, as read by dyn_step<false, false, AXI> (inv_m / inv_Iz are
// only read by the disturbance variant, which never runs in this kernel)
template <bool AXI>
__device__ __forceinline__ void coef_store_full(const Coef32& g, float4* row) {
  row[0] = make_float4(g.aj[0], g.aj[1], g.aj[2], g.com);
  row[32] = make_float4(g.kdm[0], g.kdm[1], g.xc[0], g.xc[1]);
  row[64] = make_float4(g.com_rate2, g.com_acc, g.tj1, g.tj2);
  row[96] = make_float4(g.kqI[0], g.kqI[1], g.klI[0], g.klI[1]);
  if (AXI) {
    row[128] = make_float4(g.JdI[1], g.AdI[1], 0.f, 0.f);
  } else {
    row[128] = make_float4(g.JdI[0], g.JdI[1], g.JdI[2], g.AdI[0]);
    row[160] = make_float4(g.AdI[1], g.AdI[2], g.kdm[2], g.xc[2]);
    row[192] = make_float4(g.kqI[2], g.klI[2], 0.f, 0.f);
  }
}
template <bool AXI>
__device__ __forceinline__ void coef_load_full(Coef32& g, const float4* row) {
  const float4 a = row[0], b = row[32], c = row[64], d = row[96], e = row[128];
  g.aj[0] = a.x; g.aj[1] = a.y; g.aj[2] = a.z; g.com = a.w;
  g.kdm[0] = b.x; g.kdm[1] = b.y; g.xc[0] = b.z; g.xc[1] = b.w;
  g.com_rate2 = c.x; g.com_acc = c.y; g.tj1 = c.z; g.tj2 = c.w;
  g.kqI[0] = d.x; g.kqI[1] = d.y; g.klI[0] = d.z; g.klI[1] = d.w;
  if (AXI) {
    g.JdI[1] = e.x; g.AdI[1] = e.y;
  } else {
    const float4 f = row[160], h = row[192];
    g.JdI[0] = e.x; g.JdI[1] = e.y; g.JdI[2] = e.z; g.AdI[0] = e.w;
    g.AdI[1] = f.x; g.AdI[2] = f.y; g.kdm[2] = f.z; g.xc[2] = f.w;
    g.kqI[2] = h.x; g.klI[2] = h.y;
  }
}

// Iterations j = j0..je of one hand-off chunk, for ALL lanes and without any lane test: a full chunk
// is one unrolled basic block.  Lanes whose cycle has ended (j >= K) simply keep integrating -- their
// result was put aside when they ended: each consumer warp stores its per-lane state to a snapshot
// plane in shared memory with PREDICATED stores at the lane's last iteration (j == K - 1; six
// issue slots per substep, no branch), and its fp64 totals at the flushes the lane was still alive
// for; after the loops every lane continues from its snapshot.  (Round 2 first cut the chunks at the
// substeps where lanes end -- warp-wide min of the remaining K, one segment loop per cut --, which cost
// ~20 us of a 4096-env step: tools/diag_stamps.py, profiles/r02_pipe4_clock_stamps.txt.  A lane test per
// unrolled iteration was worse still: 0.189 instead of 0.153 ms.)
// iter(j, at32): at32 = j is a multiple of the 32-substep flush interval (in an unrolled chunk only
// its last iteration can be, so the other seven stay free of branches).
template <class Iter>
__device__ __forceinline__ void p4_run_chunk(int j0, int je, Iter&& iter) {
  constexpr int C = SALP_P4_CHUNK;
  static_assert(SALP_MIXED_CHUNK % C == 0, "flush positions must fall on the last iteration of a chunk");
  if (je - j0 + 1 == C) {
#pragma unroll
    for (int u = 0; u < C; u++) iter(j0 + u, u == C - 1 && (je & (SALP_MIXED_CHUNK - 1)) == 0);
    return;
  }
#pragma unroll 1
  for (int j = j0; j <= je; j++) iter(j, (j & (SALP_MIXED_CHUNK - 1)) == 0);
}
// predicated 16-byte shared-memory store (a select-free, branch-free "if (p) *dst = v")
__device__ __forceinline__ void p4_sts128_if(bool p, void* dst, float x, float y, float z, float w) {
  asm volatile(
      "{\n\t.reg .pred q;\n\t"
      "setp.ne.b32 q, %5, 0;\n\t"
      "@q st.shared.v4.f32 [%0], {%1, %2, %3, %4};\n\t}" ::"r"((uint32_t)__cvta_generic_to_shared(dst)),
      "f"(x), "f"(y), "f"(z), "f"(w), "r"((int)p)
      : "memory");
}
__device__ __forceinline__ void p4_sts128_if(bool p, void* dst, double x, double y) {
  asm volatile(
      "{\n\t.reg .pred q;\n\t"
      "setp.ne.b32 q, %3, 0;\n\t"
      "@q st.shared.v2.f64 [%0], {%1, %2};\n\t}" ::"r"((uint32_t)__cvta_generic_to_shared(dst)),
      "d"(x), "d"(y), "r"((int)p)
      : "memory");
}

// CHECK (SALP_STEP_CHECK_HANDOFF): every ring row carries the substep index it was written for, in a
// separate tag plane; the consumer compares it with the substep it is about to use and raises
// SALP_ERR_HANDOFF otherwise.  A row read before its producer wrote it, or overwritten before its
// consumer read it, shows up as a wrong tag.  (compute-sanitizer is closed on the measurement pool;
// this is the repo's own race evidence, tests/test_gpu_parity.py.)
#define SALP_P4_FLAG_SHARED_SM 0x40000000u     // launcher-internal: more blocks than SMs, see the role assignment
#define SALP_P4_MAX_SMS 256
__device__ unsigned int salp_p4_sm_ticket[SALP_P4_MAX_SMS];
// diagnostic (tools/diag_stamps.py): with flag bit 29 the dyn warp of block 0 records clock64() at the
// boundaries of prologue / substep loops / epilogue; salp_debug_p4_stamps() reads them back
#define SALP_P4_FLAG_STAMPS 0x20000000u
__device__ long long salp_p4_stamps[16];
#define P4_STAMP(k)                                                                          \
  do {                                                                                       \
    if ((flags & SALP_P4_FLAG_STAMPS) && blockIdx.x == 0 && warp == 0 && lane == 0) salp_p4_stamps[k] = clock64(); \
  } while (0)

template <bool AXI, bool CHECK, bool WIDE>
__device__ __forceinline__ void salp_pipe4_body(const SalpParams& p, const SalpDerived& dv, const SalpView& v,
                                                const SalpStepIO& io, uint32_t flags, const int32_t* __restrict__ order,
                                                unsigned char* smem) {
  using L = std::conditional_t<WIDE, P4WLayout<AXI>, P4Layout<AXI>>;
  constexpr int Q2 = P4Layout<AXI>::Q2;
  constexpr int QC = P4WLayout<AXI>::QC;
  constexpr int C = SALP_P4_CHUNK;
  constexpr int NP = SALP_P4W_PRODUCERS;
  float4* ring1 = nullptr;
  float4* ring2 = nullptr;
  float4* ringC = nullptr;
  if constexpr (WIDE) {
    ringC = reinterpret_cast<float4*>(smem + L::ringC);
  } else {
    ring2 = reinterpret_cast<float4*>(smem + L::ring2);
    ring1 = reinterpret_cast<float4*>(smem + L::ring1);
  }
  float4* ring3a = reinterpret_cast<float4*>(smem + L::ring3a);
  float2* ring3b = reinterpret_cast<float2*>(smem + L::ring3b);
  double* merge = reinterpret_cast<double*>(smem + L::merge);
  float4* snap_dyn = reinterpret_cast<float4*>(smem + L::snap);                 // [5][32]
  float4* snap_kin = snap_dyn + 5 * 32;                                          // [5][32]
  double2* tot_dyn = reinterpret_cast<double2*>(snap_kin + 5 * 32);             // [3][32]
  double2* tot_kin = tot_dyn + 3 * 32;                                           // [3][32]
  int* tags1 = reinterpret_cast<int*>(smem + L::tags);          // (wide form: ring C's tags)
  int* tags2 = tags1 + SALP_P4_SLOTS1 * 32;
  int* tags3 = WIDE ? tags1 + SALP_P4W_SLOTSC * 32 : tags2 + SALP_P4_SLOTS2 * 32;
  float* tile = reinterpret_cast<float*>(smem + L::tile);
  const int lane = threadIdx.x & 31;
  // Role of this warp: 0 dyn, 1 kin, 2 coefs R, 3 front, one per SM sub-partition.  With two blocks
  // per SM (4737-9472 envs; flags bit 30, set by the launcher) the block that arrives second on its SM
  // rotates its roles by two, so that during the coast -- when only dyn and kin are busy -- the four
  // busy warps of the two co-resident blocks sit on four different sub-partitions: 110 instead of 185
  // cycles per coast substep.  Two things had to be measured to get there: the sub-partition of a warp
  // is its hardware slot (%warpid & 3), which for the second block on an SM is NOT threadIdx.x / 32 & 3;
  // and "second on its SM" is not blockIdx.x / #SMs & 1 once every SM holds two blocks, so the blocks
  // draw a ticket from a per-SM counter (never reset: co-resident blocks draw consecutive tickets).
  const int widx = threadIdx.x >> 5;
  int warp = widx;
  if (flags & SALP_P4_FLAG_SHARED_SM) {
    __shared__ int slot_of_warp[4];
    __shared__ unsigned ticket;
    unsigned hw, sm;
    asm volatile("mov.u32 %0, %%warpid;" : "=r"(hw));
    asm volatile("mov.u32 %0, %%smid;" : "=r"(sm));
    if (lane == 0) slot_of_warp[widx] = (int)(hw & 3u);
    if (threadIdx.x == 0) ticket = atomicAdd(&salp_p4_sm_ticket[sm & (SALP_P4_MAX_SMS - 1)], 1u);
    __syncthreads();
    const int seen = (1 << slot_of_warp[0]) | (1 << slot_of_warp[1]) | (1 << slot_of_warp[2]) | (1 << slot_of_warp[3]);
    const int base = seen == 15 ? slot_of_warp[widx] : widx;
    warp = (base + 2 * (int)(ticket & 1u)) & 3;
  }
  if constexpr (WIDE) {
    // Eight warps, two per sub-partition.  Roles by sub-partition (hardware slot %warpid & 3, as above):
    // the dyn warp shares its sub-partition with the idle warp only, so it issues alone; kin shares
    // with the other idle warp (it trails dyn at ~82 cycles per substep and must keep pace); the four
    // producers fill the other two sub-partitions.  Roles: 0 dyn, 1 kin, 2..5 producers, 6 / 7 idle.
    // If the slots do not come out two per sub-partition, the roles follow threadIdx.x instead.
    __shared__ int hw_slot[8];
    unsigned hw;
    asm volatile("mov.u32 %0, %%warpid;" : "=r"(hw));
    if (lane == 0) hw_slot[widx] = (int)(hw & 3u);
    __syncthreads();
    unsigned counts = 0;                           // four 4-bit counters, one per sub-partition
    int rank = 0;
#pragma unroll
    for (int w = 0; w < 8; w++) {
      counts += 1u << (4 * hw_slot[w]);
      if (w < widx && hw_slot[w] == hw_slot[widx]) rank++;
    }
    const bool paired = counts == 0x2222u;
    const int sub = paired ? hw_slot[widx] : (widx & 3), r = paired ? rank : (widx >> 2);
    warp = sub >= 2 ? 2 + 2 * (sub - 2) + r : (r ? 6 + sub : sub);   // {0 dyn, 6} {1 kin, 7} {2, 3} {4, 5}
  }
  const bool idle = WIDE && warp >= 2 + NP;
  const int64_t tid = (int64_t)blockIdx.x * 32 + lane;
  const bool live = tid < v.n;
  const int64_t i = live ? (order ? (int64_t)order[tid] : tid) : 0;
  P4_STAMP(0);

  // All four warps read the env's action and state themselves (reads only; every write happens in
  // the dyn warp's epilogue after the block-wide barrier) and derive the same integer plan.
  StepCtx cx;
  Body64 b;
  int Kraw = 0;
  PhasePlan pp;
  pp.k_ref = pp.k_T0 = pp.k_jet = pp.upd_a_end = pp.upd_b_begin = pp.upd_b_end = 0;
  if (live && !idle) {
    env_step_begin(p, v, io, i, cx, b);
    P4_STAMP(1);
    Kraw = plan_substeps(cx.plan, v.time_table);
    if (Kraw > 0) pp = make_phase_plan(cx.plan, v.time_table, dv.inv_dt);
  }
  const int K = Kraw > 0 ? Kraw : 0;
  const double pos0[3] = {b.pos[0], b.pos[1], b.pos[2]};
  const double ang0[3] = {b.ang[0], b.ang[1], b.ang[2]};
  // the same warp-uniform end of the shape-update part as run_cycle_mixed (updates j = 1..min(W, K))
  const int lane_end = pp.upd_a_end > pp.upd_b_end ? pp.upd_a_end : pp.upd_b_end;
  const int W = __reduce_max_sync(0xffffffffu, K > 0 ? (lane_end < K ? lane_end : K) : 0);
  const int Kw = __reduce_max_sync(0xffffffffu, K);
  const int kA = W < K ? W : K;                      // this lane's last shape update
  const int Wmax = W < Kw ? W : Kw;                  // the producers run updates j = 1..Wmax
  const int WA = Wmax < Kw - 1 ? Wmax : Kw - 1;      // substeps j = 1..K-1 exist; those <= W use g_j
  const int nch2 = (Wmax + C - 1) / C;               // chunk c = substeps c C + 1 .. (c + 1) C
  const int nch3 = Kw > 1 ? (Kw - 1 + C - 1) / C : 0;
  const float dir[3] = {(float)cx.plan.dir[0], (float)cx.plan.dir[1], (float)cx.plan.dir[2]};
  P4_STAMP(2);
  if ((flags & SALP_P4_FLAG_STAMPS) && blockIdx.x == 0 && warp == 0 && lane == 0) {
    salp_p4_stamps[8] = Kw; salp_p4_stamps[9] = Wmax; salp_p4_stamps[10] = blockDim.x;   // (blockDim: which form ran)
  }
  // ring rows of substep j (planes of quads)
  auto row1 = [&](int j) { return ring1 + (j % SALP_P4_SLOTS1) * 2 * 32 + lane; };
  auto row2 = [&](int j) { return ring2 + (j % SALP_P4_SLOTS2) * Q2 * 32 + lane; };
  auto rowC = [&](int j) { return ringC + (j % SALP_P4W_SLOTSC) * QC * 32 + lane; };
  auto put_tag = [&](int* plane, int slots, int j) { if (CHECK) plane[(j % slots) * 32 + lane] = j; };
  auto check_tag = [&](const int* plane, int slots, int j, bool mine = true) {     // mine: a row was produced for this lane
    if (CHECK && mine && plane[(j % slots) * 32 + lane] != j) raise_status(v, SALP_ERR_HANDOFF);
  };

  if (WIDE && warp >= 2) {
    // ---------------- wide form: producer f computes whole coefficient sets for chunks c = f mod NP ----------------
    // Every coefficient set depends on the action and the substep index only, so the producers work
    // side by side in time.  Each one seeds its fp64 shape track at the first substep j0 of a chunk by
    // running the two updates before it (j0 - 2 sets the centre of mass, j0 - 1 the carried rate; every
    // other field the later updates read is a pure function of t_j), with t_j from the table, which
    // holds the same chain of additions as the carried sum.  tests/test_emu_shape_seed.py checks that
    // the seeded track gives the bits of the carried one.  The seeding updates go through the same two
    // inlined shape_front calls as the others, with all their outputs live: a copy whose ShapeFront is
    // discarded was measured to contract its fp64 arithmetic differently (one ulp of the centre of
    // mass).  make_coefs is the fused kernel's arithmetic.
    if (!idle) {
      const int f = warp - 2;
      ShapeTrack st;
      if (K > 0) {
        Coef32 g0;
        mixed_init_shape<AXI>(p, dv, b, dir, st, g0);
      }
      for (int c = f; c < nch2; c += NP) {
        const int j0 = c * C + 1;
        const int je = (c + 1) * C < Wmax ? (c + 1) * C : Wmax;
        auto one = [&](double tj, int j) {
          ShapeFront fr;
          shape_front(p, dv, cx.plan, tj, j, pp.k_T0, pp.k_jet, st, fr);
          if (j >= j0) {
            Coef32 g;
            make_coefs<AXI>(dv, dir, fr, g);
            coef_store_full<AXI>(g, rowC(j));
            put_tag(tags1, SALP_P4W_SLOTSC, j);
          }
        };
        if (c >= NP) pipe_bar_sync(P4W_EMPTYC(f));
        // (a lane whose updates end at j0 - 2 or j0 - 1 seeds part-way: its last update belongs to the
        //  previous chunk, hence to another producer, whose track stays untouched)
        const int js = c > 0 ? j0 - 2 : j0;
        double tj = v.time_table[js];
        for (int j = js; j <= je; j += 2) {      // two updates per trip (independent chains, as in the front warp)
          const double tj1 = rn::dadd(tj, p.dt);
          if (j + 1 <= je && j + 1 <= kA) {
            one(tj, j);
            one(tj1, j + 1);
          } else if (j <= kA) {
            one(tj, j);
          }
          tj = rn::dadd(tj1, p.dt);
        }
        __syncwarp();
        pipe_bar_arrive(P4W_FULLC(f));
      }
      // the fp64 shape columns of a lane come from the producer that ran its last update (chunk 0's
      // producer for a lane without one)
      const int last_chunk = kA > 0 ? (kA - 1) / C : 0;
      if (K > 0 && last_chunk % NP == f) {
        mixed_finish_shape(p, st, K, b);
        merge[0 * 32 + lane] = b.length; merge[1 * 32 + lane] = b.width; merge[2 * 32 + lane] = b.prev_volume;
        merge[3 * 32 + lane] = b.prevI[0]; merge[4 * 32 + lane] = b.prevI[1];
        merge[5 * 32 + lane] = b.com; merge[6 * 32 + lane] = b.com_rate; merge[7 * 32 + lane] = b.prev_com_rate;
        merge[8 * 32 + lane] = b.com_acc;
      }
    }
  } else if (!WIDE && warp == 3) {
    // ---------------- front: fp64 shape chain + backward differences, j = 1..kA ----------------
    // ring 1 has TWO readers (coefs R and dyn): a buffer is free when both have arrived (96 threads);
    // "full" is signalled to coefs R only -- the dyn warp reads chunk c after ring 2's chunk c is full
    ShapeTrack st;
    if (K > 0) {
      Coef32 g0;
      mixed_init_shape<AXI>(p, dv, b, dir, st, g0);
    }
    double tj = v.time_table[1];                   // carried by the same additions as the table (robot.py:674)
    int j = 1;
    for (int c = 0; c < nch2; c++) {
      if (c >= SALP_P4_NBUF1) pipe_bar_sync(P4_EMPTY1(c % SALP_P4_NBUF1), 96);
      const int je = (c + 1) * C < Wmax ? (c + 1) * C : Wmax;
      // two updates per trip: consecutive updates are independent chains until their backward
      // differences (shape64_step carries nothing), so the scheduler overlaps them.  (Four per trip:
      // 134 instead of 167 cycles per update for a lone warp, but no gain in situ and slower on mixed
      // batches, where lanes whose shape motion ends inside a trip diverge.)
      while (j <= je) {
        const double tj1 = rn::dadd(tj, p.dt);
        ShapeFront f0, f1;
        if (j + 1 <= je) {
          if (j + 1 <= kA) {
            shape_front(p, dv, cx.plan, tj, j, pp.k_T0, pp.k_jet, st, f0);
            shape_front(p, dv, cx.plan, tj1, j + 1, pp.k_T0, pp.k_jet, st, f1);
            front_store(f0, row1(j));
            front_store(f1, row1(j + 1));
            put_tag(tags1, SALP_P4_SLOTS1, j);
            put_tag(tags1, SALP_P4_SLOTS1, j + 1);
          } else if (j <= kA) {
            shape_front(p, dv, cx.plan, tj, j, pp.k_T0, pp.k_jet, st, f0);
            front_store(f0, row1(j));
            put_tag(tags1, SALP_P4_SLOTS1, j);
          }
          tj = rn::dadd(tj1, p.dt);
          j += 2;
        } else {
          if (j <= kA) {
            shape_front(p, dv, cx.plan, tj, j, pp.k_T0, pp.k_jet, st, f0);
            front_store(f0, row1(j));
            put_tag(tags1, SALP_P4_SLOTS1, j);
          }
          tj = tj1;
          j += 1;
        }
      }
      __syncwarp();
      pipe_bar_arrive(P4_FULL1(c % SALP_P4_NBUF1));
    }
    if (K > 0) {
      mixed_finish_shape(p, st, K, b);
      merge[0 * 32 + lane] = b.length; merge[1 * 32 + lane] = b.width; merge[2 * 32 + lane] = b.prev_volume;
      merge[3 * 32 + lane] = b.prevI[0]; merge[4 * 32 + lane] = b.prevI[1];
      merge[5 * 32 + lane] = b.com; merge[6 * 32 + lane] = b.com_rate; merge[7 * 32 + lane] = b.prev_com_rate;
      merge[8 * 32 + lane] = b.com_acc;
    }
  } else if (!WIDE && warp == 2) {
    // ---------------- coefs R: the rotational half of the coefficient set of each ShapeFront ----------------
    auto one = [&](int j) {
      ShapeFront f;
      Coef32 g;
      front_load(f, row1(j));
      check_tag(tags1, SALP_P4_SLOTS1, j);
      make_coefs_R<AXI>(dv, dir, f, g);
      coef_store_R<AXI>(g, row2(j));
      put_tag(tags2, SALP_P4_SLOTS2, j);
    };
    int j = 1;
    for (int c = 0; c < nch2; c++) {
      pipe_bar_sync(P4_FULL1(c % SALP_P4_NBUF1));
      if (c >= SALP_P4_NBUF2) pipe_bar_sync(P4_EMPTY2(c % SALP_P4_NBUF2));
      const int je = (c + 1) * C < Wmax ? (c + 1) * C : Wmax;
      while (j <= je) {                            // two updates per trip (independent chains)
        if (j + 1 <= je) {
          if (j + 1 <= kA) { one(j); one(j + 1); }
          else if (j <= kA) one(j);
          j += 2;
        } else {
          if (j <= kA) one(j);
          j += 1;
        }
      }
      __syncwarp();
      pipe_bar_arrive(P4_EMPTY1(c % SALP_P4_NBUF1), 96);
      pipe_bar_arrive(P4_FULL2(c % SALP_P4_NBUF2));
    }
  } else if (warp == 1) {
    // ---------------- kin: Euler angles and world position from the (v, w) stream ----------------
    // kin step j uses (v, w) after dyn(j).  Step 0's input is recomputed here (g_0 and dyn(0): cheaper
    // than a one-off hand-off), steps 1..K-1 come through ring 3.  The lane's LAST step and the final
    // flush run converged after the loop, like in the fused kernel.
    Motion32 s;
    if (K > 0) {
      ShapeTrack st0;
      Coef32 g;
      mixed_init_shape<AXI>(p, dv, b, dir, st0, g);
      mixed_init_dyn(b, s);
      mixed_init_kin(b, s);
      dyn_step<false, false, AXI>(dv, g, s);
    }
    // snapshot of this warp's per-lane state (20 floats) / fp64 totals, see p4_run_chunk
    auto put_state = [&](bool pr) {
      p4_sts128_if(pr, snap_kin + 0 * 32 + lane, s.v0, s.v1, s.v2, s.w0);
      p4_sts128_if(pr, snap_kin + 1 * 32 + lane, s.w1, s.w2, s.phi_lo, s.theta_lo);
      p4_sts128_if(pr, snap_kin + 2 * 32 + lane, s.psi_lo, s.sph, s.cph, s.sth);
      p4_sts128_if(pr, snap_kin + 3 * 32 + lane, s.cth, s.sps, s.cps, s.pw0);
      p4_sts128_if(pr, snap_kin + 4 * 32 + lane, s.pw1, s.pw2, s.vw0, s.vw1);
    };
    auto put_totals = [&](bool pr) {
      p4_sts128_if(pr, tot_kin + 0 * 32 + lane, b.eul[0], b.eul[1]);
      p4_sts128_if(pr, tot_kin + 1 * 32 + lane, b.eul[2], b.pw[0]);
      p4_sts128_if(pr, tot_kin + 2 * 32 + lane, b.pw[1], b.pw[2]);
    };
    put_state(true);                                            // (a lane with K = 1 ends here)
    put_totals(true);
    // iteration j: kin step j - 1 on the (v, w) in registers, then the (v, w) of step j from the ring
    auto kin_iter = [&](int j, bool at32) {
      const float4 a = ring3a[(j % SALP_P4_SLOTS3) * 32 + lane];
      const float2 bb = ring3b[(j % SALP_P4_SLOTS3) * 32 + lane];
      check_tag(tags3, SALP_P4_SLOTS3, j);
      kin_world(dv, s);
      if (at32) {
        flush_world(b, s);
        put_totals(K > j);
      }
      s.v0 = a.x; s.v1 = a.y; s.v2 = a.z; s.w0 = a.w; s.w1 = bb.x; s.w2 = bb.y;
      put_state(j + 1 == K);
    };
    for (int c = 0; c < nch3; c++) {
      pipe_bar_sync(P4_FULL3(c % SALP_P4_NBUF3));
      p4_run_chunk(c * C + 1, (c + 1) * C < Kw - 1 ? (c + 1) * C : Kw - 1, kin_iter);
      __syncwarp();
      pipe_bar_arrive(P4_EMPTY3(c % SALP_P4_NBUF3));
    }
    if (K > 0) {
      {                                                         // continue from where this lane's cycle ended
        const float4 q0 = snap_kin[0 * 32 + lane], q1 = snap_kin[1 * 32 + lane], q2 = snap_kin[2 * 32 + lane],
                     q3 = snap_kin[3 * 32 + lane], q4 = snap_kin[4 * 32 + lane];
        s.v0 = q0.x; s.v1 = q0.y; s.v2 = q0.z; s.w0 = q0.w; s.w1 = q1.x; s.w2 = q1.y; s.phi_lo = q1.z; s.theta_lo = q1.w;
        s.psi_lo = q2.x; s.sph = q2.y; s.cph = q2.z; s.sth = q2.w; s.cth = q3.x; s.sps = q3.y; s.cps = q3.z; s.pw0 = q3.w;
        s.pw1 = q4.x; s.pw2 = q4.y; s.vw0 = q4.z; s.vw1 = q4.w;
        const double2 t0 = tot_kin[0 * 32 + lane], t1 = tot_kin[1 * 32 + lane], t2 = tot_kin[2 * 32 + lane];
        b.eul[0] = t0.x; b.eul[1] = t0.y; b.eul[2] = t1.x; b.pw[0] = t1.y; b.pw[1] = t2.x; b.pw[2] = t2.y;
      }
      kin_world(dv, s);                                         // step K - 1
      flush_world(b, s);
      merge[9 * 32 + lane] = b.eul[0]; merge[10 * 32 + lane] = b.eul[1]; merge[11 * 32 + lane] = b.eul[2];
      merge[12 * 32 + lane] = b.pw[0]; merge[13 * 32 + lane] = b.pw[1]; merge[14 * 32 + lane] = b.pw[2];
      merge[15 * 32 + lane] = (double)sqrtf(s.vw0 * s.vw0 + s.vw1 * s.vw1);
    }
  } else {
    // ---------------- dyn: the (v, w, a, alpha) recurrence + body-frame integrals ----------------
    Motion32 s;
    Coef32 g;
    if (K > 0) {
      ShapeTrack st0;
      mixed_init_shape<AXI>(p, dv, b, dir, st0, g);      // g_0 (once; cheaper than a hand-off)
      mixed_init_dyn(b, s);
      s.pos0 = s.pos1 = s.pos2 = 0.f; s.ang0 = s.ang1 = s.ang2 = 0.f;
      dyn_step<false, false, AXI>(dv, g, s);
    }
    P4_STAMP(3);
    // g_j: translational half computed here from the ShapeFront (independent of the motion state: it
    // fills the latency shadows of the recurrence), rotational half from ring 2.  Wide form: the whole
    // set from ring C.
    auto coefs_of = [&](int j) {
      if constexpr (WIDE) {
        coef_load_full<AXI>(g, rowC(j));
        check_tag(tags1, SALP_P4W_SLOTSC, j, j < K);          // (the producers stop at each lane's own K)
      } else {
        ShapeFront f;
        front_load(f, row1(j));
        coef_load_R<AXI>(g, row2(j));
        check_tag(tags1, SALP_P4_SLOTS1, j, j < K);
        check_tag(tags2, SALP_P4_SLOTS2, j, j < K);
        make_coefs_T<AXI>(dv, dir, f, g);
      }
    };
    auto wait_coefs = [&](int c) {      // (ring 1 chunk c was full before ring 2 chunk c)
      if (WIDE) pipe_bar_sync(P4W_FULLC(c % NP));
      else pipe_bar_sync(P4_FULL2(c % SALP_P4_NBUF2));
    };
    auto release_coefs = [&](int c) {
      if (WIDE) {
        pipe_bar_arrive(P4W_EMPTYC(c % NP));
      } else {
        pipe_bar_arrive(P4_EMPTY1(c % SALP_P4_NBUF1), 96);
        pipe_bar_arrive(P4_EMPTY2(c % SALP_P4_NBUF2));
      }
    };
    // snapshot of this warp's per-lane state (18 floats) / fp64 totals, see p4_run_chunk
    auto put_state = [&](bool pr) {
      p4_sts128_if(pr, snap_dyn + 0 * 32 + lane, s.v0, s.v1, s.v2, s.w0);
      p4_sts128_if(pr, snap_dyn + 1 * 32 + lane, s.w1, s.w2, s.ac0, s.ac1);
      p4_sts128_if(pr, snap_dyn + 2 * 32 + lane, s.ac2, s.al0, s.al1, s.al2);
      p4_sts128_if(pr, snap_dyn + 3 * 32 + lane, s.pos0, s.pos1, s.pos2, s.ang0);
      p4_sts128_if(pr, snap_dyn + 4 * 32 + lane, s.ang1, s.ang2, 0.f, 0.f);
    };
    auto put_totals = [&](bool pr) {
      p4_sts128_if(pr, tot_dyn + 0 * 32 + lane, b.pos[0], b.pos[1]);
      p4_sts128_if(pr, tot_dyn + 1 * 32 + lane, b.pos[2], b.ang[0]);
      p4_sts128_if(pr, tot_dyn + 2 * 32 + lane, b.ang[1], b.ang[2]);
    };
    put_state(true);                                            // (a lane with K = 1 ends here)
    put_totals(true);
    auto hand_over = [&](int j) {
      ring3a[(j % SALP_P4_SLOTS3) * 32 + lane] = make_float4(s.v0, s.v1, s.v2, s.w0);
      ring3b[(j % SALP_P4_SLOTS3) * 32 + lane] = make_float2(s.w1, s.w2);
      put_tag(tags3, SALP_P4_SLOTS3, j);
    };
    // iteration j: body-frame integrals of step j - 1, dynamics of substep j, (v, w) of step j to the ring
    auto dyn_iter_load = [&](int j, bool at32) {         // the shape is moving
      coefs_of(j);
      kin_body(dv, s);
      dyn_step<false, false, AXI>(dv, g, s);
      hand_over(j);
      if (at32) {
        flush_body(b, s);
        put_totals(K > j);
      }
      put_state(j + 1 == K);
    };
    auto dyn_iter_moving = [&](int j, bool at32) {       // the one chunk in which the warp's shape motion ends (W)
      if (j <= WA) coefs_of(j);
      kin_body(dv, s);
      dyn_step<false, false, AXI>(dv, g, s);            // (j > W: com_rate = com_acc = 0, same bits as the static form)
      hand_over(j);
      if (at32) {
        flush_body(b, s);
        put_totals(K > j);
      }
      put_state(j + 1 == K);
    };
    auto dyn_iter_static = [&](int j, bool at32) {       // the coast: coefficients stay in registers
      kin_body(dv, s);
      dyn_step<false, true, AXI>(dv, g, s);
      hand_over(j);
      if (at32) {
        flush_body(b, s);
        put_totals(K > j);
      }
      put_state(j + 1 == K);
    };
    // Three loops instead of one with per-chunk conditions (a lone warp pays ~30 cycles per branch):
    //   A  chunks whose substeps all use fresh coefficients (the shape moves),
    //   W  the chunks up to nch2 (the one in which the warp's shape motion ends; producers' last chunk),
    //   B  the coast: coefficients stay in registers, only ring 3 is fed.
    int c = 0;
    auto chunk_end = [&](int cc) { return (cc + 1) * C < Kw - 1 ? (cc + 1) * C : Kw - 1; };
    const int nA = WA / C < nch3 ? WA / C : nch3;              // chunks with je <= WA (and ring-3 traffic)
    for (; c < nA; c++) {
      wait_coefs(c);
      if (c >= SALP_P4_NBUF3) pipe_bar_sync(P4_EMPTY3(c % SALP_P4_NBUF3));
      p4_run_chunk(c * C + 1, (c + 1) * C, dyn_iter_load);
      __syncwarp();
      release_coefs(c);
      pipe_bar_arrive(P4_FULL3(c % SALP_P4_NBUF3));
    }
    for (; c < nch2; c++) {
      wait_coefs(c);
      if (c < nch3 && c >= SALP_P4_NBUF3) pipe_bar_sync(P4_EMPTY3(c % SALP_P4_NBUF3));
      p4_run_chunk(c * C + 1, chunk_end(c), dyn_iter_moving);
      __syncwarp();
      release_coefs(c);
      if (c < nch3) pipe_bar_arrive(P4_FULL3(c % SALP_P4_NBUF3));
    }
    for (; c < nch3 && c < SALP_P4_NBUF3; c++) {               // (only when the shape motion ends within the first chunks)
      p4_run_chunk(c * C + 1, chunk_end(c), dyn_iter_static);
      __syncwarp();
      pipe_bar_arrive(P4_FULL3(c % SALP_P4_NBUF3));
    }
    for (; c < nch3; c++) {
      pipe_bar_sync(P4_EMPTY3(c % SALP_P4_NBUF3));
      p4_run_chunk(c * C + 1, chunk_end(c), dyn_iter_static);
      __syncwarp();
      pipe_bar_arrive(P4_FULL3(c % SALP_P4_NBUF3));
    }
    {   // the fp64 totals as of this lane's last flush (ALL lanes: one with K = 0 rode along through its
        // neighbours' flushes too, and this warp's b goes straight into the epilogue)
      const double2 t0 = tot_dyn[0 * 32 + lane], t1 = tot_dyn[1 * 32 + lane], t2 = tot_dyn[2 * 32 + lane];
      b.pos[0] = t0.x; b.pos[1] = t0.y; b.pos[2] = t1.x; b.ang[0] = t1.y; b.ang[1] = t2.x; b.ang[2] = t2.y;
    }
    if (K > 0) {
      {                                                         // continue from where this lane's cycle ended
        const float4 q0 = snap_dyn[0 * 32 + lane], q1 = snap_dyn[1 * 32 + lane], q2 = snap_dyn[2 * 32 + lane],
                     q3 = snap_dyn[3 * 32 + lane], q4 = snap_dyn[4 * 32 + lane];
        s.v0 = q0.x; s.v1 = q0.y; s.v2 = q0.z; s.w0 = q0.w; s.w1 = q1.x; s.w2 = q1.y; s.ac0 = q1.z; s.ac1 = q1.w;
        s.ac2 = q2.x; s.al0 = q2.y; s.al1 = q2.z; s.al2 = q2.w; s.pos0 = q3.x; s.pos1 = q3.y; s.pos2 = q3.z; s.ang0 = q3.w;
        s.ang1 = q4.x; s.ang2 = q4.y;
      }
      kin_body(dv, s);                                          // step K - 1
      flush_body(b, s);
      mixed_finish_dyn(s, b);
    }
    P4_STAMP(4);
  }
  __syncthreads();
  if (warp != 0) return;
  P4_STAMP(5);
  const int D = SALP_OBS_BASE + 2 * p.num_obstacles;
  if (live) {
    double t = 0.0;
    if (K > 0) {
      b.length = merge[0 * 32 + lane]; b.width = merge[1 * 32 + lane]; b.prev_volume = merge[2 * 32 + lane];
      b.prevI[0] = merge[3 * 32 + lane]; b.prevI[1] = merge[4 * 32 + lane]; b.prevI[2] = merge[4 * 32 + lane];
      b.com = merge[5 * 32 + lane]; b.prev_com = merge[5 * 32 + lane]; b.com_rate = merge[6 * 32 + lane];
      b.prev_com_rate = merge[7 * 32 + lane]; b.com_acc = merge[8 * 32 + lane];
      b.eul[0] = merge[9 * 32 + lane]; b.eul[1] = merge[10 * 32 + lane]; b.eul[2] = merge[11 * 32 + lane];
      b.pw[0] = merge[12 * 32 + lane]; b.pw[1] = merge[13 * 32 + lane]; b.pw[2] = merge[14 * 32 + lane];
      b.speed_world = merge[15 * 32 + lane];
      t = v.time_table[K];
      b.phase = phase_at(cx.plan, t);
    }
    env_step_end(p, v, io, flags, i, cx, pos0, ang0, b, Kraw, t, tile + lane * D,
                 io.terminal_obs ? tile + (32 + lane) * D : nullptr);
  }
  __syncwarp();
  P4_STAMP(6);
  const int rows = __popc(__ballot_sync(0xffffffffu, live));     // live lanes are the low lanes
  for (int j = lane; j < 32 * D; j += 32) {                      // warp-uniform trip count (D iterations)
    const int r = j / D, k = j - r * D;
    const int64_t e = __shfl_sync(0xffffffffu, i, r);
    if (r < rows) {
      io.obs[e * D + k] = tile[j];
      if (io.terminal_obs) io.terminal_obs[e * D + k] = tile[32 * D + j];
    }
  }
  P4_STAMP(7);
}

// WIDE: the 8-warp form for one block per SM (launcher: no SALP_P4_FLAG_SHARED_SM); otherwise two
// 4-warp blocks fit an SM
template <bool CHECK, bool WIDE>
__global__ void __launch_bounds__(WIDE ? SALP_P4W_THREADS : SALP_P4_THREADS, WIDE ? 1 : 2)
salp_step_kernel_pipe4(const __grid_constant__ SalpParams p, const __grid_constant__ SalpDerived dv,
                       const __grid_constant__ SalpView v, const __grid_constant__ SalpStepIO io, uint32_t flags,
                       const int32_t* __restrict__ order) {
  extern __shared__ __align__(16) unsigned char pipe4_smem[];
  // (block-uniform: dv is a kernel argument; both forms give the same bits for axisymmetric parameters)
  if (dv.axisym) salp_pipe4_body<true, CHECK, WIDE>(p, dv, v, io, flags, order, pipe4_smem);
  else salp_pipe4_body<false, CHECK, WIDE>(p, dv, v, io, flags, order, pipe4_smem);
}
