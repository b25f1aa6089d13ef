// shape_seed_check.cu -- TEST INFRASTRUCTURE ONLY (tests/test_emu_shape_seed.py).
//
// The wide form of the pipeline kernel (salp_pipe4_kernel.cuh) has several producer warps that each
// start the fp64 shape track at the first substep j0 of a chunk, by running shape_front for j0 - 2 and
// j0 - 1 from a track that carries nothing, instead of carrying the track from substep 1.  This host
// build of the same shape_front checks, for one action, that the seeded track gives the bits of the
// carried one: every field the later updates and mixed_finish_shape read, and every ShapeFront from j0
// to the end of the updates.  It also checks that the time table holds the carried chain of additions.
#include <cstring>
#include <vector>

#include "../../grasp_lab_salp_b200/csrc/salp_env.cuh"

constexpr int kChunk = 8;                  // SALP_P4_CHUNK: the kernel's hand-off chunk

static bool same(double a, double b) { return memcmp(&a, &b, sizeof a) == 0; }
static bool same_track(const ShapeTrack& a, const ShapeTrack& b) {
  return same(a.s.V, b.s.V) && same(a.s.I0, b.s.I0) && same(a.s.I1, b.s.I1) && same(a.s.com, b.s.com) &&
         same(a.s.com_rate, b.s.com_rate) && same(a.prev_com_rate, b.prev_com_rate) && same(a.dl, b.dl) &&
         same(a.prevV, b.prevV) && same(a.I0_prev_used, b.I0_prev_used) && same(a.I1_prev_used, b.I1_prev_used);
}

extern "C" {
// Returns the number of mismatches (0: seeded == carried everywhere); out[0..5] = K, k_T0, k_jet,
// kA, number of seeding points checked, number of ShapeFronts compared.  last_update = -1: the lane's
// own end of shape motion; otherwise updates run up to min(last_update, K) (a warp neighbour's W).
int salp_seed_check(const SalpParams* p, float a0, float a1, float a2, int last_update, int* out) {
  std::vector<double> table(SALP_MAX_SUBSTEPS + 1);
  volatile double acc = 0.0;
  for (int k = 0; k <= SALP_MAX_SUBSTEPS; k++) { table[k] = acc; acc = acc + p->dt; }
  const SalpDerived dv = make_derived(*p);
  const CyclePlan plan = make_cycle_plan(*p, a0, a1, a2, 0.0, 0.0);
  const int K = plan_substeps(plan, table.data());
  if (K <= 0) { out[0] = K; return 0; }
  const PhasePlan pp = make_phase_plan(plan, table.data(), dv.inv_dt);
  const int lane_end = pp.upd_a_end > pp.upd_b_end ? pp.upd_a_end : pp.upd_b_end;
  const int W = last_update < 0 ? lane_end : last_update;
  const int kA = W < K ? W : K;
  out[0] = K; out[1] = pp.k_T0; out[2] = pp.k_jet; out[3] = kA; out[4] = 0; out[5] = 0;
  int bad = 0;
  // the carried track and its state after every update j (index j)
  std::vector<ShapeTrack> after(kA + 1);
  std::vector<ShapeFront> front(kA + 1);
  ShapeTrack st;
  memset(&st, 0, sizeof st);
  double tj = table[1];
  for (int j = 1; j <= kA; j++) {
    if (!same(tj, table[j])) bad++;
    shape_front(*p, dv, plan, tj, j, pp.k_T0, pp.k_jet, st, front[j]);
    after[j] = st;
    tj = rn::dadd(tj, p->dt);
  }
  // seeding points: every chunk start of the kernel, plus both sides of the phase edges and of kA
  std::vector<int> seeds;
  for (int j0 = kChunk + 1; j0 <= kA; j0 += kChunk) seeds.push_back(j0);
  const int edges[] = {pp.k_T0, pp.k_jet, kA};
  for (int e : edges)
    for (int d = -2; d <= 2; d++) seeds.push_back(e + d);
  for (int j0 : seeds) {
    if (j0 < 3 || j0 > kA) continue;
    ShapeTrack s2;
    memset(&s2, 0xff, sizeof s2);              // nothing carried: every field the seeding does not set is NaN
    ShapeFront d;
    shape_front(*p, dv, plan, table[j0 - 2], j0 - 2, pp.k_T0, pp.k_jet, s2, d);
    shape_front(*p, dv, plan, table[j0 - 1], j0 - 1, pp.k_T0, pp.k_jet, s2, d);
    if (!same_track(s2, after[j0 - 1])) bad++;
    out[4]++;
    double t = table[j0];
    for (int j = j0; j <= kA; j++) {
      ShapeFront f;
      shape_front(*p, dv, plan, t, j, pp.k_T0, pp.k_jet, s2, f);
      if (memcmp(&f, &front[j], sizeof f) != 0) bad++;
      out[5]++;
      t = rn::dadd(t, p->dt);
    }
    // the end state the producer owning the last update hands to mixed_finish_shape
    if (!same_track(s2, after[kA]) || !same(s2.com_acc, after[kA].com_acc) || s2.last_update != after[kA].last_update) bad++;
  }
  return bad;
}
}  // extern "C"
