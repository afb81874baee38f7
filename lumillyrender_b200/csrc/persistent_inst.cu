// persistent_inst.cu — instantiations of the render kernel (persistent.cuh, pool.cuh).  Compiled by build.py once per
// (integrator, scene has a BVH, scene has a GGX material) triple:
//   -DLR_INST_INTEGRATOR=0|1 -DLR_INST_TREE=0|1 -DLR_INST_GGX=0|1
// The tree units also get -DLR_DIV_OUT_OF_LINE, the units for scenes without GGX get -DLR_GGX_OUT_OF_LINE (both are
// code-size decisions measured A/B, see device_path.cuh), so the eight translation units build in parallel.
//
// Which organisation runs (A/B on one box, profiles/r01_e_ab_*.txt, r02_e_sweep.txt): the pool kernel (pool.cuh) for every
// scene with a BVH — pure path tracing (sample.toml: 49.0 -> 36.3 ms) and pt-direct (welcome-2018: 50.4 -> 45.8 ms once its
// slots were fetched lazily and the far light had left the tree, bvh_build.cpp: peel_outliers) — the one-path-per-lane
// kernel (persistent.cuh) for the flat-only scenes (no phase B to feed).  The units for scenes with a BVH hold both:
// DevParams.organisation == 1 (LR_ORGANISATION=persistent, api.cpp) runs the one-path-per-lane kernel there, so that tests
// can compare the two organisations' images bit for bit.  The instrumented (COUNT) kernel is the pool kernel of the tree +
// GGX units.
#include "persistent.cuh"
#include "pool.cuh"
#if !defined(LR_INST_INTEGRATOR) || !defined(LR_INST_TREE) || !defined(LR_INST_GGX)
#error "compile with -DLR_INST_INTEGRATOR=0|1 -DLR_INST_TREE=0|1 -DLR_INST_GGX=0|1"
#endif

namespace lr {

#define LR_PASTE2(a, b, c, d) a##b##_t##c##_g##d
#define LR_PASTE(a, b, c, d) LR_PASTE2(a, b, c, d)

cudaError_t LR_PASTE(launch_render_i, LR_INST_INTEGRATOR, LR_INST_TREE, LR_INST_GGX)(
    const DevScene& sc, const DevParams& p, bool count, float* out_sum, float* out_sumsq, unsigned long long* counters,
    unsigned int* next_unit, int sm_count, cudaStream_t stream) {
  (void)count;
#if LR_INST_TREE && LR_INST_GGX
  if (count) return launch_pool_one<LR_INST_INTEGRATOR, true, true, LR_INST_GGX>(sc, p, out_sum, out_sumsq, counters, next_unit, sm_count, stream);
#endif
#if LR_INST_TREE
  if (p.organisation != 1) return launch_pool_one<LR_INST_INTEGRATOR, true, false, LR_INST_GGX>(sc, p, out_sum, out_sumsq, counters, next_unit, sm_count, stream);
#endif
  return launch_persistent_one<LR_INST_INTEGRATOR, LR_INST_TREE, false, LR_INST_GGX>(sc, p, out_sum, out_sumsq, counters, next_unit, sm_count, stream);
}

}  // namespace lr
