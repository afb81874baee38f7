// persistent.cuh — the render kernel: a persistent megakernel with deferred BVH traversal (sm_100a).
//
// K1-K7 of SURVEY.md §2 in one kernel: camera ray generation -> nearest hit -> emission / Russian roulette ->
// next-event estimation -> BSDF sample + eval -> sky lookup -> fp32 accumulation.  How a warp is organised comes
// from ncu (profiles/r01_b_*, DESIGN.md §4):
//   * in a lock-step megakernel (kernels.cu: render_kernel) the BVH node loop runs with 3.8 of 32 lanes active on
//     scenes/sample.toml: the few rays of a warp that enter the mesh take ~10x more steps than the many that only
//     see walls, and every lane waits for them at every path vertex;
//   * the kernels are instruction-fetch bound when their hot code is big: a pt-direct kernel with two inlined copies
//     of every trace stage (extension + shadow ray) stalls 5-10 cycles per issued instruction on `no_instruction`.
// So: (1) the candidates every ray tests — spheres and the flat list of large triangles (walls, floor, lights:
// bvh_build.cpp) — are tested in lock-step right where the ray is made (phase A), together with the bounds of the
// tree; a lane whose ray cannot reach the tree has its hit and goes on to its next path vertex, a lane whose ray
// can SUSPENDS; after `defer_iters` vertices, or once `defer_thresh` lanes wait, the suspended lanes traverse the
// BVH together (phase B), so the node loop runs with many lanes instead of one or two stragglers.  (2) Threads
// are persistent: a lane that finished its unit (a pixel's sample range, summed in sample order: main.rs:92-104)
// takes the next one from a global cursor, so no lane idles until the slowest pixel of its tile is done.
// (3) Extension and shadow rays share ONE call site of each trace stage, the two Material::brdf evaluations of a vertex
// share one, and the strict re-trace fallback is out of line: the hot code stays small (welcome-2018: 115 -> 84 ms).
// Specialising the kernel on the materials / camera / sky a scene contains was measured too and gave nothing.
// Per-lane arithmetic is unchanged, so every sample equals the lock-step kernel's bit for bit.
#pragma once
#include <algorithm>

#include "device_path.cuh"
#include "kernels.h"

namespace lr {

namespace pk {

constexpr unsigned kFull = 0xffffffffu;
enum { F_DEPTH_MASK = 0xffff, F_ALLOW_EMISSION = 1 << 16, F_HAS_RAY = 1 << 17, F_HAS_SHADOW = 1 << 18, F_HAS_UNIT = 1 << 20 };

LR_DEV unsigned lanemask_lt() { unsigned m; asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m)); return m; }
LR_DEV unsigned int warp_sum_u(unsigned int v) { return __reduce_add_sync(kFull, v); }

// a render kernel's counters at its end: warp sums (left in the arguments), one atomic per counter and warp
template <bool COUNT>
LR_DEV void flush_counters(unsigned long long* counters, int lane, unsigned int& n_rays, unsigned int& n_nonfinite, unsigned int& n_retrace,
                           TraceCounters& tc) {
  n_rays = warp_sum_u(n_rays);
  n_nonfinite = warp_sum_u(n_nonfinite);
  n_retrace = warp_sum_u(n_retrace);
  if (COUNT) {
    tc.nodes = warp_sum_u(tc.nodes); tc.tris = warp_sum_u(tc.tris); tc.spheres = warp_sum_u(tc.spheres);
    tc.flat_tris = warp_sum_u(tc.flat_tris); tc.flat_boxes = warp_sum_u(tc.flat_boxes);
  }
  if (lane == 0) {
    if (n_rays) atomicAdd(counters + C_RAYS, (unsigned long long)n_rays);
    if (n_nonfinite) atomicAdd(counters + C_NONFINITE, (unsigned long long)n_nonfinite);
    if (n_retrace) atomicAdd(counters + C_RETRACE, (unsigned long long)n_retrace);
    if (COUNT) {
      atomicAdd(counters + C_NODES, (unsigned long long)tc.nodes);
      atomicAdd(counters + C_TRIS, (unsigned long long)tc.tris);
      atomicAdd(counters + C_SPHERES, (unsigned long long)tc.spheres);
      atomicAdd(counters + C_FLAT_TRIS, (unsigned long long)tc.flat_tris);
      atomicAdd(counters + C_FLAT_BOXES, (unsigned long long)tc.flat_boxes);
    }
  }
}

// unit -> (split, crop-relative pixel, first sample index): the shard's 8x4 pixel tiles (or those of p.tile_list) lane by
// lane, so a warp starts on one tile
LR_DEV bool decode_unit(const DevParams& p, unsigned int u, int& lx, int& ly, int& split, int& begin) {
  const unsigned int per_split = (unsigned int)p.unit_tiles * 32u;
  split = (int)(u / per_split);
  const unsigned int r = u % per_split;
  unsigned int tile = (unsigned int)shard_tile((int)(r >> 5), p.shard, p.n_shards);
  begin = p.spp_begin;
  if (p.tile_list) {
    const int2 e = __ldg(p.tile_list + (r >> 5));
    tile = (unsigned int)e.x;
    begin = e.y;
  }
  const unsigned int lane = r & 31u;
  lx = (int)(tile % p.tiles_x) * 8 + (int)(lane & 7u);
  ly = (int)(tile / p.tiles_x) * 4 + (int)(lane >> 3);
  return lx < p.crop_w && ly < p.crop_h;
}

}  // namespace pk

// Resident CTAs per SM asked of the register allocator, by integrator and by whether the scene has a BVH (TREE).
// Measured A/B on one box (profiles/r01_c_ab_s16.txt, s17, s24): the pt-direct tree kernel is latency bound and wants
// warps (welcome-2018: 61.0 / 57.9 / 57.0 / 56.1 ms at 8 / 10 / 12 / 16 CTAs, spills and all), the flat-only pt-direct
// kernel is pure arithmetic and wants registers (brdf: 25.1 / 23.7 / 22.7 ms at 8 / 6 / 4), the pt kernels sit between.
#ifndef LR_MB_PT_TREE
#define LR_MB_PT_TREE 6
#endif
#ifndef LR_MB_PT_FLAT
#define LR_MB_PT_FLAT 8
#endif
#ifndef LR_MB_PTD_TREE
#define LR_MB_PTD_TREE 16
#endif
#ifndef LR_MB_PTD_FLAT
#define LR_MB_PTD_FLAT 4
#endif
template <int INTEGRATOR, bool TREE>
struct MinBlocks {
  static constexpr int value = INTEGRATOR == LR_INTEGRATOR_PT_DIRECT ? (TREE ? LR_MB_PTD_TREE : LR_MB_PTD_FLAT) : (TREE ? LR_MB_PT_TREE : LR_MB_PT_FLAT);
};

// TREE = false: the scene has no BVH (spheres and flat triangles only); phase B is compiled out.
// BUILD tags the translation unit's code-size choices (persistent_inst.cu: GGX inline or out of line).  It changes
// nothing inside the kernel, but it makes the instantiations of different units DIFFERENT symbols — two units defining
// the same instantiation with different macros would be merged by the linker into whichever it saw first.
template <int INTEGRATOR, bool TREE, bool COUNT, int BUILD>
__global__ void __launch_bounds__(kBlockThreads, MinBlocks<INTEGRATOR, TREE>::value)
render_persistent_kernel(const __grid_constant__ DevScene sc, const __grid_constant__ DevParams p, float* __restrict__ out_sum,
                         float* __restrict__ out_sumsq, unsigned long long* __restrict__ counters, unsigned int* __restrict__ next_unit) {
  using namespace pk;
  constexpr int NR = INTEGRATOR == LR_INTEGRATOR_PT_DIRECT ? 2 : 1;     // rays a vertex can issue: extension (+ shadow)
  const int lane = (int)(threadIdx.x & 31);
  const unsigned int n_units = render_units(p);
  const bool want_sumsq = out_sumsq != nullptr;
  // the flat list every ray gates and tests, staged into shared memory by the bulk-copy engine (device_path.cuh)
  __shared__ __align__(16) float4 flat_tab[kFlatListFloat4];
  __shared__ __align__(8) unsigned long long flat_bar;
  const FlatList flat = stage_flat_list(sc, flat_tab, &flat_bar);

  F3 o = f3(0, 0, 0), T = f3(1, 1, 1), L = f3(0, 0, 0), sum = f3(0, 0, 0), sumsq = f3(0, 0, 0);
  // the rays in flight (same origin o): 0 = extension ray, 1 = shadow ray
  F3 d0 = f3(0, 0, 1), d1 = f3(0, 0, 1);                         // directions
  float t0 = 3.0e38f, t1 = 3.0e38f;                              // nearest hit distance
  int id0 = -1, id1 = -1;                                        // ... and its primitive code
  bool pend0 = false, pend1 = false;                             // the ray still has to traverse the BVH
  float cam_g = 1.0f, cam_w = 1.0f;
  int4 un = make_int4(0, 0, 0, 0);                               // crop-relative pixel, sample index, end, split
  Pcg rng;
  rng.state = 0;
  // what the resolve of a shadow ray needs (scene.rs:127-150), kept from the vertex that issued it
  F3 q_T = f3(0, 0, 0), q_brdf = f3(0, 0, 0);
  float q_prr = 1.0f, q_point_cos = 0.0f, q_dist = 0.0f, q_sqr = 1.0f, q_pdf = 1.0f;
  int flags = 0;
  bool alive = true;
  unsigned int n_nonfinite = 0, n_retrace = 0, n_rays = 0;
  TraceCounters tc;
  tc.nodes = tc.tris = tc.spheres = tc.flat_tris = tc.flat_boxes = 0;

  while (true) {
    // ================================================================ phase A
    for (int it = 0; it < p.defer_iters; it++) {
      const bool ready = alive && !(pend0 || pend1);
      if (!__any_sync(kFull, ready)) break;
      // one path vertex for the lanes that hold a resolved hit: shade, regenerate, flat list + tree bounds for the new ray(s)
      // (a lane owns its path: the whole state stays in the lane's variables, the hooks are empty)
#define PV_LOAD_SHADOW()
#define PV_STORE_SHADOW()
#define PV_STORE_QBRDF()
#define PV_LOAD_FILM()
#define PV_STORE_FILM()
#include "path_vertex.inc"
#undef PV_LOAD_SHADOW
#undef PV_STORE_SHADOW
#undef PV_STORE_QBRDF
#undef PV_LOAD_FILM
#undef PV_STORE_FILM
      if (__popc(__ballot_sync(kFull, pend0 || pend1)) >= p.defer_thresh) break;
    }

    // ================================================================ phase B
    // the suspended rays traverse the BVH together (one call site, one node and one triangle test per iteration:
    // trav_step)
#pragma unroll 1
    for (int r = 0; TREE && r < NR; r++) {
      const bool on = r == 0 ? pend0 : pend1;
      if (!__any_sync(kFull, on)) continue;
      if (on) {
        const F3 d = r == 0 ? d0 : d1;
        const F3 inv = f3(1.0f / d.x, 1.0f / d.y, 1.0f / d.z);
        float t = r == 0 ? t0 : t1;
        int id = r == 0 ? id0 : id1;
        finish_tree_query<COUNT>(sc, o, d, inv, t, id, tc, n_retrace);
        if (r == 0) { t0 = t; id0 = id; pend0 = false; } else { t1 = t; id1 = id; pend1 = false; }
      }
    }
    if (!__any_sync(kFull, alive)) break;
  }

  flush_counters<COUNT>(counters, lane, n_rays, n_nonfinite, n_retrace, tc);
}

// One launch = the whole sample range of every unit: a persistent grid that fills the SMs.  Blocks for every unit at
// units_per_block, at most as many as are resident at once (the occupancy query's blocks per SM, or `fallback` if it fails).
inline unsigned int render_grid(const void* kernel, size_t smem, long long units_per_block, int fallback, const DevParams& p, int sm_count) {
  int nb = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kernel, kBlockThreads, smem) != cudaSuccess || nb <= 0) nb = fallback;
  const long long want = ((long long)render_units(p) + units_per_block - 1) / units_per_block;
  return (unsigned int)std::max<long long>(1, std::min<long long>(want, (long long)nb * sm_count));
}

template <int INTEGRATOR, bool TREE, bool COUNT, int BUILD>
cudaError_t launch_persistent_one(const DevScene& sc, const DevParams& p, float* out_sum, float* out_sumsq,
                                  unsigned long long* counters, unsigned int* next_unit, int sm_count, cudaStream_t stream) {
  auto kernel = render_persistent_kernel<INTEGRATOR, TREE, COUNT, BUILD>;
  const unsigned int blocks = render_grid((const void*)kernel, 0, kBlockThreads, 4, p, sm_count);     // a lane serves one unit at a time
  kernel<<<blocks, kBlockThreads, 0, stream>>>(sc, p, out_sum, out_sumsq, counters, next_unit);
  return cudaGetLastError();
}

}  // namespace lr
