// pool.cuh — the render kernel as a persistent megakernel over a per-warp POOL of paths in shared memory (sm_100a).
//
// Same per-path arithmetic as persistent.cuh (K1-K7 of SURVEY.md §2, every statement citing the same reference lines),
// different scheduling.  In persistent.cuh a lane owns ONE path: a lane whose ray has to traverse the BVH idles until
// `defer_thresh` lanes wait, and the BVH phase then runs with those ~12 lanes, of which 4 are active per instruction
// (profiles/r01_d_phaseB_histograms.txt) — 39 % of the kernel's warp instructions at an eighth of the SIMD width.
// Here a warp owns LR_POOL_SLOTS (64) paths whose whole state lives in shared memory (structure of arrays, one word
// column per field), and lanes are bound to paths only for the length of one step:
//   * phase A (one path vertex): the lanes take up to 32 slots whose nearest hit is known — shade it (sky / emission /
//     Russian roulette / NEE / BSDF sample), regenerate finished paths from the unit cursor, and test the new ray(s)
//     against spheres + flat list + the bounds of the tree; a ray that can reach the tree marks its slot PENDING;
//   * phase B: the lanes take up to 32 pending rays (extension or shadow) and traverse the BVH together.
// With twice as many paths as lanes one of the two kinds of work always has >= 32 items (pigeonhole), so both phases
// start at full width whatever fraction of the rays reaches the tree.  A path's unit (a pixel's sample range) is
// summed in its slot in sample order (main.rs:92-104) and its RNG stream is a function of (seed, pixel, sample), so
// every sample — and the image — equals persistent.cuh's bit for bit, whichever lane ran which step.
#pragma once
#include "device_path.cuh"
#include "kernels.h"
#include "persistent.cuh"

namespace lr {

// Tunables, each settled by A/B runs on one box (profiles/r01_e_ab_s39.txt, s43-s49): paths per warp (64, 96 or 128: no gain
// beyond 64), pending rays that start a BVH phase (24: slower, 48: same), resident CTAs per SM asked of the register
// allocator (pt: 4..8 within 3 %, 6 = 80 registers; pt-direct: 6 since the vertex fetches its shadow and film records where
// it uses them — with the whole 42-word slot live across the vertex it needed 125 registers).
#ifndef LR_POOL_SLOTS
#define LR_POOL_SLOTS 64
#endif
// pt-direct slots hold the shadow-ray record too (42 words against 26): 48 of them per warp keep a CTA at 32 KB, so that
// six CTAs (24 warps) fit an SM's 227 KB like the pt build's; 64 leave room for five
#ifndef LR_POOL_SLOTS_PTD
#define LR_POOL_SLOTS_PTD 48
#endif
#ifndef LR_POOL_BSTART
#define LR_POOL_BSTART 32
#endif
#ifndef LR_PMB_PT_TREE
#define LR_PMB_PT_TREE 6
#endif
#ifndef LR_PMB_PTD_TREE
#define LR_PMB_PTD_TREE 6
#endif

namespace pl {

// word columns of a slot
enum {
  W_OX = 0, W_OY, W_OZ, W_DX, W_DY, W_DZ, W_T0, W_ID0, W_TX, W_TY, W_TZ, W_LX, W_LY, W_LZ, W_SX, W_SY, W_SZ,
  W_CAMG, W_CAMW, W_UNX, W_UNY, W_UNZ, W_UNW, W_RNGLO, W_RNGHI, W_FLAGS, W_PT_COUNT,
  W_D1X = W_PT_COUNT, W_D1Y, W_D1Z, W_T1, W_ID1, W_QTX, W_QTY, W_QTZ, W_QBX, W_QBY, W_QBZ, W_QPRR, W_QPC, W_QDIST, W_QSQR, W_QPDF,
  W_PTD_COUNT
};

// paths per warp: more than the 32 lanes (that is the point), a multiple of 16; the last mask word may be partly used
template <int INTEGRATOR>
__host__ __device__ constexpr int slots() { return INTEGRATOR == LR_INTEGRATOR_PT_DIRECT ? LR_POOL_SLOTS_PTD : LR_POOL_SLOTS; }
static_assert(LR_POOL_SLOTS % 16 == 0 && LR_POOL_SLOTS >= 48 && LR_POOL_SLOTS <= 128, "a warp's pool holds 48 .. 128 paths");
static_assert(LR_POOL_SLOTS_PTD % 8 == 0 && LR_POOL_SLOTS_PTD >= 40 && LR_POOL_SLOTS_PTD <= 128, "a warp's pool holds 40 .. 128 paths");
template <int INTEGRATOR>
__host__ __device__ constexpr int mask_words() { return (slots<INTEGRATOR>() + 31) / 32; }     // mask words per kind of work

template <int INTEGRATOR>
__host__ __device__ constexpr int words_per_slot(bool want_sumsq) {
  return (INTEGRATOR == LR_INTEGRATOR_PT_DIRECT ? (int)W_PTD_COUNT : (int)W_PT_COUNT) + (want_sumsq ? 3 : 0);
}
template <int INTEGRATOR>
__host__ __device__ constexpr int warp_words(bool want_sumsq) { return words_per_slot<INTEGRATOR>(want_sumsq) * slots<INTEGRATOR>() + 32; }   // + the selection list

// Takes the first `quota` set bits of the concatenation words[rot] | words[rot + 1] | ... (cyclic): their codes
// word * 32 + bit go to list[0, n) in that order, the bits are cleared in `words`.  Returns n (warp-uniform).  Lane j
// looks after bit j of every word: it scatters the code to the bit's rank, and a ballot over "my bit is taken" is the
// mask of taken bits.  `rot` (warp-uniform, < N) moves the starting word so that no part of the pool is always served
// last — a starved slot would still hold most of its unit when the units run out, and the warp would finish it alone.
// The caller reads list and then calls __syncwarp() before the next selection.
template <int N>
LR_DEV int select_take(int* list, int lane, unsigned (&words)[N], int quota, int rot) {
  const unsigned lt = pk::lanemask_lt();
  const unsigned bit = 1u << lane;
  int base = 0;
#pragma unroll
  for (int r = 0; r < N; r++) {
    if (r != rot) continue;                              // warp-uniform: one of the N unrolled orders runs
#pragma unroll
    for (int k = 0; k < N; k++) {
      const int i = (k + r) % N;                         // compile-time
      const unsigned w = words[i];
      const int rank = base + __popc(w & lt);
      const bool mine = (w & bit) != 0u && rank < quota;
      if (mine) list[rank] = i * 32 + lane;
      words[i] = w & ~__ballot_sync(pk::kFull, mine);
      base += __popc(w);
    }
  }
  __syncwarp();
  return min(base, quota);
}

}  // namespace pl

template <int INTEGRATOR, bool TREE>
struct PoolMinBlocks {
  static_assert(TREE, "the pool kernel is built for scenes with a BVH only (persistent_inst.cu)");
  static constexpr int value = INTEGRATOR == LR_INTEGRATOR_PT_DIRECT ? LR_PMB_PTD_TREE : LR_PMB_PT_TREE;
};

template <int INTEGRATOR, bool TREE, bool COUNT, int BUILD>
__global__ void __launch_bounds__(kBlockThreads, PoolMinBlocks<INTEGRATOR, TREE>::value)
render_pool_kernel(const __grid_constant__ DevScene sc, const __grid_constant__ DevParams p, float* __restrict__ out_sum,
                   float* __restrict__ out_sumsq, unsigned long long* __restrict__ counters, unsigned int* __restrict__ next_unit) {
  using namespace pk;
  using namespace pl;
  constexpr int NR = INTEGRATOR == LR_INTEGRATOR_PT_DIRECT ? 2 : 1;     // rays a vertex can issue: extension (+ shadow)
  constexpr int NS = slots<INTEGRATOR>();
  constexpr int kWords = mask_words<INTEGRATOR>();
  // the flat list every ray gates and tests, staged into shared memory by the bulk-copy engine (device_path.cuh)
  __shared__ __align__(16) float4 flat_tab[kFlatListFloat4];
  __shared__ __align__(8) unsigned long long flat_bar;
  const FlatList flat = stage_flat_list(sc, flat_tab, &flat_bar);
  extern __shared__ float pool_smem[];
  const int lane = (int)(threadIdx.x & 31);
  const unsigned int n_units = render_units(p);
  const bool want_sumsq = out_sumsq != nullptr;
  float* const pool = pool_smem + (threadIdx.x >> 5) * warp_words<INTEGRATOR>(want_sumsq);
  int* const list = (int*)(pool + words_per_slot<INTEGRATOR>(want_sumsq) * NS);
  constexpr int W_SQ = NR == 2 ? (int)W_PTD_COUNT : (int)W_PT_COUNT;    // sumsq columns, present only on request
#define SLF(w) pool[(w) * NS + s]
#define SLI(w) ((int*)pool)[(w) * NS + s]

  // every slot starts fresh: no unit, no ray -> its first step fetches a unit and makes a camera ray
  for (int s = lane; s < NS; s += 32) SLI(W_FLAGS) = 0;
  __syncwarp();

  // slot states (warp-uniform): ray r of slot s still has to traverse the BVH (pend[r * kWords + s / 32]); slot is
  // dead (no units left).  A slot that is neither is READY: its nearest hit is known.
  unsigned pend[NR * kWords], dead[kWords];
#pragma unroll
  for (int i = 0; i < NR * kWords; i++) pend[i] = 0u;
#pragma unroll
  for (int i = 0; i < kWords; i++) dead[i] = (i + 1) * 32 <= NS ? 0u : ~0u << (NS - i * 32);   // slots beyond NS do not exist
  unsigned int n_nonfinite = 0, n_retrace = 0, n_rays = 0;
  TraceCounters tc;
  tc.nodes = tc.tris = tc.spheres = tc.flat_tris = tc.flat_boxes = 0;
  int rot_a = 0, rot_b = 0;

  while (true) {
    unsigned rdy[kWords];
    int nA = 0, nB = 0;
#pragma unroll
    for (int i = 0; i < kWords; i++) {
      rdy[i] = ~(pend[i] | (NR == 2 ? pend[(NR - 1) * kWords + i] : 0u) | dead[i]);
      nA += __popc(rdy[i]);
    }
#pragma unroll
    for (int i = 0; i < NR * kWords; i++) nB += __popc(pend[i]);
    if (nA + nB == 0) break;

    if (!TREE || !(nB >= LR_POOL_BSTART || nB >= nA)) {
      // ================================================================ phase A: one path vertex of up to 32 slots
      const int n_sel = select_take<kWords>(list, lane, rdy, 32, rot_a);
      rot_a = rot_a + 1 == kWords ? 0 : rot_a + 1;
      const bool ready = lane < n_sel;
      const int s = ready ? list[lane] : 0;
      __syncwarp();
      bool alive = true;
      bool pend0 = false, pend1 = false;

      F3 o = f3(0, 0, 0), T = f3(1, 1, 1), L = f3(0, 0, 0), sum = f3(0, 0, 0), sumsq = f3(0, 0, 0);
      F3 d0 = f3(0, 0, 1), d1 = f3(0, 0, 1);
      float t0 = 3.0e38f, t1 = 3.0e38f;
      int id0 = -1, id1 = -1;
      float cam_g = 1.0f, cam_w = 1.0f;
      int4 un = make_int4(0, 0, 0, 0);
      Pcg rng;
      rng.state = 0;
      F3 q_T = f3(0, 0, 0), q_brdf = f3(0, 0, 0);
      float q_prr = 1.0f, q_point_cos = 0.0f, q_dist = 0.0f, q_sqr = 1.0f, q_pdf = 1.0f;
      int flags = 0;
      // the state every vertex needs: ray, hit, throughput, radiance, RNG, flags.  The shadow-ray record (16 words) and the
      // film record (pixel sums, unit, camera weights: 12-15 words) are fetched by the vertex code where it needs them
      // (PV_LOAD_* hooks below) and are not live across the surface / light-sample / BSDF code in between
      if (ready) {
        o = f3(SLF(W_OX), SLF(W_OY), SLF(W_OZ));
        d0 = f3(SLF(W_DX), SLF(W_DY), SLF(W_DZ));
        t0 = SLF(W_T0); id0 = SLI(W_ID0);
        T = f3(SLF(W_TX), SLF(W_TY), SLF(W_TZ));
        L = f3(SLF(W_LX), SLF(W_LY), SLF(W_LZ));
        rng.state = (unsigned long long)(unsigned int)SLI(W_RNGLO) | ((unsigned long long)(unsigned int)SLI(W_RNGHI) << 32);
        flags = SLI(W_FLAGS);
      }
#define PV_LOAD_SHADOW()                                                                                                  \
  do {                                                                                                                    \
    d1 = f3(SLF(W_D1X), SLF(W_D1Y), SLF(W_D1Z));                                                                          \
    t1 = SLF(W_T1); id1 = SLI(W_ID1);                                                                                     \
    q_T = f3(SLF(W_QTX), SLF(W_QTY), SLF(W_QTZ));                                                                         \
    q_brdf = f3(SLF(W_QBX), SLF(W_QBY), SLF(W_QBZ));                                                                      \
    q_prr = SLF(W_QPRR); q_point_cos = SLF(W_QPC); q_dist = SLF(W_QDIST); q_sqr = SLF(W_QSQR); q_pdf = SLF(W_QPDF);       \
  } while (0)
#define PV_STORE_SHADOW()                                                                                                 \
  do {                                                                                                                    \
    SLF(W_QTX) = q_T.x; SLF(W_QTY) = q_T.y; SLF(W_QTZ) = q_T.z;                                                           \
    SLF(W_QPRR) = q_prr; SLF(W_QPC) = q_point_cos; SLF(W_QDIST) = q_dist; SLF(W_QSQR) = q_sqr; SLF(W_QPDF) = q_pdf;       \
  } while (0)
#define PV_STORE_QBRDF() do { SLF(W_QBX) = q_brdf.x; SLF(W_QBY) = q_brdf.y; SLF(W_QBZ) = q_brdf.z; } while (0)
#define PV_LOAD_FILM()                                                                                                    \
  do {                                                                                                                    \
    sum = f3(SLF(W_SX), SLF(W_SY), SLF(W_SZ));                                                                            \
    cam_g = SLF(W_CAMG); cam_w = SLF(W_CAMW);                                                                             \
    un = make_int4(SLI(W_UNX), SLI(W_UNY), SLI(W_UNZ), SLI(W_UNW));                                                       \
    if (want_sumsq) sumsq = f3(SLF(W_SQ), SLF(W_SQ + 1), SLF(W_SQ + 2));                                                  \
  } while (0)
#define PV_STORE_FILM()                                                                                                   \
  do {                                                                                                                    \
    SLF(W_SX) = sum.x; SLF(W_SY) = sum.y; SLF(W_SZ) = sum.z;                                                              \
    SLF(W_CAMG) = cam_g; SLF(W_CAMW) = cam_w;                                                                             \
    SLI(W_UNX) = un.x; SLI(W_UNY) = un.y; SLI(W_UNZ) = un.z; SLI(W_UNW) = un.w;                                           \
    if (want_sumsq) { SLF(W_SQ) = sumsq.x; SLF(W_SQ + 1) = sumsq.y; SLF(W_SQ + 2) = sumsq.z; }                            \
  } while (0)

      // the vertex itself: the code of persistent.cuh's phase A, on the variables loaded above
#include "path_vertex.inc"

#undef PV_LOAD_SHADOW
#undef PV_STORE_SHADOW
#undef PV_STORE_QBRDF
#undef PV_LOAD_FILM
#undef PV_STORE_FILM
      if (go) {
        SLF(W_OX) = o.x; SLF(W_OY) = o.y; SLF(W_OZ) = o.z;
        SLF(W_DX) = d0.x; SLF(W_DY) = d0.y; SLF(W_DZ) = d0.z;
        SLF(W_T0) = t0; SLI(W_ID0) = id0;
        SLF(W_TX) = T.x; SLF(W_TY) = T.y; SLF(W_TZ) = T.z;
        SLF(W_LX) = L.x; SLF(W_LY) = L.y; SLF(W_LZ) = L.z;
        SLI(W_RNGLO) = (int)(unsigned int)rng.state; SLI(W_RNGHI) = (int)(unsigned int)(rng.state >> 32);
        SLI(W_FLAGS) = flags;
        if (NR == 2 && (flags & F_HAS_SHADOW)) {               // the shadow ray made by this vertex (its record went to the slot where it was computed)
          SLF(W_D1X) = d1.x; SLF(W_D1Y) = d1.y; SLF(W_D1Z) = d1.z;
          SLF(W_T1) = t1; SLI(W_ID1) = id1;
        }
      }
      // new slot states
      const unsigned bit = 1u << (s & 31);
      const int w = s >> 5;
#pragma unroll
      for (int i = 0; i < kWords; i++) {
        pend[i] |= __reduce_or_sync(kFull, (go && pend0 && w == i) ? bit : 0u);
        if (NR == 2) pend[(NR - 1) * kWords + i] |= __reduce_or_sync(kFull, (go && pend1 && w == i) ? bit : 0u);
        dead[i] |= __reduce_or_sync(kFull, (ready && !alive && w == i) ? bit : 0u);
      }
    } else {
      // ================================================================ phase B
      // a batch of up to 32 pending rays (extension or shadow) traverses the BVH: one loop that advances every lane by
      // at most one inner node and one triangle test per iteration (trav_step).  (Measured and dropped, each bit-exact: idle
      // lanes refilled from the pending rays inside this loop — r01 and again r02 with pools of 64 / 96 slots: 14-22 % slower;
      // two rays per lane: 23 % slower; the tree collapsed to 4-wide nodes: 4 % slower; batches formed from one class of rays —
      // bounces off the mesh apart from rays that come from a wall or the camera: 2-6 % slower.  profiles/r02_{b,c,h}_ab.txt.)
      const int n_sel = select_take<NR * kWords>(list, lane, pend, 32, rot_b);
      rot_b = rot_b + 1 == NR * kWords ? 0 : rot_b + 1;
      if (lane < n_sel) {
        const int item = list[lane];                          // mask word * 32 + bit; the shadow rays' words follow the kWords extension words
        const int s = item % (32 * kWords);
        const bool shadow = NR == 2 && item >= 32 * kWords;
        const F3 o = f3(SLF(W_OX), SLF(W_OY), SLF(W_OZ));
        const F3 d = shadow ? f3(SLF(W_D1X), SLF(W_D1Y), SLF(W_D1Z)) : f3(SLF(W_DX), SLF(W_DY), SLF(W_DZ));
        const F3 inv = f3(1.0f / d.x, 1.0f / d.y, 1.0f / d.z);
        float t = shadow ? SLF(W_T1) : SLF(W_T0);
        int id = shadow ? SLI(W_ID1) : SLI(W_ID0);
        finish_tree_query<COUNT>(sc, o, d, inv, t, id, tc, n_retrace);
        if (shadow) { SLF(W_T1) = t; SLI(W_ID1) = id; } else { SLF(W_T0) = t; SLI(W_ID0) = id; }
      }
    }
    __syncwarp();
  }
#undef SLF
#undef SLI

  flush_counters<COUNT>(counters, lane, n_rays, n_nonfinite, n_retrace, tc);
}

template <int INTEGRATOR, bool TREE, bool COUNT, int BUILD>
cudaError_t launch_pool_one(const DevScene& sc, const DevParams& p, float* out_sum, float* out_sumsq, unsigned long long* counters,
                            unsigned int* next_unit, int sm_count, cudaStream_t stream) {
  auto kernel = render_pool_kernel<INTEGRATOR, TREE, COUNT, BUILD>;
  const size_t smem = (size_t)(kBlockThreads / 32) * pl::warp_words<INTEGRATOR>(out_sumsq != nullptr) * sizeof(float);
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  // a warp serves as many units at a time as it has slots
  const unsigned int blocks = render_grid((const void*)kernel, smem, (long long)(kBlockThreads / 32) * pl::slots<INTEGRATOR>(), 2, p, sm_count);
  kernel<<<blocks, kBlockThreads, smem, stream>>>(sc, p, out_sum, out_sumsq, counters, next_unit);
  return cudaGetLastError();
}

}  // namespace lr
