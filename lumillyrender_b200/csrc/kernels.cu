// kernels.cu — the small sm_100a kernels around the render kernel (which lives in persistent.cuh and is
// instantiated in persistent_inst.cu): ordered reduction of spp splits, normalisation, the cross-device reduce and
// gather, the nearest-hit parity probes, and the read-bandwidth microbenchmark.
//
// Compiled with -fmad=false (see device_path.cuh for the numerics contract).
#include <algorithm>

#include "device_path.cuh"
#include "kernels.h"

namespace lr {

// dst[i] += sum_k partial[k][i] in k order
__global__ void reduce_splits_kernel(float* __restrict__ dst, const float* __restrict__ partial, size_t n, int splits) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float acc = 0.0f;
  for (int k = 0; k < splits; k++) acc += partial[(size_t)k * n + i];
  dst[i] += acc;
}

__global__ void scale_kernel(float* __restrict__ dst, size_t n, float divisor) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = dst[i] / divisor;   // `estimated_sum / spp as f32` (main.rs:104): a true division
}

// K7 across GPUs, fused: one kernel on the first device reads every device's per-pixel sums — its own and, through
// peer access over NVLink, the others' — adds them in device order (a fixed order: the image does not depend on which
// GPU finished first) and divides by the total sample count (main.rs:104; divisor <= 0: sums only, for the sum of
// squares).  32 MB per peer at 1920x1370: a few hundred microseconds next to a render of tens of milliseconds.
__global__ void reduce_peers_kernel(float* __restrict__ dst, PeerBuffers src, size_t n, float divisor) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float acc = src.p[0][i];
  for (int k = 1; k < src.count; k++) acc = acc + src.p[k][i];
  dst[i] = divisor > 0.0f ? acc / divisor : acc;
}

// The image of a pixel-sharded film (lr_multi_film_*), on the first device: every device's buffer spans the whole crop but
// holds only the pixels of its own shards (stale values or zeros elsewhere), so each pixel is taken from the device that
// owns its tile, never summed across devices.  Divided by the sample count with the expression of scale_kernel, so the
// bits equal lr_film_read's; divisor <= 0: the raw sums (sums of squares, checkpoints).
__global__ void gather_shards_kernel(float* __restrict__ dst, const __grid_constant__ PeerBuffers src, int crop_w, int crop_h, int n_shards, float divisor) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)crop_w * crop_h * 3) return;
  const int px = (int)(i / 3), lx = px % crop_w, ly = px / crop_w;
  const int tiles_x = (crop_w + 7) / 8;
  const int shard = shard_of_tile((ly >> 2) * tiles_x + (lx >> 3), n_shards);
  const float v = src.p[shard_device(shard, src.count)][i];
  dst[i] = divisor > 0.0f ? v / divisor : v;
}

// parity probe: nearest hit of the primary ray of every film pixel with fixed random numbers
__global__ void __launch_bounds__(kBlockThreads)
primary_kernel(const __grid_constant__ DevScene sc, int tiles_x, int tiles_y, float u, float v, float ua, float va,
               int* __restrict__ prim, float* __restrict__ tout) {
  const long long gid = (long long)blockIdx.x * kBlockThreads + threadIdx.x;
  const long long tile = gid >> 5;
  const int lane = (int)(gid & 31);
  if (tile >= (long long)tiles_x * tiles_y) return;
  const int x = (int)(tile % tiles_x) * 8 + (lane & 7), y = (int)(tile / tiles_x) * 4 + (lane >> 3);
  if (x >= sc.cam.width || y >= sc.cam.height) return;
  const float draws[4] = {u, v, ua, va};
  int k = 0;
  F3 o, d;
  float g, w;
  camera_sample(sc.cam, x, y, [&]() { return draws[k++]; }, o, d, g, w);
  float t;
  int id;
  TraceCounters tc;
  trace<false>(sc, o, d, t, id, tc);
  const size_t i = (size_t)y * sc.cam.width + x;
  if (id == -1) { prim[i] = -1; tout[i] = 0.0f; }
  else { const Surface s = surface_at(sc, o, d, t, id); prim[i] = s.prim; tout[i] = t; }
}

// RENDER_QUERY = false: the strict query (the reference's gate on every candidate).  true: the query exactly as the render
// kernels run it (path_vertex.inc + the BVH phase): flat list, tree-bounds test, optimistic traversal (trav_step), the
// nearest tree hit gated once, strict re-trace if the gate rejects it — so a replay divergence can be pinned on a ray.
template <bool RENDER_QUERY>
__global__ void __launch_bounds__(kBlockThreads)
rays_kernel(const __grid_constant__ DevScene sc, long long n, const float* __restrict__ org, const float* __restrict__ dir,
            int* __restrict__ prim, float* __restrict__ tout, float* __restrict__ nout) {
  const long long i = (long long)blockIdx.x * kBlockThreads + threadIdx.x;
  if (i >= n) return;
  const F3 o = f3(org + 3 * i), d = f3(dir + 3 * i);
  float t;
  int id;
  TraceCounters tc;
  if (RENDER_QUERY) {
    const F3 inv = f3(1.0f / d.x, 1.0f / d.y, 1.0f / d.z);
    t = 3.0e38f;
    id = -1;
    flat_hits<false>(sc, flat_list_global(sc), o, d, inv, t, id, tc);
    if (sc.n_nodes > 0 && bvh_bounds_hit(sc, o, inv, t < 3.0e38f ? t * 1.0001f + 1e-4f : 3.0e38f)) {
      bvh_traverse_unified<false>(sc, o, d, inv, t, id, tc);
      if (id >= 0 && id < sc.n_bvh_tris && !bvh_hit_is_gated(sc, o, inv, id)) trace<false>(sc, o, d, t, id, tc);
    }
  } else {
    trace<false>(sc, o, d, t, id, tc);
  }
  if (id == -1) {
    prim[i] = -1; tout[i] = 0.0f;
    if (nout) { nout[3 * i] = 0.0f; nout[3 * i + 1] = 0.0f; nout[3 * i + 2] = 0.0f; }
  } else {
    const Surface s = surface_at(sc, o, d, t, id);
    prim[i] = s.prim; tout[i] = t;
    if (nout) { nout[3 * i] = s.n.x; nout[3 * i + 1] = s.n.y; nout[3 * i + 2] = s.n.z; }
  }
}

// AOVs: Scene::normal / Scene::depth (scene.rs:48-62) of the camera ray of every sample of the range — the SAME camera rays
// the render draws (same counter-based stream, camera draws first) — averaged per pixel in sample order.
//   normal: hit ? n / 2 + (0.5, 0.5, 0.5) : (0, 0, 0)   (3 floats per pixel)      depth: hit ? distance : 0   (1 float per pixel)
__global__ void __launch_bounds__(kBlockThreads)
aov_kernel(const __grid_constant__ DevScene sc, const __grid_constant__ DevParams p, int kind, float* __restrict__ out) {
  const long long gid = (long long)blockIdx.x * kBlockThreads + threadIdx.x;
  const long long tile = gid >> 5;
  const int lane = (int)(gid & 31);
  if (tile >= (long long)p.tiles_x * p.tiles_y) return;
  const int lx = (int)(tile % p.tiles_x) * 8 + (lane & 7), ly = (int)(tile / p.tiles_x) * 4 + (lane >> 3);
  if (lx >= p.crop_w || ly >= p.crop_h) return;
  const int x = p.crop_x + lx, y = p.crop_y + ly;
  const unsigned int pixel = (unsigned int)(y * sc.cam.width + x);
  F3 sum = f3(0.0f, 0.0f, 0.0f);
  for (int si = 0; si < p.spp_count; si++) {
    Pcg rng;
    rng.seed(p.seed, pixel, (unsigned int)(p.spp_begin + si));
    F3 o, d;
    float g, w;
    camera_sample(sc.cam, x, y, [&]() { return rng.next(); }, o, d, g, w);
    float t;
    int id;
    TraceCounters tc;
    trace<false>(sc, o, d, t, id, tc);
    F3 v = f3(0.0f, 0.0f, 0.0f);
    if (id != -1) {
      if (kind == LR_AOV_NORMAL) v = surface_at(sc, o, d, t, id).n / 2.0f + f3(0.5f, 0.5f, 0.5f);   // scene.rs:52
      else v = f3(t, 0.0f, 0.0f);                                                                    // scene.rs:60
    }
    sum = sum + v;
  }
  const size_t i = (size_t)ly * p.crop_w + lx;
  const float n = (float)p.spp_count;
  if (kind == LR_AOV_NORMAL) { out[3 * i] = sum.x / n; out[3 * i + 1] = sum.y / n; out[3 * i + 2] = sum.z / n; }
  else out[i] = sum.x / n;
}

// bandwidth microbenchmark: every thread streams 128-bit loads over a working set `n4` float4s,
// `iters` passes.  With a working set << 126 MB it measures the L2 read peak, >> 126 MB the HBM read peak.
__global__ void __launch_bounds__(256) read_bw_kernel(const float4* __restrict__ buf, size_t n4, int iters, float* __restrict__ sink) {
  float acc = 0.0f;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (int it = 0; it < iters; it++) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (; i + 3 * stride < n4; i += 4 * stride) {
      float4 a, b, c, d;
      asm volatile("ld.global.cg.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w) : "l"(buf + i));
      asm volatile("ld.global.cg.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w) : "l"(buf + i + stride));
      asm volatile("ld.global.cg.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(c.x), "=f"(c.y), "=f"(c.z), "=f"(c.w) : "l"(buf + i + 2 * stride));
      asm volatile("ld.global.cg.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(d.x), "=f"(d.y), "=f"(d.z), "=f"(d.w) : "l"(buf + i + 3 * stride));
      acc += a.x + b.y + c.z + d.w;
    }
    for (; i < n4; i += stride) {
      float4 a;
      asm volatile("ld.global.cg.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w) : "l"(buf + i));
      acc += a.x;
    }
  }
  if (acc == 1.2345e-30f) *sink = acc;
}

// ------------------------------------------------------------------ launchers
cudaError_t launch_render_persistent(const DevScene& sc, const DevParams& p, bool has_ggx, bool count, float* out_sum, float* out_sumsq,
                                     unsigned long long* counters, unsigned int* next_unit, int sm_count, cudaStream_t stream) {
  // the instrumented kernel exists in the (tree, GGX inline) units only: it is the most general code
  const bool tree = sc.n_nodes > 0 || count, ggx = has_ggx || count;
  using Fn = cudaError_t (*)(const DevScene&, const DevParams&, bool, float*, float*, unsigned long long*, unsigned int*, int, cudaStream_t);
  static const Fn table[2][2][2] = {
      {{launch_persistent_i0_t0_g0, launch_persistent_i0_t0_g1}, {launch_persistent_i0_t1_g0, launch_persistent_i0_t1_g1}},
      {{launch_persistent_i1_t0_g0, launch_persistent_i1_t0_g1}, {launch_persistent_i1_t1_g0, launch_persistent_i1_t1_g1}}};
  return table[p.integrator == LR_INTEGRATOR_PT ? 0 : 1][tree ? 1 : 0][ggx ? 1 : 0](sc, p, count, out_sum, out_sumsq, counters, next_unit,
                                                                                   sm_count, stream);
}

cudaError_t launch_reduce_splits(float* dst, const float* partial, size_t n, int splits, cudaStream_t stream) {
  reduce_splits_kernel<<<(unsigned int)((n + 255) / 256), 256, 0, stream>>>(dst, partial, n, splits);
  return cudaGetLastError();
}

cudaError_t launch_scale(float* dst, size_t n, float divisor, cudaStream_t stream) {
  scale_kernel<<<(unsigned int)((n + 255) / 256), 256, 0, stream>>>(dst, n, divisor);
  return cudaGetLastError();
}

cudaError_t launch_reduce_peers(float* dst, const PeerBuffers& src, size_t n, float divisor, cudaStream_t stream) {
  reduce_peers_kernel<<<(unsigned int)((n + 255) / 256), 256, 0, stream>>>(dst, src, n, divisor);
  return cudaGetLastError();
}

cudaError_t launch_gather_shards(float* dst, const PeerBuffers& src, int crop_w, int crop_h, int n_shards, float divisor, cudaStream_t stream) {
  const size_t n = (size_t)crop_w * crop_h * 3;
  gather_shards_kernel<<<(unsigned int)((n + 255) / 256), 256, 0, stream>>>(dst, src, crop_w, crop_h, n_shards, divisor);
  return cudaGetLastError();
}

cudaError_t launch_primary(const DevScene& sc, float u, float v, float ua, float va, int* prim, float* t, cudaStream_t stream) {
  const int tiles_x = (sc.cam.width + 7) / 8, tiles_y = (sc.cam.height + 3) / 4;
  const long long threads = (long long)tiles_x * tiles_y * 32;
  primary_kernel<<<(unsigned int)((threads + kBlockThreads - 1) / kBlockThreads), kBlockThreads, 0, stream>>>(sc, tiles_x, tiles_y, u, v, ua, va, prim, t);
  return cudaGetLastError();
}

cudaError_t launch_aov(const DevScene& sc, const DevParams& p, int kind, float* out, cudaStream_t stream) {
  const long long threads = (long long)p.tiles_x * p.tiles_y * 32;
  aov_kernel<<<(unsigned int)((threads + kBlockThreads - 1) / kBlockThreads), kBlockThreads, 0, stream>>>(sc, p, kind, out);
  return cudaGetLastError();
}

cudaError_t launch_rays(const DevScene& sc, long long n, const float* org, const float* dir, int* prim, float* t, float* nout, bool render_query,
                        cudaStream_t stream) {
  const unsigned int blocks = (unsigned int)((n + kBlockThreads - 1) / kBlockThreads);
  if (render_query) rays_kernel<true><<<blocks, kBlockThreads, 0, stream>>>(sc, n, org, dir, prim, t, nout);
  else rays_kernel<false><<<blocks, kBlockThreads, 0, stream>>>(sc, n, org, dir, prim, t, nout);
  return cudaGetLastError();
}

cudaError_t launch_read_bw(const float4* buf, size_t n4, int iters, int blocks, float* sink, cudaStream_t stream) {
  read_bw_kernel<<<blocks, 256, 0, stream>>>(buf, n4, iters, sink);
  return cudaGetLastError();
}

}  // namespace lr
