// device_scene.h — layout of the scene in HBM and the kernel parameter blocks.
//
// Everything the kernels read is a flat, 16-byte aligned array so that every fetch on the
// traversal path is a 128-bit load:
//   nodes    : 4 x float4 per BVH node   (64 B)   — two child boxes + child codes
//   tris     : 3 x float4 per triangle   (48 B)   — p0|prim_id, e1 = p1-p0|material, e2 = p2-p0|0   (BVH leaf order,
//                                                   then the flat list of large triangles every ray tests)
//   tri_box  : 2 x float4 per triangle   (32 B)   — box of the vertices (lo | same-box-as-predecessor flag, hi | 0): the reference's
//                                                   leaf-AABB gate — once per ray for the nearest tree hit, once per flat box
//   tri_n    : 1 x float4 per triangle   (16 B)   — unit geometric normal | 0 (read once per path vertex)
//   spheres  : 1 x float4 per sphere     (16 B)   — centre|radius     (+ int2 material/prim_id)
//   mats     : 3 x float4 per material   (48 B)   — colour|type, emission|param0, param1|weight|emissive|0
//   emitters : 3 x float4 per emitter    (48 B)   — tri: p0|kind, p1|area, p2|0 ; sphere: centre|kind, radius,0,0|area
//   sky      : 1 x float4 per texel (rgb|0), nearest-texel lookup
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/lumilly.h"

namespace lr {

constexpr int kStackDepth = 64;          // per-thread traversal stack entries
constexpr int kBlockThreads = 128;       // 4 warps, each warp owns an 8x4 pixel tile

struct DevScene {
  const float4* nodes;
  const float4* tris;
  const float4* tri_box;                 // 2 x float4 per triangle: box lo | hi of the vertices (the reference's leaf-AABB gate)
  const float4* tri_n;                   // geometric normal per triangle, precomputed like Triangle::new does (triangle.rs:36)
  const float4* spheres;
  const int2* sphere_meta;
  const float4* mats;
  const float* emitter_cdf;
  const float4* emitters;
  const float4* sky_pixels;
  int n_nodes, n_tris, n_spheres, n_emitters;
  int n_bvh_tris;                        // tris[0, n_bvh_tris) are in BVH leaf order; tris[n_bvh_tris, n_tris) is the flat list
  float bvh_lo[3], bvh_hi[3];            // bounds of the tree (union of the root's child boxes, padded like them)
  float emission_area;
  int sky_type;
  float sky_color[3];
  int sky_height;
  float sky_longitude_offset;
  LrCamera cam;
};

struct DevParams {
  int integrator;
  int spp_begin, spp_count;
  int depth, depth_limit, no_direct_emitter;
  unsigned long long seed;
  int crop_x, crop_y, crop_w, crop_h;
  int splits;
  int tiles_x, tiles_y;                  // 8x4 pixel tiles over the crop window
  int shard, n_shards;                   // this launch renders the tiles t with shard_of_tile(t, n_shards) == shard (default 0 of 1)
  int unit_tiles;                        // how many tiles that is: shard_tile_count(tiles_x * tiles_y, ...), set once on the host
  int defer_iters, defer_thresh;         // path vertices per phase A; suspended lanes that end it early (persistent.cuh)
  int organisation;                      // BVH scenes only: 1 = one path per lane (persistent.cuh), otherwise the pool (pool.cuh)
  const int2* tile_list;                 // null: the shard's tiles from spp_begin; else the j-th tile is {global tile, first
                                         // sample index} = tile_list[j], j < unit_tiles (a film whose tiles hold different counts)
};

// Pixel sharding of a film over several devices (lr_multi_film_*): the crop's 8x4 tiles are dealt round-robin, shard k of
// S owns the tiles t with t % S == k, and shard k renders on device k % n_devices.  Round-robin balances the load without
// knowing where the expensive pixels are.  Every pixel is rendered by exactly one shard, so its samples are still added
// in sample order on one device and the image does not depend on S or on the device count.  The render kernels (decode_unit)
// and the gather kernel (kernels.cu) both go through these functions.
__host__ __device__ inline int shard_of_tile(int tile, int n_shards) { return tile % n_shards; }
__host__ __device__ inline int shard_tile(int j, int shard, int n_shards) { return j * n_shards + shard; }   // j-th tile of the shard
__host__ __device__ inline int shard_tile_count(int n_tiles, int shard, int n_shards) {
  return shard < n_tiles ? (n_tiles - shard + n_shards - 1) / n_shards : 0;
}
__host__ __device__ inline int shard_device(int shard, int n_devices) { return shard % n_devices; }
// A sample range [begin, begin + count) cut into n_parts consecutive ranges whose sizes differ by at most one: the range of
// part `part`.  The devices of lr_render_multi (lr_shard_range) and the spp splits of one launch (path_vertex.inc) are cut so.
struct SampleRange { int begin, count; };
__host__ __device__ inline SampleRange range_part(int begin, int count, int part, int n_parts) {
  const int per = count / n_parts, rem = count % n_parts;
  return {begin + part * per + (part < rem ? part : rem), per + (part < rem ? 1 : 0)};
}
// Adaptive sampling of a film (lr_film_render_adaptive): which 8x4 tiles get more samples.  A tile holding n samples of each
// of its pixels, with per-pixel sums S and sums of squares Q, has the error max over its in-crop pixels and channels of
//   sqrt(var / n) / max(m, kAdaptiveFloor),   m = S / n,   var = max(0, (Q - S m) / (n - 1))
// (the relative standard error of the pixel mean), all in fp64 without contraction (kernels.cu is built with -fmad=false), so
// a numpy float64 restatement decides the same.  The floor keeps black pixels from asking for samples forever.
constexpr double kAdaptiveFloor = 1e-3;
__host__ __device__ inline double adaptive_error(double s, double q, double n) {
  const double m = s / n;
  const double var = fmax(0.0, (q - s * m) / (n - 1.0));
  return sqrt(var / n) / fmax(m, kAdaptiveFloor);
}
// Fewer than two samples say nothing about the noise; a tile with a non-finite sum is left alone once it has two (more samples
// cannot make its sum finite again); max_spp > 0 caps the samples a tile gets.
__host__ __device__ inline bool adaptive_selects(int n, bool finite, double error, float threshold, int max_spp) {
  return (n < 2 || (finite && error > (double)threshold)) && (max_spp == 0 || n < max_spp);
}
// work items of one render launch: one per (split, pixel slot of the shard's tiles)
__host__ __device__ inline unsigned int render_units(const DevParams& p) { return (unsigned int)p.unit_tiles * 32u * (unsigned int)p.splits; }

// device counter block (unsigned long long each)
enum CounterSlot { C_RAYS = 0, C_NONFINITE = 1, C_NODES = 2, C_TRIS = 3, C_SPHERES = 4, C_RETRACE = 5, C_FLAT_TRIS = 6, C_NEXT_UNIT = 7, C_FLAT_BOXES = 8, C_COUNT = 9 };

}  // namespace lr
