/* lumilly.h — C ABI of the B200-native path-tracing hot path (liblumilly_b200.so).
 *
 * This is the drop-in boundary for LumillyRender's per-pixel Monte Carlo loop.
 * The reference has no FFI of its own; the seam these entry points replace is the
 * block `pool.scoped(|scope| { ... })` + channel gather in  src/main.rs:70-132,
 * i.e. per pixel:  cam.sample(x,y)  (src/camera.rs:9-13)  ->  scene.radiance /
 * scene.radiance_nee (src/scene.rs:20,34)  ->  output.set(x,y,..) (src/img.rs:25).
 *
 * Conventions
 *   - plain C, POD structs, plain pointers and sizes; no C++/torch types.
 *   - every function returns 0 on success, a negative LrStatus on failure and
 *     never aborts/throws across the ABI; lr_last_error() gives the message
 *     (thread-local).  The reference panics instead (SURVEY.md §5).
 *   - host pointers unless a parameter is named d_* (device pointer).
 *   - images are row-major, y = 0 is the top row, 3 floats (r,g,b) per pixel:
 *     exactly Img.data[y][x] of src/img.rs:6-27.
 *   - primitive ids are indices into the reference's `Loader.instances`
 *     (src/description.rs:90-144): objects in TOML order, OBJ faces in file order.
 *   - there is NO CPU fallback: without a CUDA device every compute entry point
 *     fails with LR_ERR_NO_DEVICE.
 */
#ifndef LUMILLY_H
#define LUMILLY_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LR_ABI_VERSION 3

typedef enum LrStatus {
  LR_OK = 0,
  LR_ERR_INVALID = -1,     /* bad argument / inconsistent description          */
  LR_ERR_NO_DEVICE = -2,   /* no CUDA device or CUDA runtime failure at init   */
  LR_ERR_CUDA = -3,        /* CUDA runtime error during a call                 */
  LR_ERR_IO = -4,          /* file not found / unreadable / unwritable         */
  LR_ERR_PARSE = -5,       /* malformed TOML / OBJ / HDR                       */
  LR_ERR_UNSUPPORTED = -6  /* valid input the library does not handle          */
} LrStatus;

/* ---- materials: src/material/{lambert,phong,blinn_phong,ggx,ideal_refraction}.rs ---- */
typedef enum LrMaterialType {
  LR_MAT_LAMBERT = 0,          /* lambert.rs:13-55 (+ hard-coded checker 58-90)  */
  LR_MAT_PHONG = 1,            /* phong.rs:16-69       param0 = alpha            */
  LR_MAT_BLINN_PHONG = 2,      /* blinn_phong.rs:16-73 param0 = alpha            */
  LR_MAT_GGX = 3,              /* ggx.rs:18-113        param0 = roughness, param1 = ior */
  LR_MAT_IDEAL_REFRACTION = 4  /* ideal_refraction.rs:16-160 param0 = absorbtance, param1 = ior */
} LrMaterialType;

typedef struct LrMaterial {
  int32_t type;        /* LrMaterialType                                         */
  float color[3];      /* albedo (lambert) or reflectance (all others)           */
  float emission[3];   /* only honoured for LR_MAT_LAMBERT (description.rs:94-101) */
  float param0;
  float param1;
} LrMaterial;

/* ---- primitives: src/triangle.rs:25-40, src/sphere.rs:21-39 (world space) ---- */
typedef struct LrTriangle {
  float p0[3], p1[3], p2[3];
  int32_t material;    /* index into LrSceneDesc.materials                       */
  int32_t prim_id;     /* index in `Loader.instances` order                      */
} LrTriangle;

typedef struct LrSphere {
  float center[3];
  float radius;
  int32_t material;
  int32_t prim_id;
} LrSphere;

/* ---- camera block: fields of the camera structs after their constructors ran.
 * IdealPinholeCamera camera.rs:16-62, PinholeCamera 200-264, LensCamera 340-409,
 * OmnidirectionalCamera 137-166.  Computed once on the host so that the oracle and
 * the device consume identical bits (SURVEY.md §7 hard part 1).                    */
typedef enum LrCameraType {
  LR_CAM_IDEAL_PINHOLE = 0,
  LR_CAM_PINHOLE = 1,          /* "realistic pinhole", finite aperture disc      */
  LR_CAM_THIN_LENS = 2,
  LR_CAM_OMNIDIRECTIONAL = 3
} LrCameraType;

typedef struct LrCamera {
  int32_t type;
  int32_t width, height;       /* film resolution the block was built for        */
  float forward[3], right[3], up[3];
  float position[3];           /* sensor centre                                  */
  float aperture_position[3];
  float sensor_size[2];
  float aperture_radius;
  float aperture_sensor_distance;
  float sensor_pixel_area;
  float sensor_sensitivity;    /* 1 for ideal pinhole / omnidirectional          */
  float focus_distance;
} LrCamera;

/* ---- sky: src/sky.rs:13-21 (uniform), 35-79 (equirect, nearest texel) ---- */
typedef enum LrSkyType { LR_SKY_UNIFORM = 0, LR_SKY_IBL = 1 } LrSkyType;

typedef struct LrSky {
  int32_t type;
  float color[3];              /* uniform radiance                               */
  const float* pixels;         /* IBL: decoded RGB fp32, row-major, n_pixels*3    */
  int64_t n_pixels;            /* must be >= 2*height*height (sky.rs:64-72 assumes width = 2*height) */
  int32_t height;
  float longitude_offset;      /* radians                                        */
} LrSky;

/* ---- flattened BVH over the triangles (spheres are kept in a flat list).
 * Replaces the boxed tree of src/bvh.rs:10-49.  64-byte node, two children with
 * their boxes stored in the parent:
 *   f[0..5]  = child0 lo.xyz, hi.xyz      f[6..11] = child1 lo.xyz, hi.xyz
 *   c[0],c[1]= child index: >= 0 inner node; < 0 leaf, first triangle = ~c
 *   n[0],n[1]= triangle count of a leaf child (0 for inner, <0 for "no child")
 * Leaves reference contiguous ranges of the first n_triangles - n_flat_triangles entries of
 * LrSceneDesc.triangles (already permuted into leaf order by the host front end).             */
typedef struct LrBvhNode {
  float f[12];
  int32_t c[2];
  int32_t n[2];
} LrBvhNode;

typedef struct LrSceneDesc {
  const LrMaterial* materials; int32_t n_materials;
  const LrTriangle* triangles; int32_t n_triangles;   /* in BVH leaf order      */
  const LrSphere* spheres;     int32_t n_spheres;
  const LrBvhNode* nodes;      int32_t n_nodes;       /* 0 nodes iff no triangle is in the BVH */
  int32_t bvh_depth;                                    /* max stack depth needed */
  int32_t n_flat_triangles;    /* the LAST n_flat_triangles entries of `triangles` are outside the BVH: large
                                  primitives (walls, floors, area lights) that every ray tests in a flat loop,
                                  like the spheres.  0 <= n_flat_triangles <= n_triangles.                   */
  LrCamera camera;
  LrSky sky;
} LrSceneDesc;

typedef enum LrIntegrator {
  LR_INTEGRATOR_PT = 0,        /* Scene::radiance      scene.rs:20-32,153-171    */
  LR_INTEGRATOR_PT_DIRECT = 1  /* Scene::radiance_nee  scene.rs:34-46,173-193    */
} LrIntegrator;

typedef struct LrRenderParams {
  int32_t integrator;          /* LrIntegrator                                   */
  int32_t spp_begin;           /* first sample index of this call                */
  int32_t spp_count;           /* number of sample indices rendered by this call */
  int32_t depth;               /* renderer.depth        (default 5,  description.rs:75) */
  int32_t depth_limit;         /* renderer.depth-limit  (default 64, description.rs:76) */
  int32_t no_direct_emitter;   /* renderer.no-direct-emitter (description.rs:79) */
  uint64_t seed;               /* key of the counter-based RNG                   */
  int32_t crop_x, crop_y;      /* crop window in film pixels; crop_w = 0 => full film */
  int32_t crop_w, crop_h;
  int32_t splits;              /* threads per pixel over the spp range; 0 = auto, 1 = one
                                  thread per pixel summing in sample order        */
  int32_t count_traversal;     /* 1 = instrumented traversal (node/tri/sphere counters) */
} LrRenderParams;

typedef struct LrStats {
  uint64_t rays;               /* closest-hit queries (camera + bounce + shadow) */
  uint64_t samples;            /* crop_w*crop_h*spp_count                        */
  uint64_t nodes_visited;      /* only if count_traversal                         */
  uint64_t tris_tested;
  uint64_t spheres_tested;
  uint64_t nonfinite_samples;  /* samples whose estimate was NaN/Inf (kept, as the reference does) */
  uint64_t gate_retraces;      /* rays re-traced strictly because their optimistic nearest BVH hit failed the
                                  reference's leaf-AABB gate (a few per 10^8 rays)                  */
  uint64_t flat_tris_tested;   /* only if count_traversal: the part of tris_tested that ran on the flat list ...   */
  uint64_t flat_boxes_tested;  /* ... and the leaf-AABB gate tests that selected those candidates                  */
  float kernel_ms;             /* CUDA-event time of the render kernel(s)        */
  int32_t launches;            /* kernels launched by the call                    */
  int32_t splits;              /* splits actually used                            */
} LrStats;

typedef struct LrScene LrScene;   /* opaque; owns device memory on the library's device (lr_init) at lr_scene_create.
                                     Every entry point that takes a scene (or a film of it) switches the calling thread to
                                     that device for the call and restores the caller's device on return.               */

/* ---- lifetime ---- */
int lr_abi_version(void);
int lr_init(int device);                       /* cudaSetDevice + context; LR_ERR_NO_DEVICE if none */
void lr_shutdown(void);
const char* lr_last_error(void);
int lr_device_info(int* sm_count, int* l2_bytes, int* sm_clock_khz, char* name, int name_len);

/* ---- scene upload (H2D of the flat arrays) ---- */
int lr_scene_create(const LrSceneDesc* desc, LrScene** out);
void lr_scene_destroy(LrScene* scene);
int lr_scene_bytes(const LrScene* scene, uint64_t* h2d_bytes);

/* ---- the hot path.  Replaces main.rs:70-132 for one sample range. ----
 * lr_render: synchronous; out_rgb = per-pixel MEAN over the call's spp_count samples
 * (crop_w*crop_h*3 floats, host). out_sumsq (nullable) = per-pixel SUM of squared
 * per-sample estimates (for the variance test).                                   */
int lr_render(const LrScene* scene, const LrRenderParams* params,
              float* out_rgb, float* out_sumsq, LrStats* stats);

/* lr_render_accumulate_device: adds the per-pixel SUM of the sample range into device
 * buffers (d_sum += ..., d_sumsq += ... if non-null), asynchronously on `cuda_stream`
 * (a cudaStream_t passed as void*; NULL = default stream).  Used for spp sharding:
 * every GPU accumulates its range, then the buffers are summed with one NCCL reduce. */
int lr_render_accumulate_device(const LrScene* scene, const LrRenderParams* params,
                                float* d_sum, float* d_sumsq, void* cuda_stream);
/* fetch + reset the device counters of the accumulate calls issued so far (synchronises the stream) */
int lr_stats_fetch(const LrScene* scene, void* cuda_stream, LrStats* stats);

/* lr_render_multi: the whole loop of main.rs:70-132 on SEVERAL GPUs of one box from one process (what a
   single-process host such as the reference's `main` calls; one process per GPU uses
   lr_render_accumulate_device instead).  The scene is uploaded to every listed device; the sample range
   [spp_begin, spp_begin + spp_count) is cut into n_devices consecutive ranges whose sizes differ by <= 1
   (samples are counter-indexed, so any device can render any range); the devices render concurrently, each
   into its own per-pixel sum buffer; then ONE kernel on devices[0] reads the peers' buffers over NVLink
   (peer access; staged copies where peer access is unavailable), adds them in list order and divides by
   spp_count.  out_rgb / out_sumsq / stats as lr_render (stats are totals, kernel_ms the slowest device's).
   1 <= n_devices <= 8, device ids distinct.  The result for a given device COUNT is bit-reproducible and
   differs from other counts only by fp32 summation order.  It switches the calling thread's CUDA device as it
   works and restores it on return; the library's device (lr_init) is untouched.  Not re-entrant: call it from
   one thread at a time and not concurrently with other entry points. */
/* The sample-range sharding rule, for any host that shards by itself (one process per GPU): part `part` of
   `n_parts` of the range [spp_begin, spp_begin + spp_count) — consecutive ranges that tile it exactly, sizes
   differing by <= 1, the larger ones first.  lr_render_multi and bench.py's ranks use this rule. */
int lr_shard_range(int32_t spp_begin, int32_t spp_count, int32_t part, int32_t n_parts, int32_t* begin, int32_t* count);

int lr_render_multi(const LrSceneDesc* desc, const LrRenderParams* params, int32_t n_devices, const int32_t* devices,
                    float* out_rgb, float* out_sumsq, LrStats* stats);
/* The same as a handle, for a host that renders more than once (progressive previews, animations, a benchmark loop): the
   scene is uploaded to every device, the per-device streams / events are made and the peer mappings that let devices[0]
   read the others' film buffers are established ONCE (first use of a mapping costs ~100 ms per device pair);
   lr_multi_render then only launches, reduces and copies.  lr_render_multi is create + render + destroy.            */
typedef struct LrMultiScene LrMultiScene;
int lr_multi_scene_create(const LrSceneDesc* desc, int32_t n_devices, const int32_t* devices, LrMultiScene** out);
int lr_multi_render(LrMultiScene* ms, const LrRenderParams* params, float* out_rgb, float* out_sumsq, LrStats* stats);
void lr_multi_scene_destroy(LrMultiScene* ms);

/* ---- AOVs: Scene::normal / Scene::depth (src/scene.rs:48-62) of the camera ray of every sample in
 * [spp_begin, spp_begin + spp_count) — the very camera rays lr_render draws for those samples (same seed, same
 * stream) — averaged per pixel in sample order.  Honours seed / spp range / crop of `params`; integrator, depth,
 * splits are ignored.  out: crop_w*crop_h*3 floats for LR_AOV_NORMAL (hit ? n/2 + 0.5 : 0), crop_w*crop_h floats
 * for LR_AOV_DEPTH (hit ? Intersection.distance : 0).  Host pointer, synchronous.                              */
typedef enum LrAovKind { LR_AOV_NORMAL = 0, LR_AOV_DEPTH = 1 } LrAovKind;
int lr_render_aov(const LrScene* scene, const LrRenderParams* params, int32_t kind, float* out);

/* ---- progressive / resumable rendering: the progress hook the reference abandoned (src/main.rs:81-91) as a handle.
 * An LrFilm owns the per-pixel SUM buffers of one render (and the sums of squares if asked for) on the scene's device
 * and remembers how many sample indices it holds.  lr_film_render adds the next `spp_count` sample indices (it
 * overrides params->spp_begin with the film's count; seed / integrator / depths / crop must stay what the film was
 * created with); lr_film_read gives the mean so far; lr_film_save / lr_film_load write and restore a checkpoint
 * (raw sums + the parameters), in this or another process.  With params->splits == 1 every pixel's samples are added
 * in sample order starting from the stored sum — the fold of main.rs:92-104 — so ANY cut of [0, n) into
 * consecutive lr_film_render calls, with or without a save / load in between, gives bit for bit the image of one
 * lr_render over [0, n).  (splits != 1 is deterministic but adds per-call partial sums.)                          */
typedef struct LrFilm LrFilm;
int lr_film_create(const LrScene* scene, const LrRenderParams* params, int32_t want_sumsq, LrFilm** out);
int lr_film_render(LrFilm* film, int32_t spp_count, LrStats* stats /* nullable */);
int lr_film_info(const LrFilm* film, int32_t* spp_done, int32_t* crop_w, int32_t* crop_h, int32_t* has_sumsq);   /* each nullable */
int lr_film_read(const LrFilm* film, float* out_rgb /* mean so far */, float* out_sumsq /* nullable */);
int lr_film_save(const LrFilm* film, const char* path);
int lr_film_load(const LrScene* scene, const char* path, LrFilm** out);
void lr_film_destroy(LrFilm* film);

/* ---- the same film on the devices of an LrMultiScene.  The crop's 8x4 pixel tiles are dealt round-robin: shard k of
 * n_devices owns the tiles t with t % n_devices == k and renders on devices[k].  Every pixel's samples are still added in
 * sample order on one device, starting from the stored sum, so the image, the sums of squares and the ray count equal
 * those of one lr_render with splits = 1, bit for bit, for ANY device count (lr_multi_render, which shards by sample
 * index, cannot promise that).  lr_multi_film_render launches every device at once, each on its own stream, and returns
 * when all are done (stats: totals, kernel_ms the slowest device's).  read / save gather the image on devices[0], each
 * pixel from the device that owns it (peer reads over NVLink, staged copies where a peer cannot be mapped).
 * params->splits must be 0 or 1 (it is always 1).  save writes the checkpoint format of lr_film_save, byte for byte
 * what lr_film_save writes for the same state; lr_film_load resumes it on one device, and lr_multi_film_load resumes a
 * checkpoint of either kind on any LrMultiScene (its header must say splits = 1).  Destroy the films of an LrMultiScene
 * before the LrMultiScene.  Not re-entrant, like lr_multi_render: the calls switch the calling thread's CUDA device as
 * they work and restore it on return; the library's device (lr_init) is untouched.                                */
typedef struct LrMultiFilm LrMultiFilm;
int lr_multi_film_create(LrMultiScene* ms, const LrRenderParams* params, int32_t want_sumsq, LrMultiFilm** out);
int lr_multi_film_render(LrMultiFilm* film, int32_t spp_count, LrStats* stats /* nullable */);
int lr_multi_film_info(const LrMultiFilm* film, int32_t* spp_done, int32_t* crop_w, int32_t* crop_h, int32_t* has_sumsq);   /* each nullable */
int lr_multi_film_read(const LrMultiFilm* film, float* out_rgb /* mean so far */, float* out_sumsq /* nullable */);
int lr_multi_film_save(const LrMultiFilm* film, const char* path);
int lr_multi_film_load(LrMultiScene* ms, const char* path, LrMultiFilm** out);
void lr_multi_film_destroy(LrMultiFilm* film);

/* ---- adaptive sampling on either film: samples only where the image is still noisy.  Each 8x4 pixel tile of the crop holds
 * its own sample count n.  A tile's error is the largest relative standard error of a pixel mean over its pixels and
 * channels, sqrt(var / n) / max(mean, 1e-3) with var = max(0, (Q - S * mean) / (n - 1)), computed in double precision
 * from the sums S and the sums of squares Q.  A tile is rendered when (n < 2 or (its S and Q are finite and its error >
 * threshold)) and (max_spp == 0 or n < max_spp).  Every tile continues from its own count with one thread per pixel, so each
 * pixel is bit for bit lr_render(splits = 1) at its tile's count, for any device count.  lr_film_render on a film whose
 * tiles differ renders every tile from its own count; lr_film_info's spp_done is then the fewest samples any pixel holds,
 * and lr_film_read divides every pixel by its tile's count.  A film whose tiles hold equal counts saves the LRFILM1
 * checkpoint; otherwise save writes LRFILM2, the same followed by the tile counts (int32, row-major), and both handles load
 * both. */
/* Adds spp_count samples to every tile of the film whose noise exceeds `threshold` (the rule above), each tile from its own
   sample count; tiles holding max_spp samples or more (max_spp > 0) are left alone, so a tile ends with fewer than
   max_spp + spp_count.  Without a cap a tile whose estimates can be negative may never converge.  *active_tiles (nullable)
   = tiles rendered; 0 means nothing was rendered.  Needs a film made with sums of squares; renders with splits = 1. */
int lr_film_render_adaptive(LrFilm* film, int32_t spp_count, float threshold, int32_t max_spp, int32_t* active_tiles, LrStats* stats);
int lr_film_spp_map(const LrFilm* film, int32_t* out /* crop_w*crop_h: samples held by each pixel */);
int lr_multi_film_render_adaptive(LrMultiFilm* film, int32_t spp_count, float threshold, int32_t max_spp, int32_t* active_tiles, LrStats* stats);
int lr_multi_film_spp_map(const LrMultiFilm* film, int32_t* out);

/* ---- parity probe: nearest hit of the primary ray through every film pixel with the
 * sensor jitter fixed to (u,v) and the aperture sample fixed to (ua,va).
 * prim[i] = primitive id or -1, t[i] = Intersection.distance (bvh.rs:131-141).      */
int lr_trace_primary(const LrScene* scene, float u, float v, float ua, float va,
                     int32_t* prim, float* t);
/* nearest hit of arbitrary rays (n rays, origins/directions 3 floats each) */
int lr_trace_rays(const LrScene* scene, int64_t n, const float* origins, const float* directions,
                  int32_t* prim, float* t, float* normal /* nullable, n*3 */);

/* the same with the kind of query stated: LR_QUERY_STRICT — the reference's leaf-AABB gate on every candidate (what
 * lr_trace_rays and lr_trace_primary run); LR_QUERY_RENDER — the query exactly as the render kernels run it (flat list,
 * tree-bounds test, optimistic traversal, the nearest tree hit gated once, strict re-trace if the gate rejects it).  Both
 * must answer alike; the second exists so that a replay divergence can be pinned on a ray.                         */
typedef enum LrQueryKind { LR_QUERY_STRICT = 0, LR_QUERY_RENDER = 1 } LrQueryKind;
int lr_trace_rays_query(const LrScene* scene, int64_t n, const float* origins, const float* directions, int32_t query,
                        int32_t* prim, float* t, float* normal /* nullable, n*3 */);

/* ---- measurement helpers ---- */
int lr_measure_l2_read_gbs(uint64_t working_set_bytes, int iters, float* gbs);
int lr_measure_hbm_read_gbs(uint64_t bytes, int iters, float* gbs);

/* ---- host front end (C++ restatement of scene_loader.rs + description.rs) ---- */
typedef struct LrHostScene LrHostScene;   /* owns the flat arrays an LrSceneDesc points into */

typedef struct LrSceneConfig {            /* [renderer] + [film] of the TOML          */
  int32_t samples, depth, depth_limit, no_direct_emitter, threads;
  int32_t integrator;                     /* LrIntegrator                              */
  int32_t width, height;
  int32_t output;                         /* 0 = png, 1 = hdr                          */
  float gamma;
  int32_t n_prims, n_emitters;
  float bvh_build_seconds;                /* host triangles -> host node array, whichever builder ran */
  int32_t bvh_builder;                    /* LrBvhBuilder that built the tree                          */
  float bvh_device_kernel_ms;             /* LR_BVH_DEVICE: CUDA-event time of the build kernels alone */
} LrSceneConfig;

/* Who builds the BVH (replaces BVH::new, src/bvh.rs:57-127; the nearest hit does not depend on the tree's topology):
 * LR_BVH_HOST   binned SAH on the host's cores — the better tree, seconds for a million triangles;
 * LR_BVH_DEVICE Morton-order radix tree (LBVH) built by CUDA kernels — milliseconds; needs a CUDA device.
 * lr_host_scene_load uses LR_BVH_HOST unless the environment says LR_BVH_BUILDER=device.                       */
typedef enum LrBvhBuilder { LR_BVH_HOST = 0, LR_BVH_DEVICE = 1 } LrBvhBuilder;
/* rebuilds the scene's BVH with the given builder (the LrSceneDesc pointer stays valid, its arrays are replaced) */
int lr_host_scene_rebuild_bvh(LrHostScene* hs, int32_t builder);

/* Parses `toml_path` (mesh/IBL paths resolved against asset_root, or the CWD if NULL — the
 * reference resolves against the CWD, description.rs:155, sky.rs:44).  width/height > 0
 * override [film] resolution (BASELINE configs 1 and 5 do). */
int lr_host_scene_load(const char* toml_path, const char* asset_root,
                       int32_t override_width, int32_t override_height, LrHostScene** out);
const LrSceneDesc* lr_host_scene_desc(const LrHostScene* hs);
int lr_host_scene_config(const LrHostScene* hs, LrSceneConfig* cfg);
void lr_host_scene_free(LrHostScene* hs);

/* Builds a host scene from raw arrays (triangles in any order; they are copied and permuted). */
int lr_host_scene_from_arrays(const LrMaterial* materials, int32_t n_materials,
                              const LrTriangle* triangles, int32_t n_triangles,
                              const LrSphere* spheres, int32_t n_spheres,
                              const LrCamera* camera, const LrSky* sky, LrHostScene** out);

/* camera constructors (host setup): matrix = 16 floats row-major as Matrix4.v (matrix4.rs:5-7) */
int lr_camera_ideal_pinhole(const float* matrix, float xfov_deg, int32_t w, int32_t h, LrCamera* out);
int lr_camera_thin_lens(const float* matrix, float xfov_deg, float focus_distance, float f_number,
                        int32_t w, int32_t h, LrCamera* out);
int lr_camera_omnidirectional(const float* matrix, int32_t w, int32_t h, LrCamera* out);
int lr_camera_pinhole(const float* position, const float* aperture_position, const float* sensor_size,
                      int32_t w, int32_t h, float aperture_radius, LrCamera* out);
/* transform helpers mirroring matrix4.rs:20-68 and scene_loader.rs:99-104 */
void lr_matrix_unit(float* m);
void lr_matrix_translate(const float* v, float* m);
void lr_matrix_scale(const float* v, float* m);
void lr_matrix_axis_angle(const float* axis, float angle_deg, float* m);
void lr_matrix_look_at(const float* origin, const float* target, const float* up, float* m);
void lr_matrix_mul(const float* a, const float* b, float* out);       /* out = a * b            */
void lr_matrix_apply(const float* m, const float* v3, float* out3);   /* M * (v,1), first 3 rows */

/* ---- output stage (main.rs:147-173, img.rs:40-63) ---- */
int lr_save_png(const char* path, const float* rgb, int32_t w, int32_t h, float gamma);
int lr_save_hdr(const char* path, const float* rgb, int32_t w, int32_t h);
int lr_load_hdr(const char* path, float** rgb /* malloc'ed, free with lr_free */, int32_t* w, int32_t* h);
void lr_free(void* p);

#ifdef __cplusplus
}
#endif
#endif /* LUMILLY_H */
