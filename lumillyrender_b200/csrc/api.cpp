// api.cpp — C ABI of liblumilly_b200.so: scene upload, render, probes, measurement helpers.
// The boundary replaces main.rs:70-132 (see include/lumilly.h).  No CPU fallback exists: every
// compute entry point needs a CUDA device and fails with LR_ERR_NO_DEVICE / LR_ERR_CUDA otherwise.
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <system_error>
#include <thread>
#include <vector>

#include "common.h"
#include "kernels.h"

namespace lr {

thread_local std::string g_error;
void set_error(const std::string& s) { g_error = s; }
int fail(int code, const std::string& s) { g_error = s; return code; }

static int g_device = -1;
static int g_sm_count = 0;
// pinned staging arena of lr_scene_create (grow-only, shared by all calls)
static std::mutex g_stage_mu;
static void* g_stage = nullptr;
static size_t g_stage_cap = 0;

#define LR_CUDA(call)                                                                      \
  do {                                                                                     \
    cudaError_t e__ = (call);                                                              \
    if (e__ != cudaSuccess)                                                                \
      return fail(LR_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));       \
  } while (0)

static int ensure_device() {
  if (g_device >= 0) return LR_OK;
  return lr_init(0);
}

// Device memory of the scene handle comes from the stream-ordered allocator with a pool that never trims (lr_init): a
// scene is created and destroyed once per end-to-end render, and cudaFree of tens of MB was measured to stall for
// 100-500 ms every few calls (tools/e2e_breakdown.py) while the pool hands the same blocks back in microseconds.
static cudaError_t dev_alloc(void** p, size_t bytes) {
  cudaError_t e = cudaMallocAsync(p, bytes, 0);
  if (e == cudaSuccess) e = cudaStreamSynchronize(0);      // usable from any stream afterwards
  return e;
}
static void dev_free(void* p) { if (p) cudaFreeAsync(p, 0); }

// Every entry point that works on a scene runs on the device that owns it, whichever device the calling thread has current
// (a host that talks to several GPUs switches devices between calls); the caller's device is restored on return.
struct OnDevice {
  int prev = -1;
  explicit OnDevice(int device) {
    int cur = -1;
    if (cudaGetDevice(&cur) == cudaSuccess && cur != device && cudaSetDevice(device) == cudaSuccess) prev = cur;
  }
  ~OnDevice() { if (prev >= 0) cudaSetDevice(prev); }
  OnDevice(const OnDevice&) = delete;
  OnDevice& operator=(const OnDevice&) = delete;
};

static inline float4 mk4(float x, float y, float z, float w) { float4 r; r.x = x; r.y = y; r.z = z; r.w = w; return r; }
static inline float as_float(int32_t i) { float f; std::memcpy(&f, &i, 4); return f; }

}  // namespace lr

using namespace lr;

struct LrScene {
  DevScene dev{};
  std::vector<void*> allocs;
  uint64_t h2d_bytes = 0;
  size_t block_bytes = 0;                          // size of the one device block (scene arrays + counter words)
  int width = 0, height = 0;
  unsigned long long* d_counters = nullptr;
  // scratch (mutable: owned by the handle, one caller thread at a time per LrScene)
  mutable float* d_film = nullptr; mutable size_t film_floats = 0;           // lr_render's sum / sum-of-squares buffers
  mutable float* d_film_sq = nullptr; mutable size_t film_sq_floats = 0;
  mutable float* d_partial = nullptr; mutable size_t partial_floats = 0;
  mutable float* d_partial_sq = nullptr; mutable size_t partial_sq_floats = 0;
  mutable uint64_t acc_samples = 0;
  mutable int acc_launches = 0;
  mutable int last_splits = 1;
  mutable float acc_kernel_ms = 0.0f;
  mutable cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  mutable bool ev_pending = false;
  bool has_ggx = false;                            // selects the render kernel built with GGX inline
  int device = 0, sm_count = 1;                    // the device that owns every pointer above, and its SM count
};

extern "C" {

int lr_abi_version(void) { return LR_ABI_VERSION; }
const char* lr_last_error(void) { return g_error.c_str(); }

int lr_init(int device) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n <= 0)
    return fail(LR_ERR_NO_DEVICE, std::string("no CUDA device available (") + (e != cudaSuccess ? cudaGetErrorString(e) : "count = 0") +
                                      "); liblumilly_b200 has no CPU fallback");
  if (device < 0 || device >= n) return fail(LR_ERR_INVALID, "device index out of range");
  e = cudaSetDevice(device);
  if (e != cudaSuccess) return fail(LR_ERR_NO_DEVICE, std::string("cudaSetDevice: ") + cudaGetErrorString(e));
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) return fail(LR_ERR_NO_DEVICE, std::string("cudaGetDeviceProperties: ") + cudaGetErrorString(e));
  g_device = device;
  g_sm_count = prop.multiProcessorCount;
  {
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
      unsigned long long keep = ~0ull;                    // never give freed blocks back to the driver
      cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
  }
  return LR_OK;
}

void lr_shutdown(void) { g_device = -1; }

int lr_device_info(int* sm_count, int* l2_bytes, int* sm_clock_khz, char* name, int name_len) {
  if (int rc = ensure_device()) return rc;
  cudaDeviceProp prop;
  LR_CUDA(cudaGetDeviceProperties(&prop, g_device));
  if (sm_count) *sm_count = prop.multiProcessorCount;
  if (l2_bytes) *l2_bytes = prop.l2CacheSize;
  if (sm_clock_khz) { int khz = 0; cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, g_device); *sm_clock_khz = khz; }
  if (name && name_len > 0) { std::strncpy(name, prop.name, name_len - 1); name[name_len - 1] = 0; }
  return LR_OK;
}

static int lr_scene_create_body(const LrSceneDesc* d, LrScene** out) {
  if (!d || !out) return fail(LR_ERR_INVALID, "null argument");
  *out = nullptr;
  if (int rc = validate_desc(*d)) return rc;
  if (int rc = ensure_device()) return rc;

  // ---- sizes.  Everything goes into ONE device block, packed on the host straight into a pinned staging arena and
  // uploaded with one copy (lr_scene_create is inside the timed region of an end-to-end render: 11 ms -> 4 ms).
  std::vector<char> emissive(d->n_materials, 0);
  for (int i = 0; i < d->n_materials; i++) {
    const LrMaterial& m = d->materials[i];
    // only Lambert carries emission (description.rs:94-101; every other material returns zero, e.g. ggx.rs:60-62)
    const bool lam = m.type == LR_MAT_LAMBERT;
    const float ex = lam ? m.emission[0] : 0.0f, ey = lam ? m.emission[1] : 0.0f, ez = lam ? m.emission[2] : 0.0f;
    emissive[i] = (ex * ex + ey * ey + ez * ez) > 0.0f;                 // emission().sqr_norm() > 0.0 (objects.rs:21)
  }
  // emitter table in instance (prim_id) order: objects.rs:18-29
  struct Em { int prim; float4 a, b, c; float area; };
  std::vector<Em> ems;
  for (int i = 0; i < d->n_triangles; i++) {
    const LrTriangle& t = d->triangles[i];
    if (!emissive[t.material]) continue;
    Em e; e.prim = t.prim_id; e.area = triangle_area(t.p0, t.p1, t.p2);
    e.a = mk4(t.p0[0], t.p0[1], t.p0[2], as_float(0));
    e.b = mk4(t.p1[0], t.p1[1], t.p1[2], e.area);
    e.c = mk4(t.p2[0], t.p2[1], t.p2[2], 0.0f);
    ems.push_back(e);
  }
  for (int i = 0; i < d->n_spheres; i++) {
    const LrSphere& sp = d->spheres[i];
    if (!emissive[sp.material]) continue;
    Em e; e.prim = sp.prim_id; e.area = sphere_area(sp.radius);
    e.a = mk4(sp.center[0], sp.center[1], sp.center[2], as_float(1));
    e.b = mk4(sp.radius, 0.0f, 0.0f, e.area);
    e.c = mk4(0.0f, 0.0f, 0.0f, 0.0f);
    ems.push_back(e);
  }
  std::sort(ems.begin(), ems.end(), [](const Em& x, const Em& y) { return x.prim < y.prim; });
  const size_t n_sky = d->sky.type == LR_SKY_IBL ? 2 * (size_t)d->sky.height * d->sky.height : 0;

  size_t total = 0;
  auto take = [&](size_t bytes) { const size_t at = total; total += (bytes + 255) & ~(size_t)255; return at; };
  const size_t o_nodes = take((size_t)d->n_nodes * 4 * sizeof(float4)), o_tris = take((size_t)d->n_triangles * 3 * sizeof(float4));
  const size_t o_tri_n = take((size_t)d->n_triangles * sizeof(float4)), o_tri_box = take((size_t)d->n_triangles * 2 * sizeof(float4));
  const size_t o_spheres = take((size_t)d->n_spheres * sizeof(float4)), o_sphere_meta = take((size_t)d->n_spheres * sizeof(int2));
  const size_t o_mats = take((size_t)d->n_materials * 3 * sizeof(float4));
  const size_t o_cdf = take(ems.size() * sizeof(float)), o_emitters = take(ems.size() * 3 * sizeof(float4));
  const size_t o_sky = take(n_sky * sizeof(float4));
  const size_t upload_bytes = total;
  const size_t o_counters = take(C_COUNT * sizeof(unsigned long long));

  struct SceneGuard { LrScene* s; ~SceneGuard() { if (s) lr_scene_destroy(s); } } guard{new LrScene()};   // released on success
  LrScene* s = guard.s;
  s->device = g_device; s->sm_count = std::max(g_sm_count, 1);
  cudaError_t e = cudaSuccess;
  DevScene& dv = s->dev;
  float area = 0.0f;
  {
    std::lock_guard<std::mutex> lock(g_stage_mu);
    if (g_stage_cap < upload_bytes) {
      if (g_stage) cudaFreeHost(g_stage);
      g_stage = nullptr; g_stage_cap = 0;
      e = cudaHostAlloc(&g_stage, upload_bytes + (upload_bytes >> 2), cudaHostAllocDefault);
      if (e == cudaSuccess) g_stage_cap = upload_bytes + (upload_bytes >> 2);
    }
    if (e == cudaSuccess) {
      char* h = (char*)g_stage;
      // ---- pack (layout documented in device_scene.h)
      float4* nodes = (float4*)(h + o_nodes); float4* tris = (float4*)(h + o_tris);
      float4* tri_n = (float4*)(h + o_tri_n); float4* tri_box = (float4*)(h + o_tri_box);
      float4* spheres = (float4*)(h + o_spheres); int2* sphere_meta = (int2*)(h + o_sphere_meta);
      float4* mats = (float4*)(h + o_mats); float* cdf = (float*)(h + o_cdf); float4* emitters = (float4*)(h + o_emitters);
      float4* sky = (float4*)(h + o_sky);
      if (d->n_nodes > 0) std::memcpy(nodes, d->nodes, (size_t)d->n_nodes * sizeof(LrBvhNode));
      // the per-triangle work (edges, box, normal: ~40 flops each) is independent: large meshes are packed by a few threads,
      // each writing its own range of the arena (lr_scene_create is inside the timed region of an end-to-end render)
      auto pack_tris = [&](int i0, int i1) {
        for (int i = i0; i < i1; i++) {
          const LrTriangle& t = d->triangles[i];
          // p0 and the edges of Moller-Trumbore, e1 = p1 - p0, e2 = p2 - p0 (triangle.rs:71-72): single fp32 subtractions
          const Vec3 e1 = vsub(vec3(t.p1), vec3(t.p0)), e2 = vsub(vec3(t.p2), vec3(t.p0));
          tris[3 * (size_t)i + 0] = mk4(t.p0[0], t.p0[1], t.p0[2], as_float(t.prim_id));
          tris[3 * (size_t)i + 1] = mk4(e1[0], e1[1], e1[2], as_float(t.material));
          tris[3 * (size_t)i + 2] = mk4(e2[0], e2[1], e2[2], 0.0f);
          // Triangle::aabb (triangle.rs:102-119): min / max of the vertices
          tri_box[2 * (size_t)i + 0] = mk4(std::fmin(std::fmin(t.p0[0], t.p1[0]), t.p2[0]), std::fmin(std::fmin(t.p0[1], t.p1[1]), t.p2[1]),
                                           std::fmin(std::fmin(t.p0[2], t.p1[2]), t.p2[2]), 0.0f);   // .w: same box as the predecessor (flat list, below)
          tri_box[2 * (size_t)i + 1] = mk4(std::fmax(std::fmax(t.p0[0], t.p1[0]), t.p2[0]), std::fmax(std::fmax(t.p0[1], t.p1[1]), t.p2[1]),
                                           std::fmax(std::fmax(t.p0[2], t.p1[2]), t.p2[2]), 0.0f);
          // triangle.rs:36  normal = (p1 - p0).cross(p2 - p0).normalize(), in the reference's fp32 operation order
          const Vec3 n = vnormalize(vcross(e1, e2));
          tri_n[i] = mk4(n[0], n[1], n[2], 0.0f);
        }
      };
      {
        const int hw = (int)std::thread::hardware_concurrency();
        const int workers = d->n_triangles >= 65536 ? std::max(1, std::min(8, hw)) : 1;
        // joined on every way out of this scope: a joinable std::thread that is destroyed calls std::terminate
        struct Joiner { std::vector<std::thread> v; ~Joiner() { for (std::thread& th : v) if (th.joinable()) th.join(); } } pool;
        pool.v.reserve(workers);                                 // no reallocation (and no bad_alloc) while threads run
        const int per = (d->n_triangles + workers - 1) / workers;
        int started = 1;                                         // ranges [0, started * per) are taken care of
        try {
          for (int w = 1; w < workers; w++) {
            pool.v.emplace_back(pack_tris, std::min(d->n_triangles, w * per), std::min(d->n_triangles, (w + 1) * per));
            started = w + 1;
          }
        } catch (const std::system_error&) {}                    // no thread to be had: this thread packs the rest
        pack_tris(0, std::min(d->n_triangles, per));
        if (started < workers) pack_tris(std::min(d->n_triangles, started * per), d->n_triangles);
        for (std::thread& th : pool.v) th.join();
      }
      // flat list: a triangle whose box equals its predecessor's (the two halves of a wall quad) shares that gate test
      for (int i = d->n_triangles - d->n_flat_triangles + 1; i < d->n_triangles; i++) {
        const float4 *a = tri_box + 2 * (size_t)(i - 1), *b = tri_box + 2 * (size_t)i;
        if (a[0].x == b[0].x && a[0].y == b[0].y && a[0].z == b[0].z && a[1].x == b[1].x && a[1].y == b[1].y && a[1].z == b[1].z)
          tri_box[2 * (size_t)i].w = 1.0f;
      }
      for (int i = 0; i < d->n_spheres; i++) {
        const LrSphere& sp = d->spheres[i];
        spheres[i] = mk4(sp.center[0], sp.center[1], sp.center[2], sp.radius);
        sphere_meta[i].x = sp.material; sphere_meta[i].y = sp.prim_id;
      }
      for (int i = 0; i < d->n_materials; i++) {
        const LrMaterial& m = d->materials[i];
        const bool lam = m.type == LR_MAT_LAMBERT;
        const float ex = lam ? m.emission[0] : 0.0f, ey = lam ? m.emission[1] : 0.0f, ez = lam ? m.emission[2] : 0.0f;
        const float weight = std::fmax(std::fmax(m.color[0], m.color[1]), m.color[2]);   // lambert.rs:27-30
        mats[3 * (size_t)i + 0] = mk4(m.color[0], m.color[1], m.color[2], as_float(m.type));
        mats[3 * (size_t)i + 1] = mk4(ex, ey, ez, m.param0);
        mats[3 * (size_t)i + 2] = mk4(m.param1, weight, emissive[i] ? 1.0f : 0.0f, 0.0f);
      }
      for (size_t i = 0; i < ems.size(); i++) {
        area += ems[i].area;                                            // `area += obj.area()` objects.rs:41
        cdf[i] = area;
        emitters[3 * i] = ems[i].a; emitters[3 * i + 1] = ems[i].b; emitters[3 * i + 2] = ems[i].c;
      }
      for (size_t i = 0; i < n_sky; i++) sky[i] = mk4(d->sky.pixels[3 * i], d->sky.pixels[3 * i + 1], d->sky.pixels[3 * i + 2], 0.0f);

      // ---- upload: one allocation, one copy
      char* block = nullptr;
      e = dev_alloc((void**)&block, total);
      if (e == cudaSuccess) {
        s->allocs.push_back(block);
        s->block_bytes = total;
        if (upload_bytes > 0) e = cudaMemcpyAsync(block, h, upload_bytes, cudaMemcpyHostToDevice, 0);
        if (e == cudaSuccess) e = cudaMemsetAsync(block + o_counters, 0, C_COUNT * sizeof(unsigned long long), 0);
        if (e == cudaSuccess) e = cudaStreamSynchronize(0);             // the arena is reused by the next call
        s->h2d_bytes = upload_bytes;
        auto at = [&](size_t off, size_t count) -> const void* { return count ? (const void*)(block + off) : nullptr; };
        dv.nodes = (const float4*)at(o_nodes, d->n_nodes); dv.tris = (const float4*)at(o_tris, d->n_triangles);
        dv.tri_n = (const float4*)at(o_tri_n, d->n_triangles); dv.tri_box = (const float4*)at(o_tri_box, d->n_triangles);
        dv.spheres = (const float4*)at(o_spheres, d->n_spheres); dv.sphere_meta = (const int2*)at(o_sphere_meta, d->n_spheres);
        dv.mats = (const float4*)at(o_mats, d->n_materials);
        dv.emitter_cdf = (const float*)at(o_cdf, ems.size()); dv.emitters = (const float4*)at(o_emitters, ems.size());
        dv.sky_pixels = (const float4*)at(o_sky, n_sky);
        s->d_counters = (unsigned long long*)(block + o_counters);
      }
    }
  }
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->ev0, cudaEventDefault);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->ev1, cudaEventDefault);
  if (e != cudaSuccess) return fail(LR_ERR_CUDA, std::string("scene upload: ") + cudaGetErrorString(e));   // the guard frees the scene
  dv.n_nodes = d->n_nodes; dv.n_tris = d->n_triangles; dv.n_spheres = d->n_spheres; dv.n_emitters = (int)ems.size();
  dv.n_bvh_tris = d->n_triangles - d->n_flat_triangles;
  for (int k = 0; k < 3; k++) {
    dv.bvh_lo[k] = d->n_nodes > 0 ? std::fmin(d->nodes[0].f[k], d->nodes[0].f[6 + k]) : 0.0f;
    dv.bvh_hi[k] = d->n_nodes > 0 ? std::fmax(d->nodes[0].f[3 + k], d->nodes[0].f[9 + k]) : 0.0f;
  }
  dv.emission_area = area;
  dv.sky_type = d->sky.type;
  dv.sky_color[0] = d->sky.color[0]; dv.sky_color[1] = d->sky.color[1]; dv.sky_color[2] = d->sky.color[2];
  dv.sky_height = d->sky.height;
  dv.sky_longitude_offset = d->sky.longitude_offset;
  dv.cam = d->camera;
  s->width = d->camera.width; s->height = d->camera.height;
  for (int i = 0; i < d->n_materials; i++) s->has_ggx = s->has_ggx || d->materials[i].type == LR_MAT_GGX;
  guard.s = nullptr;
  *out = s;
  return LR_OK;
}
int lr_scene_create(const LrSceneDesc* d, LrScene** out) { LR_GUARDED(lr_scene_create_body(d, out)); }

void lr_scene_destroy(LrScene* s) {
  if (!s) return;
  // work of this handle may still be in flight on a caller stream the legacy stream does not order against
  if (s->ev_pending && s->ev1) cudaEventSynchronize(s->ev1);
  int cur = -1;
  const bool hop = cudaGetDevice(&cur) == cudaSuccess && cur != s->device && !s->allocs.empty();
  if (hop) cudaSetDevice(s->device);                    // frees go to the owning device's stream
  for (void* p : s->allocs) dev_free(p);                // one block: scene arrays + the counter words
  dev_free(s->d_film);
  dev_free(s->d_film_sq);
  dev_free(s->d_partial);
  dev_free(s->d_partial_sq);
  if (s->ev0) cudaEventDestroy(s->ev0);
  if (s->ev1) cudaEventDestroy(s->ev1);
  if (hop) cudaSetDevice(cur);
  delete s;
}

int lr_scene_bytes(const LrScene* s, uint64_t* h2d_bytes) {
  if (!s || !h2d_bytes) return fail(LR_ERR_INVALID, "null argument");
  *h2d_bytes = s->h2d_bytes;
  return LR_OK;
}

// One part of a pixel-sharded film (lr_multi_film_*): shard `index` of `count` (device_scene.h: shard_of_tile).  Such a
// render always runs one thread per pixel, adding its samples in order (splits = 1), whatever LR_SPLITS says.
struct FilmShard { int index, count; };

static int resolve_params(const LrScene* s, const LrRenderParams* p, DevParams& dp, const FilmShard* shard = nullptr) {
  if (!s || !p) return fail(LR_ERR_INVALID, "null argument");
  if (p->integrator != LR_INTEGRATOR_PT && p->integrator != LR_INTEGRATOR_PT_DIRECT)
    return fail(LR_ERR_INVALID, "Unknown integrator type");            // main.rs:124
  if (p->spp_count <= 0 || p->spp_begin < 0) return fail(LR_ERR_INVALID, "spp range must be non-empty and non-negative");
  if (p->depth < 0 || p->depth_limit < 0) return fail(LR_ERR_INVALID, "depth and depth_limit must be >= 0");
  dp.integrator = p->integrator;
  dp.spp_begin = p->spp_begin; dp.spp_count = p->spp_count;
  dp.depth = p->depth; dp.depth_limit = p->depth_limit; dp.no_direct_emitter = p->no_direct_emitter ? 1 : 0;
  dp.seed = p->seed;
  if (p->crop_w > 0) {
    if (p->crop_h <= 0 || p->crop_x < 0 || p->crop_y < 0 || p->crop_x + p->crop_w > s->width || p->crop_y + p->crop_h > s->height)
      return fail(LR_ERR_INVALID, "crop window outside the film");
    dp.crop_x = p->crop_x; dp.crop_y = p->crop_y; dp.crop_w = p->crop_w; dp.crop_h = p->crop_h;
  } else {
    dp.crop_x = 0; dp.crop_y = 0; dp.crop_w = s->width; dp.crop_h = s->height;
  }
  dp.tiles_x = (dp.crop_w + 7) / 8; dp.tiles_y = (dp.crop_h + 3) / 4;
  int splits = shard ? 1 : p->splits;
  if (const char* e_splits = std::getenv("LR_SPLITS"); e_splits && !shard) splits = std::atoi(e_splits);   // development knob
  if (splits <= 0) {
    // auto: enough threads for ~2 full waves of 148 SMs x 2048 resident threads, >= 4 samples per thread
    const long long px_threads = (long long)dp.tiles_x * dp.tiles_y * 32;
    const long long target = 2LL * std::max(g_sm_count, 1) * 2048;
    splits = (int)std::min<long long>((target + px_threads - 1) / px_threads, std::max(1, p->spp_count / 4));
  }
  splits = std::max(1, std::min(splits, p->spp_count));
  // partial buffers must stay modest (<= 1 GiB)
  const size_t px = (size_t)dp.crop_w * dp.crop_h;
  while (splits > 1 && px * 3 * sizeof(float) * splits > (1ull << 30)) splits--;
  dp.splits = splits;
  dp.shard = shard ? shard->index : 0;
  dp.n_shards = shard ? shard->count : 1;
  dp.unit_tiles = shard_tile_count(dp.tiles_x * dp.tiles_y, dp.shard, dp.n_shards);
  // kernel organisation knobs (development / profiling only; defaults are the measured best, DESIGN.md §4)
  const char* e_di = std::getenv("LR_DEFER_ITERS");
  const char* e_dt = std::getenv("LR_DEFER_THRESH");
  dp.defer_iters = e_di ? std::max(1, std::atoi(e_di)) : 3;
  dp.defer_thresh = e_dt ? std::max(1, std::min(32, std::atoi(e_dt))) : 12;
  // both organisations of the render kernel are built for scenes with a BVH; tests render with each and compare bits
  const char* e_org = std::getenv("LR_ORGANISATION");
  dp.organisation = !e_org ? 0 : (std::strcmp(e_org, "persistent") == 0 ? 1 : (std::strcmp(e_org, "pool") == 0 ? 2 : 0));

  return LR_OK;
}

static int ensure_scratch(float** buf, size_t* have, size_t need) {
  if (*have >= need) return LR_OK;
  dev_free(*buf);
  *buf = nullptr; *have = 0;
  LR_CUDA(dev_alloc((void**)buf, need * sizeof(float)));
  *have = need;
  return LR_OK;
}

// pixels of the crop inside the shard's tiles (the tiles on the right and bottom edges may be partly outside the crop)
static uint64_t shard_pixels(const DevParams& dp) {
  if (dp.n_shards == 1) return (uint64_t)dp.crop_w * dp.crop_h;
  uint64_t n = 0;
  for (int j = 0; j < dp.unit_tiles; j++) {
    const int t = shard_tile(j, dp.shard, dp.n_shards), tx = t % dp.tiles_x, ty = t / dp.tiles_x;
    n += (uint64_t)std::min(8, dp.crop_w - 8 * tx) * (uint64_t)std::min(4, dp.crop_h - 4 * ty);
  }
  return n;
}

// lr_render_accumulate_device for the whole crop (shard = nullptr) or for one shard of its tiles (lr_multi_film_render)
static int accumulate(const LrScene* s, const LrRenderParams* p, float* d_sum, float* d_sumsq, void* cuda_stream, const FilmShard* shard) {
  if (!s) return fail(LR_ERR_INVALID, "null argument");
  const OnDevice on(s->device);
  DevParams dp;
  if (int rc = resolve_params(s, p, dp, shard)) return rc;
  if (!d_sum) return fail(LR_ERR_INVALID, "d_sum is null");
  if (int rc = ensure_device()) return rc;
  cudaStream_t st = (cudaStream_t)cuda_stream;
  const size_t n = (size_t)dp.crop_w * dp.crop_h * 3;
  float* ksum = d_sum; float* ksq = d_sumsq;
  // The previous launch (possibly on a non-blocking stream the legacy stream does not order against) may still be using
  // the partial buffers: wait for it BEFORE ensure_scratch can hand them back to the pool, and fold its time while here.
  if (s->ev_pending) {
    float ms = 0.0f;
    if (cudaEventSynchronize(s->ev1) == cudaSuccess && cudaEventElapsedTime(&ms, s->ev0, s->ev1) == cudaSuccess) s->acc_kernel_ms += ms;
    s->ev_pending = false;
  }
  if (dp.unit_tiles == 0) return LR_OK;                   // a shard without tiles (a crop smaller than the shard count)
  if (dp.splits > 1) {
    if (int rc = ensure_scratch(&s->d_partial, &s->partial_floats, n * dp.splits)) return rc;
    ksum = s->d_partial;
    if (d_sumsq) {
      if (int rc = ensure_scratch(&s->d_partial_sq, &s->partial_sq_floats, n * dp.splits)) return rc;
      ksq = s->d_partial_sq;
    }
  }
  LR_CUDA(cudaEventRecord(s->ev0, st));
  {
    // the unit cursor lives in the last word of the counter block (reset on the stream before every launch)
    unsigned int* next_unit = reinterpret_cast<unsigned int*>(s->d_counters + C_NEXT_UNIT);
    LR_CUDA(cudaMemsetAsync(next_unit, 0, sizeof(unsigned long long), st));
    LR_CUDA(launch_render_persistent(s->dev, dp, s->has_ggx, p->count_traversal != 0, ksum, d_sumsq ? ksq : nullptr, s->d_counters, next_unit,
                                     std::max(s->sm_count, 1), st));
    s->acc_launches++;
  }
  if (dp.splits > 1) {
    LR_CUDA(launch_reduce_splits(d_sum, s->d_partial, n, dp.splits, st));
    s->acc_launches++;
    if (d_sumsq) { LR_CUDA(launch_reduce_splits(d_sumsq, s->d_partial_sq, n, dp.splits, st)); s->acc_launches++; }
  }
  LR_CUDA(cudaEventRecord(s->ev1, st));
  s->ev_pending = true;
  s->acc_samples += shard_pixels(dp) * (uint64_t)dp.spp_count;
  s->last_splits = dp.splits;
  return LR_OK;
}

int lr_render_accumulate_device(const LrScene* s, const LrRenderParams* p, float* d_sum, float* d_sumsq, void* cuda_stream) {
  return accumulate(s, p, d_sum, d_sumsq, cuda_stream, nullptr);
}

int lr_stats_fetch(const LrScene* s, void* cuda_stream, LrStats* stats) {
  if (!s || !stats) return fail(LR_ERR_INVALID, "null argument");
  const OnDevice on(s->device);
  if (!s || !stats) return fail(LR_ERR_INVALID, "null argument");
  cudaStream_t st = (cudaStream_t)cuda_stream;
  LR_CUDA(cudaStreamSynchronize(st));
  if (s->ev_pending) {
    float ms = 0.0f;
    LR_CUDA(cudaEventSynchronize(s->ev1));
    LR_CUDA(cudaEventElapsedTime(&ms, s->ev0, s->ev1));
    s->acc_kernel_ms += ms;
    s->ev_pending = false;
  }
  unsigned long long c[C_COUNT];
  LR_CUDA(cudaMemcpy(c, s->d_counters, sizeof(c), cudaMemcpyDeviceToHost));
  LR_CUDA(cudaMemset(s->d_counters, 0, sizeof(c)));
  std::memset(stats, 0, sizeof(*stats));
  stats->rays = c[C_RAYS]; stats->nonfinite_samples = c[C_NONFINITE]; stats->gate_retraces = c[C_RETRACE];
  stats->nodes_visited = c[C_NODES]; stats->tris_tested = c[C_TRIS]; stats->spheres_tested = c[C_SPHERES];
  stats->flat_tris_tested = c[C_FLAT_TRIS]; stats->flat_boxes_tested = c[C_FLAT_BOXES];
  stats->samples = s->acc_samples; stats->kernel_ms = s->acc_kernel_ms; stats->launches = s->acc_launches; stats->splits = s->last_splits;
  s->acc_samples = 0; s->acc_kernel_ms = 0.0f; s->acc_launches = 0;
  return LR_OK;
}

int lr_render(const LrScene* s, const LrRenderParams* p, float* out_rgb, float* out_sumsq, LrStats* stats) {
  if (!s) return fail(LR_ERR_INVALID, "null argument");
  const OnDevice on(s->device);
  DevParams dp;
  if (int rc = resolve_params(s, p, dp)) return rc;
  if (!out_rgb) return fail(LR_ERR_INVALID, "out_rgb is null");
  if (int rc = ensure_device()) return rc;
  const size_t n = (size_t)dp.crop_w * dp.crop_h * 3;
  // the film buffers live in the scene handle between calls (no cudaMalloc / cudaFree inside an end-to-end render)
  if (int rc = ensure_scratch(&s->d_film, &s->film_floats, n)) return rc;
  if (out_sumsq) if (int rc = ensure_scratch(&s->d_film_sq, &s->film_sq_floats, n)) return rc;
  float *d_sum = s->d_film, *d_sq = out_sumsq ? s->d_film_sq : nullptr;
  int rc = LR_OK;
  do {
    if (cudaMemsetAsync(d_sum, 0, n * sizeof(float), 0) != cudaSuccess) { rc = fail(LR_ERR_CUDA, "cudaMemsetAsync failed"); break; }
    if (out_sumsq && cudaMemsetAsync(d_sq, 0, n * sizeof(float), 0) != cudaSuccess) { rc = fail(LR_ERR_CUDA, "cudaMemsetAsync failed"); break; }
    LrStats dummy;
    if (stats == nullptr) stats = &dummy;
    // drop counters of earlier accumulate calls so the stats describe this call only
    if ((rc = lr_stats_fetch(s, nullptr, stats)) != LR_OK) break;
    if ((rc = lr_render_accumulate_device(s, p, d_sum, d_sq, nullptr)) != LR_OK) break;
    cudaError_t e = launch_scale(d_sum, n, (float)dp.spp_count, 0);     // main.rs:104
    if (e != cudaSuccess) { rc = fail(LR_ERR_CUDA, std::string("scale: ") + cudaGetErrorString(e)); break; }
    if ((rc = lr_stats_fetch(s, nullptr, stats)) != LR_OK) break;
    stats->launches += 1;
    e = cudaMemcpy(out_rgb, d_sum, n * sizeof(float), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && out_sumsq) e = cudaMemcpy(out_sumsq, d_sq, n * sizeof(float), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) { rc = fail(LR_ERR_CUDA, std::string("D2H: ") + cudaGetErrorString(e)); break; }
  } while (0);
  return rc;
}

int lr_render_aov(const LrScene* s, const LrRenderParams* p, int32_t kind, float* out) {
  if (!s) return fail(LR_ERR_INVALID, "null argument");
  const OnDevice on(s->device);
  if (!s || !p || !out) return fail(LR_ERR_INVALID, "null argument");
  if (kind != LR_AOV_NORMAL && kind != LR_AOV_DEPTH) return fail(LR_ERR_INVALID, "unknown AOV kind");
  LrRenderParams q = *p;
  q.integrator = LR_INTEGRATOR_PT;                      // not used by the AOVs
  DevParams dp;
  if (int rc = resolve_params(s, &q, dp)) return rc;
  if (int rc = ensure_device()) return rc;
  const size_t n = (size_t)dp.crop_w * dp.crop_h * (kind == LR_AOV_NORMAL ? 3 : 1);
  float* d_out = nullptr;
  LR_CUDA(dev_alloc((void**)&d_out, n * sizeof(float)));
  cudaError_t e = launch_aov(s->dev, dp, kind, d_out, 0);
  if (e == cudaSuccess) e = cudaMemcpy(out, d_out, n * sizeof(float), cudaMemcpyDeviceToHost);
  dev_free(d_out);
  if (e != cudaSuccess) return fail(LR_ERR_CUDA, std::string("render_aov: ") + cudaGetErrorString(e));
  return LR_OK;
}

int lr_shard_range(int32_t spp_begin, int32_t spp_count, int32_t part, int32_t n_parts, int32_t* begin, int32_t* count) {
  if (!begin || !count) return fail(LR_ERR_INVALID, "null argument");
  if (n_parts <= 0 || part < 0 || part >= n_parts || spp_count < 0 || spp_begin < 0) return fail(LR_ERR_INVALID, "bad shard request");
  const int per = spp_count / n_parts, rem = spp_count % n_parts;
  *begin = spp_begin + part * per + std::min(part, rem);
  *count = per + (part < rem ? 1 : 0);
  return LR_OK;
}

// A copy of a device scene on the CURRENT device: the packed block travels device to device (NVLink) instead of being
// packed and uploaded from the host again, and the array pointers are rebased into the new block.
static int scene_clone(const LrScene* src, int src_device, int dst_device, LrScene** out) {
  *out = nullptr;
  if (src->allocs.size() != 1 || src->block_bytes == 0) return fail(LR_ERR_INVALID, "scene_clone: unexpected scene layout");
  LrScene* s = new LrScene();
  s->device = dst_device; s->sm_count = std::max(g_sm_count, 1);       // lr_init(dst_device) ran just before
  char* block = nullptr;
  const char* from = (const char*)src->allocs[0];
  cudaError_t e = dev_alloc((void**)&block, src->block_bytes);
  if (e == cudaSuccess) {
    s->allocs.push_back(block);
    s->block_bytes = src->block_bytes;
    e = cudaMemcpyPeerAsync(block, dst_device, from, src_device, src->h2d_bytes, 0);
  }
  const size_t o_counters = (const char*)src->d_counters - from;
  if (e == cudaSuccess) e = cudaMemsetAsync(block + o_counters, 0, C_COUNT * sizeof(unsigned long long), 0);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->ev0, cudaEventDefault);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->ev1, cudaEventDefault);
  if (e != cudaSuccess) {
    const std::string msg = std::string("scene clone: ") + cudaGetErrorString(e);
    lr_scene_destroy(s);
    return fail(LR_ERR_CUDA, msg);
  }
  s->dev = src->dev;
  auto rebase = [&](const void* p) -> const void* { return p ? (const void*)(block + ((const char*)p - from)) : nullptr; };
  s->dev.nodes = (const float4*)rebase(src->dev.nodes); s->dev.tris = (const float4*)rebase(src->dev.tris);
  s->dev.tri_n = (const float4*)rebase(src->dev.tri_n); s->dev.tri_box = (const float4*)rebase(src->dev.tri_box);
  s->dev.spheres = (const float4*)rebase(src->dev.spheres); s->dev.sphere_meta = (const int2*)rebase(src->dev.sphere_meta);
  s->dev.mats = (const float4*)rebase(src->dev.mats);
  s->dev.emitter_cdf = (const float*)rebase(src->dev.emitter_cdf); s->dev.emitters = (const float4*)rebase(src->dev.emitters);
  s->dev.sky_pixels = (const float4*)rebase(src->dev.sky_pixels);
  s->d_counters = (unsigned long long*)(block + o_counters);
  s->h2d_bytes = src->h2d_bytes;
  s->width = src->width; s->height = src->height; s->has_ggx = src->has_ggx;
  *out = s;
  return LR_OK;
}

// ---------------------------------------------------------------- one process, several GPUs
}  // extern "C"

// The scene on every listed device, with everything a render needs set up ONCE: the clones, a non-blocking stream and a
// completion event per device, the peer mappings that let devices[0] read the others' film buffers (pool access has a
// first-use cost of ~100 ms per device pair: it was the "set-up spike" of calling lr_render_multi repeatedly).
struct LrMultiScene {
  int n = 0;
  int devices[kMaxPeers] = {};
  LrScene* scenes[kMaxPeers] = {};
  cudaStream_t streams[kMaxPeers] = {};
  cudaEvent_t done[kMaxPeers] = {};
  bool mapped[kMaxPeers] = {};
  float* staged = nullptr;                 // on devices[0]: copies of the film buffers it cannot map
  size_t staged_floats = 0;
  int home = 0;
};

namespace {

// device i's stream-ordered pool grants `reader` access (plain cudaDeviceEnablePeerAccess covers cudaMalloc memory only)
bool map_peer(int reader, int owner) {
  int can = 0;
  if (std::getenv("LR_MULTI_NO_PEER") != nullptr) return false;          // development / tests: force the staged path
  if (cudaDeviceCanAccessPeer(&can, reader, owner) != cudaSuccess || !can) { cudaGetLastError(); return false; }
  if (cudaSetDevice(reader) != cudaSuccess) return false;
  const cudaError_t pe = cudaDeviceEnablePeerAccess(owner, 0);
  if (pe != cudaSuccess && pe != cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); return false; }
  cudaGetLastError();
  cudaMemPool_t pool;
  cudaMemAccessDesc ad;
  std::memset(&ad, 0, sizeof(ad));
  ad.location.type = cudaMemLocationTypeDevice;
  ad.location.id = reader;
  ad.flags = cudaMemAccessFlagsProtReadWrite;
  if (cudaDeviceGetDefaultMemPool(&pool, owner) != cudaSuccess || cudaMemPoolSetAccess(pool, &ad, 1) != cudaSuccess) { cudaGetLastError(); return false; }
  return true;
}

int multi_create(const LrSceneDesc* desc, int32_t n_devices, const int32_t* devices, LrMultiScene** out) {
  if (!desc || !devices || !out) return fail(LR_ERR_INVALID, "null argument");
  *out = nullptr;
  if (n_devices < 1 || n_devices > kMaxPeers) return fail(LR_ERR_INVALID, "lr_render_multi takes 1..8 devices");
  int n_visible = 0;
  if (cudaGetDeviceCount(&n_visible) != cudaSuccess || n_visible <= 0)
    return fail(LR_ERR_NO_DEVICE, "no CUDA device available; liblumilly_b200 has no CPU fallback");
  for (int i = 0; i < n_devices; i++) {
    if (devices[i] < 0 || devices[i] >= n_visible) return fail(LR_ERR_INVALID, "device index out of range");
    for (int j = 0; j < i; j++) if (devices[j] == devices[i]) return fail(LR_ERR_INVALID, "device listed twice");
  }
  int prev_device = 0;
  cudaGetDevice(&prev_device);
  LrMultiScene* m = new LrMultiScene();
  m->n = n_devices;
  m->home = g_device >= 0 ? g_device : devices[0];
  for (int i = 0; i < n_devices; i++) m->devices[i] = devices[i];
  int rc = LR_OK;
  // scenes first: the first device gets the scene from the host, the others a device-to-device copy of its packed block
  for (int i = 0; i < n_devices && rc == LR_OK; i++) {
    if ((rc = lr_init(devices[i])) != LR_OK) break;          // cudaSetDevice + the non-trimming memory pool
    if ((rc = i == 0 ? lr_scene_create(desc, &m->scenes[0]) : scene_clone(m->scenes[0], devices[0], devices[i], &m->scenes[i])) != LR_OK) break;
    cudaError_t e = cudaStreamCreateWithFlags(&m->streams[i], cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&m->done[i], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaStreamSynchronize(0);      // the clone has landed
    if (e != cudaSuccess) rc = fail(LR_ERR_CUDA, std::string("lr_multi_scene_create: ") + cudaGetErrorString(e));
  }
  m->mapped[0] = true;
  for (int i = 1; i < n_devices && rc == LR_OK; i++) m->mapped[i] = map_peer(devices[0], devices[i]);
  cudaSetDevice(m->home >= 0 && m->home < n_visible ? m->home : prev_device);
  g_device = m->home;
  if (rc != LR_OK) {
    const std::string err = g_error;
    lr_multi_scene_destroy(m);
    g_error = err;
    return rc;
  }
  *out = m;
  return LR_OK;
}

// statistics of several devices: totals, the slowest device's kernel time
void add_device_stats(LrStats& total, const LrStats& st) {
  total.rays += st.rays; total.samples += st.samples; total.nodes_visited += st.nodes_visited; total.tris_tested += st.tris_tested;
  total.spheres_tested += st.spheres_tested; total.nonfinite_samples += st.nonfinite_samples; total.gate_retraces += st.gate_retraces;
  total.flat_tris_tested += st.flat_tris_tested; total.flat_boxes_tested += st.flat_boxes_tested;
  total.kernel_ms = std::max(total.kernel_ms, st.kernel_ms);
  total.launches += st.launches;
  total.splits = std::max(total.splits, st.splits);
}

int multi_render(LrMultiScene* m, const LrRenderParams* p, float* out_rgb, float* out_sumsq, LrStats* stats) {
  if (!m || !p || !out_rgb) return fail(LR_ERR_INVALID, "null argument");
  if (p->spp_count <= 0 || p->spp_begin < 0) return fail(LR_ERR_INVALID, "spp range must be non-empty and non-negative");
  const int n_devices = m->n;
  // LR_MULTI_TRACE=1: wall-clock milliseconds of each phase on stderr (development)
  const bool trace_on = std::getenv("LR_MULTI_TRACE") != nullptr;
  auto t_prev = std::chrono::steady_clock::now();
  auto lap = [&](const char* what) {
    if (!trace_on) return;
    const auto now = std::chrono::steady_clock::now();
    std::fprintf(stderr, "lr_multi_render %-10s %8.2f ms\n", what, std::chrono::duration<float, std::milli>(now - t_prev).count());
    t_prev = now;
  };
  LrRenderParams parts[kMaxPeers];
  size_t n = 0;
  int rc = LR_OK;
  LrStats total;
  std::memset(&total, 0, sizeof(total));
  do {
    // ---- launch: asynchronous on every device's own stream, so the devices render concurrently
    for (int i = 0; i < n_devices && rc == LR_OK; i++) {
      cudaError_t e = cudaSetDevice(m->devices[i]);
      if (e != cudaSuccess) { rc = fail(LR_ERR_CUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(e)); break; }
      g_device = m->devices[i];
      const LrScene* s = m->scenes[i];
      parts[i] = *p;
      if ((rc = lr_shard_range(p->spp_begin, p->spp_count, i, n_devices, &parts[i].spp_begin, &parts[i].spp_count)) != LR_OK) break;
      DevParams dp;
      LrRenderParams probe = parts[i];
      if (probe.spp_count == 0) probe.spp_count = 1;         // more devices than samples: this one only contributes zeros
      if ((rc = resolve_params(s, &probe, dp)) != LR_OK) break;
      n = (size_t)dp.crop_w * dp.crop_h * 3;
      if ((rc = ensure_scratch(&s->d_film, &s->film_floats, n)) != LR_OK) break;
      if (out_sumsq && (rc = ensure_scratch(&s->d_film_sq, &s->film_sq_floats, n)) != LR_OK) break;
      e = cudaMemsetAsync(s->d_film, 0, n * sizeof(float), m->streams[i]);
      if (e == cudaSuccess && out_sumsq) e = cudaMemsetAsync(s->d_film_sq, 0, n * sizeof(float), m->streams[i]);
      if (e != cudaSuccess) { rc = fail(LR_ERR_CUDA, std::string("lr_multi_render set-up: ") + cudaGetErrorString(e)); break; }
      if (parts[i].spp_count > 0 &&
          (rc = lr_render_accumulate_device(s, &parts[i], s->d_film, out_sumsq ? s->d_film_sq : nullptr, m->streams[i])) != LR_OK) break;
      e = cudaEventRecord(m->done[i], m->streams[i]);
      if (e != cudaSuccess) { rc = fail(LR_ERR_CUDA, std::string("cudaEventRecord: ") + cudaGetErrorString(e)); break; }
    }
    if (rc != LR_OK) break;
    lap("launch");

    // ---- reduce + normalise on devices[0]: one kernel reads every device's sums (peer access over NVLink; a staged copy
    // where a peer cannot be mapped), adds them in list order and divides by spp (main.rs:104)
    cudaError_t e = cudaSetDevice(m->devices[0]);
    g_device = m->devices[0];
    cudaStream_t st0 = m->streams[0];
    PeerBuffers sum_src, sq_src;
    sum_src.count = sq_src.count = n_devices;
    size_t need_staged = 0;
    for (int i = 1; i < n_devices; i++) if (!m->mapped[i]) need_staged += n * (out_sumsq ? 2 : 1);
    if (e == cudaSuccess && need_staged > m->staged_floats) {
      dev_free(m->staged);
      m->staged = nullptr; m->staged_floats = 0;
      e = dev_alloc((void**)&m->staged, need_staged * sizeof(float));
      if (e == cudaSuccess) m->staged_floats = need_staged;
    }
    float* stage_next = m->staged;
    for (int i = 0; i < n_devices && e == cudaSuccess; i++) {
      if (i > 0) e = cudaStreamWaitEvent(st0, m->done[i], 0);     // devices[0]'s stream waits for device i's render
      if (e != cudaSuccess) break;
      sum_src.p[i] = m->scenes[i]->d_film;
      sq_src.p[i] = out_sumsq ? m->scenes[i]->d_film_sq : nullptr;
      if (!m->mapped[i]) {
        e = cudaMemcpyPeerAsync(stage_next, m->devices[0], m->scenes[i]->d_film, m->devices[i], n * sizeof(float), st0);
        sum_src.p[i] = stage_next; stage_next += n;
        if (e == cudaSuccess && out_sumsq) {
          e = cudaMemcpyPeerAsync(stage_next, m->devices[0], m->scenes[i]->d_film_sq, m->devices[i], n * sizeof(float), st0);
          sq_src.p[i] = stage_next; stage_next += n;
        }
      }
    }
    if (e == cudaSuccess) e = launch_reduce_peers(m->scenes[0]->d_film, sum_src, n, (float)p->spp_count, st0);   // main.rs:104
    if (e == cudaSuccess && out_sumsq) e = launch_reduce_peers(m->scenes[0]->d_film_sq, sq_src, n, 0.0f, st0);
    if (e == cudaSuccess) e = cudaMemcpyAsync(out_rgb, m->scenes[0]->d_film, n * sizeof(float), cudaMemcpyDeviceToHost, st0);
    if (e == cudaSuccess && out_sumsq) e = cudaMemcpyAsync(out_sumsq, m->scenes[0]->d_film_sq, n * sizeof(float), cudaMemcpyDeviceToHost, st0);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st0);
    if (e != cudaSuccess) { rc = fail(LR_ERR_CUDA, std::string("lr_multi_render reduce: ") + cudaGetErrorString(e)); break; }
    lap("render+d2h");

    // ---- statistics: totals over the devices, the slowest device's kernel time
    for (int i = 0; i < n_devices && rc == LR_OK; i++) {
      if (cudaSetDevice(m->devices[i]) != cudaSuccess) { rc = fail(LR_ERR_CUDA, "cudaSetDevice failed"); break; }
      g_device = m->devices[i];
      LrStats st;
      if ((rc = lr_stats_fetch(m->scenes[i], m->streams[i], &st)) != LR_OK) break;
      add_device_stats(total, st);
    }
    total.launches += out_sumsq ? 2 : 1;
  } while (0);
  const std::string err = g_error;
  if (rc != LR_OK) for (int i = 0; i < n_devices; i++) { cudaSetDevice(m->devices[i]); cudaDeviceSynchronize(); }   // nothing of this call stays in flight
  cudaSetDevice(m->home);
  g_device = m->home;
  lap("stats");
  if (rc != LR_OK) { g_error = err; return rc; }
  if (stats) *stats = total;
  return LR_OK;
}

}  // namespace

extern "C" {

int lr_multi_scene_create(const LrSceneDesc* desc, int32_t n_devices, const int32_t* devices, LrMultiScene** out) {
  LR_GUARDED(multi_create(desc, n_devices, devices, out));
}

int lr_multi_render(LrMultiScene* m, const LrRenderParams* p, float* out_rgb, float* out_sumsq, LrStats* stats) {
  LR_GUARDED(multi_render(m, p, out_rgb, out_sumsq, stats));
}

void lr_multi_scene_destroy(LrMultiScene* m) {
  if (!m) return;
  int prev = 0;
  cudaGetDevice(&prev);
  for (int i = 0; i < m->n; i++) {
    if (!m->scenes[i] && !m->streams[i] && !m->done[i]) continue;
    cudaSetDevice(m->devices[i]);
    cudaDeviceSynchronize();
    if (i == 0 && m->staged) dev_free(m->staged);
    lr_scene_destroy(m->scenes[i]);
    if (m->done[i]) cudaEventDestroy(m->done[i]);
    if (m->streams[i]) cudaStreamDestroy(m->streams[i]);
  }
  cudaSetDevice(prev);
  delete m;
}

// one-shot form: set-up, one render, tear-down
int lr_render_multi(const LrSceneDesc* desc, const LrRenderParams* p, int32_t n_devices, const int32_t* devices, float* out_rgb,
                    float* out_sumsq, LrStats* stats) {
  if (!desc || !p || !devices || !out_rgb) return fail(LR_ERR_INVALID, "null argument");
  if (p->spp_count <= 0 || p->spp_begin < 0) return fail(LR_ERR_INVALID, "spp range must be non-empty and non-negative");
  LrMultiScene* m = nullptr;
  if (int rc = lr_multi_scene_create(desc, n_devices, devices, &m)) return rc;
  const int rc = lr_multi_render(m, p, out_rgb, out_sumsq, stats);
  const std::string err = g_error;
  lr_multi_scene_destroy(m);
  g_error = err;
  return rc;
}

int lr_trace_primary(const LrScene* s, float u, float v, float ua, float va, int32_t* prim, float* t) {
  if (!s) return fail(LR_ERR_INVALID, "null argument");
  const OnDevice on(s->device);
  if (!s || !prim || !t) return fail(LR_ERR_INVALID, "null argument");
  if (int rc = ensure_device()) return rc;
  const size_t n = (size_t)s->width * s->height;
  int* d_prim = nullptr; float* d_t = nullptr;
  LR_CUDA(cudaMalloc((void**)&d_prim, n * sizeof(int)));
  cudaError_t e = cudaMalloc((void**)&d_t, n * sizeof(float));
  if (e == cudaSuccess) e = launch_primary(s->dev, u, v, ua, va, d_prim, d_t, 0);
  if (e == cudaSuccess) e = cudaMemcpy(prim, d_prim, n * sizeof(int), cudaMemcpyDeviceToHost);
  if (e == cudaSuccess) e = cudaMemcpy(t, d_t, n * sizeof(float), cudaMemcpyDeviceToHost);
  cudaFree(d_prim);
  if (d_t) cudaFree(d_t);
  if (e != cudaSuccess) return fail(LR_ERR_CUDA, std::string("trace_primary: ") + cudaGetErrorString(e));
  return LR_OK;
}

int lr_trace_rays(const LrScene* s, int64_t n, const float* origins, const float* directions, int32_t* prim, float* t, float* normal) {
  return lr_trace_rays_query(s, n, origins, directions, LR_QUERY_STRICT, prim, t, normal);
}

int lr_trace_rays_query(const LrScene* s, int64_t n, const float* origins, const float* directions, int32_t query, int32_t* prim, float* t,
                        float* normal) {
  if (!s) return fail(LR_ERR_INVALID, "bad argument");
  const OnDevice on(s->device);
  if (!s || !origins || !directions || !prim || !t || n < 0) return fail(LR_ERR_INVALID, "bad argument");
  if (query != LR_QUERY_STRICT && query != LR_QUERY_RENDER) return fail(LR_ERR_INVALID, "unknown query kind");
  if (n == 0) return LR_OK;
  if (int rc = ensure_device()) return rc;
  float *d_o = nullptr, *d_d = nullptr, *d_t = nullptr, *d_n = nullptr; int* d_p = nullptr;
  cudaError_t e = cudaMalloc((void**)&d_o, n * 3 * sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc((void**)&d_d, n * 3 * sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc((void**)&d_t, n * sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc((void**)&d_p, n * sizeof(int));
  if (e == cudaSuccess && normal) e = cudaMalloc((void**)&d_n, n * 3 * sizeof(float));
  if (e == cudaSuccess) e = cudaMemcpy(d_o, origins, n * 3 * sizeof(float), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(d_d, directions, n * 3 * sizeof(float), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = launch_rays(s->dev, n, d_o, d_d, d_p, d_t, d_n, query == LR_QUERY_RENDER, 0);
  if (e == cudaSuccess) e = cudaMemcpy(prim, d_p, n * sizeof(int), cudaMemcpyDeviceToHost);
  if (e == cudaSuccess) e = cudaMemcpy(t, d_t, n * sizeof(float), cudaMemcpyDeviceToHost);
  if (e == cudaSuccess && normal) e = cudaMemcpy(normal, d_n, n * 3 * sizeof(float), cudaMemcpyDeviceToHost);
  cudaFree(d_o); cudaFree(d_d); cudaFree(d_t); cudaFree(d_p); if (d_n) cudaFree(d_n);
  if (e != cudaSuccess) return fail(LR_ERR_CUDA, std::string("trace_rays: ") + cudaGetErrorString(e));
  return LR_OK;
}

// ---------------------------------------------------------------- progressive / resumable rendering (main.rs:81-91)
}  // extern "C"

struct LrFilm {
  const LrScene* scene = nullptr;
  LrRenderParams params{};               // spp_begin = first sample index of the film, spp_count unused
  int32_t spp_done = 0;
  int32_t crop_w = 0, crop_h = 0;        // resolved window
  float* d_sum = nullptr;
  float* d_sumsq = nullptr;
};

namespace {
constexpr char kFilmMagic[8] = {'L', 'R', 'F', 'I', 'L', 'M', '1', 0};
struct FilmHeader {                      // checkpoint file: this header, then crop_w*crop_h*3 floats (and again for the squares)
  char magic[8];
  int32_t film_w, film_h, crop_x, crop_y, crop_w, crop_h;
  int32_t integrator, depth, depth_limit, no_direct_emitter, splits, spp_begin, spp_done, has_sumsq;
  uint64_t seed;
};

// The checkpoint format, shared by LrFilm and LrMultiFilm: a film of either kind saves the same bytes for the same state
// and loads the other's checkpoints.
FilmHeader film_header(int film_w, int film_h, const LrRenderParams& p, int32_t crop_w, int32_t crop_h, int32_t spp_done, bool has_sumsq) {
  FilmHeader h;
  std::memset(&h, 0, sizeof(h));
  std::memcpy(h.magic, kFilmMagic, 8);
  h.film_w = film_w; h.film_h = film_h;
  h.crop_x = p.crop_w > 0 ? p.crop_x : 0; h.crop_y = p.crop_w > 0 ? p.crop_y : 0; h.crop_w = crop_w; h.crop_h = crop_h;
  h.integrator = p.integrator; h.depth = p.depth; h.depth_limit = p.depth_limit; h.no_direct_emitter = p.no_direct_emitter;
  h.splits = p.splits; h.spp_begin = p.spp_begin; h.spp_done = spp_done; h.has_sumsq = has_sumsq ? 1 : 0; h.seed = p.seed;
  return h;
}

// `data`: the raw sums, then the sums of squares if the header says so
int film_write(const char* path, const FilmHeader& h, const std::vector<float>& data) {
  // written next to the target and renamed: a crash mid-write never leaves a torn checkpoint under `path`
  const std::string tmp = std::string(path) + ".part";
  FILE* fp = std::fopen(tmp.c_str(), "wb");
  if (!fp) return fail(LR_ERR_IO, std::string("cannot write `") + tmp + "`");
  const bool ok = std::fwrite(&h, sizeof(h), 1, fp) == 1 && std::fwrite(data.data(), sizeof(float), data.size(), fp) == data.size();
  const bool closed = std::fclose(fp) == 0;
  if (!ok || !closed || std::rename(tmp.c_str(), path) != 0) { std::remove(tmp.c_str()); return fail(LR_ERR_IO, std::string("cannot write `") + path + "`"); }
  return LR_OK;
}

// reads a checkpoint made for a film_w x film_h film: its header, its data (as film_write) and the parameters to resume with
int film_read(const char* path, int film_w, int film_h, FilmHeader* hp, std::vector<float>* data, LrRenderParams* params) {
  FILE* fp = std::fopen(path, "rb");
  if (!fp) return fail(LR_ERR_IO, std::string("File `") + path + "` is not found.");
  FilmHeader& h = *hp;
  int rc = LR_OK;
  do {
    if (std::fread(&h, sizeof(h), 1, fp) != 1 || std::memcmp(h.magic, kFilmMagic, 8) != 0) { rc = fail(LR_ERR_PARSE, "not a film checkpoint"); break; }
    if (h.film_w != film_w || h.film_h != film_h) { rc = fail(LR_ERR_INVALID, "the checkpoint was made for another film resolution"); break; }
    if (h.crop_w <= 0 || h.crop_h <= 0 || h.crop_x < 0 || h.crop_y < 0 || h.crop_x + h.crop_w > film_w || h.crop_y + h.crop_h > film_h ||
        h.spp_done < 0 || h.spp_begin < 0) { rc = fail(LR_ERR_PARSE, "corrupt film checkpoint header"); break; }
    const size_t n = (size_t)h.crop_w * h.crop_h * 3;
    data->resize(n * (h.has_sumsq ? 2 : 1));
    if (std::fread(data->data(), sizeof(float), data->size(), fp) != data->size()) { rc = fail(LR_ERR_PARSE, "truncated film checkpoint"); break; }
  } while (0);
  std::fclose(fp);
  if (rc != LR_OK) return rc;
  LrRenderParams& p = *params;
  std::memset(&p, 0, sizeof(p));
  p.integrator = h.integrator; p.depth = h.depth; p.depth_limit = h.depth_limit; p.no_direct_emitter = h.no_direct_emitter;
  p.splits = h.splits; p.spp_begin = h.spp_begin; p.seed = h.seed;
  const bool whole = h.crop_x == 0 && h.crop_y == 0 && h.crop_w == film_w && h.crop_h == film_h;
  if (!whole) { p.crop_x = h.crop_x; p.crop_y = h.crop_y; p.crop_w = h.crop_w; p.crop_h = h.crop_h; }
  return LR_OK;
}

int film_alloc(const LrScene* s, const LrRenderParams* p, int want_sumsq, LrFilm** out) {
  if (!s) return fail(LR_ERR_INVALID, "null argument");
  const OnDevice on(s->device);
  if (!s || !p || !out) return fail(LR_ERR_INVALID, "null argument");
  *out = nullptr;
  LrRenderParams probe = *p;
  probe.spp_count = 1;
  DevParams dp;
  if (int rc = resolve_params(s, &probe, dp)) return rc;
  if (int rc = ensure_device()) return rc;
  LrFilm* f = new LrFilm();
  f->scene = s; f->params = *p; f->params.spp_count = 0;
  f->crop_w = dp.crop_w; f->crop_h = dp.crop_h;
  const size_t bytes = (size_t)dp.crop_w * dp.crop_h * 3 * sizeof(float);
  cudaError_t e = dev_alloc((void**)&f->d_sum, bytes);
  if (e == cudaSuccess) e = cudaMemset(f->d_sum, 0, bytes);
  if (e == cudaSuccess && want_sumsq) e = dev_alloc((void**)&f->d_sumsq, bytes);
  if (e == cudaSuccess && want_sumsq) e = cudaMemset(f->d_sumsq, 0, bytes);
  if (e != cudaSuccess) {
    const std::string msg = std::string("film: ") + cudaGetErrorString(e);
    lr_film_destroy(f);
    return fail(LR_ERR_CUDA, msg);
  }
  *out = f;
  return LR_OK;
}
}  // namespace

extern "C" {

int lr_film_create(const LrScene* s, const LrRenderParams* p, int32_t want_sumsq, LrFilm** out) { LR_GUARDED(film_alloc(s, p, want_sumsq, out)); }

void lr_film_destroy(LrFilm* f) {
  if (!f) return;
  const OnDevice on(f->scene->device);
  if (!f) return;
  cudaDeviceSynchronize();
  dev_free(f->d_sum);
  dev_free(f->d_sumsq);
  delete f;
}

int lr_film_info(const LrFilm* f, int32_t* spp_done, int32_t* crop_w, int32_t* crop_h, int32_t* has_sumsq) {
  if (!f) return fail(LR_ERR_INVALID, "null argument");
  if (spp_done) *spp_done = f->spp_done;
  if (crop_w) *crop_w = f->crop_w;
  if (crop_h) *crop_h = f->crop_h;
  if (has_sumsq) *has_sumsq = f->d_sumsq ? 1 : 0;
  return LR_OK;
}

int lr_film_render(LrFilm* f, int32_t spp_count, LrStats* stats) {
  if (!f) return fail(LR_ERR_INVALID, "null argument");
  if (spp_count <= 0) return fail(LR_ERR_INVALID, "spp_count must be positive");
  LrRenderParams q = f->params;
  q.spp_begin = f->params.spp_begin + f->spp_done;
  q.spp_count = spp_count;
  LrStats dummy;
  if (!stats) stats = &dummy;
  if (int rc = lr_stats_fetch(f->scene, nullptr, stats)) return rc;       // drop counters of earlier calls
  if (int rc = lr_render_accumulate_device(f->scene, &q, f->d_sum, f->d_sumsq, nullptr)) return rc;
  if (int rc = lr_stats_fetch(f->scene, nullptr, stats)) return rc;       // synchronises: the samples are in the film
  f->spp_done += spp_count;
  return LR_OK;
}

int lr_film_read(const LrFilm* f, float* out_rgb, float* out_sumsq) {
  if (!f) return fail(LR_ERR_INVALID, "null argument");
  const OnDevice on(f->scene->device);
  if (!f || !out_rgb) return fail(LR_ERR_INVALID, "null argument");
  if (out_sumsq && !f->d_sumsq) return fail(LR_ERR_INVALID, "the film was created without sums of squares");
  if (f->spp_done <= 0) return fail(LR_ERR_INVALID, "the film holds no samples yet");
  const size_t n = (size_t)f->crop_w * f->crop_h * 3;
  float* d_tmp = nullptr;
  LR_CUDA(dev_alloc((void**)&d_tmp, n * sizeof(float)));
  cudaError_t e = cudaMemcpyAsync(d_tmp, f->d_sum, n * sizeof(float), cudaMemcpyDeviceToDevice, 0);
  if (e == cudaSuccess) e = launch_scale(d_tmp, n, (float)f->spp_done, 0);            // main.rs:104
  if (e == cudaSuccess) e = cudaMemcpy(out_rgb, d_tmp, n * sizeof(float), cudaMemcpyDeviceToHost);
  if (e == cudaSuccess && out_sumsq) e = cudaMemcpy(out_sumsq, f->d_sumsq, n * sizeof(float), cudaMemcpyDeviceToHost);
  dev_free(d_tmp);
  if (e != cudaSuccess) return fail(LR_ERR_CUDA, std::string("film read: ") + cudaGetErrorString(e));
  return LR_OK;
}

static int film_save_body(const LrFilm* f, const char* path) {
  if (!f) return fail(LR_ERR_INVALID, "null argument");
  const OnDevice on(f->scene->device);
  if (!f || !path) return fail(LR_ERR_INVALID, "null argument");
  const size_t n = (size_t)f->crop_w * f->crop_h * 3;
  std::vector<float> host(n * (f->d_sumsq ? 2 : 1));
  LR_CUDA(cudaMemcpy(host.data(), f->d_sum, n * sizeof(float), cudaMemcpyDeviceToHost));
  if (f->d_sumsq) LR_CUDA(cudaMemcpy(host.data() + n, f->d_sumsq, n * sizeof(float), cudaMemcpyDeviceToHost));
  return film_write(path, film_header(f->scene->width, f->scene->height, f->params, f->crop_w, f->crop_h, f->spp_done, f->d_sumsq != nullptr), host);
}
int lr_film_save(const LrFilm* f, const char* path) { LR_GUARDED(film_save_body(f, path)); }

static int film_load_body(const LrScene* s, const char* path, LrFilm** out) {
  if (!s || !path || !out) return fail(LR_ERR_INVALID, "null argument");
  *out = nullptr;
  FilmHeader h;
  std::vector<float> host;
  LrRenderParams p;
  int rc = film_read(path, s->width, s->height, &h, &host, &p);
  if (rc != LR_OK) return rc;
  LrFilm* f = nullptr;
  if ((rc = film_alloc(s, &p, h.has_sumsq, &f)) != LR_OK) return rc;
  const size_t n = (size_t)h.crop_w * h.crop_h * 3;
  cudaError_t e = cudaMemcpy(f->d_sum, host.data(), n * sizeof(float), cudaMemcpyHostToDevice);
  if (e == cudaSuccess && h.has_sumsq) e = cudaMemcpy(f->d_sumsq, host.data() + n, n * sizeof(float), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) { lr_film_destroy(f); return fail(LR_ERR_CUDA, std::string("film load: ") + cudaGetErrorString(e)); }
  f->spp_done = h.spp_done;
  *out = f;
  return LR_OK;
}
int lr_film_load(const LrScene* s, const char* path, LrFilm** out) { LR_GUARDED(film_load_body(s, path, out)); }

// ---------------------------------------------------------------- progressive / resumable rendering on several GPUs
}  // extern "C"

// A film of an LrMultiScene, sharded by pixel: shard k of n_shards (device_scene.h: shard_of_tile) renders on device
// shard_device(k, n).  Every device keeps a crop-sized sum buffer but writes only the pixels of its own shards; the image
// is gathered on devices[0], each pixel from the device that owns it.
struct LrMultiFilm {
  LrMultiScene* ms = nullptr;
  LrRenderParams params{};               // as LrFilm's, with splits = 1
  int32_t spp_done = 0;
  int32_t crop_w = 0, crop_h = 0;
  int n_shards = 1;
  bool has_sumsq = false;
  float* d_sum[kMaxPeers] = {};          // on ms->devices[i]
  float* d_sumsq[kMaxPeers] = {};
};

namespace {

int use_device(const LrMultiScene* m, int i) {
  const cudaError_t e = cudaSetDevice(m->devices[i]);
  if (e != cudaSuccess) return fail(LR_ERR_CUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(e));
  g_device = m->devices[i];
  return LR_OK;
}

// the end of every multi-film call: after a failure nothing of the call stays in flight; the calling thread and the library
// are back on the multi scene's home device, as lr_multi_render leaves them
int multi_finish(const LrMultiScene* m, int rc) {
  const std::string err = g_error;
  if (rc != LR_OK) for (int i = 0; i < m->n; i++) { cudaSetDevice(m->devices[i]); cudaDeviceSynchronize(); }
  cudaSetDevice(m->home);
  g_device = m->home;
  g_error = err;
  return rc;
}

void mfilm_free(LrMultiFilm* f) {
  const LrMultiScene* m = f->ms;
  int prev = 0;
  cudaGetDevice(&prev);
  for (int i = 0; i < m->n; i++) {
    if (!f->d_sum[i] && !f->d_sumsq[i]) continue;
    cudaSetDevice(m->devices[i]);
    cudaDeviceSynchronize();
    dev_free(f->d_sum[i]);
    dev_free(f->d_sumsq[i]);
  }
  cudaSetDevice(prev);
  delete f;
}

int mfilm_alloc(LrMultiScene* m, const LrRenderParams* p, int want_sumsq, LrMultiFilm** out) {
  if (!m || !p || !out) return fail(LR_ERR_INVALID, "null argument");
  *out = nullptr;
  // the bit-for-bit contract (every pixel's samples added in order from the stored sum) holds for one thread per pixel only
  if (p->splits != 0 && p->splits != 1) return fail(LR_ERR_INVALID, "a multi-device film renders with splits = 1");
  LrRenderParams probe = *p;
  probe.spp_count = 1;
  const FilmShard whole{0, 1};
  DevParams dp;
  if (int rc = resolve_params(m->scenes[0], &probe, dp, &whole)) return rc;
  LrMultiFilm* f = new LrMultiFilm();
  f->ms = m; f->params = *p; f->params.spp_count = 0; f->params.splits = 1;
  f->crop_w = dp.crop_w; f->crop_h = dp.crop_h; f->has_sumsq = want_sumsq != 0;
  f->n_shards = m->n;
  // LR_FILM_SHARDS=S (development / tests): S shards over the devices, so that one GPU runs the interleaved kernels too
  if (const char* e_shards = std::getenv("LR_FILM_SHARDS")) f->n_shards = std::max(1, std::atoi(e_shards));
  const size_t bytes = (size_t)dp.crop_w * dp.crop_h * 3 * sizeof(float);
  int rc = LR_OK;
  for (int i = 0; i < m->n && rc == LR_OK; i++) {
    if ((rc = use_device(m, i)) != LR_OK) break;
    cudaError_t e = dev_alloc((void**)&f->d_sum[i], bytes);
    if (e == cudaSuccess) e = cudaMemsetAsync(f->d_sum[i], 0, bytes, 0);
    if (e == cudaSuccess && want_sumsq) e = dev_alloc((void**)&f->d_sumsq[i], bytes);
    if (e == cudaSuccess && want_sumsq) e = cudaMemsetAsync(f->d_sumsq[i], 0, bytes, 0);
    if (e == cudaSuccess) e = cudaStreamSynchronize(0);       // the render streams do not order against the legacy stream
    if (e != cudaSuccess) rc = fail(LR_ERR_CUDA, std::string("multi film: ") + cudaGetErrorString(e));
  }
  if ((rc = multi_finish(m, rc)) != LR_OK) {
    const std::string err = g_error;
    mfilm_free(f);
    g_error = err;
    return rc;
  }
  *out = f;
  return LR_OK;
}

int mfilm_render(LrMultiFilm* f, int32_t spp_count, LrStats* stats) {
  if (!f) return fail(LR_ERR_INVALID, "null argument");
  if (spp_count <= 0) return fail(LR_ERR_INVALID, "spp_count must be positive");
  LrMultiScene* m = f->ms;
  LrRenderParams q = f->params;
  q.spp_begin = f->params.spp_begin + f->spp_done;
  q.spp_count = spp_count;
  LrStats total;
  std::memset(&total, 0, sizeof(total));
  int rc = LR_OK;
  do {
    for (int i = 0; i < m->n && rc == LR_OK; i++) {          // drop the counters of earlier calls
      LrStats dropped;
      if ((rc = use_device(m, i)) == LR_OK) rc = lr_stats_fetch(m->scenes[i], m->streams[i], &dropped);
    }
    if (rc != LR_OK) break;
    // launch: asynchronous on every device's own stream, so the devices render concurrently; a device with several shards
    // renders them one after the other (disjoint pixels of the same buffer)
    for (int k = 0; k < f->n_shards && rc == LR_OK; k++) {
      const int i = shard_device(k, m->n);
      const FilmShard shard{k, f->n_shards};
      if ((rc = use_device(m, i)) == LR_OK) rc = accumulate(m->scenes[i], &q, f->d_sum[i], f->d_sumsq[i], m->streams[i], &shard);
    }
    if (rc != LR_OK) break;
    // wait for every device; statistics are totals, kernel_ms the slowest device's
    for (int i = 0; i < m->n && rc == LR_OK; i++) {
      LrStats st;
      if ((rc = use_device(m, i)) != LR_OK || (rc = lr_stats_fetch(m->scenes[i], m->streams[i], &st)) != LR_OK) break;
      add_device_stats(total, st);
    }
  } while (0);
  if ((rc = multi_finish(m, rc)) != LR_OK) return rc;
  f->spp_done += spp_count;
  if (stats) *stats = total;
  return LR_OK;
}

// The film's crop on devices[0] into dst (device memory there): each pixel from the buffer of the device that owns it
// (`bufs`: one per device), read over NVLink where devices[0] maps the peer and from a staged copy where it does not;
// divided by `divisor` if it is > 0.  Asynchronous on devices[0]'s stream; the caller has made devices[0] current.
int mfilm_gather(const LrMultiFilm* f, float* const* bufs, float* dst, float divisor) {
  LrMultiScene* m = f->ms;
  const size_t n = (size_t)f->crop_w * f->crop_h * 3;
  cudaStream_t st0 = m->streams[0];
  size_t need_staged = 0;
  for (int i = 1; i < m->n; i++) if (!m->mapped[i]) need_staged += n;
  cudaError_t e = cudaSuccess;
  if (need_staged > m->staged_floats) {
    e = cudaStreamSynchronize(st0);                           // an earlier gather may still read the old staging buffer
    if (e == cudaSuccess) {
      dev_free(m->staged);
      m->staged = nullptr; m->staged_floats = 0;
      e = dev_alloc((void**)&m->staged, need_staged * sizeof(float));
      if (e == cudaSuccess) m->staged_floats = need_staged;
    }
  }
  PeerBuffers src;
  src.count = m->n;
  float* stage_next = m->staged;
  for (int i = 0; i < m->n && e == cudaSuccess; i++) {
    src.p[i] = bufs[i];
    if (!m->mapped[i]) {
      e = cudaMemcpyPeerAsync(stage_next, m->devices[0], bufs[i], m->devices[i], n * sizeof(float), st0);
      src.p[i] = stage_next;
      stage_next += n;
    }
  }
  if (e == cudaSuccess) e = launch_gather_shards(dst, src, f->crop_w, f->crop_h, f->n_shards, divisor, st0);
  if (e != cudaSuccess) return fail(LR_ERR_CUDA, std::string("multi film gather: ") + cudaGetErrorString(e));
  return LR_OK;
}

// the gathered sums (sums of squares after them if asked for) or the mean, to host memory
int mfilm_download(const LrMultiFilm* f, float divisor, float* out, float* out_sumsq) {
  const LrMultiScene* m = f->ms;
  const size_t n = (size_t)f->crop_w * f->crop_h * 3;
  int rc = use_device(m, 0);
  float* d_tmp = nullptr;
  cudaError_t e = cudaSuccess;
  if (rc == LR_OK) {
    e = dev_alloc((void**)&d_tmp, n * sizeof(float));
    if (e != cudaSuccess) rc = fail(LR_ERR_CUDA, std::string("multi film: ") + cudaGetErrorString(e));
  }
  if (rc == LR_OK && (rc = mfilm_gather(f, f->d_sum, d_tmp, divisor)) == LR_OK) {
    e = cudaMemcpyAsync(out, d_tmp, n * sizeof(float), cudaMemcpyDeviceToHost, m->streams[0]);
    if (e == cudaSuccess && out_sumsq && (rc = mfilm_gather(f, f->d_sumsq, d_tmp, 0.0f)) == LR_OK)
      e = cudaMemcpyAsync(out_sumsq, d_tmp, n * sizeof(float), cudaMemcpyDeviceToHost, m->streams[0]);
    if (e == cudaSuccess) e = cudaStreamSynchronize(m->streams[0]);
    if (rc == LR_OK && e != cudaSuccess) rc = fail(LR_ERR_CUDA, std::string("multi film D2H: ") + cudaGetErrorString(e));
  }
  if (d_tmp) { if (rc != LR_OK) cudaStreamSynchronize(m->streams[0]); dev_free(d_tmp); }
  return multi_finish(m, rc);
}

int mfilm_read(const LrMultiFilm* f, float* out_rgb, float* out_sumsq) {
  if (!f || !out_rgb) return fail(LR_ERR_INVALID, "null argument");
  if (out_sumsq && !f->has_sumsq) return fail(LR_ERR_INVALID, "the film was created without sums of squares");
  if (f->spp_done <= 0) return fail(LR_ERR_INVALID, "the film holds no samples yet");
  return mfilm_download(f, (float)f->spp_done, out_rgb, out_sumsq);   // main.rs:104, as lr_film_read
}

int mfilm_save(const LrMultiFilm* f, const char* path) {
  if (!f || !path) return fail(LR_ERR_INVALID, "null argument");
  const size_t n = (size_t)f->crop_w * f->crop_h * 3;
  std::vector<float> host(n * (f->has_sumsq ? 2 : 1));
  if (int rc = mfilm_download(f, 0.0f, host.data(), f->has_sumsq ? host.data() + n : nullptr)) return rc;
  const LrScene* s0 = f->ms->scenes[0];
  return film_write(path, film_header(s0->width, s0->height, f->params, f->crop_w, f->crop_h, f->spp_done, f->has_sumsq), host);
}

int mfilm_load(LrMultiScene* m, const char* path, LrMultiFilm** out) {
  if (!m || !path || !out) return fail(LR_ERR_INVALID, "null argument");
  *out = nullptr;
  FilmHeader h;
  std::vector<float> host;
  LrRenderParams p;
  int rc = film_read(path, m->scenes[0]->width, m->scenes[0]->height, &h, &host, &p);
  if (rc != LR_OK) return rc;
  if (h.splits != 1) return fail(LR_ERR_INVALID, "the checkpoint was rendered with splits != 1; a multi-device film adds samples in order");
  LrMultiFilm* f = nullptr;
  if ((rc = mfilm_alloc(m, &p, h.has_sumsq, &f)) != LR_OK) return rc;
  // the sums go to devices[0], and from there to every other device
  const size_t bytes = (size_t)h.crop_w * h.crop_h * 3 * sizeof(float);
  cudaStream_t st0 = m->streams[0];
  rc = use_device(m, 0);
  cudaError_t e = cudaSuccess;
  if (rc == LR_OK) {
    e = cudaMemcpyAsync(f->d_sum[0], host.data(), bytes, cudaMemcpyHostToDevice, st0);
    if (e == cudaSuccess && h.has_sumsq) e = cudaMemcpyAsync(f->d_sumsq[0], host.data() + bytes / sizeof(float), bytes, cudaMemcpyHostToDevice, st0);
    for (int i = 1; i < m->n && e == cudaSuccess; i++) {
      e = cudaMemcpyPeerAsync(f->d_sum[i], m->devices[i], f->d_sum[0], m->devices[0], bytes, st0);
      if (e == cudaSuccess && h.has_sumsq) e = cudaMemcpyPeerAsync(f->d_sumsq[i], m->devices[i], f->d_sumsq[0], m->devices[0], bytes, st0);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(st0);
    if (e != cudaSuccess) rc = fail(LR_ERR_CUDA, std::string("multi film load: ") + cudaGetErrorString(e));
  }
  if ((rc = multi_finish(m, rc)) != LR_OK) {
    const std::string err = g_error;
    mfilm_free(f);
    g_error = err;
    return rc;
  }
  f->spp_done = h.spp_done;
  *out = f;
  return LR_OK;
}

}  // namespace

extern "C" {

int lr_multi_film_create(LrMultiScene* ms, const LrRenderParams* p, int32_t want_sumsq, LrMultiFilm** out) {
  LR_GUARDED(mfilm_alloc(ms, p, want_sumsq, out));
}
int lr_multi_film_render(LrMultiFilm* f, int32_t spp_count, LrStats* stats) { LR_GUARDED(mfilm_render(f, spp_count, stats)); }
int lr_multi_film_info(const LrMultiFilm* f, int32_t* spp_done, int32_t* crop_w, int32_t* crop_h, int32_t* has_sumsq) {
  if (!f) return fail(LR_ERR_INVALID, "null argument");
  if (spp_done) *spp_done = f->spp_done;
  if (crop_w) *crop_w = f->crop_w;
  if (crop_h) *crop_h = f->crop_h;
  if (has_sumsq) *has_sumsq = f->has_sumsq ? 1 : 0;
  return LR_OK;
}
int lr_multi_film_read(const LrMultiFilm* f, float* out_rgb, float* out_sumsq) { LR_GUARDED(mfilm_read(f, out_rgb, out_sumsq)); }
int lr_multi_film_save(const LrMultiFilm* f, const char* path) { LR_GUARDED(mfilm_save(f, path)); }
int lr_multi_film_load(LrMultiScene* ms, const char* path, LrMultiFilm** out) { LR_GUARDED(mfilm_load(ms, path, out)); }
void lr_multi_film_destroy(LrMultiFilm* f) {
  if (f) mfilm_free(f);
}

static int measure_read(uint64_t bytes, int iters, int warm, float* gbs) {
  if (!gbs || bytes < (1u << 20) || iters <= 0) return fail(LR_ERR_INVALID, "bad argument");
  if (int rc = ensure_device()) return rc;
  const size_t n4 = bytes / 16;
  float4* buf = nullptr; float* sink = nullptr;
  LR_CUDA(cudaMalloc((void**)&buf, n4 * 16));
  cudaError_t e = cudaMalloc((void**)&sink, 4);
  if (e == cudaSuccess) e = cudaMemset(buf, 0, n4 * 16);
  cudaEvent_t a = nullptr, b = nullptr;
  if (e == cudaSuccess) e = cudaEventCreate(&a);
  if (e == cudaSuccess) e = cudaEventCreate(&b);
  const int blocks = std::max(g_sm_count, 1) * 8;
  float best = 0.0f;
  for (int rep = 0; rep < 5 && e == cudaSuccess; rep++) {
    e = launch_read_bw(buf, n4, warm, blocks, sink, 0);                 // warm the cache level under test
    if (e == cudaSuccess) e = cudaEventRecord(a, 0);
    if (e == cudaSuccess) e = launch_read_bw(buf, n4, iters, blocks, sink, 0);
    if (e == cudaSuccess) e = cudaEventRecord(b, 0);
    if (e == cudaSuccess) e = cudaEventSynchronize(b);
    float ms = 0.0f;
    if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, a, b);
    if (e == cudaSuccess && ms > 0.0f) best = std::max(best, (float)((double)n4 * 16.0 * iters / (ms * 1e-3) / 1e9));
  }
  if (a) cudaEventDestroy(a);
  if (b) cudaEventDestroy(b);
  cudaFree(buf);
  if (sink) cudaFree(sink);
  if (e != cudaSuccess) return fail(LR_ERR_CUDA, std::string("measure_read: ") + cudaGetErrorString(e));
  *gbs = best;
  return LR_OK;
}

int lr_measure_l2_read_gbs(uint64_t working_set_bytes, int iters, float* gbs) { return measure_read(working_set_bytes, iters, 2, gbs); }
int lr_measure_hbm_read_gbs(uint64_t bytes, int iters, float* gbs) { return measure_read(bytes, iters, 1, gbs); }

}  // extern "C"
