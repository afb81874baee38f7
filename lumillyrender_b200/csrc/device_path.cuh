// device_path.cuh — device-side building blocks of the path-tracing hot path (sm_100a).
//
// NUMERICS CONTRACT.  This translation unit is compiled with -fmad=false, IEEE division and
// square root (-prec-div=true -prec-sqrt=true, no fast-math), so every expression below rounds
// exactly like the reference's fp32 code compiled by rustc without FMA (README.md:12,
// SURVEY.md §7 hard part 1).  The BVH *node* slab test uses the cancellation-safe
// (box - origin) * inv form on boxes the host padded outward; it is a conservative cull and
// never decides a hit.  A hit is decided only by (a) the reference's primitive test (triangle.rs:69-100,
// sphere.rs:42-63) and (b) the reference's slab test on the primitive's own AABB
// (aabb.rs:75-92 as applied by Leaf::may_intersect, bvh.rs:21-25), so the nearest hit equals
// the reference's regardless of BVH topology.
#pragma once
#include "device_scene.h"

namespace lr {

#define LR_DEV __device__ __forceinline__
// Code that most scenes never run (IBL lookup, Phong / Blinn-Phong / refraction, lens cameras, library fmodf) is kept out
// of line when LR_OUTLINE_COLD is set (build.py sets it for the render kernel): the kernel is instruction-fetch bound and
// every inlined cold branch dilutes the hot code (profiles/r01_c_ab_s23.txt).  Arguments go by value so that no hot
// variable has its address taken.
#ifdef LR_OUTLINE_COLD
#define LR_COLD static __device__ __noinline__
#else
#define LR_COLD __device__ __forceinline__
#endif

constexpr float kPI = 3.14159265358979323846264338327950288f;   // constant.rs:1
constexpr float kEPS = 1e-3f;                                   // constant.rs:2
constexpr float kINF = 1e5f;                                    // constant.rs:3

// ------------------------------------------------------------------ vector math (math/vector3.rs)
struct F3 { float x, y, z; };
LR_DEV F3 f3(float x, float y, float z) { F3 r; r.x = x; r.y = y; r.z = z; return r; }
LR_DEV F3 f3(const float* p) { return f3(p[0], p[1], p[2]); }
LR_DEV F3 f3(float4 v) { return f3(v.x, v.y, v.z); }
LR_DEV F3 operator-(F3 a) { return f3(-a.x, -a.y, -a.z); }
LR_DEV F3 operator+(F3 a, F3 b) { return f3(a.x + b.x, a.y + b.y, a.z + b.z); }
LR_DEV F3 operator-(F3 a, F3 b) { return f3(a.x - b.x, a.y - b.y, a.z - b.z); }
LR_DEV F3 operator*(F3 a, float s) { return f3(a.x * s, a.y * s, a.z * s); }
LR_DEV F3 operator*(float s, F3 a) { return f3(s * a.x, s * a.y, s * a.z); }
LR_DEV F3 operator*(F3 a, F3 b) { return f3(a.x * b.x, a.y * b.y, a.z * b.z); }
// ------------------------------------------------------------------ exact quotients that avoid the general division
// Under -prec-div=true every a / b is MUFU.RCP, five FFMA and an FCHK whose check sends the quotient to an out-of-line slow
// path (__cuda_sm3x_div_rn_noftz_f32_slowpath) when an operand is outside the range the fast sequence handles.  A zero
// dividend is outside that range (tools/div_probe.py on a B200: 242 cycles against 48 for a normal quotient,
// profiles/r03_a_div_probe.txt), and the hot path divides zeros on every bounce: the ONB's cross(a, n) has one component
// that is exactly +-0, two on an axis-aligned wall.  The helpers below give the IEEE
// quotient bit for bit (tests/test_exact_quotients.py checks them exhaustively) without that slow path.
//
// div_zero_dividend: 0 / s for a nonzero, non-NaN s is by IEEE definition a zero whose sign is the XOR of the operands'
// signs; the divide is handed a harmless dividend (s / s) in that case and its result is discarded.  Every other
// combination (0 / 0, 0 / NaN, any nonzero dividend) is the real division.
LR_DEV float div_zero_dividend(float a, float s) {
  const bool z = a == 0.0f && fabsf(s) > 0.0f;
  const float q = (z ? s : a) / s;
  return z ? __uint_as_float((__float_as_uint(a) ^ __float_as_uint(s)) & 0x80000000u) : q;
}
// a / kPI correctly rounded in three operations (Markstein: y = RN(1 / b) and q0 = RN(a * y) within one ulp of a / b make
// the residual r = a - b * q0 exact and RN(q0 + r * y) the correctly rounded quotient), for |a| >= 2^-95, where no step
// underflows (exhaustively: the sequence is exact for every dividend with a biased exponent of 23 or more, inf / NaN
// excepted).  A zero dividend gives a zero of its own sign; NaN, inf and tiny dividends take the real division, out of
// line (the render never reaches it).
constexpr float kPI_RCP = 0x1.45f306p-2f;                          // RN(1 / kPI)
LR_COLD float div_cold(float a, float b) { return a / b; }
LR_DEV float div_pi(float a) {
  const unsigned e = (__float_as_uint(a) >> 23) & 0xffu;
  if (e - 32u <= 254u - 32u) {
    const float q0 = __fmul_rn(a, kPI_RCP);
    const float r = __fmaf_rn(-kPI, q0, a);
    return __fmaf_rn(r, kPI_RCP, q0);
  }
  return a == 0.0f ? a : div_cold(a, kPI);
}

// IEEE quotient of a vector by a scalar, each component through div_zero_dividend: zero components are common (the ONB's
// cross product, axis-aligned normals and directions, black colour channels), and the guard is cheaper than the slow path
// they would take (A/B, profiles/r03_a_ab.txt: sample.toml 36.4 -> 31.8 ms, welcome-2018 43.2 -> 40.9 ms; with the guard
// in orthonormal_basis only, 32.6 / 44.4 ms).  In the one-path-per-lane kernel for pt-direct over a BVH the three
// divisions live in ONE out-of-line function (LR_DIV_OUT_OF_LINE, set by build.py for that translation unit): ~20 inlined
// copies of 3 x 14 instructions are a fifth of the kernel's code, and the kernel is instruction-fetch bound (A/B,
// profiles/r01_c_ab_s22.txt: +4.6 % on sample.toml; the flat-only kernels are 3 % faster with the divisions inlined).
LR_DEV F3 div3_inline(F3 a, float s) { return f3(div_zero_dividend(a.x, s), div_zero_dividend(a.y, s), div_zero_dividend(a.z, s)); }
#ifdef LR_DIV_OUT_OF_LINE
static __device__ __noinline__ F3 div3_call(F3 a, float s) { return div3_inline(a, s); }
LR_DEV F3 operator/(F3 a, float s) { return div3_call(a, s); }
#else
LR_DEV F3 operator/(F3 a, float s) { return div3_inline(a, s); }
#endif
LR_DEV float dot(F3 a, F3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
LR_DEV F3 cross(F3 a, F3 b) { return f3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x); }
LR_DEV float sqr_norm(F3 a) { return dot(a, a); }
LR_DEV float norm(F3 a) { return sqrtf(sqr_norm(a)); }
LR_DEV F3 normalize(F3 a) { return a / norm(a); }            // three true divisions (traits.rs:38-42)
LR_DEV float comp(F3 a, int i) { return i == 0 ? a.x : (i == 1 ? a.y : a.z); }

// ------------------------------------------------------------------ sin/cos
// The reference calls f32::sin / f32::cos, i.e. whatever the platform libm provides (not bit-defined).
// The hot path needs them only for angles 2*pi*xi (BSDF / emitter / aperture sampling) and the
// omnidirectional camera.  One fp32 algorithm is specified here and restated verbatim in the oracle
// (oracle.cpp: spec_sincos) so that sampled directions — and therefore every later hit — replay bit
// for bit on CPU and GPU: Cody-Waite reduction by pi/2 in three parts, then the Cephes sinf/cosf
// minimax polynomials on [-pi/4, pi/4] (<= 2 ulp), all in unfused fp32 operations.
LR_DEV void spec_sincos(float x, float* sn, float* cs) {
  const float kf = rintf(x * 0.636619772367581343f);           // round-to-nearest-even of x * 2/pi
  const int k = (int)kf;
  float r = x - kf * 1.5703125f;
  r = r - kf * 4.837512969970703125e-4f;
  r = r - kf * 7.54978995489188216e-8f;
  const float z = r * r;
  const float s = ((-1.9515295891e-4f * z + 8.3321608736e-3f) * z - 1.6666654611e-1f) * z * r + r;
  const float c = ((2.443315711809948e-5f * z - 1.388731625493765e-3f) * z + 4.166664568298827e-2f) * z * z - 0.5f * z + 1.0f;
  // quadrant k & 3: (s, c), (c, -s), (-s, -c), (-c, s) — as selects and exact negations, not a four-way branch (the
  // lanes of a warp are spread over all four quadrants: ncu showed this function at 12 of 32 lanes)
  const bool swap = (k & 1) != 0;
  const float a = swap ? c : s, b = swap ? s : c;
  *sn = (k & 2) ? -a : a;
  *cs = ((k + 1) & 2) ? -b : b;
}

// ------------------------------------------------------------------ RNG (replaces rand::random, SURVEY §8 a21)
// Counter-based: the stream of a sample is a pure function of (seed, pixel, sample index), so any
// GPU can render any sample range and reproduce it bit for bit.  PCG32 (XSH-RR 64/32) stepped from
// a splitmix64-hashed start; floats are (u32 >> 8) * 2^-24 in [0,1) like rand 0.3's f32.
LR_DEV unsigned long long splitmix64(unsigned long long z) {
  z += 0x9E3779B97F4A7C15ULL;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
  return z ^ (z >> 31);
}
struct Pcg {
  unsigned long long state;
  LR_DEV unsigned int next_u32() {
    const unsigned long long old = state;
    state = old * 6364136223846793005ULL + 1442695040888963407ULL;
    const unsigned int xorshifted = (unsigned int)(((old >> 18u) ^ old) >> 27u);
    const unsigned int rot = (unsigned int)(old >> 59u);
    return __funnelshift_r(xorshifted, xorshifted, rot);
  }
  LR_DEV float next() { return (float)(next_u32() >> 8) * (1.0f / 16777216.0f); }
  LR_DEV void seed(unsigned long long seed, unsigned int pixel, unsigned int sample) {
    state = splitmix64(splitmix64(seed + 0x632BE59BD9B4E019ULL * (unsigned long long)pixel) ^
                       ((unsigned long long)sample * 0xD1B54A32D192ED03ULL));
    next_u32();
  }
};

// ------------------------------------------------------------------ reference slab test (aabb.rs:75-92)
// inv = 1.0f / direction (the same IEEE quotient the reference recomputes at every node)
LR_DEV bool ref_slab_pass(F3 lo, F3 hi, F3 o, F3 inv) {
  float mn = -kINF, mx = kINF;
#pragma unroll
  for (int i = 0; i < 3; i++) {
    const float t1 = (comp(lo, i) - comp(o, i)) * comp(inv, i);
    const float t2 = (comp(hi, i) - comp(o, i)) * comp(inv, i);
    float t_min, t_max;
    if (t1 > t2) { t_min = t2; t_max = t1; } else { t_min = t1; t_max = t2; }
    if (mn < t_min) mn = t_min;
    if (mx > t_max) mx = t_max;
    if (mn > mx) return false;
  }
  return true;
}

// ------------------------------------------------------------------ primitive tests
// triangle.rs:69-100.  Returns t or a negative value for a miss.  The edges e1 = p1 - p0, e2 = p2 - p0 (triangle.rs:71-72)
// are single fp32 subtractions, so they are computed once at upload (api.cpp) instead of once per test: same bits.
LR_DEV float triangle_mt(F3 p0, F3 e1, F3 e2, F3 o, F3 d) {
  const F3 pv = cross(d, e2);
  const float det = dot(e1, pv);
  if (fabsf(det) < kEPS) return -1.0f;
  const float invdet = 1.0f / det;
  const F3 tv = o - p0;
  const float u = dot(tv, pv) * invdet;
  if (u < 0.0f || u > 1.0f) return -1.0f;
  const F3 qv = cross(tv, e1);
  const float v = dot(d, qv) * invdet;
  if (v < 0.0f || u + v > 1.0f) return -1.0f;
  const float t = dot(e2, qv) * invdet;
  if (!(t >= kEPS)) return -1.0f;      // `t < EPS` rejects; a NaN t (reference: panic) is a miss
  return t;
}
// sphere.rs:42-56.  Returns t or a negative value for a miss.
LR_DEV float sphere_hit(F3 c, float r, F3 o, F3 d) {
  const F3 co = o - c;
  const float cod = dot(co, d);
  const float det = cod * cod - sqr_norm(co) + r * r;
  if (!(det > 0.0f)) return -1.0f;
  const float sq = sqrtf(det);
  const float t1 = -cod - sq;
  const float t2 = -cod + sq;
  if (t1 < kEPS && t2 < kEPS) return -1.0f;
  const float t = t1 > kEPS ? t1 : t2;
  if (!(t == t)) return -1.0f;
  return t;
}

// The same test without the early exits (select form): mn only rises and mx only falls from axis to axis (a NaN bound fails
// its comparison and changes nothing, as in the reference), so `mn > mx` after some axis implies `mn > mx` at the end.
LR_DEV bool ref_slab_pass_select(F3 lo, F3 hi, F3 o, F3 inv) {
  float mn = -kINF, mx = kINF;
#pragma unroll
  for (int i = 0; i < 3; i++) {
    const float t1 = (comp(lo, i) - comp(o, i)) * comp(inv, i);
    const float t2 = (comp(hi, i) - comp(o, i)) * comp(inv, i);
    const bool sw = t1 > t2;
    const float t_min = sw ? t2 : t1, t_max = sw ? t1 : t2;
    mn = mn < t_min ? t_min : mn;
    mx = mx > t_max ? t_max : mx;
  }
  return !(mn > mx);
}

// ------------------------------------------------------------------ the tie rule
// Two primitives can answer with bit-identical distances (a ray through a shared vertex or edge of a mesh).  The reference
// keeps the first such candidate in the depth-first order of ITS tree (min_by, bvh.rs:136-140) — an order only its own SAH
// build defines.  The device's trees differ from it and from each other (host SAH, device radix tree, flat list), so the
// device rule is: among equal distances the LOWEST PRIMITIVE ID wins.  The nearest hit is then a function of the scene
// alone — argmin over the valid candidates of (t, prim_id) — whatever the tree, the visiting order or the scheduling.
// `best` is a candidate code: >= 0 triangle index, <= -2 sphere index = -2 - id (never -1 here: t == best_t implies a hit).
static __device__ __noinline__ bool tie_goes_to(const float4* __restrict__ tris, const int2* __restrict__ sphere_meta, int cand_prim, int best) {
  const int best_prim = best >= 0 ? __float_as_int(__ldg(tris + 3 * (size_t)best).w) : __ldg(sphere_meta + (-2 - best)).y;
  return cand_prim < best_prim;
}
#define LR_NEARER(sc, t, cand_prim, best_t, best) ((t) < (best_t) || ((t) == (best_t) && tie_goes_to((sc).tris, (sc).sphere_meta, (cand_prim), (best))))

struct TraceCounters { unsigned int nodes, tris, spheres, flat_tris, flat_boxes; };

LR_DEV float4 ldg4(const float4* p) { return __ldg(p); }

// the reference's gate (aabb.rs:75-92 on the triangle's own box, as Leaf::may_intersect applies it, bvh.rs:21-25)
// (the box is the min / max of the vertices, triangle.rs:102-119: exact operations, stored at upload in tri_box)
LR_DEV bool tri_gate(const DevScene& sc, F3 o, F3 inv, int id) {
  const float4* bp = sc.tri_box + 2 * (size_t)id;
  return ref_slab_pass(f3(ldg4(bp + 0)), f3(ldg4(bp + 1)), o, inv);
}
// Candidates every ray tests in a fixed order, with the reference's exact arithmetic and its leaf-AABB gate:
// the spheres (no culling at all: the r = 1e5 ground sphere of scenes/primitive.toml has a t error far larger
// than any box slack), then the flat list of large triangles tris[n_bvh_tris, n_tris) (bvh_build.cpp).
// id: -1 miss, >= 0 triangle index, <= -2 sphere index = -2 - id.
//
// Flat triangles go through the reference's own two steps in the reference's order: Leaf::may_intersect — the line-slab
// test on the triangle's own box (bvh.rs:21-25, aabb.rs:75-92) — selects the candidates, then the primitive test runs on
// those alone (nearest wins; among equal distances the lowest primitive id: the tie rule above).  The gate is what makes a
// candidate valid, so testing it first is exact by construction; it is also cheap and selective: the line of a ray inside
// a room crosses the (flat) boxes of two walls, so a lane runs Moller-Trumbore on ~4-6 of the ~12-16 flat triangles.
//   * lanes hold DIFFERENT candidates in the second loop (a bit mask per lane, lowest bit first): the loop is as long as the
//     lane with the most candidates needs, not as long as the list;
//   * consecutive flat triangles with the same box (the two halves of a wall quad) share one gate test: tri_box[2i].w is 1
//     where triangle i's box equals its predecessor's (set at upload, api.cpp).
// Where the flat list is read from: boxes (2 x float4 per flat triangle, tri_box layout) and triangles (3 x float4, tris
// layout), indexed by the position k in the flat list.  The probes read the scene arrays in global memory; the render
// kernels stage both tables into shared memory once per CTA with one TMA bulk copy each (stage_flat_list below).
struct FlatList { const float4* box; const float4* tri; };
LR_DEV FlatList flat_list_global(const DevScene& sc) {
  FlatList f;
  f.box = sc.tri_box + 2 * (size_t)sc.n_bvh_tris;
  f.tri = sc.tris + 3 * (size_t)sc.n_bvh_tris;
  return f;
}
constexpr int kFlatListMax = 32;                                   // validate_desc (bvh_build.cpp) refuses longer lists
constexpr int kFlatListFloat4 = kFlatListMax * 5;                  // 2 box + 3 triangle float4 per entry: 2560 B

// Stages the flat list (the handful of wall / floor / light triangles EVERY ray gates and tests, path_vertex.inc) into the
// CTA's shared memory with the bulk-copy engine: one thread arms an mbarrier with the byte count and issues two
// cp.async.bulk copies (global -> shared, completion counted on the mbarrier: SASS UBLKCP + SYNCS), every thread then
// waits on the barrier's phase.  Called once at kernel start by all threads of the CTA; `tab` holds kFlatListFloat4 float4.
LR_DEV FlatList stage_flat_list(const DevScene& sc, float4* tab, unsigned long long* bar) {
  const int nf = sc.n_tris - sc.n_bvh_tris;
  FlatList f;
  f.box = tab;
  f.tri = tab + 2 * nf;
  if (nf <= 0) return f;
  const unsigned bar_s = (unsigned)__cvta_generic_to_shared(bar);
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_s));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned box_bytes = (unsigned)nf * 32u, tri_bytes = (unsigned)nf * 48u;
    const unsigned dst_box = (unsigned)__cvta_generic_to_shared(tab), dst_tri = (unsigned)__cvta_generic_to_shared(tab + 2 * nf);
    const float4* src_box = sc.tri_box + 2 * (size_t)sc.n_bvh_tris;
    const float4* src_tri = sc.tris + 3 * (size_t)sc.n_bvh_tris;
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_s), "r"(box_bytes + tri_bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst_box), "l"(src_box), "r"(box_bytes), "r"(bar_s) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst_tri), "l"(src_tri), "r"(tri_bytes), "r"(bar_s) : "memory");
  }
  unsigned done = 0;
  do {
    asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                 : "=r"(done) : "r"(bar_s), "r"(0u) : "memory");
  } while (!done);
  return f;
}

template <bool COUNT>
LR_DEV void flat_hits(const DevScene& sc, const FlatList fl, F3 o, F3 d, F3 inv, float& best_t, int& best, TraceCounters& tc) {
  for (int i = 0; i < sc.n_spheres; i++) {
    const float4 s = ldg4(sc.spheres + i);
    if (COUNT) tc.spheres++;
    const float t = sphere_hit(f3(s), s.w, o, d);
    if (t >= 0.0f && LR_NEARER(sc, t, __ldg(sc.sphere_meta + i).y, best_t, best)) {
      const F3 c = f3(s);
      const F3 r = f3(s.w, s.w, s.w);
      if (ref_slab_pass(c - r, c + r, o, inv)) { best_t = t; best = -2 - i; }
    }
  }
  const int n_flat = sc.n_tris - sc.n_bvh_tris;                    // <= 24 (bvh_build.cpp: kFlatMax)
  unsigned cand = 0u;
  bool pass = false;
#pragma unroll 1
  for (int k = 0; k < n_flat; k++) {
    const float4 lo = fl.box[2 * k], hi = fl.box[2 * k + 1];
    if (lo.w == 0.0f) {                                            // warp-uniform: a new box
      pass = ref_slab_pass_select(f3(lo), f3(hi), o, inv);
      if (COUNT) tc.flat_boxes++;
    }
    if (pass) cand |= 1u << k;
  }
#pragma unroll 1
  while (cand != 0u) {
    const int k = __ffs(cand) - 1;
    cand &= cand - 1u;
    const float4* tp = fl.tri + 3 * k;
    const float4 v0 = tp[0], v1 = tp[1], v2 = tp[2];
    if (COUNT) { tc.tris++; tc.flat_tris++; }
    const float t = triangle_mt(f3(v0), f3(v1), f3(v2), o, d);
    if (t >= 0.0f && LR_NEARER(sc, t, __float_as_int(v0.w), best_t, best)) { best_t = t; best = sc.n_bvh_tris + k; }
  }
}

// conservative: can the ray reach the tree's bounds within [0, cull_t]?  (same padded-box form as the node test)
LR_DEV bool bvh_bounds_hit(const DevScene& sc, F3 o, F3 inv, float cull_t) {
  const float ax = (sc.bvh_lo[0] - o.x) * inv.x, bx = (sc.bvh_hi[0] - o.x) * inv.x;
  const float ay = (sc.bvh_lo[1] - o.y) * inv.y, by = (sc.bvh_hi[1] - o.y) * inv.y;
  const float az = (sc.bvh_lo[2] - o.z) * inv.z, bz = (sc.bvh_hi[2] - o.z) * inv.z;
  const float en = fmaxf(fmaxf(fminf(ax, bx), fminf(ay, by)), fmaxf(fminf(az, bz), 0.0f));
  const float ex = fminf(fminf(fmaxf(ax, bx), fmaxf(ay, by)), fminf(fmaxf(az, bz), cull_t));
  return en <= ex;
}

// BVH part of the STRICT nearest-hit query (probes, and the re-trace of the rare ray whose optimistic hit fails the gate):
// "while-while" traversal (every lane first descends inner nodes until it holds a leaf or is done, the warp
// reconverges, then the lanes that hold leaves test triangles together), near child first, per-thread stack, nodes
// culled against [0, cull_t] on host-padded boxes.  best_t / best come in holding the nearest flat candidate (or
// 3e38 / -1) and are replaced only by something strictly nearer that also passes the reference's gate on the
// triangle's own AABB (bvh.rs:21-25) — the reference's semantics, candidate by candidate.  The render kernels use the
// optimistic form below (trav_step: accept on the primitive test alone, gate the final nearest hit once).
template <bool COUNT>
LR_DEV void bvh_traverse(const DevScene& sc, F3 o, F3 d, F3 inv, float& best_t, int& best, TraceCounters& tc) {
  // conservative cull distance: a primitive's computed t may precede its box's computed entry
  float cull_t = best_t < 3.0e38f ? best_t * 1.0001f + 1e-4f : 3.0e38f;
  constexpr int kDone = (int)0x80000000;       // not a valid leaf code (first triangle would be 2^28 - 1)
  int stack[kStackDepth];
  int sp = 0;
  stack[sp++] = kDone;
  int cur = 0;
  while (cur != kDone) {
    while (cur >= 0) {
      const float4* np = sc.nodes + 4 * (size_t)cur;
      const float4 n0 = ldg4(np + 0), n1 = ldg4(np + 1), n2 = ldg4(np + 2), n3 = ldg4(np + 3);
      if (COUNT) tc.nodes++;
      // child 0: lo = (n0.x,n0.y,n0.z) hi = (n0.w,n1.x,n1.y); child 1: lo = (n1.z,n1.w,n2.x) hi = (n2.y,n2.z,n2.w)
      const float ax0 = (n0.x - o.x) * inv.x, bx0 = (n0.w - o.x) * inv.x;
      const float ay0 = (n0.y - o.y) * inv.y, by0 = (n1.x - o.y) * inv.y;
      const float az0 = (n0.z - o.z) * inv.z, bz0 = (n1.y - o.z) * inv.z;
      const float ax1 = (n1.z - o.x) * inv.x, bx1 = (n2.y - o.x) * inv.x;
      const float ay1 = (n1.w - o.y) * inv.y, by1 = (n2.z - o.y) * inv.y;
      const float az1 = (n2.x - o.z) * inv.z, bz1 = (n2.w - o.z) * inv.z;
      const float en0 = fmaxf(fmaxf(fminf(ax0, bx0), fminf(ay0, by0)), fmaxf(fminf(az0, bz0), 0.0f));
      const float ex0 = fminf(fminf(fmaxf(ax0, bx0), fmaxf(ay0, by0)), fminf(fmaxf(az0, bz0), cull_t));
      const float en1 = fmaxf(fmaxf(fminf(ax1, bx1), fminf(ay1, by1)), fmaxf(fminf(az1, bz1), 0.0f));
      const float ex1 = fminf(fminf(fmaxf(ax1, bx1), fmaxf(ay1, by1)), fminf(fmaxf(az1, bz1), cull_t));
      const bool h0 = en0 <= ex0, h1 = en1 <= ex1;
      const int c0 = __float_as_int(n3.x), c1 = __float_as_int(n3.y);
      if (h0 && h1) {
        const bool first0 = en0 <= en1;
        stack[sp++] = first0 ? c1 : c0;
        cur = first0 ? c0 : c1;
      } else if (h0) {
        cur = c0;
      } else if (h1) {
        cur = c1;
      } else {
        cur = stack[--sp];
      }
    }
    if (cur != kDone) {
      const int code = ~cur;
      const int first = code >> 3;
      const int count = (code & 7) + 1;
      for (int k = 0; k < count; k++) {
        const float4* tp = sc.tris + 3 * (size_t)(first + k);
        const float4 v0 = ldg4(tp + 0), v1 = ldg4(tp + 1), v2 = ldg4(tp + 2);
        if (COUNT) tc.tris++;
        const float t = triangle_mt(f3(v0), f3(v1), f3(v2), o, d);
        if (t >= 0.0f && LR_NEARER(sc, t, __float_as_int(v0.w), best_t, best)) {
          // the leaf's own AABB gate (triangle.rs:102-119 box, aabb.rs:75-92 test)
          if (tri_gate(sc, o, inv, first + k)) {
            best_t = t;
            best = first + k;
            cull_t = best_t * 1.0001f + 1e-4f;
          }
        }
      }
      cur = stack[--sp];
    }
  }
}

// The optimistic form of the same query (accept on the primitive test, the caller gates the final nearest hit once with
// bvh_hit_is_gated and falls back to the strict query if it fails: if the nearest candidate passes, it IS the gated nearest
// hit — the minimum over a superset that lies in the subset), organised as ONE loop whose every iteration advances a lane by at most
// one inner node AND at most one triangle test: a leaf the descent reaches is moved to a one-entry leaf slot and the
// descent goes on with the next stack entry while the slot's (<= 8) triangles are tested one per iteration.  In the
// while-while form the lanes of a warp wait at the leaf step for the lane with the longest run of inner nodes (ncu:
// 7 of 32 lanes active in the node loop with 28 rays in flight); here a lane idles only when it has neither a node nor
// a triangle.  Nodes are culled against a cull_t that may lag one triangle test behind, which only makes the cull more
// conservative: a triangle reached that way lies beyond the current nearest hit and fails `t < best_t`, so the nearest
// hit (and the first-minimum tie rule, the triangle order being unchanged) is the same.
struct TravState {
  F3 o, d, inv;
  float best_t, cull_t;
  int best, cur, sp, leaf_first, leaf_left;
};
constexpr int kTravDone = (int)0x80000000;       // not a valid leaf code (first triangle would be 2^28 - 1)
LR_DEV void trav_begin(TravState& s, int* stack, F3 o, F3 d, F3 inv, float best_t, int best) {
  s.o = o; s.d = d; s.inv = inv;
  s.best_t = best_t; s.best = best;
  s.cull_t = best_t < 3.0e38f ? best_t * 1.0001f + 1e-4f : 3.0e38f;
  s.sp = 0;
  stack[s.sp++] = kTravDone;
  s.cur = 0;
  s.leaf_first = 0; s.leaf_left = 0;
}
LR_DEV bool trav_done(const TravState& s) { return s.cur == kTravDone && s.leaf_left == 0; }
template <bool COUNT>
LR_DEV void trav_step(const DevScene& sc, TravState& s, int* stack, TraceCounters& tc) {
  if (s.cur >= 0) {
    const float4* np = sc.nodes + 4 * (size_t)s.cur;
    const float4 n0 = ldg4(np + 0), n1 = ldg4(np + 1), n2 = ldg4(np + 2), n3 = ldg4(np + 3);
    if (COUNT) tc.nodes++;
    const F3 o = s.o, inv = s.inv;
    const float cull_t = s.cull_t;
    const float ax0 = (n0.x - o.x) * inv.x, bx0 = (n0.w - o.x) * inv.x;
    const float ay0 = (n0.y - o.y) * inv.y, by0 = (n1.x - o.y) * inv.y;
    const float az0 = (n0.z - o.z) * inv.z, bz0 = (n1.y - o.z) * inv.z;
    const float ax1 = (n1.z - o.x) * inv.x, bx1 = (n2.y - o.x) * inv.x;
    const float ay1 = (n1.w - o.y) * inv.y, by1 = (n2.z - o.y) * inv.y;
    const float az1 = (n2.x - o.z) * inv.z, bz1 = (n2.w - o.z) * inv.z;
    const float en0 = fmaxf(fmaxf(fminf(ax0, bx0), fminf(ay0, by0)), fmaxf(fminf(az0, bz0), 0.0f));
    const float ex0 = fminf(fminf(fmaxf(ax0, bx0), fmaxf(ay0, by0)), fminf(fmaxf(az0, bz0), cull_t));
    const float en1 = fmaxf(fmaxf(fminf(ax1, bx1), fminf(ay1, by1)), fmaxf(fminf(az1, bz1), 0.0f));
    const float ex1 = fminf(fminf(fmaxf(ax1, bx1), fmaxf(ay1, by1)), fminf(fmaxf(az1, bz1), cull_t));
    const bool h0 = en0 <= ex0, h1 = en1 <= ex1;
    const int c0 = __float_as_int(n3.x), c1 = __float_as_int(n3.y);
    if (h0 && h1) {
      const bool first0 = en0 <= en1;
      stack[s.sp++] = first0 ? c1 : c0;
      s.cur = first0 ? c0 : c1;
    } else if (h0) {
      s.cur = c0;
    } else if (h1) {
      s.cur = c1;
    } else {
      s.cur = stack[--s.sp];
    }
  }
  if (s.cur < 0 && s.cur != kTravDone && s.leaf_left == 0) {
    const int code = ~s.cur;
    s.leaf_first = code >> 3;
    s.leaf_left = (code & 7) + 1;
    s.cur = stack[--s.sp];
  }
  if (s.leaf_left > 0) {
    const float4* tp = sc.tris + 3 * (size_t)s.leaf_first;
    const float4 v0 = ldg4(tp + 0), v1 = ldg4(tp + 1), v2 = ldg4(tp + 2);
    if (COUNT) tc.tris++;
    const float t = triangle_mt(f3(v0), f3(v1), f3(v2), s.o, s.d);
    if (t >= 0.0f && LR_NEARER(sc, t, __float_as_int(v0.w), s.best_t, s.best)) {
      s.best_t = t;
      s.best = s.leaf_first;
      s.cull_t = t * 1.0001f + 1e-4f;
    }
    s.leaf_first++;
    s.leaf_left--;
  }
}
template <bool COUNT>
LR_DEV void bvh_traverse_unified(const DevScene& sc, F3 o, F3 d, F3 inv, float& best_t, int& best, TraceCounters& tc) {
  int stack[kStackDepth];
  TravState s;
  trav_begin(s, stack, o, d, inv, best_t, best);
  while (!trav_done(s)) trav_step<COUNT>(sc, s, stack, tc);
  best_t = s.best_t;
  best = s.best;
}

LR_DEV bool bvh_hit_is_gated(const DevScene& sc, F3 o, F3 inv, int id) { return tri_gate(sc, o, inv, id); }

// Nearest hit: flat candidates first, then the BVH; among equal distances the lowest primitive id wins (the tie rule above).
template <bool COUNT>
LR_DEV void trace(const DevScene& sc, F3 o, F3 d, float& t_out, int& id_out, TraceCounters& tc) {
  const F3 inv = f3(1.0f / d.x, 1.0f / d.y, 1.0f / d.z);
  float best_t = 3.0e38f;
  int best = -1;
  flat_hits<COUNT>(sc, flat_list_global(sc), o, d, inv, best_t, best, tc);
  if (sc.n_nodes > 0) bvh_traverse<COUNT>(sc, o, d, inv, best_t, best, tc);
  t_out = best_t;
  id_out = best;
}

struct Surface {
  F3 pos, n;
  int mat, prim;
};

// Intersection record of the nearest hit (triangle.rs:93-99, sphere.rs:55-62)
LR_DEV Surface surface_at(const DevScene& sc, F3 o, F3 d, float t, int id) {
  Surface s;
  s.pos = o + d * t;
  if (id >= 0) {
    const float4* tp = sc.tris + 3 * (size_t)id;
    s.n = f3(ldg4(sc.tri_n + id));                     // triangle.rs:36, computed once at upload like Triangle::new
    s.prim = __float_as_int(ldg4(tp + 0).w);
    s.mat = __float_as_int(ldg4(tp + 1).w);
  } else {
    const int i = -2 - id;
    const float4 sp = ldg4(sc.spheres + i);
    const int2 meta = __ldg(sc.sphere_meta + i);
    s.n = normalize(s.pos - f3(sp));                   // sphere.rs:56
    s.mat = meta.x;
    s.prim = meta.y;
  }
  return s;
}

// ------------------------------------------------------------------ sampling utilities (util.rs)
LR_DEV void orthonormal_basis(F3 n, F3& tangent, F3& binormal) {   // util.rs:12-21
  const F3 a = fabsf(n.x) > kEPS ? f3(0.0f, 1.0f, 0.0f) : f3(1.0f, 0.0f, 0.0f);
  tangent = normalize(cross(a, n));                                // one component is +-0 whatever n is
  binormal = cross(n, tangent);
}
LR_DEV F3 reflect(F3 v, F3 normal) { return -v + normal * (dot(v, normal) * 2.0f); }   // util.rs:30-32
LR_DEV bool refract(F3 v, F3 normal, float eta, F3& out) {                               // util.rs:34-42
  const float dn = dot(v, normal);
  const float cos2theta = 1.0f - (eta * eta) * (1.0f - dn * dn);
  if (cos2theta > 0.0f) {
    out = -v * eta - normal * (eta * -dn + sqrtf(cos2theta));
    return true;
  }
  return false;
}
LR_DEV F3 orienting_normal(F3 out_, F3 normal) {                   // lambert.rs:14-21
  if (dot(normal, out_) < 0.0f) return normal * -1.0f;
  return normal;
}

// ------------------------------------------------------------------ materials
struct Mat {
  F3 color; int type;
  F3 emission; float param0;
  float param1, weight; bool emissive;
};
LR_DEV Mat load_mat(const DevScene& sc, int i) {
  const float4 a = ldg4(sc.mats + 3 * i), b = ldg4(sc.mats + 3 * i + 1), c = ldg4(sc.mats + 3 * i + 2);
  Mat m;
  m.color = f3(a); m.type = __float_as_int(a.w);
  m.emission = f3(b); m.param0 = b.w;
  m.param1 = c.x; m.weight = c.y; m.emissive = c.z != 0.0f;
  return m;
}

// fmodf(x, m) for x >= 0 and a positive module m (the checker's 30 / 150 / 300), exactly and without a division, given
// m_rcp = RN(1 / m): q0 = trunc(RN(x * m_rcp)) is the integer quotient floor(x / m) or one off IN EITHER DIRECTION (the
// product carries two roundings of at most half an ulp each, so it can land just below an integer the true quotient
// reaches as well as just above it), r0 = x - q0*m by one FMA tells which (rounding is monotonic, so r0 < 0 and
// r0 >= m are decided as for the exact value), and x - q*m with the corrected q is the remainder itself, exactly
// representable (fmod is exact), so the last FMA does not round.  Beyond a quotient of 2^23 (and for NaN / inf) the
// library routine.  Checked against fmod for every float32 x in tests/test_exact_quotients.py.
LR_COLD float fmodf_cold(float x, float m) { return fmodf(x, m); }
LR_DEV float fmod_pos(float x, float m, float m_rcp) {
  if (!(x < m * 8388608.0f)) return fmodf_cold(x, m);                   // quotient beyond 2^23: the library routine (also NaN / inf)
  const float q0 = truncf(__fmul_rn(x, m_rcp));
  const float r0 = __fmaf_rn(-q0, m, x);
  const float q = r0 < 0.0f ? q0 - 1.0f : (r0 >= m ? q0 + 1.0f : q0);
  return __fmaf_rn(-q, m, x);
}
LR_DEV float signed_mod(float base, float module, float module_rcp) {   // lambert.rs:58-64  (base % module on |base|)
  const float r = fmod_pos(fabsf(base), module, module_rcp);
  return base > 0.0f ? r : module - r;
}
LR_DEV float checker(float u, float v) {                           // lambert.rs:66-90 (grey value)
  const float lw = 2.0f, li = 150.0f, sw = 1.0f, si = 30.0f, cw = 150.0f, ci = 300.0f;
  const float li_rcp = 0x1.b4e81cp-8f, si_rcp = 0x1.111112p-5f, ci_rcp = 0x1.b4e81cp-9f;   // RN(1 / 150), RN(1 / 30), RN(1 / 300)
  const float lu = signed_mod(u, li, li_rcp), lv = signed_mod(v, li, li_rcp);
  if (lu < lw || lv < lw) return 0.5f;
  const float su = signed_mod(u, si, si_rcp), sv = signed_mod(v, si, si_rcp);
  if (su < sw || sv < sw) return 0.6f;
  const float cu = signed_mod(u, ci, ci_rcp), cv = signed_mod(v, ci, ci_rcp);
  if ((cu < cw || cv < cw) && !(cu < cw && cv < cw)) return 0.8f;
  return 1.0f;
}
LR_DEV float powi5(float x) { const float x2 = x * x; const float x4 = x2 * x2; return x * x4; }   // llvm.powi(x, 5)

LR_DEV float ggx_g1(float a2, F3 v, F3 n) {                        // ggx.rs:27-32
  const float c = dot(v, n);
  const float tan = 1.0f / (c * c) - 1.0f;
  return 2.0f / (1.0f + sqrtf(1.0f + a2 * tan * tan));
}
LR_DEV float ggx_ndf(float a2, F3 m, F3 n) {                       // ggx.rs:34-39
  const float mdn = dot(m, n);
  const float x = (a2 - 1.0f) * mdn * mdn + 1.0f;
  return a2 / (kPI * x * x);
}
LR_DEV void ior_pair(const Mat& m, F3 out_, F3 n, float& from_ior, float& to_ior) {   // ideal_refraction.rs:117-135
  if (dot(out_, n) > 0.0f) { from_ior = 1.0f; to_ior = m.param1; } else { from_ior = m.param1; to_ior = 1.0f; }
}
LR_DEV float fresnel_exact(float n1, float n2, F3 out_, F3 in_, F3 on) {               // ideal_refraction.rs:137-147
  const float cos1 = dot(out_, on);
  const float cos2 = dot(in_, -on);
  const float a = (n1 * cos1 - n2 * cos2) / (n1 * cos1 + n2 * cos2);
  const float b = (n1 * cos2 - n2 * cos1) / (n1 * cos2 + n2 * cos1);
  return (a * a + b * b) / 2.0f;
}

// Material::brdf of Phong, Blinn-Phong and ideal refraction
LR_COLD F3 mat_brdf_other(int type, F3 color, float param0, float param1, F3 out_, F3 in_, F3 n) {
  if (type == LR_MAT_PHONG) {                                      // phong.rs:39-47
    const F3 on = orienting_normal(out_, n);
    if (dot(in_, on) <= 0.0f) return f3(0.0f, 0.0f, 0.0f);
    const F3 r = reflect(out_, on);
    const float c = dot(r, in_);
    const float a = param0;
    return color * ((a + 2.0f) / (2.0f * kPI) * powf(c, a));
  }
  if (type == LR_MAT_BLINN_PHONG) {                                // blinn_phong.rs:39-49
    const F3 on = orienting_normal(out_, n);
    if (dot(in_, on) <= 0.0f) return f3(0.0f, 0.0f, 0.0f);
    const F3 h = normalize(in_ + out_);
    const float c = dot(h, on);
    const float a = param0;
    return color * ((a + 2.0f) * (a + 4.0f) / (8.0f * kPI * (powf(2.0f, -a / 2.0f) + a)) * powf(c, a));
  }
  {                                                                // ideal_refraction.rs:40-68
    const F3 on = orienting_normal(out_, n);
    float from_ior, to_ior;
    if (dot(out_, n) > 0.0f) { from_ior = 1.0f; to_ior = param1; } else { from_ior = param1; to_ior = 1.0f; }   // ior_pair
    F3 r;
    if (refract(out_, on, from_ior / to_ior, r)) {
      const float fr = fresnel_exact(from_ior, to_ior, out_, r, on);
      if (dot(in_, on) > 0.0f) return color * 1.0f / dot(in_, n) * fr;
      const float q = to_ior / from_ior;
      const float ft = (1.0f - fr) * (q * q);
      return color * 1.0f / dot(in_, n) * ft;
    }
    return color * 1.0f / dot(in_, n);
  }
}

// GGX is hot in scenes that use it and dead weight elsewhere: the render kernel is built both ways and chosen by what the
// scene contains (LR_GGX_OUT_OF_LINE, build.py; A/B profiles/r01_c_ab_s26.txt: +3.6 % on sample.toml out of line, -5.5 %
// on brdf.toml, so each gets its own)
#ifdef LR_GGX_OUT_OF_LINE
#define LR_GGX static __device__ __noinline__
#else
#define LR_GGX __device__ __forceinline__
#endif
LR_GGX F3 ggx_brdf(F3 color, float roughness, float ior, F3 out_, F3 in_, F3 n) {      // ggx.rs:71-85
  const F3 on = orienting_normal(out_, n);
  if (dot(in_, on) <= 0.0f) return f3(0.0f, 0.0f, 0.0f);
  const F3 h = normalize(in_ + out_);
  const float alpha = roughness * roughness;
  const float a2 = alpha * alpha;
  const float nnn = 1.0f - ior, nnp = 1.0f + ior;                  // ggx.rs:41-47
  const float f_0 = (nnn * nnn) / (nnp * nnp);
  const float f = f_0 + (1.0f - f_0) * powi5(1.0f - dot(in_, h));
  const float g = ggx_g1(a2, in_, on) * ggx_g1(a2, out_, on);
  const float d = ggx_ndf(a2, h, on);
  return color * f * g * d / (4.0f * dot(in_, on) * dot(out_, on));
}
LR_GGX void ggx_sample(float roughness, F3 out_, F3 on, float xi2, float s1, float c1, F3* in_, float* pdf) {   // ggx.rs:87-113
  F3 u, v;
  orthonormal_basis(on, u, v);
  const float alpha = roughness * roughness;
  const float a2 = alpha * alpha;
  const float tan = alpha * sqrtf(xi2 / (1.0f - xi2));
  const float x = 1.0f + tan * tan;
  const float c = 1.0f / sqrtf(x);
  const float s = tan / sqrtf(x);
  const F3 h = u * c1 * s + v * s1 * s + on * c;
  const float o_h = dot(out_, h);
  *in_ = h * (2.0f * o_h) - out_;
  const float jacobian = 1.0f / (4.0f * o_h);
  *pdf = ggx_ndf(a2, h, on) * dot(h, on) * jacobian;
}

// Material::brdf
LR_DEV F3 mat_brdf(const Mat& m, F3 out_, F3 in_, F3 n, F3 pos) {
  if (m.type == LR_MAT_LAMBERT) {                                  // lambert.rs:32-35
    const float c = checker(pos.x, pos.z);
    const F3 cc = m.color * f3(c, c, c);
    return f3(div_pi(cc.x), div_pi(cc.y), div_pi(cc.z));          // cc / kPI, exactly
  }
  if (m.type == LR_MAT_GGX) return ggx_brdf(m.color, m.param0, m.param1, out_, in_, n);
  return mat_brdf_other(m.type, m.color, m.param0, m.param1, out_, in_, n);
}

// Material::sample of ideal refraction (one draw) and of Phong / Blinn-Phong (xi2 and the sin / cos of 2 pi xi1 drawn by the caller)
LR_COLD void mat_sample_refraction(float ior, F3 out_, F3 n, F3 on, unsigned long long rng_state, unsigned long long* rng_out,
                                   F3* in_, float* pdf) {          // ideal_refraction.rs:70-104
  Pcg rng;
  rng.state = rng_state;
  float from_ior, to_ior;
  if (dot(out_, n) > 0.0f) { from_ior = 1.0f; to_ior = ior; } else { from_ior = ior; to_ior = 1.0f; }
  F3 r;
  if (refract(out_, on, from_ior / to_ior, r)) {
    const float fr = fresnel_exact(from_ior, to_ior, out_, r, on);
    if (rng.next() < fr) { *in_ = reflect(out_, on); *pdf = 1.0f * fr; }
    else { *in_ = r; *pdf = 1.0f * (1.0f - fr); }
  } else { *in_ = reflect(out_, on); *pdf = 1.0f; }
  *rng_out = rng.state;
}
LR_COLD void mat_sample_phong_blinn(int type, float a, F3 out_, F3 on, float xi2, float s1, float c1, F3* in_, float* pdf) {
  if (type == LR_MAT_PHONG) {                                      // phong.rs:49-69
    const F3 r = reflect(out_, on);
    F3 u, v;
    orthonormal_basis(r, u, v);
    const float t = powf(xi2, 1.0f / (a + 2.0f));
    const float ts = sqrtf(1.0f - t * t);
    *in_ = u * c1 * ts + v * s1 * ts + r * t;
    *pdf = (a + 2.0f) / (2.0f * kPI) * powf(dot(r, *in_), a);
  } else {                                                         // blinn_phong.rs:51-73
    F3 u, v;
    orthonormal_basis(on, u, v);
    const float t = powf(xi2, 1.0f / (a + 2.0f));
    const float ts = sqrtf(1.0f - t * t);
    const F3 h = u * c1 * ts + v * s1 * ts + on * t;
    *in_ = h * (2.0f * dot(out_, h)) - out_;
    *pdf = (a + 2.0f) / (2.0f * kPI) * powf(dot(on, h), a);
  }
}

// Material::sample (draw order as the reference)
LR_DEV void mat_sample(const Mat& m, F3 out_, F3 n, Pcg& rng, F3& in_, float& pdf) {
  const F3 on = orienting_normal(out_, n);
  if (m.type == LR_MAT_IDEAL_REFRACTION) {
    F3 wi; float pd;
    unsigned long long st;
    mat_sample_refraction(m.param1, out_, n, on, rng.state, &st, &wi, &pd);
    rng.state = st; in_ = wi; pdf = pd;
    return;
  }
  const float xi1 = rng.next();
  const float xi2 = rng.next();
  const float r1 = 2.0f * kPI * xi1;
  float s1, c1;
  spec_sincos(r1, &s1, &c1);
  if (m.type == LR_MAT_LAMBERT) {                                  // lambert.rs:37-55 + util.rs:87-96
    F3 u, v;
    orthonormal_basis(on, u, v);
    const float r2s = sqrtf(xi2);
    const F3 s = f3(c1 * r2s, s1 * r2s, sqrtf(1.0f - xi2));
    in_ = u * s.x + v * s.y + on * s.z;
    pdf = div_pi(dot(in_, n));                                     // dot(in_, n) / kPI, exactly
    return;
  }
  if (m.type == LR_MAT_GGX) {
    F3 wi; float pd;
    ggx_sample(m.param0, out_, on, xi2, s1, c1, &wi, &pd);
    in_ = wi; pdf = pd;
    return;
  }
  F3 wi; float pd;
  mat_sample_phong_blinn(m.type, m.param0, out_, on, xi2, s1, c1, &wi, &pd);
  in_ = wi; pdf = pd;
}

// Material::coef (traits.rs:20-22; ideal_refraction.rs:106-113)
LR_COLD F3 beer_absorption(F3 color, float absorbtance, float fly_distance) {     // ideal_refraction.rs:106-113
  const F3 v = -(f3(1.0f, 1.0f, 1.0f) - color) * absorbtance * fly_distance;
  return f3(expf(v.x), expf(v.y), expf(v.z));
}
LR_DEV F3 mat_coef(const Mat& m, F3 out_, F3 n, float fly_distance) {
  if (m.type == LR_MAT_IDEAL_REFRACTION && dot(out_, n) < 0.0f) return beer_absorption(m.color, m.param0, fly_distance);
  return f3(1.0f, 1.0f, 1.0f);
}

// ------------------------------------------------------------------ sky (sky.rs)
LR_DEV unsigned long long f32_to_usize(float v) {   // Rust `as usize`: saturating, NaN -> 0
  if (!(v > 0.0f)) return 0ull;
  if (v >= 1.8446744e19f) return 0xFFFFFFFFFFFFFFFFull;
  return (unsigned long long)v;
}
// IBLSky::radiance sky.rs:57-79: nearest texel of a 2H x H equirect image
LR_COLD F3 sky_ibl(const float4* __restrict__ pixels, int sky_height, float longitude_offset, F3 d) {
  const float theta = acosf(d.y);
  const float phi = atan2f(d.z, d.x);
  // `x % 1.0` (sky.rs:60-61) is x - trunc(x) EXACTLY: below 2^23 the difference of x and its integer part needs no more
  // bits than x has, above it x is an integer (the signed zero fmod would give there indexes the same texel), NaN and inf
  // give NaN either way.  Two subtractions instead of two calls of the library's fmodf loop on every path that ends in the sky.
  const float uq = (phi + kPI + longitude_offset) / (2.0f * kPI);
  const float vq = theta / kPI;
  const float u = uq - truncf(uq);
  const float v = vq - truncf(vq);
  const unsigned long long height = (unsigned long long)sky_height;
  const unsigned long long width = height * 2ull;
  const unsigned long long all = width * height;
  const unsigned long long x = f32_to_usize(floorf((float)width * u));
  const unsigned long long y = f32_to_usize(floorf((float)height * v));
  const unsigned long long index = y * width + x;
  return f3(ldg4(pixels + (index % all)));
}
LR_DEV F3 sky_radiance(const DevScene& sc, F3 d) {
  if (sc.sky_type == LR_SKY_UNIFORM) return f3(sc.sky_color);      // sky.rs:17-21
  return sky_ibl(sc.sky_pixels, sc.sky_height, sc.sky_longitude_offset, d);
}

// ------------------------------------------------------------------ cameras (camera.rs)
LR_DEV F3 cam_sensor_point(const LrCamera& c, int left, int top, float u, float v) {   // camera.rs:64-81
  const float px = ((((float)left + u) / (float)c.width) - 0.5f) * c.sensor_size[0];
  const float py = ((((float)top + v) / (float)c.height) - 0.5f) * c.sensor_size[1];
  return f3(c.position) - f3(c.right) * px + f3(c.up) * py;
}
LR_DEV F3 cam_aperture_point(const LrCamera& c, float xi1, float xi2) {                // camera.rs:285-300
  const float u = 2.0f * kPI * xi1;
  const float v = sqrtf(xi2) * c.aperture_radius;
  float su, cu;
  spec_sincos(u, &su, &cu);
  return f3(c.aperture_position) + f3(c.right) * (cu * v) + f3(c.up) * (su * v);
}
LR_DEV float cam_geometry_term(const LrCamera& c, F3 direction) {                      // camera.rs:302-309
  const float cos_term = dot(direction, f3(c.forward));
  const float d = c.aperture_sensor_distance / cos_term;
  return cos_term * cos_term / (d * d);
}
// Returns the ray and the per-sample weight  g_term * (sensor_sensitivity / pdf)  (main.rs:99-101);
// `draw` supplies the U[0,1) numbers in the reference's order: sensor u, v, then aperture 2.
template <class Draw>
LR_DEV void camera_sample(const LrCamera& c, int x, int y, Draw&& draw, F3& o, F3& d, float& g_term, float& sens_over_pdf) {
  const float u = draw();
  const float v = draw();
  if (c.type == LR_CAM_IDEAL_PINHOLE) {                            // camera.rs:100-115
    const F3 sensor = cam_sensor_point(c, x, y, u, v);
    o = f3(c.aperture_position);
    d = normalize(o - sensor);
    g_term = 1.0f;
    sens_over_pdf = c.sensor_sensitivity / (1.0f * 1.0f);
  } else if (c.type == LR_CAM_OMNIDIRECTIONAL) {                   // camera.rs:168-188
    const float p = ((float)x + u) / (float)c.width * kPI * 2.0f;
    const float t = ((float)y + v) / (float)c.height * kPI;
    float sp, cp, st, ct;
    spec_sincos(p, &sp, &cp);
    spec_sincos(t, &st, &ct);
    o = f3(c.aperture_position);
    d = f3(st * cp, st * sp, ct);
    g_term = 1.0f;
    sens_over_pdf = c.sensor_sensitivity / 1.0f;
  } else {
    const F3 sensor = cam_sensor_point(c, x, y, u, v);
    const float sensor_pdf = 1.0f / c.sensor_pixel_area;
    const float a1 = draw();
    const float a2 = draw();
    const F3 ap = cam_aperture_point(c, a1, a2);
    const float ap_pdf = 1.0f / (kPI * c.aperture_radius * c.aperture_radius);
    o = ap;
    if (c.type == LR_CAM_PINHOLE) {                                // camera.rs:313-328
      d = normalize(ap - sensor);
      g_term = cam_geometry_term(c, d);
    } else {                                                       // camera.rs:458-476
      const F3 apc = f3(c.aperture_position);
      const F3 sensor_center = apc - sensor;
      const F3 object_plane = sensor_center * (c.focus_distance / dot(sensor_center, f3(c.forward)));
      d = normalize(apc + object_plane - ap);
      g_term = cam_geometry_term(c, normalize(ap - sensor));
    }
    sens_over_pdf = c.sensor_sensitivity / (sensor_pdf * ap_pdf);
  }
}

// camera.sample for the render kernel: the ideal pinhole inline, the lens cameras out of line
LR_COLD void camera_sample_lens(const LrCamera* c, int x, int y, unsigned long long rng_state, unsigned long long* rng_out, F3* o, F3* d,
                                float* g_term, float* sens_over_pdf) {
  Pcg rng;
  rng.state = rng_state;
  F3 oo, dd;
  float g, w;
  camera_sample(*c, x, y, [&]() { return rng.next(); }, oo, dd, g, w);
  *rng_out = rng.state; *o = oo; *d = dd; *g_term = g; *sens_over_pdf = w;
}
LR_DEV void camera_sample_rng(const LrCamera& c, int x, int y, Pcg& rng, F3& o, F3& d, float& g_term, float& sens_over_pdf) {
  if (c.type == LR_CAM_IDEAL_PINHOLE) {                            // camera.rs:100-115
    const float u = rng.next();
    const float v = rng.next();
    const F3 sensor = cam_sensor_point(c, x, y, u, v);
    o = f3(c.aperture_position);
    d = normalize(o - sensor);
    g_term = 1.0f;
    sens_over_pdf = c.sensor_sensitivity / (1.0f * 1.0f);
  } else {
    unsigned long long st;
    F3 oo, dd;
    float g, w;
    camera_sample_lens(&c, x, y, rng.state, &st, &oo, &dd, &g, &w);
    rng.state = st; o = oo; d = dd; g_term = g; sens_over_pdf = w;
  }
}

}  // namespace lr
