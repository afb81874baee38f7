//! UNTESTED SOURCE (no Rust toolchain offline).  `extern "C"` declarations of include/lumilly.h — the
//! drop-in boundary that replaces the `pool.scoped(..)` + channel-gather block of the reference's
//! `src/main.rs:70-132`.  Field order and types mirror the C structs one to one.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

#[repr(C)] #[derive(Clone, Copy)] pub struct LrMaterial { pub type_: i32, pub color: [f32; 3], pub emission: [f32; 3], pub param0: f32, pub param1: f32 }
#[repr(C)] #[derive(Clone, Copy)] pub struct LrTriangle { pub p0: [f32; 3], pub p1: [f32; 3], pub p2: [f32; 3], pub material: i32, pub prim_id: i32 }
#[repr(C)] #[derive(Clone, Copy)] pub struct LrSphere { pub center: [f32; 3], pub radius: f32, pub material: i32, pub prim_id: i32 }
#[repr(C)] #[derive(Clone, Copy)] pub struct LrCamera {
    pub type_: i32, pub width: i32, pub height: i32,
    pub forward: [f32; 3], pub right: [f32; 3], pub up: [f32; 3], pub position: [f32; 3], pub aperture_position: [f32; 3],
    pub sensor_size: [f32; 2], pub aperture_radius: f32, pub aperture_sensor_distance: f32,
    pub sensor_pixel_area: f32, pub sensor_sensitivity: f32, pub focus_distance: f32,
}
#[repr(C)] #[derive(Clone, Copy)] pub struct LrSky { pub type_: i32, pub color: [f32; 3], pub pixels: *const f32, pub n_pixels: i64, pub height: i32, pub longitude_offset: f32 }
#[repr(C)] #[derive(Clone, Copy)] pub struct LrBvhNode { pub f: [f32; 12], pub c: [i32; 2], pub n: [i32; 2] }
#[repr(C)] pub struct LrSceneDesc {
    pub materials: *const LrMaterial, pub n_materials: i32,
    pub triangles: *const LrTriangle, pub n_triangles: i32,
    pub spheres: *const LrSphere, pub n_spheres: i32,
    pub nodes: *const LrBvhNode, pub n_nodes: i32,
    pub bvh_depth: i32, pub n_flat_triangles: i32, pub camera: LrCamera, pub sky: LrSky,
}
#[repr(C)] #[derive(Clone, Copy, Default)] pub struct LrRenderParams {
    pub integrator: i32, pub spp_begin: i32, pub spp_count: i32, pub depth: i32, pub depth_limit: i32, pub no_direct_emitter: i32,
    pub seed: u64, pub crop_x: i32, pub crop_y: i32, pub crop_w: i32, pub crop_h: i32, pub splits: i32, pub count_traversal: i32,
}
#[repr(C)] #[derive(Clone, Copy, Default)] pub struct LrStats {
    pub rays: u64, pub samples: u64, pub nodes_visited: u64, pub tris_tested: u64, pub spheres_tested: u64, pub nonfinite_samples: u64,
    pub gate_retraces: u64, pub flat_tris_tested: u64, pub flat_boxes_tested: u64, pub kernel_ms: f32, pub launches: i32, pub splits: i32,
}
#[repr(C)] #[derive(Clone, Copy, Default)] pub struct LrSceneConfig {
    pub samples: i32, pub depth: i32, pub depth_limit: i32, pub no_direct_emitter: i32, pub threads: i32, pub integrator: i32,
    pub width: i32, pub height: i32, pub output: i32, pub gamma: f32, pub n_prims: i32, pub n_emitters: i32, pub bvh_build_seconds: f32,
    pub bvh_builder: i32, pub bvh_device_kernel_ms: f32,
}
pub enum LrScene {}
pub enum LrHostScene {}
pub enum LrFilm {}
pub enum LrMultiScene {}
pub enum LrMultiFilm {}
pub const LR_AOV_NORMAL: i32 = 0;
pub const LR_AOV_DEPTH: i32 = 1;
pub const LR_BVH_HOST: i32 = 0;
pub const LR_BVH_DEVICE: i32 = 1;
pub const LR_QUERY_STRICT: i32 = 0;
pub const LR_QUERY_RENDER: i32 = 1;

extern "C" {
    pub fn lr_abi_version() -> c_int;
    pub fn lr_init(device: c_int) -> c_int;
    pub fn lr_shutdown();
    pub fn lr_last_error() -> *const c_char;
    pub fn lr_scene_create(desc: *const LrSceneDesc, out: *mut *mut LrScene) -> c_int;
    pub fn lr_scene_destroy(scene: *mut LrScene);
    pub fn lr_render(scene: *const LrScene, params: *const LrRenderParams, out_rgb: *mut f32, out_sumsq: *mut f32, stats: *mut LrStats) -> c_int;
    pub fn lr_render_accumulate_device(scene: *const LrScene, params: *const LrRenderParams, d_sum: *mut f32, d_sumsq: *mut f32, stream: *mut c_void) -> c_int;
    pub fn lr_stats_fetch(scene: *const LrScene, stream: *mut c_void, stats: *mut LrStats) -> c_int;
    pub fn lr_shard_range(spp_begin: i32, spp_count: i32, part: i32, n_parts: i32, begin: *mut i32, count: *mut i32) -> c_int;
    /// main.rs:70-132 on several GPUs of one box from this one process (scene on every device, sample ranges sharded,
    /// one peer-reading reduce kernel on devices[0])
    pub fn lr_render_multi(desc: *const LrSceneDesc, params: *const LrRenderParams, n_devices: i32, devices: *const i32,
                           out_rgb: *mut f32, out_sumsq: *mut f32, stats: *mut LrStats) -> c_int;
    /// the multi-GPU scene as a handle: set-up once, then renders only
    pub fn lr_multi_scene_create(desc: *const LrSceneDesc, n_devices: i32, devices: *const i32, out: *mut *mut LrMultiScene) -> c_int;
    pub fn lr_multi_render(ms: *mut LrMultiScene, params: *const LrRenderParams, out_rgb: *mut f32, out_sumsq: *mut f32, stats: *mut LrStats) -> c_int;
    pub fn lr_multi_scene_destroy(ms: *mut LrMultiScene);
    /// Scene::normal / Scene::depth (scene.rs:48-62) of the camera rays of the sample range, averaged per pixel
    pub fn lr_render_aov(scene: *const LrScene, params: *const LrRenderParams, kind: i32, out: *mut f32) -> c_int;
    /// progressive / resumable rendering (the hook main.rs:81-91 abandoned): per-pixel sums kept on the device
    pub fn lr_film_create(scene: *const LrScene, params: *const LrRenderParams, want_sumsq: i32, out: *mut *mut LrFilm) -> c_int;
    pub fn lr_film_render(film: *mut LrFilm, spp_count: i32, stats: *mut LrStats) -> c_int;
    pub fn lr_film_info(film: *const LrFilm, spp_done: *mut i32, crop_w: *mut i32, crop_h: *mut i32, has_sumsq: *mut i32) -> c_int;
    pub fn lr_film_read(film: *const LrFilm, out_rgb: *mut f32, out_sumsq: *mut f32) -> c_int;
    pub fn lr_film_save(film: *const LrFilm, path: *const c_char) -> c_int;
    pub fn lr_film_load(scene: *const LrScene, path: *const c_char, out: *mut *mut LrFilm) -> c_int;
    pub fn lr_film_destroy(film: *mut LrFilm);
    pub fn lr_multi_film_create(ms: *mut LrMultiScene, params: *const LrRenderParams, want_sumsq: i32, out: *mut *mut LrMultiFilm) -> c_int;
    pub fn lr_multi_film_render(film: *mut LrMultiFilm, spp_count: i32, stats: *mut LrStats) -> c_int;
    pub fn lr_multi_film_info(film: *const LrMultiFilm, spp_done: *mut i32, crop_w: *mut i32, crop_h: *mut i32, has_sumsq: *mut i32) -> c_int;
    pub fn lr_multi_film_read(film: *const LrMultiFilm, out_rgb: *mut f32, out_sumsq: *mut f32) -> c_int;
    pub fn lr_multi_film_save(film: *const LrMultiFilm, path: *const c_char) -> c_int;
    pub fn lr_multi_film_load(ms: *mut LrMultiScene, path: *const c_char, out: *mut *mut LrMultiFilm) -> c_int;
    pub fn lr_multi_film_destroy(film: *mut LrMultiFilm);
    /// adaptive sampling: spp_count more samples on the tiles whose relative standard error exceeds `threshold`, each from
    /// its own count (max_spp > 0 caps a tile's samples); the per-pixel sample counts of either film
    pub fn lr_film_render_adaptive(film: *mut LrFilm, spp_count: i32, threshold: f32, max_spp: i32, active_tiles: *mut i32, stats: *mut LrStats) -> c_int;
    pub fn lr_film_spp_map(film: *const LrFilm, out: *mut i32) -> c_int;
    pub fn lr_multi_film_render_adaptive(film: *mut LrMultiFilm, spp_count: i32, threshold: f32, max_spp: i32, active_tiles: *mut i32,
                                         stats: *mut LrStats) -> c_int;
    pub fn lr_multi_film_spp_map(film: *const LrMultiFilm, out: *mut i32) -> c_int;
    pub fn lr_trace_primary(scene: *const LrScene, u: f32, v: f32, ua: f32, va: f32, prim: *mut i32, t: *mut f32) -> c_int;
    pub fn lr_trace_rays(scene: *const LrScene, n: i64, origins: *const f32, directions: *const f32, prim: *mut i32, t: *mut f32, normal: *mut f32) -> c_int;
    pub fn lr_trace_rays_query(scene: *const LrScene, n: i64, origins: *const f32, directions: *const f32, query: i32, prim: *mut i32, t: *mut f32,
                               normal: *mut f32) -> c_int;
    /// BVH::new (bvh.rs:57-127) again, by the host's binned-SAH builder or by the device's radix-tree builder
    pub fn lr_host_scene_rebuild_bvh(hs: *mut LrHostScene, builder: i32) -> c_int;
    pub fn lr_host_scene_load(toml_path: *const c_char, asset_root: *const c_char, w: i32, h: i32, out: *mut *mut LrHostScene) -> c_int;
    pub fn lr_host_scene_from_arrays(materials: *const LrMaterial, n_materials: i32, triangles: *const LrTriangle, n_triangles: i32,
                                     spheres: *const LrSphere, n_spheres: i32, camera: *const LrCamera, sky: *const LrSky,
                                     out: *mut *mut LrHostScene) -> c_int;
    pub fn lr_host_scene_desc(hs: *const LrHostScene) -> *const LrSceneDesc;
    pub fn lr_host_scene_config(hs: *const LrHostScene, cfg: *mut LrSceneConfig) -> c_int;
    pub fn lr_host_scene_free(hs: *mut LrHostScene);
}
