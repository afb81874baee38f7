"""Host-side mirror of the reference's driver interface for the hot path, on top of the C ABI.

Names follow the reference: `Description` (description.rs:26-81: parse the TOML, expose `config`,
`camera()`, `scene()`), `Scene` (scene.rs:11-17: owns the objects, renders radiance).  Everything that
computes goes through liblumilly_b200.so; Python only moves arguments and numpy buffers.
"""
import ctypes as C

import numpy as np

from . import capi
from .capi import LrRenderParams, LrStats, check

INTEGRATORS = {"pt": capi.LR_INTEGRATOR_PT, "pt-direct": capi.LR_INTEGRATOR_PT_DIRECT}


def _fptr(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _iptr(a):
    return a.ctypes.data_as(C.POINTER(C.c_int32))


def params_from_config(cfg, integrator=None, spp=None, spp_begin=0, seed=0, crop=None, splits=0, count=False,
                       depth=None, depth_limit=None, no_direct_emitter=None):
    """LrRenderParams from the scene's [renderer] table with optional overrides."""
    p = LrRenderParams()
    if integrator is None:
        p.integrator = cfg.integrator
    else:
        p.integrator = INTEGRATORS[integrator] if isinstance(integrator, str) else int(integrator)
    p.spp_begin = int(spp_begin)
    p.spp_count = int(spp if spp is not None else cfg.samples)
    p.depth = int(cfg.depth if depth is None else depth)
    p.depth_limit = int(cfg.depth_limit if depth_limit is None else depth_limit)
    p.no_direct_emitter = int(cfg.no_direct_emitter if no_direct_emitter is None else no_direct_emitter)
    p.seed = int(seed)
    if crop:
        p.crop_x, p.crop_y, p.crop_w, p.crop_h = [int(v) for v in crop]
    p.splits = int(splits)
    p.count_traversal = 1 if count else 0
    return p


class Description:
    """`Description::new(path)` — loads a scene TOML through the host front end (C++)."""

    def __init__(self, path=None, asset_root=None, resolution=None, _handle=None):
        self._lib = capi.load_library()
        self._h = C.c_void_p()
        if _handle is not None:
            self._h = _handle
        else:
            w, h = resolution if resolution else (0, 0)
            check(self._lib.lr_host_scene_load(str(path).encode(), (str(asset_root).encode() if asset_root else None),
                                               int(w), int(h), C.byref(self._h)))
        cfg = capi.LrSceneConfig()
        check(self._lib.lr_host_scene_config(self._h, C.byref(cfg)))
        self.config = cfg
        self.path = path

    @classmethod
    def from_arrays(cls, materials, triangles, spheres, camera, sky=None):
        """Builds a description from ctypes arrays (materials/triangles/spheres) — used by tests and tools."""
        lib = capi.load_library()
        h = C.c_void_p()
        nm, nt, ns = len(materials), len(triangles), len(spheres)
        check(lib.lr_host_scene_from_arrays(materials if nm else None, nm, triangles if nt else None, nt,
                                            spheres if ns else None, ns, C.byref(camera),
                                            C.byref(sky) if sky is not None else None, C.byref(h)))
        return cls(_handle=h)

    @property
    def desc(self):
        return self._lib.lr_host_scene_desc(self._h)

    def rebuild_bvh(self, builder="device"):
        """Rebuilds the BVH (BVH::new, bvh.rs:57-127): "host" = binned SAH on the host's cores, "device" = radix tree built
        by CUDA kernels (needs a GPU).  Returns the build's wall seconds; `config` is refreshed."""
        b = {"host": capi.LR_BVH_HOST, "device": capi.LR_BVH_DEVICE}[builder] if isinstance(builder, str) else int(builder)
        check(self._lib.lr_host_scene_rebuild_bvh(self._h, b))
        check(self._lib.lr_host_scene_config(self._h, C.byref(self.config)))
        return self.config.bvh_build_seconds

    def camera(self):
        return self.desc.contents.camera

    def scene(self):
        return Scene(self)

    def render_multi(self, devices, sumsq=False, **kw):
        """One process, several GPUs (lr_render_multi): the scene goes to every device in `devices`, the sample range is
        sharded by sample index, one kernel on devices[0] sums the peers' buffers over NVLink and divides by spp.
        Returns (mean image, sumsq or None, stats dict) like Scene.render."""
        p = kw.pop("params", None) or params_from_config(self.config, **kw)
        shape = (p.crop_h, p.crop_w, 3) if p.crop_w > 0 else (self.config.height, self.config.width, 3)
        img = np.empty(shape, dtype=np.float32)
        sq = np.empty(shape, dtype=np.float32) if sumsq else None
        st = LrStats()
        dev = (C.c_int32 * len(devices))(*[int(d) for d in devices])
        check(self._lib.lr_render_multi(self.desc, C.byref(p), len(devices), dev, _fptr(img), _fptr(sq) if sumsq else None, C.byref(st)))
        return img, sq, st.as_dict()

    def multi_scene(self, devices):
        """The scene on several GPUs of this box, set up once (lr_multi_scene_create): see MultiScene."""
        return MultiScene(self, devices)

    def close(self):
        if self._h:
            self._lib.lr_host_scene_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Scene:
    """Device-resident scene (`Description::scene()`); `render` replaces main.rs:70-132."""

    def __init__(self, description):
        self._lib = capi.load_library()
        self.description = description
        self.config = description.config
        self._s = C.c_void_p()
        check(self._lib.lr_scene_create(description.desc, C.byref(self._s)))
        self.width, self.height = self.config.width, self.config.height

    @property
    def h2d_bytes(self):
        b = C.c_uint64()
        check(self._lib.lr_scene_bytes(self._s, C.byref(b)))
        return b.value

    def params(self, **kw):
        return params_from_config(self.config, **kw)

    def _shape(self, p):
        return (p.crop_h, p.crop_w, 3) if p.crop_w > 0 else (self.height, self.width, 3)

    def render(self, sumsq=False, **kw):
        """Synchronous render to host buffers: returns (mean image HxWx3 fp32, sumsq or None, stats dict)."""
        p = kw.pop("params", None) or self.params(**kw)
        img = np.empty(self._shape(p), dtype=np.float32)
        sq = np.empty(self._shape(p), dtype=np.float32) if sumsq else None
        st = LrStats()
        check(self._lib.lr_render(self._s, C.byref(p), _fptr(img), _fptr(sq) if sumsq else None, C.byref(st)))
        return img, sq, st.as_dict()

    def render_accumulate(self, d_sum, d_sumsq=None, stream=0, **kw):
        """Adds the sample range's per-pixel sums into device buffers (raw device pointers, e.g.
        torch tensor .data_ptr()), asynchronously on `stream` (a cudaStream_t handle as int)."""
        p = kw.pop("params", None) or self.params(**kw)
        check(self._lib.lr_render_accumulate_device(self._s, C.byref(p), C.c_void_p(int(d_sum)),
                                                    C.c_void_p(int(d_sumsq)) if d_sumsq else None,
                                                    C.c_void_p(int(stream)) if stream else None))
        return p

    def stats(self, stream=0):
        st = LrStats()
        check(self._lib.lr_stats_fetch(self._s, C.c_void_p(int(stream)) if stream else None, C.byref(st)))
        return st.as_dict()

    def render_aov(self, kind, **kw):
        """`Scene::normal` / `Scene::depth` (scene.rs:48-62) of the camera rays of the sample range, averaged per pixel:
        kind "normal" -> HxWx3 (hit ? n/2 + 0.5 : 0), "depth" -> HxW (hit ? distance : 0)."""
        p = kw.pop("params", None) or self.params(**kw)
        k = {"normal": capi.LR_AOV_NORMAL, "depth": capi.LR_AOV_DEPTH}[kind] if isinstance(kind, str) else int(kind)
        shape = self._shape(p) if k == capi.LR_AOV_NORMAL else self._shape(p)[:2]
        out = np.empty(shape, dtype=np.float32)
        check(self._lib.lr_render_aov(self._s, C.byref(p), k, _fptr(out)))
        return out

    def film(self, sumsq=False, **kw):
        """A resumable render of this scene (the progress hook the reference abandoned, main.rs:81-91): see Film."""
        return Film(self, params=kw.pop("params", None) or self.params(**kw), sumsq=sumsq)

    def load_film(self, path):
        return Film(self, path=path)

    def trace_primary(self, u=0.5, v=0.5, ua=0.5, va=0.5):
        prim = np.empty((self.height, self.width), dtype=np.int32)
        t = np.empty((self.height, self.width), dtype=np.float32)
        check(self._lib.lr_trace_primary(self._s, u, v, ua, va, _iptr(prim), _fptr(t)))
        return prim, t

    def trace_rays(self, origins, directions, normals=False, render_query=False):
        """Nearest hits of arbitrary rays: the strict query, or (render_query=True) the query as the render kernels run it."""
        o = np.ascontiguousarray(origins, dtype=np.float32).reshape(-1, 3)
        d = np.ascontiguousarray(directions, dtype=np.float32).reshape(-1, 3)
        n = o.shape[0]
        prim = np.empty(n, dtype=np.int32)
        t = np.empty(n, dtype=np.float32)
        nrm = np.empty((n, 3), dtype=np.float32) if normals else None
        check(self._lib.lr_trace_rays_query(self._s, n, _fptr(o), _fptr(d), 1 if render_query else 0, _iptr(prim), _fptr(t),
                                            _fptr(nrm) if normals else None))
        return (prim, t, nrm) if normals else (prim, t)

    def close(self):
        if self._s:
            self._lib.lr_scene_destroy(self._s)
            self._s = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class MultiScene:
    """One process, several GPUs (lr_multi_scene_create / lr_multi_render): scenes, streams and peer mappings are made once,
    `render` shards the sample range over the devices and returns what Scene.render returns."""

    def __init__(self, description, devices):
        self._lib = capi.load_library()
        self.description = description
        self.config = description.config
        self._m = C.c_void_p()
        dev = (C.c_int32 * len(devices))(*[int(d) for d in devices])
        check(self._lib.lr_multi_scene_create(description.desc, len(devices), dev, C.byref(self._m)))

    def render(self, sumsq=False, **kw):
        p = kw.pop("params", None) or params_from_config(self.config, **kw)
        shape = (p.crop_h, p.crop_w, 3) if p.crop_w > 0 else (self.config.height, self.config.width, 3)
        img = np.empty(shape, dtype=np.float32)
        sq = np.empty(shape, dtype=np.float32) if sumsq else None
        st = LrStats()
        check(self._lib.lr_multi_render(self._m, C.byref(p), _fptr(img), _fptr(sq) if sumsq else None, C.byref(st)))
        return img, sq, st.as_dict()

    def film(self, sumsq=False, **kw):
        """A resumable render on all the devices, sharded by pixel (lr_multi_film_*): see MultiFilm."""
        return MultiFilm(self, params=kw.pop("params", None) or params_from_config(self.config, **kw), sumsq=sumsq)

    def load_film(self, path):
        """Resumes a checkpoint written by Film.save or MultiFilm.save on these devices."""
        return MultiFilm(self, path=path)

    def close(self):
        if self._m:
            self._lib.lr_multi_scene_destroy(self._m)
            self._m = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class _FilmBase:
    """A render in progress behind one of the two film handles of the C ABI; `_API` is the prefix of its entry points
    (lr_film_* or lr_multi_film_*), `owner` the handle they are created on."""
    _API = None

    def __init__(self, owner, params=None, sumsq=False, path=None):
        self._lib = capi.load_library()
        self._fn = {n: getattr(self._lib, "%s_%s" % (self._API, n))
                    for n in ("create", "load", "render", "render_adaptive", "info", "spp_map", "read", "save", "destroy")}
        self._f = C.c_void_p()
        if path is not None:
            check(self._fn["load"](owner, str(path).encode(), C.byref(self._f)))
        else:
            check(self._fn["create"](owner, C.byref(params), 1 if sumsq else 0, C.byref(self._f)))
        _, w, h, self.has_sumsq = self._info()
        self._shape = (h, w, 3)

    def _info(self):
        v = [C.c_int32() for _ in range(4)]
        check(self._fn["info"](self._f, *[C.byref(x) for x in v]))
        return [x.value for x in v]

    @property
    def spp(self):
        return self._info()[0]

    def render(self, spp):
        st = LrStats()
        check(self._fn["render"](self._f, int(spp), C.byref(st)))
        return st.as_dict()

    def render_adaptive(self, spp, threshold, max_spp=0):
        """Adds `spp` samples to every 8x4 tile whose relative standard error exceeds `threshold`, each tile from its own
        count; tiles holding `max_spp` samples (if > 0) are left alone.  Needs a film made with sumsq=True.  Returns the
        stats dict plus `active_tiles`, the tiles rendered (0: the film has converged)."""
        st = LrStats()
        active = C.c_int32()
        check(self._fn["render_adaptive"](self._f, int(spp), float(threshold), int(max_spp), C.byref(active), C.byref(st)))
        d = st.as_dict()
        d["active_tiles"] = active.value
        return d

    def spp_map(self):
        """The samples every pixel of the crop holds, (h, w) int32."""
        out = np.empty(self._shape[:2], dtype=np.int32)
        check(self._fn["spp_map"](self._f, _iptr(out)))
        return out

    def read(self, sumsq=False):
        img = np.empty(self._shape, dtype=np.float32)
        sq = np.empty(self._shape, dtype=np.float32) if sumsq else None
        check(self._fn["read"](self._f, _fptr(img), _fptr(sq) if sumsq else None))
        return (img, sq) if sumsq else img

    def save(self, path):
        check(self._fn["save"](self._f, str(path).encode()))

    def close(self):
        if self._f:
            self._fn["destroy"](self._f)
            self._f = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Film(_FilmBase):
    """Per-pixel sums of a render in progress on the scene's device (lr_film_*): `render(n)` adds the next n sample
    indices, `read()` gives the mean so far, `save(path)` / `Scene.load_film(path)` checkpoint and resume.  With
    splits = 1 any cut of the sample range into `render` calls gives bit for bit the image of one `Scene.render`."""
    _API = "lr_film"

    def __init__(self, scene, params=None, sumsq=False, path=None):
        self.scene = scene
        super().__init__(scene._s, params, sumsq, path)


class MultiFilm(_FilmBase):
    """The same film on the devices of a MultiScene (lr_multi_film_*), sharded by 8x4 pixel tile: the image, sums of
    squares and ray count are bit for bit those of `Scene.render(splits=1)` for any device count, and its checkpoints
    are those of Film (either kind resumes the other's)."""
    _API = "lr_multi_film"

    def __init__(self, multi_scene, params=None, sumsq=False, path=None):
        self.multi_scene = multi_scene
        super().__init__(multi_scene._m, params, sumsq, path)


def init(device=0):
    check(capi.load_library().lr_init(int(device)))


def device_info():
    lib = capi.load_library()
    sm, l2, khz = C.c_int32(), C.c_int32(), C.c_int32()
    name = C.create_string_buffer(256)
    check(lib.lr_device_info(C.byref(sm), C.byref(l2), C.byref(khz), name, 256))
    return {"sm_count": sm.value, "l2_bytes": l2.value, "sm_clock_khz": khz.value, "name": name.value.decode()}


def measure_l2_read_gbs(working_set_bytes=48 << 20, iters=20):
    g = C.c_float()
    check(capi.load_library().lr_measure_l2_read_gbs(int(working_set_bytes), int(iters), C.byref(g)))
    return g.value


def measure_hbm_read_gbs(nbytes=4 << 30, iters=2):
    g = C.c_float()
    check(capi.load_library().lr_measure_hbm_read_gbs(int(nbytes), int(iters), C.byref(g)))
    return g.value


def save_png(path, img, gamma=2.2):
    a = np.ascontiguousarray(img, dtype=np.float32)
    check(capi.load_library().lr_save_png(str(path).encode(), _fptr(a), a.shape[1], a.shape[0], float(gamma)))


def save_hdr(path, img):
    a = np.ascontiguousarray(img, dtype=np.float32)
    check(capi.load_library().lr_save_hdr(str(path).encode(), _fptr(a), a.shape[1], a.shape[0]))


def load_hdr(path):
    lib = capi.load_library()
    p = C.POINTER(C.c_float)()
    w, h = C.c_int32(), C.c_int32()
    check(lib.lr_load_hdr(str(path).encode(), C.byref(p), C.byref(w), C.byref(h)))
    try:
        return np.ctypeslib.as_array(p, shape=(h.value, w.value, 3)).copy()
    finally:
        lib.lr_free(p)
