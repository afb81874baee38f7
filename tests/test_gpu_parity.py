"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle on the same inputs.

Bars (BASELINE.json north_star / SURVEY.md §8d):
  * primary-ray nearest hit: primitive index equal on >= 99.99 % of pixels, |t_gpu - t_ref| <= 1e-5 * t_ref;
  * replay (shared counter-based RNG + the specified fp32 sincos): the path GEOMETRY replays bit for bit, so
    the ray counts are equal and per-pixel means agree within rtol 1e-4 on >= 99.9 % of pixels (the residue
    is fp32 rounding of the iterative throughput form vs the reference's recursion; Phong / Blinn-Phong also
    call powf, where CUDA and glibc differ by an ulp and a path may diverge: rtol 1e-3 on >= 99.5 %);
  * statistical (independent RNG streams): per channel |mean_g - mean_r| <= 3 sigma on >= 99 % of channels and
    the image-mean difference within 4 standard errors; relMSE printed.
"""
import numpy as np
import pytest

from conftest import load_scene, make_params, mc_agreement

pytestmark = pytest.mark.gpu

SCENE_RES = {
    "primitive": (256, 256),
    "new-cbox": (128, 128),
    "brdf": (240, 135),
    "brdf-phong": (240, 135),
    "brdf-blinn": (240, 135),
    "brdf-thinlens": (240, 135),
    "sample": (160, 160),
    "welcome-2018": (214, 154),
    "primitive-pinhole": (128, 128),
    # the rest of the reference's scenes/ (SURVEY.md §8f-3): ideal refraction + Beer absorption, omnidirectional camera
    "ridaisai-2018": (214, 154),
    "vr": (128, 128),
    "debug-nee": (128, 128),
    "welcome-2018-geo": (214, 154),
}


@pytest.fixture(scope="module")
def scenes(lr, orc, assets, gpu):
    cache = {}

    def get(name):
        if name not in cache:
            d = load_scene(lr, name, SCENE_RES[name])
            cache[name] = (d, d.scene(), orc.OracleScene(d.desc, keepalive=d))
        return cache[name]
    return get


@pytest.mark.parametrize("name", list(SCENE_RES))
@pytest.mark.parametrize("jitter", [(0.5, 0.5, 0.5, 0.5), (0.137, 0.859, 0.301, 0.644)])
def test_primary_hits_match_oracle(scenes, name, jitter):
    d, s, o = scenes(name)
    pg, tg = s.trace_primary(*jitter)
    po, to = o.trace_primary(*jitter, traversal=0)
    assert (pg == po).mean() >= 0.9999, "index agreement %.6f" % (pg == po).mean()
    both = (pg == po) & (po >= 0)
    rel = np.abs(tg[both] - to[both]) / np.abs(to[both])
    assert rel.size == 0 or rel.max() <= 1e-5, "max rel dt %.3e" % rel.max()
    if jitter[2] == 0.5 and d.camera().type in (0,):
        # ideal pinhole: no transcendental on the ray path -> bit-exact distances
        assert np.array_equal(tg[both], to[both])


def _soup(rng, n, scale=10.0, size=1.0):
    c = rng.uniform(-scale, scale, (n, 1, 3))
    return (c + rng.normal(0, size, (n, 3, 3))).astype(np.float32)


def _scene_from_tris(lr, tri, spheres=()):
    from lumillyrender_b200 import capi
    mats = (capi.LrMaterial * 1)()
    mats[0].type = capi.LR_MAT_LAMBERT
    mats[0].color[:] = [0.5, 0.5, 0.5]
    T = (capi.LrTriangle * max(len(tri), 1))()
    pid = 0
    for i, t in enumerate(tri):
        T[i].p0[:] = t[0]; T[i].p1[:] = t[1]; T[i].p2[:] = t[2]
        T[i].material = 0; T[i].prim_id = pid; pid += 1
    S = (capi.LrSphere * max(len(spheres), 1))()
    for i, (c, r) in enumerate(spheres):
        S[i].center[:] = c; S[i].radius = r; S[i].material = 0; S[i].prim_id = pid; pid += 1
    m = (capi.C.c_float * 16)()
    lib = capi.load_library()
    lib.lr_matrix_look_at((capi.C.c_float * 3)(0, 0, 40), (capi.C.c_float * 3)(0, 0, 0), (capi.C.c_float * 3)(0, 1, 0), m)
    cam = capi.LrCamera()
    lib.lr_camera_ideal_pinhole(m, 60.0, 64, 64, capi.C.byref(cam))
    Tn = (capi.LrTriangle * len(tri)).from_buffer(T) if len(tri) else []
    Sn = (capi.LrSphere * len(spheres)).from_buffer(S) if len(spheres) else []
    return lr.Description.from_arrays(mats, Tn, Sn, cam)


@pytest.mark.parametrize("n_tris,n_spheres", [(0, 0), (1, 0), (2, 3), (37, 0), (1000, 5), (20000, 2)])
def test_random_rays_match_brute_force_oracle(lr, orc, gpu, n_tris, n_spheres):
    rng = np.random.RandomState(n_tris + 17 * n_spheres)
    tri = _soup(rng, n_tris)
    spheres = [(rng.uniform(-8, 8, 3).astype(np.float32), float(rng.uniform(0.2, 2.0))) for _ in range(n_spheres)]
    d = _scene_from_tris(lr, tri, spheres)
    s = d.scene()
    o = orc.OracleScene(d.desc, keepalive=d)
    n = 20000
    org = rng.uniform(-12, 12, (n, 3)).astype(np.float32)
    dirs = rng.normal(size=(n, 3)).astype(np.float32)
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True).astype(np.float32)
    # edge cases: axis-parallel directions (1/0 = inf in the slab tests) and rays starting on a surface
    dirs[:60] = np.tile(np.eye(3, dtype=np.float32), (20, 1)) * np.where(np.arange(60) % 2, 1, -1)[:, None]
    if n_tris:
        k = rng.randint(0, n_tris, 200)
        w = rng.dirichlet([1, 1, 1], 200).astype(np.float32)
        org[100:300] = (tri[k] * w[:, :, None]).sum(1)
    pg, tg, ng = s.trace_rays(org, dirs, normals=True)
    po, to, no = o.trace_rays(org, dirs, brute_force=(n_tris <= 1000))
    assert (pg == po).mean() >= 0.9999, "index agreement %.6f" % (pg == po).mean()
    both = (pg == po) & (po >= 0)
    assert np.array_equal(tg[both], to[both]), "hit distances must be bit-identical"
    assert np.array_equal(ng[both], no[both]), "hit normals must be bit-identical"
    if n_tris == 0 and n_spheres == 0:
        assert (pg == -1).all()


@pytest.mark.parametrize("name,spp", [("primitive", 8), ("new-cbox", 8), ("brdf", 8), ("brdf-phong", 8), ("brdf-blinn", 8),
                                      ("brdf-thinlens", 8), ("sample", 4), ("welcome-2018", 4), ("primitive-pinhole", 8),
                                      ("ridaisai-2018", 4), ("vr", 8), ("debug-nee", 8), ("welcome-2018-geo", 4)])
def test_replay_matches_oracle(scenes, lr, name, spp):
    d, s, o = scenes(name)
    img, sq, st = s.render(spp=spp, seed=11, splits=1, sumsq=True)
    ref_sum, ref_sq, ost = o.render(make_params(lr, d.config, spp=spp, seed=11), traversal=0, rng_mode=0, math_mode=1)
    ref = ref_sum / spp
    finite = np.isfinite(ref).all(-1) & np.isfinite(img).all(-1)
    uses_powf = name in ("brdf-phong", "brdf-blinn", "ridaisai-2018")   # powf / expf: libdevice vs glibc may differ by an ulp
    rtol, need = (1e-3, 0.995) if uses_powf else (1e-4, 0.999)
    frac = np.isclose(img, ref, rtol=rtol, atol=rtol * 0.1).all(-1)[finite].mean()
    frac_sq = np.isclose(sq, ref_sq, rtol=10 * rtol, atol=rtol).all(-1)[finite].mean()
    print("%s: replay agreement %.5f (sumsq %.5f) at rtol %g, rays gpu %d oracle %d" % (name, frac, frac_sq, rtol, st["rays"], ost["rays"]))
    assert frac >= need and frac_sq >= need
    if uses_powf:
        assert abs(st["rays"] - ost["rays"]) <= 1e-3 * ost["rays"]
    else:
        assert st["rays"] == ost["rays"], "path geometry must replay exactly"
    assert st["nonfinite_samples"] == ost["nonfinite_samples"] or uses_powf


@pytest.mark.parametrize("name,spp", [("primitive", 32), ("new-cbox", 64), ("brdf", 32), ("brdf-phong", 32), ("brdf-blinn", 32),
                                      ("sample", 32), ("welcome-2018", 16), ("ridaisai-2018", 16), ("vr", 32), ("debug-nee", 32),
                                      ("welcome-2018-geo", 16)])
def test_statistical_parity_independent_streams(scenes, lr, name, spp):
    d, s, o = scenes(name)
    img, sq, st = s.render(spp=spp, seed=5, sumsq=True)
    ref_sum, ref_sq, _ = o.render(make_params(lr, d.config, spp=spp, seed=99), traversal=1, rng_mode=1)
    ok = np.isfinite(img).all(-1) & np.isfinite(ref_sum).all(-1)
    frac, z, relmse = mc_agreement(img[ok], sq[ok], spp, ref_sum[ok] / spp, ref_sq[ok], spp)
    print("%s: within-3sigma %.4f, image-mean z %.2f, relMSE %.4g" % (name, frac, z, relmse))
    assert frac >= 0.99
    # 4 standard errors here: at 16-32 spp the firefly scenes (sun-disc IBL, caustic paths) have heavy-tailed pixel sums and the
    # normal approximation of the image mean is loose (measured: z up to 3.2, oracle vs oracle with two seeds gives the
    # same); the full-size runs at 64 spp hold the 3-sigma bar without slack (tests/test_gpu_fullsize.py)
    assert z <= 4.0


def test_furnace_white_sky_albedo_one(lr, orc, gpu):
    """Albedo-1 Lambert sphere (placed where the hard-coded checker is 1) under a radiance-1 sky: L == 1."""
    from lumillyrender_b200 import capi
    d = _scene_from_tris(lr, np.zeros((0, 3, 3), np.float32), [((15.0, 0.0, 15.0), 1.0)])
    desc = d.desc.contents
    desc.materials[0].color[:] = [1.0, 1.0, 1.0]
    desc.sky.type = capi.LR_SKY_UNIFORM
    desc.sky.color[:] = [1.0, 1.0, 1.0]
    lib = capi.load_library()
    m = (capi.C.c_float * 16)()
    lib.lr_matrix_look_at((capi.C.c_float * 3)(15, 0, 20), (capi.C.c_float * 3)(15, 0, 15), (capi.C.c_float * 3)(0, 1, 0), m)
    lib.lr_camera_ideal_pinhole(m, 40.0, 64, 64, capi.C.byref(desc.camera))
    s = d.scene()
    img, _, st = s.render(integrator="pt", spp=16, seed=3, depth=5, depth_limit=64, no_direct_emitter=0)
    assert np.allclose(img, 1.0, atol=2e-5), (img.min(), img.max())


def test_determinism_crop_and_sharding(scenes, lr):
    d, s, o = scenes("new-cbox")
    a, _, _ = s.render(spp=8, seed=2, splits=1)
    b, _, _ = s.render(spp=8, seed=2, splits=1)
    assert np.array_equal(a, b), "same seed, same splits -> bit-identical"
    c, _, _ = s.render(spp=8, seed=2, splits=1, crop=(40, 24, 32, 16))
    assert np.array_equal(c, a[24:40, 40:72]), "crop renders the same pixels (RNG keyed by film pixel)"
    e, _, _ = s.render(spp=8, seed=3, splits=1)
    assert not np.array_equal(a, e)
    # spp sharding: two ranges summed == one range, up to fp32 summation order
    lo, _, _ = s.render(spp=4, spp_begin=0, seed=2, splits=1)
    hi, _, _ = s.render(spp=4, spp_begin=4, seed=2, splits=1)
    assert np.allclose((lo + hi) / 2, a, rtol=1e-5, atol=1e-6)
    # splits > 1: deterministic too, equal to the unsplit sum up to summation order
    f, _, st = s.render(spp=8, seed=2, splits=4)
    g, _, _ = s.render(spp=8, seed=2, splits=4)
    assert st["splits"] == 4 and np.array_equal(f, g)
    assert np.allclose(f, a, rtol=1e-5, atol=1e-6)


def test_accumulate_device_matches_render(scenes, lr):
    torch = pytest.importorskip("torch")
    d, s, o = scenes("brdf")
    ref, ref_sq, _ = s.render(spp=6, seed=4, splits=1, sumsq=True)
    acc = torch.zeros((s.height, s.width, 3), dtype=torch.float32, device="cuda")
    acc_sq = torch.zeros_like(acc)
    stream = torch.cuda.current_stream().cuda_stream
    s.render_accumulate(acc.data_ptr(), acc_sq.data_ptr(), stream=stream, spp=6, seed=4, splits=1)
    st = s.stats(stream)
    assert st["samples"] == s.width * s.height * 6 and st["rays"] > 0
    assert np.array_equal(acc.cpu().numpy() / np.float32(6.0), ref)
    assert np.array_equal(acc_sq.cpu().numpy(), ref_sq)


@pytest.mark.parametrize("name,spp", [("sample", 6), ("welcome-2018", 4), ("vr", 4)])
def test_kernel_organisations_agree_bit_for_bit(scenes, monkeypatch, name, spp):
    """Scenes with a BVH have two organisations of the render kernel in the library: one path per lane with a deferred
    BVH phase (persistent.cuh) and a per-warp pool of 64 paths in shared memory (pool.cuh).  Scheduling must not change
    a bit: same image, same sum of squares, same ray count, with and without sample-range splits and on a crop."""
    d, s, o = scenes(name)
    out = {}
    for org in ("persistent", "pool"):
        monkeypatch.setenv("LR_ORGANISATION", org)
        img, sq, st = s.render(spp=spp, seed=5, splits=1, sumsq=True)
        split, _, st3 = s.render(spp=spp, seed=5, splits=3)
        crop, _, _ = s.render(spp=spp, seed=5, splits=1, crop=(37, 21, 50, 33))
        assert st3["splits"] == 3
        assert np.array_equal(crop, img[21:21 + 33, 37:37 + 50], equal_nan=True)
        out[org] = (img, sq, split, st["rays"], st["nonfinite_samples"])
    monkeypatch.delenv("LR_ORGANISATION")
    a, b = out["persistent"], out["pool"]
    assert a[3] == b[3] and a[4] == b[4]
    assert all(np.array_equal(a[i], b[i], equal_nan=True) for i in range(3))
    default, _, st = s.render(spp=spp, seed=5, splits=1)
    assert np.array_equal(default, a[0], equal_nan=True) and st["rays"] == a[3]


def test_pool_kernel_small_work(scenes):
    """The pool kernel (sample.toml: pt over a BVH) when there is less work than one warp's pool holds: single-pixel
    and single-row crops, one sample per pixel, more splits than samples — same pixels as the full render."""
    d, s, o = scenes("sample")
    full, _, st = s.render(spp=3, seed=11, splits=1)
    for crop in ((0, 0, 1, 1), (159, 159, 1, 1), (3, 77, 157, 1), (80, 0, 1, 160), (5, 6, 7, 9)):
        x, y, w, h = crop
        c, _, _ = s.render(spp=3, seed=11, splits=1, crop=crop)
        assert c.shape == (h, w, 3) and np.array_equal(c, full[y:y + h, x:x + w]), crop
    one, _, st1 = s.render(spp=1, seed=11, splits=1)
    many, _, stm = s.render(spp=1, seed=11, splits=8)            # clamped to the sample count
    assert stm["splits"] == 1 and np.array_equal(one, many) and st1["rays"] == stm["rays"]
    lo, _, _ = s.render(spp=2, spp_begin=0, seed=11, splits=1)
    hi, _, _ = s.render(spp=1, spp_begin=2, seed=11, splits=1)
    assert np.allclose((lo * 2 + hi) / 3, full, rtol=1e-5, atol=1e-6)


def test_render_multi_single_process(scenes, lr, gpu, monkeypatch):
    """lr_render_multi (one process, the scene on every listed device, sample ranges sharded, one peer-reading reduce
    kernel): with one device it is lr_render bit for bit; with two it equals the single-device render up to the fp32
    order of the cross-device sum, ray counts add up exactly, and it is reproducible.  Error paths return codes."""
    from lumillyrender_b200.capi import LumillyError
    torch = pytest.importorskip("torch")
    d, s, o = scenes("sample")
    ref, ref_sq, st = s.render(spp=6, seed=13, splits=1, sumsq=True)
    one, one_sq, st1 = d.render_multi([0], spp=6, seed=13, splits=1, sumsq=True)
    assert np.array_equal(one, ref) and np.array_equal(one_sq, ref_sq) and st1["rays"] == st["rays"] and st1["samples"] == st["samples"]
    ms1 = d.multi_scene([0])
    a1, _, sta = ms1.render(spp=6, seed=13, splits=1)
    b1, _, _ = ms1.render(spp=3, spp_begin=3, seed=13, splits=1)
    hi3, _, _ = s.render(spp=3, spp_begin=3, seed=13, splits=1)
    assert np.array_equal(a1, ref) and sta["rays"] == st["rays"] and np.array_equal(b1, hi3)
    ms1.close()
    with pytest.raises(LumillyError):
        d.render_multi([0, 0], spp=2)
    with pytest.raises(LumillyError):
        d.render_multi([0, 99], spp=2)
    with pytest.raises(LumillyError):
        d.render_multi([], spp=2)
    # the library is still usable on device 0 afterwards
    again, _, _ = s.render(spp=6, seed=13, splits=1)
    assert np.array_equal(again, ref)
    if torch.cuda.device_count() < 2:
        pytest.skip("the two-device half needs 2 GPUs")
    two, two_sq, st2 = d.render_multi([0, 1], spp=6, seed=13, splits=1, sumsq=True)
    rep, _, _ = d.render_multi([0, 1], spp=6, seed=13, splits=1)
    assert np.array_equal(two, rep)
    monkeypatch.setenv("LR_MULTI_NO_PEER", "1")                  # the staged-copy path where a peer cannot be mapped
    staged, staged_sq, _ = d.render_multi([0, 1], spp=6, seed=13, splits=1, sumsq=True)
    monkeypatch.delenv("LR_MULTI_NO_PEER")
    assert np.array_equal(staged, two) and np.array_equal(staged_sq, two_sq)
    assert st2["rays"] == st["rays"] and st2["samples"] == st["samples"] and st2["nonfinite_samples"] == st["nonfinite_samples"]
    assert np.allclose(two, ref, rtol=1e-5, atol=1e-6) and np.allclose(two_sq, ref_sq, rtol=1e-5, atol=1e-6)
    # the ranges are the ones a 2-rank run renders: [0, 3) and [3, 6)
    lo, _, _ = s.render(spp=3, spp_begin=0, seed=13, splits=1)
    hi, _, _ = s.render(spp=3, spp_begin=3, seed=13, splits=1)
    assert np.allclose(two, (lo + hi) / 2, rtol=1e-6, atol=1e-7)
    # more devices than samples: the idle device contributes zeros
    few, _, stf = d.render_multi([1, 0], spp=1, seed=13, splits=1)
    solo, _, sts = s.render(spp=1, seed=13, splits=1)
    assert np.array_equal(few, solo) and stf["rays"] == sts["rays"]
    # a scene stays on the device it was created on, whichever device the calling thread makes current afterwards
    lr.init(1)
    s1 = d.scene()                                              # lives on device 1
    on1, _, st_on1 = s1.render(spp=6, seed=13, splits=1)
    lr.init(0)
    again1, _, _ = s1.render(spp=6, seed=13, splits=1)          # called with device 0 current: runs on device 1
    depth1 = s1.render_aov("depth", spp=1, seed=13)
    film1 = s1.film(seed=13, splits=1)
    film1.render(6)
    assert np.array_equal(on1, ref) and np.array_equal(again1, ref) and st_on1["rays"] == st["rays"]
    assert np.array_equal(film1.read(), ref) and np.array_equal(depth1, s.render_aov("depth", spp=1, seed=13))
    film1.close()
    s1.close()
    still, _, _ = s.render(spp=6, seed=13, splits=1)            # the device-0 scene is untouched by all that
    assert np.array_equal(still, ref)
    # the handle form (scenes, streams, peer mappings set up once): same bits as the one-shot call, call after call
    ms = d.multi_scene([0, 1])
    for _ in range(3):
        h, h_sq, sth = ms.render(spp=6, seed=13, splits=1, sumsq=True)
        assert np.array_equal(h, two) and np.array_equal(h_sq, two_sq) and sth["rays"] == st["rays"]
    hc, _, _ = ms.render(spp=6, seed=13, splits=1, crop=(37, 21, 50, 33))
    assert np.array_equal(hc, two[21:21 + 33, 37:37 + 50])
    ms.close()


@pytest.mark.parametrize("sphere_light", [0.0, 8.0])
@pytest.mark.parametrize("integrator,with_mesh", [(0, False), (1, False), (0, True), (1, True)])
def test_direct_lighting_matches_the_point_to_rectangle_form_factor(lr, gpu, integrator, with_mesh, sphere_light):
    """The closed-form check of tests/test_oracle_known_answers.py on the CUDA path: a floor point under a rectangular
    emitter reflects albedo * L_e * F(point -> rectangle), for pt (BSDF sampling finds the light) and pt-direct (light
    sampling).  with_mesh puts a BVH into the scene: pt then runs the pool kernel, pt-direct the deferred-traversal one."""
    from conftest import form_factor_scene
    d, exact = form_factor_scene(lr, with_mesh=with_mesh, sphere_light=sphere_light)   # 8.0: spherical emitter, F = (r / h)^2
    assert (d.desc.contents.n_nodes > 0) == with_mesh
    s = d.scene()
    prim, t = s.trace_primary()
    assert set(np.unique(prim)) <= {0, 1}, "the camera must look at the floor"
    spp = (16384 if integrator == 1 else 65536) * (4 if sphere_light > 0 else 1)
    img, sq, st = s.render(integrator=integrator, spp=spp, seed=3, depth=5, depth_limit=64, no_direct_emitter=0, sumsq=True)
    n = spp * img.shape[0] * img.shape[1]
    mean = img.mean(axis=(0, 1), dtype=np.float64)
    var = sq.sum(axis=(0, 1), dtype=np.float64) / n - mean ** 2
    se = np.sqrt(np.maximum(var, 0.0) / n)
    assert st["nonfinite_samples"] == 0
    assert np.all(np.abs(mean - exact) <= 4.0 * se + 2e-4 * exact), (mean, exact, se)
    assert np.all(se < 0.005 * exact)


@pytest.mark.parametrize("kind", ["thin-lens", "pinhole"])
def test_lens_cameras_image_a_uniform_sky_as_cos4(lr, gpu, kind):
    """The radiometric camera pin of tests/test_oracle_known_answers.py on the CUDA path: a radiance-1 sky through the
    thin-lens / realistic-pinhole camera is the cos^4 vignetting averaged over pixel and aperture."""
    from conftest import lens_cos4_case
    d, expect = lens_cos4_case(lr, kind)
    s = d.scene()
    spp = 200000
    img, sq, st = s.render(integrator=0, spp=spp, seed=5, depth=5, depth_limit=64, no_direct_emitter=0, sumsq=True)
    mean = img[..., 0].astype(np.float64)
    se = np.sqrt(np.maximum(sq[..., 0].astype(np.float64) / spp - mean ** 2, 0.0) / spp)
    assert st["nonfinite_samples"] == 0
    assert np.all(np.abs(mean - expect) <= 4.5 * se + 2e-3 * expect), float(np.abs(mean - expect).max())


def test_error_paths(scenes, lr):
    from lumillyrender_b200.capi import LumillyError
    d, s, o = scenes("primitive")
    with pytest.raises(LumillyError):
        s.render(spp=0)
    with pytest.raises(LumillyError):
        s.render(spp=1, crop=(0, 0, 100000, 4))
    with pytest.raises(LumillyError):
        s.render(spp=1, integrator=7)


def test_counters_instrumented_traversal(scenes):
    d, s, o = scenes("sample")
    a, _, st0 = s.render(spp=2, seed=1, splits=1)
    b, _, st1 = s.render(spp=2, seed=1, splits=1, count=True)
    assert np.array_equal(a, b)
    assert st0["nodes_visited"] == 0 and st1["nodes_visited"] > st1["rays"] and st1["tris_tested"] > 0
    assert st0["rays"] == st1["rays"]


def test_gate_retrace_and_flat_list(lr, orc, gpu):
    """Triangles beyond t = 1e5 are invisible in the reference (the AABB line test is clipped to +-1e5, aabb.rs:76-77).
    The render kernel accepts BVH hits optimistically and gates the nearest one once: here the gate must reject it
    and the strict re-trace must answer like the oracle.  A wall-sized triangle exercises the flat list the same way."""
    from lumillyrender_b200 import capi
    rng = np.random.RandomState(3)
    far = (rng.normal(0, 1, (60, 3, 3)) * 2.0e4 + np.array([0, 0, -1.5e5]) + rng.uniform(-6e4, 6e4, (60, 1, 3)) * [1, 1, 0]).astype(np.float32)
    near = _soup(rng, 40, scale=6.0, size=1.5)
    wall = np.array([[[-3e5, -3e5, -2.0e5], [3e5, -3e5, -2.0e5], [0, 4e5, -2.0e5]]], dtype=np.float32)    # large: goes to the flat list
    tri = np.concatenate([near, far, wall])
    d = _scene_from_tris(lr, tri)
    desc = d.desc.contents
    assert 1 <= desc.n_flat_triangles < len(tri) and desc.n_nodes > 0
    desc.sky.type = capi.LR_SKY_UNIFORM
    desc.sky.color[:] = [1.0, 0.9, 0.8]
    s = d.scene()
    o = orc.OracleScene(d.desc, keepalive=d)
    # nearest hits of rays aimed at the far triangles and the wall: invisible, like the oracle's brute force says
    n = 4000
    org = np.zeros((n, 3), np.float32) + np.array([0, 0, 40], np.float32)
    k = rng.randint(len(near), len(tri), n)
    w = rng.dirichlet([1, 1, 1], n).astype(np.float32)
    dirs = (tri[k] * w[:, :, None]).sum(1) - org
    dirs = (dirs / np.linalg.norm(dirs, axis=1, keepdims=True)).astype(np.float32)
    pg, tg, _ = s.trace_rays(org, dirs, normals=True)
    po, to, _ = o.trace_rays(org, dirs, brute_force=True)
    assert np.array_equal(pg, po) and np.array_equal(tg[po >= 0], to[po >= 0])
    assert (po < len(near)).all(), "nothing beyond t = 1e5 may be hit"
    # the render path: same image as the oracle's replay, and the gate did fire
    img, _, st = s.render(integrator="pt", spp=4, seed=9, splits=1, depth=5, depth_limit=64, no_direct_emitter=0)
    ref_sum, _, ost = o.render(make_params(lr, d.config, integrator=0, spp=4, seed=9, depth=5, depth_limit=64, no_direct_emitter=0),
                               traversal=0, rng_mode=0, math_mode=1)
    assert st["rays"] == ost["rays"]
    assert np.isclose(img, ref_sum / 4, rtol=1e-4, atol=1e-5).all(-1).mean() >= 0.999
    assert st["gate_retraces"] > 0, "the far triangles must have been found optimistically and rejected by the gate"


def test_full_size_properties(lr, assets, gpu):
    """BASELINE configs[4] at its full film size (1920x1370), through properties that do not need the oracle:
    sample-range sharding is exact up to fp32 summation order, ray counts add up, a crop renders the same pixels,
    the render is finite and deterministic."""
    d = load_scene(lr, "sample", (1920, 1370))
    s = d.scene()
    full, _, st = s.render(spp=4, seed=21)
    again, _, _ = s.render(spp=4, seed=21)
    assert np.array_equal(full, again)
    assert full.shape == (1370, 1920, 3) and np.isfinite(full).all() and st["nonfinite_samples"] == 0
    lo, _, st_lo = s.render(spp=2, spp_begin=0, seed=21)
    hi, _, st_hi = s.render(spp=2, spp_begin=2, seed=21)
    assert st_lo["rays"] + st_hi["rays"] == st["rays"]
    assert np.allclose((lo + hi) / 2, full, rtol=1e-5, atol=1e-6)
    crop, _, _ = s.render(spp=4, seed=21, crop=(901, 333, 257, 129))
    assert np.array_equal(crop, full[333:333 + 129, 901:901 + 257])
    assert 0.2 < float(full.mean()) < 0.6 and st["rays"] > 4 * 1920 * 1370 * 3


@pytest.mark.parametrize("name", ["primitive", "sample", "welcome-2018", "vr"])
def test_aovs_match_oracle(scenes, lr, name):
    """Scene::normal / Scene::depth (scene.rs:48-62) over the camera rays of a sample range: the CUDA path against the
    oracle, bit for bit on pixels whose samples all hit the same primitives (every operation is an exact-rounded fp32 one
    applied in the same order; the lens / omnidirectional cameras go through the specified sincos on both sides)."""
    d, s, o = scenes(name)
    for kw in (dict(spp=1, seed=3), dict(spp=5, spp_begin=2, seed=9, crop=(31, 17, 64, 48))):
        p = make_params(lr, d.config, **kw)
        for kind in ("normal", "depth"):
            g = s.render_aov(kind, params=p)
            r = o.render_aov(p, kind)
            assert g.shape == r.shape
            same = (g == r).mean()
            print("%s %s %s: bit-equal on %.6f of the values" % (name, kind, kw, same))
            assert same >= 0.9999 and np.allclose(g, r, rtol=1e-5, atol=1e-6)
    # the AOV of sample 0 with a fixed jitter is the primary probe
    depth = s.render_aov("depth", spp=1, seed=3)
    normal = s.render_aov("normal", spp=1, seed=3)
    assert ((depth > 0) == (normal != 0).any(-1)).all()
    hit = depth > 0
    assert np.allclose(np.linalg.norm(normal[hit] * 2 - 1, axis=-1), 1.0, atol=1e-5)


def test_aov_error_paths(scenes, lr):
    from lumillyrender_b200.capi import LumillyError
    d, s, o = scenes("primitive")
    with pytest.raises(LumillyError):
        s.render_aov(7, spp=1)
    with pytest.raises(LumillyError):
        s.render_aov("depth", spp=0)


@pytest.mark.parametrize("name", ["new-cbox", "sample", "welcome-2018"])
def test_resumable_render_equals_one_pass_bit_for_bit(scenes, lr, name, tmp_path):
    """Progressive / resumable rendering (the hook main.rs:81-91 abandoned): a film rendered as [0,3) + [3,4) + [4,9) — with a
    checkpoint written to disk and restored into a NEW film in between — is bit for bit the image (and sum of squares,
    and ray count) of one lr_render over [0,9): with splits = 1 every pixel's samples are added in sample order starting
    from the stored sum, the fold of main.rs:92-104."""
    d, s, o = scenes(name)
    ref, ref_sq, st = s.render(spp=9, seed=21, splits=1, sumsq=True)
    film = s.film(sumsq=True, seed=21, splits=1)
    rays = film.render(3)["rays"]
    assert film.spp == 3
    part = film.read()
    first, _, _ = s.render(spp=3, seed=21, splits=1)
    assert np.array_equal(part, first, equal_nan=True)
    rays += film.render(1)["rays"]
    ck = str(tmp_path / "film.ck")
    film.save(ck)
    film.close()
    resumed = s.load_film(ck)
    assert resumed.spp == 4 and resumed.has_sumsq
    rays += resumed.render(5)["rays"]
    img, sq = resumed.read(sumsq=True)
    assert resumed.spp == 9 and rays == st["rays"]
    assert np.array_equal(img, ref, equal_nan=True) and np.array_equal(sq, ref_sq, equal_nan=True)
    # a crop film resumes the same way
    crop = (8, 4, 40, 24)
    cf = s.film(seed=21, splits=1, crop=crop)
    cf.render(4)
    cf.save(ck)
    cf2 = s.load_film(ck)
    cf2.render(5)
    assert np.array_equal(cf2.read(), ref[4:28, 8:48], equal_nan=True)


@pytest.mark.parametrize("name", ["new-cbox", "sample"])
def test_film_honours_splits(scenes, name):
    """A film of one scene renders with the splits it was created with, as lr_render does: one call with splits = 4 gives
    lr_render's image, sums of squares and ray count bit for bit."""
    d, s, o = scenes(name)
    ref, ref_sq, st = s.render(spp=8, seed=9, splits=4, sumsq=True)
    film = s.film(sumsq=True, seed=9, splits=4)
    fst = film.render(8)
    img, sq = film.read(sumsq=True)
    film.close()
    assert st["splits"] == 4 and fst["splits"] == 4 and fst["rays"] == st["rays"] and fst["samples"] == st["samples"]
    assert np.array_equal(img.view(np.uint32), ref.view(np.uint32)) and np.array_equal(sq.view(np.uint32), ref_sq.view(np.uint32))


def test_film_error_paths(scenes, lr, tmp_path):
    from lumillyrender_b200.capi import LumillyError
    d, s, o = scenes("new-cbox")
    film = s.film(seed=1, splits=1)
    with pytest.raises(LumillyError):
        film.read()                                   # no samples yet
    with pytest.raises(LumillyError):
        film.render(0)
    film.render(1)
    with pytest.raises(LumillyError):
        film.read(sumsq=True)                         # created without sums of squares
    with pytest.raises(LumillyError) as e:
        s.load_film(str(tmp_path / "absent.ck"))
    assert e.value.code == -4
    bad = tmp_path / "bad.ck"
    bad.write_bytes(b"not a film checkpoint at all" * 8)
    with pytest.raises(LumillyError) as e:
        s.load_film(str(bad))
    assert e.value.code == -5
    ck = str(tmp_path / "f.ck")
    film.save(ck)
    with open(ck, "rb") as f:
        data = f.read()
    (tmp_path / "short.ck").write_bytes(data[:len(data) // 2])
    with pytest.raises(LumillyError) as e:
        s.load_film(str(tmp_path / "short.ck"))
    assert e.value.code == -5
    d2, s2, _ = scenes("primitive")                    # another film resolution
    with pytest.raises(LumillyError):
        s2.load_film(ck)
