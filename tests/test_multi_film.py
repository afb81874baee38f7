"""Progressive, resumable rendering on several GPUs (lr_multi_film_*): the film's 8x4 pixel tiles are dealt round-robin over
shards, each pixel's samples are added in sample order on the one device that owns it, and the image is gathered pixel by
pixel on the first device.  So a multi film is bit for bit lr_render with splits = 1 for any device count and any shard
count (LR_FILM_SHARDS cuts one device's film into several shards), and its checkpoints are those of lr_film_*."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, load_scene

RES = {"sample": (160, 160), "welcome-2018": (214, 154), "new-cbox": (128, 128), "vr": (128, 128), "primitive": (256, 256)}


@pytest.fixture(scope="module")
def scenes(lr, assets, gpu):
    cache = {}

    def get(name):
        if name not in cache:
            d = load_scene(lr, name, RES[name])
            cache[name] = (d, d.scene(), d.multi_scene([0]))
        return cache[name]
    yield get
    for d, s, ms in cache.values():
        ms.close()
        s.close()


def bits_equal(a, b):
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["sample", "welcome-2018", "new-cbox", "vr"])
def test_one_device_equals_the_film(scenes, name, tmp_path):
    d, s, ms = scenes(name)
    ref, ref_sq, st = s.render(spp=9, seed=21, splits=1, sumsq=True)
    film = ms.film(sumsq=True, seed=21, splits=1)
    rays = film.render(3)["rays"]
    first, _, _ = s.render(spp=3, seed=21, splits=1)
    assert film.spp == 3 and bits_equal(film.read(), first)
    rays += film.render(1)["rays"]
    ck = str(tmp_path / "film.ck")
    film.save(ck)
    film.close()
    resumed = ms.load_film(ck)
    assert resumed.spp == 4 and resumed.has_sumsq
    rays += resumed.render(5)["rays"]
    img, sq = resumed.read(sumsq=True)
    resumed.close()
    assert rays == st["rays"]
    assert bits_equal(img, ref) and bits_equal(sq, ref_sq)


def crops(w, h):
    # single pixels, a row, a column, and a crop with fewer tiles (3) than most shard counts
    return ((0, 0, 1, 1), (w - 1, h - 1, 1, 1), (3, h // 2, w - 3, 1), (w // 2, 0, 1, h), (5, 6, 7, 9))


@pytest.mark.gpu
@pytest.mark.parametrize("shards", [2, 3, 8])
@pytest.mark.parametrize("name,org", [("sample", "persistent"), ("sample", "pool"), ("welcome-2018", "persistent"),
                                      ("welcome-2018", "pool"), ("new-cbox", None)])
def test_sharded_on_one_device(scenes, monkeypatch, name, org, shards):
    d, s, ms = scenes(name)
    if org:
        monkeypatch.setenv("LR_ORGANISATION", org)
    monkeypatch.setenv("LR_FILM_SHARDS", str(shards))
    ref, ref_sq, st = s.render(spp=4, seed=5, splits=1, sumsq=True)
    film = ms.film(sumsq=True, seed=5, splits=1)
    fst = film.render(4)
    img, sq = film.read(sumsq=True)
    film.close()
    assert bits_equal(img, ref) and bits_equal(sq, ref_sq)
    assert fst["rays"] == st["rays"] and fst["nonfinite_samples"] == st["nonfinite_samples"]
    assert fst["samples"] == st["samples"] and fst["splits"] == 1
    for crop in crops(s.width, s.height):
        x, y, w, h = crop
        c_ref, _, cst = s.render(spp=3, seed=5, splits=1, crop=crop)
        cf = ms.film(seed=5, splits=1, crop=crop)
        cfs = cf.render(2)
        cfs2 = cf.render(1)
        c = cf.read()
        cf.close()
        assert c.shape == (h, w, 3) and bits_equal(c, c_ref), crop
        assert cfs["rays"] + cfs2["rays"] == cst["rays"], crop
        assert cfs["nonfinite_samples"] + cfs2["nonfinite_samples"] == cst["nonfinite_samples"], crop
        assert cfs["samples"] == w * h * 2, crop


@pytest.mark.gpu
@pytest.mark.parametrize("crop", [None, (8, 4, 40, 24)])
def test_checkpoints_move_between_device_counts(scenes, monkeypatch, crop, tmp_path):
    d, s, ms = scenes("sample")
    kw = dict(seed=17, splits=1, crop=crop)
    ref, ref_sq, st = s.render(spp=9, sumsq=True, **kw)
    # a 3-shard multi film, resumed by a single-device film
    monkeypatch.setenv("LR_FILM_SHARDS", "3")
    mf = ms.film(sumsq=True, **kw)
    mf.render(4)
    multi_ck = str(tmp_path / "multi.ck")
    mf.save(multi_ck)
    mf.close()
    monkeypatch.delenv("LR_FILM_SHARDS")
    f = s.load_film(multi_ck)
    assert f.spp == 4 and f.has_sumsq
    f.render(5)
    img, sq = f.read(sumsq=True)
    f.close()
    assert bits_equal(img, ref) and bits_equal(sq, ref_sq)
    # a single-device film, resumed by a 5-shard multi film
    sf = s.film(sumsq=True, **kw)
    sf.render(4)
    single_ck = str(tmp_path / "single.ck")
    sf.save(single_ck)
    sf.close()
    monkeypatch.setenv("LR_FILM_SHARDS", "5")
    mf = ms.load_film(single_ck)
    assert mf.spp == 4 and mf.has_sumsq
    resaved = str(tmp_path / "resaved.ck")
    mf.save(resaved)
    mf.render(5)
    img, sq = mf.read(sumsq=True)
    mf.close()
    assert bits_equal(img, ref) and bits_equal(sq, ref_sq)
    # one checkpoint format: the same state saves to the same bytes through either kind of film
    with open(multi_ck, "rb") as a, open(single_ck, "rb") as b, open(resaved, "rb") as c:
        ma, sb, rc = a.read(), b.read(), c.read()
    assert ma == sb and rc == sb


@pytest.mark.gpu
def test_error_paths(scenes, lr, tmp_path):
    from lumillyrender_b200.capi import LumillyError
    d, s, ms = scenes("new-cbox")
    ref, _, _ = s.render(spp=2, seed=1, splits=1)
    with pytest.raises(LumillyError) as e:
        ms.film(seed=1, splits=2)
    assert e.value.code == -1
    film = ms.film(seed=1, splits=1)
    with pytest.raises(LumillyError) as e:
        film.read()                                   # no samples yet
    assert e.value.code == -1
    with pytest.raises(LumillyError) as e:
        film.render(0)
    assert e.value.code == -1
    film.render(1)
    with pytest.raises(LumillyError) as e:
        film.read(sumsq=True)                         # created without sums of squares
    assert e.value.code == -1
    ck = str(tmp_path / "f.ck")
    film.save(ck)
    film.close()
    _, s_other, ms_other = scenes("primitive")        # another film resolution
    with pytest.raises(LumillyError) as e:
        ms_other.load_film(ck)
    assert e.value.code == -1
    split_film = s.film(seed=1, splits=2)             # a single-device checkpoint with splits = 2 in its header
    split_film.render(2)
    split_ck = str(tmp_path / "split.ck")
    split_film.save(split_ck)
    split_film.close()
    with pytest.raises(LumillyError) as e:
        ms.load_film(split_ck)
    assert e.value.code == -1
    with pytest.raises(LumillyError) as e:
        ms.load_film(str(tmp_path / "absent.ck"))
    assert e.value.code == -4
    bad = tmp_path / "bad.ck"
    bad.write_bytes(b"not a film checkpoint at all" * 8)
    with pytest.raises(LumillyError) as e:
        ms.load_film(str(bad))
    assert e.value.code == -5
    with open(ck, "rb") as f:
        data = f.read()
    (tmp_path / "short.ck").write_bytes(data[:len(data) // 2])
    with pytest.raises(LumillyError) as e:
        ms.load_film(str(tmp_path / "short.ck"))
    assert e.value.code == -5
    # the library still renders correctly on device 0, through both paths
    again, _, _ = s.render(spp=2, seed=1, splits=1)
    film = ms.film(seed=1, splits=1)
    film.render(2)
    assert bits_equal(again, ref) and bits_equal(film.read(), ref)
    film.close()


def device_count():
    torch = pytest.importorskip("torch")
    return torch.cuda.device_count()


@pytest.mark.gpu
@pytest.mark.parametrize("no_peer", [False, True])
def test_two_or_more_devices(scenes, lr, monkeypatch, no_peer, tmp_path):
    n = device_count()
    if n < 2:
        pytest.skip("needs 2 GPUs")
    d, s, _ = scenes("sample")
    if no_peer:
        monkeypatch.setenv("LR_MULTI_NO_PEER", "1")   # the staged-copy path where a peer cannot be mapped
    ref, ref_sq, st = s.render(spp=9, seed=29, splits=1, sumsq=True)
    for devices in sorted({(0, 1), tuple(range(min(n, 8)))}):
        ms = d.multi_scene(list(devices))
        film = ms.film(sumsq=True, seed=29, splits=1)
        rays = film.render(4)["rays"]
        ck = str(tmp_path / "multi.ck")
        film.save(ck)
        film.close()
        resumed = ms.load_film(ck)
        fst = resumed.render(5)
        img, sq = resumed.read(sumsq=True)
        resumed.close()
        ms.close()
        assert bits_equal(img, ref) and bits_equal(sq, ref_sq), devices
        assert rays + fst["rays"] == st["rays"] and fst["samples"] == s.width * s.height * 5, devices
        # the checkpoint of several devices resumes on one
        one = s.load_film(ck)
        one.render(5)
        assert bits_equal(one.read(), ref), devices
        one.close()


@pytest.mark.gpu
def test_multi_device_calls_keep_the_callers_device(scenes, lr, tmp_path):
    """Calls on a multi scene switch devices as they work, then give the calling thread its device back and leave the
    library's device (lr_init) alone: after them a new scene still lands on the device the caller chose."""
    torch = pytest.importorskip("torch")
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    _, _, ms = scenes("sample")                       # the multi scene lives on [0]
    ck = str(tmp_path / "film.ck")
    lr.init(1)
    try:
        def still_on_1(after):
            assert torch.cuda.current_device() == 1, after
        ms.render(spp=1, seed=3)
        still_on_1("render")
        film = ms.film(seed=3, splits=1)
        still_on_1("film create")
        film.render(1)
        still_on_1("film render")
        film.read()
        still_on_1("film read")
        film.save(ck)
        still_on_1("film save")
        film.close()
        ms.load_film(ck).close()
        still_on_1("film load")
        # the pool never trims, so device 1's free memory shows where a new scene and its film buffers go: two buffers of
        # 126 MB at 3840x2740, more than the earlier tests left in device 1's pool
        w, h = 3840, 2740
        big = load_scene(lr, "new-cbox", (w, h))
        free = torch.cuda.mem_get_info(1)[0]
        s1 = big.scene()
        s1.render(spp=1, seed=3, sumsq=True)
        assert free - torch.cuda.mem_get_info(1)[0] >= w * h * 3 * 4
        still_on_1("a render of a new scene")
        s1.close()
    finally:
        lr.init(0)


@pytest.fixture(scope="module")
def cli(lr, assets):
    from lumillyrender_b200 import build
    path = build.build_cli()
    assert path and os.path.exists(path)
    return path


def run(cli, *args, cwd=None):
    return subprocess.run([cli, *args], capture_output=True, text=True, cwd=cwd or ROOT, timeout=300)


def test_cli_accepts_gpus_with_progress_then_refuses_without_a_gpu(cli):
    torch = pytest.importorskip("torch")
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    r = run(cli, "scenes/primitive.toml", "--spp", "2", "--resolution", "32x32", "--gpus", "2", "--progress", "2")
    assert r.returncode == 1, (r.returncode, r.stderr)
    assert "no CPU fallback" in r.stderr
    assert run(cli, "scenes/primitive.toml", "--gpus", "2", "--aov", "depth").returncode == 2


def test_multi_film_create_rejects_null_arguments(lr):
    lib = lr.load_library()
    out = C.c_void_p()
    assert lib.lr_multi_film_create(None, None, 0, C.byref(out)) == -1
    assert lib.lr_multi_film_load(None, None, C.byref(out)) == -1
    assert lib.lr_multi_film_render(None, 1, None) == -1
    assert lib.lr_multi_film_info(None, None, None, None, None) == -1


@pytest.mark.gpu
def test_cli_gpus_progress_and_resume_write_the_same_png(cli, tmp_path):
    if device_count() < 2:
        pytest.skip("needs 2 GPUs")
    scene = os.path.join(ROOT, "scenes", "primitive.toml")
    common = ("--resolution", "64x64", "--assets", ROOT, "--seed", "3")

    def png(p):
        files = sorted(os.listdir(os.path.join(str(p), "images")))
        with open(os.path.join(str(p), "images", files[-1]), "rb") as f:
            return f.read()
    one, two, res = tmp_path / "one", tmp_path / "two", tmp_path / "resume"
    for p in (one, two, res):
        p.mkdir()
    r = run(cli, scene, "--spp", "8", "--progress", "3", *common, cwd=str(one))
    assert r.returncode == 0, r.stderr
    r = run(cli, scene, "--spp", "8", "--progress", "3", "--gpus", "2", *common, cwd=str(two))
    assert r.returncode == 0 and "processing... (8/8 : 100%)" in r.stdout, r.stderr
    assert png(two) == png(one)
    ck = str(res / "film.ck")
    r = run(cli, scene, "--spp", "4", "--progress", "4", "--gpus", "2", "--checkpoint", ck, *common, cwd=str(res))
    assert r.returncode == 0 and os.path.exists(ck), r.stderr
    for f in os.listdir(str(res / "images")):
        os.remove(str(res / "images" / f))
    r = run(cli, scene, "--spp", "8", "--progress", "2", "--checkpoint", ck, *common, cwd=str(res))
    assert r.returncode == 0 and "resuming: 4 of 8 spp" in r.stdout, r.stderr
    assert png(res) == png(one)
