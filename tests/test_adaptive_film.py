"""Adaptive sampling on films (lr_film_render_adaptive, lr_multi_film_render_adaptive): each 8x4 tile of the crop holds its own
sample count, a round adds samples only to the tiles whose relative standard error is above a threshold, and every tile
continues from its own count with one thread per pixel.  So every pixel of an adaptive film is bit for bit lr_render(splits = 1)
at its tile's count, for any device or shard count and across checkpoints.  The selection rule is restated here in numpy
float64 from the raw sums of a checkpoint."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, load_scene
from lumillyrender_b200.film_checkpoint import read_checkpoint, tile_errors

RES = {"sample": (160, 160), "welcome-2018": (214, 154), "new-cbox": (128, 128), "vr": (128, 128)}


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


def restate_selection(s, q, counts, threshold, max_spp):
    err, finite = tile_errors(s, q, counts)
    noisy = (counts < 2) | (finite & (err > np.float64(np.float32(threshold))))
    return noisy & ((max_spp == 0) | (counts < max_spp))


def tile_pixels(cw, ch):
    ty, tx = (ch + 3) // 4, (cw + 7) // 8
    w = np.minimum(8, cw - 8 * np.arange(tx))
    h = np.minimum(4, ch - 4 * np.arange(ty))
    return h[:, None] * w[None, :]


def run_rounds(film, tmp_path, spp, rounds, max_spp, thresholds=None):
    """Adaptive rounds, each checked against the restated rule from the checkpoint saved before it.  The threshold of a round
    is thresholds[i] if given, else the median tile error before it (so the counts end up mixed).  Returns the thresholds
    used and the summed stats."""
    used, rays, samples = [], 0, 0
    ck = str(tmp_path / "round.ck")
    for i in range(rounds):
        film.save(ck)
        _, _, s, q, before = read_checkpoint(ck)
        if thresholds is not None:
            thr = thresholds[i]
        else:
            err, finite = tile_errors(s, q, before)
            ok = finite & (before >= 2)
            thr = float(np.median(err[ok])) if ok.any() else 0.0
        used.append(thr)
        want = restate_selection(s, q, before, thr, max_spp)
        st = film.render_adaptive(spp, thr, max_spp=max_spp)
        assert st["active_tiles"] == int(want.sum()), i
        assert st["samples"] == int(tile_pixels(s.shape[1], s.shape[0])[want].sum()) * spp, i
        film.save(ck)
        after = read_checkpoint(ck)[4]
        assert np.array_equal(after - before, np.where(want, spp, 0)), i
        rays += st["rays"]
        samples += st["samples"]
    return used, rays, samples


def expand(counts, cw, ch):
    return np.repeat(np.repeat(counts, 4, axis=0), 8, axis=1)[:ch, :cw]


@pytest.mark.gpu
@pytest.mark.parametrize("name,org,integrator", [("sample", "persistent", None), ("sample", "pool", None),
                                                 ("welcome-2018", "persistent", None), ("welcome-2018", "pool", None),
                                                 ("new-cbox", None, None), ("vr", None, "pt"), ("vr", None, "pt-direct")])
def test_every_tile_is_lr_render_at_its_count(scenes, monkeypatch, tmp_path, name, org, integrator):
    d, s, ms = scenes(name)
    if org:
        monkeypatch.setenv("LR_ORGANISATION", org)
    kw = dict(seed=11, splits=1, integrator=integrator)
    film = s.film(sumsq=True, **kw)
    run_rounds(film, tmp_path, 2, 4, max_spp=0)
    spp_map = film.spp_map()
    img, sq = film.read(sumsq=True)
    assert film.spp == spp_map.min() >= 2
    ks = np.unique(spp_map)
    assert len(ks) >= 2, ks                           # the median threshold leaves a mix of counts
    for k in ks:
        ref, ref_sq, _ = s.render(spp=int(k), sumsq=True, **kw)
        mask = spp_map == k
        assert bits_equal(img[mask], ref[mask]) and bits_equal(sq[mask], ref_sq[mask]), k
    # a film whose tiles differ renders every tile from its own count
    film.render(1)
    assert np.array_equal(film.spp_map(), spp_map + 1)
    img = film.read()
    for k in ks:
        ref, _, _ = s.render(spp=int(k) + 1, **kw)
        assert bits_equal(img[spp_map == k], ref[spp_map == k]), k
    film.close()


@pytest.mark.gpu
@pytest.mark.parametrize("crop", [(5, 6, 21, 11), (0, 0, 1, 1), (3, 2, 8, 4)])
def test_crops_caps_and_rays(scenes, tmp_path, crop):
    """Partial edge tiles and one-pixel crops, max_spp capping, and the rays of the rounds tile by tile."""
    d, s, ms = scenes("sample")
    kw = dict(seed=3, splits=1, crop=crop)
    film = s.film(sumsq=True, **kw)
    _, rays, _ = run_rounds(film, tmp_path, 3, 4, max_spp=7)
    x0, y0, cw, ch = crop
    counts = read_checkpoint(str(tmp_path / "round.ck"))[4]
    assert counts.max() <= 9 and np.all((counts == 0) | (counts >= 3))   # 7 caps: a tile at 6 gets one more round
    spp_map = film.spp_map()
    assert np.array_equal(spp_map, expand(counts, cw, ch))
    img, sq = film.read(sumsq=True)
    film.close()
    want_rays = 0
    for ty in range(counts.shape[0]):
        for tx in range(counts.shape[1]):
            k = int(counts[ty, tx])
            tile = (x0 + 8 * tx, y0 + 4 * ty, min(8, cw - 8 * tx), min(4, ch - 4 * ty))
            ref, ref_sq, st = s.render(spp=k, seed=3, splits=1, crop=tile, sumsq=True)
            want_rays += st["rays"]
            sl = (slice(4 * ty, 4 * ty + tile[3]), slice(8 * tx, 8 * tx + tile[2]))
            assert bits_equal(img[sl], ref) and bits_equal(sq[sl], ref_sq), (tx, ty)
    assert rays == want_rays


def adaptive_state(film, path):
    film.save(path)
    img, sq = film.read(sumsq=True)
    with open(path, "rb") as f:
        return img, sq, film.spp_map(), f.read()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["sample", "welcome-2018"])
def test_shard_count_does_not_matter(scenes, monkeypatch, tmp_path, name):
    d, s, ms = scenes(name)
    film = s.film(sumsq=True, seed=19, splits=1)
    thresholds, rays, samples = run_rounds(film, tmp_path, 2, 4, max_spp=0)
    ref = adaptive_state(film, str(tmp_path / "single.ck"))
    film.close()
    for shards in (2, 3, 8):
        monkeypatch.setenv("LR_FILM_SHARDS", str(shards))
        mf = ms.film(sumsq=True, seed=19, splits=1)
        _, mrays, msamples = run_rounds(mf, tmp_path, 2, 4, max_spp=0, thresholds=thresholds)
        got = adaptive_state(mf, str(tmp_path / "multi.ck"))
        mf.close()
        assert (mrays, msamples) == (rays, samples), shards
        assert all(bits_equal(a, b) if isinstance(a, np.ndarray) else a == b for a, b in zip(got, ref)), shards


@pytest.mark.gpu
@pytest.mark.parametrize("first", ["single", "multi"])
def test_interrupted_run_resumes_in_the_other_handle(scenes, monkeypatch, tmp_path, first):
    d, s, ms = scenes("sample")
    kw = dict(seed=23, splits=1)
    film = s.film(sumsq=True, **kw)
    thresholds, _, _ = run_rounds(film, tmp_path, 2, 5, max_spp=0)
    whole = adaptive_state(film, str(tmp_path / "whole.ck"))
    film.close()
    assert whole[3][:8] == b"LRFILM2\0"
    monkeypatch.setenv("LR_FILM_SHARDS", "3")
    a = s.film(sumsq=True, **kw) if first == "single" else ms.film(sumsq=True, **kw)
    for t in thresholds[:3]:
        a.render_adaptive(2, t)
    ck = str(tmp_path / "cut.ck")
    a.save(ck)
    a.close()
    with open(ck, "rb") as f:
        assert f.read(8) == b"LRFILM2\0"
    b = ms.load_film(ck) if first == "single" else s.load_film(ck)
    for t in thresholds[3:]:
        b.render_adaptive(2, t)
    got = adaptive_state(b, str(tmp_path / "resumed.ck"))
    b.close()
    assert all(bits_equal(x, y) if isinstance(x, np.ndarray) else x == y for x, y in zip(got, whole))


@pytest.mark.gpu
def test_uniform_adaptive_film_still_saves_lrfilm1(scenes, tmp_path):
    d, s, ms = scenes("new-cbox")
    film = s.film(sumsq=True, seed=2, splits=1)
    assert film.render_adaptive(2, 0.0)["active_tiles"] == ((s.width + 7) // 8) * ((s.height + 3) // 4)
    ck = str(tmp_path / "u.ck")
    film.save(ck)
    plain = s.film(sumsq=True, seed=2, splits=1)
    plain.render(2)
    ck2 = str(tmp_path / "p.ck")
    plain.save(ck2)
    film.close()
    plain.close()
    with open(ck, "rb") as f, open(ck2, "rb") as g:
        assert f.read() == g.read()


def device_count():
    torch = pytest.importorskip("torch")
    return torch.cuda.device_count()


@pytest.mark.gpu
@pytest.mark.parametrize("no_peer", [False, True])
def test_two_or_more_devices(scenes, monkeypatch, tmp_path, no_peer):
    n = device_count()
    if n < 2:
        pytest.skip("needs 2 GPUs")
    d, s, _ = scenes("sample")
    if no_peer:
        monkeypatch.setenv("LR_MULTI_NO_PEER", "1")   # the staged-copy path where a peer cannot be mapped
    film = s.film(sumsq=True, seed=31, splits=1)
    thresholds, rays, _ = run_rounds(film, tmp_path, 2, 3, max_spp=0)
    ref = adaptive_state(film, str(tmp_path / "single.ck"))
    film.close()
    for devices in sorted({(0, 1), tuple(range(min(n, 8)))}):
        ms = d.multi_scene(list(devices))
        mf = ms.film(sumsq=True, seed=31, splits=1)
        _, mrays, _ = run_rounds(mf, tmp_path, 2, 3, max_spp=0, thresholds=thresholds)
        got = adaptive_state(mf, str(tmp_path / "multi.ck"))
        mf.close()
        ms.close()
        assert mrays == rays, devices
        assert all(bits_equal(a, b) if isinstance(a, np.ndarray) else a == b for a, b in zip(got, ref)), devices


@pytest.mark.gpu
def test_invalid_arguments(scenes):
    from lumillyrender_b200.capi import LumillyError
    d, s, ms = scenes("new-cbox")
    no_sq = s.film(seed=1, splits=1)
    with pytest.raises(LumillyError) as e:
        no_sq.render_adaptive(2, 0.1)
    assert e.value.code == -1
    no_sq.close()
    for film in (s.film(sumsq=True, seed=1, splits=1), ms.film(sumsq=True, seed=1, splits=1)):
        for spp, thr, cap in ((0, 0.1, 0), (-1, 0.1, 0), (2, -0.5, 0), (2, float("nan"), 0), (2, 0.1, -1)):
            with pytest.raises(LumillyError) as e:
                film.render_adaptive(spp, thr, max_spp=cap)
            assert e.value.code == -1, (spp, thr, cap)
        assert film.spp == 0 and film.spp_map().max() == 0
        film.close()


def test_adaptive_entry_points_reject_null_handles(lr):
    lib = lr.load_library()
    out = (C.c_int32 * 4)()
    assert lib.lr_film_render_adaptive(None, 1, 0.1, 0, None, None) == -1
    assert lib.lr_multi_film_render_adaptive(None, 1, 0.1, 0, None, None) == -1
    assert lib.lr_film_spp_map(None, out) == -1
    assert lib.lr_multi_film_spp_map(None, out) == -1


@pytest.fixture(scope="module")
def cli(lr):
    from lumillyrender_b200 import build
    path = build.build_cli()
    assert path and os.path.exists(path)
    return path


def run(cli, *args, cwd=None):
    return subprocess.run([cli, *args], capture_output=True, text=True, cwd=cwd or ROOT, timeout=600)


@pytest.mark.parametrize("args,message", [
    (("--adaptive", "0.05"), "--adaptive needs --progress"),
    (("--adaptive", "0.05", "--progress", "4", "--aov", "depth"), "not an AOV"),
    (("--adaptive", "-1", "--progress", "4"), "relative error >= 0"),
    (("--adaptive", "nan", "--progress", "4"), "relative error >= 0"),
    (("--adaptive", "0.1x", "--progress", "4"), "relative error >= 0"),
])
def test_cli_refuses_bad_adaptive_arguments(cli, args, message):
    r = run(cli, "scenes/primitive.toml", *args)
    assert r.returncode == 2 and message in r.stderr, (r.returncode, r.stderr)


@pytest.mark.gpu
def test_cli_adaptive_resume_writes_the_same_png(cli, assets, tmp_path):
    scene = os.path.join(ROOT, "scenes", "new-cbox.toml")
    common = ("--resolution", "64x64", "--assets", ROOT, "--seed", "5", "--progress", "4", "--adaptive", "0.05")

    def png(p):
        files = sorted(os.listdir(os.path.join(str(p), "images")))
        with open(os.path.join(str(p), "images", files[-1]), "rb") as f:
            return f.read()
    whole, res = tmp_path / "whole", tmp_path / "resume"
    for p in (whole, res):
        p.mkdir()
    r = run(cli, scene, "--spp", "16", *common, cwd=str(whole))
    assert r.returncode == 0 and "adaptive round 1:" in r.stdout and "mean" in r.stdout, r.stderr
    ck = str(res / "film.ck")
    r = run(cli, scene, "--spp", "8", "--checkpoint", ck, *common, cwd=str(res))
    assert r.returncode == 0 and os.path.exists(ck), r.stderr
    for f in os.listdir(str(res / "images")):
        os.remove(str(res / "images" / f))
    r = run(cli, scene, "--spp", "16", "--checkpoint", ck, *common, cwd=str(res))
    assert r.returncode == 0 and "resuming:" in r.stdout, r.stderr
    assert png(res) == png(whole)


def test_checkpoint_reader_and_error_rule(tmp_path):
    """film_checkpoint reads an LRFILM2 file and restates the error: one pixel of samples 1 and 3 (S = 4, Q = 10, n = 2) has
    m = 2, var = (10 - 8) / 1 = 2 and error sqrt(2 / 2) / 2 = 0.5; a black pixel has error 0."""
    cw, ch = 9, 5                                     # 2 x 2 tiles, partial on the right and the bottom
    s = np.zeros((ch, cw, 3), np.float32)
    q = np.zeros((ch, cw, 3), np.float32)
    s[4, 8, 1], q[4, 8, 1] = 4.0, 10.0
    counts = np.array([[3, 2], [2, 2]], np.int32)
    from lumillyrender_b200.film_checkpoint import HEADER
    head = HEADER.pack(b"LRFILM2\0", 16, 16, 0, 0, cw, ch, 0, 5, 5, 0, 1, 0, 2, 1, 7)
    path = tmp_path / "t.ck"
    path.write_bytes(head + s.tobytes() + q.tobytes() + counts.tobytes())
    magic, spp_done, s2, q2, c2 = read_checkpoint(str(path))
    assert magic == b"LRFILM2\0" and spp_done == 2 and np.array_equal(c2, counts)
    assert np.array_equal(s2, s) and np.array_equal(q2, q)
    err, finite = tile_errors(s2, q2, c2)
    assert finite.all() and err[1, 1] == 0.5 and err[0, 0] == 0.0
