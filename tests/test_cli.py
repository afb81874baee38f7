"""The command line (csrc/cli_main.cpp), which keeps the reference's surface `<binary> scenes/x.toml` (main.rs:43-51) and
its progress lines.  What can be checked without a GPU: argument handling, the reference's messages for a missing
argument / file, the host-side lines printed before the device is touched, and the loud refusal without a device."""
import os
import subprocess

import pytest

from conftest import ROOT


@pytest.fixture(scope="module")
def cli(lr, assets):
    from lumillyrender_b200 import build
    path = build.build_cli()
    assert path and os.path.exists(path)
    return path


def run(cli, *args, cwd=None):
    return subprocess.run([cli, *args], capture_output=True, text=True, cwd=cwd or ROOT, timeout=120)


def test_missing_argument_is_the_reference_message(cli):
    r = run(cli)
    assert r.returncode == 2 and "Path for .toml must be specified." in r.stderr      # main.rs:47-49
    assert r.stdout.startswith("start: ")                                              # main.rs:44


def test_bad_flags_exit_2(cli):
    assert run(cli, "--spp").returncode == 2
    assert run(cli, "scenes/primitive.toml", "--resolution", "banana").returncode == 2
    assert run(cli, "scenes/primitive.toml", "extra.toml").returncode == 2
    assert run(cli, "scenes/primitive.toml", "--aov", "albedo").returncode == 2
    assert run(cli, "scenes/primitive.toml", "--checkpoint", "x.ck").returncode == 2          # needs --progress


def test_missing_scene_file_is_an_error_not_a_crash(cli):
    r = run(cli, "scenes/does-not-exist.toml")
    assert r.returncode == 1 and "is not found" in r.stderr                           # description.rs:34
    assert "loading: scenes/does-not-exist.toml" in r.stdout


def test_host_side_lines_then_loud_refusal_without_a_gpu(cli):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    r = run(cli, "scenes/primitive.toml", "--spp", "2", "--resolution", "32x32")
    assert r.returncode == 1
    assert "resolution: 32x32" in r.stdout and "spp: 2" in r.stdout                   # main.rs:52-59, printed before the device is touched
    assert "no CPU fallback" in r.stderr


@pytest.mark.gpu
def test_cli_renders_and_writes_the_image(cli, tmp_path):
    r = run(cli, os.path.join(ROOT, "scenes", "primitive.toml"), "--spp", "4", "--resolution", "64x64", "--assets", ROOT, cwd=str(tmp_path))
    assert r.returncode == 0, r.stderr
    for line in ("start: ", "loading: ", "resolution: 64x64", "spp: 4", "integrator: pt", "polygons: ", "bvh construction: ", "saving...", "end: ", "elapse: "):
        assert line in r.stdout, line
    files = os.listdir(os.path.join(str(tmp_path), "images"))
    assert len(files) == 1 and files[0].startswith("image_") and files[0].endswith("_4.png")   # main.rs:147-169


@pytest.mark.gpu
def test_cli_progress_checkpoint_resume_and_aov(cli, tmp_path):
    """--progress renders in chunks through a film on the devices of --gpus (here one) and prints the reference's abandoned progress line (main.rs:81-91);
    an interrupted run (here: a first run asked for 4 of the 8 spp) resumed from its checkpoint writes byte for byte the
    PNG of an uninterrupted one; --aov writes Scene::normal / Scene::depth (scene.rs:48-62)."""
    scene = os.path.join(ROOT, "scenes", "primitive.toml")
    common = ("--resolution", "64x64", "--assets", ROOT, "--seed", "3")

    def png(d):
        files = sorted(os.listdir(os.path.join(d, "images")))
        with open(os.path.join(d, "images", files[-1]), "rb") as f:
            return f.read()
    a, b = tmp_path / "a", tmp_path / "b"
    a.mkdir(); b.mkdir()
    r = run(cli, scene, "--spp", "8", "--progress", "3", *common, cwd=str(a))
    assert r.returncode == 0 and "processing... (8/8 : 100%)" in r.stdout, r.stderr
    ck = str(b / "film.ck")
    r = run(cli, scene, "--spp", "4", "--progress", "4", "--checkpoint", ck, *common, cwd=str(b))
    assert r.returncode == 0 and os.path.exists(ck), r.stderr
    for f in os.listdir(str(b / "images")):
        os.remove(str(b / "images" / f))
    r = run(cli, scene, "--spp", "8", "--progress", "2", "--checkpoint", ck, *common, cwd=str(b))
    assert r.returncode == 0 and "resuming: 4 of 8 spp" in r.stdout, r.stderr
    assert png(str(a)) == png(str(b))
    for kind in ("normal", "depth"):
        c = tmp_path / kind
        c.mkdir()
        r = run(cli, scene, "--spp", "2", "--aov", kind, *common, cwd=str(c))
        assert r.returncode == 0 and ("aov: " + kind) in r.stdout, r.stderr
        assert len(png(str(c))) > 100
