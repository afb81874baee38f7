"""What a pixel-sharded film (lr_multi_film_*) delivers on the bench workload: sample.toml at 1920x1370 with the 144,046-
triangle mesh, 1024 spp rendered in chunks of 64 with a checkpoint written after every chunk, on 1 / 2 / 4 / 8 GPUs as
the box has them, against lr_multi_render (samples sharded by index) of the same 1024 spp on the same devices.
Prints, per device count: multi-film Msamples/s (render calls only, and with the checkpoints), the per-chunk wall time,
the gather + save time per checkpoint, lr_multi_render's Msamples/s, and whether the image equals the 1-GPU film's bits.
usage (GPU box): python tools/multi_film_probe.py [spp_total] [chunk] [n_max]"""
import os, statistics, sys, tempfile, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch
import lumillyrender_b200 as lr

spp = int(sys.argv[1]) if len(sys.argv) > 1 else 1024
chunk = int(sys.argv[2]) if len(sys.argv) > 2 else 64
n_max = int(sys.argv[3]) if len(sys.argv) > 3 else min(8, torch.cuda.device_count())
if n_max < 1:
    sys.exit("no CUDA device: this probe measures the GPU path only")
lr.init(0)
print("device:", lr.device_info(), flush=True)
lr.ensure_assets(ROOT, bunny_tris=144046, need_ibl=False)
d = lr.Description(os.path.join(ROOT, "scenes", "sample.toml"), asset_root=ROOT, resolution=(1920, 1370))
tmp = tempfile.mkdtemp(prefix="multi_film_probe_")
ck = os.path.join(tmp, "film.ck")
ref = None
n = 1
try:
    while n <= n_max:
        ms = d.multi_scene(list(range(n)))
        ms.render(spp=chunk, seed=1)                         # warm-up: modules, pools, peer mappings
        warm = ms.film(seed=1, splits=1)
        warm.render(chunk)
        warm.save(ck)
        warm.close()
        # lr_multi_render: the same 1024 spp in one call
        t0 = time.perf_counter()
        _, _, mst = ms.render(spp=spp, seed=0, splits=1)
        multi_wall = time.perf_counter() - t0
        # the film: chunks of `chunk` spp, a checkpoint after each
        film = ms.film(seed=0, splits=1)
        chunks, saves, samples = [], [], 0
        for _ in range(spp // chunk):
            t0 = time.perf_counter()
            st = film.render(chunk)
            chunks.append(time.perf_counter() - t0)
            samples += st["samples"]
            t0 = time.perf_counter()
            film.save(ck)
            saves.append(time.perf_counter() - t0)
        img = film.read()
        film.close()
        ms.close()
        if ref is None:
            ref = img
        same = np.array_equal(img.view(np.uint32), ref.view(np.uint32))
        render_s, total_s = sum(chunks), sum(chunks) + sum(saves)
        print("N=%d spp=%d: multi film %.0f Msamples/s in render calls, %.0f with a checkpoint per %d spp | chunk wall min %.1f / median %.1f / "
              "max %.1f ms | gather + save min %.1f / median %.1f / max %.1f ms | lr_multi_render %.0f Msamples/s (wall %.1f ms, slowest kernel "
              "%.1f ms) | film / lr_multi_render %.3f | image bits equal to N=1: %s"
              % (n, spp, samples / render_s / 1e6, samples / total_s / 1e6, chunk, min(chunks) * 1e3, statistics.median(chunks) * 1e3,
                 max(chunks) * 1e3, min(saves) * 1e3, statistics.median(saves) * 1e3, max(saves) * 1e3, mst["samples"] / multi_wall / 1e6,
                 multi_wall * 1e3, mst["kernel_ms"], (samples / render_s) / (mst["samples"] / multi_wall), same), flush=True)
        n *= 2
finally:
    for f in os.listdir(tmp):
        os.remove(os.path.join(tmp, f))
    os.rmdir(tmp)
