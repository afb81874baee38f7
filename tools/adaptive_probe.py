"""What adaptive sampling buys on a full-size film: a uniform film and an adaptive film (lr_film_render_adaptive) of the same
scene, against a high-spp uniform reference of another seed.  Per round: samples and kernel time so far, RMSE against the
reference, the largest tile error (the rule of device_scene.h, restated in float64 from a checkpoint's raw sums), and for the
adaptive film the tiles selected, the render's Msamples/s, Mrays/s and rays per sample (the tiles left are the hard ones, so
Msamples/s alone mixes longer paths with lower occupancy) and the selection kernels' time (select_tiles_kernel +
compact_tiles_kernel, from torch.profiler in a second, identical pass; the selection is deterministic).
usage: python tools/adaptive_probe.py [--scenes sample,welcome-2018] [--ref-spp 1024] [--round 4] [--max-spp 64] [--threshold 0.05]"""
import argparse
import os
import sys
import tempfile
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import lumillyrender_b200 as lr                                        # noqa: E402
from lumillyrender_b200.film_checkpoint import read_checkpoint, tile_errors   # noqa: E402


def max_tile_error(film, ck):
    film.save(ck)
    _, _, s, q, counts = read_checkpoint(ck)
    err, finite = tile_errors(s, q, counts)
    return float(err[finite & (counts >= 2)].max())


def rmse(img, ref):
    return float(np.sqrt(np.mean((img.astype(np.float64) - ref) ** 2)))


def select_ms(prof):
    return sum(e.device_time_total for e in prof.key_averages()
               if "select_tiles_kernel" in e.key or "compact_tiles_kernel" in e.key) / 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenes", default="sample,welcome-2018")
    ap.add_argument("--ref-spp", type=int, default=1024)
    ap.add_argument("--round", type=int, default=4)
    ap.add_argument("--max-spp", type=int, default=64)
    ap.add_argument("--threshold", type=float, default=0.05)
    a = ap.parse_args()
    lr.init(0)
    lr.ensure_assets(ROOT, bunny_tris=144046, ibl_height=1600)
    print(lr.device_info())
    ck = os.path.join(tempfile.mkdtemp(), "probe.ck")
    for name in a.scenes.split(","):
        d = lr.Description(os.path.join(ROOT, "scenes", name + ".toml"), asset_root=ROOT)
        s = d.scene()
        ref = np.zeros((s.height, s.width, 3))
        for k in range(0, a.ref_spp, 64):                                   # independent of the films' seed
            img, _, _ = s.render(spp=min(64, a.ref_spp - k), spp_begin=k, seed=999)
            ref += img.astype(np.float64) * min(64, a.ref_spp - k)
        ref /= a.ref_spp
        n_tiles = ((s.width + 7) // 8) * ((s.height + 3) // 4)
        print("== %s %dx%d, %d tiles; reference %d spp (seed 999); rounds of %d spp, max %d spp, threshold %g"
              % (name, s.width, s.height, n_tiles, a.ref_spp, a.round, a.max_spp, a.threshold))

        uni = []
        film = s.film(sumsq=True, seed=1, splits=1)
        samples, ms = 0, 0.0
        while film.spp < a.max_spp:
            st = film.render(a.round)
            samples += st["samples"]; ms += st["kernel_ms"]
            uni.append((film.spp, samples, ms, rmse(film.read(), ref), max_tile_error(film, ck), st["rays"] / st["kernel_ms"] / 1e3))
        film.close()
        neg = (read_checkpoint(ck)[2] < 0).any(axis=2)
        print("uniform film at %d spp: %d pixels hold a negative sum (per-sample estimates below zero)" % (uni[-1][0], int(neg.sum())))
        print("uniform: spp | Msamples | kernel ms | RMSE | max tile error | render Mrays/s")
        for r in uni:
            print("  %3d | %9.1f | %9.2f | %.6f | %.4f | %8.1f" % (r[0], r[1] / 1e6, r[2], r[3], r[4], r[5]))

        ada = []
        film = s.film(sumsq=True, seed=1, splits=1)
        samples, ms = 0, 0.0
        while True:
            st = film.render_adaptive(a.round, a.threshold, max_spp=a.max_spp)
            if st["active_tiles"] == 0:
                break
            samples += st["samples"]; ms += st["kernel_ms"]
            ada.append((st["active_tiles"], st["samples"] / st["kernel_ms"] / 1e3, samples, ms, rmse(film.read(), ref),
                        max_tile_error(film, ck), float(film.spp_map().mean()), st["rays"] / st["kernel_ms"] / 1e3,
                        st["rays"] / st["samples"]))
        film.close()
        sel = [float("nan")] * (len(ada) + 1)
        try:
            import torch
            from torch.profiler import ProfilerActivity, profile
            warnings.filterwarnings("ignore", message=".*Profiler clears events")   # one profile per round, by design
            film = s.film(sumsq=True, seed=1, splits=1)
            for i in range(len(ada) + 1):
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    film.render_adaptive(a.round, a.threshold, max_spp=a.max_spp)
                torch.cuda.synchronize()
                sel[i] = select_ms(prof)
            film.close()
        except Exception as e:                                              # the rest of the report stands without it
            print("selection timing unavailable: %r" % (e,))
        print("adaptive: round | tiles | select ms | render Msamples/s | render Mrays/s | rays/sample | Msamples | kernel ms | RMSE"
              " | max tile error | mean spp")
        for i, r in enumerate(ada):
            print("  %3d | %6d | %8.3f | %8.1f | %8.1f | %6.3f | %9.1f | %9.2f | %.6f | %.4f | %.2f"
                  % (i + 1, r[0], sel[i], r[1], r[7], r[8], r[2] / 1e6, r[3], r[4], r[5], r[6]))

        # equal total samples / equal kernel time: the last uniform round that does not exceed the adaptive film's totals
        if ada:
            a_samples, a_ms, a_rmse = ada[-1][2], ada[-1][3], ada[-1][4]
            eq_s = [u for u in uni if u[1] <= a_samples]
            eq_t = [u for u in uni if u[2] <= a_ms]
            print("adaptive, converged: %.1f Msamples, %.2f ms, RMSE %.6f" % (a_samples / 1e6, a_ms, a_rmse))
            if eq_s:
                print("uniform at <= equal samples: %d spp, %.1f Msamples, RMSE %.6f" % (eq_s[-1][0], eq_s[-1][1] / 1e6, eq_s[-1][3]))
            if eq_t:
                print("uniform at <= equal kernel time: %d spp, %.2f ms, RMSE %.6f" % (eq_t[-1][0], eq_t[-1][2], eq_t[-1][3]))
        for target in (0.2, 0.1, a.threshold):
            u = next((r for r in uni if r[4] <= target), None)
            v = next((r for r in ada if r[5] <= target), None)
            print("max tile error <= %g: uniform %s, adaptive %s" % (
                target, "%.2f ms (%d spp)" % (u[2], u[0]) if u else "not reached by %d spp" % a.max_spp,
                "%.2f ms (round %d)" % (v[3], ada.index(v) + 1) if v else "not reached (tiles capped at %d spp)" % a.max_spp))
        s.close()


if __name__ == "__main__":
    main()
