#!/usr/bin/env python
"""bench.py — headline benchmark of the path-tracing hot path (BASELINE.json metric: Msamples/s, Mrays/s).

Workload (BASELINE.json configs[4], the configuration the multi-GPU metric is quoted on):
  scenes/sample.toml at 1920x1370, pure path tracing, Cornell box + 144,046-triangle synthetic stand-in for the
  absent bunny.obj, ONE render of SPP_TOTAL = 1024 samples per pixel whose sample indices are sharded over the GPUs
  (strong scaling: rank r of N renders indices [r*1024/N, (r+1)*1024/N) of every pixel), per-pixel sums accumulated in
  HBM and ONE NCCL reduce to rank 0.  A "step" is one full pass: render + reduce + normalise.

  python bench.py --gpus N --steps K --warmup W          (N > 1: launched by torchrun, one rank per GPU)
  python bench.py --impl reference ...                   (the CPU restatement of the reference algorithm)
  python bench.py ... --dump-outputs DIR                 (writes the image of the last timed step to DIR/image.npy)

Writes nothing into the source tree: the synthetic scene assets are generated into a temporary directory.
Prints ONE JSON line (rank 0).  `value` is device-timed with the scene resident in HBM; `e2e` goes through
the C ABI with host buffers (scene upload H2D + image D2H inside the timed region).  At N = 1 the line also carries
`configs`: BASELINE configs 1-4 (primitive / new-cbox / brdf / welcome-2018 at 144 k and 1 M triangles) measured in the
same run, each with its roofline fractions and the CPU restatement timed beside it (--no-configs skips them).
"""
import argparse
import json
import os
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True                         # the source tree may be read-only; leave no __pycache__ in it

WIDTH, HEIGHT = 1920, 1370
SPP_TOTAL = 1024                                       # BASELINE.md §4 config 5: 256 / 1024 / 4096
BUNNY_TRIS = 144046
CPU_SAMPLE_SPP = 64                                   # the CPU arm renders 64 of the 1024 sample indices of a pixel subset
SCENE = "sample"
NODE_BYTES, TRI_BYTES, SPHERE_BYTES = 64, 48, 16      # 128-bit loads per visit: 4 / 3 / 1 (DESIGN.md)
# BASELINE.json configs[0..3] (BASELINE.md §4): scene, film, spp, mesh triangles (0: the scene has no mesh asset)
CONFIGS = [
    ("1 primitive", "primitive", (2048, 2048), 16, 0),
    ("2 new-cbox", "new-cbox", (256, 256), 64, 0),
    ("3 brdf", "brdf", (960, 540), 64, 0),
    ("4 welcome-2018 (144k)", "welcome-2018", (2138, 1536), 64, 144046),
    ("4 welcome-2018 (1M)", "welcome-2018", (2138, 1536), 64, 1048576),
]


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons during the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz, self.stop_flag = index, [], set(), None, False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if mask & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.05)

    def result(self):
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def oracle_sample(desc_owner, params_fn, spp, target_seconds=12.0, size=(WIDTH, HEIGHT)):
    """Times the CPU restatement (faithful reference algorithm, all host threads) on a bounded pixel-strided
    sample of the same workload.  Returns (Msamples/s, Mrays/s, stats, description of the sample)."""
    from oracle import oracle_py as orc
    o = orc.OracleScene(desc_owner.desc, keepalive=desc_owner)
    cores = os.cpu_count() or 1
    w, h = size
    # calibrate on a coarse stride, then pick the stride that gives ~target_seconds of wall time
    _, _, st = o.render(params_fn(spp=spp), traversal=0, rng_mode=1, math_mode=0, threads=cores, pixel_stride=16, sumsq=False)
    per_sample = max(st["render_seconds"], 1e-4) / max(st["samples"], 1)
    stride = 16
    for cand in (1, 2, 3, 4, 6, 8, 12, 16):
        n = ((w + cand - 1) // cand) * ((h + cand - 1) // cand) * spp
        if n * per_sample <= target_seconds:
            stride = cand
            break
    p = params_fn(spp=spp)
    _, _, st = o.render(p, traversal=0, rng_mode=1, math_mode=0, threads=cores, pixel_stride=stride, sumsq=False)
    sec = st["render_seconds"]
    desc = "every %d-th pixel in x and y of the %dx%d film (%d pixels) at %d spp, faithful unordered BVH traversal" % (
        stride, w, h, st["samples"] // spp, spp)
    o.close()
    return st["samples"] / sec / 1e6, st["rays"] / sec / 1e6, st, desc, cores


def reference_traversal(st):
    """What the reference's own traversal costs per ray (SURVEY.md §8d, 'for context'): bvh.rs:131-141 visits every node
    whose box the ray's LINE hits, unordered and unpruned, then fully tests every candidate leaf.  Counters of the
    restatement; bytes at the reference's sizes (AABB 36 B per node visited, aabb.rs:10-14; 3 x 12 B of vertices per
    primitive tested, triangle.rs:25-40)."""
    rays = max(st.get("rays", 0), 1)
    nodes, prims = st.get("nodes_visited", 0) / rays, st.get("prims_tested", 0) / rays
    return {"nodes_per_ray": nodes, "prims_per_ray": prims, "bytes_per_ray": 36.0 * nodes + 36.0 * prims}


def run_reference(args, asset_root):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import lumillyrender_b200 as lr
    lr.ensure_assets(asset_root, bunny_tris=BUNNY_TRIS, need_ibl=False)
    d = lr.Description(os.path.join(ROOT, "scenes", SCENE + ".toml"), asset_root=asset_root, resolution=(WIDTH, HEIGHT))
    from lumillyrender_b200.renderer import params_from_config

    def params_fn(spp):
        return params_from_config(d.config, spp=spp, seed=1)

    vals, rays, secs = [], [], []
    desc, cores, st = "", 1, None
    budget = 150.0 / max(args.steps + args.warmup, 1)
    for i in range(args.warmup + args.steps):
        ms, mr, st, desc, cores = oracle_sample(d, params_fn, CPU_SAMPLE_SPP, target_seconds=min(12.0, budget))
        if i >= args.warmup:
            vals.append(ms)
            rays.append(mr)
            secs.append(st["render_seconds"])
    v = sum(vals) / len(vals)
    line = {
        "impl": "reference", "metric": "Msamples/s", "value": v, "unit": "Msamples/s", "mrays_per_s": sum(rays) / len(rays),
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * sum(secs) / len(secs),
        "ms_per_step_note": "measured: each timed step renders the bounded sample named in cpu_baseline.sample; the whole workload "
                            "(%d x %d x %d samples) at this rate would take ms_per_full_step" % (WIDTH, HEIGHT, SPP_TOTAL),
        "ms_per_full_step": 1e3 * (WIDTH * HEIGHT * SPP_TOTAL) / (v * 1e6),
        "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.gpus, d.config.n_prims),
        "cpu_baseline": {"value": v, "unit": "Msamples/s", "cores": cores, "kind": "port", "sample": desc,
                         "reference_traversal": reference_traversal(st),
                         "note": "C++ restatement of the reference CPU algorithm (oracle/); the Rust reference cannot be built offline"},
        "e2e": {"value": v, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def workload_config(n_gpus, n_prims):
    return {"workload": "scenes/sample.toml (BASELINE configs[4]) at %dx%d, integrator pt, Cornell box + %d-triangle synthetic bunny stand-in, "
                        "one render of %d spp whose sample indices are sharded over the GPUs, one NCCL reduce per step" % (
                            WIDTH, HEIGHT, BUNNY_TRIS, SPP_TOTAL),
            "resolution": [WIDTH, HEIGHT], "spp_total": SPP_TOTAL, "spp_per_gpu": SPP_TOTAL / n_gpus, "n_prims": int(n_prims),
            "integrator": "pt", "parallelism": "spp-range sharding x%d" % n_gpus,
            "l2": "256 MiB write between steps flushes L2 (scene arrays are ~19 MB and are re-read from L2 within a step by design)"}


def byte_model(cst, n_flat):
    """Algorithmic bytes per ray from the instrumented kernel's counters (DESIGN.md §4): 64 B per BVH node visited, 48 B per
    triangle tested, 32 B per flat-list box gated, 16 B per sphere tested — split into what the TREE costs (nodes + leaf
    triangles: ray-dependent addresses, served by L2) and what the FLAT LIST costs (every ray gates the same few boxes in the
    same order and tests the triangles whose box its line crosses: a handful of cache lines that live in L1)."""
    rays = max(cst["rays"], 1)
    nodes, tris, sph = cst["nodes_visited"] / rays, cst["tris_tested"] / rays, cst["spheres_tested"] / rays
    flat, boxes = cst["flat_tris_tested"] / rays, cst["flat_boxes_tested"] / rays
    tree_b = NODE_BYTES * nodes + TRI_BYTES * (tris - flat)
    flat_b = TRI_BYTES * flat + 32 * boxes + SPHERE_BYTES * sph
    return {"bytes_per_ray": tree_b + flat_b, "tree_bytes_per_ray": tree_b, "flat_list_bytes_per_ray": flat_b,
            "nodes_per_ray": nodes, "tree_tris_per_ray": tris - flat, "flat_tris_per_ray": flat, "flat_boxes_per_ray": boxes,
            "flat_list_size": int(n_flat), "spheres_per_ray": sph}


def kernel_name(d):
    desc = d.desc.contents
    integ = "pt" if d.config.integrator == 0 else "pt-direct"
    tree = desc.n_nodes > 0
    pool = tree                                         # persistent_inst.cu: LR_USE_POOL
    return "%s<%s, %s>" % ("render_pool_kernel" if pool else "render_persistent_kernel", integ, "tree" if tree else "flat")


def run_configs(lr, torch, l2_peak, hbm_peak, asset_root):
    """BASELINE configs 1-4 in the same run: device-timed render at the scene's own film size and spp (CUDA events on the
    launching stream, 3 repeats after a warm-up, L2 flushed between them), the byte model from one instrumented launch,
    and the CPU restatement on a bounded sample (~4 s) beside it."""
    from lumillyrender_b200.renderer import params_from_config
    out = []
    roots = {0: asset_root, BUNNY_TRIS: asset_root}
    stream = torch.cuda.current_stream().cuda_stream
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    for label, name, (w, h), spp, tris in CONFIGS:
        if tris not in roots:
            roots[tris] = lr.ensure_assets(os.path.join(asset_root, "m%d" % tris), bunny_tris=tris, ibl_height=1600)
        elif tris == BUNNY_TRIS:
            lr.ensure_assets(asset_root, bunny_tris=BUNNY_TRIS, ibl_height=1600)
        t0 = time.perf_counter()
        d = lr.Description(os.path.join(ROOT, "scenes", name + ".toml"), asset_root=roots[tris], resolution=(w, h))
        load_s = time.perf_counter() - t0
        host_build_s = float(d.config.bvh_build_seconds)
        s = d.scene()
        accum = torch.zeros((h, w, 3), dtype=torch.float32, device="cuda")
        s.render_accumulate(accum.data_ptr(), None, stream=stream, spp=min(spp, 4), seed=1)      # warm-up
        torch.cuda.synchronize()
        s.stats(stream)
        ms = []
        for rep in range(3):
            flush.fill_(rep)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            s.render_accumulate(accum.data_ptr(), None, stream=stream, spp=spp, seed=10 + rep)
            b.record()
            torch.cuda.synchronize()
            ms.append(a.elapsed_time(b))
        st = s.stats(stream)
        sec = sum(ms) * 1e-3
        _, _, cst = s.render(spp=2, seed=7, count=True)
        bm = byte_model(cst, d.desc.contents.n_flat_triangles)
        rays_per_s = st["rays"] / sec
        cpu_ms, cpu_mr, ost, sample, cores = oracle_sample(d, lambda spp: params_from_config(d.config, spp=spp, seed=1), min(spp, CPU_SAMPLE_SPP),
                                                          target_seconds=4.0, size=(w, h))
        device_bvh = None
        if tris > 0:
            # the same scene with the BVH built on the device (bvh_build_gpu.cu): build time and what the tree costs the render
            host_nodes, host_depth = int(d.desc.contents.n_nodes), int(d.desc.contents.bvh_depth)
            d.rebuild_bvh("device")                              # first call: loads the kernels, grows the memory pool
            wall = d.rebuild_bvh("device")
            s_dev = d.scene()
            s_dev.render_accumulate(accum.data_ptr(), None, stream=stream, spp=min(spp, 4), seed=1)
            torch.cuda.synchronize()
            s_dev.stats(stream)
            dms = []
            for rep in range(2):
                flush.fill_(rep)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                s_dev.render_accumulate(accum.data_ptr(), None, stream=stream, spp=spp, seed=10 + rep)
                b.record()
                torch.cuda.synchronize()
                dms.append(a.elapsed_time(b))
            dst = s_dev.stats(stream)
            device_bvh = {"build_ms_wall": 1e3 * wall, "build_ms_kernels": float(d.config.bvh_device_kernel_ms),
                          "nodes": int(d.desc.contents.n_nodes), "depth": int(d.desc.contents.bvh_depth),
                          "host_sah": {"build_s": host_build_s, "nodes": host_nodes, "depth": host_depth},
                          "msamples_per_s": dst["samples"] / (sum(dms) * 1e-3) / 1e6, "ms_per_render": sum(dms) / len(dms),
                          "what": "Morton-order radix tree (LBVH) built by CUDA kernels from the host triangle array to the host node array "
                                  "(H2D + kernels + D2H); same images bit for bit, a slower tree than the host's binned SAH"}
            s_dev.close()
        out.append({
            "config": label, "scene": "scenes/%s.toml" % name, "resolution": [w, h], "spp": spp,
            "integrator": "pt" if d.config.integrator == 0 else "pt-direct", "n_prims": int(d.config.n_prims),
            "bvh_nodes": int(d.desc.contents.n_nodes), "kernel": kernel_name(d),
            "msamples_per_s": st["samples"] / sec / 1e6, "mrays_per_s": rays_per_s / 1e6, "ms_per_render": sum(ms) / len(ms),
            "launches": int(st["launches"]), "splits": int(st["splits"]),
            "bytes": bm,
            "l2_frac": (bm["bytes_per_ray"] * rays_per_s / 1e9 / l2_peak) if l2_peak else None,
            "l2_frac_tree_only": (bm["tree_bytes_per_ray"] * rays_per_s / 1e9 / l2_peak) if l2_peak else None,
            "hbm_frac": bm["bytes_per_ray"] * rays_per_s / 1e9 / hbm_peak,
            "host_seconds": {"scene_load_s": load_s, "bvh_build_s": host_build_s},
            "device_bvh": device_bvh,
            "cpu": {"msamples_per_s": cpu_ms, "mrays_per_s": cpu_mr, "cores": cores, "kind": "port", "sample": sample,
                    "oracle_bvh_build_s": ost["build_seconds"]},
            "gpu_over_cpu": st["samples"] / sec / 1e6 / cpu_ms,
        })
        s.close()
        d.close()
        del accum
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the mean image of the last timed step (HxWx3 float32) to DIR/image.npy, for comparing builds")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU implementation only")
    with tempfile.TemporaryDirectory(prefix="lumilly_bench_") as asset_root:
        if args.impl == "reference":
            return run_reference(args, asset_root)
        run_b200(args, asset_root)


def run_b200(args, asset_root):
    import numpy as np
    import torch
    import lumillyrender_b200 as lr
    from lumillyrender_b200.distributed import env_rank_world, render_sharded

    rank, local_rank, world = env_rank_world()
    if world != args.gpus and world > 1:
        raise SystemExit("WORLD_SIZE %d != --gpus %d" % (world, args.gpus))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: liblumilly_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    lr.init(local_rank)
    lr.ensure_assets(asset_root, bunny_tris=BUNNY_TRIS, need_ibl=False)     # every rank its own (deterministic) copy
    t0 = time.perf_counter()
    d = lr.Description(os.path.join(ROOT, "scenes", SCENE + ".toml"), asset_root=asset_root, resolution=(WIDTH, HEIGHT))
    load_s = time.perf_counter() - t0
    s = d.scene()
    stream = torch.cuda.current_stream().cuda_stream
    accum = torch.zeros((HEIGHT, WIDTH, 3), dtype=torch.float32, device="cuda")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    spp_total = SPP_TOTAL

    def step(i):
        accum.zero_()
        render_sharded(lambda b, n: s.render_accumulate(accum.data_ptr(), None, stream=stream, spp_begin=b, spp=n, seed=1000 + i),
                       accum, spp_total, rank, world, dist=dist)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        step(i)
        flush.fill_(i & 255)
    barrier()
    s.stats(stream)                                    # reset counters
    sampler = ClockSampler(local_rank)
    sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    for i in range(args.steps):
        ev[i][0].record()
        step(args.warmup + i)
        ev[i][1].record()
        flush.fill_(i & 255)                           # L2 flush between timed iterations (outside the events)
    barrier()
    sampler.stop_flag = True
    step_ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = torch.tensor([sum(step_ms)], dtype=torch.float64, device="cuda")
    st = s.stats(stream)
    counts = torch.tensor([st["rays"], st["samples"], st["launches"]], dtype=torch.float64, device="cuda")
    kernel_ms = torch.tensor([st["kernel_ms"]], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(counts, op=dist.ReduceOp.SUM)
        dist.all_reduce(kernel_ms, op=dist.ReduceOp.MAX)
    total_s = float(total_ms.item()) * 1e-3
    rays, samples, launches = [float(x) for x in counts.tolist()]
    image_mean = float(accum.mean().item()) if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        # the last timed step's result as its caller receives it: the reduced, normalised image (seed 1000 + warmup + steps - 1)
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "image.npy"), accum.cpu().numpy())

    # ---- e2e through the C ABI with host buffers: scene upload (H2D) + render + image download (D2H) per step
    host_img = torch.empty((HEIGHT, WIDTH, 3), dtype=torch.float32).pin_memory()
    e2e_t = []
    h2d = d2h = 0
    import ctypes as C
    from lumillyrender_b200 import capi
    lib = capi.load_library()
    e2e_steps = args.steps
    for i in range(1 + e2e_steps):
        barrier()
        t0 = time.perf_counter()
        s2 = d.scene()                                  # lr_scene_create: H2D of the flat arrays
        h2d = s2.h2d_bytes
        if world == 1:
            p = s2.params(spp=spp_total, seed=2000 + i)
            stats = capi.LrStats()
            capi.check(lib.lr_render(s2._s, C.byref(p), C.cast(host_img.data_ptr(), C.POINTER(C.c_float)), None, C.byref(stats)))
        else:
            accum.zero_()
            render_sharded(lambda b, n: s2.render_accumulate(accum.data_ptr(), None, stream=stream, spp_begin=b, spp=n, seed=2000 + i),
                           accum, spp_total, rank, world, dist=dist)
            if rank == 0:
                host_img.copy_(accum, non_blocking=True)
        torch.cuda.synchronize()
        s2.close()
        d2h = HEIGHT * WIDTH * 3 * 4
        barrier()
        if i >= 1:
            e2e_t.append(time.perf_counter() - t0)
    e2e_s = torch.tensor([sum(e2e_t)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_value = WIDTH * HEIGHT * spp_total * e2e_steps / float(e2e_s.item()) / 1e6

    if rank == 0:
        # ---- roofline inputs: algorithmic bytes per ray from ONE instrumented launch (outside the timed region)
        _, _, cst = s.render(spp=4, seed=7, count=True)
        bm = byte_model(cst, d.desc.contents.n_flat_triangles)
        b_ray = bm["bytes_per_ray"]
        # this rank's launches: rays and milliseconds per launch of the render kernel (launches are per rank; the totals
        # above are sums over ranks)
        rank_launches = max(st["launches"], 1)
        rays_per_launch = st["rays"] / rank_launches
        launch_ms = st["kernel_ms"] / rank_launches
        achieved = b_ray * rays_per_launch / (launch_ms * 1e-3) / 1e9
        achieved_tree = bm["tree_bytes_per_ray"] * rays_per_launch / (launch_ms * 1e-3) / 1e9
        hbm_peak, which = measured_peaks()
        traffic = {}
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            with open(tp) as f:
                traffic = json.load(f)
        try:
            l2_peak = lr.measure_l2_read_gbs(48 << 20, 20)
        except Exception:
            l2_peak = None
        dram = traffic.get("dram_bytes_per_launch")
        algorithmic = b_ray * rays_per_launch
        # the ncu capture is one launch of `spp_of_capture` samples per pixel (ncu cannot replay the bench's 2 s launch): the
        # algorithmic bytes of THAT launch are what its DRAM traffic is compared with
        cap_spp = traffic.get("spp_of_capture") or (spp_total / world)
        algorithmic_capture = algorithmic * cap_spp / (spp_total / world)
        # the scene is L2-resident when the kernel's measured DRAM traffic is a small fraction of the bytes the traversal
        # asks for: the bound is then L2 (tree fetches) / L1 + shared memory (flat list), not HBM
        l2_resident = dram is not None and dram < 0.1 * algorithmic_capture
        measured_l2 = None
        if traffic.get("lts_bytes_per_launch") and traffic.get("kernel_ms_of_capture"):
            measured_l2 = traffic["lts_bytes_per_launch"] / (traffic["kernel_ms_of_capture"] * 1e-3) / 1e9
        roof_l2 = {"bound": "l2", "achieved": achieved, "peak": l2_peak, "unit": "GB/s",
                   "frac": (achieved / l2_peak) if l2_peak else None, "traffic": dram,
                   "peak_source": "lr_measure_l2_read_gbs: 48 MiB working set, ld.global.cg.v4, measured in this run "
                                  "(MEASURED_PEAKS.json supplies no L2 figure)",
                   "achieved_tree_only": achieved_tree, "frac_tree_only": (achieved_tree / l2_peak) if l2_peak else None,
                   "measured_l2_gbs": measured_l2, "measured_l2_frac": (measured_l2 / l2_peak) if (measured_l2 and l2_peak) else None,
                   "measured_l2_source": traffic.get("source"),
                   "kernel": kernel_name(d) + " (pool.cuh)", "kernel_ms_per_launch": launch_ms, "rays_per_launch": rays_per_launch,
                   "algorithmic_bytes_per_launch": algorithmic,
                   "traffic_note": "traffic = dram__bytes_read + dram__bytes_write of ONE %s-spp launch of this kernel on this workload (profiles/traffic.json); "
                                   "the same launch asks for %.3g algorithmic bytes" % (cap_spp, algorithmic_capture)}
        roof_l2.update(bm)
        roof_hbm = {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak, "traffic": dram,
                    "peak_source": "MEASURED_PEAKS.json hbm_gbs (of %s)" % which,
                    "dram_gbs_measured": (dram / (traffic["kernel_ms_of_capture"] * 1e-3) / 1e9) if (dram and traffic.get("kernel_ms_of_capture")) else None,
                    "note": "algorithmic bytes against the HBM peak; the scene is L2-resident, so the DRAM actually moves `traffic` bytes per launch"}
        line = {
            "metric": "Msamples/s", "value": samples / total_s / 1e6, "unit": "Msamples/s",
            "mrays_per_s": rays / total_s / 1e6, "rays_per_sample": rays / max(samples, 1),
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total_s / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(world, d.config.n_prims),
            "e2e": {"value": e2e_value, "unit": "Msamples/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "steps": e2e_steps,
                    "what": "lr_scene_create (H2D of BVH/triangles/materials) + render + D2H of the fp32 image to pinned host memory, wall clock, max over ranks",
                    "outside": {"scene_load_s": load_s, "bvh_build_s": float(d.config.bvh_build_seconds),
                                "note": "TOML + OBJ parse and the BVH build run once per scene file, before e2e's timed region (the reference "
                                        "prints `bvh construction` separately too, description.rs:67-73); the CPU arm's build time is cpu_baseline.oracle_bvh_build_s"}},
            "gpu_launches": int(launches),
            "clocks": sampler.result(),
            "roofline": roof_l2 if (l2_resident or dram is None) else roof_hbm,
            "roofline_hbm" if (l2_resident or dram is None) else "roofline_l2": roof_hbm if (l2_resident or dram is None) else roof_l2,
            "image_mean": image_mean,
        }
        if world == 1 and not args.no_cpu_baseline:
            from lumillyrender_b200.renderer import params_from_config
            ms, mr, ost, desc, cores = oracle_sample(d, lambda spp: params_from_config(d.config, spp=spp, seed=1), CPU_SAMPLE_SPP)
            line["cpu_baseline"] = {"value": ms, "unit": "Msamples/s", "mrays_per_s": mr, "cores": cores, "kind": "port", "sample": desc,
                                    "reference_traversal": reference_traversal(ost), "oracle_bvh_build_s": ost["build_seconds"]}
        if world == 1 and not args.no_configs:
            del accum, flush
            s.close()
            line["configs"] = run_configs(lr, torch, l2_peak, hbm_peak, asset_root)
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
