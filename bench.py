#!/usr/bin/env python
"""bench.py — the reference's headline metric (camera samples/s and Mrays/s of the path integrator) on the
configuration BASELINE.json's north_star scales on: configs[4], the 262 k-triangle atrium at 3840x2160, max_depth 15,
under STRONG scaling — a fixed total number of samples per pixel dealt over the GPUs.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload c1|c2|c3|c5] [--spp S] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...      (one rank per GPU; the driver's way)
    python bench.py --gpus N            (no torchrun: one process drives N devices through ptrs_multi_render)

A step = one full render of the workload into a cleared film: every rank renders the Sobol sample numbers
s = rank (mod N) of every pixel, then the films are summed into rank 0's with ONE NCCL reduce inside the library
(ptrs_film_reduce) — inside the timed region.
  value     camera paths of all ranks / max-over-ranks step time, scene and film resident in HBM (CUDA events on the launching stream)
  e2e       the same through the C ABI with HOST buffers: ptrs_scene_create from host arrays, render, film reduce,
            ptrs_film_download — host<->device copies inside the timed region
  roofline  the BVH traversal kernels (extend_kernel + connect_kernel, one traversal engine; the dominant kernels of the
            workload): algorithmic bytes (32 B x nodes tested + 36 B x triangles tested + 28 B ray + 20 B / 1 B result,
            SURVEY.md §8d) / their summed launch time, against the measured HBM copy bandwidth in MEASURED_PEAKS.json
            (frac), and against the memory system's own figures for this access pattern measured in the same process
            (frac_of_l2_gather, frac_of_l2_stream: the tree is L2 resident on this workload); roofline.stages lists every
            stage of the step; roofline.traffic is the measured DRAM traffic per launch of the same kernels on this
            workload (ncu, profiles/traversal_dram_bytes.json)
  cpu_baseline  the C++ oracle (a restatement of the reference's rayon integrator; the Rust crate cannot be built in
            this image) on a bounded, strided sample of the same workload's 16x16 tiles
  bvh_microbench  BASELINE configs[3] (10 M triangles, 2^24 coherent / incoherent rays): the HBM-bound traversal case
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

# BASELINE.json configs.  "spp" is the TOTAL over all GPUs (strong scaling).  The default is configs[4]; its 1024 spp
# are run as 128: the largest power of two for which the driver's 25 steps at N=1 (~5 s each) fit its per-N time limit.
# The metric is a rate; samples/s does not depend on how many of the 1024 sample numbers a step renders.
WORKLOADS = {
    "c1": {"name": "cornell 512x512 16spp depth15 (BASELINE configs[0])", "res": (512, 512), "spp": 16, "max_depth": 15,
           "scene": "SCENE_CORNELL", "n_tris": 0, "data": "data/cornell-box.xml geometry, built procedurally"},
    "c2": {"name": "cornell + abandoned_tank_farm_04_1k.hdr environment map 1024x1024 64spp depth15 (BASELINE configs[1])", "res": (1024, 1024),
           "spp": 64, "max_depth": 15, "scene": "SCENE_CORNELL_ENV", "n_tris": 0, "env_hdr": True,
           "data": "cornell box + the reference's own data/abandoned_tank_farm_04_1k.hdr (fixture under tests/golden)"},
    "c3": {"name": "1M-triangle material field (glass/substrate/metal/Disney/matte + env + area lights) 1920x1080 256spp depth15 (BASELINE configs[2])",
           "res": (1920, 1080), "spp": 256, "max_depth": 15, "scene": "SCENE_MATERIAL_FIELD", "n_tris": 1000000, "data": "synthetic (seeded procedural scene)"},
    "c5": {"name": "262k-triangle atrium 3840x2160 depth15, 128 of the 1024 spp per step (BASELINE configs[4], strong scaling over the GPUs)",
           "res": (3840, 2160), "spp": 128, "max_depth": 15, "scene": "SCENE_ATRIUM", "n_tris": 262144, "data": "synthetic (seeded procedural scene)"},
}
DEFAULT_WORKLOAD = "c5"
HBM_FALLBACK_GBS = 6650.0  # GB/s of HBM copy bandwidth assumed for a B200 when MEASURED_PEAKS.json is absent
DUMP_PIXELS = 1 << 20  # film pixels --dump-outputs writes at most: 16 MiB of film sums + 8 MiB of pixel indices


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        return HBM_FALLBACK_GBS, "fallback (no MEASURED_PEAKS.json)"


def dump_outputs(out_dir, film_rgbw, counts):
    """--dump-outputs: what the timed path handed back in its last step, for comparing two builds output for output.
    film_rgbw.npy         (N, 4) f32 raw film sums (r, g, b, filter weight) of N pixels: the whole film when it has at most
                          DUMP_PIXELS pixels, else a fixed seeded sample of DUMP_PIXELS of them (the same for every run)
    film_pixel_index.npy  (N,) f64 row-major index y * width + x of each of those pixels
    step_counts.npy       (2,) f64 camera paths and rays (extension + shadow + MIS) of the step over all GPUs"""
    os.makedirs(out_dir, exist_ok=True)
    px = film_rgbw.reshape(-1, 4)
    idx = np.arange(px.shape[0])
    if idx.size > DUMP_PIXELS:
        idx = np.sort(np.random.default_rng(0).choice(idx.size, DUMP_PIXELS, replace=False))
    np.save(os.path.join(out_dir, "film_rgbw.npy"), np.ascontiguousarray(px[idx], dtype=np.float32))
    np.save(os.path.join(out_dir, "film_pixel_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(out_dir, "step_counts.npy"), np.array(counts, dtype=np.float64))


class ClockSampler(threading.Thread):
    """Samples SM clocks and throttle reasons with nvidia-smi while the timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu_index, self.samples, self.stop_flag = gpu_index, [], threading.Event()

    def run(self):
        if self._run_nvml():
            return
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu_index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def _run_nvml(self):
        """The same readings through NVML every 20 ms (an nvidia-smi process takes ~100 ms per sample, too coarse for a
        timed region of half a second).  False if NVML is not usable: the caller falls back to nvidia-smi."""
        try:
            import pynvml as nv

            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.gpu_index)
            mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
        except Exception:
            return False
        bits = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))
        while not self.stop_flag.is_set():
            try:
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.samples.append([str(sm), str(mx)] + ["Active" if r & b else "Not Active" for _, b in bits])
            except Exception:
                pass
            self.stop_flag.wait(0.02)
        return True

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=6)
        sm = [float(s[0]) for s in self.samples if s and s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if len(s) > 1 and s[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for s in self.samples for n, v in zip(names, s[2:6]) if v.lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def host_threads():
    """Threads the CPU arm uses: every core this process may run on.  Passed explicitly because torchrun exports
    OMP_NUM_THREADS=1 to its workers, which would silently make the reference arm single-threaded."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_sample_plan(oracle, flat, cam, params, target_s=12.0):
    """Pick a tile stride so that the oracle renders a uniform subset of the workload's 16x16 tiles in
    roughly target_s seconds on this host."""
    n_tiles = oracle.tile_count(cam, params)
    probe_stride = max(1, n_tiles // 64)
    t0 = time.perf_counter()
    _, st = oracle.render(flat, cam, params, n_threads=host_threads(), tile_stride=probe_stride)
    dt = time.perf_counter() - t0
    per_tile = dt / max(1, (n_tiles + probe_stride - 1) // probe_stride)
    want = max(16, int(target_s / max(per_tile, 1e-9)))
    return n_tiles, max(1, n_tiles // want)


def load_workload(args):
    w = dict(WORKLOADS[args.workload])
    if args.spp:
        w["name"] += f" [run at {args.spp} spp in total]"
        w["spp"] = args.spp
    return w


def build_scene(host, w):
    env = host.TANK_FARM_HDR if w.get("env_hdr") else None
    return host.make_scene(getattr(host, w["scene"]), seed=1, n_tris=w["n_tris"], res=w["res"], env_hdr=env)


def make_config(w, n_gpus):
    """The same dict in both arms (the driver compares them)."""
    W, H = w["res"]
    return {"workload": w["name"], "resolution": [W, H], "spp_total": w["spp"], "max_depth": w["max_depth"],
            "camera_paths_per_step": (W + 4) * (H + 4) * w["spp"],
            "sharding": f"sample number mod {n_gpus} per GPU, films summed by one NCCL reduce inside the timed region",
            "l2": "inputs larger than L2 (368 B of path state per path slot, wavefront batches of up to 2^27 slots = 49 GB) and a 256 MiB buffer written between timed iterations"}


def run_reference(args):
    """--impl reference: the reference algorithm's CPU path (C++ oracle, tile-parallel like
    integrator.rs:617-637, all host threads) on this arm's config; each step = a bounded tile sample."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import pathtracer_rs_b200.host as host
    from oracle import oracle

    w = load_workload(args)
    flat, cam = build_scene(host, w)
    params = host.default_render_params(spp=w["spp"], max_depth=w["max_depth"])
    n_tiles, stride = cpu_sample_plan(oracle, flat, cam, params, target_s=6.0)
    cores = host_threads()
    for _ in range(args.warmup):
        oracle.render(flat, cam, params, n_threads=cores, tile_stride=stride * 8)
    times, paths, rays = [], 0, 0
    for _ in range(args.steps):
        t0 = time.perf_counter()
        film, st = oracle.render(flat, cam, params, n_threads=cores, tile_stride=stride)
        times.append(time.perf_counter() - t0)
        paths = st["camera_paths"]
        rays = st["extension_rays"] + st["shadow_rays"] + st["mis_rays"]
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, film, [paths, rays])
    t = float(np.mean(times))
    value = paths / t
    sample = f"every {stride}th of the {n_tiles} 16x16 tiles, all {w['spp']} spp ({paths} camera paths per step)"
    line = {"impl": "reference", "metric": "samples/sec", "value": value, "unit": "samples/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": w["data"], "mrays_per_s": rays / t / 1e6,
            "config": make_config(w, args.gpus),
            "cpu_baseline": {"value": value, "unit": "samples/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "reference = C++ restatement of the reference's rayon path integrator (oracle/); the Rust crate itself cannot be built in this image"}
    emit(line)


def bvh_microbench(gpu, host, torch, peak_gbs, checker=None):
    """BASELINE configs[3]: fixed-ray intersection microbenchmark on a synthetic 10 M-triangle mesh,
    2^24 coherent and 2^24 incoherent rays; HBM-bound for incoherent rays."""
    n_tris = int(os.environ.get("PTRS_BENCH_BVH_TRIS", "10000000"))
    n_side = int(os.environ.get("PTRS_BENCH_BVH_SIDE", "4096"))
    flat, cam = host.make_scene(host.SCENE_TERRAIN, seed=1, n_tris=n_tris, res=(n_side, n_side))
    scene = gpu.RenderScene(flat)
    bmin, bmax = flat.world_bound()
    out = {"n_tris": flat.n_prims, "n_nodes": flat.n_nodes, "bvh_build_s": flat.bvh_seconds, "scene_mb": scene.device_bytes / 1e6}
    stream = torch.cuda.current_stream().cuda_stream
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    for name in ("coherent", "incoherent"):
        rays = host.coherent_rays(cam, n_side) if name == "coherent" else host.incoherent_rays(bmin, bmax, 42, n_side * n_side)
        n = rays.shape[0]
        d_rays = torch.from_numpy(rays.view(np.uint8).reshape(-1)).cuda()
        d_hits = torch.empty(n * 20, dtype=torch.uint8, device="cuda")
        d_occ = torch.empty(n, dtype=torch.uint8, device="cuda")
        for any_hit in (False, True):
            d_out = d_occ if any_hit else d_hits
            nodes, tris = scene.intersect_counted_device(d_rays.data_ptr(), n, d_out.data_ptr(), any_hit=any_hit, stream=stream)
            alg_bytes = 32 * nodes + 36 * tris + n * (28 + (1 if any_hit else 20))
            ms = []
            for it in range(6):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                if any_hit:
                    scene.intersect_p_device(d_rays.data_ptr(), n, d_occ.data_ptr(), stream)
                else:
                    scene.intersect_device(d_rays.data_ptr(), n, d_hits.data_ptr(), stream)
                e1.record()
                e1.synchronize()
                if it >= 3:
                    ms.append(e0.elapsed_time(e1))
            t = float(np.mean(ms)) * 1e-3
            key = f"{name}_{'any' if any_hit else 'closest'}"
            if checker is not None:  # a strided sample of the results against the oracle: ids, t, barycentrics bit for bit
                pick = np.arange(0, n, max(1, n // 4096))
                if any_hit:
                    got = d_occ.cpu().numpy()[pick]
                    want, _ = checker.intersect_p(flat, rays[pick])
                else:
                    got = d_hits.cpu().numpy().view(host.HIT_DTYPE)[pick]
                    want, _ = checker.intersect(flat, rays[pick])
                same = np.array_equal(got, want) if any_hit else (
                    np.array_equal(got["prim"], want["prim"]) and all(np.array_equal(got[f][want["prim"] >= 0], want[f][want["prim"] >= 0]) for f in ("t", "b0", "b1", "b2")))
                if not same:
                    raise RuntimeError(f"bvh_microbench {key}: device hits differ from the oracle's on the checked sample")
                out.setdefault("hits_checked_against_oracle", {})[key] = int(pick.shape[0])
            out[key] = {"mrays_per_s": n / t / 1e6, "ms": t * 1e3, "nodes_per_ray": nodes / n, "tris_per_ray": tris / n,
                        "achieved_gbs": alg_bytes / t / 1e9, "frac": alg_bytes / t / 1e9 / peak_gbs}
        del d_rays, d_hits, d_occ
    scene.close()
    # the same mesh with the BVH built on the device (ptrs_scene_create_device_bvh, csrc/k_bvh.cu)
    dev = {}
    for tag in ("build_ms_cold", "build_ms_warm"):
        scene = gpu.RenderScene(flat, device_bvh=True)
        dev["n_nodes"], dev[tag] = scene.bvh_info()
        if tag == "build_ms_cold":
            scene.close()
    dev["speedup_vs_host_sah"] = flat.bvh_seconds * 1e3 / dev["build_ms_warm"]
    rays = host.incoherent_rays(bmin, bmax, 42, n_side * n_side)
    n = rays.shape[0]
    d_rays = torch.from_numpy(rays.view(np.uint8).reshape(-1)).cuda()
    d_hits = torch.empty(n * 20, dtype=torch.uint8, device="cuda")
    nodes, tris = scene.intersect_counted_device(d_rays.data_ptr(), n, d_hits.data_ptr(), any_hit=False, stream=stream)
    ms = []
    for it in range(6):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        scene.intersect_device(d_rays.data_ptr(), n, d_hits.data_ptr(), stream)
        e1.record()
        e1.synchronize()
        if it >= 3:
            ms.append(e0.elapsed_time(e1))
    t = float(np.mean(ms)) * 1e-3
    alg_bytes = 32 * nodes + 36 * tris + n * 48
    dev["incoherent_closest"] = {"mrays_per_s": n / t / 1e6, "ms": t * 1e3, "nodes_per_ray": nodes / n, "tris_per_ray": tris / n,
                                 "achieved_gbs": alg_bytes / t / 1e9, "frac": alg_bytes / t / 1e9 / peak_gbs}
    out["device_bvh"] = dev
    scene.close()
    try:  # the memory system's answer to this tree's access pattern: random 64-byte gathers over a buffer of the tree's size
        tree_bytes = int(out["n_nodes"]) * 32 + int(out["n_tris"]) * 48
        out["hbm_gather64_gbs_tree_sized"] = gpu.gather_bandwidth(tree_bytes, 256)
    except Exception:
        pass
    return out


def traffic_record(workload):
    """Measured DRAM traffic per launch (ncu dram__bytes_read.sum + dram__bytes_write.sum) of the traversal kernels on this
    workload, from the committed capture; None when this workload was not captured."""
    try:
        with open(os.path.join(ROOT, "profiles", "traversal_dram_bytes.json")) as f:
            return json.load(f).get(workload)
    except Exception:
        return None


def run_gpu(args):
    import torch
    import torch.distributed as dist

    import pathtracer_rs_b200.gpu as gpu
    import pathtracer_rs_b200.host as host
    from pathtracer_rs_b200._abi import PtrsRenderParams
    from pathtracer_rs_b200.dist import exchange_comm_id, sample_shard

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("no CUDA device: the rendering hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    gpu.set_device(local_rank)
    # "ranks": one process per GPU (torchrun); "threads": this process drives args.gpus devices through ptrs_multi_render
    mode = "ranks" if world > 1 else ("threads" if args.gpus > 1 else "single")
    n_gpus = world if world > 1 else args.gpus
    comm = None
    if mode == "ranks":
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        comm = gpu.Comm(exchange_comm_id(gpu.Comm.unique_id, rank, world), world, rank)  # the film reduce lives in the library
    peak_gbs, peak_src = measured_peaks()

    w = load_workload(args)
    W, H = w["res"]
    flat, cam = build_scene(host, w)
    dev_bvh = args.tree == "device"  # whole run over the tree the library builds (ptrs_scene_create_device_bvh); default: the reference-built tree
    if dev_bvh:
        w["name"] += " [tree built on the device: ptrs_scene_create_device_bvh]"
    integ = gpu.PathIntegrator(gpu.SamplerBuilder(w["spp"]), max_depth=w["max_depth"])
    shard = sample_shard(rank, n_gpus) if mode == "ranks" else (1, 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2
    stream = torch.cuda.current_stream().cuda_stream

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def agg(per_device):
        """one stats dict from the per-device ones: counts add, times take the slowest device"""
        out = dict(per_device[0])
        for st in per_device[1:]:
            for k, v in st.items():
                out[k] = max(out[k], v) if k.startswith("ms_") else out[k] + v
        return out

    if mode == "threads":
        multi = gpu.MultiScene(flat, n_gpus, device_bvh=dev_bvh)
        scene = gpu.RenderScene(flat, device_bvh=dev_bvh)  # device 0 replica for the counted pass

        def step():
            per_dev, ms = multi.render_into(cam, integ.params, None)
            return agg(per_dev), ms

        def counted():
            scene.set_stats_mode(True)
            f = gpu.Film(W, H)
            st = integ.render(cam, scene, f, sample_stride=(n_gpus, 0))
            scene.set_stats_mode(False)
            return st

        def last_film():
            """device 0's film, into which the last step reduced every device's"""
            f, out = C.c_void_p(), np.empty((H, W, 4), dtype=np.float32)
            gpu._check(gpu.lib().ptrs_multi_root_film(multi._h, C.byref(f)))
            gpu._check(gpu.lib().ptrs_film_download(f, out.ctypes.data_as(C.POINTER(C.c_float))))
            return out
    else:
        scene = gpu.RenderScene(flat, device_bvh=dev_bvh)
        integ.preprocess(scene)
        film_t = torch.zeros(H, W, 4, dtype=torch.float32, device="cuda")
        film = gpu.Film(W, H, device_ptr=film_t.data_ptr())

        def step():
            film.clear(stream)
            st = integ.render(cam, scene, film, stream=stream, sample_stride=shard)
            if comm:
                comm.reduce_film(film, root=0, stream=stream)
            return st, None

        def counted():
            scene.set_stats_mode(True)
            st, _ = step()
            scene.set_stats_mode(False)
            return st

        def last_film():
            return film_t.cpu().numpy()

    # one untimed pass with visit counters on: algorithmic bytes of this rank's (deterministic) share of the step
    st_count = counted()
    for _ in range(args.warmup):
        step()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    barrier()
    step_ms, stats = [], None
    for _ in range(args.steps):
        flush.zero_()  # L2 flush between timed iterations
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        stats, lib_ms = step()
        e1.record()
        barrier()
        # "threads": the devices run on the library's own streams, so the step time is the library's clock around the whole
        # call (all streams synchronised on both sides); otherwise CUDA events on the launching stream
        step_ms.append(lib_ms if lib_ms is not None else e0.elapsed_time(e1))
    clocks = sampler.summary() if sampler else None
    t_local = torch.tensor([sum(step_ms)], dtype=torch.float64, device="cuda")
    paths_t = torch.tensor([float(stats["camera_paths"])], dtype=torch.float64, device="cuda")
    rays_t = torch.tensor([float(stats["extension_rays"] + stats["shadow_rays"] + stats["mis_rays"])], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t_local, op=dist.ReduceOp.MAX)  # max over ranks
        dist.all_reduce(paths_t, op=dist.ReduceOp.SUM)
        dist.all_reduce(rays_t, op=dist.ReduceOp.SUM)
    ms_per_step = float(t_local.item()) / args.steps
    paths_step, rays_step = int(paths_t.item()), int(rays_t.item())
    value = paths_step / (ms_per_step * 1e-3)
    if args.dump_outputs and rank == 0:  # rank 0's film holds the sum of all ranks' after the reduce
        dump_outputs(args.dump_outputs, last_film(), [paths_step, rays_step])

    # ---- end to end through the C ABI with host buffers -----------------------------------------------
    host_film = np.empty((H, W, 4), dtype=np.float32)
    e2e_ms, e2e_parts = [], {}
    for it in range(max(2, min(args.steps, 3)) + 1):
        barrier()
        t0 = time.perf_counter()
        if mode == "threads":
            m2 = gpu.MultiScene(flat, n_gpus, device_bvh=dev_bvh, device_tables=True)  # ptrs_multi_create: H2D of the flattened scene to every device
            t1 = time.perf_counter()
            m2.render_into(cam, integ.params, host_film.ctypes.data)  # render + reduce + D2H of the film
            t2 = t3 = time.perf_counter()
            m2.close()
        else:
            sc2 = gpu.RenderScene(flat, device_bvh=dev_bvh, device_tables=True)  # ptrs_scene_create: H2D of the flattened scene; MIP pyramids / env distribution built on the device
            f2 = gpu.Film(W, H)
            t1 = time.perf_counter()
            integ.render(cam, sc2, f2, sample_stride=shard)
            t2 = time.perf_counter()
            if comm:
                comm.reduce_film(f2, root=0)
            if rank == 0:
                gpu._check(gpu.lib().ptrs_film_download(f2._h, host_film.ctypes.data_as(C.POINTER(C.c_float))))
            else:
                torch.cuda.synchronize()
            t3 = time.perf_counter()
            sc2.close()
            del f2
        barrier()
        if it > 0:
            e2e_ms.append((time.perf_counter() - t0) * 1e3)
            e2e_parts = {"scene_create_ms": (t1 - t0) * 1e3, "render_ms": (t2 - t1) * 1e3, "film_reduce_download_ms": (t3 - t2) * 1e3,
                         "destroy_ms": (time.perf_counter() - t3) * 1e3}
    e2e_local = torch.tensor([float(np.mean(e2e_ms))], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(e2e_local, op=dist.ReduceOp.MAX)
    e2e_value = paths_step / (float(e2e_local.item()) * 1e-3)
    h2d = (int(flat.host_bytes_device_tables) + C.sizeof(type(cam)) + C.sizeof(PtrsRenderParams)) * n_gpus
    d2h = H * W * 16

    if rank != 0:
        if comm:
            comm.close()
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernels: BVH traversal (extend + connect) -------------------------------------
    # byte counts from the counted pass, times from the timed steps (this rank's / device 0's share: 1/N of the step)
    ext_rays = st_count["extension_rays"]
    nee_rays = st_count["shadow_rays"] + st_count["mis_rays"]
    ext_bytes = 32 * st_count["nodes_tested"] + 36 * st_count["tris_tested"] + ext_rays * (28 + 20)
    nee_bytes = 32 * st_count["nee_nodes_tested"] + 36 * st_count["nee_tris_tested"] + 28 * nee_rays + 1 * st_count["shadow_rays"] + 20 * st_count["mis_rays"]
    step_mean = sum(step_ms) / len(step_ms)
    ext_ms, con_ms = stats["ms_extend"], stats["ms_connect_trace"]
    trav_bytes, trav_ms = ext_bytes + nee_bytes, ext_ms + con_ms
    trav_launches = stats["extend_launches"] + stats["connect_launches"]
    achieved = trav_bytes / (trav_ms * 1e-3) / 1e9
    tr = traffic_record(args.workload)
    roofline = {"bound": "hbm", "kernel": "extend_kernel<false, DIST> + connect_kernel<false, DIST> (closest-hit / any-hit BVH traversal, one engine: dev_accel.cuh trace_fast; DIST = false on the reference-built tree)",
                "achieved": achieved, "peak": peak_gbs, "unit": "GB/s", "frac": achieved / peak_gbs,
                "traffic": tr.get("dram_bytes_per_launch") if tr else None, "traffic_source": tr.get("source") if tr else None,
                "peak_source": peak_src, "algorithmic_bytes_per_step": trav_bytes, "algorithmic_bytes_per_launch": trav_bytes / max(1, trav_launches),
                "launches_per_step": trav_launches, "avg_launch_ms": trav_ms / max(1, trav_launches),
                "share_of_step": trav_ms / step_mean,
                "extend": {"ms": ext_ms, "achieved_gbs": ext_bytes / (ext_ms * 1e-3) / 1e9, "bytes_per_ray": ext_bytes / max(1, ext_rays),
                           "nodes_per_ray": st_count["nodes_tested"] / max(1, ext_rays), "tris_per_ray": st_count["tris_tested"] / max(1, ext_rays),
                           "mrays_per_s": ext_rays / (ext_ms * 1e-3) / 1e6},
                "connect": {"ms": con_ms, "achieved_gbs": nee_bytes / max(con_ms * 1e-3, 1e-9) / 1e9, "bytes_per_ray": nee_bytes / max(1, nee_rays),
                            "nodes_per_ray": st_count["nee_nodes_tested"] / max(1, nee_rays), "mrays_per_s": nee_rays / max(con_ms * 1e-3, 1e-9) / 1e6},
                "note": f"scene: {flat.n_prims} triangles, {flat.n_nodes} nodes ({(flat.n_nodes * 32 + flat.n_prims * 48) / 1e6:.1f} MB of nodes + triangles: L2 resident; "
                        "`frac` is quoted against the HBM copy peak as the contract asks, frac_of_l2_gather is the roof of this access pattern); the HBM-bound case is bvh_microbench"}
    shade_bytes = (84 + 176) * ext_rays
    roofline["stages"] = {
        "generate": {"ms": stats["ms_generate"], "share_of_step": stats["ms_generate"] / step_mean},
        "extend": {"ms": ext_ms, "share_of_step": ext_ms / step_mean},
        "shade (all materials + miss)": {"ms": stats["ms_shade"], "share_of_step": stats["ms_shade"] / step_mean,
                                         "achieved_gbs": shade_bytes / (stats["ms_shade"] * 1e-3) / 1e9,
                                         "note": "latency bound (dependent scene / table loads), not a bandwidth kernel; record bytes are an upper bound"},
        "connect (trace)": {"ms": con_ms, "share_of_step": con_ms / step_mean},
        "connect_resolve": {"ms": stats["ms_resolve"], "share_of_step": stats["ms_resolve"] / step_mean},
        "accumulate": {"ms": stats["ms_accumulate"], "share_of_step": stats["ms_accumulate"] / step_mean},
    }
    # What the memory system gives THIS access pattern, measured here and now (MEASURED_PEAKS.json has a copy
    # bandwidth only): streaming 256-bit reads and independent random 64-byte gathers (one sibling pair of nodes),
    # from an L2-resident buffer and from one far larger than L2 (ptrs_read_bandwidth / ptrs_gather_bandwidth).
    try:
        probes = {"l2_stream_read_gbs_64MiB": gpu.read_bandwidth(64 << 20, 30), "l2_gather64_gbs_64MiB": gpu.gather_bandwidth(64 << 20, 512),
                  "hbm_stream_read_gbs_4GiB": gpu.read_bandwidth(4 << 30, 2), "hbm_gather64_gbs_1GiB": gpu.gather_bandwidth(1 << 30, 256)}
        roofline["probes"] = probes
        roofline["frac_of_hbm"] = achieved / peak_gbs
        roofline["frac_of_l2_gather"] = achieved / probes["l2_gather64_gbs_64MiB"]
        roofline["frac_of_l2_stream"] = achieved / probes["l2_stream_read_gbs_64MiB"]
    except Exception as e:  # diagnostic only
        roofline["probes"] = {"error": str(e)}

    # ---- CPU baseline: the oracle on a bounded sample of the same workload ----------------------------
    cpu = None
    if n_gpus == 1 and not args.no_cpu_baseline:
        from oracle import oracle

        p1 = host.default_render_params(spp=w["spp"], max_depth=w["max_depth"])
        n_tiles, stride = cpu_sample_plan(oracle, flat, cam, p1, target_s=12.0)
        t0 = time.perf_counter()
        _, ost = oracle.render(flat, cam, p1, n_threads=host_threads(), tile_stride=stride)
        dt = time.perf_counter() - t0
        cpu = {"value": ost["camera_paths"] / dt, "unit": "samples/s", "cores": host_threads(), "kind": "port",
               "sample": f"every {stride}th of the {n_tiles} 16x16 tiles, all {w['spp']} spp ({ost['camera_paths']} camera paths, {dt:.1f} s)",
               "mrays_per_s": (ost["extension_rays"] + ost["shadow_rays"] + ost["mis_rays"]) / dt / 1e6}

    # ---- the same render over the tree the library builds itself (ptrs_scene_create_device_bvh: PLOC clustering, k_bvh.cu) ----
    # An eighth of the step's samples through both trees, one warm-up and one timed pass each.  The headline above stays on
    # the reference-built tree (what the north star names and what the bit-exact hit parity is defined on).
    dev_tree = None
    if n_gpus == 1 and mode == "single" and not args.no_device_bvh_render and not dev_bvh:
        try:
            spp_d = max(1, w["spp"] // 8)
            sc_d = gpu.RenderScene(flat, device_bvh=True)
            dev_tree = {"spp": spp_d, "device_nodes": sc_d.bvh_info()[0], "device_build_ms": sc_d.bvh_info()[1], "reference_nodes": int(flat.n_nodes)}
            for name, sc in (("reference_built_tree", scene), ("device_built_tree", sc_d)):
                for it in range(2):
                    film.clear(stream)
                    flush.zero_()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    std = integ.render(cam, sc, film, stream=stream, sample_range=(0, spp_d))
                    e1.record()
                    e1.synchronize()
                dev_tree[name] = {"ms": e0.elapsed_time(e1), "samples_per_s": std["camera_paths"] / (e0.elapsed_time(e1) * 1e-3),
                                  "ms_extend": std["ms_extend"], "ms_connect_trace": std["ms_connect_trace"]}
            dev_tree["speedup"] = dev_tree["reference_built_tree"]["ms"] / dev_tree["device_built_tree"]["ms"]
            sc_d.close()
        except Exception as e:  # an extra, never the reason a bench line is missing
            dev_tree = {"error": str(e)}

    micro = None
    if n_gpus == 1 and not args.no_bvh_microbench:
        if mode != "threads":
            del film, film_t
        scene.close()
        torch.cuda.empty_cache()
        checker = None
        if not args.no_cpu_baseline:  # the cpu_baseline leg's oracle doubles as the checker of the microbenchmark's hits
            from oracle import oracle as checker
        micro = bvh_microbench(gpu, host, torch, peak_gbs, checker)

    line = {"metric": "samples/sec", "value": value, "unit": "samples/s", "n_gpus": n_gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": w["data"], "mrays_per_s": rays_step / (ms_per_step * 1e-3) / 1e6,
            "config": make_config(w, n_gpus), "launch": {"ranks": "one process per GPU (torchrun), ptrs_comm_* + ptrs_film_reduce", "threads": "one process, ptrs_multi_render",
                                                         "single": "one GPU"}[mode],
            "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": float(e2e_local.item()),
                    "includes": "ptrs_scene_create from host arrays (every rank) + render + NCCL film reduce + ptrs_film_download + ptrs_scene_destroy; excludes the host-side BVH build / scene assembly",
                    "parts_last_step": e2e_parts},
            "gpu_launches": int(stats["launches"]) * args.steps * (n_gpus if mode == "ranks" else 1), "roofline": roofline, "cpu_baseline": cpu, "clocks": clocks,
            "stage_ms": {k: stats[k] for k in ("ms_generate", "ms_extend", "ms_shade", "ms_connect_trace", "ms_resolve", "ms_accumulate", "ms_total")},
            "rays_per_step": rays_step, "rays_rank0": {k: stats[k] for k in ("extension_rays", "shadow_rays", "mis_rays")}, "device_bvh_render": dev_tree, "bvh_microbench": micro}
    emit(line)
    if comm:
        comm.close()
    if world > 1:
        dist.destroy_process_group()


def _claim_stdout():
    """The contract is ONE JSON line on stdout.  Native libraries (NCCL prints its version banner) write to
    file descriptor 1 directly, so fd 1 is pointed at stderr for the whole run and the JSON line goes to a
    private duplicate of the original stdout."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    return os.fdopen(real, "w")


_OUT = None


def emit(line):
    _OUT.write(json.dumps(line) + "\n")
    _OUT.flush()


def main():
    global _OUT
    _OUT = _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-bvh-microbench", action="store_true")
    ap.add_argument("--no-device-bvh-render", action="store_true")
    ap.add_argument("--tree", default="reference", choices=["reference", "device"],
                    help="reference: the host-built SAH tree handed over as LinearBVHNode records (default); device: built by the library")
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--spp", type=int, default=0, help="override the workload's total samples per pixel")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write the last step's film (a seeded sample of a large one) and counts as DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
