#!/usr/bin/env python
"""bench.py -- camera paths/s of the render hot path on N B200s (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W]            one rank per GPU (torchrun for N > 1)
    python bench.py --impl reference ...                           the reference's own CPU code on the host cores
    python bench.py --dump-outputs DIR ...                         also write the last timed step's film to DIR/*.npy
                                                                   (one GPU, or N > 1 with --merge nccl: the default sharded
                                                                   merge leaves the film split over the ranks, and is refused)

One "step" is one complete render of the workload: every pixel, all its samples, film accumulated, and (N > 1) the
per-GPU films combined.  Default workload = BASELINE.json configs[1] / the north-star target: init_cornell.scn, 1024x1024,
1024 spp, max_cast_depth 4, pixel_random.  Scaling is STRONG by default: the 1024 samples of every pixel are split over the
GPUs by sample index (rank r renders global samples [r*spp/N, (r+1)*spp/N)); --scaling weak gives every GPU `spp` samples
(an N*spp image); the other mode is measured too and reported under its own key.  For every N the film that the end-to-end
leg reads back is checked on a tile against the reference's own code over the same global sample indices (image_rmse).
Prints ONE JSON line on rank 0.
"""
import argparse
import ctypes as C
import importlib
import json
import os
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True          # the tree may be read-only: the benchmark leaves nothing in it
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tests"))

PKG = "daily-ray-trace_b200"
import atexit
import shutil
import tempfile
SCRATCH = os.environ.get("DRT_BENCH_SCRATCH") or tempfile.mkdtemp(prefix="drt_bench_")
os.environ["DRT_BENCH_SCRATCH"] = SCRATCH          # pool workers (spawned) share the parent's directory
if os.environ.get("DRT_BENCH_SCRATCH_OWNER") is None:
    os.environ["DRT_BENCH_SCRATCH_OWNER"] = str(os.getpid())
    atexit.register(lambda: shutil.rmtree(SCRATCH, ignore_errors=True))


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scene", default="init_cornell")
    ap.add_argument("--width", type=int, default=1024)
    ap.add_argument("--height", type=int, default=1024)
    ap.add_argument("--spp", type=int, default=1024)
    ap.add_argument("--depth", type=int, default=4)
    ap.add_argument("--seed", type=int, default=20261018)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--geometry", default="f32", choices=["f32", "f64"])
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="N > 1: strong = --spp samples per pixel IN TOTAL, spp/N per GPU (the north-star workload, default); "
                         "weak = --spp samples per pixel PER GPU (an N*spp image).  The other mode is reported as an extra key.")
    ap.add_argument("--spp-sweep", default="", help="comma-separated samples-per-pixel values measured after the main workload "
                                                    "(BASELINE configs[2]: 1,4,16,64,256,1024), reported under spp_sweep")
    ap.add_argument("--no-other-scaling", action="store_true", help="skip the extra measurement in the other scaling mode")
    ap.add_argument("--merge", default="sharded", choices=["sharded", "nccl"],
                    help="multi-GPU film combination: sharded = render kernel scatters finished pixels to their owner over NVLink, "
                         "device-side flags, local merge, film stays sharded (default); nccl = 2 all_reduce + 1 reduce")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the film of the last timed step to DIR/<plane>.npy (float32; a fixed, seeded "
                         "sample of pixels when the whole film is over 60 MB, their indices in pixel_index.npy) to compare two builds")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.gpus > 1 and a.merge == "sharded":
        ap.error("--dump-outputs needs one GPU or --merge nccl (the sharded film is never whole on one device)")
    return a


def samples(a, world):
    """(samples per pixel in total, per GPU) of the chosen scaling mode"""
    if a.scaling == "weak":
        return a.spp * world, a.spp
    return a.spp, max(1, a.spp // world)


def workload_name(a):
    total, per = samples(a, max(1, a.gpus))
    split = "" if a.gpus <= 1 else f" ({a.scaling} scaling: {per} spp on each of {a.gpus} GPUs, sample-index sharded)"
    return f"{a.scene}.scn {a.width}x{a.height} @{total}spp depth{a.depth} pixel_random, N=69 wavelengths{split}"


# ----------------------------------------------------------------------------------------------- CPU arms

def _cpu_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


_W = {}


def _cpu_worker_init(kind, scene, width, height, depth, seed):
    """Runs in every pool process: load the scene once into the reference library (or the oracle port)."""
    import common
    host = importlib.import_module(PKG + ".host")
    assets = os.path.join(REPO, "assets")
    if kind == "reference":
        import refdriver
        parsed = host.parse_scene_text(open(common.scene_path(scene)).read())
        root = os.path.join(SCRATCH, f"ref_root_{os.getpid()}")
        refdriver.make_root(root, assets, host.scene_to_text(parsed), "bench_scene.scn")
        cfg = host.make_config_text(scene="scenes\\bench_scene.scn", width=width, height=height, spp=1, depth=depth)
        devnull = os.open(os.devnull, os.O_WRONLY)
        saved = os.dup(1)
        os.dup2(devnull, 1)          # the reference's CSV loader and scene dump are chatty (read_scene.c:803-844)
        try:
            _W["ref"] = refdriver.Ref(root, cfg, seed=seed)
        finally:
            os.dup2(saved, 1)
            os.close(devnull)
            os.close(saved)
    else:
        import oracledriver
        cfg, tables, sc, cam = common.load(scene, width, height, 1, depth)
        _W["oracle"] = (oracledriver, sc, cam, cfg)
    _W["kind"], _W["dims"], _W["depth"], _W["seed"] = kind, (width, height), depth, seed


def _cpu_worker_render(job):
    """Renders rows [y0, y1) of sample index s through the reference's sample_scene; returns the number of paths."""
    y0, y1, s = job
    w, h = _W["dims"]
    if _W["kind"] == "reference":
        _W["ref"].render_tile(0, y0, w, y1, s, s + 1)
    else:
        od, sc, cam, cfg = _W["oracle"]
        prm = od.params(w, h, s, s + 1, _W["depth"], cfg.pixel_scheme, _W["seed"])
        od.render_tile(sc, cam, prm, 0, y0, w, y1)
    return (y1 - y0) * w


def _cpu_worker_tile(job):
    """Per-path spectra [(pixels), samples, N] of a pixel rectangle through the reference's sample_scene (same per-path streams)."""
    x0, y0, x1, y1, s0, s1 = job
    w, h = _W["dims"]
    if _W["kind"] == "reference":
        return _W["ref"].render_tile(x0, y0, x1, y1, s0, s1, want_paths=True)[3]
    od, sc, cam, cfg = _W["oracle"]
    prm = od.params(w, h, s0, s1, _W["depth"], cfg.pixel_scheme, _W["seed"])
    return od.render_tile(sc, cam, prm, x0, y0, x1, y1, want_paths=True)[3]


def _cpu_worker_tile_film(job):
    """Film (sum, mean, M2) of a pixel rectangle over samples [s0, s1) through the reference's sample_scene."""
    x0, y0, x1, y1, s0, s1 = job
    w, h = _W["dims"]
    if _W["kind"] == "reference":
        return _W["ref"].render_tile(x0, y0, x1, y1, s0, s1)[:3]
    od, sc, cam, cfg = _W["oracle"]
    prm = od.params(w, h, s0, s1, _W["depth"], cfg.pixel_scheme, _W["seed"])
    return od.render_tile(sc, cam, prm, x0, y0, x1, y1)[:3]


class CpuArm:
    """The reference's CPU implementation of the path on all host cores: one single-threaded process per core (the
    reference has global RNG/scratch state, SURVEY.md 8b), rows of the image split between them."""

    def __init__(self, a):
        import multiprocessing as mp
        import refdriver
        self.kind = "reference" if refdriver.available() else "port"
        self.cores = _cpu_cores()
        self.a = a
        os.makedirs(SCRATCH, exist_ok=True)
        self.pool = mp.get_context("spawn").Pool(self.cores, _cpu_worker_init,
                                                (self.kind, a.scene, a.width, a.height, a.depth, a.seed))

    def step(self, sample_index, rows=None):
        """One bounded sample of the workload: `rows` image rows (default all) at ONE sample per pixel."""
        h = self.a.height if rows is None else min(rows, self.a.height)
        per = max(1, h // (self.cores * 4))
        jobs = [(y, min(y + per, h), sample_index) for y in range(0, h, per)]
        t0 = time.perf_counter()
        paths = sum(self.pool.map(_cpu_worker_render, jobs, chunksize=1))
        return paths, time.perf_counter() - t0

    def tile_paths(self, x0, y0, x1, y1, s0, s1):
        import numpy as np
        rows = self.pool.map(_cpu_worker_tile, [(x0, y, x1, y + 1, s0, s1) for y in range(y0, y1)], chunksize=1)
        return np.concatenate(rows, axis=0)

    def tile_film(self, x0, y0, x1, y1, s0, s1):
        """(sum[(px, N+1)], mean, m2) of the tile over ALL samples [s0, s1): pixels split over the pool, every pixel whole."""
        import numpy as np
        cols = max(1, (x1 - x0) // 4)
        jobs = [(x, y, min(x + cols, x1), y + 1, s0, s1) for y in range(y0, y1) for x in range(x0, x1, cols)]
        parts = self.pool.map(_cpu_worker_tile_film, jobs, chunksize=1)
        return tuple(np.concatenate([p[i] for p in parts], axis=0) for i in range(3))

    def close(self):
        self.pool.close()
        self.pool.join()


def run_reference_arm(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    arm = CpuArm(a)
    for i in range(a.warmup):
        arm.step(i)
    paths, secs = 0, 0.0
    for i in range(a.steps):
        p, t = arm.step(a.warmup + i)
        paths += p
        secs += t
    arm.close()
    value = paths / secs
    sample = f"{a.width}x{a.height} at 1 sample per pixel per step ({paths // a.steps} paths/step), rows split over {arm.cores} processes"
    line = {
        "impl": "reference", "metric": "camera_paths_per_sec", "value": value, "unit": "paths/s", "n_gpus": a.gpus,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * secs / a.steps, "higher_is_better": True,
        "scaling": a.scaling, "vs_baseline": None, "dtype": "f64", "data": f"shipped scene assets/scenes/{a.scene}.scn",
        "config": {"workload": workload_name(a), "note": "CPU arm renders a bounded sample of the same workload: cost per sample pass is independent of spp"},
        "cpu_baseline": {"value": value, "unit": "paths/s", "cores": arm.cores, "kind": arm.kind, "sample": sample},
        "e2e": {"value": value, "unit": "paths/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------- clocks

class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.proc = None
        self.lines = []
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={gpu_index}", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        mhz, mx, reasons = [], None, set()
        for t, line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8 or not (t0 - 0.05 <= t <= t1 + 0.15):
                continue
            try:
                mhz.append(float(f[1]))
                mx = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        mhz.sort()
        return {"sm_mhz": mhz[len(mhz) // 2] if mhz else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(mhz)}


# ----------------------------------------------------------------------------------------------- roofline arithmetic

def algorithmic_flops_per_path(scene, st, n):
    """SURVEY.md 8d: flops/path = R_c*F_c + R_s*F_s + B*19N + 8N + 40, with per-surface costs 33 (plane) / 24 (sphere)
    and the ray, shadow-ray and shaded-bounce counts measured by the kernel itself."""
    per_ray = 0
    for i in range(scene.num_surfaces):
        t = scene.surfaces[i].type
        per_ray += 33 if t == 3 else 24 if t == 2 else 0
    rc, rs, b = st.closest_rays / st.paths, st.shadow_rays / st.paths, st.shaded_bounces / st.paths
    return rc * (per_ray + 32) + rs * (per_ray + 33) + b * 19 * n + 8 * n + 40, rc, rs, b


# ----------------------------------------------------------------------------------------------- GPU arm

def pin_to_gpu_numa_node(gpu_index):
    """Bind this rank's host thread to the CPUs NVML reports as local to its GPU, so that the pages of the host film it first
    touches (its own slice) sit on the memory controllers next to its PCIe link.  Returns the number of CPUs, or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * i + b for i, w in enumerate(mask) for b in range(64) if (w >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


class SharedHostFilm:
    """One page-locked host film that every rank of the node writes its own slice into (POSIX shared memory mapped and
    cudaHostRegister-ed by every process): the host-side destination of the per-rank read-back.  Plumbing only."""

    def __init__(self, torch, dist, npix, n, rank, world, pixel_range=None):
        import mmap
        import numpy as np
        self.torch = torch
        self.bytes = (3 * npix * n + npix) * 4
        name = [f"/dev/shm/drt_film_{os.getpid()}" if rank == 0 else None]
        if world > 1:
            dist.broadcast_object_list(name, src=0)
        self.path, self.owner = name[0], rank == 0
        if rank == 0:
            with open(self.path, "wb") as f:
                f.truncate(self.bytes)
        if world > 1:
            dist.barrier()
        self.fd = os.open(self.path, os.O_RDWR)
        self.mm = mmap.mmap(self.fd, self.bytes)
        flat = np.frombuffer(self.mm, dtype=np.float32)
        base = flat.ctypes.data
        # page-lock what this rank's DMA writes: the whole film when it is small, else only the rank's slice of every plane
        # (one registration of a 13.9 GB film per process is refused by the driver)
        p0, p1 = pixel_range if pixel_range is not None else (0, npix)
        if self.bytes <= (2 << 30) or pixel_range is None:
            ranges = [(0, self.bytes)]
        else:
            page = 4096
            ranges = []
            for plane, width in ((0, n), (1, n), (2, n)):
                ranges.append(((plane * npix * n + p0 * width) * 4, (plane * npix * n + p1 * width) * 4))
            ranges.append(((3 * npix * n + p0) * 4, (3 * npix * n + p1) * 4))
            ranges = sorted((lo // page * page, min(self.bytes, -(-hi // page) * page)) for lo, hi in ranges if hi > lo)
            merged = []
            for lo, hi in ranges:
                if merged and lo <= merged[-1][1]:
                    merged[-1] = (merged[-1][0], max(hi, merged[-1][1]))
                else:
                    merged.append((lo, hi))
            ranges = merged
        # first touch by the rank that will DMA into the pages (NUMA placement; see pin_to_gpu_numa_node)
        if pixel_range is not None:
            for plane, width in ((0, n), (1, n), (2, n)):
                flat[plane * npix * n + p0 * width:plane * npix * n + p1 * width] = 0.0
            flat[3 * npix * n + p0:3 * npix * n + p1] = 0.0
        else:
            flat[:] = 0.0
        if world > 1:
            dist.barrier()
        self.registered = []
        for lo, hi in ranges:
            rc = torch.cuda.cudart().cudaHostRegister(base + lo, hi - lo, 0)
            if int(rc) != 0:
                raise RuntimeError(f"cudaHostRegister({hi - lo} bytes) failed: error {int(rc)}")
            self.registered.append(base + lo)
        self.planes = {"sum": flat[:npix * n].reshape(npix, n), "mean": flat[npix * n:2 * npix * n].reshape(npix, n),
                       "m2": flat[2 * npix * n:3 * npix * n].reshape(npix, n), "filter": flat[3 * npix * n:]}

    def drt_film(self, cuda):
        p = self.planes
        return cuda.Film(p["sum"].ctypes.data, p["filter"].ctypes.data, p["mean"].ctypes.data, p["m2"].ctypes.data)

    def close(self):
        for ptr in self.registered:
            try:
                self.torch.cuda.cudart().cudaHostUnregister(ptr)
            except Exception:
                pass
        self.planes = None
        if self.owner:
            try:
                os.unlink(self.path)
            except OSError:
                pass


def run_b200_arm(a):
    import numpy as np
    import torch
    import torch.distributed as dist
    import common
    cuda = importlib.import_module(PKG + ".cuda")
    film_mod = importlib.import_module(PKG + ".film")

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if a.gpus > 1 and world != a.gpus:
        raise SystemExit(f"--gpus {a.gpus} needs torchrun with {a.gpus} ranks (WORLD_SIZE={world})")
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: the product has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    numa = pin_to_gpu_numa_node(local) if world > 1 else None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    spp_total, spp_rank = samples(a, world)
    if a.scaling == "strong" and spp_total % world:
        raise SystemExit(f"--spp {a.spp} is not a multiple of {world} ranks")
    cfg, tables, scene, camera = common.load(a.scene, a.width, a.height, spp_rank, a.depth)
    n = scene.num_wavelengths
    npix = a.width * a.height
    ctx = cuda.Context(local)
    ctx.upload_scene(scene, camera, tables)
    ctx.set_geometry_precision(cuda.GEOMETRY_F64 if a.geometry == "f64" else cuda.GEOMETRY_F32)
    dev = torch.device("cuda", local)
    stream = torch.cuda.current_stream()

    group, film, merge_kind = None, None, "none (one GPU)"
    if world > 1 and a.merge == "sharded":
        group = film_mod.ShardedFilmGroup(ctx, a.width, a.height)
        merge_kind = ("sharded: the render kernel stores each finished pixel into its owner's staging film over NVLink (CUDA IPC), device-side "
                      "arrival flags instead of host barriers, one local merge+images kernel per rank, merged film stays sharded over the owners")
    elif world > 1:
        merge_kind = "nccl: 2 all_reduce + 1 reduce into rank 0"
    if group is None:
        film = film_mod.FilmPlanes(a.width, a.height, n, dev)
        drt_film = film.as_drt_film()

    def params_for(per_rank):
        return common.structs.RenderParams(a.width, a.height, rank * per_rank, (rank + 1) * per_rank, a.depth, cfg.pixel_scheme, a.seed)

    prm = params_for(spp_rank)
    paths_per_step = npix * spp_total
    marks = None

    def mark(name):
        if marks is not None:
            ev = torch.cuda.Event(enable_timing=True)
            ev.record(stream)
            marks[-1][name] = ev

    def step(p=None):
        """One complete render of the workload on this rank's stream; returns the number of kernels launched."""
        p = p or prm
        if group is not None:
            return group.step(p, stream.cuda_stream, mark if marks is not None else None)
        ctx.render_device(p, drt_film, accumulate=False, stream=stream.cuda_stream)
        mark("render")
        if world > 1:
            film_mod.merge_distributed_(film)       # NCCL collectives + torch elementwise kernels: library work, not counted
        return 1

    def fence():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(p, steps):
        """(ms per step: max over ranks of the CUDA-event time of `steps` steps, launches per step, per-step phase events)"""
        nonlocal marks
        fence()
        marks = []
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        launches = 0
        e0.record(stream)
        for _ in range(steps):
            marks.append({})
            mark("start")
            launches += step(p)
        e1.record(stream)
        fence()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        got, marks = marks, None
        return float(ms.item()) / steps, launches // steps, got

    peak_tf = ctx.measure_fp32_peak(False) if rank == 0 else 0.0
    for _ in range(max(a.warmup, 3)):
        step()
    fence()
    sampler = ClockSampler(local) if rank == 0 else None
    t0 = time.perf_counter()
    ms_step, launches_step, ev = timed(prm, a.steps)
    t1 = time.perf_counter()
    clocks = sampler.stop(t0, t1) if sampler else None
    if a.dump_outputs and rank == 0:
        dump_film(a.dump_outputs, film, npix, n, a.seed)
    kernel_ms = sum(m["start"].elapsed_time(m["render"]) for m in ev) / len(ev)
    exchange_ms = None
    if group is not None:
        group.check()
        phases = {"render_kernel": ("start", "render"), "signal_and_wait_for_all_ranks": ("render", "arrived"),
                  "merge_kernel": ("arrived", "merged"), "completion_flags": ("merged", "done")}
        mine = torch.tensor([sum(m[x].elapsed_time(m[y]) for m in ev) / len(ev) for x, y in phases.values()], device="cuda")
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        exchange_ms = {k: {"rank0": float(allr[0][i]), "max_over_ranks": float(max(t[i] for t in allr))} for i, k in enumerate(phases)}
    st = ctx.stats()

    # ---- the other scaling mode as an extra figure (N > 1): weak = every GPU renders `spp` samples, strong = `spp` in total
    other = None
    if world > 1 and not a.no_other_scaling:
        per = a.spp if a.scaling == "strong" else a.spp // world
        if per >= 1:
            p2 = params_for(per)
            step(p2)
            ms2, _, _ = timed(p2, a.steps)
            other = {"scaling": "weak" if a.scaling == "strong" else "strong", "samples_per_pixel_total": per * world,
                     "value": npix * per * world / (ms2 * 1e-3), "unit": "paths/s", "ms_per_step": ms2}

    # ---- sample-count sweep (BASELINE configs[2]): for every value the frame with that many samples per pixel IN TOTAL, split over
    # the GPUs when it divides (strong), and with that many PER GPU (weak); same timing rules, fewer steps for the long ones
    sweep = []
    for v in [int(x) for x in a.spp_sweep.split(",") if x.strip()]:
        entry = {"spp": v}
        for mode, per in (("strong", v // world if v % world == 0 else 0), ("weak", v)):
            if per < 1 or (mode == "weak" and world == 1):
                continue
            pv = params_for(per)
            for _ in range(3):
                step(pv)
            ms_v, _, _ = timed(pv, max(2, min(a.steps, 5)))
            entry[mode] = {"samples_per_pixel_total": per * world, "ms_per_step": ms_v, "value": npix * per * world / (ms_v * 1e-3)}
        sweep.append(entry)

    # ---- end to end through host buffers, every step: scene upload (H2D) + render + exchange + film read-back (D2H).
    # N = 1: the C-ABI host-buffer call drt_cuda_render_host.  N > 1 (sharded): every rank reads ITS merged slice back into one
    # shared page-locked host film over its own PCIe link (drt_cuda_film_read_slice); nccl: rank 0 reads the whole film back.
    host = SharedHostFilm(torch, dist, npix, n, rank, world, (group.p0, group.p1) if group is not None else None) \
        if (world == 1 or group is not None) else None
    pinned = None
    if host is None and rank == 0:
        pinned = {k: torch.empty(shape, dtype=torch.float32).pin_memory()
                  for k, shape in (("sum", (npix, n)), ("filter", (npix,)), ("mean", (npix, n)), ("m2", (npix, n)))}
    host_film = host.drt_film(cuda) if host is not None else None
    d2h = [0]

    e2e_marks = None

    copy_stream = torch.cuda.Stream() if group is not None else None

    def mark_e2e(name, on=None):
        ev = torch.cuda.Event(enable_timing=True)
        ev.record(on or stream)
        e2e_marks[name] = ev

    def e2e_step():
        ctx.upload_scene(scene, camera, tables)
        if e2e_marks is not None:
            mark_e2e("uploaded")
        if world == 1:
            ctx.render_host_into(prm, host_film)
            d2h[0] = (3 * npix * n + npix) * 4
        elif group is not None:
            _, d2h[0] = group.step_bands_to_host(prm, host_film, stream.cuda_stream, copy_stream.cuda_stream)
            if e2e_marks is not None:
                mark_e2e("rendered")
                mark_e2e("on_host", copy_stream)
            copy_stream.synchronize()
            stream.synchronize()
        else:
            step()
            if rank == 0:
                for k, t in (("sum", film.sum), ("filter", film.filter), ("mean", film.mean), ("m2", film.m2)):
                    pinned[k].copy_(t, non_blocking=True)
                d2h[0] = (3 * npix * n + npix) * 4
            torch.cuda.synchronize()
        if world > 1:
            dist.barrier()          # the step is over when the whole film is in host memory

    e2e_step()
    fence()
    te0 = time.perf_counter()
    for _ in range(a.steps):
        e2e_step()
    fence()
    e2e_s = torch.tensor([time.perf_counter() - te0], device="cuda")
    d2h_all = torch.tensor([float(d2h[0])], device="cuda")
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
        dist.all_reduce(d2h_all, op=dist.ReduceOp.SUM)
    e2e_s = float(e2e_s.item())
    e2e_phases = None
    if group is not None:       # one more step with events between its phases (device times; max over ranks)
        e2e_marks = {}
        e2e_step()
        fence()
        mine = torch.tensor([e2e_marks["uploaded"].elapsed_time(e2e_marks["rendered"]), e2e_marks["uploaded"].elapsed_time(e2e_marks["on_host"])], device="cuda")
        e2e_marks = None
        dist.all_reduce(mine, op=dist.ReduceOp.MAX)
        e2e_phases = {"render_stream_ms": float(mine[0]), "until_slice_on_host_ms": float(mine[1]), "bands": len(group.BAND_CUTS) - 1,
                      "host_threads_numa_bound_cpus": numa,
                      "note": "the frame is rendered in bands (the same part of every owner's slice per band); owners merge and read back band b "
                              "on a second stream while band b + 1 renders"}
    upload_bytes = ctx.scene_upload_bytes() * world
    d2h_bytes = int(d2h_all.item())
    if group is not None:
        group.check()

    if rank == 0:
        kinfo = ctx.render_kernel_info(prm)
        flops_path, rc, rs, b = algorithmic_flops_per_path(scene, st, n)
        paths_launch = npix * spp_rank
        achieved_tf = flops_path * paths_launch / (kernel_ms * 1e-3) / 1e12
        # pixels outside the scene's screen-space bound are counted, not traced (exact; drt_cuda_analyse_scene): the fraction of
        # camera paths the kernel executes, and the roofline fraction on executed work alone
        hx0, hy0, hx1, hy1 = cuda.analyse_scene(scene, camera, a.width, a.height)[0]
        traced_fraction = (hx1 - hx0) * (hy1 - hy0) / npix
        per_ray = sum(33 if scene.surfaces[i].type == 3 else 24 if scene.surfaces[i].type == 2 else 0 for i in range(scene.num_surfaces))
        culled_flops = (1.0 - traced_fraction) * ((per_ray + 32) + 8 * n + 40)       # one closest-hit ray, film update, camera
        executed_tf = (flops_path - culled_flops) * paths_launch / (kernel_ms * 1e-3) / 1e12
        film_bytes = (3 * npix * n + npix) * 4
        try:
            hbm_peak = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))["hbm_gbs"]
        except Exception:
            hbm_peak = 6650.0
        value = paths_per_step / (ms_step * 1e-3)
        traffic = None
        try:
            tj = json.load(open(os.path.join(REPO, "profiles", "ncu_traffic.json")))
            if (a.width, a.height) == (1024, 1024):
                traffic = tj["dram_bytes_read_per_launch"] + tj["dram_bytes_written_per_launch"]
        except Exception:
            traffic = None
        line = {
            "metric": "camera_paths_per_sec", "value": value, "unit": "paths/s", "n_gpus": world, "steps": a.steps,
            "warmup": max(a.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": a.scaling,
            "vs_baseline": None, "dtype": "f32", "impl": "b200",
            "data": f"shipped scene assets/scenes/{a.scene}.scn through the legacy-compat parser; per-path Philox4x32-10 streams, seed {a.seed}",
            "config": {"workload": workload_name(a), "geometry": a.geometry, "film_merge": merge_kind,
                       "l2": "inputs (scene + spectra, < 64 KB) live in shared memory; each step writes fresh film planes "
                             f"({film_bytes / 1e6:.0f} MB in all > 126 MB L2), nothing is re-read between steps",
                       "samples_per_pixel_total": spp_total, "samples_per_pixel_per_gpu": spp_rank},
            "rays_per_sec": value * (rc + rs),
            "rays_per_path": {"closest": rc, "shadow": rs, "shaded_bounces": b},
            "paths_traced_fraction": traced_fraction,
            "clocks": clocks,
            "e2e": {"value": paths_per_step * a.steps / e2e_s, "unit": "paths/s", "h2d_bytes_per_step": upload_bytes,
                    "d2h_bytes_per_step": d2h_bytes, "phases": e2e_phases,
                    "note": "scene upload + render (+ exchange) + film read-back into page-locked host memory, wall clock, max over ranks"
                            + ("; every rank reads its own merged slice back over its own PCIe link into one shared host film, band by band under the render" if group is not None else "")},
            "gpu_launches": launches_step * a.steps,
            "film_exchange_ms": exchange_ms,
            "roofline": {"bound": "fp32", "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s",
                         "frac": achieved_tf / peak_tf if peak_tf else None,
                         "frac_executed": executed_tf / peak_tf if peak_tf else None,
                         "frac_note": "frac bills every camera path at the reference's arithmetic (SURVEY.md 8d), frac_executed leaves out the "
                                      "paths of pixels that provably see nothing and are counted instead of traced (paths_traced_fraction)",
                         "traffic": traffic,
                         "traffic_note": "dram__bytes_read.sum + dram__bytes_write.sum of one launch from the committed ncu --set full capture (profiles/ncu_traffic.json); null for other image sizes",
                         "kernel": kinfo[0], "warps_per_cta": kinfo[1], "ctas_per_sm": kinfo[2], "kernel_ms": kernel_ms,
                         "algorithmic_flops_per_path": flops_path,
                         "peak_source": "measured in this run by drt_cuda_measure_fp32_peak (FFMA, 2 flops); MEASURED_PEAKS.json has no FP32 entry",
                         "hbm": {"achieved": film_bytes / (kernel_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                 "frac": film_bytes / (kernel_ms * 1e-3) / 1e9 / hbm_peak,
                                 "note": "algorithmic HBM bytes per launch = one write of the four film planes"}},
        }
        if other is not None:
            line[other["scaling"]] = other
        if sweep:
            line["spp_sweep"] = {"unit": "paths/s", "note": "whole frames at other sample counts, same scene and image size; strong = that many samples "
                                 "per pixel in total split over the GPUs (where it divides), weak = that many per GPU", "points": sweep}
        if not a.no_cpu_baseline:
            try:
                arm = CpuArm(a)
                # image RMSE against the reference on the SAME per-path random streams, every N: a tile of the film the e2e leg left
                # in host memory (for N > 1 it straddles two owners' slices) against the reference's film of all GLOBAL sample indices
                try:
                    line["image_rmse"] = image_check(a, arm, ctx, common, cfg, host.planes if host is not None else {k: v.numpy() for k, v in pinned.items()},
                                                     n, spp_total, world)
                except Exception as exc:
                    line["image_rmse"] = {"value": None, "error": repr(exc)}
                if world == 1:
                    arm.step(0, rows=max(64, a.height // 8))
                    paths, secs, passes = 0, 0.0, 0
                    while secs < 10.0 and passes < 256:   # a bounded sample: about 10 s of work on all host cores
                        p, t = arm.step(1 + passes)
                        paths += p
                        secs += t
                        passes += 1
                    line["cpu_baseline"] = {"value": paths / secs, "unit": "paths/s", "cores": arm.cores, "kind": arm.kind,
                                            "sample": f"{passes} full-frame passes of {a.width}x{a.height} at 1 sample per pixel ({paths} paths, {secs:.1f} s), "
                                                      f"one single-threaded process per core"}
                arm.close()
            except Exception as exc:   # the baseline is reported, never a gate
                line["cpu_baseline"] = {"value": None, "unit": "paths/s", "cores": _cpu_cores(), "kind": "unavailable", "sample": repr(exc)}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
    if host is not None:
        host.close()
    if group is not None:
        group.close()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def dump_film(out_dir, film, npix, n, seed, budget=60_000_000):
    """The four film planes a caller of the render receives, as float32 .npy files.  A film over `budget` bytes is sampled: the
    same pixels (drawn from `seed`) every run, so that two builds can be compared plane by plane."""
    import numpy as np
    import torch
    per_pixel = (3 * n + 1) * 4 + 8
    k = min(npix, budget // per_pixel)
    idx = np.arange(npix) if k == npix else np.sort(np.random.default_rng(seed).choice(npix, k, replace=False))
    sel = torch.from_numpy(idx).to(film.sum.device)
    os.makedirs(out_dir, exist_ok=True)
    for name in ("sum", "filter", "mean", "m2"):
        np.save(os.path.join(out_dir, name + ".npy"), getattr(film, name).index_select(0, sel).cpu().numpy())
    np.save(os.path.join(out_dir, "pixel_index.npy"), idx.astype(np.float64))


def image_check(a, arm, ctx, common, cfg, planes, n, spp_total, world):
    """Film of a centre tile, GPU (as read back by the e2e leg) against the reference over the same global sample indices."""
    import numpy as np
    tw, th = min(32, a.width), min(32, a.height)
    # keep the CPU side bounded (about 4 M paths): a thinner tile for very large sample counts
    while tw * th * spp_total > (1 << 22) and th > 2:
        th //= 2
    x0, y0 = (a.width - tw) // 2, (a.height - th) // 2
    r_sum, r_mean, r_m2 = arm.tile_film(x0, y0, x0 + tw, y0 + th, 0, spp_total)
    idx = np.array([(y0 + j) * a.width + x0 + i for j in range(th) for i in range(tw)])
    g_sum, g_mean, g_m2, g_cnt = (planes[k][idx].astype(np.float64) for k in ("sum", "mean", "m2", "filter"))
    rmse = float(np.sqrt(np.mean((g_mean - r_mean) ** 2)))
    rel = rmse / float(np.abs(r_mean).mean())

    def worst(g, r):
        return float((np.abs(g - r) / np.maximum(np.abs(r), 1e-4 * np.abs(r).max())).max())
    out = {"value": rmse, "relative": rel, "unit": "spectral radiance, RMSE over pixels and wavelengths of the film mean",
           "tile": f"{tw}x{th} at the image centre, all {spp_total} global samples per pixel ({tw * th * spp_total} paths), film as read back by the e2e leg",
           "rng": "matched: both sides draw the same per-path Philox streams (keyed by pixel and GLOBAL sample index)",
           "sample_count_exact": bool((g_cnt == spp_total).all()),
           "max_rel_err": {"sum": worst(g_sum, r_sum[:, :n]), "mean": worst(g_mean, r_mean), "m2": worst(g_m2, r_m2)},
           "reference": arm.kind, "n_gpus": world,
           "ok": bool(rel <= 1e-3 and (g_cnt == spp_total).all())}
    if world == 1:
        prm8 = common.structs.RenderParams(a.width, a.height, 0, 8, a.depth, cfg.pixel_scheme, a.seed)
        ref_paths = arm.tile_paths(x0, y0, x0 + tw, y0 + th, 0, 8)
        gpu_paths = ctx.sample_paths(prm8, x0, y0, x0 + tw, y0 + th)
        out["paths_within_1e-3"] = float((common.path_errors(gpu_paths, ref_paths) <= 1e-3).mean())
    return out


def main():
    a = parse_args()
    if a.impl == "reference":
        run_reference_arm(a)
    else:
        run_b200_arm(a)


if __name__ == "__main__":
    main()
