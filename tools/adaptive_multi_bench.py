"""Adaptive sampling on several GPUs of one process, sharded by rows (drt_cuda_render_host_multi_adaptive):

    python tools/adaptive_multi_bench.py [--size 1024] [--reps 3] [--out profiles/adaptive_multi_r6.jsonl]

Device g renders the rows y = g (mod G) of the frame and reads them back over its own PCIe link; nothing is merged.  Workloads:
init_cornell at size x size, cap 4096, min_samples 64, rel_error 0.01 and 0.02.  cornell_plane_light (the classed kernel) at cap 1024,
rel_error 0.02 runs only when named in --workloads (cornell_plane_light:1024:0.02): at 1024² that launch has not finished (DESIGN.md
section 9).  For G = 1, 2, 4, 8 (as many as the machine has), after a warm-up of every G, each line gives
  - e2e_ms: the best of --reps end-to-end calls of render_host_multi_adaptive into a pinned host film (host clock; the call waits);
    e2e_pageable_ms: the same for the binding's default call, which returns new (pageable) numpy planes;
  - kernel_ms / copy_ms per device: CUDA events around each device's drt_cuda_render_device_adaptive_rows launch and around its
    drt_cuda_film_read_rows copy, all devices at once on their own streams (best of --reps); paths per device;
  - imbalance: max / mean of the per-device kernel times and of the per-device paths;
  - exposed_copy_ms: the copy time left after the slowest render, max_g (kernel_g + copy_g) - max_g kernel_g (a device's copy starts
    when its render ends; it hides only under the renders of slower devices);
  - efficiency: T_1 / (G T_G) for the end-to-end time and for the slowest device's kernel time.
Every G's film must equal the G = 1 film bit for bit, else the script fails.  Each workload runs in a child process with a timeout, so a
launch that does not finish is recorded as such; the child's progress goes to stderr.  The cards' names and power limits (nvidia-smi,
read only) are part of every line."""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.join(HERE, "..")
sys.path.insert(0, os.path.join(REPO, "tests"))
sys.path.insert(0, REPO)

WORKLOADS = [("init_cornell", 4096, 0.01), ("init_cornell", 4096, 0.02)]
# scenes whose launch at 1024² with >= 1024 samples per pixel has not finished (the classed kernel; DESIGN.md section 9)
NOT_FINISHING = {"cornell_plane_light", "classed_all"}
MIN_SAMPLES, DEPTH, SEED = 64, 4, 7


def cards():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True)
    rows = [r.split(",") for r in q.stdout.strip().splitlines()[1:]] if q.returncode == 0 else []
    return {"gpus": [{"name": r[0].strip(), "power_limit": r[1].strip()} for r in rows if len(r) >= 2], "gpu_count": len(rows)}


def one(scene, cap, rel_error, size, reps, hw):
    """All G for one workload; returns the JSON lines."""
    import numpy as np
    import torch
    import common
    import oracledriver
    cuda = importlib.import_module("daily-ray-trace_b200.cuda")
    ndev = cuda.device_count()
    counts = [g for g in (1, 2, 4, 8) if g <= ndev]
    w = h = size
    cfg, tables, sc, cam = common.load(scene, w, h, cap, DEPTH)
    n = sc.num_wavelengths
    prm = oracledriver.params(w, h, 0, cap, DEPTH, cfg.pixel_scheme, SEED)
    ctxs = [cuda.Context(d) for d in range(counts[-1])]
    for c in ctxs:
        c.upload_scene(sc, cam, tables)
    # pinned host film of the end-to-end call
    pinned = {k: torch.empty((w * h, n) if k != "filter" else (w * h,), dtype=torch.float32).pin_memory() for k in ("sum", "filter", "mean", "m2")}
    host_film = cuda.Film(*(pinned[k].data_ptr() for k in ("sum", "filter", "mean", "m2")))
    # device films and streams of the event-timed runs
    planes = [[torch.zeros(w * h * n if i != 1 else w * h, device=f"cuda:{d}") for i in range(4)] for d in range(len(ctxs))]
    films = [cuda.film_from_tensors(*p) for p in planes]
    streams = [torch.cuda.Stream(device=d) for d in range(len(ctxs))]

    def e2e(g):
        t0 = time.perf_counter()
        cuda.render_host_multi_adaptive(ctxs[:g], prm, rel_error, MIN_SAMPLES, film=host_film)
        return (time.perf_counter() - t0) * 1e3

    def e2e_pageable(g):
        t0 = time.perf_counter()
        cuda.render_host_multi_adaptive(ctxs[:g], prm, rel_error, MIN_SAMPLES)
        return (time.perf_counter() - t0) * 1e3

    def evented(g):
        ev = []
        for d in range(g):
            with torch.cuda.device(d):
                e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
                s = streams[d]
                e[0].record(s)
                ctxs[d].render_device_adaptive_rows(prm, rel_error, MIN_SAMPLES, films[d], g, d, stream=s.cuda_stream)
                e[1].record(s)
                ctxs[d].film_read_rows(films[d], w, h, g, d, host_film, stream=s.cuda_stream)
                e[2].record(s)
                ev.append(e)
        for d in range(g):
            streams[d].synchronize()
        paths = [int(ctxs[d].stats().paths) for d in range(g)]
        return [e[0].elapsed_time(e[1]) for e in ev], [e[1].elapsed_time(e[2]) for e in ev], paths

    for g in counts:   # warm-up of every G
        e2e(g)
        evented(g)
    lines, ref, t1 = [], None, {}
    for g in counts:
        e2e_ms = min(e2e(g) for _ in range(reps))
        film = {k: v.numpy().view(np.uint32).copy() for k, v in pinned.items()}
        pageable_ms = min(e2e_pageable(g) for _ in range(reps))
        if ref is None:
            ref = film
        identical = all(np.array_equal(film[k], ref[k]) for k in film)
        best = None
        for _ in range(reps):
            k_ms, c_ms, paths = evented(g)
            if best is None or max(k_ms) < max(best[0]):
                best = (k_ms, c_ms, paths)
        k_ms, c_ms, paths = best
        kmax = max(k_ms)
        if g == 1:
            t1 = {"e2e": e2e_ms, "kernel": kmax}
        lines.append({"kind": "adaptive_multi", "scene": scene, "size": size, "cap": cap, "min_samples": MIN_SAMPLES, "rel_error": rel_error,
                      "depth": DEPTH, "gpus_used": g, "e2e_ms": round(e2e_ms, 3), "e2e_pageable_ms": round(pageable_ms, 3),
                      "kernel_ms": [round(x, 3) for x in k_ms], "copy_ms": [round(x, 3) for x in c_ms], "paths": paths,
                      "mean_spp": round(sum(paths) / (w * h), 2),
                      "imbalance_kernel": round(kmax / (sum(k_ms) / g), 4), "imbalance_paths": round(max(paths) / (sum(paths) / g), 4),
                      "exposed_copy_ms": round(max(k + c for k, c in zip(k_ms, c_ms)) - kmax, 3),
                      "efficiency_e2e": round(t1["e2e"] / (g * e2e_ms), 4), "efficiency_kernel": round(t1["kernel"] / (g * kmax), 4),
                      "film_identical_to_g1": identical, **hw})
        print(json.dumps(lines[-1]), file=sys.stderr, flush=True)
    for c in ctxs:
        c.close()
    return lines


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--timeout", type=float, default=300.0, help="seconds per workload (all G)")
    ap.add_argument("--workloads", default=",".join(f"{s}:{c}:{r}" for s, c, r in WORKLOADS), help="scene:cap:rel_error,...")
    ap.add_argument("--out", default=os.path.join(REPO, "profiles", "adaptive_multi_r6.jsonl"))
    ap.add_argument("--one", default=None, help=argparse.SUPPRESS)   # child: scene,cap,rel_error
    a = ap.parse_args()
    hw = json.loads(os.environ["DRT_BENCH_HW"]) if a.one else cards()
    if a.one:
        scene, cap, rel = a.one.split(",")
        for line in one(scene, int(cap), float(rel), a.size, a.reps, hw):
            print(json.dumps(line), flush=True)
        return
    ok = True
    with open(a.out, "w") as out:
        out.write(json.dumps({"kind": "cards", **hw}) + "\n")
        for scene, cap, rel in (w.split(":") for w in a.workloads.split(",")):
            cap, rel = int(cap), float(rel)
            if scene in NOT_FINISHING:
                print(f"warning: {scene} runs the classed kernel, whose launches at 1024² with 1024 or more samples per pixel have not "
                      f"finished (DESIGN.md section 9); the child is stopped after {a.timeout:g} s", file=sys.stderr, flush=True)
            cmd = [sys.executable, os.path.abspath(__file__), "--one", f"{scene},{cap},{rel}", "--size", str(a.size), "--reps", str(a.reps)]
            try:
                r = subprocess.run(cmd, stdout=subprocess.PIPE, text=True, timeout=a.timeout, env=dict(os.environ, DRT_BENCH_HW=json.dumps(hw)))
                lines = [json.loads(x) for x in r.stdout.splitlines() if x.startswith("{")]
                if r.returncode != 0:
                    lines.append({"kind": "failed", "scene": scene, "cap": cap, "rel_error": rel, "returncode": r.returncode, **hw})
            except subprocess.TimeoutExpired:
                lines = [{"kind": "did_not_finish", "scene": scene, "cap": cap, "rel_error": rel, "timeout_s": a.timeout, **hw}]
            for line in lines:
                print(json.dumps(line), flush=True)
                out.write(json.dumps(line) + "\n")
                out.flush()
                ok = ok and line["kind"] == "adaptive_multi" and line["film_identical_to_g1"]
    if not ok:
        sys.exit("a workload failed, did not finish, or gave a film that differs from G = 1")


if __name__ == "__main__":
    main()
