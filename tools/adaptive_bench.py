"""Adaptive sampling against uniform sampling on one GPU, in one process:

    python tools/adaptive_bench.py [--scenes init_cornell,cornell_plane_light] [--size 1024] [--ref-spp 16384] [--out FILE]

For each scene at size x size: a uniform reference render (--ref-spp, another seed); uniform renders at 256, 512, 1024 and 4096 spp;
adaptive renders with cap 4096, min_samples 64 and rel_error 0.05, 0.02, 0.01, 0.005.  Each line gives the CUDA-event time of the
device render (best of --reps after a warm-up), the paths taken, the mean samples per pixel and the RMSE of the luminance
Y = sum_l w_l mean_l (w = cmf_y * ref_white, the weights of the adaptive rule) against the reference.  A summary line per scene gives
the time at which adaptive sampling reaches the error of uniform 1024 spp (log-log interpolation between the adaptive renders that
bracket it) and the speed-up at equal error, for the luminance RMSE and for the relative luminance RMSE over the pixels the reference
sees lit (the error the adaptive rule bounds).  Two more lines measure the cost of the check itself in paths/s against uniform 1024 spp:
rel_error 1e-6 with min_samples 64 (no lit pixel stops early; unlit pixels stop at 64), and min_samples = cap (no pixel stops early, so
the two renders trace the same paths).  The card's name and power limit are printed with the numbers."""
import argparse
import importlib
import json
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", "tests"))
sys.path.insert(0, os.path.join(HERE, ".."))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import common  # noqa: E402
import oracledriver  # noqa: E402

cuda = importlib.import_module("daily-ray-trace_b200.cuda")

UNIFORM = [256, 512, 1024, 4096]
ADAPTIVE_CAP, ADAPTIVE_MIN = 4096, 64
REL_ERRORS = [0.05, 0.02, 0.01, 0.005]


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    fields = [f.strip() for f in q.stdout.strip().split(",")] if q.returncode == 0 else []
    return {"device": torch.cuda.get_device_name(0), "power_limit": fields[1] if len(fields) > 1 else None,
            "sm_max_clock": fields[2] if len(fields) > 2 else None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenes", default="init_cornell,cornell_plane_light")
    ap.add_argument("--size", type=int, default=1024)
    ap.add_argument("--ref-spp", type=int, default=16384)
    ap.add_argument("--depth", type=int, default=4)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    a = ap.parse_args()
    out = open(a.out, "a") if a.out else None

    def emit(rec):
        line = json.dumps(rec)
        print(line, flush=True)
        if out:
            out.write(line + "\n")
            out.flush()

    hw = card()
    emit({"kind": "card", **hw})
    ctx = cuda.Context(0)
    w = h = a.size
    for scene in a.scenes.split(","):
        cfg, tables, sc, cam = common.load(scene, w, h, ADAPTIVE_CAP, a.depth)
        ctx.upload_scene(sc, cam, tables)
        n = sc.num_wavelengths
        yw = torch.tensor((np.array(tables.cmf_y[:n]) * np.array(tables.ref_white[:n])).astype(np.float32), device="cuda")
        planes = [torch.zeros(w * h * n, device="cuda"), torch.zeros(w * h, device="cuda"),
                  torch.zeros(w * h * n, device="cuda"), torch.zeros(w * h * n, device="cuda")]
        film = cuda.film_from_tensors(*planes)

        def render(spp, seed, rel_error=None, min_samples=ADAPTIVE_MIN, reps=a.reps):
            print(f"{scene}: {'uniform' if rel_error is None else f'adaptive {rel_error:g}'} {spp} spp", file=sys.stderr, flush=True)
            prm = oracledriver.params(w, h, 0, spp, a.depth, cfg.pixel_scheme, seed)
            go = (lambda: ctx.render_device(prm, film)) if rel_error is None else \
                 (lambda: ctx.render_device_adaptive(prm, rel_error, min_samples, film))
            go()
            torch.cuda.synchronize()
            best = float("inf")
            for _ in range(reps):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                go()
                e1.record()
                torch.cuda.synchronize()
                best = min(best, e0.elapsed_time(e1))
            paths = ctx.stats().paths
            lum = planes[2].view(w * h, n) @ yw
            return best, paths, lum

        # the reference in accumulated chunks of 4096 samples: no launch takes more than 2^32 paths
        ref_ms = 0.0
        for s0 in range(0, a.ref_spp, 4096):
            print(f"{scene}: reference samples [{s0}, {min(s0 + 4096, a.ref_spp)})", file=sys.stderr, flush=True)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            ctx.render_device(oracledriver.params(w, h, s0, min(s0 + 4096, a.ref_spp), a.depth, cfg.pixel_scheme, 99991), film, accumulate=s0 > 0)
            e1.record()
            torch.cuda.synchronize()
            ref_ms += e0.elapsed_time(e1)
        ref = planes[2].view(w * h, n) @ yw
        lit = ref > 0
        emit({"kind": "reference", "scene": scene, "size": w, "spp": a.ref_spp, "ms": round(ref_ms, 2), "lit_pixels": int(lit.sum()),
              "kernel": ctx.render_kernel_info(oracledriver.params(w, h, 0, a.ref_spp, a.depth, cfg.pixel_scheme, 1))[0], **hw})

        def rmse(lum):
            return float(torch.sqrt(torch.mean((lum.double() - ref.double()) ** 2)))

        def rel_rmse(lum):   # over the pixels the reference sees lit: the error the adaptive rule bounds
            return float(torch.sqrt(torch.mean(((lum.double() - ref.double())[lit] / ref.double()[lit]) ** 2)))

        uni = {}
        for spp in UNIFORM:
            ms, paths, lum = render(spp, 7)
            uni[spp] = (ms, rmse(lum), rel_rmse(lum))
            emit({"kind": "uniform", "scene": scene, "size": w, "spp": spp, "ms": round(ms, 3), "paths": paths,
                  "mean_spp": paths / (w * h), "gpaths_per_s": round(paths / ms * 1e-6, 3), "lum_rmse": uni[spp][1], "lum_rel_rmse": rel_rmse(lum), **hw})
        ada = []
        for rel in REL_ERRORS:
            ms, paths, lum = render(ADAPTIVE_CAP, 7, rel)
            ada.append((ms, rmse(lum), rel_rmse(lum)))
            emit({"kind": "adaptive", "scene": scene, "size": w, "cap": ADAPTIVE_CAP, "min_samples": ADAPTIVE_MIN, "rel_error": rel,
                  "ms": round(ms, 3), "paths": paths, "mean_spp": round(paths / (w * h), 2), "gpaths_per_s": round(paths / ms * 1e-6, 3),
                  "lum_rmse": ada[-1][1], "lum_rel_rmse": ada[-1][2], **hw})
        # time at which adaptive sampling reaches the error of uniform 1024 spp: log-log interpolation between bracketing renders
        for metric, col in (("lum_rmse", 1), ("lum_rel_rmse", 2)):
            target_ms, target = uni[1024][0], uni[1024][col]
            t_eq = None
            for r0, r1 in zip(ada, ada[1:]):
                if r1[col] <= target <= r0[col] and r0[col] > r1[col]:
                    f = (np.log(r0[col]) - np.log(target)) / (np.log(r0[col]) - np.log(r1[col]))
                    t_eq = float(np.exp(np.log(r0[0]) + f * (np.log(r1[0]) - np.log(r0[0]))))
                    break
            emit({"kind": "equal_error", "scene": scene, "size": w, "metric": metric, "uniform_spp": 1024, "uniform_ms": round(target_ms, 3),
                  metric: target, "adaptive_ms_at_equal_error": None if t_eq is None else round(t_eq, 3),
                  "speedup": None if t_eq is None else round(target_ms / t_eq, 3),
                  "note": None if t_eq is not None else "no two adaptive renders bracket the uniform error", **hw})
        # cost of the check: alternate the uniform and the adaptive render of the same cap
        for label, mn in (("rel_error 1e-6, min_samples 64", ADAPTIVE_MIN), ("rel_error 1e-6, min_samples = cap", 1024)):
            rates_u, rates_a = [], []
            for _ in range(3):
                ms, paths, _ = render(1024, 7)
                rates_u.append(paths / ms * 1e-6)
                ms, paths_a, _ = render(1024, 7, 1e-6, mn)
                rates_a.append(paths_a / ms * 1e-6)
            u, ad = float(np.median(rates_u)), float(np.median(rates_a))
            emit({"kind": "check_cost", "scene": scene, "size": w, "spp": 1024, "adaptive": label, "uniform_gpaths_per_s": round(u, 3),
                  "adaptive_gpaths_per_s": round(ad, 3), "adaptive_paths": paths_a, "uniform_paths": paths,
                  "cost_percent": round(100 * (1 - ad / u), 2), **hw})
        del planes, film
        torch.cuda.empty_cache()
    ctx.close()


if __name__ == "__main__":
    main()
