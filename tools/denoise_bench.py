"""Cost and quality of the non-local-means film filter (drt_cuda_film_denoise) on one GPU, in one process:

    python tools/denoise_bench.py [--scenes init_cornell] [--size 1024] [--ref-spp 4096] [--out FILE]

For each scene at size x size with the 69-wavelength grid: a uniform reference render (--ref-spp, another seed, accumulated in launches
of 1024 samples so that no launch takes 2^32 paths); uniform renders at 16, 32, 64, 128, 256 and 512 spp (16 and 64 spp and 2x, 4x, 8x
each), each timed with CUDA events (best of --reps after a warm-up); the filter at the defaults (r = 7, f = 3, k = 0.45) on the 16 and
64 spp films, timed the same way over --filter-reps back-to-back launches per timing.  Each line gives the luminance MSE
(Y = sum_l w_l mean_l, w = cmf_y * ref_white) against the reference over the pixels usable to the filter (n >= 2, finite statistics),
for the noisy film and for the denoised one, so that "denoised 16 spp ~ uniform X spp" can be read off.  The card's name and power limit
are printed with the numbers."""
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

NOISY = [16, 64]
UNIFORM = [16, 32, 64, 128, 256, 512]


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    fields = [f.strip() for f in q.stdout.strip().split(",")] if q.returncode == 0 else []
    return {"device": torch.cuda.get_device_name(0), "power_limit": fields[1] if len(fields) > 1 else None,
            "sm_max_clock": fields[2] if len(fields) > 2 else None}


def main():
    ap = argparse.ArgumentParser()
    # cornell_plane_light only when named: its classed-kernel render at 1024 x 1024 did not finish (DESIGN.md section 9)
    ap.add_argument("--scenes", default="init_cornell")
    ap.add_argument("--size", type=int, default=1024)
    ap.add_argument("--ref-spp", type=int, default=4096)
    ap.add_argument("--depth", type=int, default=4)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--filter-reps", type=int, default=20)
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
        cfg, tables, sc, cam = common.load(scene, w, h, a.ref_spp, a.depth)
        ctx.upload_scene(sc, cam, tables)
        n = sc.num_wavelengths
        yw = torch.tensor((np.array(tables.cmf_y[:n]) * np.array(tables.ref_white[:n])).astype(np.float32), device="cuda").double()
        planes = [torch.zeros(w * h * n, device="cuda"), torch.zeros(w * h, device="cuda"),
                  torch.zeros(w * h * n, device="cuda"), torch.zeros(w * h * n, device="cuda")]
        film = cuda.film_from_tensors(*planes)
        den = torch.empty(w * h * n, device="cuda")

        def timed(go, reps, inner=1):
            go()
            torch.cuda.synchronize()
            best = float("inf")
            for _ in range(reps):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(inner):
                    go()
                e1.record()
                torch.cuda.synchronize()
                best = min(best, e0.elapsed_time(e1) / inner)
            return best

        ref_ms = 0.0
        for s0 in range(0, a.ref_spp, 1024):
            print(f"{scene}: reference samples [{s0}, {min(s0 + 1024, a.ref_spp)})", file=sys.stderr, flush=True)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            ctx.render_device(oracledriver.params(w, h, s0, min(s0 + 1024, a.ref_spp), a.depth, cfg.pixel_scheme, 99991), film, accumulate=s0 > 0)
            e1.record()
            torch.cuda.synchronize()
            ref_ms += e0.elapsed_time(e1)
        ref = planes[2].view(w * h, n).double() @ yw
        emit({"kind": "reference", "scene": scene, "size": w, "spp": a.ref_spp, "ms": round(ref_ms, 2), **hw})

        def usable():
            cnt = planes[1]
            fin = torch.isfinite(planes[2].view(w * h, n)).all(dim=1) & torch.isfinite(planes[3].view(w * h, n)).all(dim=1)
            return (cnt >= 2) & fin

        def mse(lum, mask):
            return float(torch.mean((lum - ref)[mask] ** 2))

        uni, dens = {}, {}
        for spp in UNIFORM:
            print(f"{scene}: uniform {spp} spp", file=sys.stderr, flush=True)
            prm = oracledriver.params(w, h, 0, spp, a.depth, cfg.pixel_scheme, 7)
            ms = timed(lambda: ctx.render_device(prm, film), a.reps)
            mask = usable()
            noisy = mse(planes[2].view(w * h, n).double() @ yw, mask)
            uni[spp] = noisy
            rec = {"kind": "uniform", "scene": scene, "size": w, "spp": spp, "render_ms": round(ms, 3), "lum_mse": noisy}
            if spp in NOISY:
                f_ms = timed(lambda: ctx.film_denoise(film, w, h, out=den.data_ptr()), a.reps, a.filter_reps)
                denoised = dens[spp] = mse(den.view(w * h, n).double() @ yw, mask)
                rec.update({"filter_ms": round(f_ms, 3), "filter": "r=7 f=3 k=0.45", "lum_mse_denoised": denoised,
                            "mse_ratio": round(denoised / noisy, 4)})
            emit({**rec, **hw})
        for spp in NOISY:
            # the uniform spp whose MSE the denoised film reaches: log-log interpolation between the uniform renders that bracket it
            target, eq = dens[spp], None
            for s0, s1 in zip(UNIFORM, UNIFORM[1:]):
                if uni[s1] <= target <= uni[s0]:
                    t = (np.log(uni[s0]) - np.log(target)) / (np.log(uni[s0]) - np.log(uni[s1]))
                    eq = float(np.exp(np.log(s0) + t * (np.log(s1) - np.log(s0))))
                    break
            emit({"kind": "equal_error", "scene": scene, "size": w, "denoised_spp": spp, "lum_mse_denoised": target,
                  "uniform_spp_at_equal_mse": None if eq is None else round(eq, 1),
                  "note": None if eq is not None else f"outside the uniform renders {UNIFORM[0]}..{UNIFORM[-1]} spp", **hw})
        del planes, film, den
        torch.cuda.empty_cache()
    ctx.close()


if __name__ == "__main__":
    main()
