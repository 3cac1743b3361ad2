"""Where a render kernel's warps spend their cycles, by part of a batch (needs a GPU and a diagnostic build of the library):

    tools/build_variant.sh clocks "-DDRT_PHASE_CLOCKS"
    DRT_CUDA_LIB=build_variants/libdrt_cuda_clocks.so python tools/phase_split.py [--scene S] [--size W] [--spp S] [--depth D]

Defaults are the bench.py workload (init_cornell 1024x1024, 1024 spp, depth 4, seed 20261018).  Prints one JSON line: the SM-clock
cycles the warps spent in phase 1 (trace), the batch bookkeeping, phase 2 (replay) and the rest (task fetch, film load and store), as
shares and per traced path.  The cuts themselves cost a few instructions per batch, so the diagnostic build runs a little slower than
the default one; compare shares between two diagnostic builds, never their times against a default build."""
import argparse
import ctypes as C
import importlib
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", "tests"))
sys.path.insert(0, os.path.join(HERE, ".."))
import common          # noqa: E402
import oracledriver    # noqa: E402

cuda = importlib.import_module("daily-ray-trace_b200.cuda")
PARTS = ("trace", "bookkeeping", "replay", "other")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scene", default="init_cornell")
    ap.add_argument("--size", type=int, default=1024)
    ap.add_argument("--spp", type=int, default=1024)
    ap.add_argument("--depth", type=int, default=4)
    ap.add_argument("--seed", type=int, default=20261018)
    ap.add_argument("--label", default="")
    a = ap.parse_args()
    lib = cuda.lib()
    if not hasattr(lib, "drt_cuda_phase_clocks"):
        raise SystemExit(f"{cuda.library_path()} is not a -DDRT_PHASE_CLOCKS build (tools/build_variant.sh NAME -DDRT_PHASE_CLOCKS)")
    lib.drt_cuda_phase_clocks.argtypes = [C.c_void_p, C.POINTER(C.c_uint64 * 4)]
    import torch
    w = h = a.size
    cfg, tables, sc, cam = common.load(a.scene, w, h, a.spp, a.depth)
    ctx = cuda.Context(0)
    ctx.upload_scene(sc, cam, tables)
    n = sc.num_wavelengths
    planes = [torch.zeros(w * h * n, device="cuda"), torch.zeros(w * h, device="cuda"),
              torch.zeros(w * h * n, device="cuda"), torch.zeros(w * h * n, device="cuda")]
    film = cuda.film_from_tensors(*planes)
    prm = oracledriver.params(w, h, 0, a.spp, a.depth, cfg.pixel_scheme, a.seed)
    ctx.render_device(prm, film)        # warm-up
    ctx.render_device(prm, film)
    clocks = (C.c_uint64 * 4)()
    rc = lib.drt_cuda_phase_clocks(ctx._h, C.byref(clocks))
    if rc != 0:
        raise SystemExit(f"drt_cuda_phase_clocks failed: {rc}")
    st = ctx.stats()
    kinfo = ctx.render_kernel_info(prm)
    ctx.close()
    total = sum(clocks)
    line = {"label": a.label, "workload": f"{a.scene} {w}x{h} {a.spp} spp depth {a.depth}", "kernel": kinfo[0],
            "warp_cycles": {p: int(c) for p, c in zip(PARTS, clocks)},
            "share": {p: c / total for p, c in zip(PARTS, clocks)},
            "warp_cycles_per_camera_path": {p: c / st.paths for p, c in zip(PARTS, clocks)},
            "paths": int(st.paths), "shaded_bounces_per_path": st.shaded_bounces / st.paths}
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
