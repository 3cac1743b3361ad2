"""GPU tier: non-local-means denoising of finished films (drt_cuda_film_denoise / _host, csrc/drt_denoise.cu) against the f64
reference of tests/denoise_ref.py, its exact properties, its quality against a converged render, its error codes and
`drt_raytrace --denoise`."""
import importlib
import os
import subprocess

import numpy as np
import pytest

import common
import denoise_ref
import oracledriver
import refdriver
import test_wavelength_grids_model as grids

cuda = importlib.import_module("daily-ray-trace_b200.cuda")

pytestmark = pytest.mark.gpu

BIN = os.path.join(common.REPO, "daily-ray-trace_b200", "drt_raytrace")
GRID = {n: (lo, hi, step) for n, ns, lo, hi, step in grids.RENDER_GRIDS}


@pytest.fixture(scope="module")
def ctx():
    c = cuda.Context(0)
    yield c
    c.close()


def _setup(ctx, scene, w, h, spp, seed, n=69, depth=4):
    grid = {} if n == 69 else dict(zip(("min_wl", "max_wl", "wl_interval"), GRID[n]))
    cfg, tables, sc, camera = common.load(scene, w, h, spp, depth, **grid)
    assert sc.num_wavelengths == n
    ctx.upload_scene(sc, camera, tables)
    ctx.set_geometry_precision(cuda.GEOMETRY_F32)
    return oracledriver.params(w, h, 0, spp, depth, cfg.pixel_scheme, seed), denoise_ref.luminance_weights(tables, n)


def _check(film, out, yw, w, h, r=7, f=3, k=0.45):
    """The GPU result against the f64 reference: relative 1e-4 (floor 1e-6 max) for >= 99.9 % of the values and 1e-3 for all;
    pass-through pixels bit for bit."""
    ref = denoise_ref.denoise(film["mean"], film["m2"], film["filter"], yw, w, h, r=r, f=f, k=np.float32(k))
    _, _, usable = denoise_ref.guide(film["mean"], film["m2"], film["filter"], yw)
    assert np.array_equal(out[~usable].view(np.uint32), film["mean"][~usable].view(np.uint32))
    floor = 1e-6 * float(np.abs(ref[usable]).max()) if usable.any() else 1.0
    rel = np.abs(out[usable].astype(np.float64) - ref[usable]) / np.maximum(np.abs(ref[usable]), floor)
    print(f"  {int(usable.sum())} of {w * h} pixels usable; rel error max {rel.max() if rel.size else 0:.2e}, "
          f"99.9 % {np.quantile(rel, 0.999) if rel.size else 0:.2e}")
    if rel.size:
        assert np.quantile(rel, 0.999) <= 1e-4 and rel.max() <= 1e-3
    return usable


SCENES = [("init_cornell", 37, 23), ("cornell_plane_light", 37, 23), ("sky_cornell", 37, 23),
          ("init_cornell", 64, 48), ("cornell_plane_light", 64, 48), ("sky_cornell", 64, 48)]


@pytest.mark.parametrize("scene,w,h", SCENES)
def test_matches_reference(ctx, scene, w, h):
    prm, yw = _setup(ctx, scene, w, h, 16, 5)
    film = ctx.render_host(prm)
    usable = _check(film, ctx.film_denoise_host(film, w, h), yw, w, h)
    if scene == "init_cornell":
        # the culled pixels (outside the hit rectangle: counted, black) keep their edge next to the lit ones
        cfg, tables, sc, camera = common.load(scene, w, h, 16, 4)
        x0, y0, x1, y1 = cuda.analyse_scene(sc, camera, w, h)[0]
        yy, xx = np.divmod(np.arange(w * h), w)
        culled = (xx < x0) | (xx >= x1) | (yy < y0) | (yy >= y1)
        assert culled.any() and (film["mean"][culled] == 0).all() and usable[culled].all()
        out = ctx.film_denoise_host(film, w, h)
        print(f"  culled pixels: max {np.abs(out[culled]).max():.3e} of a peak mean {np.abs(film['mean']).max():.3e}")
        assert np.abs(out[culled]).max() <= 1e-3 * np.abs(film["mean"]).max()


@pytest.mark.parametrize("r", [1, 7, 15])
@pytest.mark.parametrize("f", [0, 3, 4])
def test_radii(ctx, r, f):
    w, h = 37, 23
    prm, yw = _setup(ctx, "cornell_plane_light", w, h, 16, 8)
    film = ctx.render_host(prm)
    _check(film, ctx.film_denoise_host(film, w, h, search_radius=r, patch_radius=f, strength=0.7), yw, w, h, r=r, f=f, k=0.7)


def test_adaptive_film(ctx):
    """Counts vary from pixel to pixel."""
    w, h = 37, 23
    prm, yw = _setup(ctx, "init_cornell", w, h, 512, 3)
    film = ctx.render_host_adaptive(prm, 0.05, 64)
    assert len(np.unique(film["filter"])) > 1
    _check(film, ctx.film_denoise_host(film, w, h), yw, w, h)


@pytest.mark.parametrize("n,r,f", [(32, 7, 3), (128, 15, 4), (2, 2, 1)])
def test_wavelength_grids(ctx, n, r, f):
    w, h = 37, 23
    prm, yw = _setup(ctx, "cornell_plane_light", w, h, 16, 4, n=n)
    film = ctx.render_host(prm)
    out = ctx.film_denoise_host(film, w, h, search_radius=r, patch_radius=f)
    assert out.shape == (w * h, n)
    _check(film, out, yw, w, h, r=r, f=f)


def test_unusable_pixels_injected(ctx):
    """An n = 1 pixel, a NaN pixel and an infinite-M2 pixel are copied bit for bit and enter no other pixel's sum."""
    w, h = 64, 48
    prm, yw = _setup(ctx, "cornell_plane_light", w, h, 16, 6)
    film = ctx.render_host(prm)
    film["filter"][100] = 1.0
    film["mean"][777, 5] = np.nan
    film["m2"][1500, 0] = np.inf
    out = ctx.film_denoise_host(film, w, h)
    usable = _check(film, out, yw, w, h)
    assert not usable[[100, 777, 1500]].any() and np.isfinite(out[usable]).all()
    assert np.isnan(out[777, 5])


def test_zero_variance_is_the_identity(ctx):
    w, h = 37, 23
    _setup(ctx, "cornell_plane_light", w, h, 16, 1)
    n = 69
    lum = (np.random.default_rng(2).permutation(w * h) + 1.0).astype(np.float32)
    film = {"mean": (lum[:, None] * np.linspace(0.5, 1.5, n, dtype=np.float32)[None, :]).astype(np.float32),
            "m2": np.zeros((w * h, n), np.float32), "filter": np.full(w * h, 4.0, np.float32)}
    out = ctx.film_denoise_host(film, w, h)
    assert np.array_equal(out.view(np.uint32), film["mean"].view(np.uint32))


def test_constant_film_is_unchanged(ctx):
    w, h = 37, 23
    _setup(ctx, "cornell_plane_light", w, h, 16, 1)
    n = 69
    film = {"mean": np.tile(np.linspace(0.1, 2.0, n, dtype=np.float32), (w * h, 1)), "m2": np.full((w * h, n), 0.25, np.float32),
            "filter": np.full(w * h, 16.0, np.float32)}
    out = ctx.film_denoise_host(film, w, h)
    assert np.allclose(out, film["mean"], rtol=1e-5, atol=0)      # f32 sums of up to 225 equal terms


def test_device_form_exact_properties(ctx):
    """The device call leaves its input planes untouched, two runs are bit-identical, and the host call equals it bit for bit."""
    import torch
    w, h = 64, 48
    prm, yw = _setup(ctx, "init_cornell", w, h, 16, 12)
    n = 69
    planes = [torch.zeros(w * h * n, device="cuda"), torch.zeros(w * h, device="cuda"),
              torch.zeros(w * h * n, device="cuda"), torch.zeros(w * h * n, device="cuda")]
    film = cuda.film_from_tensors(*planes)
    ctx.render_device(prm, film)
    torch.cuda.synchronize()
    before = [p.clone() for p in planes]
    a = ctx.film_denoise(film, w, h)
    out = torch.full((w * h * n,), float("nan"), device="cuda")
    assert ctx.film_denoise(film, w, h, out=out.data_ptr()) is None
    torch.cuda.synchronize()
    for p, q in zip(planes, before):
        assert torch.equal(p.view(torch.int32), q.view(torch.int32))
    assert torch.equal(a.view(torch.int32), out.view(torch.int32))
    host = {"mean": planes[2].cpu().numpy().reshape(w * h, n), "m2": planes[3].cpu().numpy().reshape(w * h, n),
            "filter": planes[1].cpu().numpy()}
    h_out = ctx.film_denoise_host(host, w, h)
    assert np.array_equal(h_out.view(np.uint32), a.cpu().numpy().reshape(w * h, n).view(np.uint32))
    _check(host, h_out, yw, w, h)


@pytest.mark.parametrize("scene", ["init_cornell", "cornell_plane_light"])
def test_quality_against_converged_render(ctx, scene):
    """At 16 spp the denoised luminance is closer to a 4096-spp render with another seed than the noisy one (MSE over usable pixels)."""
    w, h = 128, 96
    prm, yw = _setup(ctx, scene, w, h, 16, 101)
    film = ctx.render_host(prm)
    out = ctx.film_denoise_host(film, w, h)
    ref = ctx.render_host(oracledriver.params(w, h, 0, 4096, 4, prm.pixel_scheme, 202))
    _, _, usable = denoise_ref.guide(film["mean"], film["m2"], film["filter"], yw)
    y_ref = ref["mean"].astype(np.float64) @ yw
    mse_noisy = float(((film["mean"].astype(np.float64) @ yw - y_ref)[usable] ** 2).mean())
    mse_den = float(((out.astype(np.float64) @ yw - y_ref)[usable] ** 2).mean())
    print(f"\n{scene} {w}x{h} 16 spp: luminance MSE noisy {mse_noisy:.4e}, denoised {mse_den:.4e}, ratio {mse_den / mse_noisy:.3f}")
    assert mse_den < mse_noisy


def test_error_codes(ctx):
    w, h = 16, 12
    prm, _ = _setup(ctx, "init_cornell", w, h, 8, 1)
    film = ctx.render_host(prm)
    n = 69
    keep = {k: np.ascontiguousarray(film[k]) for k in ("mean", "m2", "filter")}
    F = cuda.Film(None, keep["filter"].ctypes.data, keep["mean"].ctypes.data, keep["m2"].ctypes.data)
    out = np.empty((w * h, n), np.float32)
    L = cuda.lib()

    def call(film=F, width=w, height=h, opt=cuda.Denoise(7, 3, 0.45), dst=out.ctypes.data, c=ctx._h):
        rc = L.drt_cuda_film_denoise_host(c, cuda.C.byref(film), width, height, cuda.C.byref(opt), dst)
        return rc, L.drt_cuda_last_error().decode()

    assert call()[0] == 0
    for film_, wd, ht, opt, dst, word in [
            (cuda.Film(None, None, F.mean, F.m2), w, h, cuda.Denoise(7, 3, 0.45), out.ctypes.data, "planes"),
            (cuda.Film(None, F.filter, None, F.m2), w, h, cuda.Denoise(7, 3, 0.45), out.ctypes.data, "planes"),
            (cuda.Film(None, F.filter, F.mean, None), w, h, cuda.Denoise(7, 3, 0.45), out.ctypes.data, "planes"),
            (F, 0, h, cuda.Denoise(7, 3, 0.45), out.ctypes.data, "width"),
            (F, w, 0, cuda.Denoise(7, 3, 0.45), out.ctypes.data, "height"),
            (F, w, h, cuda.Denoise(0, 3, 0.45), out.ctypes.data, "search_radius"),
            (F, w, h, cuda.Denoise(16, 3, 0.45), out.ctypes.data, "search_radius"),
            (F, w, h, cuda.Denoise(7, 5, 0.45), out.ctypes.data, "patch_radius"),
            (F, w, h, cuda.Denoise(7, 3, 0.0), out.ctypes.data, "strength"),
            (F, w, h, cuda.Denoise(7, 3, -1.0), out.ctypes.data, "strength"),
            (F, w, h, cuda.Denoise(7, 3, float("nan")), out.ctypes.data, "strength"),
            (F, w, h, cuda.Denoise(7, 3, float("inf")), out.ctypes.data, "strength"),
            (F, w, h, cuda.Denoise(7, 3, 0.45), F.mean, "overlaps"),
            (F, w, h, cuda.Denoise(7, 3, 0.45), F.mean + 4 * 100, "overlaps"),
            (F, w, h, cuda.Denoise(7, 3, 0.45), F.m2, "overlaps")]:
        rc, msg = call(film_, wd, ht, opt, dst)
        assert rc == -103 and word in msg, (rc, msg, word)
    assert np.array_equal(keep["mean"], film["mean"])
    # the device call takes the same checks
    rc = L.drt_cuda_film_denoise(ctx._h, cuda.C.byref(F), w, h, cuda.C.byref(cuda.Denoise(7, 3, 0.45)), F.mean, None)
    assert rc == -103 and "overlaps" in L.drt_cuda_last_error().decode()
    fresh = cuda.Context(0)
    try:
        rc, msg = call(c=fresh._h)
        assert rc == -105 and "scene" in msg
        rc = L.drt_cuda_film_denoise(fresh._h, cuda.C.byref(F), w, h, cuda.C.byref(cuda.Denoise(7, 3, 0.45)), out.ctypes.data, None)
        assert rc == -105
    finally:
        fresh.close()


def _run_main(root, args):
    out = subprocess.run([BIN, "--seed", "5"] + args, cwd=root, check=True, capture_output=True, text=True).stdout
    assert "Converted." in out
    return out, {k: open(os.path.join(root, "output", k), "rb").read() for k in
                 ("output.spd", "average.spd", "variance.spd", "output.bmp", "average.bmp", "variance.bmp")}


@pytest.mark.parametrize("extra", [[], ["--adaptive", "0.05", "--min-spp", "32"], ["--gpus", "2"]])
def test_linux_main_denoise(ctx, host, tmp_path, extra):
    """`drt_raytrace --denoise` writes denoised.spd (film_denoise_host of its own film, read back from average.spd / output.spd) and
    denoised.bmp, and leaves the six usual files as a run without the flag writes them."""
    if "--gpus" in extra:
        import torch
        if torch.cuda.device_count() < 2:
            pytest.skip("needs 2 GPUs")
    if not os.path.exists(BIN):
        pytest.fail("drt_raytrace is not built (make -C daily-ray-trace_b200)")
    root = refdriver.make_root(str(tmp_path), common.ASSETS)
    w, h, spp, n = 37, 23, 64, 69
    open(os.path.join(root, "config.cfg"), "w").write(host.make_config_text(scene="scenes\\init_cornell.scn", width=w, height=h, spp=spp))
    _, plain = _run_main(root, extra)
    assert not os.path.exists(os.path.join(root, "output", "denoised.spd"))
    log, files = _run_main(root, extra + ["--denoise"])
    assert "Denoise time:" in log
    assert files == plain
    den = open(os.path.join(root, "output", "denoised.spd"), "rb").read()
    assert den[:40] == files["average.spd"][:40] and len(den) == len(files["average.spd"])
    bmp = open(os.path.join(root, "output", "denoised.bmp"), "rb").read()
    assert bmp[:2] == b"BM" and len(bmp) == 54 + w * h * 4
    # the film of the run: mean from average.spd, count from output.spd; M2 does not survive in the files (variance.spd is normalised),
    # so it comes from the library's own render of the same samples, whose mean and count equal the files'
    prm, _ = _setup(ctx, "init_cornell", w, h, spp, 5)
    body = np.frombuffer(files["output.spd"][40:], dtype=np.float64).reshape(w * h, n + 1)
    mean = np.frombuffer(files["average.spd"][40:], dtype=np.float64).reshape(w * h, n).astype(np.float32)
    if extra[:1] == ["--adaptive"]:
        lib_film = ctx.render_host_adaptive(prm, 0.05, 32)
    elif extra[:1] == ["--gpus"]:
        other = cuda.Context(1)
        try:
            cfg, tables, sc, camera = common.load("init_cornell", w, h, spp, 4)
            other.upload_scene(sc, camera, tables)
            lib_film = cuda.render_host_multi([ctx, other], prm)
        finally:
            other.close()
    else:
        lib_film = ctx.render_host(prm)
    assert np.array_equal(lib_film["filter"], body[:, n].astype(np.float32))
    assert np.array_equal(lib_film["mean"], mean)
    film = {"mean": mean, "m2": lib_film["m2"], "filter": lib_film["filter"]}
    expect = ctx.film_denoise_host(film, w, h)
    got = np.frombuffer(den[40:], dtype=np.float64).reshape(w * h, n)
    assert np.array_equal(got.astype(np.float32), expect)
