"""GPU tier: the compact-record replay (plastic-only kernel, mode 1) and its per-batch film statistics.

The compact-record kernels replay a path from its last bounce to its first and fold the samples of a batch into the film in units
of the light's emission (drt_render.cuh: replay_compact, BatchStats, PixelFilm::add_batch).  These tests render films with many
batches, a partial last batch and both task shapes (spp >= 32: one pixel per task; spp < 32: several pixels per task), and check
them against the oracle and against the exact statistics of the same paths as the kernel dumps them."""
import importlib

import numpy as np
import pytest

import common
import oracledriver

cuda = importlib.import_module("daily-ray-trace_b200.cuda")

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = cuda.Context(0)
    yield c
    c.close()


def _rel(a, b, floor):
    return np.abs(a.astype(np.float64) - b) / np.maximum(np.abs(b), floor)


def _setup(ctx, scene, w, h, spp, depth, seed, deep=False):
    cfg, tables, sc, camera = common.load(scene, w, h, spp, depth)
    ctx.upload_scene(sc, camera, tables)
    ctx.set_geometry_precision(cuda.GEOMETRY_F32)
    prm = oracledriver.params(w, h, 0, spp, depth, cfg.pixel_scheme, seed)
    name = ctx.render_kernel_info(prm)[0]
    assert name.startswith("drt::render_kernel<float,") and name.endswith(f",1,{'true' if spp >= 32 else 'false'},{'true' if deep else 'false'}>"), name
    return sc, camera, prm


# scene, W, H, spp, depth: 1024 spp = 32 full batches per pixel; 97 = 3 full batches and one path; 7 = four pixels per task
FILM_CASES = [("init_cornell", 24, 16, 1024, 4), ("init_cornell", 32, 24, 97, 4), ("init_cornell", 32, 24, 7, 4),
              ("cornell_large_box", 24, 16, 1024, 4), ("cornell_large_box", 32, 24, 97, 4), ("cornell_large_box", 32, 24, 7, 4)]


@pytest.mark.parametrize("scene,w,h,spp,depth", FILM_CASES)
def test_film_matches_oracle(ctx, scene, w, h, spp, depth):
    """Sum, mean and M2 of every pixel within 2e-3 of the oracle's per-sample Welford film for at least 99 % of the pixels (the rest
    hold a path that took another branch in f32 geometry).  cornell_large_box sees its light directly: paths that end on the emitter,
    with and without shaded bounces."""
    sc, camera, prm = _setup(ctx, scene, w, h, spp, depth, 77)
    film = ctx.render_host(prm)
    o_sum, o_avg, o_m2, _, cnt = oracledriver.render_tile(sc, camera, prm, 0, 0, w, h)
    n = sc.num_wavelengths
    assert np.array_equal(film["filter"], np.full(w * h, spp, np.float32))
    for name, ref in (("sum", o_sum[:, :n]), ("mean", o_avg), ("m2", o_m2)):
        rel = _rel(film[name], ref, 1e-5 * np.abs(ref).max()).max(axis=1)
        print(f"\n{scene} {w}x{h}x{spp} {name}: pixels over 2e-3: {(rel > 2e-3).sum()} of {w * h}")
        assert (rel <= 2e-3).mean() >= 0.99, name


@pytest.mark.parametrize("scene,w,h,spp,depth,deep",
                         [c + (False,) for c in FILM_CASES] + [("cornell_large_box", 16, 12, 97, 100, True)])
def test_film_is_the_statistics_of_its_paths(ctx, scene, w, h, spp, depth, deep):
    """The film equals the sum, mean and M2 (f64) of the very paths the kernel dumps (drt_cuda_sample_paths writes E * r): the
    batched shifted sums lose nothing against a per-sample update.  Free of branch flips, so it holds for every pixel.  The depth-100
    case walks the overflow row in global memory before the shared-memory record."""
    sc, camera, prm = _setup(ctx, scene, w, h, spp, depth, 5, deep)
    film = ctx.render_host(prm)
    paths = ctx.sample_paths(prm, 0, 0, w, h).astype(np.float64)       # [pixels, spp, N]
    s = paths.sum(axis=1)
    m = s / spp
    m2 = ((paths - m[:, None, :]) ** 2).sum(axis=1)
    assert np.array_equal(film["filter"], np.full(w * h, spp, np.float32))
    lit = np.abs(paths).max(axis=(1, 2)) > 0
    assert np.array_equal(lit, np.abs(film["sum"]).max(axis=1) > 0)
    assert np.all(film["mean"][~lit] == 0) and np.all(film["m2"][~lit] == 0)   # an unlit pixel's film is exactly zero
    for name, ref, tol in (("sum", s, 1e-4), ("mean", m, 1e-4), ("m2", m2, 1e-3)):
        rel = _rel(film[name], ref, 1e-5 * np.abs(ref).max())
        print(f"\n{scene} {w}x{h}x{spp} {name}: max rel {rel.max():.2e}")
        assert rel.max() <= tol, name


@pytest.mark.parametrize("a,b", [(20, 48), (40, 97)])
def test_accumulate_composes(ctx, a, b):
    """Mode 1: rendering [0,a) and then accumulating [a,b) equals rendering [0,b) -- count exactly, planes to rounding."""
    import torch
    w, h, depth = 32, 24, 4
    cfg, tables, sc, camera = common.load("init_cornell", w, h, b, depth)
    ctx.upload_scene(sc, camera, tables)
    ctx.set_geometry_precision(cuda.GEOMETRY_F32)
    assert ctx.render_kernel_info(oracledriver.params(w, h, 0, b, depth, cfg.pixel_scheme, 5))[0] == "drt::render_kernel<float,5,1,true,false>"
    n = sc.num_wavelengths

    def planes():
        return [torch.zeros(w * h * n, device="cuda"), torch.zeros(w * h, device="cuda"),
                torch.zeros(w * h * n, device="cuda"), torch.zeros(w * h * n, device="cuda")]

    one, two = planes(), planes()
    ctx.render_device(oracledriver.params(w, h, 0, b, depth, cfg.pixel_scheme, 5), cuda.film_from_tensors(*one))
    ctx.render_device(oracledriver.params(w, h, 0, a, depth, cfg.pixel_scheme, 5), cuda.film_from_tensors(*two))
    ctx.render_device(oracledriver.params(w, h, a, b, depth, cfg.pixel_scheme, 5), cuda.film_from_tensors(*two), accumulate=True)
    torch.cuda.synchronize()
    assert torch.equal(one[1], two[1])
    for x, y in zip((one[0], one[2], one[3]), (two[0], two[2], two[3])):
        scale = float(x.abs().max())
        assert scale > 0
        assert float((x - y).abs().max()) <= 2e-5 * scale
