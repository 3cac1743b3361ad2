"""Phase-1 trims of the compact-record kernels (modes 1 and 2):

* the inline reduced-range sin / cos of pi u of the concentric disc map (sincospi_quarter in csrc/drt_render.cuh), modelled here in
  float32 with the coefficients read from the source, against float64 -- runs without a GPU;
* the direction sample of a bounce at the depth cap, which is never cast and is not drawn any more: per-path radiance and the work
  counters against the oracle at several depth caps, in the plastic-only, the classed and a deep render, and the record weights it
  leaves (GPU tier).
"""
import importlib
import os
import re

import numpy as np
import pytest

import common
import oracledriver

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUH = os.path.join(REPO, "daily-ray-trace_b200", "csrc", "drt_render.cuh")
F32 = np.float32

# ----------------------------------------------------------------------------------------------- CPU: sincospi_quarter


def _coefficients():
    """The float32 literals of sincospi_quarter, in source order: S3, S2, S1, S0, C4, C3, C2, C1."""
    src = open(CUH).read()
    body = re.search(r"void sincospi_quarter\(float u, float &s, float &c\)\s*\{(.*?)\n\}", src, re.S).group(1)
    lits = [F32(float.fromhex(x[:-1])) for x in re.findall(r"-?0x[0-9a-f.]+p[+-]\d+f", body)]
    assert len(lits) == 8, lits
    return lits


def _fma(a, b, c):
    """fmaf in float32: the product of two float32 values is exact in float64, then one rounding of the sum (twice: to f64, to f32)."""
    return (np.asarray(a, np.float64) * np.asarray(b, np.float64) + np.asarray(c, np.float64)).astype(F32)


def sincospi_quarter(u):
    """float32 model of sincospi_quarter's evaluation, operation by operation."""
    s3, s2, s1, s0, c4, c3, c2, c1 = _coefficients()
    u = np.asarray(u, F32)
    v = u * u
    ps = _fma(_fma(s3, v, s2), v, s1)
    s = _fma(u, s0, (u * v) * ps)
    pc = _fma(_fma(_fma(c4, v, c3), v, c2), v, c1)
    c = _fma(v, pc, F32(1))
    return s, c


def _ulps(got, ref):
    """|got - ref| in units of the float32 spacing at ref"""
    r = np.abs(ref).astype(F32)
    spacing = np.nextafter(r, F32(np.inf)).astype(np.float64) - r
    return np.abs(got.astype(np.float64) - ref) / spacing


def _near_quarter_and_zero():
    q = np.arange(0x3E800000 - (1 << 21), 0x3E800000 + 16, dtype=np.uint32).view(F32)   # 2M floats up to 1/4 and 16 past it
    z = np.arange(0, 0x3A000000, 97, dtype=np.uint32).view(F32)                           # +0, subnormals, up to 4.9e-4
    u = np.concatenate([q, z])
    return np.concatenate([u, -u])


@pytest.mark.parametrize("grid", ["dense", "near_quarter_and_zero"])
def test_sincospi_quarter_within_2_ulp(grid):
    u = np.linspace(-0.25, 0.25, 4_000_001, dtype=np.float64).astype(F32) if grid == "dense" else _near_quarter_and_zero()
    s, c = sincospi_quarter(u)
    x = np.pi * u.astype(np.float64)
    es, ec = _ulps(s, np.sin(x)), _ulps(c, np.cos(x))
    print(f"\n{grid}: {u.size} arguments, max error sin {es.max():.3f} ulp, cos {ec.max():.3f} ulp")
    assert es.max() <= 2.0 and ec.max() <= 2.0


def test_sincospi_quarter_swap_identity():
    """The steep octants of the disc map take sin and cos of pi (1/2 - u) as cos and sin of pi u.  Against float64 sin / cos of
    pi (1/2 - u) -- for |u| >= 2^-20, where rounding 1/2 - u and pi (1/2 - u) in float64 is far below a float32 ulp of the result."""
    u = np.linspace(-0.25, 0.25, 4_000_001, dtype=np.float64).astype(F32)
    u = np.concatenate([u, _near_quarter_and_zero()])
    u = u[np.abs(u) >= 2.0 ** -20]
    s, c = sincospi_quarter(u)
    x = np.pi * (0.5 - u.astype(np.float64))
    es, ec = _ulps(c, np.sin(x)), _ulps(s, np.cos(x))
    print(f"\nswap: max error sin {es.max():.3f} ulp, cos {ec.max():.3f} ulp")
    assert es.max() <= 2.0 and ec.max() <= 2.0


def test_coefficients_match_their_generator():
    import importlib.util
    spec = importlib.util.spec_from_file_location("fit_sincospi_quarter", os.path.join(REPO, "tools", "fit_sincospi_quarter.py"))
    fit = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(fit)
    s, c = fit.fit()
    s3, s2, s1, s0, c4, c3, c2, c1 = _coefficients()
    assert [s0, s1, s2, s3] == s and [c1, c2, c3, c4] == c


# ----------------------------------------------------------------------------------------------- GPU: the kernels against the oracle

REL_TOL = 1e-3


@pytest.fixture(scope="module")
def ctx():
    cuda = importlib.import_module("daily-ray-trace_b200.cuda")
    c = cuda.Context(0)
    yield c
    c.close()


def _parity(ctx, scene_name, w, h, tile, spp, depth, seed=0x7A11):
    cuda = importlib.import_module("daily-ray-trace_b200.cuda")
    cfg, tables, scene, camera = common.load(scene_name, w, h, spp, depth)
    ctx.upload_scene(scene, camera, tables)
    ctx.set_geometry_precision(cuda.GEOMETRY_F32)
    prm = oracledriver.params(w, h, 0, spp, depth, cfg.pixel_scheme, seed)
    x0, y0, x1, y1 = tile
    gpu = ctx.sample_paths(prm, x0, y0, x1, y1)
    st = ctx.stats()
    kernel = ctx.render_kernel_info(prm)[0]
    _, _, _, ref, cnt = oracledriver.render_tile(scene, camera, prm, x0, y0, x1, y1, want_paths=True)
    err = common.path_errors(gpu, ref)
    ok = (err <= REL_TOL).mean()
    print(f"\n{scene_name} depth {depth} [{kernel}]: {err.size} paths, within {REL_TOL:g}: {100 * ok:.3f} %, "
          f"rng draws {st.rng_draws} vs {cnt.rng_draws}, capped {st.reached_depth_cap}")
    assert ok >= 0.995
    assert st.paths == cnt.paths == err.size
    for a, b in ((st.closest_rays, cnt.closest_rays), (st.shadow_rays, cnt.shadow_rays), (st.rng_draws, cnt.rng_draws)):
        assert abs(a - b) <= 0.01 * b + 8
    return kernel, st


@pytest.mark.gpu
@pytest.mark.parametrize("depth", [1, 2, 4])
@pytest.mark.parametrize("scene", ["init_cornell", "cornell_plane_light"])
def test_depth_cap_parity(ctx, scene, depth):
    kernel, st = _parity(ctx, scene, 64, 48, (0, 0, 64, 48), 4, depth)
    assert kernel.split(",")[2] in ("1", "2"), kernel     # a compact-record kernel
    assert st.reached_depth_cap > 0


@pytest.mark.gpu
def test_classed_all_depth4(ctx):
    kernel, _ = _parity(ctx, "classed_all", 64, 48, (0, 0, 64, 48), 6, 4)
    assert kernel.split(",")[2] == "2", kernel


@pytest.mark.gpu
def test_deep_render_cap_in_overflow_row(ctx):
    """depth 40: the records overflow to global memory, and the capped bounce is written there"""
    _, st = _parity(ctx, "cornell_large_box", 48, 48, (8, 8, 40, 40), 8, 40)
    assert st.reached_depth_cap > 0


@pytest.mark.gpu
def test_capped_bounce_has_no_sampled_direction_weights(ctx):
    """init_cornell (plastic-only kernel, cosine sampler everywhere): a path that reaches the cap has sampled-direction weights 0 in its
    last bounce, and its first bounce has them (the diffuse weight is cos / pi x pi / cos x vignette > 0)"""
    depth, spp = 3, 4
    cfg, tables, scene, camera = common.load("init_cornell", 32, 32, spp, depth)
    ctx.upload_scene(scene, camera, tables)
    prm = oracledriver.params(32, 32, 0, spp, depth, cfg.pixel_scheme, 11)
    rec = ctx.debug_records(prm, 0, 0, 32, 32)
    words = rec.shape[-1]
    rec = rec.reshape(-1, words)
    head = words - 4 * depth
    nb = rec[:, 0] & 0xFFFF
    capped = rec[nb == depth].view(np.float32)
    assert len(capped) > 0
    last = capped[:, head + 4 * (depth - 1):head + 4 * depth]
    assert (last[:, 2:] == 0).all()
    first = capped[:, head:head + 4]
    assert (first[:, 2] > 0).all()
