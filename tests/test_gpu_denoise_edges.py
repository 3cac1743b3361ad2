"""GPU tier: drt_cuda_film_denoise (csrc/drt_denoise.cu) against the f64 reference of tests/denoise_ref.py where an indexing kernel goes
wrong: images narrower, shorter and smaller than a tile or the search window, every search and patch radius, every wavelength layout,
frames past 2^32 bytes of plane, extreme statistics, exact scaling, the ends of the strength range and calls on several streams.

The films are synthetic (film() below): a piecewise-smooth luminance of rectangles and gradients, per-wavelength noise independent from
pixel to pixel, counts of 2 to 64 and M2 consistent with the noise.  test_denoise_reference.py checks that these films make the
reference's weights informative and that each plausible indexing slip moves the output far beyond the tolerance of _agree().  Nothing
here reads the kernel's tile shape: this file is the acceptance suite of a rewrite of the filter kernel (DESIGN.md section 9)."""
import importlib

import numpy as np
import pytest

import common
import denoise_ref
import test_wavelength_grids_model as grids

cuda = importlib.import_module("daily-ray-trace_b200.cuda")

pytestmark = pytest.mark.gpu

GRID = {**{n: (lo, hi, step) for n, ns, lo, hi, step in grids.RENDER_GRIDS}, **{n: (lo, hi, step) for n, lo, hi, step in grids.EPILOGUE_GRIDS}}
WIDTHS = [1, 2, 5, 31, 32, 33, 65, 100]
HEIGHTS = [1, 2, 3, 4, 5, 8, 9, 15, 16, 17, 33]
SHAPE_RADII = [(1, 0), (7, 3), (15, 4)]
LAYOUT_RADII = [(7, 3), (3, 1)]
E_ARG = -103


def film(width, height, n, seed, device="cpu", rel=0.5, band=512):
    """A seeded synthetic film of width x height pixels and n wavelengths: {"mean": [W*H, N], "m2": [W*H, N], "filter": [W*H]} as f32
    numpy arrays (device "cpu") or torch tensors on `device`, generated in bands of `band` rows.  rel is the relative standard deviation
    of one sample."""
    import torch
    rng = np.random.default_rng(seed)
    rects = []
    for _ in range(4):
        x0, x1 = np.sort(rng.integers(0, width + 1, 2))
        y0, y1 = np.sort(rng.integers(0, height + 1, 2))
        rects.append((x0, x1, y0, y1, rng.uniform(0.3, 3.0), rng.uniform(-1, 1, 2), rng.uniform(-1, 1)))
    fx, fy, px, py = rng.uniform(0.9, 1.7), rng.uniform(0.7, 1.3), rng.uniform(0, 6.3), rng.uniform(0, 6.3)
    gen = torch.Generator(device=device).manual_seed(seed)
    f32 = dict(dtype=torch.float32, device=device)
    lw = torch.linspace(-1.0, 1.0, n, **f32)
    shape = 1.0 + 0.3 * torch.sin(3.1 * lw)
    mean, m2 = torch.empty(width * height, n, **f32), torch.empty(width * height, n, **f32)
    cnt = torch.empty(width * height, **f32)
    for b0 in range(0, height, band):
        b1 = min(height, b0 + band)
        yy, xx = torch.meshgrid(torch.arange(b0, b1, **f32), torch.arange(width, **f32), indexing="ij")
        lum = 1.0 + 0.8 * xx / width + 0.4 * yy / height
        tilt = torch.zeros_like(lum)
        for x0, x1, y0, y1, level, g, t in rects:
            m = (xx >= x0) & (xx < x1) & (yy >= y0) & (yy < y1)
            ramp = level * (1.0 + 0.3 * (g[0] * (xx - x0) / max(x1 - x0, 1) + g[1] * (yy - y0) / max(y1 - y0, 1)))
            lum, tilt = torch.where(m, ramp, lum), torch.where(m, torch.full_like(tilt, t), tilt)
        lum = lum * (1.0 + 0.25 * torch.sin(fx * xx + px) * torch.sin(fy * yy + py))
        base = lum.reshape(-1, 1) * (1.0 + 0.5 * tilt.reshape(-1, 1) * lw) * shape
        c = torch.randint(2, 65, (base.shape[0],), generator=gen, device=device).to(torch.float32)
        sd = rel * base
        s = slice(b0 * width, b1 * width)
        mean[s] = base + sd * torch.randn(base.shape, generator=gen, **f32) / c.sqrt()[:, None]
        m2[s] = sd * sd * (c - 1.0)[:, None] * (0.5 + torch.rand(base.shape, generator=gen, **f32))
        cnt[s] = c
    if device == "cpu":
        return {"mean": mean.numpy(), "m2": m2.numpy(), "filter": cnt.numpy()}
    return {"mean": mean, "m2": m2, "filter": cnt}


def shape_seed(w, h):
    return 1000 + 7 * w + h


@pytest.fixture(scope="module")
def ctx():
    c = cuda.Context(0)
    yield c
    c.close()


def _scene(c, n):
    """Upload a scene of n wavelengths to c (if it holds another N); returns the luminance weights of the filter."""
    grid = {} if n == 69 else dict(zip(("min_wl", "max_wl", "wl_interval"), GRID[n]))
    cfg, tables, sc, camera = common.load("init_cornell", 8, 8, 1, 4, **grid)
    assert sc.num_wavelengths == n
    if getattr(c, "_denoise_n", None) != n:
        c.upload_scene(sc, camera, tables)
        c._denoise_n = n
    return denoise_ref.luminance_weights(tables, n)


def _agree(out, ref, mean, usable):
    """The criteria of test_gpu_denoise._check: usable values within 1e-4 relative (floor 1e-6 of the peak) for >= 99.9 % and 1e-3 for
    all; unusable pixels copied bit for bit."""
    out, mean = np.asarray(out).reshape(ref.shape), np.asarray(mean).reshape(ref.shape)
    assert np.array_equal(out[~usable].view(np.uint32), mean[~usable].view(np.uint32))
    if not usable.any():
        return 0.0
    floor = 1e-6 * float(np.abs(ref[usable]).max())
    rel = np.abs(out[usable].astype(np.float64) - ref[usable]) / np.maximum(np.abs(ref[usable]), floor)
    assert np.quantile(rel, 0.999) <= 1e-4 and rel.max() <= 1e-3, (np.quantile(rel, 0.999), rel.max())
    return float(rel.max())


def _check(c, f, w, h, yw, r=7, f_=3, k=0.45):
    out = c.film_denoise_host(f, w, h, search_radius=r, patch_radius=f_, strength=k)
    ref = denoise_ref.denoise(f["mean"], f["m2"], f["filter"], yw, w, h, r=r, f=f_, k=np.float32(k))
    usable = denoise_ref.guide(f["mean"], f["m2"], f["filter"], yw)[2]
    _agree(out, ref, f["mean"], usable)
    return out, usable


@pytest.mark.parametrize("r,f", SHAPE_RADII)
@pytest.mark.parametrize("h", HEIGHTS)
@pytest.mark.parametrize("w", WIDTHS)
def test_shapes(ctx, w, h, r, f):
    """Images narrower and shorter than a tile, of 1 to 3 rows, smaller than the search window, and just either side of 32 columns and
    of 4, 8 and 16 rows."""
    yw = _scene(ctx, 18)
    _check(ctx, film(w, h, 18, shape_seed(w, h)), w, h, yw, r, f)


@pytest.mark.parametrize("f", range(5))
@pytest.mark.parametrize("r", range(1, 16))
def test_radii(ctx, r, f):
    yw = _scene(ctx, 69)
    _check(ctx, film(45, 19, 69, 19), 45, 19, yw, r, f)


@pytest.mark.parametrize("r,f", LAYOUT_RADII)
@pytest.mark.parametrize("n", sorted(GRID))
def test_wavelength_layouts(ctx, n, r, f):
    """Every N of the render and epilogue grids: every residue of N mod 4 and one to four groups of 32 wavelengths."""
    yw = _scene(ctx, n)
    _check(ctx, film(41, 13, n, 500 + n), 41, 13, yw, r, f)


def _device_film(f):
    return cuda.Film(None, f["filter"].data_ptr(), f["mean"].data_ptr(), f["m2"].data_ptr())


def _windows_agree(f, out, yw, w, h, windows, n):
    for x0, y0, x1, y1 in windows:
        ref = denoise_ref.denoise_window(f["mean"], f["m2"], f["filter"], yw, w, h, x0, y0, x1, y1, r=7, f=3, k=np.float32(0.45))
        sub = lambda p: denoise_ref.host_array(p.reshape(h, w, -1)[y0:y1, x0:x1]).reshape((y1 - y0) * (x1 - x0), -1)
        mean = sub(f["mean"])
        usable = denoise_ref.guide(mean, sub(f["m2"]), sub(f["filter"]).reshape(-1), yw)[2]
        got = sub(out.reshape(w * h, n))
        err = _agree(got, ref, mean, usable)
        print(f"  window x {x0}..{x1} y {y0}..{y1}: rel error max {err:.2e}")


def test_1024_square_windows(ctx):
    import torch
    yw = _scene(ctx, 69)
    w = h = 1024
    f = film(w, h, 69, 1024, device="cuda")
    out = ctx.film_denoise(_device_film(f), w, h)
    torch.cuda.synchronize()
    s = 40
    _windows_agree(f, out, yw, w, h, [(0, 0, s, s), (w - s, 0, w, s), (0, h - s, s, h), (w - s, h - s, w, h),
                                      (512 - s // 2, 300, 512 + s // 2, 300 + s), (w // 2 - s // 2, h // 2 - s // 2, w // 2 + s // 2, h // 2 + s // 2)], 69)


def test_4096_square_windows(ctx):
    """Planes of 4.6 GB: offsets past 2^32 bytes."""
    import torch
    free, _ = torch.cuda.mem_get_info()
    if free < 20 * 2 ** 30:
        pytest.skip("needs 20 GB of free device memory")
    yw = _scene(ctx, 69)
    w = h = 4096
    f = film(w, h, 69, 4096, device="cuda")
    out = ctx.film_denoise(_device_film(f), w, h)
    torch.cuda.synchronize()
    s = 32
    _windows_agree(f, out, yw, w, h, [(0, 0, s, s), (w - s, 0, w, s), (0, h - s, s, h), (w - s, h - s, w, h),
                                      (1000, h - 3, 1000 + 2 * s, h)], 69)
    del f, out
    torch.cuda.empty_cache()


def test_extreme_statistics(ctx):
    """Counts of 0, 1, 2, inf and NaN; -0.0 in mean and M2; one tiny negative M2; a zero-variance region where the 1e-10 floor decides;
    a usable pixel among unusable ones; a checkerboard of unusable pixels."""
    n, w, h = 18, 40, 24
    yw = _scene(ctx, n)
    f = film(w, h, n, 77)
    mean, m2, cnt = f["mean"], f["m2"], f["filter"]
    at = lambda x, y: y * w + x
    cnt[at(3, 3)], cnt[at(4, 3)], cnt[at(5, 3)], cnt[at(6, 3)], cnt[at(7, 3)] = 0.0, 1.0, 2.0, np.inf, np.nan
    mean[at(10, 2), 4] = -0.0
    m2[at(11, 2), :] = -0.0
    m2[at(12, 5), 7] = -1e-30                                 # a single tiny negative M2
    # a zero-variance region: equal spectra, M2 = 0, v = 0 for every pair inside it
    zy, zx = np.mgrid[14:20, 2:12]
    zero = (zy * w + zx).ravel()
    mean[zero] = mean[at(2, 14)]
    m2[zero] = 0.0
    mean[at(5, 16)] *= 1.0 + 1e-6                             # one pixel of the region a little apart: only the floor weighs it
    # a usable pixel whose neighbours within r = 7 are all unusable
    iy, ix = np.mgrid[2:20, 22:40]
    iso = (iy * w + ix).ravel()
    cnt[iso] = 1.0
    cnt[at(31, 10)] = 16.0
    # a checkerboard of unusable pixels in the last rows
    cy, cx = np.mgrid[20:24, 0:w]
    cnt[(cy * w + cx).ravel()[((cy + cx) % 2 == 1).ravel()]] = 1.0
    out, usable = _check(ctx, f, w, h, yw)
    assert usable[at(5, 3)] and usable[at(6, 3)] and usable[at(12, 5)] and usable[at(31, 10)]
    assert not usable[[at(3, 3), at(4, 3), at(7, 3)]].any()
    assert np.array_equal(out[at(31, 10)].view(np.uint32), mean[at(31, 10)].view(np.uint32))
    assert np.isfinite(out[usable]).all()


def test_negative_m2_counts_as_zero_variance(ctx):
    """A negative M2 value gives the guide no NaN: its pixel keeps a finite v and no pixel around it takes a weight of 1 from NaN."""
    n, w, h = 69, 37, 21
    yw = _scene(ctx, n)
    f = film(w, h, n, 88)
    f["m2"][10 * w + 17, 30] = -5.0
    out, usable = _check(ctx, f, w, h, yw)
    assert usable[10 * w + 17] and np.isfinite(out).all()


def test_guide_overflow(ctx):
    """Finite statistics near the top of the f32 range.  Columns 10..15: mean x 1e17, count 2 and M2 1e38, so v lies beyond FLT_MAX:
    unusable, copied bit for bit, and no other pixel takes them in.  Columns 20..25: mean x 1e25 with small M2, usable, whose luminance differences
    overflow f32 when squared.  Columns 32..37: mean x 1e12, M2 x 1e24, usable.  Every usable output is finite."""
    n, w, h = 69, 48, 20
    yw = _scene(ctx, n)
    f = film(w, h, n, 99)
    col = np.arange(w * h) % w
    vbig, huge, big = (col >= 10) & (col < 16), (col >= 20) & (col < 26), (col >= 32) & (col < 38)
    for m, sm, s2 in ((huge, 1e25, 1e12), (big, 1e12, 1e24)):
        f["mean"][m] *= np.float32(sm)
        f["m2"][m] *= np.float32(s2)
    f["mean"][vbig] *= np.float32(1e17)
    f["m2"][vbig], f["filter"][vbig] = 1e38, 2.0
    assert np.isfinite(f["mean"]).all() and np.isfinite(f["m2"]).all()
    out, usable = _check(ctx, f, w, h, yw)
    assert not usable[vbig].any() and usable[huge].all() and usable[big].all()
    assert np.isfinite(out[usable]).all()


def test_scale_is_exact(ctx):
    """mean x 2^k and M2 x 2^2k give out x 2^k bit for bit (film with v >= 1: the 1e-10 floor is absorbed, the weights are unchanged)."""
    n, w, h = 69, 45, 19
    yw = _scene(ctx, n)
    f = film(w, h, n, 123)
    v = denoise_ref.guide(f["mean"], f["m2"], f["filter"], yw)[1]
    c = np.float32(2.0 ** np.ceil(-0.5 * np.log2(v.min())))
    f["mean"], f["m2"] = f["mean"] * c, f["m2"] * c * c
    assert denoise_ref.guide(f["mean"], f["m2"], f["filter"], yw)[1].min() >= 1.0
    base = ctx.film_denoise_host(f, w, h)
    for k in (8, 16, 24):
        s = np.float32(2.0 ** k)
        out = ctx.film_denoise_host({"mean": f["mean"] * s, "m2": f["m2"] * s * s, "filter": f["filter"]}, w, h)
        want = base * s
        ulp = np.abs(out.view(np.int32).astype(np.int64) - want.view(np.int32).astype(np.int64))
        print(f"  k = {k}: max difference {int(ulp.max())} ulp")
        assert np.array_equal(out.view(np.uint32), want.view(np.uint32))


def test_strength_limits(ctx):
    """strength^2 must be a normal f32: strength in [2^-63, 2^64).  Just outside returns DRT_CUDA_E_ARG naming strength; the two ends
    match the reference."""
    n, w, h = 18, 33, 9
    yw = _scene(ctx, n)
    f = film(w, h, n, 5)
    lo, hi = np.float32(2.0 ** -63), np.nextafter(np.float32(2.0 ** 64), np.float32(0))
    assert np.isfinite(hi * hi) and lo * lo >= np.finfo(np.float32).tiny
    for k in (np.nextafter(lo, np.float32(0)), np.float32(2.0 ** 64), np.float32(1e20), np.float32(1e-30)):
        with pytest.raises(cuda.CudaError) as e:
            ctx.film_denoise_host(f, w, h, strength=float(k))
        assert e.value.code == E_ARG and "strength" in str(e.value), str(e.value)
    # a zero-variance pair where the floor alone is the denominator
    f["m2"][:w] = 0.0
    f["mean"][1:w] = f["mean"][0]
    for k in (lo, hi):
        _check(ctx, f, w, h, yw, 7, 3, float(k))


def _solo(c, f, w, h):
    import torch
    out = c.film_denoise(_device_film(f), w, h)
    torch.cuda.synchronize()
    return out


def test_two_streams(ctx):
    """Two same-size films on two streams, queued back to back: each output equals the output of the same call made alone."""
    import torch
    _scene(ctx, 69)
    w = h = 1024
    a, b = film(w, h, 69, 31, device="cuda"), film(w, h, 69, 32, device="cuda")
    want_a, want_b = _solo(ctx, a, w, h), _solo(ctx, b, w, h)
    out_a, out_b = torch.full_like(want_a, float("nan")), torch.full_like(want_b, float("nan"))
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    ctx.film_denoise(_device_film(a), w, h, out=out_a.data_ptr(), stream=s1.cuda_stream)
    ctx.film_denoise(_device_film(b), w, h, out=out_b.data_ptr(), stream=s2.cuda_stream)
    torch.cuda.synchronize()
    assert torch.equal(out_a.view(torch.int32), want_a.view(torch.int32))
    assert torch.equal(out_b.view(torch.int32), want_b.view(torch.int32))


def test_small_large_small(ctx):
    """One context filters a small film, a large one and the small one again: each output equals a fresh context's, bit for bit."""
    _scene(ctx, 69)
    small, large = film(41, 13, 69, 7), film(512, 384, 69, 8)
    got = [ctx.film_denoise_host(small, 41, 13), ctx.film_denoise_host(large, 512, 384), ctx.film_denoise_host(small, 41, 13)]
    for out, (f, w, h) in zip(got, [(small, 41, 13), (large, 512, 384), (small, 41, 13)]):
        fresh = cuda.Context(0)
        try:
            _scene(fresh, 69)
            want = fresh.film_denoise_host(f, w, h)
        finally:
            fresh.close()
        assert np.array_equal(out.view(np.uint32), want.view(np.uint32))
