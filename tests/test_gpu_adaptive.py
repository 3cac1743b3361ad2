"""GPU tier: adaptive sampling (drt_cuda_render_host_adaptive / _device_adaptive, render_kernel_adaptive).

A pixel takes batches of 32 samples and stops at the end of the first batch after which n >= min_samples and
err = sum_l w_l sqrt(M2_l / (n (n - 1))) <= rel_error * Y, Y = sum_l w_l mean_l (w = cmf_y * ref_white), or when the call's samples
run out.  Sample s of a pixel is the same path as in a uniform render, so these tests dump the paths of the whole range with
sample_paths (the kernel's own paths: f32 branch flips do not matter), and check that every pixel's film is the statistics of a prefix
of them and that the prefix ends where the rule, evaluated in f64 on the same paths, says it does."""
import importlib
import os
import subprocess

import numpy as np
import pytest

import common
import oracledriver
import refdriver
import test_converged

cuda = importlib.import_module("daily-ray-trace_b200.cuda")

pytestmark = pytest.mark.gpu

BIN = os.path.join(common.REPO, "daily-ray-trace_b200", "drt_raytrace")


@pytest.fixture(scope="module")
def ctx():
    c = cuda.Context(0)
    yield c
    c.close()


def _setup(ctx, scene, w, h, cap, depth, seed):
    cfg, tables, sc, camera = common.load(scene, w, h, cap, depth)
    ctx.upload_scene(sc, camera, tables)
    ctx.set_geometry_precision(cuda.GEOMETRY_F32)
    prm = oracledriver.params(w, h, 0, cap, depth, cfg.pixel_scheme, seed)
    n = sc.num_wavelengths
    # the weights as the device holds them: (float)(cmf_y * ref_white), drt_fill_rgb_tables
    yw = (np.array(tables.cmf_y[:n]) * np.array(tables.ref_white[:n])).astype(np.float32).astype(np.float64)
    return sc, prm, yw


def _rel(a, b, floor):
    return np.abs(a.astype(np.float64) - b) / np.maximum(np.abs(b), floor)


def _prefix_stats(paths, counts):
    """f64 sum, mean and M2 of paths [0, n_p) of every pixel."""
    s = np.zeros((paths.shape[0], paths.shape[2]))
    m2 = np.zeros_like(s)
    for p, k in enumerate(counts.astype(np.int64)):
        x = paths[p, :k]
        s[p] = x.sum(axis=0)
        m2[p] = ((x - s[p] / k) ** 2).sum(axis=0)
    return s, s / counts[:, None], m2


def _check_prefix(film, paths, counts):
    """The film of every pixel is the statistics of its first counts[p] dumped paths."""
    s, m, m2 = _prefix_stats(paths, counts)
    for name, ref, tol in (("sum", s, 1e-4), ("mean", m, 1e-4), ("m2", m2, 1e-3)):
        rel = _rel(film[name], ref, 1e-5 * max(np.abs(ref).max(), 1e-30))
        print(f"  {name}: max rel {rel.max():.2e}")
        assert rel.max() <= tol, name


def _rule(paths, yw, rel_error, min_samples, begin, cap):
    """f64 stopping rule at every batch end of a call over samples [begin, cap), with `paths` the paths [0, cap) of every pixel (those
    before `begin` are the film an accumulating call loaded): (batch ends, stop[pixel, end], ratio err / (rel_error Y))."""
    b = np.array(sorted(set(range(begin + 32, cap, 32)) | {cap}))
    c1 = np.cumsum(paths, axis=1)[:, b - 1]                      # [pixels, batch ends, N]
    c2 = np.cumsum(paths * paths, axis=1)[:, b - 1]
    n = b.astype(np.float64)[None, :, None]
    y = (c1 / n) @ yw
    err = np.sqrt(np.maximum(c2 - c1 * c1 / n, 0.0) / (n * (n - 1))) @ yw
    with np.errstate(invalid="ignore", divide="ignore"):
        ratio = err / (rel_error * y)
    stop = (b[None, :] >= min_samples) & (err <= rel_error * y)
    return b, stop, ratio


def _check_rule(counts, paths, yw, rel_error, min_samples, begin, cap):
    """Every pixel stopped at the first batch end where the rule holds, or at the cap.  A disagreement is allowed only where the f64
    ratio err / (rel_error Y) at the disputed batch end is within 1e-3 of 1 (the kernel evaluates the rule in f32)."""
    b, stop, ratio = _rule(paths, yw, rel_error, min_samples, begin, cap)
    disputed = 0
    for p, c in enumerate(counts.astype(np.int64)):
        k = int(np.searchsorted(b, c))
        assert k < len(b) and b[k] == c, (p, c)
        # went on past every earlier batch end and stopped at b[k] (unless b[k] is the cap)
        want = np.concatenate([~stop[p, :k], [stop[p, k]] if c < cap else []]).astype(bool)
        if not want.all():
            assert np.all(np.abs(ratio[p, :len(want)][~want] - 1.0) <= 1e-3), (p, c, ratio[p, :len(want)][~want])
            disputed += 1
    print(f"  pixels whose stop only f32 rounding explains: {disputed} of {len(counts)}")


# scene, W, H, cap, depth, rel_error, min_samples, kernel mode
CASES = [("init_cornell", 16, 12, 2048, 4, 0.05, 64, 1),
         ("cornell_plane_light", 16, 12, 2048, 4, 0.05, 64, 2),
         ("classed_all", 16, 12, 2048, 4, 0.05, 64, 2),
         ("stress_all", 16, 12, 2048, 4, 0.05, 64, 0),
         ("sky_cornell", 16, 12, 2048, 4, 0.05, 64, 0),
         ("cornell_large_box", 16, 12, 1024, 100, 0.05, 64, 1),
         ("init_cornell", 16, 12, 1000, 4, 0.02, 96, 1)]


@pytest.mark.parametrize("scene,w,h,cap,depth,rel_error,min_samples,mode", CASES)
def test_adaptive_film_is_the_prefix_the_rule_picks(ctx, scene, w, h, cap, depth, rel_error, min_samples, mode):
    sc, prm, yw = _setup(ctx, scene, w, h, cap, depth, 31)
    name = ctx.render_kernel_info(prm)[0]
    assert name.split(",")[2] == str(mode) and name.endswith(",true,true>" if depth == 100 else ",true,false>"), name
    film = ctx.render_host_adaptive(prm, rel_error, min_samples)
    paths_taken = ctx.stats().paths
    counts = film["filter"].astype(np.float64)
    print(f"\n{scene} {w}x{h} cap {cap}: counts {counts.min():.0f}..{counts.max():.0f}, mean {counts.mean():.1f}")
    assert np.all((counts == cap) | ((counts % 32 == 0) & (counts >= min_samples)))
    assert len(np.unique(counts)) > 1                              # it adapts
    assert paths_taken == int(counts.sum())
    paths = ctx.sample_paths(prm, 0, 0, w, h).astype(np.float64)   # [pixels, cap, N]
    _check_prefix(film, paths, counts)
    _check_rule(counts, paths, yw, rel_error, min_samples, 0, cap)


def test_large_rel_error_gives_min_samples(ctx):
    """Every pixel stops at min_samples, and the film is the uniform render of [0, min_samples)."""
    w, h, mn = 24, 16, 64
    sc, prm, _ = _setup(ctx, "cornell_plane_light", w, h, 1024, 4, 3)
    film = ctx.render_host_adaptive(prm, 1e30, mn)
    assert np.array_equal(film["filter"], np.full(w * h, mn, np.float32))
    assert ctx.stats().paths == w * h * mn
    prm.sample_end = mn
    ref = ctx.render_host(prm)
    for k in ("sum", "mean", "m2"):
        scale = float(np.abs(ref[k]).max())
        assert scale > 0
        assert float(np.abs(film[k] - ref[k]).max()) <= 2e-5 * scale, k


def test_accumulate_continues_a_uniform_film(ctx):
    """Uniform [0, 256), then adaptive [256, 2048) with accumulate=1: each film is the statistics of paths [0, n_p), and the rule
    counts the loaded samples."""
    import torch
    w, h, a, cap, rel_error, mn = 16, 12, 256, 2048, 0.02, 64
    sc, prm, yw = _setup(ctx, "init_cornell", w, h, cap, 4, 9)
    n = sc.num_wavelengths
    planes = [torch.zeros(w * h * n, device="cuda"), torch.zeros(w * h, device="cuda"),
              torch.zeros(w * h * n, device="cuda"), torch.zeros(w * h * n, device="cuda")]
    f = cuda.film_from_tensors(*planes)
    first = oracledriver.params(w, h, 0, a, 4, prm.pixel_scheme, 9)
    rest = oracledriver.params(w, h, a, cap, 4, prm.pixel_scheme, 9)
    ctx.render_device(first, f)
    ctx.render_device_adaptive(rest, rel_error, mn, f, accumulate=True)
    taken = ctx.stats().paths
    torch.cuda.synchronize()
    film = {"sum": planes[0].cpu().numpy().reshape(w * h, n), "filter": planes[1].cpu().numpy(),
            "mean": planes[2].cpu().numpy().reshape(w * h, n), "m2": planes[3].cpu().numpy().reshape(w * h, n)}
    counts = film["filter"].astype(np.float64)
    print(f"\naccumulate: counts {counts.min():.0f}..{counts.max():.0f}")
    assert np.all((counts == cap) | ((counts - a) % 32 == 0)) and np.all(counts > a)
    assert len(np.unique(counts)) > 1 and taken == int((counts - a).sum())
    paths = ctx.sample_paths(prm, 0, 0, w, h).astype(np.float64)     # [0, cap)
    _check_prefix(film, paths, counts)
    _check_rule(counts, paths, yw, rel_error, mn, a, cap)


def test_host_bands_match_device(ctx):
    """render_host_adaptive on a frame large enough for the six-band read-back gives the counts of render_device_adaptive."""
    import torch
    w, h, cap, rel_error, mn = 256, 256, 1024, 0.05, 64
    sc, prm, _ = _setup(ctx, "cornell_plane_light", w, h, cap, 4, 21)
    n = sc.num_wavelengths
    assert w * h * cap >= 1 << 26
    host = ctx.render_host_adaptive(prm, rel_error, mn)
    host_paths = ctx.stats().paths
    assert ctx.stats().kernel_launches == 6
    planes = [torch.zeros(w * h * n, device="cuda"), torch.zeros(w * h, device="cuda"),
              torch.zeros(w * h * n, device="cuda"), torch.zeros(w * h * n, device="cuda")]
    ctx.render_device_adaptive(prm, rel_error, mn, cuda.film_from_tensors(*planes))
    dev_paths = ctx.stats().paths
    torch.cuda.synchronize()
    assert np.array_equal(host["filter"], planes[1].cpu().numpy())
    assert host_paths == dev_paths == int(host["filter"].astype(np.int64).sum())
    assert len(np.unique(host["filter"])) > 1
    for k, t in (("sum", planes[0]), ("mean", planes[2]), ("m2", planes[3])):
        d = t.cpu().numpy().reshape(w * h, n)
        scale = float(np.abs(d).max())
        assert float(np.abs(host[k] - d).max()) <= 1e-6 * scale, k


@pytest.mark.parametrize("name", test_converged.CASES)
def test_adaptive_image_within_noise_of_reference(ctx, name):
    """The adaptive image of the converged-reference tiles passes the uniform renders' noise bound, with per-pixel counts n_p in
    sigma^2 = var (1 / n_p + 1 / K_ref)."""
    w, h, k_ref, depth, ref_mean = test_converged._fixture(name)
    cfg, tables, sc, camera = common.load(name, w, h, 4096, depth)
    ctx.upload_scene(sc, camera, tables)
    ctx.set_geometry_precision(cuda.GEOMETRY_F32)
    film = ctx.render_host_adaptive(oracledriver.params(w, h, 0, 4096, depth, cfg.pixel_scheme, 778), 0.01, 64)
    counts = film["filter"].astype(np.float64)
    print(f"\n{name}: counts {counts.min():.0f}..{counts.max():.0f}, mean {counts.mean():.1f}")
    test_converged._check(name + " adaptive", counts[:, None], film["mean"], film["m2"], ref_mean, k_ref)


def test_adaptive_error_codes(ctx):
    w, h = 8, 8
    sc, prm, _ = _setup(ctx, "init_cornell", w, h, 256, 4, 1)
    bad = [(0.0, 64, prm), (-0.1, 64, prm), (float("nan"), 64, prm), (float("inf"), 64, prm), (0.05, 31, prm), (0.05, 257, prm),
           (0.05, 32, oracledriver.params(w, h, 0, 16, 4, prm.pixel_scheme, 1))]
    for rel_error, mn, p in bad:
        with pytest.raises(cuda.CudaError) as e:
            ctx.render_host_adaptive(p, rel_error, mn)
        assert e.value.code == -103, (rel_error, mn, str(e.value))
        assert "rel_error" in str(e.value) or "min_samples" in str(e.value)
    ctx.set_geometry_precision(cuda.GEOMETRY_F64)
    try:
        with pytest.raises(cuda.CudaError) as e:
            ctx.render_host_adaptive(prm, 0.05, 64)
        assert e.value.code == -104 and "f64" in str(e.value)
    finally:
        ctx.set_geometry_precision(cuda.GEOMETRY_F32)


def test_linux_main_adaptive(host, tmp_path):
    """`drt_raytrace --adaptive 0.02` writes .spd files whose per-pixel counts (the filter column) vary and stay within the cap."""
    if not os.path.exists(BIN):
        pytest.fail("drt_raytrace is not built (make -C daily-ray-trace_b200)")
    root = refdriver.make_root(str(tmp_path), common.ASSETS)
    w, h, spp, n = 40, 24, 512, 69
    open(os.path.join(root, "config.cfg"), "w").write(host.make_config_text(scene="scenes\\init_cornell.scn", width=w, height=h, spp=spp))
    out = subprocess.run([BIN, "--seed", "3", "--adaptive", "0.02"], cwd=root, check=True, capture_output=True, text=True).stdout
    assert "Render complete." in out and "Converted." in out and "samples per pixel" in out
    body = np.frombuffer(open(os.path.join(root, "output", "output.spd"), "rb").read()[40:], dtype=np.float64).reshape(w * h, n + 1)
    counts = body[:, n]
    assert counts.max() <= spp and counts.min() >= 64 and len(np.unique(counts)) > 1
    for k in ("output.bmp", "average.bmp", "variance.bmp"):
        assert open(os.path.join(root, "output", k), "rb").read()[:2] == b"BM"
