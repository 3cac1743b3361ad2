"""GPU tier: the render kernels and the film epilogues at every wavelength-slot layout, not only the 69-wavelength default.

The render kernel is instantiated for NS = 2, 3, 5 and 8 slots per lane of a half warp (a lane holds wavelengths l16 + 16 k), for
three modes (0 general, 1 plastic-only, 2 classed), two task shapes (spp >= 32: one pixel per task, "paired"; fewer: several pixels per
task) and shallow / deep records; the adaptive kernel for every mode, NS and depth class.  The compact-record kernels (modes 1, 2)
treat slot pairs and, for odd NS, a last single slot separately (BatchStats, PixelFilm::add_batch, the light's E in light_pairs), so a
lane or pair mapping that is wrong only for even NS passes every test at N = 69.  The film epilogues hold wavelengths lane + 32 k in up
to four slots.  The grids are those of tests/test_wavelength_grids_model.py, which checks their N and NS without a GPU.

  (a) every f32 instantiation: the film is the f64 statistics of the kernel's own dumped paths (adaptive: of the prefix the f64
      stopping rule picks) -- free of f32 branch flips;
  (b) per mode and NS, three cases against the oracle with the allowances of test_gpu_parity.py / test_deep_paths, and f64 geometry;
  (c) the same paths on different grids are the same at the wavelengths the grids share (bit-identical up to branch flips);
  (d) film_to_rgb, film_merge, film_merge_many, film_merge_slices(_local) and film_read_slice against float64 on synthetic films."""
import ctypes as C
import importlib
import math

import numpy as np
import pytest

import common
import oracledriver
import test_gpu_adaptive
import test_wavelength_grids_model as grids

cuda = importlib.import_module("daily-ray-trace_b200.cuda")
film_mod = importlib.import_module("daily-ray-trace_b200.film")

pytestmark = pytest.mark.gpu

GRID = {n: (lo, hi, step) for n, ns, lo, hi, step in grids.RENDER_GRIDS}
GRID.update({n: (lo, hi, step) for n, lo, hi, step in grids.EPILOGUE_GRIDS})
NS_GRIDS = {2: (2, 32), 3: (33, 48), 5: (69, 80), 8: (81, 128)}      # two grids per NS: a partial and a full last slot
SCENES = {1: ("init_cornell", "cornell_large_box"), 2: ("cornell_plane_light", "classed_all"), 0: ("stress_all", "sky_cornell")}
DEEP_DEPTHS = (24, 48, 64, 100, 160)
SHALLOW_DEPTHS = (4, 3, 2)       # at NS = 8 a general or classed record with 4 bounces already overflows shared memory
SEEN = set()               # instantiation names the tests below launched
SEEN_ADAPTIVE = set()
RAN = set()                # (a) cases that ran (the coverage check needs the whole module)


@pytest.fixture(scope="module")
def ctx():
    c = cuda.Context(0)
    yield c
    c.close()


def _load(ctx, scene, n, w, h, spp, depth):
    lo, hi, step = GRID[n]
    cfg, tables, sc, camera = common.load(scene, w, h, spp, depth, min_wl=lo, max_wl=hi, wl_interval=step)
    assert sc.num_wavelengths == n
    ctx.upload_scene(sc, camera, tables)
    ctx.set_geometry_precision(cuda.GEOMETRY_F32)
    return cfg, tables, sc, camera


def _shallow_depth(ctx, cfg, w, h, spp):
    """The largest of SHALLOW_DEPTHS whose records fit in shared memory."""
    for d in SHALLOW_DEPTHS:
        if ctx.render_kernel_info(oracledriver.params(w, h, 0, spp, d, cfg.pixel_scheme, 1))[0].endswith(",false>"):
            return d
    pytest.fail(f"no depth of {SHALLOW_DEPTHS} gives a shallow record")


def _deep_depth(ctx, cfg, w, h, spp):
    """The smallest of DEEP_DEPTHS whose records overflow shared memory (it depends on NS through the parked film)."""
    for d in DEEP_DEPTHS:
        if ctx.render_kernel_info(oracledriver.params(w, h, 0, spp, d, cfg.pixel_scheme, 1))[0].endswith(",true>"):
            return d
    pytest.fail(f"no depth of {DEEP_DEPTHS} gives a deep record")


def _case_list():
    """(mode, NS, paired, deep, scene, N): every f32 non-adaptive instantiation once, scenes and grids alternating."""
    out = []
    for mode in (1, 2, 0):
        for ns in (2, 3, 5, 8):
            for i, (paired, deep) in enumerate(((True, False), (False, False), (True, True), (False, True))):
                out.append((mode, ns, paired, deep, SCENES[mode][i % 2], NS_GRIDS[ns][(i // 2 + i) % 2]))
    return out


CASES = _case_list()


def _setup_case(ctx, mode, ns, paired, deep, scene, n, seed=5):
    w, h = (16, 12) if deep else (24, 16)
    spp = 40 if paired else 7            # 40: one full batch and a partial one; 7: four pixels per task
    cfg, tables, sc, camera = _load(ctx, scene, n, w, h, spp, 4)
    depth = _deep_depth(ctx, cfg, w, h, spp) if deep else _shallow_depth(ctx, cfg, w, h, spp)
    prm = oracledriver.params(w, h, 0, spp, depth, cfg.pixel_scheme, seed)
    name = ctx.render_kernel_info(prm)[0]
    assert name == f"drt::render_kernel<float,{ns},{mode},{str(paired).lower()},{str(deep).lower()}>", name
    SEEN.add(name)
    return sc, camera, prm, w, h, spp


def _rel(a, b, floor):
    return np.abs(a.astype(np.float64) - b) / np.maximum(np.abs(b), floor)


# ---------------------------------------------------------------------------------------------------------------- (a) film = its paths
@pytest.mark.parametrize("mode,ns,paired,deep,scene,n", CASES)
def test_film_is_the_statistics_of_its_paths(ctx, mode, ns, paired, deep, scene, n):
    """As test_gpu_replay.py's check of the same name, for every f32 instantiation: filter exact, sum and mean within 1e-4 and M2
    within 1e-3 of the f64 statistics of the dumped paths (floor 1e-5 of the plane's peak), unlit pixels exactly zero."""
    RAN.add((mode, ns, paired, deep))
    sc, camera, prm, w, h, spp = _setup_case(ctx, mode, ns, paired, deep, scene, n)
    film = ctx.render_host(prm)
    paths = ctx.sample_paths(prm, 0, 0, w, h).astype(np.float64)
    s = paths.sum(axis=1)
    m = s / spp
    m2 = ((paths - m[:, None, :]) ** 2).sum(axis=1)
    assert np.array_equal(film["filter"], np.full(w * h, spp, np.float32))
    lit = np.abs(paths).max(axis=(1, 2)) > 0
    assert lit.any()
    assert np.array_equal(lit, np.abs(film["sum"]).max(axis=1) > 0)
    assert not film["sum"][~lit].any() and not film["mean"][~lit].any() and not film["m2"][~lit].any()
    for name, ref, tol in (("sum", s, 1e-4), ("mean", m, 1e-4), ("m2", m2, 1e-3)):
        rel = _rel(film[name], ref, 1e-5 * np.abs(ref).max())
        print(f"\n{scene} N={n} NS={ns} mode {mode} spp {spp} depth {prm.max_depth} {name}: max rel {rel.max():.2e}")
        assert rel.max() <= tol, name


ADAPTIVE_CASES = [(mode, ns, deep, SCENES[mode][(i + deep) % 2], NS_GRIDS[ns][(i + deep) % 2])
                  for mode in (1, 2, 0) for i, ns in enumerate((2, 3, 5, 8)) for deep in (False, True)]


@pytest.mark.parametrize("mode,ns,deep,scene,n", ADAPTIVE_CASES)
def test_adaptive_film_is_the_prefix_the_rule_picks(ctx, mode, ns, deep, scene, n):
    """Every adaptive instantiation: each pixel's film is the statistics of a prefix of its dumped paths, and the prefix ends where the
    f64 rule says (test_gpu_adaptive.py's checks).  rel_error is the median over the lit pixels of the f64 error ratio at 128 samples,
    so that some pixels stop early and some do not."""
    w, h, cap, mn = 16, 12, 256, 64
    cfg, tables, sc, camera = _load(ctx, scene, n, w, h, cap, 4)
    depth = _deep_depth(ctx, cfg, w, h, cap) if deep else _shallow_depth(ctx, cfg, w, h, cap)
    prm = oracledriver.params(w, h, 0, cap, depth, cfg.pixel_scheme, 31)
    name = ctx.render_kernel_info(prm)[0]
    assert name == f"drt::render_kernel<float,{ns},{mode},true,{str(deep).lower()}>", name
    SEEN_ADAPTIVE.add((ns, mode, deep))
    yw = (np.array(tables.cmf_y[:n]) * np.array(tables.ref_white[:n])).astype(np.float32).astype(np.float64)
    paths = ctx.sample_paths(prm, 0, 0, w, h).astype(np.float64)
    x = paths[:, :128]
    y = x.mean(axis=1) @ yw
    err = np.sqrt(np.maximum((x * x).sum(axis=1) - x.sum(axis=1) ** 2 / 128, 0.0) / (128 * 127)) @ yw
    lit = y > 0
    r = np.sort(err[lit] / y[lit])
    assert len(r) >= 2
    k = len(r) // 2
    rel_error = float(math.sqrt(r[k - 1] * r[k])) if r[k - 1] > 0 else float(r[k]) * 1.001
    film = ctx.render_host_adaptive(prm, rel_error, mn)
    counts = film["filter"].astype(np.float64)
    print(f"\n{scene} N={n} NS={ns} mode {mode} depth {depth}: rel_error {rel_error:.3g}, counts {counts.min():.0f}..{counts.max():.0f}")
    assert np.all((counts == cap) | ((counts % 32 == 0) & (counts >= mn)))
    assert counts.min() < cap and len(np.unique(counts)) > 1
    test_gpu_adaptive._check_prefix(film, paths, counts)
    test_gpu_adaptive._check_rule(counts, paths, yw, rel_error, mn, 0, cap)


# ---------------------------------------------------------------------------------------------------------------- (b) against the oracle
ORACLE_CASES = [c for c in CASES if not c[3] and c[2]] + [c for c in CASES if not c[3] and not c[2]] + [c for c in CASES if c[3] and c[2]]
WORST = {}


@pytest.mark.parametrize("mode,ns,paired,deep,scene,n", ORACLE_CASES)
def test_paths_match_oracle(ctx, mode, ns, paired, deep, scene, n):
    """Per-path radiance and work counters against the oracle with the allowances of test_gpu_parity.py (>= 99.5 % of paths within
    1e-3, counters within 1 % + 8) and, for the deep case, of test_deep_paths."""
    sc, camera, prm, w, h, spp = _setup_case(ctx, mode, ns, paired, deep, scene, n, seed=0xC0FFEE)
    gpu = ctx.sample_paths(prm, 0, 0, w, h)
    st = ctx.stats()
    _, _, _, ref, cnt = oracledriver.render_tile(sc, camera, prm, 0, 0, w, h, want_paths=True)
    err = common.path_errors(gpu, ref)
    ok = (err <= 1e-3).mean()
    good = err[err <= 1e-3]
    WORST[ns] = max(WORST.get(ns, 0.0), float(good.max()) if good.size else 0.0)
    print(f"\n{scene} N={n} NS={ns} mode {mode} depth {prm.max_depth}: {100 * ok:.3f} % within 1e-3, "
          f"largest error below it {WORST[ns]:.2e}, over it {int((err > 1e-3).sum())}")
    assert st.paths == cnt.paths == err.size
    if deep:
        assert ok >= (0.99 if prm.max_depth <= 24 else 0.97)
        assert abs(int(st.shaded_bounces) - int(cnt.shaded_bounces)) <= 0.02 * cnt.shaded_bounces + 8
    else:
        assert ok >= 0.995
        for a, b in ((st.closest_rays, cnt.closest_rays), (st.shadow_rays, cnt.shadow_rays), (st.rng_draws, cnt.rng_draws)):
            assert abs(a - b) <= 0.01 * b + 8


@pytest.mark.parametrize("n,scene", [(2, "stress_all"), (32, "cornell_plane_light"), (48, "classed_all"), (80, "init_cornell"),
                                     (128, "stress_all")])
def test_paths_match_oracle_f64_geometry(ctx, n, scene):
    """The f64-geometry (general) kernel at NS = 2, 3, 5 and 8, full and partial last slots: >= 99.95 % of paths within 1e-4."""
    w, h, spp = 24, 16, 33
    cfg, tables, sc, camera = _load(ctx, scene, n, w, h, spp, 5)
    ctx.set_geometry_precision(cuda.GEOMETRY_F64)
    try:
        prm = oracledriver.params(w, h, 0, spp, _shallow_depth(ctx, cfg, w, h, spp), cfg.pixel_scheme, 17)
        assert ctx.render_kernel_info(prm)[0] == f"drt::render_kernel<double,{grids.render_slots(n)},0,true,false>"
        gpu = ctx.sample_paths(prm, 0, 0, w, h)
    finally:
        ctx.set_geometry_precision(cuda.GEOMETRY_F32)
    ref = oracledriver.render_tile(sc, camera, prm, 0, 0, w, h, want_paths=True)[3]
    err = common.path_errors(gpu, ref)
    ok = (err <= 1e-4).mean()
    print(f"\n{scene} N={n} [f64 geometry]: within 1e-4: {100 * ok:.4f} %, max err {err.max():.2e}")
    assert ok >= 0.9995


# ---------------------------------------------------------------------------------------------------------------- (c) grid invariance
@pytest.mark.parametrize("scene", grids.INVARIANT_SCENES)
@pytest.mark.parametrize("spp", [40, 7])
def test_paths_are_grid_invariant(ctx, scene, spp):
    """The kernel's dumped paths at 380, 400, ..., 720 nm on the 18-, 35- (NS 2, 3), 69- (NS 5) and 128-wavelength (NS 8) grids.
    Every wavelength's arithmetic is independent and the geometry is the same scalar code, so the values must be bit-identical, up to
    the paths that take another branch in f32 (<= 0.5 % of the paths, as test_gpu_parity.py allows).  A lane or slot-pair mapping
    error moves values between wavelengths, which this check sees with no tolerance to hide behind."""
    w, h, depth = 24, 16, 4
    shared = {}
    for n, lo, hi, step in grids.INVARIANCE_GRIDS:
        cfg, tables, sc, camera = _load(ctx, scene, n, w, h, spp, depth)
        prm = oracledriver.params(w, h, 0, spp, depth, cfg.pixel_scheme, 13)
        SEEN.add(ctx.render_kernel_info(prm)[0])
        shared[n] = ctx.sample_paths(prm, 0, 0, w, h)[:, :, grids.shared_columns(n, lo, hi, step)[0]]
    base = shared[18]
    assert np.abs(base).max() > 0
    for n in (35, 69, 128):
        a, b = shared[n], base[:, :, :shared[n].shape[-1]]
        same = a.view(np.uint32) == b.view(np.uint32)
        live = (a != 0) | (b != 0)
        rel = np.abs(a.astype(np.float64) - b) / np.maximum(np.abs(b.astype(np.float64)), 1e-30)
        rel = np.where(same, 0.0, rel)
        flipped = (rel > 1e-6).any(axis=-1)                       # paths with any value beyond 1e-6
        frac, frac_live = same.mean(), same[live].mean()
        print(f"\n{scene} spp {spp} N=18 vs N={n}: bit-identical {100 * frac:.4f} % of values ({100 * frac_live:.4f} % of the non-zero ones), "
              f"max rel {rel.max():.2e}, paths over 1e-6: {int(flipped.sum())} of {flipped.size}")
        assert frac >= 0.999 and frac_live >= 0.999
        assert flipped.mean() <= 0.005


# ---------------------------------------------------------------------------------------------------------------- (d) epilogues vs f64
EPS = float(np.finfo(np.float32).eps)
EPI_GRIDS = (2, 32, 33, 64, 96, 97, 128)


def _epi_ctx(ctx, n):
    cfg, tables, sc, camera = _load(ctx, "init_cornell", n, 8, 8, 1, 4)
    return tables


def _synthetic(rng, npix, n, specials=True):
    """f32 film planes (sum, filter, mean, m2) of npix pixels with the rows where epilogues go wrong first (those that fit)."""
    cnt = rng.integers(2, 300, npix).astype(np.float64)
    mean = rng.uniform(0.0, 1.5, (npix, n)) * rng.uniform(0.1, 1.0, (npix, 1))
    m2 = rng.uniform(0.0, 0.3, (npix, n)) * cnt[:, None]
    if specials:
        cnt[0] = 0; mean[0] = 0; m2[0] = 0                                             # no samples
        cnt[1] = 1; m2[1] = 0                                                          # one sample
        cnt[2] = 1e6; m2[2] *= 1e4                                                     # a million samples
        mean[3] = 1e4 + rng.uniform(-1e-2, 1e-2, n); m2[3] = cnt[3] * 1e-4 * rng.uniform(0.5, 1.0, n)   # large mean, tiny spread
        mean[4] = rng.uniform(-1.0, 1.0, n); m2[4, ::3] = -m2[4, ::3]                  # negative entries
        mean[5, ::7] = np.nan; m2[5, 1::9] = np.nan                                    # NaN entries
        m2[6] = 0                                                                      # all-zero M2
        if npix > 7:
            mean[7] = 40.0; m2[7] = 1e3                                                # converts above 1 (clamps to 255)
    planes = {"filter": cnt.astype(np.float32), "mean": mean.astype(np.float32), "m2": m2.astype(np.float32)}
    planes["sum"] = (planes["mean"].astype(np.float64) * cnt[:, None]).astype(np.float32)
    return planes


def _to_device(planes):
    import torch
    t = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in planes.items()}
    return t, cuda.film_from_tensors(t["sum"], t["filter"], t["mean"], t["m2"])


def _host(t):
    import torch
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in t.items()}


def _rgb_f64(tables, n, spd):
    """drt_spectrum_to_rgb in float64, vectorised over rows."""
    cx, cy, cz, rw = (np.array(getattr(tables, k)[:n]) for k in ("cmf_x", "cmf_y", "cmf_z", "ref_white"))
    norm = (cy * rw).sum() * tables.wl_interval
    xyz = np.stack([spd @ (cx * rw), spd @ (cy * rw), spd @ (cz * rw)], axis=-1) * (tables.wl_interval / norm)
    x, y, z = xyz[:, 0], xyz[:, 1], xyz[:, 2]
    return np.stack([(2.3706743 * x) - (0.9000405 * y) - (0.4706338 * z), (-0.5138850 * x) + (1.4253036 * y) + (0.0885814 * z),
                     (0.0052982 * x) - (0.0146949 * y) + (1.0093968 * z)], axis=-1)


def _image_planes(p):
    """The three images' spectra in f64 as the epilogue forms them: sum / filter, mean, M2 / (largest non-negative M2 of the row)."""
    with np.errstate(invalid="ignore", divide="ignore"):
        peak = np.maximum(np.nanmax(np.where(np.isnan(p["m2"]), -np.inf, p["m2"].astype(np.float64)), axis=1), 0.0)
        return (p["sum"].astype(np.float64) / p["filter"][:, None], p["mean"].astype(np.float64), p["m2"].astype(np.float64) / peak[:, None])


def _codes(rgb):
    """drt_rgb_to_bgra8 on f64 rows, and which channels lie within 1e-4 of a code boundary (f32 may land on either side)."""
    v = np.where(np.isnan(rgb), 0.0, rgb)
    v = np.clip(v, 0.0, 1.0)
    q = (v * 255.0).astype(np.uint32)
    near = np.abs(v * 255.0 - np.round(v * 255.0)) <= 255.0 * 1e-4
    near &= (v > 0.0) & (v < 1.0)
    return (q[:, 0] << 16) | (q[:, 1] << 8) | q[:, 2], near


def _check_codes(got, rgb_ref, what):
    """Codes equal to the f64 conversion's, except one code off where the f64 value lies within 1e-4 of a boundary."""
    want, near = _codes(rgb_ref)
    got = got.view(np.uint32)
    diff = np.stack([np.abs(((got >> s) & 255).astype(int) - ((want >> s) & 255).astype(int)) for s in (16, 8, 0)], axis=-1)
    bad = (diff > 1) | ((diff == 1) & ~near)
    assert not bad.any(), (what, np.argwhere(bad)[:5])
    assert np.all(got >> 24 == 0)
    return int((diff > 0).sum())


@pytest.mark.parametrize("n", EPI_GRIDS)
def test_film_to_rgb_matches_float64(ctx, host, n):
    import torch
    tables = _epi_ctx(ctx, n)
    rng = np.random.default_rng(100 + n)
    w, h = 9, 7
    p = _synthetic(rng, w * h, n)
    t, film = _to_device(p)
    dp = C.POINTER(C.c_double)
    src = _image_planes(p)
    probe = np.ascontiguousarray(src[1][8])
    one = np.zeros(3)
    host.lib().drt_spectrum_to_rgb(C.byref(tables), probe.ctypes.data_as(dp), one.ctypes.data_as(dp))
    assert np.allclose(_rgb_f64(tables, n, probe[None])[0], one, rtol=1e-12, atol=1e-15)      # the numpy model is the host function
    rgb = torch.zeros(w * h, 3, device="cuda")
    bgra = torch.zeros(w * h, dtype=torch.int32, device="cuda")
    near_misses = 0
    for which in (0, 1, 2):
        rgb.fill_(-7.0)
        ctx.film_to_rgb(film, w, h, which, rgb.data_ptr(), bgra.data_ptr())
        torch.cuda.synchronize()
        with np.errstate(invalid="ignore"):
            ref = _rgb_f64(tables, n, src[which])
        got = rgb.cpu().numpy()
        nan = np.isnan(ref)
        assert np.array_equal(np.isnan(got), nan), which
        assert np.allclose(got[~nan], ref[~nan], rtol=2e-4, atol=2e-6), which
        near_misses += _check_codes(bgra.cpu().numpy(), ref, f"which {which}")
        q = bgra.cpu().numpy()
        assert q[0] == 0 and q[5] == 0                          # no samples (0 / 0 for the sum image), NaN entries -> byte 0
        if which == 2:
            assert q[6] == 0                                    # all-zero M2: 0 / 0
        else:
            assert any((int(q[7]) >> s) & 255 == 255 for s in (0, 8, 16))     # clamped to 255
    print(f"\nN={n}: film_to_rgb codes one off at a boundary: {near_misses}")


def _chan(parts, from_empty=False):
    """f64 Chan merge of partial films in order, with a running bound on the f32 kernel's error (see test_film_merge_matches_float64).
    from_empty: start from a film with no samples, as the gather-merge kernel does (a NaN mean then also poisons M2)."""
    if from_empty:
        parts = [{k: np.zeros_like(v) for k, v in parts[0].items()}] + list(parts)
    f = {k: parts[0][k].astype(np.float64) for k in ("sum", "filter", "mean", "m2")}
    e_mean = np.zeros_like(f["mean"])
    e_m2 = np.zeros_like(f["m2"])
    e_sum = np.zeros_like(f["sum"])
    u = EPS / 2
    for b in parts[1:]:
        na, nb = f["filter"][:, None], b["filter"].astype(np.float64)[:, None]
        nab = na + nb
        with np.errstate(invalid="ignore", divide="ignore"):
            wb = np.where(nab > 0, nb / np.where(nab > 0, nab, 1), 0.0)
        d = b["mean"] - f["mean"]
        term = d * d * na * wb
        # the f32 kernel: delta carries the running mean's error plus one rounding, wb one rounding, the M2 term 4, the sums 2 each
        e_d = e_mean + u * np.abs(d)
        e_term = term * 8 * u + (2 * np.abs(d) * e_d + e_d * e_d) * na * wb
        new_m2 = f["m2"] + b["m2"] + term
        e_m2 = e_m2 + e_term + 3 * u * (np.abs(f["m2"]) + np.abs(b["m2"]) + term)
        new_mean = f["mean"] + d * wb
        e_mean = e_mean * (1 - wb) + e_d * wb + 3 * u * (np.abs(new_mean) + np.abs(d) * wb)
        e_sum = e_sum + 2 * u * (np.abs(f["sum"]) + np.abs(b["sum"]))
        f = {"sum": f["sum"] + b["sum"], "filter": nab[:, 0], "mean": new_mean, "m2": new_m2}
    return f, {"sum": e_sum, "mean": e_mean, "m2": e_m2}


def _check_merged(got, ref, err, what, ratio_log):
    assert np.array_equal(got["filter"], ref["filter"].astype(np.float32)), what
    for k in ("sum", "mean", "m2"):
        g, r = got[k].astype(np.float64), ref[k]
        nan = np.isnan(r)
        assert np.array_equal(np.isnan(g), nan), (what, k)
        bound = 2 * err[k] + 1e-37
        d = np.abs(g - r)
        ratio_log.append(float(np.max(np.where(nan, 0.0, d / bound))))
        assert np.all(np.where(nan, True, d <= bound)), (what, k, np.argwhere(~nan & (d > bound))[:5])


MERGE_RATIOS = []


@pytest.mark.parametrize("n", EPI_GRIDS)
def test_film_merge_matches_float64(ctx, n):
    """The pairwise kernel (drt_cuda_film_merge) against the f64 Chan update under an f32 error bound: 2 x (8 u (M2a + M2b + d^2 na nb / n)
    + 3 u (M2a + M2b)) for M2, and the analogous bound for mean and sum (u = 2^-24) -- not a flat relative tolerance, which large means
    with tiny spreads would break.  Rows with na = 0, nb = 0 and both zero must merge exactly."""
    _epi_ctx(ctx, n)
    rng = np.random.default_rng(200 + n)
    npix = 40
    a, b = _synthetic(rng, npix, n), _synthetic(rng, npix, n)
    b["mean"][3] = (np.float32(1e4) + rng.uniform(-1e-2, 1e-2, n)).astype(np.float32)          # both large with tiny spreads
    b["sum"][3] = (b["mean"][3].astype(np.float64) * b["filter"][3]).astype(np.float32)
    b["filter"][2] = 1; b["m2"][2] = 0; b["sum"][2] = b["mean"][2]                                # counts 1e6 against 1
    for k in ("sum", "mean", "m2"):
        b[k][1] = 0
        b[k][8] = 0; a[k][9] = 0
    b["filter"][1] = 0; b["filter"][8] = 0; a["filter"][9] = 0                                   # nb = 0 (rows 1, 8), na = 0 (9); both zero (0)
    ref, err = _chan([a, b])
    ta, fa = _to_device(a)
    tb, fb = _to_device(b)
    ctx.film_merge(fa, fb, npix, 1)
    got = _host(ta)
    _check_merged(got, ref, err, f"N={n}", MERGE_RATIOS)
    for row, src in ((1, a), (8, a), (9, b), (0, a)):
        for k in ("sum", "mean", "m2", "filter"):
            assert np.array_equal(got[k][row], src[k][row], equal_nan=True), (row, k)
    print(f"\nN={n}: film_merge worst error / bound {max(MERGE_RATIOS[-3:]):.3f}")


def _parts(rng, count, npix, n):
    parts = [_synthetic(rng, npix, n, specials=(g == 0)) for g in range(count)]
    for g, p in enumerate(parts):
        if g % 3 == 1:                                    # empty partial films here and there, and a pixel no rank sampled
            for k in p:
                p[k][(10 + g % 5) % npix] = 0
        for k in p:
            p[k][11 % npix] = 0
        if g:                                             # the large-mean row stays a large mean with a tiny spread in every part
            p["mean"][3] = (np.float32(1e4) + rng.uniform(-1e-2, 1e-2, n)).astype(np.float32)
            p["m2"][3] = (p["filter"][3] * 1e-4 * rng.uniform(0.5, 1.0, n)).astype(np.float32)
            p["sum"][3] = (p["mean"][3].astype(np.float64) * p["filter"][3]).astype(np.float32)
    return parts


def _images_equal_film_to_rgb(ctx, merged_film, w, h, imgs, what):
    import torch
    ref = torch.zeros(w * h, dtype=torch.int32, device="cuda")
    differ = 0
    for which in range(3):
        ctx.film_to_rgb(merged_film, w, h, which, None, ref.data_ptr())
        torch.cuda.synchronize()
        differ += int((imgs[which].cpu().numpy() != ref.cpu().numpy()).sum())
    assert differ == 0, (what, differ)


@pytest.mark.parametrize("n", (2, 33, 97, 128))
@pytest.mark.parametrize("count", (1, 2, 3, 4, 5, 8, 9, 16))
def test_film_merge_many_matches_float64(ctx, n, count):
    """The fused gather-merge kernel (CHUNK 2 for <= 2 films, 4 above: 5 and 9 leave a tail of one, 16 none) over ragged pixel ranges:
    merged planes against f64 under the running f32 bound of _chan, pixels outside a call's range untouched, and the three images
    equal to film_to_rgb of the merged film (the arithmetic is the same)."""
    import torch
    _epi_ctx(ctx, n)
    rng = np.random.default_rng(1000 * count + n)
    w, h = 13, 5
    npix = w * h
    parts = _parts(rng, count, npix, n)
    dev = [_to_device(p) for p in parts]
    ref, err = _chan(parts, from_empty=True)
    out = {k: torch.full_like(v, -7.0) for k, v in dev[0][0].items()}
    dst = cuda.film_from_tensors(out["sum"], out["filter"], out["mean"], out["m2"])
    imgs = [torch.zeros(npix, dtype=torch.int32, device="cuda") for _ in range(3)]
    cuts = [0, 1, 18, 19, 47, npix]
    ctx.film_merge_many(dst, [d[1] for d in dev], w, h, cuts[1], cuts[3], bgra=[t.data_ptr() for t in imgs])
    got = _host(out)
    assert np.all(got["filter"][:cuts[1]] == -7.0) and np.all(got["filter"][cuts[3]:] == -7.0)
    assert np.all(got["sum"][cuts[3]:] == -7.0) and np.all(got["m2"][:cuts[1]] == -7.0)
    for a, b in ((0, 1), (3, 4), (4, 5)):
        ctx.film_merge_many(dst, [d[1] for d in dev], w, h, cuts[a], cuts[b], bgra=[t.data_ptr() for t in imgs])
    got = _host(out)
    _check_merged(got, ref, err, f"count {count} N={n}", MERGE_RATIOS)
    _images_equal_film_to_rgb(ctx, dst, w, h, imgs, f"count {count} N={n}")


def _staging(rng, count, slice_px, npix, n):
    """The staging film of one owner (drt_cuda_render_device_scatter's layout: rank g's partial film of the slice at pixels
    g * slice_px ...), filled with synthetic partial films, and those partial films."""
    parts = _parts(rng, count, slice_px, n)
    planes = {k: np.concatenate([p[k] for p in parts]) for k in ("sum", "filter", "mean", "m2")}
    return parts, planes


@pytest.mark.parametrize("count,w,h", [(3, 37, 23), (8, 7, 7), (16, 15, 15)])
@pytest.mark.parametrize("n", (32, 97))
def test_merge_slices_local_and_read_slice_in_bands(ctx, count, w, h, n):
    """The sharded exchange's merge and read-back, band by band (ShardedFilmGroup.BAND_CUTS) over every owner's slice, on synthetic
    staging films: the assembled host film matches the f64 merge of the partial films, the images equal film_to_rgb of it.  With
    7 x 7 pixels over 8 owners and 15 x 15 over 16 the last owner has no pixels."""
    import torch
    _epi_ctx(ctx, n)
    rng = np.random.default_rng(7 * count + n)
    npix = w * h
    slice_px, owners = film_mod.slice_partition(npix, count)
    if count in (8, 16):
        assert owners[-1][0] == owners[-1][1] == npix
    host_planes = {k: np.full((npix, n) if k != "filter" else npix, -7.0, np.float32) for k in ("sum", "filter", "mean", "m2")}
    host_film = cuda.Film(*(host_planes[k].ctypes.data for k in ("sum", "filter", "mean", "m2")))
    imgs = [torch.zeros(npix, dtype=torch.int32, device="cuda") for _ in range(3)]
    refs, errs, keep = [], [], []
    cuts = film_mod.ShardedFilmGroup.BAND_CUTS
    for o, (p0, p1) in enumerate(owners):
        parts, planes = _staging(rng, count, slice_px, npix, n)
        t, staging = _to_device(planes)
        sl = ctx.film_alloc(w, max(1, -(-slice_px // w)))
        keep.append((t, sl))
        ref, err = _chan(parts, from_empty=True)
        refs.append({k: v[:p1 - p0] for k, v in ref.items()})
        errs.append({k: v[:p1 - p0] for k, v in err.items()})
        for b in range(len(cuts) - 1):
            q0, q1 = min(p1, p0 + slice_px * cuts[b] // 16), min(p1, p0 + slice_px * cuts[b + 1] // 16)
            if q1 > q0:
                ctx.film_merge_slices_local(sl, staging, count, slice_px, w, h, q0, q1, bgra=[i.data_ptr() for i in imgs])
                ctx.film_read_slice(sl, p0, q0, q1, host_film)
    torch.cuda.synchronize()
    ref = {k: np.concatenate([r[k] for r in refs]) for k in refs[0]}
    err = {k: np.concatenate([e[k] for e in errs]) for k in errs[0]}
    _check_merged(host_planes, ref, err, f"count {count} N={n}", MERGE_RATIOS)
    t, merged = _to_device(host_planes)
    _images_equal_film_to_rgb(ctx, merged, w, h, imgs, f"count {count} N={n}")
    for _, sl in keep:
        ctx.film_free(sl)


@pytest.mark.parametrize("n", (33, 128))
def test_merge_slices_band_inside_a_slice(ctx, n):
    """drt_cuda_film_merge_slices on a range that starts inside the owner's slice (a band) reads the staging film from the slice's
    first pixel, like drt_cuda_film_merge_slices_local, and a range that crosses a slice boundary is an argument error."""
    import torch
    _epi_ctx(ctx, n)
    rng = np.random.default_rng(n)
    count, w, h = 4, 12, 10
    npix = w * h
    slice_px, owners = film_mod.slice_partition(npix, count)
    o = 2
    p0, p1 = owners[o]
    parts, planes = _staging(rng, count, slice_px, npix, n)
    t, staging = _to_device(planes)
    ref, err = _chan(parts, from_empty=True)
    out = {k: torch.full((npix, n) if k != "filter" else (npix,), -7.0, device="cuda") for k in ("sum", "filter", "mean", "m2")}
    dst = cuda.film_from_tensors(out["sum"], out["filter"], out["mean"], out["m2"])
    q0, q1 = p0 + 7, p0 + 19
    ctx.film_merge_slices(dst, staging, count, slice_px, w, h, q0, q1)
    got = _host(out)
    assert np.all(got["filter"][:q0] == -7.0) and np.all(got["filter"][q1:] == -7.0)
    part = {k: v[q0:q1] for k, v in got.items()}
    _check_merged(part, {k: v[q0 - p0:q1 - p0] for k, v in ref.items()}, {k: v[q0 - p0:q1 - p0] for k, v in err.items()},
                  f"band [{q0}, {q1}) of slice [{p0}, {p1})", MERGE_RATIOS)
    with pytest.raises(cuda.CudaError) as e:
        ctx.film_merge_slices(dst, staging, count, slice_px, w, h, p1 - 3, p1 + 3)
    assert e.value.code == -103 and "slice boundary" in str(e.value)


# ---------------------------------------------------------------------------------------------------------------- coverage
def test_every_instantiation_was_launched():
    """Runs last in this module: the tests above launched all 48 f32 render_kernel instantiations (3 modes x NS 2, 3, 5, 8 x both task
    shapes x shallow / deep) and all 24 adaptive ones (3 modes x 4 NS x shallow / deep)."""
    want = {f"drt::render_kernel<float,{ns},{mode},{p},{d}>" for ns in (2, 3, 5, 8) for mode in (0, 1, 2)
            for p in ("true", "false") for d in ("true", "false")}
    want_adaptive = {(ns, mode, d) for ns in (2, 3, 5, 8) for mode in (0, 1, 2) for d in (False, True)}
    if len(RAN) < len(CASES) or len(SEEN_ADAPTIVE) < len(ADAPTIVE_CASES):
        pytest.skip("the coverage check needs the whole module")
    f32 = {s for s in SEEN if s.startswith("drt::render_kernel<float,")}
    print(f"\ninstantiations launched: {len(f32 & want)}/{len(want)} non-adaptive, {len(SEEN_ADAPTIVE & want_adaptive)}/{len(want_adaptive)} "
          f"adaptive; largest per-path oracle error (paths within 1e-3) by NS: {WORST}; "
          f"worst merge error / bound: {max(MERGE_RATIOS) if MERGE_RATIOS else float('nan'):.3f}")
    assert f32 == want
    assert SEEN_ADAPTIVE == want_adaptive
