"""CPU tier: the wavelength grids that tests/test_gpu_slot_layouts.py renders, and the premise of its grid-invariance check.

The render kernel holds wavelengths l16 + 16 k of a half warp in NS slots per lane, instantiated for NS = 2, 3, 5 and 8
(drt_cuda_upload_scene: ceil(N / 16) rounded up to the next of these); the film epilogues hold wavelengths lane + 32 k of a full warp
in up to DRT_MAX_SLOTS = 4 slots.  The grids below reach every NS with and without padding lanes, and every epilogue slot count.

The grid-invariance check renders the same paths on several grids and compares the wavelengths the grids share.  That is only
meaningful where the reference itself gives the same radiance at a wavelength whatever the rest of the grid is, which is checked
here against the f64 oracle."""
import math

import numpy as np
import pytest

import common
import oracledriver

# (N, render slots NS, min_wl, max_wl, wl_interval): every grid of the GPU slot-layout tests
RENDER_GRIDS = [(2, 2, 620.0, 640.0, 20.0), (18, 2, 380.0, 720.0, 20.0), (32, 2, 380.0, 690.0, 10.0), (33, 3, 380.0, 700.0, 10.0),
                (35, 3, 380.0, 720.0, 10.0), (48, 3, 380.0, 709.0, 7.0), (49, 5, 380.0, 716.0, 7.0), (69, 5, 380.0, 720.0, 5.0),
                (80, 5, 380.0, 696.0, 4.0), (81, 8, 380.0, 700.0, 4.0), (114, 8, 380.0, 720.0, 3.0), (128, 8, 380.0, 697.5, 2.5)]
# the epilogue grids that are not render grids above: N = 64, 96 (no padding lanes) and 97 (one wavelength in the fourth slot)
EPILOGUE_GRIDS = [(64, 380.0, 695.0, 5.0), (96, 380.0, 712.5, 3.5), (97, 380.0, 716.0, 3.5)]

# scenes whose oracle radiance at a wavelength does not depend on the rest of the grid (checked below), and the grids compared
INVARIANT_SCENES = ["init_cornell", "cornell_large_box", "sky_cornell"]
INVARIANCE_GRIDS = [(18, 380.0, 720.0, 20.0), (35, 380.0, 720.0, 10.0), (69, 380.0, 720.0, 5.0), (128, 380.0, 697.5, 2.5)]


def render_slots(n):
    """The half-warp slot count drt_cuda_upload_scene picks for N wavelengths."""
    return {1: 2, 2: 2, 3: 3, 4: 5, 5: 5}.get(math.ceil(n / 16), 8)


def shared_columns(n, lo, hi, step):
    """Indices of the grid's wavelengths on 380, 400, ..., 720 nm (the 20 nm grid), and those wavelengths."""
    wl = lo + step * np.arange(n)
    idx = [i for i, x in enumerate(wl) if (x - 380.0) % 20.0 == 0.0]
    return idx, wl[idx]


@pytest.mark.parametrize("n,ns,lo,hi,step", RENDER_GRIDS)
def test_render_grid(n, ns, lo, hi, step):
    cfg, tables, scene, camera = common.load("init_cornell", 8, 8, 1, 4, min_wl=lo, max_wl=hi, wl_interval=step)
    assert scene.num_wavelengths == n and render_slots(n) == ns
    assert 16 * {2: 0, 3: 2, 5: 3, 8: 5}[ns] < n <= 16 * ns               # the next smaller instantiation would not hold the grid
    assert lo <= 630.0 <= lo + step * (n - 1)                             # trans_wl lies inside the grid (upload_scene refuses otherwise)
    assert math.ceil(n / 32) <= 4                                         # DRT_MAX_SLOTS of the epilogues


@pytest.mark.parametrize("n,lo,hi,step", EPILOGUE_GRIDS)
def test_epilogue_grid(n, lo, hi, step):
    cfg, tables, scene, camera = common.load("init_cornell", 8, 8, 1, 4, min_wl=lo, max_wl=hi, wl_interval=step)
    assert scene.num_wavelengths == n and lo <= 630.0 <= lo + step * (n - 1)


def test_grids_reach_every_layout():
    """Every render NS with a full last slot (N = 16 NS) and a partial one, and every epilogue slot count 1..4 full and partial."""
    ns_full = {ns for n, ns, *_ in RENDER_GRIDS if n == 16 * ns}
    ns_part = {ns for n, ns, *_ in RENDER_GRIDS if n % 16}
    assert ns_full == {2, 3, 5, 8} and ns_part == {2, 3, 5, 8}
    ns_of = {n: ns for n, ns, *_ in RENDER_GRIDS}
    assert {ns_of[n] for n in (2, 32, 33, 48, 81, 128, 69)} == {2, 3, 5, 8}
    epi = [g[0] for g in RENDER_GRIDS] + [g[0] for g in EPILOGUE_GRIDS]
    assert {math.ceil(n / 32) for n in epi if n % 32 == 0} == {1, 2, 3, 4}
    assert {math.ceil(n / 32) for n in epi if n % 32} == {1, 2, 3, 4}


def test_invariance_grids_share_the_20nm_wavelengths():
    for n, lo, hi, step in INVARIANCE_GRIDS:
        idx, wl = shared_columns(n, lo, hi, step)
        assert list(wl) == list(np.arange(380.0, min(hi, 720.0) + 1e-9, 20.0)), n
        assert len(idx) == (16 if n == 128 else 18)


def _oracle_shared(scene_name, n, lo, hi, step, w=12, h=8, spp=6, seed=3):
    cfg, tables, scene, camera = common.load(scene_name, w, h, spp, 4, min_wl=lo, max_wl=hi, wl_interval=step)
    prm = oracledriver.params(w, h, 0, spp, 4, cfg.pixel_scheme, seed)
    paths = oracledriver.render_tile(scene, camera, prm, 0, 0, w, h, want_paths=True)[3]
    return paths[:, :, shared_columns(n, lo, hi, step)[0]]


@pytest.mark.parametrize("scene", INVARIANT_SCENES)
def test_oracle_radiance_is_grid_invariant(scene):
    """The f64 oracle's per-path radiance at 380, 400, ..., 720 nm is bit-identical on the 18-, 35-, 69- and 128-wavelength grids: every
    wavelength's arithmetic is independent of the others and the path's geometry does not depend on the grid.  The GPU check compares
    its own dumped paths the same way.

    Not so for scenes with a refracting or conductor material (cornell_plane_light, classed_all, stress_all): their sampled directions
    depend on the refractive index at 630 nm (trans_wl), which is interpolated from the grid's neighbours when 630 nm is not a grid
    wavelength (N = 18), so a path's geometry, and with it every wavelength, can change between grids (up to 5e-6 relative for
    cornell_plane_light, up to 4e-2 for classed_all and stress_all).  test_excluded_scenes_are_not_invariant keeps that reason true."""
    base = _oracle_shared(scene, *INVARIANCE_GRIDS[0])
    assert np.abs(base).max() > 0
    for g in INVARIANCE_GRIDS[1:]:
        other = _oracle_shared(scene, *g)
        k = other.shape[-1]
        assert np.array_equal(other, base[:, :, :k]), (scene, g[0])


@pytest.mark.parametrize("scene", ["cornell_plane_light", "classed_all", "stress_all"])
def test_excluded_scenes_are_not_invariant(scene):
    """The scenes left out of the grid-invariance check do change between a grid without 630 nm (N = 18) and one with it (N = 35), and
    agree exactly between two grids that both hold 630 nm (N = 35 and 69)."""
    a, b, c = (_oracle_shared(scene, *g) for g in INVARIANCE_GRIDS[:3])
    assert not np.array_equal(a, b)
    assert np.array_equal(b, c)
