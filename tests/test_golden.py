"""Committed fixtures from the unmodified reference (tests/golden/*.npz, made by tests/golden/make_golden.py).

CPU tier: the host front-end and the oracle restatement reproduce them bit-for-bit -- the same pins as
test_host_vs_ref.py / test_oracle_vs_ref.py, but usable where /root/reference and oracle/_ref are absent.
GPU tier: the CUDA path against the same per-path spectra within the f32 tolerance."""
import glob
import importlib
import os

import numpy as np
import pytest

import common
import oracledriver

FIXTURES = sorted(glob.glob(os.path.join(common.GOLDEN, "*.npz")))
NAMES = [os.path.splitext(os.path.basename(f))[0] for f in FIXTURES]


def _load(name):
    z = np.load(os.path.join(common.GOLDEN, name + ".npz"))
    w, h, x0, y0, x1, y1, spp, depth, scheme, seed = [int(v) for v in z["meta"]]
    cfg, tables, scene, camera = common.load(name, w, h, spp, depth, "pixel_random" if scheme == 2 else "pixel_center")
    return z, (w, h, x0, y0, x1, y1, spp, depth, scheme, seed), cfg, tables, scene, camera


def _same(a, b):
    return ((a == b) | (np.isnan(a) & np.isnan(b))).all()


def test_fixtures_exist():
    assert len(FIXTURES) >= 7


@pytest.mark.parametrize("name", NAMES)
def test_host_setup_matches_reference_fixture(host, name):
    z, meta, cfg, tables, scene, cam = _load(name)
    # the scene text the fixture was rendered from is what the writer still produces
    parsed = host.parse_scene_text(open(common.scene_path(name)).read())
    assert host.scene_to_text(parsed).encode() == bytes(z["upgraded_scene"])
    n = scene.num_wavelengths
    mine_cam = np.array(list(cam.forward) + list(cam.right) + list(cam.up) + list(cam.aperture_position)
                        + [cam.aperture_radius, cam.focal_depth, cam.focal_length] + list(cam.film_bottom_left)
                        + [cam.pixel_width, cam.pixel_height])
    assert np.array_equal(mine_cam, z["camera"])
    mt = np.array([list(tables.ref_white)[:n], list(tables.cmf_x)[:n], list(tables.cmf_y)[:n], list(tables.cmf_z)[:n]]
                  + [list(tables.rgb_basis[k])[:n] for k in range(7)])
    assert np.array_equal(mt, z["tables"])
    assert (scene.base_material, scene.escape_material) == tuple(z["base_escape"])
    assert scene.num_materials == len(z["mat_spds"]) and scene.num_surfaces == len(z["surf_geom"])
    for i in range(scene.num_materials):
        m = scene.materials[i]
        assert np.array_equal(np.array([list(m.spd[k])[:n] for k in range(6)]), z["mat_spds"][i])
        assert [m.is_black_body, m.is_emissive, m.num_lobes, m.dir_func, m.spd_mask] == list(z["mat_flags"][i])
        assert list(m.lobes)[:m.num_lobes] == list(z["mat_lobes"][i][:m.num_lobes])
        assert [m.shininess, m.roughness] == list(z["mat_scalars"][i])
    for i in range(scene.num_surfaces):
        s = scene.surfaces[i]
        assert [s.type, s.material] == list(z["surf_types"][i])
        assert np.array_equal(np.array(list(s.position) + [s.radius] + list(s.normal) + list(s.u) + list(s.v)), z["surf_geom"][i])


@pytest.mark.parametrize("name", NAMES)
def test_spectral_helpers_match_reference_fixture(host, name):
    """drt_rgb_to_spectrum and drt_blackbody_spectrum called directly on every rgb / blackbody input of the scene, bit-for-bit
    against the reference's material spectra (init_spd, daily_ray_trace.c:79-123: blackbody normalised to its peak, then the scale)."""
    import ctypes as C
    z, meta, cfg, tables, scene, cam = _load(name)
    parsed = host.parse_scene_text(open(common.scene_path(name)).read())
    inputs = {parsed.materials[j].name: parsed.materials[j] for j in range(parsed.num_materials)}
    L = host.lib()
    dp = C.POINTER(C.c_double)
    n = scene.num_wavelengths
    checked = 0
    for i in range(scene.num_materials):
        m = inputs.get(scene.materials[i].name)
        for k in range(6) if m is not None else ():
            spd = m.spd[k]
            out = np.zeros(n)
            if spd.method == 1:
                rgb = np.array(spd.rgb[:])
                L.drt_rgb_to_spectrum(C.byref(tables), rgb.ctypes.data_as(dp), out.ctypes.data_as(dp))
            elif spd.method == 3:
                L.drt_blackbody_spectrum(C.byref(tables), spd.value, out.ctypes.data_as(dp))
                out = out / out.max()
            else:
                continue
            if spd.has_scale:
                out = out * spd.scale
            assert np.array_equal(out, z["mat_spds"][i][k]), (scene.materials[i].name, k)
            checked += 1
    assert checked > 0
    print(f"\n{name}: {checked} rgb / blackbody spectra")


@pytest.mark.parametrize("name", NAMES)
def test_oracle_matches_reference_fixture(name):
    z, (w, h, x0, y0, x1, y1, spp, depth, scheme, seed), cfg, tables, scene, cam = _load(name)
    prm = oracledriver.params(w, h, 0, spp, depth, scheme, seed)
    o_sum, o_avg, o_m2, o_paths, cnt = oracledriver.render_tile(scene, cam, prm, x0, y0, x1, y1, want_paths=True)
    assert _same(o_paths, z["paths"])
    assert _same(o_sum, z["film_sum"]) and _same(o_avg, z["film_mean"]) and _same(o_m2, z["film_m2"])


def test_classed_all_tile_sees_every_material():
    """The classed_all fixture's tile is cut to stay under 1 MB; its camera rays must still hit every material of the scene's surfaces
    (all classes of the classed kernel) other than the light, which the tile does not see."""
    z, (w, h, x0, y0, x1, y1, spp, depth, scheme, seed), cfg, tables, scene, cam = _load("classed_all")
    prm = oracledriver.params(w, h, 0, spp, depth, scheme, seed)
    hit = {oracledriver.primary_material(scene, cam, prm, x, y, s) for y in range(y0, y1) for x in range(x0, x1) for s in range(spp)}
    want = {scene.surfaces[i].material for i in range(scene.num_surfaces) if not scene.materials[scene.surfaces[i].material].is_emissive}
    assert len(want) == 9 and want <= hit, sorted(scene.materials[m].name.decode() for m in want - hit)


@pytest.mark.gpu
@pytest.mark.parametrize("name", NAMES)
def test_cuda_matches_reference_fixture(name):
    cuda = importlib.import_module("daily-ray-trace_b200.cuda")
    z, (w, h, x0, y0, x1, y1, spp, depth, scheme, seed), cfg, tables, scene, cam = _load(name)
    ctx = cuda.Context(0)
    try:
        ctx.upload_scene(scene, cam, tables)
        prm = oracledriver.params(w, h, 0, spp, depth, scheme, seed)
        for geometry, tol, need in ((cuda.GEOMETRY_F32, 1e-3, 0.995), (cuda.GEOMETRY_F64, 1e-4, 0.995)):
            ctx.set_geometry_precision(geometry)
            gpu = ctx.sample_paths(prm, x0, y0, x1, y1)
            err = common.path_errors(gpu, z["paths"])
            ok = float((err <= tol).mean())
            print(f"\n{name} geometry={'f64' if geometry else 'f32'}: {100 * ok:.3f} % of {err.size} paths within {tol:g}")
            assert ok >= need
    finally:
        ctx.close()
