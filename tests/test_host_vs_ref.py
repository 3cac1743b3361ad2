"""Host C front-end (product) pinned bit-for-bit against the unmodified reference's own parse/setup code.

The comparisons with the reference need oracle/_ref (built by oracle/Makefile where the reference sources are present).  Without
it, test_golden.py compares scene, camera, tables and the rgb / blackbody spectra with stored reference fixtures; material names,
spectrum -> RGB and the 8-bit conversion are compared with the reference only here."""
import os

import numpy as np
import pytest

import refdriver

needs_ref = pytest.mark.skipif(not refdriver.available(), reason="oracle/_ref not built")

SCENES = ["cornell_plane_light", "init_cornell", "cornell_large_box", "cornell_downward", "first_scene", "example_scene"]


def _load_both(host, assets, tmp_path, scene, w=48, h=32):
    text = open(os.path.join(assets, "scenes", scene + ".scn")).read()
    parsed = host.parse_scene_text(text)
    upgraded = host.scene_to_text(parsed)
    root = refdriver.make_root(str(tmp_path), assets, upgraded, "upgraded.scn")
    cfg_text = host.make_config_text(scene="scenes\\upgraded.scn", width=w, height=h)
    ref = refdriver.Ref(root, cfg_text)
    cfg = host.parse_config_text(cfg_text)
    tables = host.load_tables(cfg, assets)
    mine = host.load_scene_file(assets, f"scenes/{scene}.scn", tables, w, h)
    return ref, tables, mine


@pytest.mark.parametrize("scene", SCENES)
def test_upgraded_text_reparses_to_the_same_scene(host, assets, tmp_path, scene):
    """The text scene_to_text upgrades a legacy scene to parses to the same scene and camera under the STRICT (reference) grammar."""
    w, h = 48, 32
    parsed = host.parse_scene_text(open(os.path.join(assets, "scenes", scene + ".scn")).read())
    root = refdriver.make_root(str(tmp_path), assets, host.scene_to_text(parsed), "upgraded.scn")
    tables = host.load_tables(host.parse_config_text(host.make_config_text(width=w, height=h)), assets)
    sc, cam = host.load_scene_file(assets, f"scenes/{scene}.scn", tables, w, h)
    sc2, cam2 = host.load_scene_file(root, "scenes/upgraded.scn", tables, w, h, flags=0)
    assert bytes(sc) == bytes(sc2) and bytes(cam)[:160] == bytes(cam2)[:160]


@needs_ref
@pytest.mark.parametrize("scene", SCENES)
def test_scene_and_camera_bit_exact(host, assets, tmp_path, scene):
    ref, tables, (sc, cam) = _load_both(host, assets, tmp_path, scene)

    mine_cam = np.array(list(cam.forward) + list(cam.right) + list(cam.up) + list(cam.aperture_position)
                        + [cam.aperture_radius, cam.focal_depth, cam.focal_length] + list(cam.film_bottom_left)
                        + [cam.pixel_width, cam.pixel_height])
    assert np.array_equal(mine_cam, ref.camera()), (mine_cam, ref.camera())

    n = ref.n
    rt = ref.tables()
    mt = np.array([list(tables.ref_white)[:n], list(tables.cmf_x)[:n], list(tables.cmf_y)[:n], list(tables.cmf_z)[:n]]
                  + [list(tables.rgb_basis[k])[:n] for k in range(7)])
    assert np.array_equal(mt, rt)

    assert sc.num_surfaces == ref.lib.ref_num_surfaces()
    assert sc.num_materials == ref.lib.ref_num_materials()
    assert sc.base_material == ref.lib.ref_base_material()
    assert sc.escape_material == ref.lib.ref_escape_material()
    for i in range(sc.num_surfaces):
        t, m, g = ref.surface(i)
        s = sc.surfaces[i]
        assert (s.type, s.material) == (t, m)
        mine = np.array(list(s.position) + [s.radius] + list(s.normal) + list(s.u) + list(s.v))
        assert np.array_equal(mine, g), (scene, i)
    for i in range(sc.num_materials):
        r = ref.material(i)
        m = sc.materials[i]
        assert m.name.decode() == r["name"]
        assert (m.is_black_body, m.is_emissive, m.num_lobes, m.dir_func, m.spd_mask) == \
               (r["is_black_body"], r["is_emissive"], r["num_lobes"], r["dir_func"], r["spd_mask"])
        assert list(m.lobes)[:m.num_lobes] == r["lobes"]
        assert (m.shininess, m.roughness) == (r["shininess"], r["roughness"])
        mine = np.array([list(m.spd[k])[:n] for k in range(6)])
        assert np.array_equal(mine, r["spds"]), (scene, r["name"])


@needs_ref
def test_spectral_helpers_bit_exact(host, assets, tmp_path):
    import ctypes as C
    ref, tables, _ = _load_both(host, assets, tmp_path, "cornell_plane_light")
    L = host.lib()
    n = ref.n
    rng = np.random.default_rng(7)
    dp = C.POINTER(C.c_double)
    for rgb in list(rng.random((64, 3))) + [np.array([0.2, 0.2, 0.8]), np.array([1.0, 1.0, 1.0]), np.zeros(3)]:
        rgb = np.ascontiguousarray(rgb)
        out = np.zeros(n)
        L.drt_rgb_to_spectrum(C.byref(tables), rgb.ctypes.data_as(dp), out.ctypes.data_as(dp))
        assert np.array_equal(out, ref.rgb_to_spectrum(rgb))
        back = np.zeros(3)
        L.drt_spectrum_to_rgb(C.byref(tables), out.ctypes.data_as(dp), back.ctypes.data_as(dp))
        assert np.array_equal(back, ref.spectrum_to_rgb(out))
        q = L.drt_rgb_to_bgra8(back.ctypes.data_as(dp))
        r8 = ref.rgb_to_u8(back)     # r | g<<8 | b<<16
        assert ((q >> 16) & 255, (q >> 8) & 255, q & 255) == (r8 & 255, (r8 >> 8) & 255, (r8 >> 16) & 255)
    for temp in (2000.0, 4000.0, 6500.0):
        out = np.zeros(n)
        L.drt_blackbody_spectrum(C.byref(tables), temp, out.ctypes.data_as(dp))
        assert np.array_equal(out, ref.blackbody(temp))


def test_rgb_roundtrip_known_answers(host, assets, tmp_path):
    """The only numbers the reference's own test program prints (src/test.c:45-142, SURVEY.md section 4):
    11^3 RGB grid -> rgb_f64_to_spectrum -> spectrum_to_rgb_f64 error statistics."""
    import ctypes as C
    cfg = host.parse_config_text(host.make_config_text())
    tables = host.load_tables(cfg, assets)
    L = host.lib()
    dp = C.POINTER(C.c_double)
    n = tables.num_wavelengths
    errs = []
    vals = []
    v = 0.0
    while v <= 1.0:           # the reference accumulates r += 0.1 (test.c:66-72), it does not multiply
        vals.append(v)
        v += 0.1
    assert len(vals) == 11
    for r in vals:
        for g in vals:
            for b in vals:
                rgb = np.array([r, g, b])
                spd = np.zeros(n)
                back = np.zeros(3)
                L.drt_rgb_to_spectrum(C.byref(tables), rgb.ctypes.data_as(dp), spd.ctypes.data_as(dp))
                L.drt_spectrum_to_rgb(C.byref(tables), spd.ctypes.data_as(dp), back.ctypes.data_as(dp))
                errs.append(np.abs(back - rgb))
    errs = np.array(errs)
    overall = np.sqrt((errs ** 2).sum(axis=1))
    # printed by bin/test_raytrace (glibc, gcc 13.3, no FMA), to the 6 decimals of its "%f"
    assert abs(overall.max() - 0.266593) < 5e-7 and abs(overall.mean() - 0.093890) < 5e-7
    assert np.allclose(errs.max(axis=0), [0.132717, 0.208796, 0.123103], atol=5e-7, rtol=0)
    assert np.allclose(errs.mean(axis=0), [0.042695, 0.066948, 0.041327], atol=5e-7, rtol=0)
