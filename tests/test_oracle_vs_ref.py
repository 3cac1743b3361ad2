"""oracle/drt_oracle.c (the CPU restatement the CUDA path is checked against) pinned BIT-FOR-BIT against the
unmodified reference's sample_scene (oracle/_ref, per-path RNG streams) -- every shipped scene plus a stress
scene that exercises all 7 lobes, all 6 samplers, plane/sphere/point lights, multi-light NEE and the thin lens.
Where oracle/_ref is absent, test_golden.py makes the same bit-exact comparison (per path and film) for every scene here against
stored reference tiles; those are rendered at other sizes, sample counts and seeds, and cover tiles rather than whole frames."""
import os

import numpy as np
import pytest

import oracledriver
import refdriver

pytestmark = pytest.mark.skipif(not refdriver.available(), reason="oracle/_ref not built")

CASES = [
    ("cornell_plane_light", 24, 24, 3, 4, "pixel_random"),
    ("init_cornell", 24, 16, 2, 4, "pixel_random"),
    ("cornell_large_box", 16, 16, 2, 4, "pixel_random"),
    ("cornell_downward", 16, 16, 2, 4, "pixel_random"),
    ("first_scene", 16, 16, 2, 4, "pixel_center"),
    ("example_scene", 16, 16, 1, 3, "pixel_random"),
    ("stress_all", 32, 24, 4, 6, "pixel_random"),
    ("rotated_room", 32, 24, 3, 5, "pixel_random"),      # planes in general position, a tilted card and a ball inside, plane light
    ("sky_cornell", 32, 24, 3, 4, "pixel_random"),       # pinhole camera + emissive escape material (Q19), all-plastic walls
    ("classed_all", 32, 24, 4, 6, "pixel_random"),       # every material class of the classed kernel under one light
]


def _scene_text(host, assets, name):
    for d in (os.path.join(assets, "scenes"), os.path.join(os.path.dirname(__file__), "golden", "scenes")):
        p = os.path.join(d, name + ".scn")
        if os.path.exists(p):
            return open(p).read()
    raise FileNotFoundError(name)


@pytest.mark.parametrize("scene,w,h,spp,depth,scheme", CASES)
def test_per_path_and_film_bit_exact(host, assets, tmp_path, scene, w, h, spp, depth, scheme):
    parsed = host.parse_scene_text(_scene_text(host, assets, scene))
    upgraded = host.scene_to_text(parsed)
    root = refdriver.make_root(str(tmp_path), assets, upgraded, "upgraded.scn")
    cfg_text = host.make_config_text(scene="scenes\\upgraded.scn", width=w, height=h, spp=spp, depth=depth, scheme=scheme)
    seed = 0x1234ABCD5678
    ref = refdriver.Ref(root, cfg_text, seed=seed)
    cfg = host.parse_config_text(cfg_text)
    tables = host.load_tables(cfg, assets)
    sc, cam = host.build_scene(parsed, tables, assets, w, h)

    prm = oracledriver.params(w, h, 0, spp, depth, cfg.pixel_scheme, seed)
    r_sum, r_avg, r_m2, r_paths = ref.render_tile(0, 0, w, h, 0, spp, want_paths=True)
    o_sum, o_avg, o_m2, o_paths, cnt = oracledriver.render_tile(sc, cam, prm, 0, 0, w, h, want_paths=True)

    assert np.isfinite(r_paths).all() or scene == "stress_all"
    same = (o_paths == r_paths) | (np.isnan(o_paths) & np.isnan(r_paths))
    assert same.all(), f"{(~same).any(axis=(1, 2)).sum()} pixels differ"
    for a, b in ((o_sum, r_sum), (o_avg, r_avg), (o_m2, r_m2)):
        assert ((a == b) | (np.isnan(a) & np.isnan(b))).all()
    assert cnt.paths == w * h * spp
    assert r_paths.max() > 0.0
