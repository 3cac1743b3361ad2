"""Generates tests/golden/*.npz from the UNMODIFIED reference (oracle/_ref, built from /root/reference by oracle/Makefile).

Run here, where /root/reference exists:   python tests/golden/make_golden.py
For every case it stores what the reference itself computed:
  camera (20 f64), cmf/rgb tables, per-material SPDs, per-surface geometry       <- parse_scene/init_camera/init_scene
  per-path spectra of a pixel tile (sample_scene with per-path RNG streams)      <- sample_scene
  the three film tiles (sum+filter, Welford mean, M2)                             <- render_image's accumulation
The fixtures travel to the GPU box, where /root/reference does not exist."""
import importlib
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tests"))
import common      # noqa: E402
import refdriver   # noqa: E402

host = importlib.import_module("daily-ray-trace_b200.host")

# name, W, H, tile, spp, depth, scheme, seed
CASES = [
    ("cornell_plane_light", 64, 64, (24, 8, 40, 24), 3, 4, "pixel_random", 11),
    ("init_cornell", 64, 48, (20, 10, 36, 22), 2, 4, "pixel_random", 12),
    ("cornell_large_box", 48, 48, (16, 8, 32, 24), 2, 4, "pixel_random", 13),
    ("cornell_downward", 48, 48, (16, 16, 32, 32), 2, 4, "pixel_random", 14),
    ("first_scene", 32, 32, (8, 8, 24, 24), 2, 4, "pixel_center", 15),
    ("example_scene", 32, 32, (8, 8, 24, 24), 1, 3, "pixel_random", 16),
    # tiles of stress_all and classed_all are sized to keep each fixture under 1 MB; classed_all's still sees all nine materials
    ("stress_all", 64, 48, (16, 8, 39, 24), 2, 6, "pixel_random", 17),
    ("rotated_room", 64, 48, (20, 12, 44, 28), 2, 5, "pixel_random", 18),
    # pinhole camera + EMISSIVE escape material (Q19 environment light): the tile straddles the scene's screen-space edge
    ("sky_cornell", 64, 48, (0, 8, 24, 24), 2, 4, "pixel_random", 19),
    # one light, pinhole: every material class of the classed compact-record kernel (plastics with repeated / single lobes and a
    # uniform-hemisphere sampler, mirror, fs_conductor, glass R+T, transmittance only, ct_conductor)
    ("classed_all", 64, 48, (12, 20, 48, 30), 2, 6, "pixel_random", 20),
]


def main():
    assert refdriver.available(), "build oracle/_ref first (make -C oracle ref)"
    only = set(sys.argv[1:])
    for name, w, h, tile, spp, depth, scheme, seed in CASES:
        if only and name not in only:
            continue
        parsed = host.parse_scene_text(open(common.scene_path(name)).read())
        upgraded = host.scene_to_text(parsed)
        with tempfile.TemporaryDirectory() as root:
            refdriver.make_root(root, common.ASSETS, upgraded, "upgraded.scn")
            cfg = host.make_config_text(scene="scenes\\upgraded.scn", width=w, height=h, spp=spp, depth=depth, scheme=scheme)
            ref = refdriver.Ref(root, cfg, seed=seed)
            x0, y0, x1, y1 = tile
            total, avg, m2, paths = ref.render_tile(x0, y0, x1, y1, 0, spp, want_paths=True)
            mats = [ref.material(i) for i in range(ref.lib.ref_num_materials())]
            surfs = [ref.surface(i) for i in range(ref.lib.ref_num_surfaces())]
            np.savez_compressed(
                os.path.join(HERE, name + ".npz"),
                meta=np.array([w, h, x0, y0, x1, y1, spp, depth, 2 if scheme == "pixel_random" else 1, seed], dtype=np.int64),
                upgraded_scene=np.frombuffer(upgraded.encode(), dtype=np.uint8),
                camera=ref.camera(), tables=ref.tables(),
                mat_spds=np.array([m["spds"] for m in mats]),
                mat_flags=np.array([[m["is_black_body"], m["is_emissive"], m["num_lobes"], m["dir_func"], m["spd_mask"]] for m in mats], dtype=np.int64),
                mat_lobes=np.array([m["lobes"] + [-1] * (16 - len(m["lobes"])) for m in mats], dtype=np.int64),
                mat_scalars=np.array([[m["shininess"], m["roughness"]] for m in mats]),
                surf_types=np.array([[s[0], s[1]] for s in surfs], dtype=np.int64),
                surf_geom=np.array([s[2] for s in surfs]),
                base_escape=np.array([ref.lib.ref_base_material(), ref.lib.ref_escape_material()], dtype=np.int64),
                paths=paths, film_sum=total, film_mean=avg, film_m2=m2)
        print(name, "paths", paths.shape, "max", float(np.nanmax(paths)))


if __name__ == "__main__":
    main()
