"""GPU tier: the direction samplers on surfaces that face almost straight down -z.

rotate_from_z (csrc/drt_render.cuh) turns a sample about +z into a direction about the hit normal; the inline cosine-weighted sampler,
the uniform hemisphere and the `ct` sampler call it.  In f32 its reference form, a x (a x q) / (1 + n.z), divided by zero once n.z
rounded to -1 (within 2.4e-4 rad of -z) and lost most of its digits up to 1e-3 rad; tests/test_frame_model.py checks the function on
its own.  Here the kernels are compared per path with the f64 oracle on small rooms written in this file: the camera looks along +z at
a panel tilted by a small angle from facing -z, or at the -z pole of a sphere, and lit walls all around make the second bounce depend on
the sampled direction.  The rooms have no edges in view and no occluders between the walls and the lamp, so nearly every path must
agree: >= 99.9 % within 1e-3 (the shipped-scene suite allows 99.5 %), and not one non-finite path.  The same cases with f64 geometry
are the control: they show that what fails in f32 is the arithmetic, not the scene.
"""
import importlib

import numpy as np
import pytest

import common
import oracledriver

cuda = importlib.import_module("daily-ray-trace_b200.cuda")
host = importlib.import_module("daily-ray-trace_b200.host")

pytestmark = pytest.mark.gpu

REL_TOL = 1e-3
TILTS = [0.0, 3e-5, 1e-4, 2e-4, 3e-4, 1e-3, 1e-2]
AZIMUTH = 0.7          # the panel tilts towards (cos 0.7, sin 0.7, 0): both n.x and n.y are non-zero

MATERIALS = """
Material
name air
refract csv air_spec.csv
base_material

Material
name escape
is_black_body true
escape_material

Material
name lamp
emission constant 4.0
is_black_body true

Material
name white
diffuse rgb 0.7, 0.7, 0.7
glossy rgb 0.2, 0.2, 0.2
shininess 16.0
bdsfs bp_diffuse_bdsf, bp_glossy_bdsf
dir_func cos_weighted_sample_hemisphere

Material
name red
diffuse rgb 0.7, 0.1, 0.1
glossy rgb 0.2, 0.2, 0.2
shininess 16.0
bdsfs bp_diffuse_bdsf, bp_glossy_bdsf
dir_func cos_weighted_sample_hemisphere

Material
name green
diffuse rgb 0.1, 0.6, 0.15
glossy rgb 0.2, 0.2, 0.2
shininess 16.0
bdsfs bp_diffuse_bdsf, bp_glossy_bdsf
dir_func cos_weighted_sample_hemisphere

Material
name blue
diffuse rgb 0.1, 0.2, 0.7
glossy rgb 0.3, 0.3, 0.3
shininess 40.0
bdsfs bp_diffuse_bdsf, bp_glossy_bdsf
dir_func cos_weighted_sample_hemisphere

Material
name target_cos
diffuse rgb 0.5, 0.5, 0.4
glossy rgb 0.4, 0.4, 0.4
shininess 24.0
bdsfs bp_diffuse_bdsf, bp_glossy_bdsf
dir_func cos_weighted_sample_hemisphere

Material
name target_uniform
diffuse rgb 0.5, 0.5, 0.4
glossy rgb 0.4, 0.4, 0.4
shininess 24.0
bdsfs bp_diffuse_bdsf, bp_glossy_bdsf
dir_func uniform_sample_hemisphere

Material
name target_ct
refract csv au_spec_n.csv
extinct csv au_spec_k.csv
roughness 0.3
bdsfs ct_conductor_bdsf
dir_func sample_ct_direction
"""


def _v(p):
    return ", ".join(f"{float(x):.24f}" for x in p)      # the scene format has no exponents


def _plane(name, p, pu, pv, material):
    return f"\nSurface\nname {name}\ntype plane\nposition {_v(p)}\npointu {_v(pu)}\npointv {_v(pv)}\nmaterial {material}\n"


def _room(z_far, far_wall, second_lamp):
    """Walls x, y in [-3, 3], z in [-10, z_far] (red left, green right, white floor and ceiling, blue behind the camera), a lamp under
    the ceiling, a second one over the floor if asked for, and a wall at z_far if asked for."""
    s = _plane("floor", (-3, -3, -10), (3, -3, -10), (-3, -3, z_far), "white")
    s += _plane("ceiling", (-3, 3, -10), (3, 3, -10), (-3, 3, z_far), "white")
    s += _plane("left", (-3, -3, -10), (-3, 3, -10), (-3, -3, z_far), "red")
    s += _plane("right", (3, -3, -10), (3, 3, -10), (3, -3, z_far), "green")
    s += _plane("back", (-3, -3, -10), (3, -3, -10), (-3, 3, -10), "blue")
    if far_wall:
        s += _plane("far", (-3, -3, z_far), (3, -3, z_far), (-3, 3, z_far), "white")
    s += _plane("lamp", (-1, 2.9, -5), (1, 2.9, -5), (-1, 2.9, -3), "lamp")
    if second_lamp:
        s += _plane("lamp2", (-0.5, -2.9, -4), (0.5, -2.9, -4), (-0.5, -2.9, -3), "lamp")
    return s


def _camera(fov):
    return f"Camera\nposition 0.0, 0.0, -6.0\ntarget 0.0, 0.0, 0.0\nroll 0.0\nfov {fov:.24f}\nfdepth 6.0\nflength 0.5\naperture 0.0\n"


def panel_scene(tilt, material, second_lamp=False):
    """An 8 x 8 panel through the origin whose normal is `tilt` rad from -z; it reaches through the side walls, so the camera (fov 20
    degrees, 2.1 x 2.1 of the panel in view) sees no edge.  tilt = 0 is an axis-aligned plane."""
    n = np.array([np.sin(tilt) * np.cos(AZIMUTH), np.sin(tilt) * np.sin(AZIMUTH), -np.cos(tilt)])
    u = np.array([1.0, 0.0, 0.0]) - n[0] * n
    u /= np.linalg.norm(u)
    v = np.cross(n, u)
    p = -4 * u - 4 * v
    return _camera(20.0) + MATERIALS + _room(1.0, False, second_lamp) + _plane("panel", p, p + 8 * u, p + 8 * v, material)


def sphere_scene(material):
    """A unit sphere with its -z pole at the origin, seen through a field of view 1.4e-3 wide at the pole: the tile's normals tilt from 0
    to 1e-3 rad from -z."""
    fov = float(np.degrees(2 * np.arctan(7e-4 / 6.0)))
    sphere = f"\nSurface\nname ball\ntype sphere\nposition 0.0, 0.0, 1.0\nradius 1.0\nmaterial {material}\n"
    return _camera(fov) + MATERIALS + _room(3.0, True, False) + sphere


def load(text, w, h, spp, depth):
    cfg = host.parse_config_text(host.make_config_text(width=w, height=h, spp=spp, depth=depth))
    tables = host.load_tables(cfg, common.ASSETS)
    scene, camera = host.build_scene(host.parse_scene_text(text), tables, common.ASSETS, w, h)
    return cfg, tables, scene, camera


@pytest.fixture(scope="module")
def ctx():
    c = cuda.Context(0)
    yield c
    c.close()


def _parity(ctx, text, geometry, mode, w=32, h=24, spp=8, depth=3, seed=0x5EED, deep=False):
    cfg, tables, scene, camera = load(text, w, h, spp, depth)
    ctx.upload_scene(scene, camera, tables)
    ctx.set_geometry_precision(geometry)
    prm = oracledriver.params(w, h, 0, spp, depth, cfg.pixel_scheme, seed)
    kernel = ctx.render_kernel_info(prm)[0]
    real = "float" if geometry == cuda.GEOMETRY_F32 else "double"
    assert kernel.startswith(f"drt::render_kernel<{real},") and kernel.split(",")[2] == str(mode), kernel
    assert kernel.endswith(",true>" if deep else ",false>"), kernel
    gpu = ctx.sample_paths(prm, 0, 0, w, h)
    st = ctx.stats()
    _, _, _, ref, cnt = oracledriver.render_tile(scene, camera, prm, 0, 0, w, h, want_paths=True)
    err = common.path_errors(gpu, ref)
    ok = (err <= REL_TOL).mean()
    nonfinite = int((~np.isfinite(gpu)).any(axis=-1).sum())
    second = 1 - (st.terminated_at_depth[0] + st.terminated_at_depth[1]) / st.paths
    print(f"\n[{kernel}] {err.size} paths: within {REL_TOL:g} {100 * ok:.3f} %, max err {err.max():.2e}, non-finite {nonfinite}, "
          f"shade a second bounce {100 * second:.1f} %")
    assert np.isfinite(ref).all()
    assert nonfinite == 0
    assert ok >= 0.999
    assert st.paths == cnt.paths == err.size
    assert second >= 0.9                      # the sampled direction is cast, and what it hits is shaded
    for a, b in ((st.closest_rays, cnt.closest_rays), (st.shadow_rays, cnt.shadow_rays), (st.rng_draws, cnt.rng_draws)):
        assert abs(a - b) <= 0.001 * b + 8
    return scene


# material of the panel or sphere, extra lamp, kernel mode in f32 geometry
CASES = [("target_cos", False, 1), ("target_uniform", False, 1), ("target_ct", False, 2), ("target_cos", True, 0)]
CASE_IDS = ["cosine", "uniform", "ct", "two_lamps"]


@pytest.mark.parametrize("geometry", [cuda.GEOMETRY_F32, cuda.GEOMETRY_F64], ids=["f32", "f64"])
@pytest.mark.parametrize("material,second_lamp,mode", CASES, ids=CASE_IDS)
@pytest.mark.parametrize("tilt", TILTS)
def test_tilted_panel(ctx, tilt, material, second_lamp, mode, geometry):
    scene = _parity(ctx, panel_scene(tilt, material, second_lamp), geometry, mode if geometry == cuda.GEOMETRY_F32 else 0)
    nz = scene.surfaces[scene.num_surfaces - 1].normal[2]
    # the regime of each tilt: n.z of the f32 normal rounds to -1 exactly below 2.4e-4 rad
    assert (np.float32(abs(nz)) == 1) == (tilt < 2.4e-4)


@pytest.mark.parametrize("geometry", [cuda.GEOMETRY_F32, cuda.GEOMETRY_F64], ids=["f32", "f64"])
@pytest.mark.parametrize("material,mode", [("target_cos", 1), ("target_uniform", 1), ("target_ct", 2)], ids=CASE_IDS[:3])
def test_sphere_pole(ctx, material, mode, geometry):
    _parity(ctx, sphere_scene(material), geometry, mode if geometry == cuda.GEOMETRY_F32 else 0)


@pytest.mark.parametrize("geometry", [cuda.GEOMETRY_F32, cuda.GEOMETRY_F64], ids=["f32", "f64"])
def test_deep_render(ctx, geometry):
    """depth 40: the bounces past the records' shared-memory part go to the overflow rows in global memory; in the closed room a path
    ends only on the lamp, and comes back to the panel many times"""
    _parity(ctx, panel_scene(1e-4, "target_cos"), geometry, 1 if geometry == cuda.GEOMETRY_F32 else 0, w=32, h=16, spp=4, depth=40,
            deep=True)


def test_film_tilted_panel(ctx):
    """A whole film at 64 spp through render_device: every plane finite, and the film within test_gpu_replay's tolerances of the oracle
    (sum, mean and M2 within 2e-3 for >= 99 % of the pixels)."""
    import torch
    w, h, spp, depth = 16, 12, 64, 3
    cfg, tables, scene, camera = load(panel_scene(1e-4, "target_cos"), w, h, spp, depth)
    ctx.upload_scene(scene, camera, tables)
    ctx.set_geometry_precision(cuda.GEOMETRY_F32)
    prm = oracledriver.params(w, h, 0, spp, depth, cfg.pixel_scheme, 21)
    assert ctx.render_kernel_info(prm)[0] == "drt::render_kernel<float,5,1,true,false>"
    n = scene.num_wavelengths
    planes = [torch.zeros(w * h * n, device="cuda"), torch.zeros(w * h, device="cuda"),
              torch.zeros(w * h * n, device="cuda"), torch.zeros(w * h * n, device="cuda")]
    ctx.render_device(prm, cuda.film_from_tensors(*planes))
    torch.cuda.synchronize()
    film = {k: t.cpu().numpy().reshape(w * h, -1) for k, t in zip(("sum", "filter", "mean", "m2"), planes)}
    for k, v in film.items():
        assert np.isfinite(v).all(), k
    assert np.array_equal(film["filter"][:, 0], np.full(w * h, spp, np.float32))
    o_sum, o_avg, o_m2, _, _ = oracledriver.render_tile(scene, camera, prm, 0, 0, w, h)
    for name, ref in (("sum", o_sum[:, :n]), ("mean", o_avg), ("m2", o_m2)):
        rel = (np.abs(film[name].astype(np.float64) - ref) / np.maximum(np.abs(ref), 1e-5 * np.abs(ref).max())).max(axis=1)
        print(f"\nfilm {name}: max rel {rel.max():.2e}, pixels over 2e-3: {(rel > 2e-3).sum()} of {w * h}")
        assert (rel <= 2e-3).mean() >= 0.99, name
