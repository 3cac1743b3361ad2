"""CPU tier: the factorisation behind the classed kernel, against the REFERENCE's own bdsf() (oracle/_ref, daily_ray_trace.c:215-229).

The classed kernel never evaluates a specular material's lobe list per wavelength.  It stores, per bounce, two scalars (c0, c1) picked
from a table built at scene upload (drt_cuda_plan_scene: the lobe walk with the stale-scratch rule, Q7) and shades c0 + c1 X(lambda) with
X = the mirror spectrum, the dielectric reflectance or the conductor reflectance, the latter two from per-wavelength ratios formed at
upload (rel = ir / tr;  A = eta^2 - kappa^2, B = 4 eta^2 kappa^2 with eta = tr / ir, kappa = te / ir).  Here the same formulas run in
numpy f64 on the reference's own material spectra and are compared with what the reference's bdsf() returns for exact reflection and
refraction directions, both orientations of the surface.  Where the reference build is absent, the checker is the oracle's bdsf()
(oracle/drt_oracle.c), the C restatement that tests/test_golden.py pins bit-for-bit to the reference's per-path spectra of this scene."""
import functools
import importlib
import os
import types

import numpy as np
import pytest

import common
import oracledriver
import refdriver

cuda = importlib.import_module("daily-ray-trace_b200.cuda")

EMISSION, DIFFUSE, GLOSSY, MIRROR, REFRACT, EXTINCT = range(6)


def dot(a, b):                       # geometry.c: a.x*b.x + a.y*b.y + a.z*b.z, left to right, no contraction
    return (a[0] * b[0] + a[1] * b[1]) + a[2] * b[2]


def reflect(v, n):                   # vec3_reflect, geometry.c:85-90
    f = 2.0 * dot(v, n)
    return np.array([v[0] - f * n[0], v[1] - f * n[1], v[2] - f * n[2]])


def transmit(v, n, ir, tr):          # vec3_transmit, geometry.c:92-106
    if tr == 0.0:
        return np.full(3, np.nan)
    vn = dot(v, n)
    rel = ir / tr
    m = np.array([vn * n[0], vn * n[1], vn * n[2]])
    w = m - v
    perp = -(rel * w)
    with np.errstate(invalid="ignore"):
        pd = -np.sqrt(1.0 - dot(perp, perp))
    return np.array([perp[0] + pd * n[0], perp[1] + pd * n[1], perp[2] + pd * n[2]])


def dielectric_rel(rel, c):          # fresnel_dielectric_rel of csrc/drt_render.cuh (bdsf.c:44-76 with the amplitudes divided by tr, Q9 kept)
    ts = rel * rel * (1.0 - c * c)
    tc = np.sqrt(np.maximum(1.0 - ts * ts, 0.0))
    a, b = rel * tc, rel * c
    par, per = (c - a) / (c + a), (b - tc) / (b + tc)
    return np.where(ts >= 1.0, 1.0, 0.5 * (par * par + per * per))


def conductor_ab(A, B, c):           # fresnel_conductor_ab of csrc/drt_render.cuh (bdsf.c:78-101 on precomputed ratios)
    cs, ss = c * c, 1.0 - c * c
    r = A - ss
    apb = np.sqrt(r * r + B)
    a = np.sqrt(np.maximum(0.5 * (apb + r), 0.0))
    s, t = apb + cs, 2.0 * a * c
    u, v = cs * apb + ss * ss, t * ss
    par = (s - t) / (s + t)
    return 0.5 * (par + par * (u - v) / (u + v))


@pytest.fixture(scope="module")
def loaded(tmp_path_factory):
    host = importlib.import_module("daily-ray-trace_b200.host")
    cfg, tables, scene, camera = common.load("classed_all", 16, 16, 1, 4)
    if refdriver.available():
        root = str(tmp_path_factory.mktemp("ref_root"))
        parsed = host.parse_scene_text(open(common.scene_path("classed_all")).read())
        refdriver.make_root(root, common.ASSETS, host.scene_to_text(parsed), "upgraded.scn")
        ref = refdriver.Ref(root, host.make_config_text(scene="scenes\\upgraded.scn", width=16, height=16, spp=1, depth=4), seed=1)
    else:
        ref = types.SimpleNamespace(bdsf=functools.partial(oracledriver.bdsf, scene))
    mode, classes, consts = cuda.plan_scene(scene, camera)
    names = {scene.materials[m].name.decode(): m for m in range(scene.num_materials)}
    return ref, scene, classes, consts, names


@pytest.mark.parametrize("material", ["mirror", "chrome", "glass", "clear"])
@pytest.mark.parametrize("inside", [False, True])
def test_specular_materials_are_c0_plus_c1_x(loaded, material, inside):
    ref, scene, classes, consts, names = loaded
    m, base = names[material], scene.base_material
    assert classes[m] == 1
    if inside and material == "chrome":
        pytest.skip("the reference dereferences the base medium's missing extinction spectrum here (fs_conductor_reflectance, bdsf.c:78-101); "
                    "the CUDA path takes kappa = 0")
    n = scene.num_wavelengths
    spd = lambda mat, k: np.array(scene.materials[mat].spd[k][:n])
    have_k = lambda mat: bool(scene.materials[mat].spd_mask & (1 << EXTINCT))
    inc, trans = (m, base) if inside else (base, m)                  # Q11: seen from inside, the media swap
    ir, tr = spd(inc, REFRACT), spd(trans, REFRACT)
    te = spd(trans, EXTINCT) if have_k(trans) else np.zeros(n)
    lobes = list(scene.materials[m].lobes[:scene.materials[m].num_lobes])
    basis = "mirror" if 2 in lobes else "dielectric" if (4 in lobes or 5 in lobes) else "conductor"
    rng = np.random.default_rng(5)
    for _ in range(6):
        nrm = rng.normal(size=3); nrm /= np.sqrt(dot(nrm, nrm))
        out = rng.normal(size=3); out /= np.sqrt(dot(out, out))
        if dot(nrm, out) < 0:
            out = -out
        on_dot = dot(nrm, out)
        i630 = int((630.0 - scene.min_wl) / scene.wl_interval)
        directions = {0: rng.normal(size=3), 1: reflect(-out, nrm), 2: transmit(-out, nrm, ir[i630], tr[i630])}
        if basis == "mirror":
            X = spd(m, MIRROR)
        elif basis == "dielectric":
            X = dielectric_rel(ir / tr, on_dot)
        else:
            eta, kap = tr / ir, te / ir
            X = conductor_ab(eta * eta - kap * kap, 4.0 * eta * eta * kap * kap, on_dot)
        for match, d in directions.items():
            if np.isnan(d).any():
                continue                                             # total internal reflection: no refraction direction
            got = float(consts[m][match][0]) + float(consts[m][match][1]) * X
            want = ref.bdsf(m, inc, trans, nrm, out, d)
            assert np.allclose(got, want, rtol=1e-11, atol=1e-13), (material, inside, match, np.abs(got - want).max())
            if match == 1 and material != "clear":
                assert np.abs(want).max() > 0                               # the reflection-gated lobes did fire for the exact direction


def test_rough_conductor_is_w_times_f_of_the_half_vector(loaded):
    """ct_conductor_bdsf (bdsf.c:174-186) = [D G1 / (4 on_dot)] * F(|n.m|, lambda): the bracket is what ct_weight stores, F comes from the
    conductor rows at the micro-normal cosine."""
    ref, scene, classes, consts, names = loaded
    m, base = names["rough_gold"], scene.base_material
    assert classes[m] == 2
    n = scene.num_wavelengths
    ir = np.array(scene.materials[base].spd[REFRACT][:n]); tr = np.array(scene.materials[m].spd[REFRACT][:n]); te = np.array(scene.materials[m].spd[EXTINCT][:n])
    rough = scene.materials[m].roughness
    rng = np.random.default_rng(9)
    for _ in range(8):
        nrm = rng.normal(size=3); nrm /= np.sqrt(dot(nrm, nrm))
        out = rng.normal(size=3); out /= np.sqrt(dot(out, out))
        inn = rng.normal(size=3); inn /= np.sqrt(dot(inn, inn))
        if dot(nrm, out) < 0: out = -out
        if dot(nrm, inn) < 0: inn = -inn
        on_dot = dot(nrm, out)
        h = out + inn; h /= np.sqrt(dot(h, h))
        d = dot(nrm, h)
        r2 = rough * rough
        gg = r2 / (np.pi * d ** 4 * (r2 + (1.0 / (d * d) - 1.0)) ** 2) if d > 0 else 0.0               # ggx, bdsf.c:3-20
        quot = abs(dot(out, h) / dot(out, nrm))
        att = 2.0 / (1.0 + np.sqrt(1.0 + r2 * (1.0 / dot(out, nrm) ** 2 - 1.0))) if quot > 0 else 0.0    # G1(out), bdsf.c:22-42
        w = gg * att / (4.0 * on_dot)
        eta, kap = tr / ir, te / ir
        got = w * conductor_ab(eta * eta - kap * kap, 4.0 * eta * eta * kap * kap, abs(d))
        want = ref.bdsf(m, base, m, nrm, out, inn)
        assert np.allclose(got, want, rtol=1e-9, atol=1e-12), np.abs(got - want).max()


@pytest.mark.parametrize("material,nd,ng", [("grey", 1, 1), ("red", 1, 0), ("sheen", 0, 2), ("thick", 2, 1)])
def test_plastics_are_lobe_multiplicities_times_two_weights(loaded, material, nd, ng):
    """A plastic's bdsf() sum is nd * w_d * D + ng * w_g * G (both lobes always write, so a lobe listed k times counts k times,
    daily_ray_trace.c:215-229): the multiplicities live in the material's D, G block (SpdIndex::plastic2), the kernel computes the two
    weights w_d = |n.in| / pi and w_g = max(0, n.h)^shininess |n.in| (bdsf.c:105-119)."""
    ref, scene, classes, consts, names = loaded
    m, base = names[material], scene.base_material
    assert classes[m] == 0
    n = scene.num_wavelengths
    mat = scene.materials[m]
    lobes = list(mat.lobes[:mat.num_lobes])
    assert (lobes.count(0), lobes.count(1)) == (nd, ng)
    D = np.array(mat.spd[DIFFUSE][:n]) if mat.spd_mask & (1 << DIFFUSE) else np.zeros(n)
    G = np.array(mat.spd[GLOSSY][:n]) if mat.spd_mask & (1 << GLOSSY) else np.zeros(n)
    rng = np.random.default_rng(3)
    for _ in range(6):
        nrm = rng.normal(size=3); nrm /= np.sqrt(dot(nrm, nrm))
        out = rng.normal(size=3); out /= np.sqrt(dot(out, out))
        inn = rng.normal(size=3); inn /= np.sqrt(dot(inn, inn))
        if dot(nrm, out) < 0: out = -out
        h = out + inn; h /= np.sqrt(dot(h, h))
        cos_in = abs(dot(nrm, inn))
        w_d = cos_in / np.pi
        w_g = max(0.0, dot(nrm, h)) ** mat.shininess * cos_in
        got = nd * w_d * D + ng * w_g * G
        want = ref.bdsf(m, base, m, nrm, out, inn)
        assert np.allclose(got, want, rtol=1e-12, atol=1e-15), (material, np.abs(got - want).max())
