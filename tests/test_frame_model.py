"""The frame of the hemisphere samplers: rotate_from_z in csrc/drt_render.cuh maps a direction q about +z onto the hit normal n.  Three
samplers call it: the inline cosine-weighted hemisphere, the uniform hemisphere and the `ct` sampler.

The function is modelled here in float32, operation by operation as the source writes it, against a rotation about the same normal in
float64 that has no cancellation near -z: c q + a x q + (1 - c)(a.q)/(a.a) a, with a = (-n.y, n.x, 0) and c = n.z.  Its factor
1 / (1 + c) of the reference's form is ill-conditioned there: in float32, n.z rounds to exactly -1 within 2.4e-4 rad of -z while a.a
is still about 6e-8, which made the sampled direction inf / NaN.  The same check runs on the f64 oracle's rotation_between, the
reference the GPU parity tests compare the kernels with.  Runs without a GPU.
"""
import os
import re

import numpy as np
import pytest

import oracledriver

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUH = os.path.join(REPO, "daily-ray-trace_b200", "csrc", "drt_render.cuh")
F32 = np.float32
NORM_MIN = np.finfo(F32).tiny                           # Num<float>::norm_min, 2^-126

# The body of rotate_from_z that the float32 model below restates (comments and whitespace dropped).
MODELLED_BODY = """
    V3<R> a = mk<R>(-n.y, n.x, R(0));
    R c = n.z;
    R p = R(1) + c;
    R d = p * p + dot(a, a);
    V3<R> aq = mk<R>(a.y * q.z, -(a.x * q.z), a.x * q.y - a.y * q.x);
    V3<R> aaq = mk<R>(a.y * aq.z, -(a.x * aq.z), a.x * aq.y - a.y * aq.x);
    V3<R> r = (q + aq) + aaq * r_div(R(2), d);
    bool anti = d < Num<R>::norm_min() && c <= R(0);
    return mk<R>(anti ? -q.x : r.x, anti ? -q.y : r.y, anti ? -q.z : r.z);
"""


def _squash(code):
    return re.sub(r"\s+", "", re.sub(r"/\*.*?\*/", "", code, flags=re.S))


def test_model_is_the_source():
    """The model restates the source: a change to rotate_from_z must come with a change to the model."""
    src = open(CUH).read()
    body = re.search(r"V3<R> rotate_from_z\(V3<R> n, V3<R> q\)\s*\{(.*?)\n\}", src, re.S).group(1)
    assert _squash(body) == _squash(MODELLED_BODY)
    for r, lit in (("float", "0x1p-126f"), ("double", "0x1p-1022")):
        num = re.search(r"template <> struct Num<%s>\s*\{(.*?)\n\};" % r, src, re.S).group(1)
        assert re.search(r"norm_min\(\)\s*\{\s*return %s;" % re.escape(lit), num)


# ------------------------------------------------------------------------------------------------ the float32 model


def _cross(a, b):
    return np.stack([a[:, 1] * b[:, 2] - a[:, 2] * b[:, 1],
                     a[:, 2] * b[:, 0] - a[:, 0] * b[:, 2],
                     a[:, 0] * b[:, 1] - a[:, 1] * b[:, 0]], axis=1)


def _dot(a, b):
    return (a[:, 0] * b[:, 0] + a[:, 1] * b[:, 1]) + a[:, 2] * b[:, 2]


def _rcp(x, ulps):
    """r_rcp_fast: MUFU.RCP (rcp.approx.ftz) -- a subnormal argument is taken as 0, the result is within 1 ulp; `ulps` = -1, 0, +1
    picks the result one float32 below, at, or one above the correctly rounded reciprocal."""
    x = np.where(np.abs(x) < np.finfo(F32).tiny, F32(0), x).astype(F32)
    with np.errstate(divide="ignore"):
        r = (F32(1) / x).astype(F32)
    for _ in range(abs(ulps)):
        r = np.nextafter(r, F32(np.inf) if ulps > 0 else F32(-np.inf)).astype(F32)
    return np.where(np.isinf(r), r, np.where(np.abs(r) < np.finfo(F32).tiny, F32(0), r)).astype(F32)


def rotate_from_z_f32(n, q, ulps=0, reference_form=False):
    """float32 model of rotate_from_z for arrays n, q of shape (K, 3).  nvcc may contract a product and a sum into one FMA, which this
    model rounds twice; the accuracy bounds below leave room for either.  reference_form=True: the reference's factor 1 / (1 + c) and
    its exact test a.a == 0 -- the kernels' form before 2 / ((1 + c)^2 + a.a), kept here to show what the checks catch."""
    n, q = np.asarray(n, F32), np.asarray(q, F32)
    with np.errstate(all="ignore"):
        a = np.stack([-n[:, 1], n[:, 0], np.zeros(len(n), F32)], axis=1)
        c = n[:, 2]
        aq = _cross(a, q)
        aaq = _cross(a, aq)
        if reference_form:
            anti = (_dot(a, a) == 0) & (c <= 0)
            f = F32(1) * _rcp(F32(1) + c, ulps)
        else:
            p = F32(1) + c
            d = p * p + _dot(a, a)
            anti = (d < NORM_MIN) & (c <= 0)
            f = F32(2) * _rcp(d, ulps)
        r = (q + aq) + aaq * f[:, None]
    return np.where(anti[:, None], -q, r).astype(F32)


def rotate_stable_f64(n, q):
    """The rotation taking +z to n (normalised in float64), in the form without cancellation; q at +z, and -q (Q14) at -z: where n is
    exactly -z, and where n is so close to -z that (1 + c)^2 + a.a is below the float32 normal range (within 2^-63 rad), which the
    kernels take as antiparallel."""
    n32 = np.asarray(n, F32)
    with np.errstate(under="ignore"):
        anti = ((F32(1) + n32[:, 2]) ** 2 + n32[:, 0] * n32[:, 0] + n32[:, 1] * n32[:, 1] < NORM_MIN) & (n32[:, 2] <= 0)
    n = np.asarray(n, np.float64)
    n = n / np.linalg.norm(n, axis=1, keepdims=True)
    q = np.asarray(q, np.float64)
    a = np.stack([-n[:, 1], n[:, 0], np.zeros(len(n))], axis=1)
    c, aa = n[:, 2], np.einsum("ij,ij->i", a, a)
    with np.errstate(all="ignore"):
        k = (1.0 - c) * np.einsum("ij,ij->i", a, q) / aa
        out = c[:, None] * q + np.cross(a, q) + k[:, None] * a
    return np.where(anti[:, None], -q, np.where((aa == 0)[:, None], q, out))


# ------------------------------------------------------------------------------------------------ inputs


def _unit_q(rng, k):
    """unit directions in the upper hemisphere about +z, from grazing to straight up, as float32"""
    z = np.concatenate([rng.uniform(0, 1, k - 4), [1.0, 1e-3, 1e-7, 0.5]])
    phi = rng.uniform(0, 2 * np.pi, k)
    r = np.sqrt(1 - z * z)
    return np.stack([r * np.cos(phi), r * np.sin(phi), z], axis=1).astype(F32)


def _tilted(tilt, phi):
    """the float32 unit normal `tilt` rad from -z towards azimuth phi"""
    n = np.stack([np.sin(tilt) * np.cos(phi), np.sin(tilt) * np.sin(phi), -np.cos(tilt)], axis=1)
    return n.astype(F32)


TILTS = np.geomspace(1e-7, np.pi, 240)
AZIMUTHS = np.array([0.0, 0.5 * np.pi, np.pi, 1.5 * np.pi, 0.3, 2.0, 4.4])


def _grid(nq=16, seed=3):
    rng = np.random.default_rng(seed)
    t, p = np.meshgrid(TILTS, AZIMUTHS, indexing="ij")
    normals = _tilted(t.ravel(), p.ravel())
    n = np.repeat(normals, nq, axis=0)
    q = _unit_q(rng, len(n))
    tilt = np.repeat(t.ravel(), nq)
    return n, q, tilt


def _special():
    """exact +-z, signed zeros, and normals next to -z and +z whose float32 a.a is tiny, at the bottom of the normal range, subnormal, or
    underflows to 0"""
    tiny = [1e-12, 1e-15, 1e-18, 2.0 ** -62, 2.0 ** -63, 2.0 ** -64, 1e-20, 1e-22, 3e-23, 2.0 ** -126, 1e-40, 2.0 ** -149]
    rows = [(0, 0, -1), (0, 0, 1), (-0.0, 0, -1), (0, -0.0, -1), (-0.0, -0.0, -1), (-0.0, -0.0, 1), (1, -0.0, 0), (-0.0, 1, -0.0),
            (-1, 0, -0.0)]
    for t in tiny:
        rows += [(t, 0, -1), (0, -t, -1), (-t, t, -1), (t, 0, 1)]
    normals = np.array(rows, F32)
    q = _unit_q(np.random.default_rng(9), 64)
    q = np.concatenate([q, np.array([(1, 0, 0), (0, 1, 0), (-0.6, 0.8, 0), (0, 0, 1)], F32)])
    n = np.repeat(normals, len(q), axis=0)
    return n, np.tile(q, (len(normals), 1))


def _checks(n, q, out):
    """Per input: finite, unit length within 1e-6, within 1e-6 of the float64 rotation per component, and on the side of the surface
    that q.z gives (n.out = q.z within 1e-6)."""
    ref = rotate_stable_f64(n, q)
    o = out.astype(np.float64)
    finite = np.isfinite(o).all(axis=1)
    assert finite.all(), f"{(~finite).sum()} non-finite directions, first at n = {n[~finite][0]}, q = {q[~finite][0]}: {out[~finite][0]}"
    length = np.abs(np.linalg.norm(o, axis=1) - 1)
    err = np.abs(o - ref).max(axis=1)
    nn = n.astype(np.float64) / np.linalg.norm(n.astype(np.float64), axis=1, keepdims=True)
    side = np.abs(np.einsum("ij,ij->i", nn, o) - q[:, 2])
    worst = int(np.argmax(err))
    print(f"\n{len(n)} inputs: max |len - 1| {length.max():.2e}, max error {err.max():.2e} (n = {n[worst]}), max |n.out - q.z| {side.max():.2e}")
    assert length.max() <= 1e-6
    assert err.max() <= 1e-6, f"n = {n[worst]}, q = {q[worst]}: {out[worst]} against {ref[worst]}"
    assert side.max() <= 1e-6
    assert (np.sign(np.einsum("ij,ij->i", nn, o)) == np.sign(q[:, 2]))[q[:, 2] > 1e-6].all()


@pytest.mark.parametrize("ulps", [-1, 0, 1])
def test_tilt_grid(ulps):
    """Tilts from 1e-7 rad to pi (normals from -z over to +z), seven azimuths, 16 directions each; the reciprocal correctly rounded and
    one ulp either side, as MUFU.RCP may return."""
    n, q, _ = _grid()
    _checks(n, q, rotate_from_z_f32(n, q, ulps))


@pytest.mark.parametrize("ulps", [-1, 0, 1])
def test_special_normals(ulps):
    n, q = _special()
    out = rotate_from_z_f32(n, q, ulps)
    _checks(n, q, out)
    with np.errstate(under="ignore"):
        aa = n[:, 0] * n[:, 0] + n[:, 1] * n[:, 1]
    down = (aa < NORM_MIN) & (n[:, 2] < 0)
    assert np.array_equal(out[down], -q[down])                        # Q14: antiparallel gives -q, bit for bit
    assert ((aa > 0) & (aa < NORM_MIN) & (n[:, 2] < 0)).any()        # a.a subnormal: -q, no longer inf / NaN
    rot = (aa >= NORM_MIN) & (n[:, 2] < 0) & (aa < 1e-30)
    assert rot.any() and not np.array_equal(out[rot], -q[rot])        # at the bottom of the normal range: the rotation itself
    up = (n[:, 0] == 0) & (n[:, 1] == 0) & (n[:, 2] > 0)
    assert np.array_equal(np.abs(out[up]), np.abs(q[up]))


def test_reference_form_fails_the_checks():
    """The checks catch the reference's factor 1 / (1 + c) in float32: inf / NaN where n.z rounds to -1 (tilt <= 2.4e-4), errors far
    above 1e-3 up to tilts of 1e-3, and above 1e-6 past 1e-1.  For c >= 0 (tilts from pi/2 on), away from the cancellation, it
    passes."""
    n, q, tilt = _grid()
    out = rotate_from_z_f32(n, q, reference_form=True).astype(np.float64)
    err = np.abs(out - rotate_stable_f64(n, q)).max(axis=1)
    err = np.where(np.isfinite(err), err, np.inf)
    assert np.isinf(err[tilt <= 2e-4]).mean() > 0.9
    assert (err[tilt <= 1e-3] > 1e-3).mean() > 0.9
    assert err[(tilt > 0.1) & (tilt < 0.3)].max() > 1e-6
    assert err[tilt >= np.pi / 2].max() <= 1e-6


# ------------------------------------------------------------------------------------------------ the f64 oracle


def test_oracle_frame_against_stable_form():
    """The f64 oracle's rotation_between (the reference's form, 1 / (1 + c)) on f64 unit normals, as the GPU parity tests use it.  Its
    error grows as eps / tilt^2 towards -z: at most 8 eps / tilt^2 over the grid, i.e. below 1e-6 from tilts of 3e-5 on (the smallest
    tilt of tests/test_gpu_frames.py) and below 1e-9 from 1e-3 on -- far inside those tests' 1e-3 on radiance."""
    rng = np.random.default_rng(5)
    worst = {}
    for t in TILTS[TILTS >= 1e-5]:
        for phi in AZIMUTHS:
            nn = np.array([np.sin(t) * np.cos(phi), np.sin(t) * np.sin(phi), -np.cos(t)])
            nn /= np.linalg.norm(nn)
            qs = _unit_q(rng, 8).astype(np.float64)
            qs /= np.linalg.norm(qs, axis=1, keepdims=True)
            got = np.array([oracledriver.rotate_from_z(nn, qq) for qq in qs])
            err = np.abs(got - rotate_stable_f64(np.tile(nn, (len(qs), 1)), qs)).max()
            worst[t] = max(worst.get(t, 0.0), err)
    eps = np.finfo(np.float64).eps
    ts = np.array(sorted(worst))
    errs = np.array([worst[t] for t in ts])
    print("\n" + ", ".join(f"tilt {t:.1e}: {e:.1e}" for t, e in zip(ts[::24], errs[::24])))
    assert (errs <= 8 * eps / ts ** 2 + 4 * eps).all()
    assert errs[ts >= 3e-5].max() <= 1e-6
    assert errs[ts >= 1e-3].max() <= 1e-9
    # exactly -z and +z: -q and q
    q = np.array([0.3, 0.2, np.sqrt(1 - 0.13)])
    assert np.array_equal(oracledriver.rotate_from_z([0.0, 0.0, -1.0], q), -q)
    assert np.array_equal(oracledriver.rotate_from_z([0.0, 0.0, 1.0], q), q)
