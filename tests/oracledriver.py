"""TEST INFRASTRUCTURE: ctypes wrapper of oracle/libdrt_oracle.so, the plain-C f64 restatement of the hot path.
Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg may use it -- as the checker, never the product."""
import ctypes as C
import importlib
import os
import subprocess

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(REPO, "oracle")
ORACLE_LIB = os.path.join(ORACLE_DIR, "libdrt_oracle.so")

_structs = importlib.import_module("daily-ray-trace_b200._structs")


class Counters(C.Structure):
    _fields_ = [("paths", C.c_uint64), ("closest_rays", C.c_uint64), ("shadow_rays", C.c_uint64),
                ("shaded_bounces", C.c_uint64), ("rng_draws", C.c_uint64), ("terminated_at_depth", C.c_uint64 * 8),
                ("reached_depth_cap", C.c_uint64)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        # make rebuilds a library older than drt_oracle.c (one without the newer exports) and does nothing otherwise
        subprocess.check_call(["make", "-s", "-C", ORACLE_DIR, "oracle"], stdout=subprocess.DEVNULL)
        L = C.CDLL(ORACLE_LIB)
        dp = C.POINTER(C.c_double)
        L.drt_oracle_sample.argtypes = [C.POINTER(_structs.Scene), C.POINTER(_structs.Camera), C.POINTER(_structs.RenderParams),
                                        C.c_uint32, C.c_uint32, C.c_uint32, dp, dp, C.POINTER(Counters)]
        L.drt_oracle_sample.restype = None
        L.drt_oracle_render_tile.argtypes = [C.POINTER(_structs.Scene), C.POINTER(_structs.Camera), C.POINTER(_structs.RenderParams),
                                             C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, dp, dp, dp, dp, C.POINTER(Counters)]
        L.drt_oracle_render_tile.restype = None
        L.drt_oracle_bdsf.argtypes = [C.POINTER(_structs.Scene), C.c_uint32, C.c_uint32, C.c_uint32, dp, dp, dp, dp]
        L.drt_oracle_bdsf.restype = None
        L.drt_oracle_primary_material.argtypes = [C.POINTER(_structs.Scene), C.POINTER(_structs.Camera), C.POINTER(_structs.RenderParams),
                                                  C.c_uint32, C.c_uint32, C.c_uint32]
        L.drt_oracle_primary_material.restype = C.c_int
        L.drt_oracle_rotate_from_z.argtypes = [dp, dp, dp]
        L.drt_oracle_rotate_from_z.restype = None
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def params(width, height, s0, s1, max_depth=4, scheme=_structs.PIXEL_RANDOM, seed=0):
    return _structs.RenderParams(width, height, s0, s1, max_depth, scheme, seed)


def sample(scene, camera, prm, x, y, s):
    out = np.zeros(scene.num_wavelengths)
    filt = C.c_double()
    lib().drt_oracle_sample(C.byref(scene), C.byref(camera), C.byref(prm), x, y, s, _p(out), C.byref(filt), None)
    return out


def primary_material(scene, camera, prm, x, y, s):
    """Index of the material the camera ray of path (x, y, s) hits first."""
    return lib().drt_oracle_primary_material(C.byref(scene), C.byref(camera), C.byref(prm), x, y, s)


def bdsf(scene, surf_mat, inc_mat, trans_mat, normal, out_dir, in_dir):
    """The material's bdsf() sum for one incoming direction (the arguments of refdriver.Ref.bdsf)."""
    a = [np.ascontiguousarray(v, dtype=np.float64) for v in (normal, out_dir, in_dir)]
    res = np.zeros(scene.num_wavelengths)
    lib().drt_oracle_bdsf(C.byref(scene), surf_mat, inc_mat, trans_mat, _p(a[0]), _p(a[1]), _p(a[2]), _p(res))
    return res


def rotate_from_z(normal, q):
    """q, a direction about +z, rotated onto `normal` by the reference's frame (rotation_between((0,0,1), normal))."""
    a = [np.ascontiguousarray(v, dtype=np.float64) for v in (normal, q)]
    res = np.zeros(3)
    lib().drt_oracle_rotate_from_z(_p(a[0]), _p(a[1]), _p(res))
    return res


def render_tile(scene, camera, prm, x0, y0, x1, y1, want_paths=False):
    """Returns (sum[(npx, N+1)], avg[(npx, N)], m2[(npx, N)], paths[(npx, spp, N)] or None, Counters)."""
    n = scene.num_wavelengths
    npx = (x1 - x0) * (y1 - y0)
    spp = prm.sample_end - prm.sample_begin
    total = np.zeros((npx, n + 1))
    avg = np.zeros((npx, n))
    m2 = np.zeros((npx, n))
    paths = np.zeros((npx, spp, n)) if want_paths else None
    cnt = Counters()
    lib().drt_oracle_render_tile(C.byref(scene), C.byref(camera), C.byref(prm), x0, y0, x1, y1, _p(total), _p(avg), _p(m2),
                                 _p(paths) if want_paths else None, C.byref(cnt))
    return total, avg, m2, paths, cnt
