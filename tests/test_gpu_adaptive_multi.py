"""GPU tier: adaptive sampling sharded by rows (drt_cuda_render_device_adaptive_rows, drt_cuda_film_read_rows,
drt_cuda_render_host_multi_adaptive).

A pixel's film depends only on its own paths (Philox streams keyed by pixel and sample index) and on the fixed order in which one warp
folds a batch of 32 of them in, not on the device or warp that takes the pixel.  So the rows y = rank (mod count) of every rank,
rendered into one film, must equal the one-device adaptive render bit for bit, and so must the multi-device host call."""
import importlib

import numpy as np
import pytest
import torch

import common
import oracledriver
import test_gpu_adaptive
import test_wavelength_grids_model as grids

cuda = importlib.import_module("daily-ray-trace_b200.cuda")

pytestmark = pytest.mark.gpu

E_ARG, E_UNSUPPORTED, E_STATE = -103, -104, -105
NAN_BITS = 0x7FC00BAD                      # a quiet NaN that no render writes
COUNTS = (1, 2, 3, 8, 16)                  # 16 > 12 rows: ranks 12 .. 15 have no rows
WORK = ("paths", "closest_rays", "shadow_rays", "shaded_bounces", "rng_draws")


@pytest.fixture(scope="module")
def ctx():
    c = cuda.Context(0)
    yield c
    c.close()


def _setup(ctx, scene, w, h, cap, depth, seed, n=None):
    grid = {}
    if n is not None:
        lo, hi, step = next((lo, hi, step) for gn, ns, lo, hi, step in grids.RENDER_GRIDS if gn == n)
        grid = dict(min_wl=lo, max_wl=hi, wl_interval=step)
    cfg, tables, sc, camera = common.load(scene, w, h, cap, depth, **grid)
    ctx.upload_scene(sc, camera, tables)
    ctx.set_geometry_precision(cuda.GEOMETRY_F32)
    return sc, oracledriver.params(w, h, 0, cap, depth, cfg.pixel_scheme, seed)


def _planes(w, h, n, fill_bits=None):
    planes = [torch.zeros(w * h * n, device="cuda"), torch.zeros(w * h, device="cuda"),
              torch.zeros(w * h * n, device="cuda"), torch.zeros(w * h * n, device="cuda")]
    if fill_bits is not None:
        for t in planes:
            t.view(torch.int32).fill_(fill_bits)
    return planes, cuda.film_from_tensors(*planes)


def _bits(planes, w, h, n):
    """The four planes as uint32 bit patterns, rows of the frame as the leading axis: {name: [h, w(, n)]}."""
    torch.cuda.synchronize()
    out = {}
    for k, t in zip(("sum", "filter", "mean", "m2"), planes):
        a = t.cpu().numpy().view(np.uint32)
        out[k] = a.reshape(h, w) if k == "filter" else a.reshape(h, w, n)
    return out


def _host_bits(film, w, h):
    return {k: v.view(np.uint32).reshape((h, w) + v.shape[1:]) for k, v in film.items()}


def _work(s):
    return np.array([getattr(s, k) for k in WORK], dtype=np.uint64)


def _whole(ctx, prm, rel_error, mn, w, h, n):
    planes, film = _planes(w, h, n)
    ctx.render_device_adaptive(prm, rel_error, mn, film)
    work = _work(ctx.stats())
    return _bits(planes, w, h, n), work


# the seven scene cases of the one-device adaptive tests (modes 1, 2 and 0, and the depth-100 render), plus init_cornell on the
# 32-wavelength grid (NS = 2)
ROW_CASES = [c[:7] + (None,) for c in test_gpu_adaptive.CASES] + [("init_cornell", 16, 12, 2048, 4, 0.05, 64, 32)]


@pytest.mark.parametrize("scene,w,h,cap,depth,rel_error,min_samples,n_grid", ROW_CASES)
def test_rows_of_all_ranks_are_the_whole_frame(ctx, scene, w, h, cap, depth, rel_error, min_samples, n_grid):
    sc, prm = _setup(ctx, scene, w, h, cap, depth, 31, n_grid)
    n = sc.num_wavelengths
    ref, ref_work = _whole(ctx, prm, rel_error, min_samples, w, h, n)
    assert len(np.unique(ref["filter"])) > 1                      # it adapts
    for count in COUNTS:
        planes, film = _planes(w, h, n, NAN_BITS)                 # every pixel must be written by exactly its rank
        work = np.zeros(len(WORK), np.uint64)
        for rank in range(count):
            ctx.render_device_adaptive_rows(prm, rel_error, min_samples, film, count, rank)
            s = ctx.stats()
            work += _work(s)
            rows = len(range(rank, h, count))
            assert s.kernel_launches == (1 if rows else 0), (count, rank)
            if not rows:
                assert not _work(s).any(), (count, rank)
        got = _bits(planes, w, h, n)
        for k in got:
            assert np.array_equal(got[k], ref[k]), (scene, count, k)
        assert np.array_equal(work, ref_work), (scene, count, work, ref_work)
    print(f"\n{scene} N={n}: rows of {COUNTS} ranks equal the whole-frame render bit for bit; {ref_work[0]} paths")


def test_rows_leave_other_rows_untouched(ctx):
    w, h, cap, count, rank = 16, 12, 1024, 3, 1
    sc, prm = _setup(ctx, "cornell_plane_light", w, h, cap, 4, 5)
    n = sc.num_wavelengths
    ref, _ = _whole(ctx, prm, 0.05, 64, w, h, n)
    planes, film = _planes(w, h, n, NAN_BITS)
    ctx.render_device_adaptive_rows(prm, 0.05, 64, film, count, rank)
    got = _bits(planes, w, h, n)
    own = np.arange(h) % count == rank
    for k in got:
        assert np.array_equal(got[k][own], ref[k][own]), k
        assert np.all(got[k][~own] == NAN_BITS), k


def test_rows_accumulate_continue_a_uniform_film(ctx):
    """Uniform [0, 256), then adaptive [256, 2048) with accumulate = 1 rank by rank: the film of render_device_adaptive's accumulate."""
    w, h, a, cap, rel_error, mn = 16, 12, 256, 2048, 0.02, 64
    sc, prm = _setup(ctx, "init_cornell", w, h, cap, 4, 9)
    n = sc.num_wavelengths
    first = oracledriver.params(w, h, 0, a, 4, prm.pixel_scheme, 9)
    rest = oracledriver.params(w, h, a, cap, 4, prm.pixel_scheme, 9)
    ref_planes, ref_film = _planes(w, h, n)
    ctx.render_device(first, ref_film)
    ctx.render_device_adaptive(rest, rel_error, mn, ref_film, accumulate=True)
    ref_work = _work(ctx.stats())
    ref = _bits(ref_planes, w, h, n)
    counts = ref["filter"].view(np.float32)
    assert np.all(counts > a) and len(np.unique(counts)) > 1
    for count in (2, 3, 16):
        planes, film = _planes(w, h, n)
        ctx.render_device(first, film)
        work = np.zeros(len(WORK), np.uint64)
        for rank in range(count):
            ctx.render_device_adaptive_rows(rest, rel_error, mn, film, count, rank, accumulate=True)
            work += _work(ctx.stats())
        got = _bits(planes, w, h, n)
        for k in got:
            assert np.array_equal(got[k], ref[k]), (count, k)
        assert np.array_equal(work, ref_work), count


def test_film_read_rows_lands_at_global_rows(ctx):
    w, h = 16, 12
    sc, prm = _setup(ctx, "init_cornell", w, h, 64, 4, 2)
    n = sc.num_wavelengths
    planes, film = _planes(w, h, n)
    ctx.render_device(prm, film)
    dev = _bits(planes, w, h, n)
    for count, rank in ((1, 0), (3, 2), (5, 0), (16, 11), (16, 12)):
        host = {"sum": np.full((w * h, n), NAN_BITS, np.uint32), "filter": np.full(w * h, NAN_BITS, np.uint32),
                "mean": np.full((w * h, n), NAN_BITS, np.uint32), "m2": np.full((w * h, n), NAN_BITS, np.uint32)}
        hf = cuda.Film(host["sum"].ctypes.data, host["filter"].ctypes.data, host["mean"].ctypes.data, host["m2"].ctypes.data)
        ctx.film_read_rows(film, w, h, count, rank, hf)
        torch.cuda.synchronize()
        got = _host_bits(host, w, h)
        own = np.arange(h) % count == rank
        for k in got:
            assert np.array_equal(got[k][own], dev[k][own]), (count, rank, k)
            assert np.all(got[k][~own] == NAN_BITS), (count, rank, k)


def _code(call, message=None):
    with pytest.raises(cuda.CudaError) as e:
        call()
    assert message is None or message in str(e.value), str(e.value)
    return e.value.code


def test_row_shard_error_codes(ctx):
    w, h = 8, 8
    sc, prm = _setup(ctx, "init_cornell", w, h, 256, 4, 1)
    n = sc.num_wavelengths
    planes, film = _planes(w, h, n)
    host = {k: np.zeros((w * h, n) if k != "filter" else w * h, np.float32) for k in ("sum", "filter", "mean", "m2")}
    hf = cuda.Film(host["sum"].ctypes.data, host["filter"].ctypes.data, host["mean"].ctypes.data, host["m2"].ctypes.data)
    L = cuda.lib()
    ada = cuda.Adaptive(0.05, 64)
    for count, rank in ((0, 0), (17, 0), (2, -1), (2, 2), (16, 16)):
        assert _code(lambda: ctx.render_device_adaptive_rows(prm, 0.05, 64, film, count, rank)) == E_ARG, (count, rank)
        assert _code(lambda: ctx.film_read_rows(film, w, h, count, rank, hf)) == E_ARG, (count, rank)
    assert _code(lambda: cuda.render_host_multi_adaptive([ctx] * 17, prm, 0.05, 64)) == E_ARG
    assert _code(lambda: cuda._check(L.drt_cuda_render_host_multi_adaptive((cuda.C.c_void_p * 1)(ctx._h), 0, cuda.C.byref(prm),
                                                                         cuda.C.byref(ada), cuda.C.byref(hf)))) == E_ARG
    # NULL pointers
    null = cuda.Film()
    assert _code(lambda: ctx.render_device_adaptive_rows(prm, 0.05, 64, null, 2, 0)) == E_ARG
    assert _code(lambda: ctx.film_read_rows(null, w, h, 2, 0, hf)) == E_ARG
    assert _code(lambda: ctx.film_read_rows(film, w, h, 2, 0, null)) == E_ARG
    assert _code(lambda: cuda._check(L.drt_cuda_render_device_adaptive_rows(ctx._h, None, cuda.C.byref(ada), cuda.C.byref(film), 0, 2, 0, None))) == E_ARG
    assert _code(lambda: cuda._check(L.drt_cuda_render_device_adaptive_rows(ctx._h, cuda.C.byref(prm), None, cuda.C.byref(film), 0, 2, 0, None))) == E_ARG
    assert _code(lambda: cuda._check(L.drt_cuda_render_device_adaptive_rows(None, cuda.C.byref(prm), cuda.C.byref(ada), cuda.C.byref(film), 0, 2, 0, None))) == E_ARG
    assert _code(lambda: cuda._check(L.drt_cuda_render_host_multi_adaptive(None, 1, cuda.C.byref(prm), cuda.C.byref(ada), cuda.C.byref(hf)))) == E_ARG
    assert _code(lambda: cuda._check(L.drt_cuda_render_host_multi_adaptive((cuda.C.c_void_p * 1)(None), 1, cuda.C.byref(prm), cuda.C.byref(ada),
                                                                         cuda.C.byref(hf)))) == E_ARG
    assert _code(lambda: cuda._check(L.drt_cuda_render_host_multi_adaptive((cuda.C.c_void_p * 1)(ctx._h), 1, cuda.C.byref(prm), cuda.C.byref(ada),
                                                                         cuda.C.byref(null)))) == E_ARG
    # the adaptive arguments
    for rel_error, mn in ((0.0, 64), (float("nan"), 64), (float("inf"), 64), (0.05, 31), (0.05, 257)):
        assert _code(lambda: ctx.render_device_adaptive_rows(prm, rel_error, mn, film, 2, 1)) == E_ARG, (rel_error, mn)
        assert _code(lambda: cuda.render_host_multi_adaptive([ctx], prm, rel_error, mn)) == E_ARG, (rel_error, mn)
    ctx.set_geometry_precision(cuda.GEOMETRY_F64)
    try:
        assert _code(lambda: ctx.render_device_adaptive_rows(prm, 0.05, 64, film, 2, 1)) == E_UNSUPPORTED
        assert _code(lambda: cuda.render_host_multi_adaptive([ctx], prm, 0.05, 64)) == E_UNSUPPORTED
    finally:
        ctx.set_geometry_precision(cuda.GEOMETRY_F32)
    # before an upload
    fresh = cuda.Context(0)
    try:
        assert _code(lambda: fresh.render_device_adaptive_rows(prm, 0.05, 64, film, 2, 1)) == E_STATE
        assert _code(lambda: fresh.film_read_rows(film, w, h, 2, 1, hf)) == E_STATE
        assert _code(lambda: cuda._check(L.drt_cuda_render_host_multi_adaptive((cuda.C.c_void_p * 1)(fresh._h), 1, cuda.C.byref(prm),
                                                                             cuda.C.byref(ada), cuda.C.byref(hf)))) == E_STATE
        # two contexts on one device, or holding scenes with different N.  Both pairs share device 0; the messages tell the two checks
        # apart (a context's N is checked before its device)
        cfg, tables, sc2, cam2 = common.load("init_cornell", w, h, 256, 4)
        fresh.upload_scene(sc2, cam2, tables)
        assert _code(lambda: cuda.render_host_multi_adaptive([ctx, fresh], prm, 0.05, 64), "share device") == E_ARG
        lo, hi, step = next((lo, hi, step) for gn, ns, lo, hi, step in grids.RENDER_GRIDS if gn == 32)
        cfg, tables, sc3, cam3 = common.load("init_cornell", w, h, 256, 4, min_wl=lo, max_wl=hi, wl_interval=step)
        fresh.upload_scene(sc3, cam3, tables)
        assert _code(lambda: cuda.render_host_multi_adaptive([ctx, fresh], prm, 0.05, 64), "another scene") == E_ARG
    finally:
        fresh.close()


@pytest.mark.parametrize("w,h", [(16, 12), (256, 256)])
def test_host_multi_with_one_device_is_render_host_adaptive(ctx, w, h):
    """Also on a frame large enough for render_host_adaptive's six-band read-back."""
    cap, rel_error, mn = 1024, 0.05, 64
    sc, prm = _setup(ctx, "cornell_plane_light", w, h, cap, 4, 21)
    ref = ctx.render_host_adaptive(prm, rel_error, mn)
    ref_s = ctx.stats()
    assert ref_s.kernel_launches == (6 if w * h * cap >= 1 << 26 else 1)
    got = cuda.render_host_multi_adaptive([ctx], prm, rel_error, mn)
    s = ctx.stats()
    assert s.kernel_launches == 1
    for k in got:
        assert np.array_equal(got[k].view(np.uint32), ref[k].view(np.uint32)), k
    assert np.array_equal(_work(s), _work(ref_s))


def _device_contexts(count):
    return [cuda.Context(d) for d in range(count)]


def test_host_multi_on_several_devices():
    """Over 2 devices and over all of them: render_host_adaptive on device 0 bit for bit, each device reporting its own paths."""
    ndev = cuda.device_count()
    if ndev < 2:
        pytest.skip(f"needs two or more GPUs ({ndev} visible)")
    ctxs = _device_contexts(ndev)
    try:
        cases = [("init_cornell", 64, 48), ("cornell_plane_light", 64, 48), ("init_cornell", 16, max(ndev - 1, 1))]
        for scene, w, h in cases:
            cfg, tables, sc, camera = common.load(scene, w, h, 1024, 4)
            for c in ctxs:
                c.upload_scene(sc, camera, tables)
            prm = oracledriver.params(w, h, 0, 1024, 4, cfg.pixel_scheme, 17)
            ref = ctxs[0].render_host_adaptive(prm, 0.05, 64)
            ref_work = _work(ctxs[0].stats())
            for g in sorted({2, ndev}):
                got = cuda.render_host_multi_adaptive(ctxs[:g], prm, 0.05, 64)
                for k in got:
                    assert np.array_equal(got[k].view(np.uint32), ref[k].view(np.uint32)), (scene, h, g, k)
                per = [_work(c.stats()) for c in ctxs[:g]]
                assert np.array_equal(np.sum(per, axis=0, dtype=np.uint64), ref_work), (scene, h, g)
                for rank in range(g):
                    assert per[rank].any() == (rank < h), (scene, h, g, rank)
                print(f"\n{scene} {w}x{h} on {g} devices: paths per device {[int(p[0]) for p in per]}")
        # contexts that share a device, or hold scenes with different N
        twin = cuda.Context(0)
        try:
            cfg, tables, sc, camera = common.load("init_cornell", 16, 12, 256, 4)
            twin.upload_scene(sc, camera, tables)
            prm = oracledriver.params(16, 12, 0, 256, 4, cfg.pixel_scheme, 1)
            for c in ctxs:
                c.upload_scene(sc, camera, tables)
            assert _code(lambda: cuda.render_host_multi_adaptive([ctxs[0], ctxs[1], twin], prm, 0.05, 64), "share device") == E_ARG
            lo, hi, step = next((lo, hi, step) for gn, ns, lo, hi, step in grids.RENDER_GRIDS if gn == 32)
            cfg, tables, sc3, cam3 = common.load("init_cornell", 16, 12, 256, 4, min_wl=lo, max_wl=hi, wl_interval=step)
            ctxs[1].upload_scene(sc3, cam3, tables)
            assert _code(lambda: cuda.render_host_multi_adaptive(ctxs[:2], prm, 0.05, 64), "another scene") == E_ARG
        finally:
            twin.close()
    finally:
        for c in ctxs:
            c.close()
