"""ctypes binding of libdrt_cuda.so: the C ABI of include/drt_cuda.h.

There is no CPU fallback anywhere in this module: if the library is not built, or no CUDA device is visible,
every entry point raises."""
import ctypes as C
import os

import numpy as np

from . import PACKAGE_DIR
from ._structs import Adaptive, Camera, RenderParams, Scene, Tables

GEOMETRY_F32, GEOMETRY_F64 = 0, 1

EXPORTS = ["drt_cuda_last_error", "drt_cuda_device_count", "drt_cuda_create", "drt_cuda_destroy", "drt_cuda_upload_scene",
           "drt_cuda_scene_upload_bytes", "drt_cuda_set_geometry_precision", "drt_cuda_film_sizes", "drt_cuda_render_device", "drt_cuda_render_host", "drt_cuda_render_host_multi",
           "drt_cuda_get_stats", "drt_cuda_analyse_scene", "drt_cuda_validate_scene", "drt_cuda_render_kernel_info", "drt_cuda_sample_paths", "drt_cuda_film_to_rgb", "drt_cuda_film_merge",
           "drt_cuda_measure_fp32_peak", "drt_cuda_film_alloc", "drt_cuda_film_free", "drt_cuda_film_ipc_export",
           "drt_cuda_film_ipc_open", "drt_cuda_film_ipc_close", "drt_cuda_film_merge_many", "drt_cuda_film_merge_slices", "drt_cuda_render_device_scatter", "drt_cuda_debug_records", "drt_cuda_buffer_alloc", "drt_cuda_buffer_free",
           "drt_cuda_buffer_ipc_export", "drt_cuda_buffer_ipc_open", "drt_cuda_buffer_ipc_close",
           "drt_cuda_film_merge_slices_local", "drt_cuda_film_read_slice", "drt_cuda_flags_signal", "drt_cuda_flags_wait", "drt_cuda_flags_timeouts",
           "drt_cuda_host_alloc", "drt_cuda_host_free", "drt_cuda_render_host_multi_images", "drt_cuda_render_device_scatter_band", "drt_cuda_plan_scene",
           "drt_cuda_render_device_adaptive", "drt_cuda_render_host_adaptive"]


class Film(C.Structure):
    _fields_ = [("sum", C.c_void_p), ("filter", C.c_void_p), ("mean", C.c_void_p), ("m2", C.c_void_p)]


class Stats(C.Structure):
    _fields_ = [("paths", C.c_uint64), ("closest_rays", C.c_uint64), ("shadow_rays", C.c_uint64),
                ("shaded_bounces", C.c_uint64), ("rng_draws", C.c_uint64), ("terminated_at_depth", C.c_uint64 * 8),
                ("reached_depth_cap", C.c_uint64), ("kernel_launches", C.c_uint64)]


class CudaError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"drt_cuda error {code}: {message}")
        self.code = code


_lib = None


def library_path():
    """libdrt_cuda.so next to this file; DRT_CUDA_LIB names another build of the same library (A/B measurements)."""
    return os.environ.get("DRT_CUDA_LIB") or os.path.join(PACKAGE_DIR, "libdrt_cuda.so")


def lib():
    global _lib
    if _lib is None:
        path = library_path()
        if not os.path.exists(path):
            raise ImportError(f"{path} is missing: the CUDA extension must be built (make -C {PACKAGE_DIR}); "
                              "this package has no CPU render path")
        L = C.CDLL(path)
        L.drt_cuda_last_error.restype = C.c_char_p
        L.drt_cuda_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        L.drt_cuda_destroy.argtypes = [C.c_void_p]
        L.drt_cuda_destroy.restype = None
        L.drt_cuda_upload_scene.argtypes = [C.c_void_p, C.POINTER(Scene), C.POINTER(Camera), C.POINTER(Tables)]
        L.drt_cuda_scene_upload_bytes.argtypes = [C.c_void_p, C.POINTER(C.c_size_t)]
        L.drt_cuda_validate_scene.argtypes = [C.POINTER(Scene)]
        L.drt_cuda_plan_scene.argtypes = [C.POINTER(Scene), C.POINTER(Camera), C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_float)]
        L.drt_cuda_analyse_scene.argtypes = [C.POINTER(Scene), C.POINTER(Camera), C.c_uint32, C.c_uint32, C.POINTER(C.c_uint32 * 4), C.POINTER(C.c_int32)]
        L.drt_cuda_render_kernel_info.argtypes = [C.c_void_p, C.POINTER(RenderParams), C.c_char_p, C.c_size_t, C.POINTER(C.c_int), C.POINTER(C.c_int)]
        L.drt_cuda_set_geometry_precision.argtypes = [C.c_void_p, C.c_int]
        L.drt_cuda_film_sizes.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]
        L.drt_cuda_render_device.argtypes = [C.c_void_p, C.POINTER(RenderParams), C.POINTER(Film), C.c_int, C.c_void_p]
        L.drt_cuda_render_host_multi.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.POINTER(RenderParams), C.POINTER(Film)]
        L.drt_cuda_render_device_scatter.argtypes = [C.c_void_p, C.POINTER(RenderParams), C.POINTER(Film), C.c_int, C.c_int, C.c_uint64, C.c_void_p]
        L.drt_cuda_film_merge_slices.argtypes = [C.c_void_p, C.POINTER(Film), C.POINTER(Film), C.c_int, C.c_uint64, C.c_uint32, C.c_uint32,
                                                 C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.drt_cuda_render_host.argtypes = [C.c_void_p, C.POINTER(RenderParams), C.POINTER(Film)]
        L.drt_cuda_render_device_adaptive.argtypes = [C.c_void_p, C.POINTER(RenderParams), C.POINTER(Adaptive), C.POINTER(Film), C.c_int, C.c_void_p]
        L.drt_cuda_render_host_adaptive.argtypes = [C.c_void_p, C.POINTER(RenderParams), C.POINTER(Adaptive), C.POINTER(Film)]
        L.drt_cuda_film_merge_slices_local.argtypes = [C.c_void_p, C.POINTER(Film), C.POINTER(Film), C.c_int, C.c_uint64, C.c_uint32, C.c_uint32,
                                                       C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.drt_cuda_film_read_slice.argtypes = [C.c_void_p, C.POINTER(Film), C.c_uint64, C.c_uint64, C.c_uint64, C.POINTER(Film), C.c_void_p]
        L.drt_cuda_render_device_scatter_band.argtypes = [C.c_void_p, C.POINTER(RenderParams), C.POINTER(Film), C.c_int, C.c_int, C.c_uint64, C.c_uint64, C.c_uint64, C.c_int, C.c_void_p]
        L.drt_cuda_flags_signal.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.c_int, C.c_uint32, C.c_void_p]
        L.drt_cuda_flags_wait.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_uint32, C.c_void_p]
        L.drt_cuda_flags_timeouts.argtypes = [C.c_void_p, C.POINTER(C.c_uint32)]
        L.drt_cuda_host_alloc.argtypes = [C.c_size_t, C.POINTER(C.c_void_p)]
        L.drt_cuda_host_free.argtypes = [C.c_void_p]
        L.drt_cuda_get_stats.argtypes = [C.c_void_p, C.POINTER(Stats)]
        L.drt_cuda_sample_paths.argtypes = [C.c_void_p, C.POINTER(RenderParams)] + [C.c_uint32] * 4 + [C.c_void_p]
        L.drt_cuda_film_to_rgb.argtypes = [C.c_void_p, C.POINTER(Film), C.c_uint32, C.c_uint32, C.c_int, C.c_void_p,
                                           C.c_void_p, C.c_void_p]
        L.drt_cuda_film_merge.argtypes = [C.c_void_p, C.POINTER(Film), C.POINTER(Film), C.c_uint32, C.c_uint32, C.c_void_p]
        L.drt_cuda_debug_records.argtypes = [C.c_void_p, C.POINTER(RenderParams)] + [C.c_uint32] * 4 + [C.c_void_p, C.c_size_t, C.POINTER(C.c_uint32)]
        L.drt_cuda_buffer_alloc.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]
        L.drt_cuda_buffer_free.argtypes = [C.c_void_p, C.c_void_p]
        L.drt_cuda_buffer_ipc_export.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.drt_cuda_buffer_ipc_open.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]
        L.drt_cuda_buffer_ipc_close.argtypes = [C.c_void_p, C.c_void_p]
        L.drt_cuda_film_alloc.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.POINTER(Film)]
        L.drt_cuda_film_free.argtypes = [C.c_void_p, C.POINTER(Film)]
        L.drt_cuda_film_ipc_export.argtypes = [C.c_void_p, C.POINTER(Film), C.c_void_p]
        L.drt_cuda_film_ipc_open.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(Film)]
        L.drt_cuda_film_ipc_close.argtypes = [C.c_void_p, C.POINTER(Film)]
        L.drt_cuda_film_merge_many.argtypes = [C.c_void_p, C.POINTER(Film), C.POINTER(Film), C.c_int, C.c_uint32, C.c_uint32,
                                               C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.drt_cuda_measure_fp32_peak.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_double)]
        _lib = L
    return _lib


def _check(rc):
    if rc != 0:
        raise CudaError(rc, lib().drt_cuda_last_error().decode(errors="replace"))


def device_count():
    return lib().drt_cuda_device_count()


class Context:
    """One CUDA device with one uploaded scene (drt_cuda_context)."""

    def __init__(self, device=0):
        self._h = C.c_void_p()
        _check(lib().drt_cuda_create(device, C.byref(self._h)))
        self.device = device
        self.n = None

    def close(self):
        if self._h:
            lib().drt_cuda_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def upload_scene(self, scene, camera, tables):
        _check(lib().drt_cuda_upload_scene(self._h, C.byref(scene), C.byref(camera), C.byref(tables)))
        self.n = scene.num_wavelengths

    def scene_upload_bytes(self):
        v = C.c_size_t()
        _check(lib().drt_cuda_scene_upload_bytes(self._h, C.byref(v)))
        return v.value

    def render_kernel_info(self, params):
        """(kernel name, warps per CTA, CTAs per SM) the uploaded scene, the geometry precision and `params` select."""
        name = C.create_string_buffer(96)
        warps, ctas = C.c_int(), C.c_int()
        _check(lib().drt_cuda_render_kernel_info(self._h, C.byref(params), name, len(name), C.byref(warps), C.byref(ctas)))
        return name.value.decode(), warps.value, ctas.value

    def set_geometry_precision(self, precision):
        _check(lib().drt_cuda_set_geometry_precision(self._h, precision))

    def render_host(self, params):
        """End-to-end call with host buffers: returns dict of numpy f32 arrays sum[H*W,N], filter[H*W], mean, m2."""
        npix = max(params.width * params.height, 1)
        n = self.n or 1     # before upload_scene the library reports DRT_CUDA_E_STATE; buffers only need to exist
        out = {"sum": np.empty((npix, n), np.float32), "filter": np.empty(npix, np.float32),
               "mean": np.empty((npix, n), np.float32), "m2": np.empty((npix, n), np.float32)}
        film = Film(out["sum"].ctypes.data, out["filter"].ctypes.data, out["mean"].ctypes.data, out["m2"].ctypes.data)
        _check(lib().drt_cuda_render_host(self._h, C.byref(params), C.byref(film)))
        return out

    def render_host_adaptive(self, params, rel_error, min_samples):
        """render_host with adaptive sampling (drt_cuda_render_host_adaptive): every pixel stops once the error bound of its luminance
        is <= rel_error times the luminance and it has >= min_samples samples; filter holds each pixel's count."""
        npix = max(params.width * params.height, 1)
        n = self.n or 1
        out = {"sum": np.empty((npix, n), np.float32), "filter": np.empty(npix, np.float32),
               "mean": np.empty((npix, n), np.float32), "m2": np.empty((npix, n), np.float32)}
        film = Film(out["sum"].ctypes.data, out["filter"].ctypes.data, out["mean"].ctypes.data, out["m2"].ctypes.data)
        _check(lib().drt_cuda_render_host_adaptive(self._h, C.byref(params), C.byref(Adaptive(rel_error, min_samples)), C.byref(film)))
        return out

    def render_device_adaptive(self, params, rel_error, min_samples, film, accumulate=False, stream=None):
        _check(lib().drt_cuda_render_device_adaptive(self._h, C.byref(params), C.byref(Adaptive(rel_error, min_samples)), C.byref(film),
                                                     int(accumulate), stream))

    def render_host_into(self, params, film):
        _check(lib().drt_cuda_render_host(self._h, C.byref(params), C.byref(film)))

    def render_device(self, params, film, accumulate=False, stream=None):
        _check(lib().drt_cuda_render_device(self._h, C.byref(params), C.byref(film), int(accumulate), stream))

    def sample_paths(self, params, x0, y0, x1, y1):
        """The sample_scene seam: f32 array [(y1-y0)*(x1-x0), spp, N] of per-path spectral radiance."""
        spp = params.sample_end - params.sample_begin
        out = np.empty(((y1 - y0) * (x1 - x0), spp, self.n), np.float32)
        _check(lib().drt_cuda_sample_paths(self._h, C.byref(params), x0, y0, x1, y1, out.ctypes.data))
        return out

    def debug_records(self, params, x0, y0, x1, y1):
        """Raw path records [(pixels), spp, words] as uint32 (reinterpret floats with .view(np.float32))."""
        words = C.c_uint32()
        _check(lib().drt_cuda_debug_records(self._h, C.byref(params), x0, y0, x1, y1, None, 0, C.byref(words)))
        spp = params.sample_end - params.sample_begin
        out = np.empty(((y1 - y0) * (x1 - x0), spp, words.value), np.uint32)
        _check(lib().drt_cuda_debug_records(self._h, C.byref(params), x0, y0, x1, y1, out.ctypes.data, out.size, C.byref(words)))
        return out

    def stats(self):
        s = Stats()
        _check(lib().drt_cuda_get_stats(self._h, C.byref(s)))
        return s

    def film_to_rgb(self, film, width, height, which, rgb_ptr=None, bgra_ptr=None, stream=None):
        _check(lib().drt_cuda_film_to_rgb(self._h, C.byref(film), width, height, which, rgb_ptr, bgra_ptr, stream))

    def film_merge(self, dst, src, width, height, stream=None):
        _check(lib().drt_cuda_film_merge(self._h, C.byref(dst), C.byref(src), width, height, stream))

    def buffer_alloc(self, nbytes):
        p = C.c_void_p()
        _check(lib().drt_cuda_buffer_alloc(self._h, nbytes, C.byref(p)))
        return p.value

    def buffer_free(self, ptr):
        _check(lib().drt_cuda_buffer_free(self._h, ptr))

    def buffer_ipc_export(self, ptr):
        buf = C.create_string_buffer(64)
        _check(lib().drt_cuda_buffer_ipc_export(self._h, ptr, buf))
        return buf.raw

    def buffer_ipc_open(self, handle):
        p = C.c_void_p()
        _check(lib().drt_cuda_buffer_ipc_open(self._h, C.create_string_buffer(handle, 64), C.byref(p)))
        return p.value

    def buffer_ipc_close(self, ptr):
        _check(lib().drt_cuda_buffer_ipc_close(self._h, ptr))

    def film_alloc(self, width, height):
        f = Film()
        _check(lib().drt_cuda_film_alloc(self._h, width, height, C.byref(f)))
        return f

    def film_free(self, film):
        _check(lib().drt_cuda_film_free(self._h, C.byref(film)))

    def film_ipc_export(self, film):
        buf = C.create_string_buffer(256)
        _check(lib().drt_cuda_film_ipc_export(self._h, C.byref(film), buf))
        return buf.raw

    def film_ipc_open(self, handles):
        f = Film()
        _check(lib().drt_cuda_film_ipc_open(self._h, C.create_string_buffer(handles, 256), C.byref(f)))
        return f

    def film_ipc_close(self, film):
        _check(lib().drt_cuda_film_ipc_close(self._h, C.byref(film)))

    def film_merge_many(self, dst, srcs, width, height, pixel_begin, pixel_end, bgra=None, stream=None):
        arr = (Film * len(srcs))(*srcs)
        b = bgra or (None, None, None)
        _check(lib().drt_cuda_film_merge_many(self._h, C.byref(dst), arr, len(srcs), width, height, pixel_begin, pixel_end,
                                              b[0], b[1], b[2], stream))

    def render_device_scatter(self, params, staging, rank, slice_pixels, stream=None):
        arr = (Film * len(staging))(*staging)
        _check(lib().drt_cuda_render_device_scatter(self._h, C.byref(params), arr, len(staging), rank, slice_pixels, stream))

    def film_merge_slices(self, dst, staging, count, slice_pixels, width, height, pixel_begin, pixel_end, bgra=None, stream=None):
        b = bgra or (None, None, None)
        _check(lib().drt_cuda_film_merge_slices(self._h, C.byref(dst), C.byref(staging), count, slice_pixels, width, height,
                                                pixel_begin, pixel_end, b[0], b[1], b[2], stream))

    def film_merge_slices_local(self, slice_film, staging, count, slice_pixels, width, height, pixel_begin, pixel_end, bgra=None, stream=None):
        b = bgra or (None, None, None)
        _check(lib().drt_cuda_film_merge_slices_local(self._h, C.byref(slice_film), C.byref(staging), count, slice_pixels, width, height,
                                                      pixel_begin, pixel_end, b[0], b[1], b[2], stream))

    def film_read_slice(self, slice_film, slice_begin, pixel_begin, pixel_end, host_film, stream=None):
        _check(lib().drt_cuda_film_read_slice(self._h, C.byref(slice_film), slice_begin, pixel_begin, pixel_end, C.byref(host_film), stream))

    def render_device_scatter_band(self, params, staging, rank, slice_pixels, band_begin, band_end, keep_stats=False, stream=None):
        arr = (Film * len(staging))(*staging)
        _check(lib().drt_cuda_render_device_scatter_band(self._h, C.byref(params), arr, len(staging), rank, slice_pixels, band_begin, band_end,
                                                         int(keep_stats), stream))

    def flags_signal(self, targets, value, stream=None):
        arr = (C.c_void_p * len(targets))(*targets)
        _check(lib().drt_cuda_flags_signal(self._h, arr, len(targets), value & 0xffffffff, stream))

    def flags_wait(self, flags_ptr, count, value, stream=None):
        _check(lib().drt_cuda_flags_wait(self._h, flags_ptr, count, value & 0xffffffff, stream))

    def flags_timeouts(self):
        v = C.c_uint32()
        _check(lib().drt_cuda_flags_timeouts(self._h, C.byref(v)))
        return v.value

    def measure_fp32_peak(self, packed=False):
        v = C.c_double()
        _check(lib().drt_cuda_measure_fp32_peak(self._h, int(packed), C.byref(v)))
        return v.value


def render_host_multi(contexts, params):
    """render_host over several Context objects on distinct devices of this process: dict of numpy f32 arrays like Context.render_host."""
    npix, n = params.width * params.height, contexts[0].n
    out = {"sum": np.empty((npix, n), np.float32), "filter": np.empty(npix, np.float32),
           "mean": np.empty((npix, n), np.float32), "m2": np.empty((npix, n), np.float32)}
    film = Film(out["sum"].ctypes.data, out["filter"].ctypes.data, out["mean"].ctypes.data, out["m2"].ctypes.data)
    handles = (C.c_void_p * len(contexts))(*[c._h for c in contexts])
    _check(lib().drt_cuda_render_host_multi(handles, len(contexts), C.byref(params), C.byref(film)))
    return out


def validate_scene(scene):
    """Raises CudaError for a scene drt_cuda_upload_scene would reject (host arithmetic, no device needed)."""
    _check(lib().drt_cuda_validate_scene(C.byref(scene)))


def plan_scene(scene, camera):
    """(kernel mode, class per material, specular constants [materials][3][2]) of drt_cuda_plan_scene: host arithmetic, no device needed."""
    mode = C.c_int32()
    classes = (C.c_int32 * scene.num_materials)()
    consts = (C.c_float * (scene.num_materials * 6))()
    _check(lib().drt_cuda_plan_scene(C.byref(scene), C.byref(camera), C.byref(mode), classes, consts))
    return mode.value, list(classes), np.array(consts, dtype=np.float32).reshape(scene.num_materials, 3, 2)


def analyse_scene(scene, camera, width, height):
    """(hit rectangle (x0, y0, x1, y1), boundary flag per surface) of drt_cuda_analyse_scene: host arithmetic, no device needed."""
    rect = (C.c_uint32 * 4)()
    flags = (C.c_int32 * max(scene.num_surfaces, 1))()
    _check(lib().drt_cuda_analyse_scene(C.byref(scene), C.byref(camera), width, height, C.byref(rect), flags))
    return tuple(rect), [bool(flags[i]) for i in range(scene.num_surfaces)]


def film_from_tensors(total, filt, mean, m2):
    """drt_film over caller-owned torch CUDA tensors (f32, contiguous): PyTorch is only the allocator here."""
    for t in (total, filt, mean, m2):
        assert t.is_cuda and t.is_contiguous() and t.dtype.is_floating_point and t.element_size() == 4
    return Film(total.data_ptr(), filt.data_ptr(), mean.data_ptr(), m2.data_ptr())
