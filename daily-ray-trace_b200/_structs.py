"""ctypes mirrors of include/drt_scene.h and include/drt_host.h (plain-old-data, no logic)."""
import ctypes as C

MAX_WL, MAX_SURF, MAX_MAT, MAX_LOBES, SPD_COUNT = 128, 16, 17, 16, 6

GEO_NONE, GEO_POINT, GEO_SPHERE, GEO_PLANE = 0, 1, 2, 3
PIXEL_NONE, PIXEL_CENTER, PIXEL_RANDOM = 0, 1, 2
LOBE_NAMES = ["bp_diffuse_bdsf", "bp_glossy_bdsf", "mirror_bdsf", "fs_conductor_bdsf",
              "fs_dielectric_reflectance_bdsf", "fs_dielectric_transmittance_bdsf", "ct_conductor_bdsf"]
DIR_NAMES = ["cos_weighted_sample_hemisphere", "uniform_sample_hemisphere", "sample_specular_direction",
             "sample_transmit_direction", "sample_reflect_or_transmit_direction", "sample_ct_direction"]
PARSE_STRICT, PARSE_LEGACY_COMPAT = 0, 1


class Surface(C.Structure):
    _fields_ = [("type", C.c_int32), ("material", C.c_int32), ("position", C.c_double * 3), ("radius", C.c_double),
                ("normal", C.c_double * 3), ("u", C.c_double * 3), ("v", C.c_double * 3), ("name", C.c_char * 32)]


class Material(C.Structure):
    _fields_ = [("name", C.c_char * 32), ("is_black_body", C.c_int32), ("is_emissive", C.c_int32),
                ("shininess", C.c_double), ("roughness", C.c_double), ("num_lobes", C.c_int32),
                ("lobes", C.c_int32 * MAX_LOBES), ("dir_func", C.c_int32), ("spd_mask", C.c_int32),
                ("spd", (C.c_double * MAX_WL) * SPD_COUNT)]


class Scene(C.Structure):
    _fields_ = [("num_wavelengths", C.c_int32), ("min_wl", C.c_double), ("max_wl", C.c_double), ("wl_interval", C.c_double),
                ("num_surfaces", C.c_int32), ("num_materials", C.c_int32), ("base_material", C.c_int32),
                ("escape_material", C.c_int32), ("surfaces", Surface * MAX_SURF), ("materials", Material * MAX_MAT)]


class Camera(C.Structure):
    _fields_ = [("forward", C.c_double * 3), ("right", C.c_double * 3), ("up", C.c_double * 3),
                ("aperture_position", C.c_double * 3), ("aperture_radius", C.c_double), ("focal_depth", C.c_double),
                ("focal_length", C.c_double), ("film_bottom_left", C.c_double * 3), ("pixel_width", C.c_double),
                ("pixel_height", C.c_double), ("lens_rotation", C.c_double * 9)]


class Tables(C.Structure):
    _fields_ = [("num_wavelengths", C.c_int32), ("min_wl", C.c_double), ("wl_interval", C.c_double),
                ("ref_white", C.c_double * MAX_WL), ("cmf_x", C.c_double * MAX_WL), ("cmf_y", C.c_double * MAX_WL),
                ("cmf_z", C.c_double * MAX_WL), ("rgb_basis", (C.c_double * MAX_WL) * 7)]


class RenderParams(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("sample_begin", C.c_uint32), ("sample_end", C.c_uint32),
                ("max_depth", C.c_uint32), ("pixel_scheme", C.c_int32), ("seed", C.c_uint64)]


class Adaptive(C.Structure):
    _fields_ = [("rel_error", C.c_float), ("min_samples", C.c_uint32)]


class Denoise(C.Structure):
    _fields_ = [("search_radius", C.c_uint32), ("patch_radius", C.c_uint32), ("strength", C.c_float)]


class Config(C.Structure):
    _paths = ["input_scene", "output_spd", "average_spd", "variance_spd", "output_bmp", "average_bmp", "variance_bmp",
              "white_spd", "cmf_x", "cmf_y", "cmf_z", "red_spd", "green_spd", "blue_spd", "cyan_spd", "magenta_spd",
              "yellow_spd"]
    _fields_ = ([("num_pixel_samples", C.c_uint32), ("max_cast_depth", C.c_uint32), ("output_width", C.c_uint32),
                 ("output_height", C.c_uint32), ("min_wl", C.c_double), ("max_wl", C.c_double), ("wl_interval", C.c_double)]
                + [(p, C.c_char * 64) for p in _paths] + [("pixel_scheme", C.c_int32)])


class SpdInput(C.Structure):
    _fields_ = [("method", C.c_int32), ("has_scale", C.c_int32), ("scale", C.c_double), ("rgb", C.c_double * 3),
                ("csv", C.c_char * 64), ("value", C.c_double)]


class MaterialInput(C.Structure):
    _fields_ = [("name", C.c_char * 32), ("is_base", C.c_int32), ("is_escape", C.c_int32), ("is_black_body", C.c_int32),
                ("is_emissive", C.c_int32), ("shininess", C.c_double), ("roughness", C.c_double),
                ("spd", SpdInput * SPD_COUNT), ("num_lobes", C.c_int32), ("lobes", C.c_int32 * MAX_LOBES),
                ("dir_func", C.c_int32), ("has_lobes_key", C.c_int32)]


class SurfaceInput(C.Structure):
    _fields_ = [("name", C.c_char * 32), ("type", C.c_int32), ("position", C.c_double * 3), ("radius", C.c_double),
                ("pointu", C.c_double * 3), ("pointv", C.c_double * 3), ("material_name", C.c_char * 32)]


class CameraInput(C.Structure):
    _fields_ = [("position", C.c_double * 3), ("target", C.c_double * 3), ("roll", C.c_double), ("fov", C.c_double),
                ("fdepth", C.c_double), ("flength", C.c_double), ("aperture", C.c_double), ("has_target", C.c_int32),
                ("has_legacy_axes", C.c_int32), ("up", C.c_double * 3), ("right", C.c_double * 3), ("forward", C.c_double * 3)]


class SceneInput(C.Structure):
    _fields_ = [("camera", CameraInput), ("num_materials", C.c_int32), ("num_surfaces", C.c_int32),
                ("materials", MaterialInput * 16), ("surfaces", SurfaceInput * 16), ("used_legacy", C.c_int32)]
