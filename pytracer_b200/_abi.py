"""ctypes mirror of include/rt_api.h (struct layouts and enum values)."""
from __future__ import annotations

import ctypes as C

RT_API_VERSION = 1

RT_SHAPE_SPHERE, RT_SHAPE_PLANE = 0, 1
RT_BRDF_DIFFUSE, RT_BRDF_SPECULAR = 0, 1
RT_PIGMENT_UNIFORM, RT_PIGMENT_CHECKERED, RT_PIGMENT_IMAGE = 0, 1, 2
RT_CAMERA_ORTHOGONAL, RT_CAMERA_PERSPECTIVE = 0, 1
RT_ALGO_ONOFF, RT_ALGO_FLAT, RT_ALGO_PATHTRACING, RT_ALGO_POINTLIGHT = 0, 1, 2, 3
ALGORITHMS = {"onoff": 0, "flat": 1, "pathtracing": 2, "pointlight": 3}
RT_PRECISION_AUTO, RT_PRECISION_F32, RT_PRECISION_F64, RT_PRECISION_HYBRID = 0, 1, 2, 3
PRECISIONS = {"auto": 0, "f32": 1, "f64": 2, "hybrid": 3}
RT_VARIANT_AUTO, RT_VARIANT_MEGA, RT_VARIANT_WARP = 0, 1, 2
VARIANTS = {"auto": 0, "mega": 1, "warp": 2}
RT_RNG_STREAMS, RT_RNG_REPLAY = 0, 1
RT_PART_NONE, RT_PART_SPP, RT_PART_ROWS = 0, 1, 2
RT_HIT_SHAPE, RT_HIT_RAY_COUNT = 0, 1
PARTITIONS = {"none": 0, "spp": 1, "rows": 2}
RT_ROWS_FULL, RT_ROWS_COMPACT = 0, 1
RT_MAX_PEERS = 8
ACCELS = {"none": 0, "bvh": 1}  # RT_ACCEL_*

RT_OK, RT_ERR_INVALID, RT_ERR_CUDA, RT_ERR_NO_DEVICE, RT_ERR_OVERFLOW = 0, -1, -2, -3, -4
RT_ERR_EST_BATCH, RT_ERR_EST_PAIRED = 0, 1
ERROR_ESTIMATORS = {"batch": 0, "paired": 1}

c_double3 = C.c_double * 3


class rt_pigment(C.Structure):
    _fields_ = [
        ("kind", C.c_int32),
        ("num_of_steps", C.c_int32),
        ("tex_width", C.c_int32),
        ("tex_height", C.c_int32),
        ("tex_offset", C.c_int64),
        ("color1", c_double3),
        ("color2", c_double3),
    ]


class rt_material(C.Structure):
    _fields_ = [
        ("brdf_kind", C.c_int32),
        ("brdf_pigment", C.c_int32),
        ("emitted_pigment", C.c_int32),
        ("_pad", C.c_int32),
        ("threshold_angle_rad", C.c_double),
    ]


class rt_light(C.Structure):
    _fields_ = [("position", c_double3), ("color", c_double3), ("linear_radius", C.c_double)]


class rt_scene_desc(C.Structure):
    _fields_ = [
        ("n_shapes", C.c_int32),
        ("n_materials", C.c_int32),
        ("n_pigments", C.c_int32),
        ("n_lights", C.c_int32),
        ("shape_kind", C.c_void_p),
        ("shape_material", C.c_void_p),
        ("shape_m", C.c_void_p),
        ("shape_invm", C.c_void_p),
        ("materials", C.c_void_p),
        ("pigments", C.c_void_p),
        ("lights", C.c_void_p),
        ("n_texels", C.c_int64),
        ("texels", C.c_void_p),
    ]


class rt_camera(C.Structure):
    _fields_ = [
        ("kind", C.c_int32),
        ("_pad", C.c_int32),
        ("screen_distance", C.c_double),
        ("aspect_ratio", C.c_double),
        ("m", C.c_double * 12),
    ]


class rt_render_params(C.Structure):
    _fields_ = [
        ("width", C.c_int32),
        ("height", C.c_int32),
        ("samples_per_side", C.c_int32),
        ("algorithm", C.c_int32),
        ("camera", rt_camera),
        ("background", c_double3),
        ("onoff_color", c_double3),
        ("ambient", c_double3),
        ("num_of_rays", C.c_int32),
        ("max_depth", C.c_int32),
        ("rr_limit", C.c_int32),
        ("rng_mode", C.c_int32),
        ("aa_state", C.c_uint64),
        ("aa_inc", C.c_uint64),
        ("pt_state", C.c_uint64),
        ("pt_inc", C.c_uint64),
        ("replay_states", C.c_void_p),
        ("part_mode", C.c_int32),
        ("part_rank", C.c_int32),
        ("part_count", C.c_int32),
        ("variant", C.c_int32),
        ("precision", C.c_int32),
        ("out_f64", C.c_int32),
        ("hit_mode", C.c_int32),
        ("accel", C.c_int32),
        ("rows_layout", C.c_int32),
        ("n_peer_images", C.c_int32),
        ("peer_images", C.c_void_p * 8),
    ]


class rt_stats(C.Structure):
    _fields_ = [
        ("rays_closest", C.c_uint64),
        ("rays_shadow", C.c_uint64),
        ("samples", C.c_uint64),
        ("kernel_ms", C.c_float),
        ("total_ms", C.c_float),
        ("variant_used", C.c_int32),
        ("precision_used", C.c_int32),
        ("n_launches", C.c_int32),
        ("overflow", C.c_int32),
    ]

    def as_dict(self) -> dict:
        return {name: getattr(self, name) for name, _ in self._fields_}


class rt_tonemap_stats(C.Structure):
    _fields_ = [
        ("luminosity", C.c_double),
        ("lum_ms", C.c_float),
        ("map_ms", C.c_float),
        ("total_ms", C.c_float),
        ("n_launches", C.c_int32),
    ]

    def as_dict(self) -> dict:
        return {name: getattr(self, name) for name, _ in self._fields_}


class rt_adaptive_params(C.Structure):
    _fields_ = [
        ("target_error", C.c_double),
        ("error_floor", C.c_double),
        ("max_passes", C.c_int32),
        ("estimator", C.c_int32),
    ]


class rt_adaptive_stats(C.Structure):
    _fields_ = [
        ("rays_closest", C.c_uint64),
        ("rays_shadow", C.c_uint64),
        ("samples", C.c_uint64),
        ("kernel_ms", C.c_float),
        ("total_ms", C.c_float),
        ("passes", C.c_int32),
        ("n_launches", C.c_int32),
        ("pixels_in_pass", C.c_int64 * 16),
        ("overflow", C.c_int32),
        ("_pad", C.c_int32),
    ]

    def as_dict(self) -> dict:
        d = {name: getattr(self, name) for name, _ in self._fields_ if name != "_pad"}
        d["pixels_in_pass"] = [int(v) for v in self.pixels_in_pass[: min(self.passes, 16)]]
        return d


class rt_hit(C.Structure):
    _fields_ = [
        ("shape", C.c_int32),
        ("material", C.c_int32),
        ("t", C.c_double),
        ("world_point", c_double3),
        ("normal", c_double3),
        ("uv", C.c_double * 2),
    ]
