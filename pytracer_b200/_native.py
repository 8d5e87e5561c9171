"""Loads libpytracer_b200.so (the C-ABI of include/rt_api.h) through ctypes.

There is no CPU fallback: if the library is missing, cannot be loaded, or finds no CUDA device,
the call raises — it never degrades to a Python implementation.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import threading
from pathlib import Path

from . import _abi

_PKG = Path(__file__).resolve().parent
# PYTRACER_B200_LIB: another build of the same library (kernel tuning experiments)
LIB_PATH = Path(os.environ.get("PYTRACER_B200_LIB") or _PKG / "libpytracer_b200.so")
_lock = threading.Lock()
_lib = None

_P = C.c_void_p
_PROTOTYPES = {
    "rt_api_version": (C.c_int, []),
    "rt_device_count": (C.c_int, []),
    "rt_set_device": (C.c_int, [C.c_int]),
    "rt_last_error": (C.c_char_p, []),
    "rt_scene_create": (C.c_int, [C.POINTER(_abi.rt_scene_desc), C.POINTER(_P)]),
    "rt_scene_destroy": (None, [_P]),
    "rt_bvh_build_host": (C.c_int, [_P, C.c_int32, _P, C.c_int32, _P, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "rt_scene_update_transforms": (C.c_int, [_P, C.c_int32, C.c_int32, _P, _P, _P]),
    "rt_render": (C.c_int, [_P, C.POINTER(_abi.rt_render_params), _P, _P, C.POINTER(_abi.rt_stats)]),
    "rt_render_multi": (C.c_int, [C.POINTER(_P), C.c_int32, C.POINTER(_abi.rt_render_params), _P, _P, C.POINTER(_abi.rt_stats)]),
    "rt_render_device": (C.c_int, [_P, C.POINTER(_abi.rt_render_params), _P, _P, _P]),
    "rt_render_finish": (C.c_int, [_P, _P, C.POINTER(_abi.rt_stats)]),
    "rt_render_adaptive": (C.c_int, [_P, C.POINTER(_abi.rt_render_params), C.POINTER(_abi.rt_adaptive_params), _P, _P, _P,
                                     C.POINTER(_abi.rt_adaptive_stats)]),
    "rt_trace_rays": (C.c_int, [_P, C.POINTER(_abi.rt_render_params), _P, _P, C.c_int32, _P, _P]),
    "rt_intersect": (C.c_int, [_P, C.c_int32, C.c_int32, _P, C.c_int32, _P]),
    "rt_is_point_visible": (C.c_int, [_P, C.c_int32, _P, C.c_int32, _P]),
    "rt_camera_rays": (C.c_int, [C.POINTER(_abi.rt_render_params), C.c_int32, _P]),
    "rt_camera_fire": (C.c_int, [C.POINTER(_abi.rt_camera), C.c_int32, _P, C.c_int32, _P]),
    "rt_pcg_draw": (C.c_int, [_P, C.c_int32, _P]),
    "rt_pcg_seed": (C.c_int, [C.c_uint64, C.c_uint64, _P]),
    "rt_pigment_color": (C.c_int, [_P, C.c_int32, C.c_int32, _P, C.c_int32, _P]),
    "rt_scatter": (C.c_int, [_P, C.c_int32, C.c_int32, _P, C.c_int32, _P, _P]),
    "rt_onb": (C.c_int, [C.c_int32, _P, C.c_int32, _P]),
    "rt_average_luminosity": (C.c_int, [_P, C.c_int64, C.c_double, C.c_int32, _P, C.POINTER(C.c_double)]),
    "rt_tone_map": (C.c_int, [_P, C.c_int64, C.c_int32, C.c_double, C.c_double, C.c_double, C.c_int32, _P, _P, _P,
                              C.POINTER(_abi.rt_tonemap_stats)]),
    "rt_host_register": (C.c_int, [_P, C.c_uint64]),
    "rt_host_unregister": (C.c_int, [_P]),
    "rt_bench_ffma": (C.c_int, [C.c_int32, C.POINTER(C.c_double), C.POINTER(C.c_float)]),
    "rt_bench_dfma": (C.c_int, [C.c_int32, C.POINTER(C.c_double), C.POINTER(C.c_float)]),
}
EXPORTED_SYMBOLS = tuple(_PROTOTYPES)


class NativeError(RuntimeError):
    """An rt_* call returned a negative status; carries the library's error text."""

    def __init__(self, code: int, message: str):
        super().__init__(f"libpytracer_b200: {message} (status {code})")
        self.code = code


def build(verbose: bool = False) -> Path:
    """Compile the library in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    proc = subprocess.run(["bash", str(_PKG / "csrc" / "build.sh")], capture_output=True, text=True)
    if verbose or proc.returncode != 0:
        print(proc.stdout, proc.stderr)
    if proc.returncode != 0:
        raise RuntimeError("building libpytracer_b200.so failed:\n" + proc.stderr[-4000:])
    return LIB_PATH


def load() -> C.CDLL:
    """dlopen the library and attach prototypes.  Does not need a GPU (symbol checks run on CPU)."""
    global _lib
    with _lock:
        if _lib is None:
            if not LIB_PATH.exists():
                raise RuntimeError(
                    f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                    "or pytracer_b200/csrc/build.sh. There is no CPU fallback."
                )
            lib = C.CDLL(str(LIB_PATH))
            for name, (restype, argtypes) in _PROTOTYPES.items():
                fn = getattr(lib, name)
                fn.restype, fn.argtypes = restype, argtypes
            if lib.rt_api_version() != _abi.RT_API_VERSION:
                raise RuntimeError("libpytracer_b200.so does not match include/rt_api.h (rebuild it)")
            _lib = lib
    return _lib


def check(status: int) -> None:
    if status != 0:
        raise NativeError(status, load().rt_last_error().decode("utf-8", "replace"))


def require_device() -> C.CDLL:
    lib = load()
    if lib.rt_device_count() <= 0:
        raise NativeError(_abi.RT_ERR_NO_DEVICE, "no CUDA device is visible; this library has no CPU path")
    return lib
