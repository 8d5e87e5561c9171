"""DeviceScene: a flattened World resident in HBM + typed wrappers over the rt_* entry points."""
from __future__ import annotations

import ctypes as C
from typing import Optional, Tuple

import numpy as np

from . import _abi, _native
from .flatten import FlatScene, flatten_world


def _ptr(arr: Optional[np.ndarray]):
    return None if arr is None else C.c_void_p(arr.ctypes.data)


class DeviceScene:
    """Owns one ``rt_scene`` (device copies of the shape transforms in fp32 and fp64, material /
    pigment / light tables, textures).  Build it from a World (ours or the reference's) or from a
    :class:`FlatScene`."""

    def __init__(self, world_or_flat, device: Optional[int] = None):
        """``device``: the CUDA device the scene lives on (None = the current one)."""
        self._lib = _native.require_device()
        self.flat: FlatScene = world_or_flat if isinstance(world_or_flat, FlatScene) else flatten_world(world_or_flat)
        handle = C.c_void_p()
        if device is not None:
            _native.check(self._lib.rt_set_device(int(device)))
        _native.check(self._lib.rt_scene_create(C.byref(self.flat.desc), C.byref(handle)))
        self._handle = handle

    def close(self) -> None:
        if getattr(self, "_handle", None):
            self._lib.rt_scene_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def update_transforms(self, first: int, m: np.ndarray, invm: np.ndarray, stream: int = 0) -> None:
        """New Transformation.m / .invm rows 0..2 ((n, 12) fp64 each) for shapes [first, first + n) of
        World.shapes; the rest of the scene stays resident (animation frames)."""
        m = np.ascontiguousarray(m, dtype=np.float64).reshape(-1, 12)
        invm = np.ascontiguousarray(invm, dtype=np.float64).reshape(-1, 12)
        assert m.shape == invm.shape
        _native.check(self._lib.rt_scene_update_transforms(self._handle, int(first), m.shape[0], _ptr(m), _ptr(invm),
                                                           C.c_void_p(stream) if stream else None))
        self.flat.shape_m.reshape(-1, 12)[first:first + m.shape[0]] = m
        self.flat.shape_invm.reshape(-1, 12)[first:first + m.shape[0]] = invm

    def update_from_world(self, world, stream: int = 0) -> None:
        """Same shapes, materials and lights as the resident scene, new transformations (e.g. the next
        frame of an animation parsed with another `clock`)."""
        new = world if isinstance(world, FlatScene) else flatten_world(world)
        if not self.flat.differs_only_in_transforms(new):
            raise ValueError("update_from_world: more than the transformations changed; build a new DeviceScene")
        self.update_transforms(0, new.shape_m, new.shape_invm, stream)

    # ------------------------------------------------------------------ the hot path
    def render(self, params: _abi.rt_render_params, want_hit: bool = False, out: Optional[np.ndarray] = None,
               replay_states: Optional[np.ndarray] = None) -> Tuple[np.ndarray, Optional[np.ndarray], dict]:
        """rt_render: host buffers in, host image out (float32, or float64 if params.out_f64)."""
        H, W = params.height, params.width
        dtype = np.float64 if params.out_f64 else np.float32
        if out is None:
            out = np.empty((H, W, 3), dtype=dtype)
        assert out.dtype == dtype and out.shape == (H, W, 3) and out.flags.c_contiguous
        hit = np.empty((H, W), dtype=np.int32) if want_hit else None
        if replay_states is not None:
            replay_states = np.ascontiguousarray(replay_states, dtype=np.uint64)
            params.replay_states = replay_states.ctypes.data
        stats = _abi.rt_stats()
        try:
            _native.check(self._lib.rt_render(self._handle, C.byref(params), _ptr(out), _ptr(hit), C.byref(stats)))
        finally:
            params.replay_states = None
        return out, hit, stats.as_dict()

    def render_adaptive(self, params: _abi.rt_render_params, target_error: float = 0.0, max_passes: int = 1,
                        error_floor: float = 1e-2, out: Optional[np.ndarray] = None, estimator: str = "batch"):
        """rt_render_adaptive: (mean image, SE image, samples per pixel, stats) as float32 [H][W][3] x 2 and
        int32 [H][W]; ``max_passes`` passes of ``params.samples_per_side ** 2`` samples at most per pixel.
        ``estimator``: "batch" or "paired" (collapsed strata, even samples_per_side), or an RT_ERR_EST_* int."""
        H, W = params.height, params.width
        if out is None:
            out = np.empty((H, W, 3), dtype=np.float32)
        assert out.dtype == np.float32 and out.shape == (H, W, 3) and out.flags.c_contiguous
        err = np.empty((H, W, 3), dtype=np.float32)
        samples = np.empty((H, W), dtype=np.int32)
        ap = _abi.rt_adaptive_params()
        ap.target_error, ap.error_floor, ap.max_passes = float(target_error), float(error_floor), int(max_passes)
        ap.estimator = _abi.ERROR_ESTIMATORS[estimator] if isinstance(estimator, str) else int(estimator)
        stats = _abi.rt_adaptive_stats()
        _native.check(self._lib.rt_render_adaptive(self._handle, C.byref(params), C.byref(ap), _ptr(out), _ptr(err), _ptr(samples),
                                                   C.byref(stats)))
        return out, err, samples, stats.as_dict()

    def render_device(self, params: _abi.rt_render_params, out_ptr: int, hit_ptr: int = 0, stream: int = 0) -> None:
        """rt_render_device: enqueue on ``stream`` writing to device memory at ``out_ptr``."""
        _native.check(self._lib.rt_render_device(self._handle, C.byref(params), C.c_void_p(out_ptr),
                                                 C.c_void_p(hit_ptr) if hit_ptr else None,
                                                 C.c_void_p(stream) if stream else None))

    def finish(self, stream: int = 0) -> dict:
        stats = _abi.rt_stats()
        _native.check(self._lib.rt_render_finish(self._handle, C.c_void_p(stream) if stream else None, C.byref(stats)))
        return stats.as_dict()

    # ------------------------------------------------------------------ explicit rays and probes
    def trace_rays(self, params: _abi.rt_render_params, rays: np.ndarray, depth: Optional[np.ndarray] = None,
                   pcg_state_inc: Optional[Tuple[int, int]] = None):
        rays = np.ascontiguousarray(rays, dtype=np.float64).reshape(-1, 8)
        n = rays.shape[0]
        depth_arr = None if depth is None else np.ascontiguousarray(depth, dtype=np.int32)
        st = np.array(pcg_state_inc if pcg_state_inc is not None else (params.pt_state, params.pt_inc), dtype=np.uint64)
        out = np.zeros((n, 3), dtype=np.float64)
        _native.check(self._lib.rt_trace_rays(self._handle, C.byref(params), _ptr(rays), _ptr(depth_arr), n, _ptr(st), _ptr(out)))
        return out, (int(st[0]), int(st[1]))

    def intersect(self, rays: np.ndarray, precision: str = "f64", normalize: bool = True):
        rays = np.ascontiguousarray(rays, dtype=np.float64).reshape(-1, 8)
        out = (_abi.rt_hit * rays.shape[0])()
        _native.check(self._lib.rt_intersect(self._handle, _abi.PRECISIONS[precision], int(normalize), _ptr(rays), rays.shape[0], out))
        return out

    def is_point_visible(self, pairs: np.ndarray, precision: str = "f64") -> np.ndarray:
        pairs = np.ascontiguousarray(pairs, dtype=np.float64).reshape(-1, 6)
        out = np.zeros(pairs.shape[0], dtype=np.uint8)
        _native.check(self._lib.rt_is_point_visible(self._handle, _abi.PRECISIONS[precision], _ptr(pairs), pairs.shape[0], _ptr(out)))
        return out.astype(bool)

    def pigment_color(self, pigment: int, uv: np.ndarray, precision: str = "f64") -> np.ndarray:
        uv = np.ascontiguousarray(uv, dtype=np.float64).reshape(-1, 2)
        out = np.zeros((uv.shape[0], 3), dtype=np.float64)
        _native.check(self._lib.rt_pigment_color(self._handle, pigment, _abi.PRECISIONS[precision], _ptr(uv), uv.shape[0], _ptr(out)))
        return out

    def scatter(self, material: int, inputs: np.ndarray, state: int, inc: int, precision: str = "f64"):
        inputs = np.ascontiguousarray(inputs, dtype=np.float64).reshape(-1, 9)
        st = np.array([state, inc], dtype=np.uint64)
        out = np.zeros((inputs.shape[0], 8), dtype=np.float64)
        _native.check(self._lib.rt_scatter(self._handle, material, _abi.PRECISIONS[precision], _ptr(inputs), inputs.shape[0], _ptr(st), _ptr(out)))
        return out, int(st[0])


class MultiDeviceScene:
    """The same World resident on several devices of the node, rendered by ONE ``rt_render_multi`` call from
    this process: device i traces the interleaved rows i, i + n, ... and copies them into the caller's
    image; bit-identical to the single-device image (SURVEY §8b/e: ``CudaRenderer(..., gpus=n)``)."""

    def __init__(self, world_or_flat, devices):
        self._lib = _native.require_device()
        devices = list(range(devices)) if isinstance(devices, int) else [int(d) for d in devices]
        available = self._lib.rt_device_count()
        if not devices or len(set(devices)) != len(devices) or min(devices) < 0 or max(devices) >= available:
            raise ValueError(f"devices {devices}: need distinct indices below the {available} visible device(s)")
        self.flat: FlatScene = world_or_flat if isinstance(world_or_flat, FlatScene) else flatten_world(world_or_flat)
        self.devices = devices
        self.scenes = [DeviceScene(self.flat, device=d) for d in devices]
        _native.check(self._lib.rt_set_device(devices[0]))

    def close(self) -> None:
        for s in self.scenes:
            s.close()
        self.scenes = []

    def update_transforms(self, first: int, m: np.ndarray, invm: np.ndarray, stream: int = 0) -> None:
        for s in self.scenes:
            s.update_transforms(first, m, invm, stream)

    def update_from_world(self, world, stream: int = 0) -> None:
        new = world if isinstance(world, FlatScene) else flatten_world(world)
        if not self.flat.differs_only_in_transforms(new):
            raise ValueError("update_from_world: more than the transformations changed; build a new MultiDeviceScene")
        for s in self.scenes:
            s.update_transforms(0, new.shape_m, new.shape_invm, stream)

    def render(self, params: _abi.rt_render_params, want_hit: bool = False, out: Optional[np.ndarray] = None,
               replay_states: Optional[np.ndarray] = None) -> Tuple[np.ndarray, Optional[np.ndarray], dict]:
        if replay_states is not None:
            raise ValueError("replay is a single-device mode")
        H, W = params.height, params.width
        dtype = np.float64 if params.out_f64 else np.float32
        if out is None:
            out = np.empty((H, W, 3), dtype=dtype)
        assert out.dtype == dtype and out.shape == (H, W, 3) and out.flags.c_contiguous
        hit = np.empty((H, W), dtype=np.int32) if want_hit else None
        handles = (C.c_void_p * len(self.scenes))(*[s._handle for s in self.scenes])
        stats = _abi.rt_stats()
        _native.check(self._lib.rt_render_multi(handles, len(self.scenes), C.byref(params), _ptr(out), _ptr(hit), C.byref(stats)))
        return out, hit, stats.as_dict()

    def trace_rays(self, *args, **kw):
        return self.scenes[0].trace_rays(*args, **kw)


# ---------------------------------------------------------------------- scene-free probes
def camera_rays(params: _abi.rt_render_params, precision: str = "f64") -> np.ndarray:
    lib = _native.require_device()
    spp = max(1, params.samples_per_side) ** 2
    out = np.zeros((params.width * params.height * spp, 8), dtype=np.float64)
    _native.check(lib.rt_camera_rays(C.byref(params), _abi.PRECISIONS[precision], _ptr(out)))
    return out


def camera_fire(camera: _abi.rt_camera, uv: np.ndarray, precision: str = "f64") -> np.ndarray:
    lib = _native.require_device()
    uv = np.ascontiguousarray(uv, dtype=np.float64).reshape(-1, 2)
    out = np.zeros((uv.shape[0], 8), dtype=np.float64)
    _native.check(lib.rt_camera_fire(C.byref(camera), _abi.PRECISIONS[precision], _ptr(uv), uv.shape[0], _ptr(out)))
    return out


def pcg_seed(init_state: int, init_seq: int) -> Tuple[int, int]:
    lib = _native.require_device()
    st = np.zeros(2, dtype=np.uint64)
    _native.check(lib.rt_pcg_seed(init_state, init_seq, _ptr(st)))
    return int(st[0]), int(st[1])


def pcg_draw(state: int, inc: int, n: int):
    lib = _native.require_device()
    st = np.array([state, inc], dtype=np.uint64)
    out = np.zeros(n, dtype=np.uint32)
    _native.check(lib.rt_pcg_draw(_ptr(st), n, _ptr(out)))
    return out, int(st[0])


def onb(normals: np.ndarray, precision: str = "f64") -> np.ndarray:
    lib = _native.require_device()
    normals = np.ascontiguousarray(normals, dtype=np.float64).reshape(-1, 3)
    out = np.zeros((normals.shape[0], 9), dtype=np.float64)
    _native.check(lib.rt_onb(_abi.PRECISIONS[precision], _ptr(normals), normals.shape[0], _ptr(out)))
    return out


def ffma_peak_tflops(iterations: int = 4096) -> Tuple[float, float]:
    """Measured FP32 FMA throughput of the current device: (TFLOP/s, kernel ms)."""
    lib = _native.require_device()
    tf, ms = C.c_double(0.0), C.c_float(0.0)
    _native.check(lib.rt_bench_ffma(iterations, C.byref(tf), C.byref(ms)))
    return tf.value, ms.value


def dfma_peak_tflops(iterations: int = 1024) -> Tuple[float, float]:
    """Measured FP64 FMA throughput of the current device: (TFLOP/s, kernel ms)."""
    lib = _native.require_device()
    tf, ms = C.c_double(0.0), C.c_float(0.0)
    _native.check(lib.rt_bench_dfma(iterations, C.byref(tf), C.byref(ms)))
    return tf.value, ms.value
