"""ImageTracer (imagetracer.py:26-110) whose ``fire_all_rays`` is one CUDA launch.

``CudaImageTracer(image, camera, samples_per_side=0, pcg=PCG())`` has the reference's constructor
and ``fire_all_rays(func, callback=None, callback_time_s=2.0, **callback_kwargs)`` signature.

* ``func`` is a :class:`pytracer_b200.render.CudaRenderer`: the scene is flattened, ``rt_render``
  traces every pixel sample on the GPU and the image lands in ``image`` (array-backed images adopt
  the buffer; a reference ``HdrImage`` gets a lazy ``pixels`` view).  ``callback(col=0, row=0)`` is
  called first exactly like imagetracer.py:77-78, and once more for the last pixel.
* ``func`` is any other callable ``Ray -> Color`` (the reference's contract, e.g. the lambdas of its
  unit tests): the primary rays still come from the device (jittered by jump-ahead on ``pcg``), and
  ``func`` is applied to them in the reference's order on the host.

Either way ``self.pcg`` is left where the reference leaves it: 2 draws per sample further.
With a ``comm`` (see :mod:`pytracer_b200.dist`) every rank renders interleaved rows of the image and
copies them into one page-locked host image shared by the ranks of the node, which ``image`` adopts.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Optional

import numpy as np

from . import _abi, device
from .hdrimage import install_array
from .params import make_params
from .pcg import PCG
from .render import CudaRenderer
from .scene import Color, Point, Ray, Vec


@dataclass
class AdaptiveResult:
    """What ``fire_all_rays_adaptive`` returns besides the image: the standard error of every pixel's mean
    (float32 [H][W][3]), the samples every pixel received (int32 [H][W]), the passes run and the call's counters."""
    error: np.ndarray
    samples: np.ndarray
    passes: int
    stats: dict = field(default_factory=dict)


class ImageTracer:
    def __init__(self, image, camera, samples_per_side: int = 0, pcg: Optional[PCG] = None):
        self.image = image
        self.camera = camera
        self.samples_per_side = samples_per_side
        self.pcg = pcg if pcg is not None else PCG()
        self.last_stats: dict = {}

    def fire_ray(self, col: int, row: int, u_pixel: float = 0.5, v_pixel: float = 0.5) -> Ray:
        """imagetracer.py:48-58"""
        u = (col + u_pixel) / self.image.width
        v = 1.0 - (row + v_pixel) / self.image.height
        return self.camera.fire_ray(u, v)

    def _params(self, renderer: Optional[CudaRenderer], **overrides) -> _abi.rt_render_params:
        w, h = self.image.width, self.image.height
        if renderer is not None:
            return renderer.make_params(w, h, self.camera, self.samples_per_side, aa_pcg=self.pcg, **overrides)
        return make_params(w, h, self.camera, samples_per_side=self.samples_per_side, aa_pcg=self.pcg, **overrides)

    def _draws_per_image(self) -> int:
        return 2 * self.image.width * self.image.height * self.samples_per_side ** 2

    def fire_all_rays(self, func, callback=None, callback_time_s: float = 2.0, comm=None, **callback_kwargs):
        if callback:
            callback(col=0, row=0, **callback_kwargs)
        if isinstance(func, CudaRenderer):
            self._fire_cuda(func, comm)
        else:
            self._fire_callable(func)
        self.pcg.advance(self._draws_per_image())
        if callback:
            callback(col=self.image.width - 1, row=self.image.height - 1, **callback_kwargs)

    def fire_all_rays_adaptive(self, renderer, target_error: float = 0.0, max_samples_per_pixel: Optional[int] = None,
                               error_floor: float = 1e-2, callback=None, callback_time_s: float = 2.0,
                               error_estimator: str = "batch", **callback_kwargs) -> AdaptiveResult:
        """Path-traced image with a per-pixel Monte Carlo error map, optionally refined where it is noisy.

        Pass 0 is exactly ``fire_all_rays(renderer)``; every further pass traces ``samples_per_side ** 2`` more
        samples, for the pixels whose relative error max_c SE_c / max(mean_c, error_floor) is still above
        ``target_error``, until they meet it or hold ``max_samples_per_pixel`` samples (default: one pass, the
        error map only).  Pass p of a pixel is that pixel of the (p+1)-th consecutive ``fire_all_rays``; a pixel
        with P passes holds the mean of its P pass values.  ``self.image`` receives the mean image, and
        ``self.pcg`` and ``renderer.pcg`` are left where ``passes`` consecutive ``fire_all_rays`` leave them.
        ``error_estimator`` forms each pass's SE from the stratified samples: "batch" treats them as independent
        (conservative); "paired" collapses pairs of horizontally adjacent strata, which credits stratification
        and so reports less where radiance is smooth within the pixel (even ``samples_per_side`` only)."""
        spp = self.samples_per_side ** 2
        if not isinstance(renderer, CudaRenderer) or renderer.algorithm != "pathtracing":
            raise ValueError("fire_all_rays_adaptive needs a path-tracing CudaRenderer")
        if self.samples_per_side < 2:
            raise ValueError(f"the error map needs samples_per_side >= 2 (got {self.samples_per_side})")
        if not (isinstance(renderer.gpus, int) and renderer.gpus == 1):
            raise ValueError("adaptive rendering runs on one device (gpus=1)")
        if renderer.variant == "mega" or renderer.precision in ("f64", "hybrid"):
            raise ValueError("adaptive rendering uses the fp32 warp path tracer (variant auto/warp, precision auto/f32)")
        if not np.isfinite(target_error) or target_error < 0:
            raise ValueError(f"target_error must be finite and >= 0 (got {target_error})")
        if not (np.isfinite(error_floor) and error_floor > 0):
            raise ValueError(f"error_floor must be > 0 (got {error_floor})")
        if error_estimator not in _abi.ERROR_ESTIMATORS:
            raise ValueError(f"error_estimator must be one of {sorted(_abi.ERROR_ESTIMATORS)} (got {error_estimator!r})")
        if error_estimator == "paired" and self.samples_per_side % 2:
            raise ValueError(f"the paired error estimator needs an even samples_per_side (got {self.samples_per_side})")
        if max_samples_per_pixel is None:
            max_samples_per_pixel = spp
        if int(max_samples_per_pixel) != max_samples_per_pixel or max_samples_per_pixel < spp or max_samples_per_pixel % spp:
            raise ValueError(f"max_samples_per_pixel ({max_samples_per_pixel}) must be a positive multiple of the "
                             f"samples per pass ({spp})")
        max_passes = int(max_samples_per_pixel) // spp
        if max_passes >= 2 ** 31:
            raise ValueError(f"max_samples_per_pixel ({max_samples_per_pixel}) is too large")
        if callback:
            callback(col=0, row=0, **callback_kwargs)
        scene = renderer.device_scene()
        rgb, err, samples, stats = scene.render_adaptive(self._params(renderer), target_error, max_passes, error_floor,
                                                         out=self._adoptable_buffer(), estimator=error_estimator)
        passes = stats["passes"]
        self.last_stats = renderer.last_stats = stats
        for _ in range(passes):  # where `passes` consecutive fire_all_rays leave both generators
            renderer.pcg.random()
        self.pcg.advance(passes * self._draws_per_image())
        install_array(self.image, rgb)
        if callback:
            callback(col=self.image.width - 1, row=self.image.height - 1, **callback_kwargs)
        return AdaptiveResult(error=err, samples=samples, passes=passes, stats=stats)

    # -- the product path
    def _fire_cuda(self, renderer: CudaRenderer, comm=None) -> None:
        scene = renderer.device_scene()
        shared = comm is not None and comm.world_size > 1
        if shared:
            # rows of the image interleaved over the ranks, each rank's rows copied straight into ONE
            # page-locked host image shared by the node: the image object adopts that memory
            from .dist import render_rows_to_shared_host

            rgb, stats = render_rows_to_shared_host(scene, self._params(renderer), comm)
        else:
            rgb, _, stats = scene.render(self._params(renderer), out=self._adoptable_buffer())
        self.last_stats = renderer.last_stats = stats
        if renderer.algorithm == "pathtracing":
            renderer.pcg.random()  # the next image must not reuse these sample streams
        install_array(self.image, rgb, adopt=shared)  # the shared image is adopted, never copied (24.9 MB per frame)

    def _adoptable_buffer(self) -> Optional[np.ndarray]:
        arr = getattr(self.image, "_rgb", None)
        if isinstance(arr, np.ndarray) and arr.dtype == np.float32 and arr.flags.c_contiguous:
            if hasattr(self.image, "pin"):
                self.image.pin()
            return arr
        return None

    # -- arbitrary Python callables: device-generated rays, host-applied function
    def _fire_callable(self, func) -> None:
        rays = device.camera_rays(self._params(None))
        spp = max(1, self.samples_per_side) ** 2
        w, h = self.image.width, self.image.height
        out = np.zeros((h, w, 3), dtype=np.float64)
        k = 0
        for row in range(h):
            for col in range(w):
                cum = Color(0.0, 0.0, 0.0)
                for _ in range(spp):
                    r = rays[k]
                    k += 1
                    c = func(Ray(Point(*r[0:3]), Vec(*r[3:6]), float(r[6]), float(r[7]), 0))
                    cum = Color(cum.r + c.r, cum.g + c.g, cum.b + c.b) if self.samples_per_side > 0 else c
                if self.samples_per_side > 0:
                    s = 1 / self.samples_per_side ** 2
                    cum = Color(cum.r * s, cum.g * s, cum.b * s)
                out[row, col] = (cum.r, cum.g, cum.b)
        install_array(self.image, out.astype(np.float32) if hasattr(self.image, "_rgb") else out)


CudaImageTracer = ImageTracer
