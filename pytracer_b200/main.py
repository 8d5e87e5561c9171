"""`python -m pytracer_b200 render …` — the reference's `render` command (main.py:76-214: same options,
same defaults, same messages) with the image traced on the GPU.  Extra switches: --gpus/--variant/
--precision/--parser.  Scene parsing uses the reference's own parser when the `pytracer` package is
importable (`--parser reference`), otherwise this repository's reader of the same language."""
from __future__ import annotations

import sys
from math import sqrt
from time import perf_counter

import click

from .hdrimage import HdrImage
from .imagetracer import CudaImageTracer
from .pcg import PCG
from .render import RENDERERS, FlatRenderer, OnOffRenderer, PathTracer, PointLightRenderer
from .scene import BLACK


def build_variable_table(definitions):
    variables = {}
    for declaration in definitions:
        parts = declaration.split(":")
        if len(parts) != 2:
            print(f"error, the definition «{declaration}» does not follow the pattern NAME:VALUE")
            sys.exit(1)
        name, value = parts
        try:
            value = float(value)
        except ValueError:
            print(f"invalid floating-point value «{value}» in definition «{declaration}»")
            sys.exit(1)
        variables[name] = value
    return variables


def load_scene(path: str, variables, parser: str):
    if parser in ("auto", "reference"):
        try:
            from pytracer.scene_file import GrammarError as RefGrammarError, InputStream, parse_scene

            with open(path, "rt") as f:
                try:
                    return parse_scene(input_file=InputStream(stream=f, file_name=path), variables=variables)
                except RefGrammarError as e:
                    loc = e.location
                    print(f"{loc.file_name}:{loc.line_num}:{loc.col_num}: {e.message}")
                    sys.exit(1)
        except ImportError:
            if parser == "reference":
                raise
    from .scene_text import GrammarError, parse_scene_text

    with open(path, "rt") as f:
        try:
            return parse_scene_text(f.read(), variables, file_name=path)
        except GrammarError as e:
            print(str(e))
            sys.exit(1)


def adaptive_cli_problem(algorithm, samples_per_pixel, gpus, variant, precision, target_error, max_samples_per_pixel,
                         error_floor, error_estimator="batch", mean_samples_per_pixel=None, mean_rays_per_pixel=None):
    """Why `render --error-output / --target-error / --max-samples-per-pixel / --mean-samples-per-pixel /
    --mean-rays-per-pixel` cannot run as asked (None: it can)."""
    if algorithm != "pathtracing":
        return "--error-output, --target-error and --max-samples-per-pixel need --algorithm pathtracing"
    if samples_per_pixel < 4:
        return f"the error map needs at least 4 samples per pixel per pass (got {samples_per_pixel})"
    if gpus != 1:
        return "adaptive rendering runs on one GPU (--gpus 1)"
    if variant == "mega" or precision == "f64":
        return "adaptive rendering uses the fp32 warp path tracer (--variant auto|warp, --precision auto|f32)"
    if target_error is not None and (not target_error >= 0 or target_error == float("inf")):
        return f"--target-error must be a finite number >= 0 (got {target_error})"
    if not error_floor > 0:
        return f"--error-floor must be > 0 (got {error_floor})"
    if mean_rays_per_pixel is not None:
        if mean_samples_per_pixel is not None:
            return "--mean-rays-per-pixel and --mean-samples-per-pixel exclude each other"
        if not (mean_rays_per_pixel >= 0 and mean_rays_per_pixel != float("inf")):
            return f"--mean-rays-per-pixel must be a finite number >= 0 (got {mean_rays_per_pixel})"
        if max_samples_per_pixel is None:
            return "--mean-rays-per-pixel needs --max-samples-per-pixel"
    elif mean_samples_per_pixel is None:
        if (target_error is not None and target_error > 0) != (max_samples_per_pixel is not None):
            return "--target-error and --max-samples-per-pixel go together"
    elif max_samples_per_pixel is None:
        return "--mean-samples-per-pixel needs --max-samples-per-pixel"
    elif mean_samples_per_pixel < samples_per_pixel:
        return (f"--mean-samples-per-pixel ({mean_samples_per_pixel}) must be at least --samples-per-pixel "
                f"({samples_per_pixel}), the first pass")
    elif max_samples_per_pixel < mean_samples_per_pixel:
        return (f"--max-samples-per-pixel ({max_samples_per_pixel}) must be at least --mean-samples-per-pixel "
                f"({mean_samples_per_pixel})")
    if max_samples_per_pixel is not None and (max_samples_per_pixel < samples_per_pixel or max_samples_per_pixel % samples_per_pixel):
        return (f"--max-samples-per-pixel ({max_samples_per_pixel}) must be a positive multiple of "
                f"--samples-per-pixel ({samples_per_pixel})")
    if error_estimator == "paired" and int(sqrt(samples_per_pixel)) % 2:
        return (f"--error-estimator paired needs an even number of samples per side "
                f"(--samples-per-pixel 4, 16, 36, 64, ...; got {samples_per_pixel})")
    return None


@click.group()
def cli():
    pass


@cli.command("render")
@click.option("--width", type=int, default=640, help="Width of the image to render")
@click.option("--height", type=int, default=480, help="Height of the image to render")
@click.option("--algorithm", type=click.Choice(RENDERERS), default="pathtracing")
@click.option("--pfm-output", type=str, default="output.pfm", help="Name of the PFM file to create")
@click.option("--png-output", type=str, default="output.png", help="Name of the PNG file to create")
@click.option("--num-of-rays", type=int, default=10)
@click.option("--max-depth", type=int, default=3)
@click.option("--init-state", type=int, default=45)
@click.option("--init-seq", type=int, default=54)
@click.option("--samples-per-pixel", type=int, default=1)
@click.option("--declare-float", "-d", type=str, multiple=True)
@click.option("--variant", type=click.Choice(["auto", "mega", "warp"]), default="auto")
@click.option("--precision", type=click.Choice(["auto", "f32", "f64"]), default="auto")
@click.option("--parser", type=click.Choice(["auto", "reference", "builtin"]), default="auto")
@click.option("--accel", type=click.Choice(["none", "bvh"]), default="none", help="bvh: sphere hierarchy, same image")
@click.option("--gpus", type=int, default=1, help="GPUs of this node to render on: interleaved rows, one rt_render_multi call from this process")
@click.option("--launcher", type=click.Choice(["inprocess", "torchrun"]), default="inprocess",
              help="with --gpus N: drive the N devices from this process (default) or re-launch under torchrun, one process per GPU")
@click.option("--error-output", type=str, default=None, help="PFM file to receive the standard error of every pixel (path tracing)")
@click.option("--target-error", type=float, default=None,
              help="render adaptively: trace more passes of --samples-per-pixel samples where the relative error is above this")
@click.option("--max-samples-per-pixel", type=int, default=None, help="with --target-error: samples per pixel at most")
@click.option("--mean-samples-per-pixel", type=int, default=None,
              help="render to a sample budget of this many samples per pixel on average (with --max-samples-per-pixel): "
                   "after the first pass, trace the pixels of largest relative error (above --target-error, if given)")
@click.option("--mean-rays-per-pixel", type=float, default=None,
              help="render to a budget of this many closest-hit rays per pixel on average (with --max-samples-per-pixel): after "
                   "the first pass, trace the pixels whose next pass buys the most error reduction per predicted ray")
@click.option("--error-floor", type=float, default=1e-2, help="radiance below which the relative error is taken against this floor")
@click.option("--error-estimator", type=click.Choice(["batch", "paired"]), default="batch",
              help="how the standard error is formed: batch (strata as independent samples) or paired (collapsed pairs "
                   "of adjacent strata, tighter under stratification; even samples per side)")
@click.argument("input_scene_name", type=str)
def render(width, height, algorithm, pfm_output, png_output, num_of_rays, max_depth, init_state, init_seq,
           samples_per_pixel, declare_float, variant, precision, parser, accel, gpus, launcher, error_output, target_error,
           max_samples_per_pixel, mean_samples_per_pixel, mean_rays_per_pixel, error_floor, error_estimator, input_scene_name):
    import os

    if gpus > 1 and launcher == "torchrun" and "WORLD_SIZE" not in os.environ:  # one process per GPU: hand the same command line to torchrun
        import socket
        import subprocess

        with socket.socket() as sock:
            sock.bind(("127.0.0.1", 0))
            port = sock.getsockname()[1]
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={gpus}",
               "--master-addr", "127.0.0.1", "--master-port", str(port), "-m", "pytracer_b200", *sys.argv[1:]]
        sys.exit(subprocess.call(cmd))
    samples_per_side = int(sqrt(samples_per_pixel))
    if samples_per_side ** 2 != samples_per_pixel:
        print(f"Error, the number of samples per pixel ({samples_per_pixel}) must be a perfect square")
        return
    adaptive = (error_output is not None or target_error is not None or max_samples_per_pixel is not None
                or mean_samples_per_pixel is not None or mean_rays_per_pixel is not None)
    if error_estimator != "batch" and not adaptive:
        print("Error, --error-estimator applies to --error-output and --target-error")
        sys.exit(1)
    if adaptive:
        problem = adaptive_cli_problem(algorithm, samples_per_pixel, gpus, variant, precision, target_error,
                                       max_samples_per_pixel, error_floor, error_estimator,
                                       mean_samples_per_pixel=mean_samples_per_pixel, mean_rays_per_pixel=mean_rays_per_pixel)
        if problem:
            print(f"Error, {problem}")
            sys.exit(1)
    scene = load_scene(input_scene_name, build_variable_table(declare_float), parser)
    image = HdrImage(width, height)
    print(f"Generating a {width}×{height} image")
    tracer = CudaImageTracer(image=image, camera=scene.camera, samples_per_side=samples_per_side)
    extra = dict(variant=variant, precision=precision, accel=accel)
    if gpus > 1 and "WORLD_SIZE" not in os.environ:
        extra["gpus"] = gpus
    if algorithm == "onoff":
        print("Using on/off renderer")
        renderer = OnOffRenderer(world=scene.world, background_color=BLACK, **extra)
    elif algorithm == "flat":
        print("Using flat renderer")
        renderer = FlatRenderer(world=scene.world, background_color=BLACK, **extra)
    elif algorithm == "pathtracing":
        print("Using a path tracer")
        renderer = PathTracer(world=scene.world, pcg=PCG(init_state=init_state, init_seq=init_seq),
                              num_of_rays=num_of_rays, max_depth=max_depth, **extra)
    else:
        print("Using a point-light tracer")
        renderer = PointLightRenderer(world=scene.world, background_color=BLACK, **extra)

    comm = None
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:  # launched under torchrun: one rank per GPU
        from .dist import TorchComm

        comm = TorchComm.from_env()
    start = perf_counter()
    result = None
    if adaptive:
        result = tracer.fire_all_rays_adaptive(renderer, target_error=target_error or 0.0,
                                               max_samples_per_pixel=max_samples_per_pixel, error_floor=error_floor,
                                               error_estimator=error_estimator, mean_samples_per_pixel=mean_samples_per_pixel,
                                               mean_rays_per_pixel=mean_rays_per_pixel)
    else:
        tracer.fire_all_rays(renderer, comm=comm)
    elapsed = perf_counter() - start
    st = tracer.last_stats
    rays = st.get("rays_closest", 0) + st.get("rays_shadow", 0)
    print(f"Rendering completed in {elapsed:.3f} s ({rays} rays, {rays / max(elapsed, 1e-9) / 1e6:.1f} Mrays/s, "
          f"kernel {st.get('kernel_ms', 0.0):.2f} ms)")
    if result is not None:
        print(f"{result.passes} pass(es) of {samples_per_pixel} samples; pixels per pass: "
              f"{', '.join(str(n) for n in st['pixels_in_pass'])}; {st['samples']} samples in all "
              f"({st['samples'] / (width * height):.1f} per pixel)"
              + (f"; budget {st['sample_budget']} samples, {st['samples']} spent" if "sample_budget" in st else "")
              + (f"; budget {st['ray_budget']} rays, {st['rays_closest']} spent" if "ray_budget" in st else ""))
    if comm is not None and comm.rank != 0:
        return
    with open(pfm_output, "wb") as outf:
        image.write_pfm(outf)
    print(f"HDR demo image written to {pfm_output}")
    if result is not None and error_output is not None:
        from .hdrimage import install_array

        err_image = HdrImage(width, height)
        install_array(err_image, result.error)
        with open(error_output, "wb") as outf:
            err_image.write_pfm(outf)
        print(f"Standard error of every pixel written to {error_output}")
    try:
        from .tonemap import write_ldr_image

        with open(png_output, "wb") as outf:
            write_ldr_image(image, outf, "PNG", factor=1.0)
        print(f"PNG demo image written to {png_output}")
    except ImportError as e:
        print(f"PNG output skipped ({e})")


@cli.command("animate")
@click.option("--width", type=int, default=640)
@click.option("--height", type=int, default=480)
@click.option("--algorithm", type=click.Choice(RENDERERS), default="pathtracing")
@click.option("--output-prefix", type=str, default="frame", help="files are <prefix>NNN.pfm / .png")
@click.option("--num-of-rays", type=int, default=10)
@click.option("--max-depth", type=int, default=3)
@click.option("--init-state", type=int, default=45)
@click.option("--init-seq", type=int, default=54)
@click.option("--samples-per-pixel", type=int, default=1)
@click.option("--declare-float", "-d", type=str, multiple=True)
@click.option("--variable", type=str, default="clock", help="the float variable that changes from frame to frame")
@click.option("--start", type=float, default=0.0)
@click.option("--stop", type=float, default=360.0)
@click.option("--frames", type=int, default=36)
@click.option("--variant", type=click.Choice(["auto", "mega", "warp"]), default="auto")
@click.option("--precision", type=click.Choice(["auto", "f32", "f64"]), default="auto")
@click.option("--parser", type=click.Choice(["auto", "reference", "builtin"]), default="auto")
@click.option("--no-png", is_flag=True)
@click.argument("input_scene_name", type=str)
def animate(width, height, algorithm, output_prefix, num_of_rays, max_depth, init_state, init_seq, samples_per_pixel,
            declare_float, variable, start, stop, frames, variant, precision, parser, no_png, input_scene_name):
    """The loop users of the reference write around `render -d clock:VALUE` (one process, one parse and
    one full render per frame): here the scene stays resident in HBM and only the transformations that
    changed are uploaded per frame (SURVEY §8f-4)."""
    samples_per_side = int(sqrt(samples_per_pixel))
    if samples_per_side ** 2 != samples_per_pixel:
        print(f"Error, the number of samples per pixel ({samples_per_pixel}) must be a perfect square")
        return
    base = build_variable_table(declare_float)
    renderer, patched = None, 0
    t_all = perf_counter()
    for f in range(frames):
        value = start + (stop - start) * f / max(1, frames)
        scene = load_scene(input_scene_name, dict(base, **{variable: value}), parser)
        if renderer is None:
            extra = dict(variant=variant, precision=precision)
            renderer = {"onoff": OnOffRenderer, "flat": FlatRenderer, "pointlight": PointLightRenderer}.get(algorithm)
            if renderer is None:
                renderer = PathTracer(world=scene.world, pcg=PCG(init_state=init_state, init_seq=init_seq),
                                      num_of_rays=num_of_rays, max_depth=max_depth, **extra)
            else:
                renderer = renderer(world=scene.world, background_color=BLACK, **extra)
        else:
            patched += bool(renderer.set_world(scene.world))
        image = HdrImage(width, height)
        tracer = CudaImageTracer(image=image, camera=scene.camera, samples_per_side=samples_per_side)
        t0 = perf_counter()
        tracer.fire_all_rays(renderer)
        dt = perf_counter() - t0
        with open(f"{output_prefix}{f:03d}.pfm", "wb") as outf:
            image.write_pfm(outf)
        if not no_png:
            from .tonemap import write_ldr_image

            with open(f"{output_prefix}{f:03d}.png", "wb") as outf:
                write_ldr_image(image, outf, "PNG", factor=1.0)
        print(f"frame {f:03d} ({variable} = {value:g}): rendered in {dt * 1e3:.1f} ms")
    print(f"{frames} frames in {perf_counter() - t_all:.2f} s; the resident scene was patched in place for {patched} of them")


if __name__ == "__main__":
    cli()
