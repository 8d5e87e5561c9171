#!/usr/bin/env python
"""Benchmark of the rendering hot path: path-traced rays/s on BASELINE config 3, with configs 4 and 5
measured beside it in the same line (`configs`).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c3|c4|c5|tonemap]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A *step* is one full render of the workload (ImageTracer.fire_all_rays over every pixel sample).
`value` is whole-job rays/s (closest-hit + shadow queries, the events BASELINE.md §3.3 counts) with the
scene resident in HBM and the image left in HBM, timed with CUDA events on the launch stream, max over
ranks; `e2e` is the same metric through the public API (CudaImageTracer.fire_all_rays: flatten, scene
upload, launch, device->host copy of the image into a page-locked host image) timed on the host clock,
max over ranks.  With N > 1 the rows of the image are interleaved over the ranks (`scaling: strong` — the
frame is fixed, the work is split): device-resident, the render kernel stores every finished pixel into
every rank's image over NVLink (symmetric memory) and a barrier closes the step (`--exchange allgather`:
one in-place NCCL all-gather of the row slabs instead; `--partition spp`: the strata split with one NCCL
sum); end to end,
every rank copies its rows straight into one page-locked host image shared by the node.

`--impl reference` times the reference's CPU implementation on all host threads: the C restatement
(oracle/pt_oracle.c, bit-exact with the Python reference — tests/test_oracle_golden.py) as the line's
value, and the unmodified Python reference itself (baseline/_ref, BASELINE config 1) beside it.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

# Rank 0 prints exactly ONE line on stdout: the JSON.  Libraries write there too (NCCL prints its
# "NCCL version ..." banner on fd 1 whenever NCCL_DEBUG is set), so fd 1 is pointed at stderr for the
# whole run and the JSON line goes to the saved descriptor.
sys.stdout.flush()
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit(line: dict) -> None:
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

SCALE = 1
METRIC = "path-traced rays/sec (demo.txt 1080p)"
UNIT = "rays/s"
_WORKLOADS = {}


def workload(name):
    """(world, camera, render kwargs, description, flops per ray, sphere count); cached per process."""
    from pytracer_b200 import scenes

    if name in _WORKLOADS:
        return _WORKLOADS[name]
    if name == "c3":
        world, camera = scenes.demo_scene()
        kw = dict(width=1920, height=1080, samples_per_side=8, algorithm="pathtracing", num_of_rays=10, max_depth=3, rr_limit=3)
        desc = "BASELINE config 3: examples/demo.txt pathtracing 1920x1080, 64 spp, num-of-rays 10, max-depth 3, Russian roulette limit 3"
        n_sph, n_pl = 1, 2
    elif name == "c4":
        rs = scenes.random_spheres_scene(1024, 2024, 4, 20.0)
        world, camera = rs.world, rs.camera
        kw = dict(width=3840, height=2160, samples_per_side=4, algorithm="pathtracing", num_of_rays=10, max_depth=3, rr_limit=3)
        desc = "BASELINE config 4: 1024 random ellipsoids + 2 planes, checkered/image pigments, pathtracing 3840x2160, 16 spp"
        n_sph, n_pl = 1024, 2
    elif name == "c5":
        rs = scenes.random_spheres_scene(4096, 2025, 5, 40.0, with_light=True)
        world, camera = rs.world, rs.camera
        kw = dict(width=3840, height=2160, samples_per_side=2, algorithm="pointlight")
        desc = "BASELINE config 5: 4096 random ellipsoids + 2 planes, pointlight 3840x2160, 4 spp"
        n_sph, n_pl = 4096, 2
    else:
        raise SystemExit(f"unknown workload {name}")
    # SURVEY §8(d): 54 per sphere test, 12 per plane test, 60 for the winner's record, 46 scatter
    flops_per_ray = 54 * n_sph + 12 * n_pl + 60 + 46
    if SCALE > 1:
        kw["width"], kw["height"] = kw["width"] // SCALE, kw["height"] // SCALE
        desc += f" [SCALED DOWN {SCALE}x per side: experiment, not the benchmark]"
    _WORKLOADS[name] = (world, camera, kw, desc, flops_per_ray, n_sph)
    return _WORKLOADS[name]


def build_params(kw, camera, **extra):
    from pytracer_b200.params import make_params
    from pytracer_b200.pcg import PCG

    args = dict(kw)
    width, height = args.pop("width"), args.pop("height")
    args.update(aa_pcg=PCG(42, 54), pt_pcg=PCG(45, 54))  # the CLI's generators (main.py:168-185)
    args.update(extra)
    return make_params(width, height, camera, **args)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region: the sampler is started before the
    warm-up (nvidia-smi takes a few hundred ms to deliver its first line) and only the samples whose
    timestamps fall between `mark_begin()` and `mark_end()` are reported (all of them if none does)."""

    FIELDS = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.proc, self.path = None, None
        self.t0 = self.t1 = None
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "40"],
                stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    @staticmethod
    def _stamp(text):
        import datetime

        try:
            return datetime.datetime.strptime(text.strip(), "%Y/%m/%d %H:%M:%S.%f").timestamp()
        except ValueError:
            return None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        if self.t1 is None:
            self.mark_end()
        time.sleep(0.08)  # one more sampling period: the line of the last interval is on its way
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        rows = []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                parts = [x.strip() for x in line.split(",")]
                if len(parts) < 8:
                    continue
                try:
                    rows.append((self._stamp(parts[0]), float(parts[1]), float(parts[2]),
                                 [n for n, val in zip(names, parts[4:8]) if val.lower().startswith("active")]))
                except ValueError:
                    continue
            os.unlink(self.path)
        except Exception:
            pass
        inside = [r for r in rows if r[0] is not None and self.t0 is not None and self.t0 - 0.04 <= r[0] <= self.t1 + 0.04]
        used = inside or rows
        if used:
            out = {"sm_mhz": statistics.median(r[1] for r in used), "sm_max_mhz": max(r[2] for r in used),
                   "reasons": sorted({n for r in used for n in r[3]}), "samples": len(used),
                   "window": "timed region" if inside else "whole run (no sample fell inside the timed region)"}
        return out


DUMP_BYTES = 64 * 1024 * 1024  # --dump-outputs writes at most this much
DUMP_SAMPLE_PIXELS = 1 << 20


def write_outputs(directory, arrays):
    """`--dump-outputs DIR`: each array as DIR/<name>.npy, float64 where the data is float64 (the ray counters
    are passed as such), float32 otherwise.  An image of more than half of DUMP_BYTES (the 4K frames, the 8K tone-mapped frame)
    is stored as a fixed sample of DUMP_SAMPLE_PIXELS pixels, drawn without replacement with numpy seed 0:
    <name>.npy holds their values (pixels x channels), <name>_index.npy their flat indices in ascending order."""
    out = {}
    for name, a in arrays.items():
        a = np.asarray(a)
        dtype = np.float64 if a.dtype == np.float64 else np.float32
        if a.size * np.dtype(dtype).itemsize > DUMP_BYTES // 2:
            pixels = a.reshape(-1, a.shape[-1])
            index = np.sort(np.random.default_rng(0).choice(pixels.shape[0], DUMP_SAMPLE_PIXELS, replace=False))
            out[name], out[name + "_index"] = pixels[index].astype(dtype), index.astype(np.float64)
        else:
            out[name] = a.astype(dtype)
    total = sum(a.nbytes for a in out.values())
    assert total <= DUMP_BYTES, f"--dump-outputs: {total} bytes"
    os.makedirs(directory, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def cpu_baseline_sample(name, threads, width=None, height=None):
    """The oracle on a bounded sample of the same workload: the same scene and settings at 1 sample per
    pixel — the full frame for demo.txt, a crop-sized frame for the many-sphere scenes (ms per ray there;
    BASELINE.md §3.2 asks for 64x36) — on `threads` host threads."""
    from oracle import oracle
    from pytracer_b200.flatten import flatten_world

    world, camera, kw, _, _, n_sph = workload(name)
    flat = flatten_world(world)
    args = dict(kw)
    # 1 sample per pixel on one thread; the threaded arm takes 4 (about 1.6 s per step on 16 threads instead of 0.4)
    args["samples_per_side"] = 2 if (threads > 1 and n_sph <= 100 and not width) else 1
    if width:
        args["width"], args["height"] = width, height
    elif n_sph > 100:
        args["width"], args["height"] = (64, 36) if threads == 1 else (256, 144)
    p = build_params(args, camera)
    t0 = time.perf_counter()
    r = oracle.render_threaded(flat, p, threads) if threads > 1 else oracle.render(flat, p, want_hit=False)
    dt = time.perf_counter() - t0
    rays = r["rays_closest"] + r["rays_shadow"]
    sample = f"{args['width']}x{args['height']} at {args['samples_per_side'] ** 2} spp of the same scene/settings ({rays} rays, {dt:.1f} s)"
    return rays / dt, sample


def python_reference(all_cores=False):
    """The unmodified Python reference on BASELINE config 1 (oracle/python_ref.py); a dict for the JSON line."""
    try:
        from oracle import python_ref

        why = python_ref.available()
        if why:
            return {"unavailable": why}
        r = python_ref.run_config1()
        out = {"value": r["rays"] / r["wall_s"], "unit": UNIT, "cores": 1, "kind": "reference",
               "sample": f"BASELINE config 1 exactly: demo.txt pathtracing 160x120, 1 spp, N=10, depth 3, seeds 42/45 "
                         f"({r['rays']} rays, {r['wall_s']:.1f} s wall, {r['cpu_s']:.1f} s process_time as main.py:196-200 times it)",
               "rays": r["rays"], "rays_match_golden": r["rays"] == python_ref.C1_RAYS, "mean_rgb": r["mean_rgb"]}
        if all_cores:
            a = python_ref.run_config1_all_cores()
            out["all_cores"] = {"value": a["rays_per_s"], "unit": UNIT, "cores": a["processes"],
                                "sample": f"{a['processes']} independent processes, config 1 each with its own --init-state ({a['rays']} rays, {a['wall_s']:.1f} s)"}
        return out
    except Exception as exc:  # the baseline must never take the benchmark down
        return {"unavailable": f"{type(exc).__name__}: {exc}"}


def run_reference(args, rank, world_size):
    if rank != 0:
        return
    _, _, kw, desc, _, _ = workload(args.workload)
    threads = os.cpu_count() or 1
    from oracle import oracle

    oracle.build()
    for _ in range(args.warmup):
        cpu_baseline_sample(args.workload, threads, 480, 270)
    rates, sample = [], ""
    t_all = time.perf_counter()
    for _ in range(args.steps):
        rate, sample = cpu_baseline_sample(args.workload, threads)
        rates.append(rate)
    total = time.perf_counter() - t_all
    value = statistics.mean(rates)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / max(1, args.steps), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": desc},
        "run": {"note": "CPU restatement of the reference (oracle/pt_oracle.c, bit-exact with the Python reference on the golden "
                "fixtures), one bounded sample per step: a RATE on the same scene and settings"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if not args.no_python_ref:
        line["cpu_baseline"]["python_ref"] = python_reference(all_cores=True)
    emit(line)


def run_tonemap(args, rank, local_rank, world_size):
    """Extra line (not the headline): the tone-mapping step that follows a render (SURVEY §8f-2), HBM-bound.
    A step = average luminosity + normalise/clamp/quantise of one 7680x4320 fp32 frame resident in HBM."""
    import torch

    from oracle import tonemap_oracle
    from pytracer_b200 import tonemap

    if rank != 0:
        return
    torch.cuda.set_device(local_rank)
    h, w = 4320 // SCALE, 7680 // SCALE
    n = h * w
    gen = torch.Generator(device="cuda").manual_seed(11)
    img = torch.exp(torch.randn((h, w, 3), device="cuda", generator=gen)).contiguous()
    ldr = torch.empty((h, w, 3), dtype=torch.uint8, device="cuda")
    flush = torch.zeros(64 * 1024 * 1024, dtype=torch.float32, device="cuda")  # 256 MB, read to evict L2 cleanly
    lum_ms, map_ms, total_ms = [], [], []
    sampler = ClockSampler(local_rank)
    for i in range(args.warmup + args.steps):
        flush.sum()
        st = tonemap.tone_map_device(img.data_ptr(), n, 1.0, None, 1.0, 0, ldr.data_ptr())
        if i >= args.warmup:
            lum_ms.append(st["lum_ms"]); map_ms.append(st["map_ms"]); total_ms.append(st["lum_ms"] + st["map_ms"])
    clocks = sampler.stop()
    if args.dump_outputs:
        write_outputs(args.dump_outputs, {"ldr": ldr.cpu().numpy(), "luminosity": np.array([st["luminosity"]])})
    # end to end: host image in (pinned), LDR bytes out
    himg = torch.empty((h, w, 3), dtype=torch.float32).pin_memory()
    himg.copy_(img)
    e2e = []
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        _, out, _ = tonemap.tone_map(himg.numpy(), 1.0, None, 1.0, want_hdr=False)
        dt = time.perf_counter() - t0
        if i >= args.warmup:
            e2e.append(dt)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6534.5))
    traffic = None
    try:
        if SCALE == 1:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get("tonemap")
    except Exception:
        pass
    k_lum, k_map = statistics.mean(lum_ms), statistics.mean(map_ms)
    ms = statistics.mean(total_ms)
    line = {
        "metric": "tone-mapped pixels/sec (average luminosity + normalise/clamp/8-bit, fp32 frame resident in HBM)",
        "value": n / (ms * 1e-3), "unit": "pixels/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64 semantics (fp32 fast path with fp64 guard)",
        "data": "synthetic", "config": {"workload": f"tone mapping of one {w}x{h} frame (hdrimages.py:120-171)", "l2": "256 MB read between steps"},
        "e2e": {"value": n / statistics.mean(e2e), "unit": "pixels/s", "h2d_bytes_per_step": 12 * n, "d2h_bytes_per_step": 3 * n},
        "gpu_launches": 2 * args.steps, "clocks": clocks,
        "roofline": {"bound": "hbm", "achieved": 15 * n / (k_map * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                     "frac": 15 * n / (k_map * 1e-3) / 1e9 / peak, "traffic": traffic, "kernel": "k_tone_map_ldr (12 B read + 3 B written per pixel)",
                     "kernel_ms": k_map, "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6534.5 GB/s",
                     "other_kernel": {"kernel": "k_lum_sum (12 B read per pixel)", "kernel_ms": k_lum,
                                      "achieved": 12 * n / (k_lum * 1e-3) / 1e9, "frac": 12 * n / (k_lum * 1e-3) / 1e9 / peak}},
    }
    if not args.no_cpu_baseline:
        host = img[: max(1, h // 8)].cpu().numpy()
        t0 = time.perf_counter()
        tonemap_oracle.tone_map(host, 1.0, None, 1.0)
        dt = time.perf_counter() - t0
        line["cpu_baseline"] = {"value": host.shape[0] * w / dt, "unit": "pixels/s", "cores": 1, "kind": "port",
                                "sample": f"{w}x{host.shape[0]} rows of the same frame through oracle/tonemap_oracle.py ({dt:.1f} s)"}
    emit(line)


class Session:
    """Device, communicator and the buffers shared by every measurement of one bench.py process."""

    def __init__(self, rank, local_rank, world_size):
        import torch

        from pytracer_b200.dist import TorchComm

        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device (there is no CPU path); use --impl reference for the CPU arm")
        torch.cuda.set_device(local_rank)
        self.torch = torch
        self.rank, self.local_rank, self.world_size = rank, local_rank, world_size
        self.comm = TorchComm.from_env("nccl") if world_size > 1 else None
        self.flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")  # > 126 MB of L2
        self.stream = torch.cuda.current_stream().cuda_stream
        self.peaks = {}

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.comm is not None:
            self.comm.barrier()
        self.torch.cuda.synchronize()

    def reduce(self, value, op):
        import torch.distributed as dist

        t = self.torch.tensor([value], dtype=self.torch.float64, device="cuda")
        if self.comm is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX if op == "max" else dist.ReduceOp.SUM)
        return float(t.item())

    def peak(self, kind):
        from pytracer_b200 import device

        if kind not in self.peaks:
            self.peaks[kind] = (device.ffma_peak_tflops() if kind == "fp32" else device.dfma_peak_tflops())[0]
        return self.peaks[kind]


def measure_device(sess, name, steps, warmup, variant="auto", precision="auto", accel="none", partition="rows",
                   exchange="allgather", sample_clocks=False, keep_outputs=False):
    """Device-resident arm: scene and image in HBM, CUDA events on the launch stream around render (+ the
    exchange at N > 1), L2 evicted between timed steps; max over ranks.  `keep_outputs`: the result's
    `outputs` holds what the last timed step computed (the frame, and its counters summed over ranks)."""
    from pytracer_b200 import _abi
    from pytracer_b200.device import DeviceScene
    from pytracer_b200.dist import (PeerImages, RowSlabs, partition_params, render_rows_allgather, render_rows_push)

    torch = sess.torch
    world, camera, kw, desc, flops_per_ray, n_sph = workload(name)
    scene = DeviceScene(world)
    params = build_params(kw, camera, variant=variant, precision=precision, accel=accel)
    H, W = params.height, params.width
    comm, G = sess.comm, sess.world_size
    part_name = "none"
    if G == 1:
        image = torch.empty((H, W, 3), dtype=torch.float32, device="cuda")
        frame = lambda: image  # noqa: E731

        def step():
            scene.render_device(params, image.data_ptr(), 0, sess.stream)
    elif partition == "spp":
        p = partition_params(params, sess.rank, G, "spp")
        part_name = {_abi.RT_PART_SPP: "spp", _abi.RT_PART_ROWS: "rows"}[p.part_mode] + " + all-reduce"
        image = torch.empty((H, W, 3), dtype=torch.float32, device="cuda")
        frame = lambda: image  # noqa: E731

        def step():
            scene.render_device(p, image.data_ptr(), 0, sess.stream)
            comm.all_reduce_sum(image)
    else:
        peers, why = None, ""
        if exchange == "push":
            try:  # every rank must take the same branch: the outcome of the rendezvous is agreed on below
                peers = PeerImages(H, W, comm)
            except Exception as exc:
                why = f"{type(exc).__name__}: {exc}"[:120]
            if sess.reduce(0.0 if peers is not None else 1.0, "max") > 0.0:
                peers, why = None, why or "the symmetric-memory rendezvous failed on another rank"
        if peers is not None:
            part_name = "rows, pixels stored into every rank's image by the kernel over NVLink (symmetric memory) + barrier"
            frame = lambda: peers.image  # noqa: E731

            def step():
                render_rows_push(scene, params, comm, peers, sess.stream)
        else:
            slabs = RowSlabs(H, W, G)
            part_name = "rows + in-place NCCL all-gather of the row slabs" + (f" (peer images unavailable: {why})" if why else "")
            frame = slabs.gathered_image

            def step():
                render_rows_allgather(scene, params, comm, slabs, sess.stream)

    sampler = ClockSampler(sess.local_rank) if (sample_clocks and sess.rank == 0) else None
    for _ in range(max(warmup, 0)):
        step()
        scene.finish(sess.stream)
    sess.barrier()
    if sampler:
        sampler.mark_begin()
    events, rays_rank, kernel_ms, launches, st = [], 0, [], 0, {}
    wall0 = time.perf_counter()
    for _ in range(steps):
        sess.flush.zero_()  # evict L2 between timed iterations (not inside the timed interval)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        step()
        e1.record()
        st = scene.finish(sess.stream)
        events.append((e0, e1))
        rays_rank += st["rays_closest"] + st["rays_shadow"]
        kernel_ms.append(st["kernel_ms"])
        launches += st["n_launches"]
    sess.barrier()
    wall = time.perf_counter() - wall0
    if sampler:
        sampler.mark_end()
    clocks = sampler.stop() if sampler else None
    total_ms = sess.reduce(sum(a.elapsed_time(b) for a, b in events), "max")
    rays = int(round(sess.reduce(float(rays_rank), "sum")))
    outputs = None
    if keep_outputs:
        counters = [sess.reduce(float(st[k]), "sum") for k in ("rays_closest", "rays_shadow", "samples")]
        outputs = {"image": frame().cpu().numpy(), "counters": np.array(counters, dtype=np.float64)}
    scene.close()
    k_ms = statistics.mean(kernel_ms)
    precision_used = {1: "f32", 2: "f64", 3: "hybrid"}.get(st.get("precision_used"), "?")
    return dict(value=rays / (total_ms * 1e-3), ms_per_step=total_ms / max(1, steps), rays_per_step=rays // max(1, steps),
                kernel_ms=k_ms, rays_per_launch_rank=rays_rank / max(1, steps), launches=launches, wall=wall, clocks=clocks,
                partition=part_name, precision_used=precision_used, desc=desc, flops_per_ray=flops_per_ray, n_sph=n_sph,
                H=H, W=W, variant=variant, accel=accel, outputs=outputs)


def measure_e2e(sess, name, iters, warmup, variant="auto", precision="auto", accel="none"):
    """End to end through the public API: a new renderer every step (flatten + scene upload), the launch, the
    image into a page-locked host image (N > 1: every rank's rows into the node's shared one); host clock,
    max over ranks."""
    from pytracer_b200.hdrimage import HdrImage
    from pytracer_b200.imagetracer import CudaImageTracer
    from pytracer_b200.pcg import PCG
    from pytracer_b200.render import CudaRenderer

    torch = sess.torch
    world, camera, kw, _, _, _ = workload(name)
    himg = HdrImage(kw["width"], kw["height"])
    rays, t_sum, scene_bytes, params_bytes = 0, 0.0, 0, 0
    for i in range(warmup + iters):
        renderer = CudaRenderer(world, algorithm=kw["algorithm"], pcg=PCG(45, 54), num_of_rays=kw.get("num_of_rays", 10),
                                max_depth=kw.get("max_depth", 10), russian_roulette_limit=kw.get("rr_limit", 3),
                                variant=variant, precision=precision, accel=accel)
        tracer = CudaImageTracer(himg, camera, samples_per_side=kw["samples_per_side"], pcg=PCG(42, 54))
        sess.barrier()
        t0 = time.perf_counter()
        tracer.fire_all_rays(renderer, comm=sess.comm)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if i >= warmup:
            t_sum += dt
            rays += tracer.last_stats["rays_closest"] + tracer.last_stats["rays_shadow"]
        flat = renderer._scene.flat
        scene_bytes = sum(a.nbytes for a in (flat.shape_kind, flat.shape_material, flat.shape_m, flat.shape_invm, flat.texels)) + \
            sum(len(bytes(s)) for s in (flat.materials, flat.pigments, flat.lights))
        params_bytes = len(bytes(tracer._params(renderer)))
        renderer._scene.close()
    t_max = sess.reduce(t_sum, "max")
    G = sess.world_size
    d2h = kw["height"] * kw["width"] * 12 + 64 if G == 1 else ((kw["height"] + G - 1) // G) * kw["width"] * 12 + 64
    return {"value": rays / t_max, "unit": UNIT, "h2d_bytes_per_step": int(scene_bytes + params_bytes), "d2h_bytes_per_step": int(d2h),
            "bytes_are": "per rank" if G > 1 else "total"}


def roofline_of(sess, m, name):
    """Roofline object of the dominant kernel of a measurement (SURVEY §8d: FP32 FMA pipe; the fp64 kernel
    against the DFMA probe)."""
    torch = sess.torch
    fp64 = m["precision_used"] == "f64"
    peak = sess.peak("fp64" if fp64 else "fp32")
    achieved = m["rays_per_launch_rank"] * m["flops_per_ray"] / (m["kernel_ms"] * 1e-3) / 1e12
    prop = torch.cuda.get_device_properties(sess.local_rank)
    out = {"bound": "fp64" if fp64 else "fp32", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
           "traffic": None, "flops_per_ray": m["flops_per_ray"], "kernel_ms": m["kernel_ms"], "rays_per_launch": m["rays_per_launch_rank"],
           "peak_source": ("DFMA" if fp64 else "FFMA") + " micro-benchmark run in this job (rt_bench_dfma / rt_bench_ffma); MEASURED_PEAKS.json "
           "holds only HBM and bf16-tensor peaks, neither bounds this path",
           "achieved_is": "ALGORITHMIC flops (SURVEY §8d: 54 per ray-sphere test, 12 per ray-plane test, 106 per ray for record and "
           "scatter) over the kernel time, not executed flops"}
    if not fp64:
        out["peak_nominal"] = prop.multi_processor_count * 128 * 2 * 1.965e9 / 1e12
    try:
        prof = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        key = name + ("" if m["accel"] == "none" else "_bvh") + ("_" + m["precision_used"] if name == "c5" else "")
        if SCALE == 1 and sess.world_size == 1:
            out["traffic"] = prof.get(key)
            if prof.get(key + "_issue_slots_busy") is not None:
                out["issue_slots_busy"] = prof.get(key + "_issue_slots_busy")
                out["issue_slots_source"] = "smsp__issue_active.avg.pct_of_peak_sustained_active, profiles/traffic.json (committed ncu capture)"
            for pipe in ("fma", "fp64"):
                if prof.get(f"{key}_{pipe}_pipe_busy") is not None:
                    out[f"{pipe}_pipe_busy"] = prof[f"{key}_{pipe}_pipe_busy"]
                    out["pipe_busy_source"] = f"sm__pipe_{pipe}_cycles_active.avg.pct_of_peak_sustained_active, {prof.get(key + '_source', 'profiles/traffic.json')}"
            if prof.get(key + "_thread_instructions_per_ray") is not None:
                out["thread_instructions_per_ray"] = prof[key + "_thread_instructions_per_ray"]
            if prof.get(key + "_executed_flops_per_ray") is not None:
                ex = prof[key + "_executed_flops_per_ray"]
                out["executed_flops_per_ray"] = ex
                out["executed_frac"] = m["rays_per_launch_rank"] * ex / (m["kernel_ms"] * 1e-3) / 1e12 / peak
                out["executed_source"] = "FFMA/FMUL/FADD (+ 2x packed) thread instructions of the committed ncu capture, profiles/traffic.json"
    except Exception:
        pass
    if m["precision_used"] == "hybrid":
        out["note"] = ("hybrid: the sweep executes 17 packed FMAs per sphere pair and ray (34 flop per ray-sphere test) where the "
                       "straightforward evaluation SURVEY counts needs 27 (54 flop): per-(origin, sphere) terms are precomputed in fp64, so "
                       "`frac` on algorithmic flops can exceed what the FMA pipe executes; decisions and colours are the fp64 kernel's, bit for bit")
        out["sweep_executed_frac"] = m["rays_per_launch_rank"] * 34.0 * m["n_sph"] / (m["kernel_ms"] * 1e-3) / 1e12 / peak
    if m["accel"] != "none":
        out["note"] = ("flops_per_ray is the linear scan's (the reference's algorithm); the hierarchy skips most of that work, "
                       "so `frac` is a speed-up over the roofline of the linear scan, not a utilisation")
    return out


def sub_result(sess, name, steps, warmup, e2e_iters, cpu=True, **opts):
    """One entry of the line's `configs` object."""
    part = opts.pop("partition", "rows")
    exch = opts.pop("exchange", "allgather")
    m = measure_device(sess, name, steps, warmup, partition=part, exchange=exch, **opts)
    out = {"workload": m["desc"], "value": m["value"], "unit": UNIT, "ms_per_step": m["ms_per_step"], "steps": steps, "warmup": warmup,
           "rays_per_step": m["rays_per_step"], "precision": m["precision_used"], "variant": opts.get("variant", "auto"),
           "accel": opts.get("accel", "none"), "partition": m["partition"], "gpu_launches": m["launches"]}
    if e2e_iters > 0:
        out["e2e"] = measure_e2e(sess, name, e2e_iters, 0 if m["ms_per_step"] > 2000 else 1, **opts)
    if sess.rank == 0:
        out["roofline"] = roofline_of(sess, m, name)
        if cpu and sess.world_size == 1:
            v, sample = cpu_baseline_sample(name, 1)
            out["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": 1, "kind": "port", "sample": sample}
    return out


def run_ours(args, rank, local_rank, world_size):
    sess = Session(rank, local_rank, world_size)
    name = args.workload
    m = measure_device(sess, name, args.steps, args.warmup, variant=args.variant, precision=args.precision, accel=args.accel,
                       partition=args.partition, exchange=args.exchange, sample_clocks=True, keep_outputs=bool(args.dump_outputs))
    if args.dump_outputs and rank == 0:
        write_outputs(args.dump_outputs, m["outputs"])
    e2e = measure_e2e(sess, name, args.steps, args.warmup, variant=args.variant, precision=args.precision, accel=args.accel)

    # ---- the other BASELINE configs, measured in the same job (1-2 steps each; `--no-extra` skips them)
    configs = {}
    if name == "c3" and not args.no_extra and SCALE == 1:
        cpu = not args.no_cpu_baseline
        if world_size == 1:
            configs["c4_linear"] = sub_result(sess, "c4", 1, 0, 1, cpu=cpu)
            configs["c4_bvh"] = sub_result(sess, "c4", 2, 1, 1, cpu=False, accel="bvh")
            configs["c5_auto_hybrid"] = sub_result(sess, "c5", 2, 1, 2, cpu=cpu)
            configs["c5_f32"] = sub_result(sess, "c5", 2, 1, 0, cpu=False, precision="f32")
            configs["c5_f64"] = sub_result(sess, "c5", 2, 1, 0, cpu=False, precision="f64")
            configs["c5_bvh_auto_f64"] = sub_result(sess, "c5", 2, 1, 0, cpu=False, accel="bvh")
        else:
            configs["c3_spp_allreduce"] = sub_result(sess, "c3", args.steps, args.warmup, 0, cpu=False, partition="spp")
            other = "allgather" if args.exchange == "push" else "push"
            configs["c3_rows_" + other] = sub_result(sess, "c3", args.steps, args.warmup, 0, cpu=False, exchange=other)
            configs["c4_linear_rows"] = sub_result(sess, "c4", 1, 0, 1, cpu=False)
            configs["c5_auto_hybrid_rows"] = sub_result(sess, "c5", 2, 1, 2, cpu=False)
    if sess.comm is not None:  # unmap / unlink the node's shared host images (rank 0 owns the segments)
        sess.barrier()
        sess.comm.close()
    if rank != 0:
        return
    roofline = roofline_of(sess, m, name)
    line = {
        "metric": METRIC, "value": m["value"], "unit": UNIT, "n_gpus": world_size, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": m["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": {"f32": "f32", "f64": "f64", "hybrid": "f64"}.get(m["precision_used"], "f32"), "data": "synthetic",
        "config": {"workload": m["desc"]},
        "run": {"variant": args.variant, "accel": args.accel, "precision": m["precision_used"], "rays_per_step": m["rays_per_step"],
                "partition": m["partition"], "l2": "256 MB buffer zeroed between timed steps", "wall_s_timed_region": m["wall"]},
        "e2e": e2e, "gpu_launches": m["launches"], "clocks": m["clocks"], "roofline": roofline,
    }
    if configs:
        line["configs"] = configs
    if world_size == 1 and not args.no_cpu_baseline:
        v, sample = cpu_baseline_sample(name, 1)
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": 1, "kind": "port", "sample": sample}
        if not args.no_python_ref:
            line["cpu_baseline"]["python_ref"] = python_reference(all_cores=False)
    emit(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=["c3", "c4", "c5", "tonemap"])
    ap.add_argument("--variant", default="auto", choices=["auto", "mega", "warp"])
    ap.add_argument("--precision", default="auto", choices=["auto", "f32", "f64", "hybrid"])
    ap.add_argument("--partition", default="rows", choices=["rows", "spp"],
                    help="multi-GPU split: interleaved rows (default) or the strata of every pixel + one all-reduce")
    ap.add_argument("--exchange", default="push", choices=["allgather", "push"],
                    help="row split, device-resident arm: stores into every rank's image from inside the kernel over NVLink "
                         "(symmetric memory; the default: 514 vs 510 Grays/s on 8 GPUs), or an in-place NCCL all-gather of the row slabs")
    ap.add_argument("--accel", default="none", choices=["none", "bvh"],
                    help="bvh: sphere hierarchy instead of the reference's loop over all shapes (same image; separately reported mode)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-python-ref", action="store_true", help="skip the ~15 s run of the Python reference (baseline/_ref)")
    ap.add_argument("--no-extra", action="store_true", help="skip the `configs` sub-results (configs 4 and 5)")
    ap.add_argument("--scale", type=int, default=1, help="divide width and height by this (quick experiments only; "
                    "a scaled run is NOT the benchmark and says so in config)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed (the frame "
                    "and its ray counters; tonemap: the 8-bit frame and the luminosity) as DIR/<name>.npy, at most 64 MB: "
                    "the inputs are seeded, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference" and args.workload != "tonemap":
        ap.error("--dump-outputs writes the outputs of the device path (--impl ours)")
    global SCALE
    SCALE = max(1, args.scale)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world_size = int(os.environ.get("WORLD_SIZE", "1"))
    if args.workload == "tonemap":
        run_tonemap(args, rank, local_rank, world_size)
    elif args.impl == "reference":
        run_reference(args, rank, world_size)
    else:
        run_ours(args, rank, local_rank, world_size)
        if world_size > 1:
            import torch.distributed as dist

            if dist.is_initialized():
                dist.destroy_process_group()


if __name__ == "__main__":
    main()
