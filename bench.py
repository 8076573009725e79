#!/usr/bin/env python
"""bench.py -- headline benchmark of the hot path (contract: see the task statement).

Workload (every N): BASELINE.json configs[1] -- 8192x8192 RGBA Q16-HDRI images, each through

    BlurImage(image, 0, sigma=4)             separable Gaussian, 33 + 33 taps (as ConvolveImage with the broadcast taps)
    ResizeImage(blurred, W/2, H/2, Lanczos)  Lanczos 2x

A "step" is one pass of that pipeline over the rank's batch of IMAGES distinct images (weak scaling: every rank owns its
own batch, image -> rank with no pixel traffic; the only collective is one NCCL broadcast of the filter parameters).

metric   = input Mpixels/s, whole job over all ranks.
value    : batch resident in HBM; the step is captured ONCE into a CUDA graph and the timed region replays it K times
           between two events (barrier + synchronize on both sides, max over ranks).  An eager pass with events around
           every operator gives the per-operator / per-rank statistics and the roofline numbers.
e2e      : the plugin path -- the host-buffer C-ABI calls a MagickCore caller makes (mb200_convolve_image +
           mb200_resize_image on ordinary host memory attached to the pixel-cache registry, lazy mode): every image is
           uploaded from host memory (1.07 GB) and its result read back (0.27 GB) inside the timed region.
roofline : dominant kernels = the two 1-D passes of BlurImage; algorithmic bytes per launch = 32 B/pixel x 8192^2
           (SURVEY 8d).  roofline_fp64: the same launches against the measured FP64 FMA issue rate (their real bound).
config.per_config (N = 1): configs[0], [2], [3] and the other operators of DESIGN.md's table, timed in the same run.
config.config5: BASELINE.json configs[4] as written -- 256 x 4096^2 images sharded i mod N (strong scaling).
cpu_baseline / --impl reference: the reference's own CPU implementation (ImageMagick 7.1.1-45 compiled from source into
           oracle/_ref, all host threads; the oracle port when that library is absent) on the SAME 8192^2 images.
"""
from __future__ import annotations

import os as _os

# torchrun exports OMP_NUM_THREADS=1.  Only rank 0 ever runs the CPU arm (OpenMP); libgomp takes the variable when it
# is first loaded (with torch), so rank 0 -- and nobody else -- gets all host cores before anything is imported.
if _os.environ.get("RANK", "0") == "0" and _os.environ.get("OMP_NUM_THREADS", "") in ("", "1"):
    _os.environ["OMP_NUM_THREADS"] = str(_os.cpu_count() or 1)

import argparse
import ctypes as C
import json
import math
import os
import re
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

SIZE = 8192
SIGMA = 4.0
LANCZOS = 22
IMAGES = 32                # images per rank per step (34 GB of pixels per GPU)
METRIC = "Mpixels/s on 8K RGBA Gaussian-blur σ=4 + Lanczos 2×; % HBM roofline"
WORKLOAD = (f"configs[1]: {SIZE}x{SIZE} RGBA Q16-HDRI images, each BlurImage(0,{SIGMA}) (separable Gaussian, 33+33 taps) "
            f"+ ResizeImage({SIZE // 2}x{SIZE // 2}, Lanczos)")


def measured_peak():
    try:
        p = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """ONE `nvidia-smi -lms` for all GPUs of the node, started by rank 0 only (r01 ran one poller per rank)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpus: int, period_ms: int = 100):
        self.gpus, self.period_ms, self.proc, self.lines = gpus, period_ms, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", str(self.period_ms)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._drain, daemon=True).start()
            time.sleep(0.3)
        except Exception:
            self.proc = None
        return self

    def _drain(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line))

    def stop(self):
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()

    def summary(self, t0, t1):
        num = lambda x: float(x) if re.fullmatch(r"[0-9.]+", x) else None
        rows = []
        for t, line in self.lines:
            parts = [p.strip() for p in line.strip().split(",")]
            if len(parts) >= 8 and t0 - 0.05 <= t <= t1 + 0.15 and num(parts[0]) is not None and num(parts[0]) < self.gpus:
                rows.append(parts)
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = [num(r[1]) for r in rows if num(r[1]) is not None]
        pw = [num(r[3]) for r in rows if num(r[3]) is not None]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in rows for n, v in zip(names, r[4:8]) if v.lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_mhz_min": min(sm) if sm else None,
                "sm_max_mhz": num(rows[0][2]), "power_w_max": max(pw) if pw else None, "samples": len(rows),
                "gpus_sampled": self.gpus, "sampler": f"one nvidia-smi -lms {self.period_ms} on rank 0", "reasons": reasons}


# ------------------------------------------------------------------ CPU arms

def cpu_pipeline(steps: int, warmup: int, size: int = 0, dump_dir=None):
    """The reference's CPU implementation (oracle/_ref when present, else the oracle port): blur sigma=4 then Lanczos 2x
    down on one size^2 RGBA image per step, all host threads.  size defaults to the GPU arm's 8192 (the CPU test suite
    shrinks it through MB200_BENCH_CPU_SIZE to stay fast on small machines; the `sample` string always says what ran)."""
    size = size or int(os.environ.get("MB200_BENCH_CPU_SIZE", SIZE))
    cores = os.cpu_count() or 1
    fp = C.POINTER(C.c_float)
    ref_so = ROOT / "oracle" / "_ref" / "libmagickref.so"
    n = size
    rng = np.random.default_rng(42)
    src = np.empty((n, n, 4), np.float32)
    for y0 in range(0, n, 1024):                      # bounded temporaries
        src[y0:y0 + 1024] = rng.random((min(1024, n - y0), n, 4), dtype=np.float32) * np.float32(65535)
    mid = np.empty_like(src)
    out = np.empty((n // 2, n // 2, 4), np.float32)
    P = lambda a: a.ctypes.data_as(fp)
    if ref_so.exists():
        lib, kind, pre = C.CDLL(str(ref_so)), "reference", "ref"
    else:
        so = ROOT / "oracle" / "liboracle.so"
        if not so.exists():
            subprocess.run(["make", "-C", str(ROOT / "oracle"), "port"], check=True, stdout=subprocess.DEVNULL)
        lib, kind, pre = C.CDLL(str(so)), "port", "orc"
    f_blur, f_resize, f_threads = getattr(lib, pre + "_blur"), getattr(lib, pre + "_resize"), getattr(lib, pre + "_set_threads")
    f_blur.argtypes = [fp, fp, C.c_size_t, C.c_size_t, C.c_int, C.c_double, C.c_double]
    f_resize.argtypes = [fp, C.c_size_t, C.c_size_t, C.c_int, fp, C.c_size_t, C.c_size_t, C.c_int]
    f_threads.argtypes = [C.c_int]
    f_threads(cores)
    f_threads(cores)          # the resource limit is clamped to omp_get_max_threads(), which the first call raises

    def step():
        assert f_blur(P(src), P(mid), n, n, 4, 0.0, SIGMA) == 0
        assert f_resize(P(mid), n, n, 4, P(out), n // 2, n // 2, LANCZOS) == 0

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    if dump_dir:
        dump_outputs(dump_dir, out)
    name = "ImageMagick 7.1.1-45 Q16-HDRI OpenMP" if kind == "reference" else "oracle port"
    return {"value": steps * n * n / dt / 1e6, "unit": "Mpixels/s", "cores": cores, "kind": kind,
            "sample": f"{steps} x ({n}x{n} RGBA BlurImage(0,{SIGMA}) + ResizeImage {n // 2}x{n // 2} Lanczos), {name}, "
                      f"{dt:.2f} s"}, dt / steps * 1e3


def run_reference(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return 0
    cpu, ms = cpu_pipeline(max(1, args.steps), max(1, min(args.warmup, 2)), dump_dir=args.dump_outputs)
    line = {"impl": "reference", "metric": METRIC, "value": cpu["value"], "unit": "Mpixels/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "images_per_step": 1,
                       "note": "CPU arm: the unmodified reference on all host threads, pixels resident in host RAM; "
                               "one image per step (a bounded sample of the GPU arm's batch of identical images)"},
            "cpu_baseline": cpu,
            "e2e": {"value": cpu["value"], "unit": "Mpixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------- GPU arm

def med(v):
    return statistics.median(v) if v else None


def stats3(v):
    return {"min": min(v), "median": statistics.median(v), "max": max(v)} if v else None


def gpu_cpu_affinity(index: int):
    """CPU ids of the NUMA node GPU `index` hangs off (nvidia-smi topo -m, 'CPU Affinity' column)."""
    try:
        out = subprocess.run(["nvidia-smi", "topo", "-m"], capture_output=True, text=True, timeout=20).stdout
        out = re.sub(r"\x1b\[[0-9;]*m", "", out)
        header = None
        for line in out.splitlines():
            cells = [c.strip() for c in line.split("\t")]
            if header is None and any(c == "CPU Affinity" for c in cells):
                header = [c for c in cells if c]
                continue
            if header and cells and cells[0] == f"GPU{index}":
                vals = [c for c in cells if c]
                col = header.index("CPU Affinity") + 1          # the row label shifts the columns by one
                spec = vals[col]
                cpus = set()
                for part in spec.split(","):
                    a, _, b = part.partition("-")
                    cpus.update(range(int(a), int(b or a) + 1))
                return sorted(cpus), spec
    except Exception:
        pass
    return None, None


DUMP_ROWS = 512           # rows of a 4096 x 4096 RGBA result kept by --dump-outputs (32 MB)


def dump_outputs(directory, pixels):
    """What the last timed step returned -- the Lanczos result of the step's last image, an (H, W, 4) numpy array or
    tensor -- as DIR/lanczos_rows.npy in float32: a seeded, fixed choice of min(H, DUMP_ROWS) of its rows (the same rows
    in every run), so two builds can be compared output for output.  Written by rank 0 only."""
    rows = np.sort(np.random.default_rng(0).choice(pixels.shape[0], min(pixels.shape[0], DUMP_ROWS), replace=False))
    sample = pixels[rows.tolist()]
    if not isinstance(sample, np.ndarray):
        sample = sample.float().cpu().numpy()
    out = Path(directory)
    out.mkdir(parents=True, exist_ok=True)
    np.save(out / "lanczos_rows.npy", np.ascontiguousarray(sample, np.float32))


def run_gpu(args):
    import torch
    import imagemagick_b200 as im
    from imagemagick_b200 import _lib
    from imagemagick_b200 import dist as mdist

    rank, world, local = mdist.init_process_group()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the GPU arm has no CPU fallback")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    lib = _lib.load()
    W = H = SIZE
    ev = lambda: torch.cuda.Event(enable_timing=True)
    peak, peak_src = measured_peak()

    # the one collective of the data path: rank 0's filter parameters
    job = None
    if rank == 0:
        taps = im.AcquireKernelInfo(f"blur:0x{SIGMA}").arrays()[0][0].ravel()
        job = mdist.FilterJob(0.0, SIGMA, W // 2, H // 2, LANCZOS, taps)
    job = mdist.broadcast_job(job, device=dev)
    blur_kernel = mdist.blur_kernel_from_taps(job.taps)

    gen = torch.Generator(device=dev)
    gen.manual_seed(42 + rank)
    batch = [im.Image(torch.rand((H, W, 4), device=dev, generator=gen) * 65535.0) for _ in range(IMAGES)]

    def one_image(image):
        b = im.ConvolveImage(image, blur_kernel)          # == BlurImage(image, 0, sigma) with the broadcast taps
        return im.ResizeImage(b, job.out_columns, job.out_rows, job.resize_filter)

    def step_eager():
        out = None
        for image in batch:
            out = one_image(image)
        return out

    for _ in range(max(1, args.warmup - 2)):               # also builds the resize tables / fills the pools
        last = step_eager()
    torch.cuda.synchronize()

    # ---- eager pass with events around every operator: per-operator statistics, launch count per step
    launches0 = im.launch_count()
    marks = []
    host_ms = []
    for image in batch:
        e0, e1, e2 = ev(), ev(), ev()
        h0 = time.perf_counter()
        e0.record()
        b = im.ConvolveImage(image, blur_kernel)
        e1.record()
        last = im.ResizeImage(b, job.out_columns, job.out_rows, job.resize_filter)
        e2.record()
        host_ms.append((time.perf_counter() - h0) * 1e3)
        marks.append((e0, e1, e2))
    torch.cuda.synchronize()
    launches_per_step = im.launch_count() - launches0
    blur_ms = [a.elapsed_time(b) for a, b, _ in marks]
    resize_ms = [b.elapsed_time(c) for _, b, c in marks]
    check = last.pixels.reshape(-1)[:64].cpu().numpy()

    # ---- capture the step in a CUDA graph (the inner loop is 4 launches per image: launch-bound work belongs in a graph)
    timing_mode = "cuda graph of one step (batch of %d images), replayed K times" % IMAGES
    graph = None
    try:
        graph = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            step_eager()                                   # warm the side stream's allocator state
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        branches = [torch.cuda.Stream(device=dev) for _ in range(max(0, args.streams - 1))]
        with torch.cuda.graph(graph, stream=side):
            if not branches:
                graph_out = step_eager()
            else:
                # independent images on separate streams: the FP64-bound blur of one image and the HBM-bound resize of
                # another may share the SMs, and a kernel's last partial wave overlaps the next kernel's first
                lanes = [side] + branches
                for b_ in branches:
                    b_.wait_stream(side)
                outs = [None] * len(lanes)
                for k, image in enumerate(batch):
                    lane = k % len(lanes)
                    with torch.cuda.stream(lanes[lane]):
                        outs[lane] = one_image(image)
                for b_ in branches:
                    side.wait_stream(b_)
                graph_out = outs[(len(batch) - 1) % len(lanes)]
        if branches:
            timing_mode = ("cuda graph of one step (batch of %d images on %d image-parallel streams), replayed K times"
                           % (IMAGES, len(branches) + 1))
        graph.replay()
        torch.cuda.synchronize()
        assert np.array_equal(graph_out.pixels.reshape(-1)[:64].cpu().numpy(), check), "graph replay differs"
    except Exception as exc:                               # never hide it: the mode is part of the JSON line
        graph = None
        timing_mode = f"eager launches (graph capture failed: {type(exc).__name__}: {str(exc)[:120]})"
        torch.cuda.synchronize()
    run_step = graph.replay if graph is not None else step_eager

    clocks = ClockSampler(world).start() if rank == 0 else None
    for _ in range(2):
        run_step()
    torch.cuda.synchronize()
    mdist.barrier()
    torch.cuda.synchronize()
    clk_t0 = time.perf_counter()
    t_start, t_end = ev(), ev()
    t_start.record()
    for _ in range(args.steps):
        step_out = run_step()
    t_end.record()
    torch.cuda.synchronize()
    clk_t1 = time.perf_counter()
    mdist.barrier()
    local_ms = t_start.elapsed_time(t_end)
    total_ms = mdist.max_over_ranks(local_ms, device=dev)
    ms_per_step = total_ms / args.steps
    value = world * IMAGES * W * H / ms_per_step / 1e3           # Mpixels/s over all ranks
    per_rank = mdist.gather_over_ranks([local_ms / args.steps, med(blur_ms), min(blur_ms), max(blur_ms), med(resize_ms),
                                        min(resize_ms), max(resize_ms), med(host_ms), max(host_ms)], device=dev)
    clock_summary = clocks.summary(clk_t0, clk_t1) if clocks else None
    if clocks:
        clocks.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, (graph_out if graph is not None else step_out).pixels)

    # ---- roofline inputs: each pass of the blur alone (events around exactly one launch), FP64 issue-rate probe
    row_k, col_k = im.AcquireKernelInfo(f"blur:0x{SIGMA}"), im.AcquireKernelInfo(f"blur:0x{SIGMA}+90")

    def time_op(fn, reps=12, warm=2):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            a, b = ev(), ev()
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        return statistics.median(ts)

    def mma_launches():
        v = C.c_int(0)
        _lib.check(lib.mb200_get_option(b"conv_mma_launches", C.byref(v)))
        return v.value

    n_mma = mma_launches()
    row_ms = time_op(lambda: im.ConvolveImage(batch[0], row_k))
    col_ms = time_op(lambda: im.ConvolveImage(batch[1], col_k))
    blur_on_mma = mma_launches() > n_mma            # which kernels serve the 33-tap passes (conv_mma.cu / conv1d.cu)
    blur_kernels = (("conv_mma_kernel<10,0,0,0,4>", "conv_mma_kernel<10,1,0,0,4>") if blur_on_mma else
                    ("conv_pair_async_kernel<33,2,0,0>", "conv_pair_kernel<33,2,1,0,true>"))
    fma_rate = C.c_double(0.0)
    _lib.check(lib.mb200_probe_fp64_fma_rate(C.byref(fma_rate)))

    # ---- per-config table (N = 1 only: the scaling runs stay short)
    per_config = None
    if world == 1:
        per_config = {}

        def entry(name, ms, npix, alg_bytes, note=None):
            e = {"ms": ms, "mpix_s": npix / ms / 1e3, "alg_bytes": alg_bytes, "hbm_frac": alg_bytes / (ms * 1e-3) / 1e9 / peak}
            if note:
                e["note"] = note
            per_config[name] = e

        px = W * H
        entry("config2_blur_8192_sigma4", med(blur_ms), px, 64 * px, "row + column pass, 32 B/px each")
        entry("config2_blur_row_pass", row_ms, px, 32 * px, blur_kernels[0])
        entry("config2_blur_column_pass", col_ms, px, 32 * px, blur_kernels[1])
        entry("resize_8192_to_4096_lanczos", med(resize_ms), px, 36 * px, "V pass 24 B + H pass 12 B per input px")
        x = batch[2]
        entry("blur_8192_sigma2", time_op(lambda: im.BlurImage(x, 0.0, 2.0)), px, 64 * px, "17 + 17 taps")
        entry("unsharp_8192_sigma4_fused", time_op(lambda: im.UnsharpMaskImage(x, 0.0, 4.0, 1.5, 0.02)), px, 80 * px,
              "blur (64 B/px) + source read in the fused epilogue (16 B/px)")
        entry("gaussian_blur_8192_2d_29x29", time_op(lambda: im.GaussianBlurImage(x, 0.0, 4.0), reps=6), px, 32 * px,
              "rank-1 path: row pass with raw double intermediate + column pass; bytes of a one-pass evaluation")
        k7 = im.AcquireKernelInfo("Disk:3")
        entry("config4_dilate_disk3_8192", time_op(lambda: im.MorphologyImage(x, im.DilateMorphology, 1, k7)), px, 32 * px)
        lab = im.Image(x.pixels.clone())

        def to_lab():
            lab.colorspace = im.sRGBColorspace
            im.TransformImageColorspace(lab, im.LabColorspace)
        entry("config4_srgb_to_lab_8192", time_op(to_lab), px, 32 * px, "in place")

        def lab_dilate():
            lab.colorspace = im.sRGBColorspace
            im.TransformImageColorspace(lab, im.LabColorspace)
            im.MorphologyImage(lab, im.DilateMorphology, 1, k7)
        entry("config4_pipeline_lab_then_dilate", time_op(lab_dilate), px, 64 * px)
        del lab
        small = im.Image(torch.rand((1024, 1024, 4), device=dev, generator=gen) * 65535.0)
        entry("config1_blur_1024_sigma2", time_op(lambda: im.BlurImage(small, 0.0, 2.0), reps=30), 1024 * 1024, 64 * 1024 * 1024,
              "configs[0]'s image on the GPU (16.8 MB: L2 resident)")
        hd = im.Image(torch.rand((1080, 1920, 4), device=dev, generator=gen) * 65535.0)
        entry("sharpen_1920x1080_5x2", time_op(lambda: im.SharpenImage(hd, 5.0, 2.0), reps=30), 1920 * 1080, 32 * 1920 * 1080,
              "the reference's only published -bench workload (www/architecture.html:889: 9.47 Mpix/s on 6 threads); 11x11 2-D kernel")
        del small, hd
        # config 3 needs 4.3 + 2.1 + 1.1 GB next to the resident batch
        big = im.Image(torch.rand((16384, 16384, 4), device=dev, generator=gen) * 65535.0)
        entry("config3_resize_16384_to_8192_lanczos", time_op(lambda: im.ResizeImage(big, 8192, 8192, im.LanczosFilter), reps=8),
              16384 * 16384, 36 * 16384 * 16384, "Mpix/s on input pixels")
        del big
        torch.cuda.empty_cache()

    # ---- end to end through the plugin path (host buffers, C-ABI host entry points) --------------------------------------
    vp = lambda a: C.c_void_p(a.ctypes.data)
    in_bytes, out_bytes = W * H * 16, job.out_columns * job.out_rows * 16
    affinity, affinity_spec = gpu_cpu_affinity(local)

    E2E_THREADS = 2          # application threads calling the plugin path (each gets its own library stream)

    def make_host_buffers(k):
        src = np.empty((H, W, 4), np.float32)                 # the step's inputs live in ordinary host memory
        _lib.check(lib.mb200_download(vp(src), C.c_void_p(batch[k].pixels.data_ptr()), in_bytes, None))
        _lib.check(lib.mb200_synchronize(None))
        return src, np.empty((H, W, 4), np.float32), np.empty((job.out_rows, job.out_columns, 4), np.float32)

    def e2e_image(src, mid, out):
        _lib.check(lib.mb200_cache_host_written(vp(src)))                       # new pixels arrived in the host cache
        _lib.check(lib.mb200_convolve_image(vp(src), vp(mid), W, H, 4, blur_kernel._ptr))
        _lib.check(lib.mb200_resize_image(vp(mid), W, H, 4, vp(out), job.out_columns, job.out_rows, job.resize_filter))
        _lib.check(lib.mb200_cache_sync(vp(out)))                               # the caller reads the result

    def e2e_run(images, attach, nthreads):
        """`images` images through the two host-buffer calls, split over `nthreads` application threads (ctypes releases
        the GIL; every thread owns its source / intermediate / result buffers and gets its own library stream, so one
        thread's upload overlaps the other's kernels and download).  Returns ms per image (wall clock)."""
        sets = [make_host_buffers(k) for k in range(nthreads)]
        flat = [a for st in sets for a in st]
        if attach:
            for a in flat:
                _lib.check(lib.mb200_cache_attach(vp(a), a.nbytes, 1))
            lib.mb200_cache_set_lazy(1)
        errors = []

        def worker(k, n):
            try:
                _lib.check(lib.mb200_set_device(local))           # the current device is a per-thread setting
                for _ in range(n):
                    e2e_image(*sets[k])
                _lib.check(lib.mb200_synchronize(None))
            except Exception as exc:                              # surfaced after the join
                errors.append(exc)

        def run(n_each):
            ts = [threading.Thread(target=worker, args=(k, n_each)) for k in range(nthreads)]
            for t in ts:
                t.start()
            for t in ts:
                t.join()
            if errors:
                raise errors[0]

        try:
            run(2)                                                # warm-up: pins, pools, tables
            mdist.barrier()
            t0 = time.perf_counter()
            run(images // nthreads)
            ms = (time.perf_counter() - t0) * 1e3 / (images // nthreads * nthreads)
            ok = np.array_equal(sets[0][2].reshape(-1)[:64], one_image(batch[0]).pixels.reshape(-1)[:64].cpu().numpy())
        finally:
            if attach:
                lib.mb200_cache_set_lazy(0)
                for a in flat:
                    lib.mb200_cache_detach(vp(a))
        assert ok, "e2e result differs from the device-resident one"
        return ms

    e2e_steps = max(1, min(args.steps, 2))
    e2e_images = IMAGES * e2e_steps
    e2e_single = mdist.max_over_ranks(e2e_run(8, True, 1), device=dev)
    e2e_unbound = mdist.max_over_ranks(e2e_run(e2e_images, True, E2E_THREADS), device=dev)
    e2e_bound = None
    if affinity:
        original_affinity = os.sched_getaffinity(0)
        try:                                                  # experiment: run on the cores of the GPU's NUMA node and
            os.sched_setaffinity(0, affinity)                 # first-touch / pin the host buffers there
            e2e_bound = mdist.max_over_ranks(e2e_run(e2e_images, True, E2E_THREADS), device=dev)
        except Exception:
            e2e_bound = None
        finally:
            os.sched_setaffinity(0, original_affinity)        # the CPU baseline below uses every core
    e2e_ms = min(e2e_unbound, e2e_bound) if e2e_bound else e2e_unbound
    e2e_value = world * W * H / e2e_ms / 1e3
    e2e_modes = {"application_threads": E2E_THREADS, "lazy_attached_ms_per_image": e2e_unbound,
                 "lazy_attached_numa_bound_ms_per_image": e2e_bound, "numa_cpu_affinity": affinity_spec,
                 "lazy_attached_single_thread_ms_per_image": e2e_single}
    # the same two calls on UNATTACHED pageable buffers: every operator stages in and out through the bounce ring
    pageable_ms = e2e_run(4, False, 1) if world == 1 else None
    if rank == 0:
        e2e_modes["eager_pageable_ms_per_image"] = pageable_ms
        harness = ROOT / "oracle" / "_ref" / "shim" / "chain_harness"
        if world == 1 and harness.exists():                   # BlurImage -> ResizeImage through the MagickCore shim itself
            try:
                r = subprocess.run([str(harness), str(SIZE), "3", "0"], capture_output=True, text=True, timeout=600)
                shim = {}
                for line in r.stdout.splitlines():
                    m = re.match(r"(eager, pageable caches|eager, pinned caches|lazy, pinned caches)\s+best\s+([0-9.]+) ms", line)
                    if m:
                        shim[m.group(1)] = float(m.group(2))
                e2e_modes["magickcore_shim_blur_resize_ms"] = shim or r.stdout[-300:]
            except Exception as exc:
                e2e_modes["magickcore_shim_blur_resize_ms"] = f"{type(exc).__name__}"

    # ---- BASELINE.json configs[4] as written: 256 x 4096^2, image i -> rank i mod N (strong scaling) ------------------------
    del batch, last
    if graph is not None:
        del graph, graph_out
    torch.cuda.empty_cache()
    N5, S5 = 256, 4096
    mine = mdist.shard_indices(N5, rank, world)
    job5 = mdist.FilterJob(0.0, SIGMA, S5 // 2, S5 // 2, LANCZOS, job.taps)
    shard = {i: im.Image(torch.rand((S5, S5, 4), device=dev, generator=gen) * 65535.0) for i in mine}
    mdist.run_pipeline(dict(list(shard.items())[:2]), blur_kernel, job5)
    torch.cuda.synchronize()
    a, b = ev(), ev()
    a.record()
    mdist.run_pipeline(shard, blur_kernel, job5)
    b.record()
    torch.cuda.synchronize()
    one_pass = mdist.max_over_ranks(a.elapsed_time(b), device=dev)
    reps = int(min(64, max(4, math.ceil(1000.0 / max(one_pass, 1e-3)))))
    mdist.barrier()
    torch.cuda.synchronize()
    a, b = ev(), ev()
    a.record()
    for _ in range(reps):
        mdist.run_pipeline(shard, blur_kernel, job5)
    b.record()
    torch.cuda.synchronize()
    c5_local = a.elapsed_time(b) / reps
    c5_ms = mdist.max_over_ranks(c5_local, device=dev)
    c5_ranks = mdist.gather_over_ranks([c5_local, float(len(mine))], device=dev)
    config5 = {"workload": f"configs[4]: {N5} x {S5}x{S5} RGBA, BlurImage(0,{SIGMA}) + ResizeImage({S5 // 2}x{S5 // 2}, Lanczos), "
                           f"image i -> rank i mod {world}", "scaling": "strong", "passes_timed": reps,
               "ms_per_batch_pass": c5_ms, "mpix_s": N5 * S5 * S5 / c5_ms / 1e3, "timed_region_s": c5_ms * reps / 1e3,
               "per_rank_ms": [r[0] for r in c5_ranks], "per_rank_images": [int(r[1]) for r in c5_ranks]}
    del shard

    if rank != 0:
        _finish_group()
        return 0

    blur_launch_ms = med(blur_ms) / 2.0                               # two 1-D passes per BlurImage
    alg_bytes = 32.0 * W * H
    achieved = alg_bytes / (blur_launch_ms * 1e-3) / 1e9
    fma_per_launch = 33.0 * 4 * W * H
    cpu, _ = cpu_pipeline(steps=3, warmup=1)                          # ~20-25 s of the reference on all host cores
    keys = ["ms_per_step", "blur_ms_median", "blur_ms_min", "blur_ms_max", "resize_ms_median", "resize_ms_min",
            "resize_ms_max", "host_enqueue_ms_median", "host_enqueue_ms_max"]
    line = {
        "metric": METRIC, "value": value, "unit": "Mpixels/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "images_per_step": IMAGES,
                   "l2": "every image (1.07 GB) is larger than the 126 MB L2 and the batch holds 32 distinct images; no explicit flush",
                   "sharding": "one batch per rank, one NCCL broadcast of the filter taps, no pixel traffic",
                   "timing": timing_mode, "timed_region_s": total_ms / 1e3,
                   "blur_ms": med(blur_ms), "resize_ms": med(resize_ms), "blur_row_pass_ms": row_ms, "blur_column_pass_ms": col_ms,
                   "blur_mpix_s": W * H / med(blur_ms) / 1e3,
                   "resize_hbm_frac": 36.0 * W * H / (med(resize_ms) * 1e-3) / 1e9 / peak,
                   "per_rank": [dict(zip(keys, r)) for r in per_rank],
                   "per_config": per_config if per_config is not None else "measured at N=1 only (BENCH run)",
                   "config5": config5,
                   "e2e_path": "plugin path: mb200_convolve_image + mb200_resize_image on ordinary host buffers (numpy / malloc) "
                               "attached to the pixel-cache registry (cudaHostRegister once), lazy mode: per image one 1.07 GB "
                               "upload, the blurred intermediate stays in HBM, one 0.27 GB download (mb200_cache_sync); "
                               f"{E2E_THREADS} application threads, each on its own library stream",
                   "e2e_modes": e2e_modes, "copy_threads": int(lib.mb200_copy_threads())},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": None,
                     "kernel": f"{blur_kernels[0]} (row pass) / {blur_kernels[1]} (column pass) "
                               "of BlurImage; average of the two launches (median over the batch)",
                     "algorithmic_bytes_per_launch": alg_bytes, "peak_source": peak_src},
        "roofline_fp64": {"bound": "fp64", "achieved": fma_per_launch / (blur_launch_ms * 1e-3) / 1e12,
                          "peak": fma_rate.value / 1e12, "unit": "TFMA/s",
                          "frac": fma_per_launch / (blur_launch_ms * 1e-3) / fma_rate.value,
                          "algorithmic_fma_per_launch": fma_per_launch,
                          "peak_source": "measured in this run (mb200_probe_fp64_fma_rate: 16 DFMA chains/thread, 2048 threads/SM); "
                                         "profiles/r02_pipes.log has the standalone microbenchmark",
                          "note": "33 taps x 4 channels of FP64 FMA per pixel: the pass is FP64-issue bound, not HBM bound "
                                  "(DESIGN.md 5.1)"},
        "cpu_baseline": cpu,
        "e2e": {"value": e2e_value, "unit": "Mpixels/s", "ms_per_image": e2e_ms, "images_timed": e2e_images,
                "h2d_bytes_per_step": IMAGES * in_bytes, "d2h_bytes_per_step": IMAGES * out_bytes},
        "gpu_launches": int(launches_per_step * args.steps),
        "clocks": clock_summary,
    }
    try:
        prof = json.loads((ROOT / "profiles" / "r02_blur_traffic.json").read_text())
        line["roofline"]["traffic"] = prof["mma" if blur_on_mma else "dfma"].get("dram_bytes_per_launch")
    except Exception:
        try:
            prof = json.loads((ROOT / "profiles" / "r01_blur_traffic.json").read_text())
            line["roofline"]["traffic"] = prof["mma" if blur_on_mma else "dfma"].get("dram_bytes_per_launch")
        except Exception:
            pass
    print(json.dumps(line), flush=True)
    _finish_group()
    return 0


def _finish_group():
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            dist.barrier()
            dist.destroy_process_group()
    except Exception:
        pass


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--streams", type=int, default=int(os.environ.get("BENCH_STREAMS", "1")),
                    help="image-parallel branches of the timed step's CUDA graph (independent images on separate streams)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write a fixed sample of what the last step computed to DIR/*.npy "
                         "(rank 0; with --impl reference, the reference's result)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        return run_reference(args)
    return run_gpu(args)


if __name__ == "__main__":
    sys.exit(main())
