#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric: megapixels/s of fused BilateralSliceApply @4K.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A step is ONE pass of the hot path over one batch of synthetic input: one launch of the fused
slice-apply kernel over 8 frames of 3840x2160 (BASELINE.json configs[2]) per GPU, grid
16x16x8x12, has_offset.  Inputs are device-resident before the timed region; 1.86 GB are
touched per step, far more than the 126 MB L2, so no flush is needed between iterations.
Multi-GPU: the batch shards over ranks with no data-path collective (weak scaling: 8 frames
per GPU); timing is CUDA events on the launch stream, max over ranks.

Rank 0 prints ONE JSON line (keys: see the task contract).  `--impl reference` times the
reference's own CPU loops (oracle/_ref: hdrnet/ops/bilateral_slice_apply.cc compiled
unmodified; falls back to the C restatement) on the host cores.

`--dump-outputs DIR` writes, after the timed steps, a fixed seeded sample of what the last timed
step returned (see dump_outputs): the inputs are seeded too, so two builds can be compared value
for value.  The bench writes nothing into the source tree, which may be read-only.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # no __pycache__ written into the tree by the imports below

METRIC = "megapixels/s BilateralSliceApply @4K"
UNIT = "MP/s"
H4K, W4K, B_PER_GPU = 2160, 3840, 8
GH, GW, GD, N_IN, N_OUT = 16, 16, 8, 3, 3
GC = N_OUT * (N_IN + 1)
BYTES_PER_PX = 4 * (N_IN + 1 + N_OUT)  # 28 B: input 12 + guide 4 + output 12 (SURVEY 8d)
WORKLOAD = (f"4K ({W4K}x{H4K}) batch={B_PER_GPU} per GPU, fused slice-apply, "
            f"grid {GH}x{GW}x{GD}x{GC}, has_offset, f32")


KERNEL_TEXT = {
    7: "tex_async (AUTO with workspace): slice_apply_rows_async_kernel<5 texture chunks, per-quad indices, "
       "math warps + issuer warp + slab warp> -- 384 threads: the slab warp blends every row's slab inside "
       "the kernel (no pre-pass launch); 352 / 512 threads: yblend_rows_kernel pre-pass + row kernel, both "
       "inside every timed step",
    4: "tex (AUTO with workspace): yblend_rows_kernel pre-pass + "
       "slice_apply_rows_tma_kernel<GuideFromInput,4,2,512,f32,f32>, both inside every timed step",
    2: "tma: slice_apply_rows_tma_kernel (all-LSU form)",
    1: "generic: one thread per pixel",
}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic_per_launch():
    """DRAM bytes per launch of the dominant kernel from the committed ncu capture, or None."""
    path = os.path.join(ROOT, "profiles", "slice_apply_traffic.json")
    try:
        with open(path) as f:
            return json.load(f).get("dram_bytes_per_launch")
    except Exception:
        return None


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons through NVML while the timed region runs."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown",
               0x4: "sw_power_cap", 0x80: "hw_power_brake", 0x2: "applications_clocks_setting"}

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.samples = []
        self.stop_flag = threading.Event()
        self.window = [None, None]
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.max_mhz = None

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        while not self.stop_flag.is_set():
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    reasons = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((time.perf_counter(), mhz, reasons))
            except Exception:
                pass
            time.sleep(0.001)

    def summary(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        t0, t1 = self.window
        inside = [s for s in self.samples if t0 is not None and t0 <= s[0] <= t1]
        # too short a region for three samples: take everything up to its end (warm-up included),
        # never what ran AFTER it (the sampler of the headline is stopped right behind the region)
        use = inside if len(inside) >= 3 else [s for s in self.samples if t1 is None or s[0] <= t1] or self.samples
        mask = 0
        for s in use:
            mask |= s[2]
        return {"sm_mhz": float(np.median([s[1] for s in use])), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(n for b, n in self.REASONS.items() if mask & b),
                "samples": len(use),
                "window": "timed region" if use is inside else "warm-up + timed region (timed region too short)"}


# ------------------------------------------------------------------------------------------
# CPU arm (reference's own loops on the host cores)
# ------------------------------------------------------------------------------------------
def cpu_checker():
    # torchrun exports OMP_NUM_THREADS=1 to every rank; the CPU arm is meant to use all the
    # host threads it can, so undo that before libgomp is initialised by the oracle library.
    if os.environ.get("OMP_NUM_THREADS") in (None, "1"):
        os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)
    import oracle
    return oracle.best()       # the checkers __graft_entry__.build() compiled; nothing is built here


def cpu_inputs(frames: int, rows: int, seed: int = 1234):
    rng = np.random.RandomState(seed)
    grid = rng.rand(frames, GH, GW, GD, GC).astype(np.float32)
    guide = rng.rand(frames, rows, W4K).astype(np.float32)
    inp = rng.rand(frames, rows, W4K, N_IN).astype(np.float32)
    return grid, guide, inp


def cpu_rate(lib, frames: int, rows: int) -> float:
    grid, guide, inp = cpu_inputs(frames, rows)
    t = time.perf_counter()
    lib.bilateral_slice_apply(grid, guide, inp, True)
    dt = time.perf_counter() - t
    return frames * rows * W4K / dt / 1e6


def pick_frames(lib, cores: int):
    """How many frames to run at once.  The reference loops are serial per frame, so the frame count
    IS the thread count.  One frame per hardware thread is not always the fastest (SMT siblings share
    a core and the loops are memory-heavy: measured 15.5 MP/s with 128 frames against 25.1 with 64 on a
    128-thread host): time a short sample with one frame per thread and one per two, keep the faster.
    Returns (frames, MP/s of the sample)."""
    best = None
    for frames in sorted({max(1, min(cores, 256)), max(1, min(cores, 256) // 2)}, reverse=True):
        cpu_rate(lib, frames, 16)                 # first touch / thread start-up
        rate = cpu_rate(lib, frames, 64)
        if best is None or rate > best[1]:
            best = (frames, rate)
    return best


def cpu_baseline(target_seconds: float = 15.0):
    """Bounded sample of the same workload on the host cores (reported-only baseline)."""
    lib = cpu_checker()
    cores = lib.num_threads()
    frames, guess = pick_frames(lib, cores)  # calibration, ~1 s
    rows = int(min(H4K, 64 * H4K // frames, max(64, guess * 1e6 * target_seconds / (frames * W4K))))  # <= 15 GB of host arrays
    grid, guide, inp = cpu_inputs(frames, rows)
    t = time.perf_counter()
    lib.bilateral_slice_apply(grid, guide, inp, True)
    dt = time.perf_counter() - t
    return {"value": round(frames * rows * W4K / dt / 1e6, 3), "unit": UNIT,
            "cores": min(cores, frames) if lib.kind == "reference" else cores,
            "kind": lib.kind,
            "sample": f"{frames} frames of {W4K}x{rows} (rows of 4K frames, grid {GH}x{GW}x{GD}), "
                      f"{dt:.1f} s, " + ("reference .cc loops, one thread per frame"
                                         if lib.kind == "reference" else "C restatement, OpenMP over rows")}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    lib = cpu_checker()
    cores = lib.num_threads()
    frames, guess = pick_frames(lib, cores)
    budget = 120.0 / max(1, args.steps + args.warmup)  # whole run within a few minutes
    rows = int(min(H4K, 64 * H4K // frames, max(16, guess * 1e6 * budget / (frames * W4K))))  # <= 15 GB of host arrays
    grid, guide, inp = cpu_inputs(frames, rows)
    for _ in range(args.warmup):
        lib.bilateral_slice_apply(grid, guide, inp, True)
    t = time.perf_counter()
    for _ in range(args.steps):
        lib.bilateral_slice_apply(grid, guide, inp, True)
    dt = time.perf_counter() - t
    value = args.steps * frames * rows * W4K / dt / 1e6
    used = min(cores, frames) if lib.kind == "reference" else cores
    sample = (f"per step: {frames} frames of {W4K}x{rows} px rows of the 4K workload "
              f"(bounded sample), {used} host threads")
    line = {"impl": "reference", "metric": METRIC, "value": round(value, 3), "unit": UNIT,
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(dt / args.steps * 1e3, 3), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "sample": sample,
                       "path": "hdrnet/ops/bilateral_slice_apply.cc:24-82 compiled unmodified "
                               "(oracle/_ref)" if lib.kind == "reference"
                               else "oracle/hdrnet_oracle.c restatement"},
            "cpu_baseline": {"value": round(value, 3), "unit": UNIT, "cores": used,
                             "kind": lib.kind, "sample": sample},
            "e2e": {"value": round(value, 3), "unit": UNIT, "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)
    return 0



# ------------------------------------------------------------------------------------------
# Extra records of the GPU arm (BASELINE.json configs 2, 4, 5, the model path, a sustained run).
# The headline `value` above them is untouched; these ride along in the same JSON line.
# ------------------------------------------------------------------------------------------
def _time_ms(torch, stream, fn, iters, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    for _ in range(iters):
        fn()
    b.record(stream)
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def _op_case(torch, lib, _lib, dev, stream, B, H, W, gh, gw, gd, iters, peak, smooth_guide=False):
    """Device-resident op-API call (guide as an input, f32) through the C-ABI with a lent workspace.
    smooth_guide: a low-frequency guide plus 1 % noise (a natural image's luminance varies slowly:
    neighbouring pixels share a depth cell) instead of the headline's uniformly random one."""
    gen = torch.Generator(device=dev).manual_seed(7)
    grid = torch.rand(B, gh, gw, gd, GC, device=dev, generator=gen)
    guide = torch.rand(B, H, W, device=dev, generator=gen)
    if smooth_guide:
        yy = torch.linspace(0, 1, H, device=dev)[None, :, None]
        xx = torch.linspace(0, 1, W, device=dev)[None, None, :]
        bb = torch.arange(B, device=dev, dtype=torch.float32)[:, None, None] / max(B, 1)
        guide = (0.5 + 0.45 * torch.sin(6.2831853 * (3 * xx + 2 * yy + bb)) + 0.01 * (guide - 0.5)).clamp_(0, 1)
    inp = torch.rand(B, H, W, N_IN, device=dev, generator=gen)
    out = torch.empty(B, H, W, N_OUT, device=dev)
    nws = int(lib.hdrnet_slice_apply_workspace_bytes(B, H, gw, gd))
    ws = torch.empty(max(nws, 16) // 4, dtype=torch.float32, device=dev)

    def step():
        rc = lib.hdrnet_slice_apply_f32_ws(grid.data_ptr(), guide.data_ptr(), inp.data_ptr(), out.data_ptr(),
                                           B, H, W, gh, gw, gd, N_IN, N_OUT, 1, _lib.VARIANT_AUTO,
                                           ws.data_ptr(), nws, stream.cuda_stream)
        if rc != 0:
            raise RuntimeError(_lib.error_string(rc))
    ms = _time_ms(torch, stream, step, iters)
    v = ctypes.c_int()
    lib.hdrnet_slice_apply_plan_ws(B, H, W, gh, gw, gd, N_IN, N_OUT, 1, 1, ctypes.byref(v), None, None, None)
    nbytes = B * H * W * BYTES_PER_PX + grid.numel() * 4
    return {"ms": round(ms, 5), "mp_s": round(B * H * W / ms / 1e3, 1), "gb_s": round(nbytes / ms / 1e6, 1),
            "frac": round(nbytes / ms / 1e6 / peak, 4), "variant": v.value}


def extra_records(torch, dist, lib, _lib, dev, stream, world, rank, peak, args):
    """Everything is timed with CUDA events on the launch stream; multi-rank numbers take the max
    over ranks.  Synthetic inputs, seeded synthetic weights (no pretrained model in the tree)."""
    from hdrnet_b200 import models
    ex = {}

    def agg(ms):   # slowest rank
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- model path at the headline shape: guide computed in the slice-apply kernel (24 B/px) ----
    gen = torch.Generator(device=dev).manual_seed(11 + rank)
    im_f = torch.rand(B_PER_GPU, H4K, W4K, 3, device=dev, generator=gen)
    model = {}
    for name in ("HDRNetCurves", "HDRNetPointwiseNNGuide"):
        p = dict(models.DEFAULT_PARAMS, model_name=name)
        p["weights"] = models.init_weights(p, seed=0, model_name=name)
        cls = getattr(models, name)
        low = models.lowres_from_image(im_f, 256)
        coeffs = cls._coefficients(low, p)
        ms_full = agg(_time_ms(torch, stream, lambda: cls._fullres(coeffs, im_f, p, torch.float32), 20))
        ms_cnn = agg(_time_ms(torch, stream, lambda: cls._coefficients(low, p), 10))
        nbytes = B_PER_GPU * H4K * W4K * 24
        model[name] = {"ms_guide_plus_slice_apply": round(ms_full, 5), "ms_coefficient_cnn_batch8": round(ms_cnn, 5),
                       "bytes_per_px": 24, "gb_s": round(nbytes / ms_full / 1e6, 1),
                       "frac": round(nbytes / ms_full / 1e6 / peak, 4),
                       "mp_s_all_gpus": round(world * B_PER_GPU * H4K * W4K / (ms_full + ms_cnn) / 1e3, 1)}
    ex["model_4k_x8"] = model
    del im_f

    # ---- config 4: HDR+ 16-bit linear 12 MP, 8 frames per GPU (64 over 8), uint16 in -> uint8 out ----
    H12, W12 = 3024, 4032
    im16 = torch.randint(0, 32768, (B_PER_GPU, H12, W12, 3), device=dev, generator=gen, dtype=torch.int32).to(torch.uint16)
    p = dict(models.DEFAULT_PARAMS, model_name="HDRNetCurves")
    p["weights"] = models.init_weights(p, seed=0, model_name="HDRNetCurves")
    cls = models.HDRNetCurves
    low = models.lowres_from_image(im16, 256)
    coeffs = cls._coefficients(low, p)
    ms_k = agg(_time_ms(torch, stream, lambda: cls._fullres(coeffs, im16, p, torch.uint8), 10))
    ms_all = agg(_time_ms(torch, stream, lambda: cls.inference_image(im16, p), 5))
    px = B_PER_GPU * H12 * W12
    ex["C4_12mp_u16_x8_per_gpu"] = {
        "frames_all_gpus": B_PER_GPU * world, "ms_fullres_kernel": round(ms_k, 5),
        "ms_inference_image": round(ms_all, 5), "bytes_per_px": 9,
        "gb_s": round(px * 9 / ms_k / 1e6, 1), "frac": round(px * 9 / ms_k / 1e6 / peak, 4),
        "mp_s_all_gpus": round(world * px / ms_all / 1e3, 1),
        "path": "models.HDRNetCurves.inference_image: lowres_nearest_kernel + coefficient CNN + fused-guide "
                "slice-apply reading uint16, writing uint8 (hdrnet/bin/run.py:145-169, :95)"}
    del im16

    if rank == 0:   # single-GPU records
        # ---- config 2: one 1080p frame (op and model) ----
        ex["C2_1080p_x1_op"] = _op_case(torch, lib, _lib, dev, stream, 1, 1080, 1920, GH, GW, GD, 200, peak)
        im = torch.rand(1, 1080, 1920, 3, device=dev, generator=gen)
        low1 = models.lowres_from_image(im, 256)
        ms_m = _time_ms(torch, stream, lambda: cls.inference(low1, im, p), 50)
        ms_c = _time_ms(torch, stream, lambda: cls._coefficients(low1, p), 50)
        ex["C2_1080p_x1_model"] = {"ms_inference": round(ms_m, 5), "ms_coefficient_cnn": round(ms_c, 5),
                                   "mp_s": round(1080 * 1920 / ms_m / 1e3, 1),
                                   "weights": "seeded synthetic (local_laplacian_sample is not in the tree)"}
        # ---- config 5: grid sweep at 4K x 8 ----
        sweep = {}
        for gh, gw, gd in ((8, 8, 4), (16, 16, 4), (16, 16, 8), (32, 32, 8), (32, 32, 16)):
            sweep[f"{gh}x{gw}x{gd}"] = _op_case(torch, lib, _lib, dev, stream, B_PER_GPU, H4K, W4K, gh, gw, gd, 30, peak)
        ex["C5_grid_sweep_4k_x8"] = sweep
        # the same shapes with a natural-image-like guide (the random one is the worst case for the
        # shared-memory bank groups at 16 depth cells, DESIGN.md section 4)
        ex["C5_smooth_guide_4k_x8"] = {
            f"{gh}x{gw}x{gd}": _op_case(torch, lib, _lib, dev, stream, B_PER_GPU, H4K, W4K, gh, gw, gd, 30, peak,
                                        smooth_guide=True)
            for gh, gw, gd in ((16, 16, 8), (32, 32, 16))}
    return ex

# ------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------
DUMP_PIXELS = 1 << 20   # 12 MB of float32 RGB out of the 796 MB output of one step


def dump_outputs(torch, out, directory, name, pixels):
    """Writes `pixels` output pixels of the last timed step to directory/name.npy, float32 [pixels, N_OUT].
    The pixels are a seeded sample (numpy default_rng(0), sorted flat pixel indices into out[B,H,W]),
    the same on every run, so two builds' files compare element for element."""
    flat = out.view(-1, out.shape[-1])
    idx = np.sort(np.random.default_rng(0).choice(flat.shape[0], size=min(pixels, flat.shape[0]), replace=False))
    sample = flat.index_select(0, torch.from_numpy(idx).to(out.device)).cpu().numpy()
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, name + ".npy"), sample.astype(np.float32))


def run_b200_arm(args):
    import torch
    import torch.distributed as dist

    from hdrnet_b200 import _lib, hdrnet_ops

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; hdrnet_b200 has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # Bind this rank to the CPUs (and so the memory) of its GPU's NUMA node BEFORE any pinned
    # allocation: the end-to-end leg moves 1.9 GB per step and rank through host memory.
    from hdrnet_b200 import parallel
    numa_cpus = parallel.bind_to_gpu_numa(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if args.gpus != world and rank == 0:
        print(f"bench.py: --gpus {args.gpus} but WORLD_SIZE={world}; reporting n_gpus={world}",
              file=sys.stderr)

    B, H, W = B_PER_GPU, H4K, W4K
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    grid = torch.rand(B, GH, GW, GD, GC, device=dev, generator=gen)
    guide = torch.rand(B, H, W, device=dev, generator=gen)
    inp = torch.rand(B, H, W, N_IN, device=dev, generator=gen)
    out = torch.empty(B, H, W, N_OUT, device=dev)
    npix = B * H * W
    algo_bytes = npix * BYTES_PER_PX + grid.numel() * 4

    lib = _lib.load()
    stream = torch.cuda.current_stream(dev)
    # Workspace lent to the library (it never allocates): y-pre-blended slab rows for the
    # texture-assisted kernel, B*H*gw*gd*48 bytes (106 MB here).  Allocated once, outside the
    # timed region, exactly as hdrnet_ops.bilateral_slice_apply does for CUDA tensors.
    ws_bytes = int(lib.hdrnet_slice_apply_workspace_bytes(B, H, GW, GD))
    ws = torch.empty(ws_bytes // 4, dtype=torch.float32, device=dev)

    def step():
        rc = lib.hdrnet_slice_apply_f32_ws(grid.data_ptr(), guide.data_ptr(), inp.data_ptr(),
                                           out.data_ptr(), B, H, W, GH, GW, GD, N_IN, N_OUT, 1,
                                           _lib.VARIANT_AUTO, ws.data_ptr(), ws_bytes,
                                           stream.cuda_stream)
        if rc != 0:
            raise RuntimeError(_lib.error_string(rc))

    def barrier():
        if world > 1:
            dist.barrier()

    sampler = ClockSampler(local_rank)
    sampler.start()

    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    barrier()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.window[0] = time.perf_counter()
    ev0.record(stream)
    for _ in range(args.steps):
        step()
    ev1.record(stream)
    torch.cuda.synchronize()
    sampler.window[1] = time.perf_counter()
    sampler.stop_flag.set()     # the later legs (end to end, extras, sustained) are not the headline's clocks
    sampler.join(timeout=2)
    barrier()
    elapsed_ms = ev0.elapsed_time(ev1)
    t = torch.tensor([elapsed_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_max_ms = float(t.item())
    own_launch_ms = elapsed_ms / args.steps
    if args.dump_outputs:       # before any later leg runs the step again
        dump_outputs(torch, out, args.dump_outputs, "out" if world == 1 else f"out_rank{rank}",
                     DUMP_PIXELS // world)

    # ---- end to end: public API, pinned HOST buffers, H2D + kernel + D2H inside the timing --
    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    h_grid = grid.cpu().pin_memory()
    h_guide = guide.cpu().pin_memory()
    h_inp = inp.cpu().pin_memory()
    h_out = torch.empty(B, H, W, N_OUT).pin_memory()
    hdrnet_ops.bilateral_slice_apply(h_grid, h_guide, h_inp, True, out=h_out)  # warm (allocs)
    torch.cuda.synchronize()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        hdrnet_ops.bilateral_slice_apply(h_grid, h_guide, h_inp, True, out=h_out)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_s = float(te.item())
    e2e_ok = bool(torch.equal(h_out, out.cpu()))
    e2e_h2d = int((h_grid.numel() + h_guide.numel() + h_inp.numel()) * 4)
    e2e_d2h = int(h_out.numel() * 4)
    del h_grid, h_guide, h_inp, h_out

    # ---- end to end, integer image path: what hdrnet/bin/run.py moves per frame -- decoded uint8
    # pixels in, uint8 prediction out (3 + 3 B/px over PCIe), whole model (CNN + guide + slice-apply)
    from hdrnet_b200 import models
    mp = dict(models.DEFAULT_PARAMS, model_name="HDRNetCurves")
    mp["weights"] = models.init_weights(mp, seed=0, model_name="HDRNetCurves")
    h_im8 = torch.randint(0, 256, (B, H, W, 3), dtype=torch.uint8).pin_memory()
    h_out8 = torch.empty(B, H, W, 3, dtype=torch.uint8).pin_memory()

    def e2e_u8_step():   # frame-pipelined: upload i + 1 | model i | download i - 1 (host_pipeline.py)
        models.HDRNetCurves.inference_image_host(h_im8, mp, out=h_out8, device=dev)
    e2e_u8_step()
    torch.cuda.synchronize()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_u8_step()
    torch.cuda.synchronize()
    e2e8_s = time.perf_counter() - t0
    te = torch.tensor([e2e8_s], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e8_s = float(te.item())
    del h_im8, h_out8

    peak, peak_src = measured_peaks()
    extra = {} if args.no_extra else extra_records(torch, dist, lib, _lib, dev, stream, world, rank, peak, args)

    # ---- sustained: the same step for >= 2 s, LAST (the boxes power-cap under sustained load and
    # take a second to recover: anything timed right after it would carry the capped clock) ----
    sus_steps = max(args.steps, int(2200.0 / max(own_launch_ms, 1e-3)))
    sus = ClockSampler(local_rank)
    sus.start()
    torch.cuda.synchronize()
    barrier()
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sus.window[0] = time.perf_counter()
    s0.record(stream)
    for _ in range(sus_steps):
        step()
    s1.record(stream)
    torch.cuda.synchronize()
    sus.window[1] = time.perf_counter()
    sus.stop_flag.set()
    sus.join(timeout=2)
    ts = torch.tensor([s0.elapsed_time(s1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ts, op=dist.ReduceOp.MAX)
    sus_ms = float(ts.item()) / sus_steps

    if rank == 0:
        achieved = algo_bytes / (own_launch_ms * 1e-3) / 1e9
        variant, ctas, threads, smem = (ctypes.c_int() for _ in range(4))
        lib.hdrnet_slice_apply_plan_ws(B, H, W, GH, GW, GD, N_IN, N_OUT, 1, 1, ctypes.byref(variant),
                                       ctypes.byref(ctas), ctypes.byref(threads), ctypes.byref(smem))
        line = {
            "metric": METRIC,
            "value": round(world * npix * args.steps / (elapsed_max_ms * 1e-3) / 1e6, 1),
            "unit": UNIT,
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": round(elapsed_max_ms / args.steps, 5),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "frames_per_gpu": B, "global_frames": B * world,
                       "parallelism": f"batch-shard x{world}, no data-path collective",
                       "l2": "1.86 GB touched per step >> 126 MB L2: no flush between iterations",
                       "kernel": {"variant": KERNEL_TEXT.get(variant.value, f"variant {variant.value}"),
                                  "ctas": ctas.value, "threads": threads.value,
                                  "dyn_smem_bytes": smem.value, "workspace_bytes": ws_bytes}},
            "roofline": {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                         "frac": round(achieved / peak, 4), "traffic": ncu_traffic_per_launch(),
                         "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": algo_bytes,
                         "launch_ms": round(own_launch_ms, 5),
                         "note": "duration = the whole step the caller pays for (every launch of the call)"},
            "e2e": {"value": round(world * npix * e2e_steps / e2e_s / 1e6, 1), "unit": UNIT,
                    "h2d_bytes_per_step": e2e_h2d, "d2h_bytes_per_step": e2e_d2h, "steps": e2e_steps,
                    "ms_per_step": round(e2e_s / e2e_steps * 1e3, 3),
                    "path": "hdrnet_ops.bilateral_slice_apply on pinned CPU tensors -> "
                            "hdrnet_slice_apply_host_f32 (row-band H2D/kernel/D2H pipeline)",
                    "matches_device_result": e2e_ok,
                    # what bounds this leg at N > 1: every byte crosses host DRAM and the root complexes
                    "host_traffic_gb_s_all_gpus": round(world * (e2e_h2d + e2e_d2h) * e2e_steps / e2e_s / 1e9, 1),
                    "u8_image_path": {
                        "value": round(world * npix * e2e_steps / e2e8_s / 1e6, 1), "unit": UNIT,
                        "h2d_bytes_per_step": int(npix * 3), "d2h_bytes_per_step": int(npix * 3),
                        "ms_per_step": round(e2e8_s / e2e_steps * 1e3, 3),
                        "path": "pinned uint8 frames -> models.HDRNetCurves.inference_image_host: per frame upload | "
                                "inference_image (lowres gather + coefficient CNN chain + fused-guide slice-apply, "
                                "uint8 in / out) | download on three streams -> pinned uint8"},
                    "numa_cpus_bound": len(numa_cpus)},
            "gpu_launches": (1 if threads.value == 384 else 2) * args.steps * world,
            "clocks": sampler.summary(),
            "sustained": {"steps": sus_steps, "ms_per_step": round(sus_ms, 5),
                          "value": round(world * npix / sus_ms / 1e3, 1), "unit": UNIT,
                          "frac": round(algo_bytes / sus_ms / 1e6 / peak, 4), "clocks": sus.summary()},
            "extra": extra,
        }
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline()
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra records (configs 2, 4, 5, model path)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write a seeded sample of the last step's output to DIR/out.npy "
                         "(DIR/out_rank<r>.npy per rank when several GPUs run)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the GPU path's output; --impl reference has none")
    if args.impl == "reference":
        return run_reference_arm(args)
    return run_b200_arm(args)


if __name__ == "__main__":
    sys.exit(main())
