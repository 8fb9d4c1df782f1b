#!/usr/bin/env python
"""Headline benchmark: movies/s for a 40x4096x4096 fp32 movie through estimate + correct.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

One "step" = one movie through ``motion_correct`` (whole-frame XC -> patch XC on the rigidly pre-shifted windows ->
spline optimiser -> fused warp-and-sum).  At N > 1 (torchrun, one rank per GPU) every
rank aligns its own movie (independent movies, no data-path collective: weak scaling) and the value
is total movies / max-over-ranks device time.  Prints ONE JSON line (rank 0).

``--dump-outputs DIR`` writes what the last timed step returned (rank 0) as ``DIR/<name>.npy``, float32, at most
DUMP_BYTES in all.  Inputs and the optimiser's mini-batch order are seeded, so two builds run with the same arguments
can be compared output for output.  Two runs of one build still differ a little: the optimiser accumulates in float
atomics, so its field varies by about 4e-7 Angstrom, and next to the frame edge the sum is not continuous in the field
(adding 1e-6 Angstrom to the field moved one edge pixel of the sum by 2.4; measured on a B200, 1000 W power limit).

``--impl reference`` times the CPU oracle (restatement of the reference's PyTorch path; the
reference itself cannot be installed offline, see DESIGN.md) on a bounded sample of the workload.
"""

from __future__ import annotations

import argparse
import json
import os
import random
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

WORKLOADS = {
    # BASELINE.json configs[1]: K3-like 40-frame 4096^2 movie, global + (3,5,5) spline local motion
    "c2": dict(t=40, h=4096, w=4096, pixel_spacing=0.83, patch=1024, resolution=(3, 5, 5)),
    # reduced shapes for quick functional runs (NOT the headline; selected only with --workload)
    "c1": dict(t=10, h=512, w=512, pixel_spacing=1.0, patch=128, resolution=(3, 5, 5)),
    "mid": dict(t=16, h=2048, w=2048, pixel_spacing=0.83, patch=512, resolution=(3, 5, 5)),
    # BASELINE.json configs[3]: super-resolution 40 x 8192^2 movie, ONE movie split by frames over the ranks (--gpus N > 1)
    "c4": dict(t=40, h=8192, w=8192, pixel_spacing=0.415, patch=1024, resolution=(3, 5, 5)),
}


def workload_text(name, cfg, iterations):
    """The workload both arms (ours and --impl reference) name in `config.workload`."""
    return (f"{name}: {cfg['t']}x{cfg['h']}x{cfg['w']} fp32 movie, whole-frame XC + patch XC ({cfg['patch']} px, 50% overlap) on the "
            f"rigidly pre-corrected movie + {iterations}-iteration {cfg['resolution']} spline optimiser + warp-and-sum")


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--iterations", type=int, default=int(os.environ.get("TMC_BENCH_ITERATIONS", "-1")),
                    help="spline-optimiser iterations per movie (-1: default of the build)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-aten-baseline", action="store_true")
    ap.add_argument("--no-frame-split", action="store_true", help="skip the frame-split (one movie over N GPUs) sub-record at N > 1")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_BYTES = 64_000_000  # on disk, all files of --dump-outputs together
NPY_HEADER = 4096  # more than any .npy header takes


def dump_outputs(out_dir, arrays):
    """Writes every array of ``arrays`` (name -> tensor, in order) as ``out_dir/<name>.npy`` in float32.  One that does
    not fit what is left of DUMP_BYTES is replaced by a fixed, seeded sample of its elements (flattened, in index
    order): the same positions on every run with the same arguments."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    left = DUMP_BYTES
    for name, a in arrays.items():
        a = a.detach().float().cpu().numpy()
        if a.nbytes + NPY_HEADER > left:
            keep = torch.randperm(a.size, generator=torch.Generator().manual_seed(0))[: (left - NPY_HEADER) // a.itemsize]
            a = a.reshape(-1)[keep.sort().values.numpy()]
        path = os.path.join(out_dir, name + ".npy")
        np.save(path, a)
        left -= os.path.getsize(path)


# --------------------------------------------------------------------------------------------
# synthetic data
# --------------------------------------------------------------------------------------------


def synthetic_movie_gpu(t, h, w, seed, device):
    """Band-limited random specimen, integer global drift (<= +-6 px), unit Gaussian noise."""
    g = torch.Generator(device=device).manual_seed(seed)
    pad = 16
    H, W = h + 2 * pad, w + 2 * pad
    white = torch.randn((H, W), generator=g, device=device)
    fy = torch.fft.fftfreq(H, device=device)[:, None]
    fx = torch.fft.rfftfreq(W, device=device)[None, :]
    spec = torch.fft.rfftn(white) * torch.exp(-(fy**2 + fx**2) / (2 * 0.08**2))
    specimen = torch.fft.irfftn(spec, s=(H, W))
    specimen = specimen / specimen.std()
    del white, spec
    cpu_g = torch.Generator().manual_seed(seed)
    walk = torch.cumsum(torch.randn((t, 2), generator=cpu_g), dim=0)
    walk = walk - walk[t // 2]
    walk = torch.round(walk / max(float(walk.abs().max()), 1e-6) * 6.0).long()
    movie = torch.empty((t, h, w), dtype=torch.float32, device=device)
    for k in range(t):
        sy, sx = int(walk[k, 0]), int(walk[k, 1])
        movie[k] = specimen[pad - sy : pad - sy + h, pad - sx : pad - sx + w]
        movie[k] += torch.randn((h, w), generator=g, device=device)
    return movie, walk


def synthetic_frames_gpu(t, h, w, seed, device, f0=0, f1=None):
    """Frames [f0, f1) of a movie like synthetic_movie_gpu's whose frames can be generated independently (one noise seed
    per frame): every rank of a frame-split run makes its own block of the SAME movie."""
    f1 = t if f1 is None else f1
    g = torch.Generator(device=device).manual_seed(seed)
    pad = 16
    H, W = h + 2 * pad, w + 2 * pad
    white = torch.randn((H, W), generator=g, device=device)
    fy = torch.fft.fftfreq(H, device=device)[:, None]
    fx = torch.fft.rfftfreq(W, device=device)[None, :]
    spec = torch.fft.rfftn(white) * torch.exp(-(fy**2 + fx**2) / (2 * 0.08**2))
    del white
    specimen = torch.fft.irfftn(spec, s=(H, W))
    del spec
    specimen = specimen / specimen.std()
    cpu_g = torch.Generator().manual_seed(seed)
    walk = torch.cumsum(torch.randn((t, 2), generator=cpu_g), dim=0)
    walk = walk - walk[t // 2]
    walk = torch.round(walk / max(float(walk.abs().max()), 1e-6) * 6.0).long()
    frames = torch.empty((f1 - f0, h, w), dtype=torch.float32, device=device)
    for k in range(f0, f1):
        sy, sx = int(walk[k, 0]), int(walk[k, 1])
        gk = torch.Generator(device=device).manual_seed(seed * 1000 + k)
        frames[k - f0] = specimen[pad - sy : pad - sy + h, pad - sx : pad - sx + w]
        frames[k - f0] += torch.randn((h, w), generator=gk, device=device)
    return frames, walk


def frame_split_record(dev, rank, world, steps, iterations, dist):
    """BASELINE config 4 through distributed.motion_correct_frame_split: ONE 40 x 8192^2 movie split by frames over the
    ranks, spline optimiser included (Sigma + coefficient-gradient all-reduce per iteration, frame-sum all-reduce at the
    end, NCCL).  Returns the sub-record of the benchmark line (rank 0) or None."""
    import random

    import torch_motion_correction_b200 as tmc
    from torch_motion_correction_b200 import _fourier
    from torch_motion_correction_b200.distributed import frame_range, motion_correct_frame_split

    cfg = WORKLOADS["c4"]
    t, h, w, px, p = cfg["t"], cfg["h"], cfg["w"], cfg["pixel_spacing"], cfg["patch"]
    f0, f1 = frame_range(t, rank, world)
    local, _ = synthetic_frames_gpu(t, h, w, 4040, dev, f0, f1)
    kw = dict(patch_sidelength=p, n_iterations=iterations, deformation_field_resolution=cfg["resolution"])

    def step():
        random.seed(99)  # rank 0 draws the optimiser's mini-batches and broadcasts them
        return motion_correct_frame_split(local, px, f0, t, **kw)

    def barrier():
        dist.barrier()
        torch.cuda.synchronize(dev)

    total, field = step()
    step()
    barrier()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # every repetition timed on its own (device events, max over ranks), the MEDIAN reported: the 100 optimiser iterations
    # are 100 host-driven launch groups with a small all-reduce each, and one slow repetition (a host hiccup on one of
    # the N ranks) would otherwise own the mean
    per_step = []
    for _ in range(max(steps, 3)):
        barrier()
        s.record()
        total, field = step()
        e.record()
        barrier()
        one = torch.tensor([s.elapsed_time(e)], device=dev)
        dist.all_reduce(one, op=dist.ReduceOp.MAX)
        per_step.append(float(one))
    ms = torch.tensor([sorted(per_step)[len(per_step) // 2]], device=dev)
    # the one bandwidth-relevant collective alone: all-reduce of the (h, w) fp32 partial frame sums
    buf = torch.zeros((h, w), dtype=torch.float32, device=dev)
    for _ in range(2):
        dist.all_reduce(buf)
    barrier()
    s.record()
    for _ in range(5):
        dist.all_reduce(buf)
    e.record()
    barrier()
    ar_ms = torch.tensor([s.elapsed_time(e) / 5], device=dev)
    dist.all_reduce(ar_ms, op=dist.ReduceOp.MAX)
    del buf
    # single-GPU run of the same movie on rank 0 (speed-up and agreement)
    record = None
    if rank == 0:
        del local
        torch.cuda.empty_cache()
        movie, _ = synthetic_frames_gpu(t, h, w, 4040, dev)

        def single():
            random.seed(99)
            return tmc.motion_correct(movie, px, **kw)

        want_total, want_field = single()
        single()
        torch.cuda.synchronize(dev)
        s.record()
        for _ in range(steps):
            single()
        e.record()
        torch.cuda.synchronize(dev)
        single_ms = s.elapsed_time(e) / steps
        band = _fourier.BandPlan(p, p, dev, px, 500, (300, 10))
        from torch_motion_correction_b200.patch_grid import patch_grid_centers

        centres = patch_grid_centers((t, h, w), (1, p, p), (1, p // 2, p // 2))
        g = centres.shape[1] * centres.shape[2]
        record = {
            "workload": f"c4: ONE {t}x{h}x{w} fp32 movie split by frames over {world} GPUs: whole-frame XC + patch XC ({p} px, {g} "
                        f"patches) + {iterations}-iteration {cfg['resolution']} spline optimiser + warp-and-sum + NCCL frame-sum all-reduce",
            "ms_per_movie": float(ms), "ms_per_movie_repetitions": [round(v, 3) for v in per_step],
            "single_gpu_ms_per_movie": single_ms, "speedup_vs_1_gpu": single_ms / float(ms),
            "frame_sum_allreduce_ms": float(ar_ms), "frame_sum_allreduce_bytes": h * w * 4,
            "frame_sum_allreduce_busbw_gbs": h * w * 4 * 2 * (world - 1) / world / (float(ar_ms) * 1e-3) / 1e9,
            # patch XC and optimiser run patch-sharded (all frames of a share of the patches per rank): per iteration only the
            # coefficient gradient is all-reduced; the band-limited spectra are exchanged once each (XC: both mask powers)
            "optimiser_allreduce_bytes_per_iteration": 2 * cfg["resolution"][0] * cfg["resolution"][1] * cfg["resolution"][2] * 4,
            # all-to-all: every rank keeps 1/world of its own planes and receives the rest of its patches' planes
            "spectra_exchange": "all-to-all (frames -> patches)",
            "spectra_total_bytes": 3 * t * g * band.plane_elems * 8,
            "spectra_received_bytes_per_rank": int(3 * t * g * band.plane_elems * 8 * (world - 1) / world / world),
            "max_abs_field_diff_angstrom": float((field - want_field).abs().max()),
            "rel_l2_sum_diff": float(torch.linalg.norm(total - want_total) / torch.linalg.norm(want_total)),
        }
        del movie
    barrier()
    torch.cuda.empty_cache()
    return record


# --------------------------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------------------------


class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True,
            )
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) >= 6:
                self.samples.append(parts)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for p in self.samples:
            try:
                sm.append(float(p[0]))
                mx.append(float(p[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {
            "sm_mhz": sm[len(sm) // 2] if sm else None,
            "sm_max_mhz": max(mx) if mx else None,
            "samples": len(sm),
            "reasons": sorted(reasons),
        }


# --------------------------------------------------------------------------------------------
# roofline bookkeeping: ALGORITHMIC bytes per C-ABI entry point (DESIGN.md §Kernels)
# --------------------------------------------------------------------------------------------


def measured_peak_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def algorithmic_bytes(cfg, iterations, band_bins, n_patches, plane_elems, whole_plane_elems):
    """Per movie and per KERNEL (timing label of csrc/): the bytes the ALGORITHM must move (DESIGN.md §3) -- inputs that
    have to come from HBM plus the final outputs, not the intermediates an implementation happens to write.  None: the
    kernel has no HBM-bound formulation (compute on band-limited data; reported as issue-bound)."""
    t, h, w = cfg["t"], cfg["h"], cfg["w"]
    frame = 4 * h * w
    patch_spectra = 8 * t * n_patches * plane_elems  # one band-box spectrum per patch and frame
    return {
        # fused warp + frame sum: read every frame once, write one sum
        "warp_tma_kernel": t * frame + frame,
        "warp_lattice_kernel": t * frame + frame,
        # central 50% box of every frame, once per movie
        "stats_partial_kernel": t * frame // 4,
        # band-limited forward row passes: one read of every frame each (patch overlap served by L2)
        "rows_forward_poly<1>": t * frame,      # patch XC: mask^1 and mask^2 packed (quirk Q1)
        "rows_forward_poly<2>": t * frame,      # optimiser spectra, two frames packed
        "rows_forward_p2<4096>": t * frame,     # whole-frame XC
        "rows_forward_real2n<2048>": t * frame,  # whole-frame XC rows as half-length transforms (4096-point rows)
        "rows_forward_real2n<4096>": t * frame,  # the same for 8192-point rows
        "rows_forward_p2": t * frame,
        # column passes: their input is the row pass's intermediate (not algorithmic); they write the band-box spectra
        "cols_forward_p2<1024>": 3 * patch_spectra,  # XC (2 mask powers) + optimiser
        "cols_forward_p2<4096>": 8 * t * whole_plane_elems,
        # leave-one-out products: read both mask powers, write one product per patch and frame
        "xc_leave_one_out_kernel": 3 * patch_spectra,
        # optimiser iteration: the band-limited spectra are read once
        "local_loss_tile_kernel": 8 * t * n_patches * band_bins,
        # inverse transforms + peak search work on band-limited products only
        "cols_inverse_p2<1024>": None, "cols_inverse_p2<4096>": None, "rows_inverse_argmax_poly": None,
        "rows_inverse_argmax_p2<4096>": None, "rows_inverse_argmax_real2n<2048>": None,
        "rows_inverse_argmax_real2n<4096>": None, "peak_finalize_kernel": None,
    }


# --------------------------------------------------------------------------------------------
# CPU arm (oracle) on a bounded sample
# --------------------------------------------------------------------------------------------


def oracle_stages(movie, cfg, iterations):
    """One pass of the oracle (restatement of the reference's PyTorch path, op for op) over ``movie`` on movie.device:
    global XC -> patch XC on the global field -> ``iterations`` optimiser iterations -> correct + sum.  Returns wall
    seconds per stage (the device is synchronised around every stage when it is a GPU)."""
    from oracle import reference_path as rp

    px, p = cfg["pixel_spacing"], cfg["patch"]
    cuda = movie.is_cuda

    def tick():
        if cuda:
            torch.cuda.synchronize(movie.device)
        return time.perf_counter()

    t0 = tick()
    g = rp.estimate_global_motion(movie, px)
    f, _ = rp.estimate_motion_cross_correlation_patches(movie, px, patch_sidelength=p, deformation_field=g)
    t1 = tick()
    if iterations > 0:
        f = rp.estimate_local_motion(movie, px, n_iterations=iterations, patch_shape=(p, p),
                                     deformation_field_resolution=cfg["resolution"], initial_deformation_field=f, grid_type="bspline")
    t2 = tick()
    total = rp.correct_motion(movie, f, px, "bspline").sum(dim=0)
    if cuda:
        total = total.cpu()
    t3 = tick()
    return {"estimate_xc": t1 - t0, "optimiser": t2 - t1, "correct": t3 - t2}


def cpu_sample_plan(cfg, iterations):
    """A bounded sample of the workload (about 10-30 s of CPU work per pass): fewer frames, a crop, fewer iterations."""
    t, h, w = cfg["t"], cfg["h"], cfg["w"]
    if h * w <= 1024 * 1024:
        return dict(frames=min(t, 10), crop=(h, w), iterations=min(iterations, 3))
    return dict(frames=8, crop=(h // 2, w // 2), iterations=min(iterations, 3))


def run_cpu_arm(cfg, movie_cpu_full, steps, warmup, tag, iterations):
    """Times the oracle on the sample for real (every step is one full pass over the sample, nothing synthesised) and
    extrapolates stage by stage: all stages scale with frames x area, the optimiser also with its iteration count."""
    torch.set_num_threads(os.cpu_count() or 1)
    plan = cpu_sample_plan(cfg, iterations)
    n, (ch, cw), its = plan["frames"], plan["crop"], plan["iterations"]
    sample = movie_cpu_full[:n, :ch, :cw].contiguous()
    for _ in range(warmup):
        oracle_stages(sample, cfg, its)
    passes = [oracle_stages(sample, cfg, its) for _ in range(max(steps, 1))]
    stage = {k: sum(p_[k] for p_ in passes) / len(passes) for k in passes[0]}
    dt = sum(stage.values())
    frac = (n / cfg["t"]) * (ch * cw) / (cfg["h"] * cfg["w"])
    full = stage["estimate_xc"] / frac + stage["correct"] / frac
    if its > 0:
        full += stage["optimiser"] / frac * (iterations / its)
    return {
        "value": 1.0 / full,
        "unit": "movies/s",
        "cores": torch.get_num_threads(),
        "kind": "port",
        "sample": f"{tag}: one real pass of the oracle (global XC + patch XC + {its} of {iterations} optimiser iterations + correct) over "
                  f"{n} of {cfg['t']} frames, crop {ch}x{cw} of {cfg['h']}x{cfg['w']}: {dt:.1f} s measured per pass "
                  f"(xc {stage['estimate_xc']:.1f} s, optimiser {stage['optimiser']:.1f} s, correct {stage['correct']:.1f} s); value = "
                  f"1 / ({full:.0f} s per movie), every stage scaled by frames x area, the optimiser also by iterations "
                  f"(understates the reference's O(T^2) leave-one-out loop)",
        "seconds_per_step": dt,
        "extrapolated_seconds_per_movie": full,
    }


def run_aten_cuda_baseline(cfg, movie_gpu, iterations):
    """The existing Blackwell path: the same oracle (the reference's algorithm op for op) with the tensors on the B200, i.e.
    stock ATen / cuFFT sm_100 kernels (SURVEY.md §8d).  One pass over the WHOLE movie after a 4-frame warm-up pass
    (cuFFT plans, allocator)."""
    try:
        with torch.device(movie_gpu.device):
            oracle_stages(movie_gpu[:4], cfg, min(iterations, 1))
            stage = oracle_stages(movie_gpu, cfg, iterations)
        dt = sum(stage.values())
        return {"value": 1.0 / dt, "unit": "movies/s", "ms_per_movie": dt * 1e3, "kind": "oracle port on device=cuda (ATen / cuFFT)",
                "stage_seconds": {k: round(v, 3) for k, v in stage.items()},
                "sample": f"whole movie, one pass, {iterations} optimiser iterations, device-resident input, sum read back"}
    except Exception as exc:  # the baseline must not take the benchmark line down
        return {"unavailable": f"{type(exc).__name__}: {str(exc)[:200]}"}
    finally:
        torch.cuda.empty_cache()


# --------------------------------------------------------------------------------------------
# main
# --------------------------------------------------------------------------------------------


def main():
    args = parse_args()
    cfg = dict(WORKLOADS[args.workload])
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        if rank != 0:
            return 0
        cpu_g = torch.Generator().manual_seed(0)
        ref_iterations = 100 if args.iterations < 0 else args.iterations
        plan = cpu_sample_plan(cfg, ref_iterations)
        n, (ch, cw) = plan["frames"], plan["crop"]
        if torch.cuda.is_available():
            movie, _ = synthetic_movie_gpu(n, cfg["h"], cfg["w"], 0, torch.device("cuda", local_rank))
            movie_cpu = movie.cpu()
            del movie
        else:
            movie_cpu = torch.randn((n, cfg["h"], cfg["w"]), generator=cpu_g)
        base = run_cpu_arm(cfg, movie_cpu, args.steps, max(args.warmup, 0), "reference arm", ref_iterations)
        line = {
            "impl": "reference", "metric": "movies_per_second_estimate_plus_correct", "value": base["value"], "unit": "movies/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": base["seconds_per_step"] * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_text(args.workload, cfg, ref_iterations), "pixel_spacing": cfg["pixel_spacing"],
                       "arm": "CPU oracle port (the reference's algorithm op for op) on a bounded sample, see cpu_baseline.sample"},
            # ms_per_step is the measured wall time of one pass over the sample; value extrapolates it to whole movies
            "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample", "seconds_per_step",
                                                  "extrapolated_seconds_per_movie")},
            "e2e": {"value": base["value"], "unit": "movies/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        }
        print(json.dumps(line))
        return 0

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    import torch.distributed as dist

    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    import torch_motion_correction_b200 as tmc
    from torch_motion_correction_b200 import _lib

    iterations = args.iterations
    has_optimizer = hasattr(tmc, "estimate_local_motion")
    if iterations < 0:
        iterations = 100 if has_optimizer else 0  # the reference's default n_iterations
    if not has_optimizer:
        iterations = 0
    px, p = cfg["pixel_spacing"], cfg["patch"]

    movie, _ = synthetic_movie_gpu(cfg["t"], cfg["h"], cfg["w"], 1000 + rank, dev)

    def step(m):
        random.seed(0)  # the optimiser's mini-batch order: every step computes the same outputs
        return tmc.motion_correct(
            m, px, patch_sidelength=p, deformation_field_resolution=cfg["resolution"], n_iterations=iterations
        )

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- device-resident throughput ------------------------------------------------------------
    # the clock sampler (nvidia-smi) starts before the warm-up: its start-up (NVML init) must not land inside
    # the timed region; it samples clocks / throttle reasons under load through warm-up and timed steps
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        step(movie)
    barrier()
    _lib.TIMING = {}
    _lib.kernel_timing(True)  # CUDA events around the hot kernels' launches, on their stream, inside the timed region
    calls_before = dict(_lib.CALLS)
    launches_before = _lib.query("tmc_launch_count") + _lib.GRAPH_LAUNCHES
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    start.record()
    for _ in range(args.steps):
        total, field = step(movie)
    end.record()
    barrier()
    elapsed_ms = start.elapsed_time(end)
    timing, _lib.TIMING = _lib.TIMING, None
    _lib.kernel_timing(False)
    kernel_times = _lib.kernel_timing_report()
    launches = _lib.query("tmc_launch_count") + _lib.GRAPH_LAUNCHES - launches_before
    clocks = sampler.stop() if rank == 0 else None
    t_ms = torch.tensor([elapsed_ms], device=dev)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    max_ms = float(t_ms)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"field": field, "frame_sum": total})
    del total, field

    # ---- end to end through the public API with HOST buffers ----------------------------------
    # motion_correct_many: the public call for host-resident movies; it overlaps the H2D copy of the next movie
    # with the processing of the current one and copies every frame sum back to pinned host memory
    host = torch.empty(movie.shape, dtype=torch.float32, pin_memory=True)
    host.copy_(movie)
    host_out = torch.empty((cfg["h"], cfg["w"]), dtype=torch.float32, pin_memory=True)
    del movie
    torch.cuda.empty_cache()
    e2e_kwargs = dict(patch_sidelength=p, deformation_field_resolution=cfg["resolution"], n_iterations=iterations)

    def e2e_run(n):
        for _ in tmc.motion_correct_many((host for _ in range(n)), px, device=dev, out_host=host_out, **e2e_kwargs):
            pass

    e2e_run(2)
    barrier()
    s2, e2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s2.record()
    e2e_run(args.steps)
    e2.record()
    barrier()
    e_ms = torch.tensor([s2.elapsed_time(e2)], device=dev)
    if world > 1:
        dist.all_reduce(e_ms, op=dist.ReduceOp.MAX)
    e2e_ms = float(e_ms)

    # the ceiling of that number: the bare pinned-host -> device copy of the movie, all ranks at once (no compute at all)
    sink = torch.empty(host.shape, dtype=torch.float32, device=dev)
    sink.copy_(host, non_blocking=True)
    barrier()
    s2.record()
    for _ in range(3):
        sink.copy_(host, non_blocking=True)
    e2.record()
    barrier()
    c_ms = torch.tensor([s2.elapsed_time(e2) / 3], device=dev)
    if world > 1:
        dist.all_reduce(c_ms, op=dist.ReduceOp.MAX)
    h2d_ms = float(c_ms)
    del sink

    # the same with the movie held as uint16 detector counts on the host (K3 / Falcon movies are integer counts): half the
    # PCIe bytes, converted to fp32 on the device (additional record; the fp32 number above stays the headline)
    host16 = torch.empty(host.shape, dtype=torch.uint16, pin_memory=True)
    host16.copy_(torch.round(host * 16.0 + 1024.0).clamp_(0, 65535).to(torch.uint16))

    def e2e16_run(n):
        for _ in tmc.motion_correct_many((host16 for _ in range(n)), px, device=dev, out_host=host_out, **e2e_kwargs):
            pass

    e2e16_run(2)
    barrier()
    s2.record()
    e2e16_run(args.steps)
    e2.record()
    barrier()
    e16 = torch.tensor([s2.elapsed_time(e2)], device=dev)
    if world > 1:
        dist.all_reduce(e16, op=dist.ReduceOp.MAX)
    e2e16_ms = float(e16)
    del host16

    torch.cuda.empty_cache()
    split = None
    if world > 1 and not args.no_frame_split:
        split = frame_split_record(dev, rank, world, max(2, min(args.steps, 3)), iterations, dist)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ---- roofline: every timed kernel, the dominant one in front --------------------------------------------------
    # per C-ABI entry point: device time per movie from CUDA events recorded around every call inside the timed region;
    # per kernel: CUDA events recorded by the library right before / after each launch on the launching stream
    per_entry = {}
    for name, pairs in timing.items():
        per_entry[name] = sum(a.elapsed_time(b) for a, b in pairs) / args.steps  # ms per movie
    from torch_motion_correction_b200 import _fourier
    from torch_motion_correction_b200.patch_grid import patch_grid_centers

    band = _fourier.BandPlan(p, p, dev, px, 500, (300, 10))
    whole = _fourier.BandPlan(cfg["h"], cfg["w"], dev, px, 500, (300, 10))
    centres = patch_grid_centers((cfg["t"], cfg["h"], cfg["w"]), (1, p, p), (1, p // 2, p // 2))
    n_patches = centres.shape[1] * centres.shape[2]
    band_bins = int((band.weight != 0).sum())  # bins inside the pass band (the box around it holds band.plane_elems)
    bytes_tbl = algorithmic_bytes(cfg, iterations, band_bins, n_patches, band.plane_elems, whole.plane_elems)
    peak, peak_src = measured_peak_gbs()
    import csv
    import glob

    ncu_rows = {}
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "*_ncu_full_kernels.csv"))):  # later tags override
        try:
            for r in csv.DictReader(open(path)):
                if r.get("dram_read_MB"):
                    ncu_rows[r["kernel"]] = (int((float(r["dram_read_MB"]) + float(r["dram_write_MB"] or 0)) * 1e6),
                                             os.path.basename(path))
        except Exception:  # a malformed summary must not break the benchmark line
            continue

    def ncu_traffic(kernel):
        hit = [v for k, v in ncu_rows.items() if k.startswith(kernel.split("<")[0]) and (("<" not in kernel) or kernel.split("<")[1].rstrip(">") in k)]
        return hit[-1] if hit else (None, None)

    kernels = []
    for name, (count, total_ms) in kernel_times.items():
        launches_per_movie = count / args.steps
        ms_movie = total_ms / args.steps
        entry = {"kernel": name, "launches_per_movie": launches_per_movie, "ms_per_movie": round(ms_movie, 4),
                 "us_per_launch": round(1e3 * total_ms / max(count, 1), 2), "timing": "CUDA events around each launch"}
        nbytes = bytes_tbl.get(name)
        if nbytes:
            achieved = nbytes / (ms_movie * 1e-3) / 1e9 if ms_movie > 0 else 0.0
            entry.update(bound="hbm", algorithmic_bytes_per_movie=nbytes, achieved=round(achieved, 1), frac=round(achieved / peak, 4))
        else:
            entry.update(bound="issue" if name in bytes_tbl else None, algorithmic_bytes_per_movie=None, achieved=None, frac=None)
        traffic, src = ncu_traffic(name)
        if traffic is not None:
            entry.update(traffic_per_launch=traffic, traffic_source=src)
        kernels.append(entry)
    if "tmc_local_steps" in per_entry and iterations > 0:
        # the optimiser's two kernels are chained by programmatic dependent launches (events in between would serialise
        # them): the iteration time is the entry point's time / iterations and covers loss + coefficient kernel
        ms_movie = per_entry["tmc_local_steps"]
        nbytes = bytes_tbl["local_loss_tile_kernel"]
        achieved = nbytes * iterations / (ms_movie * 1e-3) / 1e9
        entry = {"kernel": "local_loss_tile_kernel", "launches_per_movie": iterations, "ms_per_movie": round(ms_movie, 4),
                 "us_per_launch": round(1e3 * ms_movie / iterations, 2),
                 "timing": "entry point tmc_local_steps / iterations (includes the dependent single-CTA coefficient kernel)",
                 "bound": "hbm", "algorithmic_bytes_per_movie": nbytes * iterations, "achieved": round(achieved, 1),
                 "frac": round(achieved / peak, 4)}
        traffic, src = ncu_traffic("local_loss_tile_kernel")
        if traffic is not None:
            entry.update(traffic_per_launch=traffic, traffic_source=src)
        kernels.append(entry)
    kernels.sort(key=lambda k: -k["ms_per_movie"])
    # the dominant kernel: largest device time per movie among ALL timed kernels
    dom = kernels[0] if kernels else None
    roof = {"bound": "hbm", "peak": peak, "peak_source": peak_src, "unit": "GB/s", "traffic": None}
    if dom is not None:
        per_launch = (dom["algorithmic_bytes_per_movie"] or 0) / max(dom["launches_per_movie"], 1)
        roof.update(kernel=dom["kernel"], ms_per_movie=dom["ms_per_movie"], launches_per_movie=dom["launches_per_movie"],
                    launch_us=dom["us_per_launch"], algorithmic_bytes_per_launch=int(per_launch), achieved=dom["achieved"],
                    frac=dom["frac"], traffic=dom.get("traffic_per_launch"), traffic_source=dom.get("traffic_source"),
                    timing=dom["timing"])
        if dom["bound"] != "hbm":
            roof["note"] = "the dominant kernel works on band-limited data: no HBM-bound formulation, issue-bound"
    roof["kernels"] = kernels
    # the two kernels BASELINE.json names (warp/sum and patch filter), whatever their rank
    roof["north_star_kernels"] = {k["kernel"]: k["frac"] for k in kernels
                                  if k["kernel"] in ("warp_tma_kernel", "warp_lattice_kernel", "rows_forward_poly<1>", "rows_forward_poly<2>")}
    breakdown = {k: round(v, 4) for k, v in sorted(per_entry.items(), key=lambda kv: -kv[1])}

    cpu_base = None
    if not args.no_cpu_baseline and world == 1:
        cpu_base = run_cpu_arm(cfg, host[:8].clone(), 1, 0, "cpu_baseline", iterations)
        cpu_base = {k: cpu_base[k] for k in ("value", "unit", "cores", "kind", "sample", "seconds_per_step",
                                             "extrapolated_seconds_per_movie")}
    aten_base = None
    if not args.no_cpu_baseline and world == 1 and not args.no_aten_baseline:
        aten_base = run_aten_cuda_baseline(cfg, host.to(dev), iterations)

    movies = args.steps * world
    calls = {k: _lib.CALLS[k] - calls_before.get(k, 0) for k in _lib.CALLS}
    line = {
        "metric": "movies_per_second_estimate_plus_correct",
        "value": movies / (max_ms * 1e-3),
        "unit": "movies/s",
        "n_gpus": world,
        "steps": args.steps,
        "warmup": max(args.warmup, 3),
        "ms_per_step": max_ms / args.steps,
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "f32",
        "data": "synthetic",
        "config": {
            "workload": workload_text(args.workload, cfg, iterations),
            "arm": "CUDA: the rigid pre-correction is served by whole-pixel shifted patch windows, the warp-and-sum is fused",
            "pixel_spacing": px, "movies_per_rank_per_step": 1, "sharding": "independent movies per rank, no collective",
            "l2_policy": "inputs (2.7 GB/movie) exceed L2 (126 MB); no explicit flush",
        },
        "e2e": {
            "value": movies / (e2e_ms * 1e-3), "unit": "movies/s", "ms_per_step": e2e_ms / args.steps,
            # whole job: every rank copies its own movie in and its frame sum out each step
            "h2d_bytes_per_step": host.numel() * 4 * world, "d2h_bytes_per_step": cfg["h"] * cfg["w"] * 4 * world,
            # machine ceiling: the bare host -> device copy of one movie per rank, all ranks copying at once
            "h2d_copy_only_ms_per_step": h2d_ms, "h2d_ceiling_gbs": host.numel() * 4 * world / (h2d_ms * 1e-3) / 1e9,
            "fraction_of_h2d_ceiling": h2d_ms / (e2e_ms / args.steps),
        },
        "e2e_uint16": {
            "value": movies / (e2e16_ms * 1e-3), "unit": "movies/s", "ms_per_step": e2e16_ms / args.steps,
            "h2d_bytes_per_step": host.numel() * 2 * world, "d2h_bytes_per_step": cfg["h"] * cfg["w"] * 4 * world,
            "note": "host movie as uint16 counts, converted to fp32 on the device (tmc_convert_stack)",
        },
        "gpu_launches": launches,
        "c_abi_calls": calls,
        "roofline": roof,
        "entry_point_ms_per_movie": breakdown,
        "cpu_baseline": cpu_base,
        "aten_cuda_baseline": aten_base,
        "frame_split": split,
        "clocks": clocks,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
