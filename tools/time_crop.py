"""Time of Fourier cropping by 2 of 40-frame movies: fourier_crop at 8192^2, K3 super-resolution 11520 x 8184 and K3
5760 x 4092 with the bytes it moves and per-kernel times of one call; at 8192^2 two chunk sizes, alternating in rounds;
motion_correct(fourier_bin=2) against motion_correct at 8192^2 end to end with peak extra device memory.

CUDA events around each call after warm-up; every movie (5.3 to 15 GB) is far larger than the 126 MB L2.  Prints the
card and its power limit, then one JSON line per measurement.  Usage: python tools/time_crop.py [--reps N] [--frames T]"""

import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

import torch_motion_correction_b200 as tmc  # noqa: E402
from torch_motion_correction_b200 import _fourier, _lib  # noqa: E402
from torch_motion_correction_b200.prepare import fourier_crop_shape  # noqa: E402


def timed(fn, reps):
    fn()  # warm-up: module load, plans, host tables
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    times = []
    for _ in range(reps):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        out = fn()
        e.record()
        torch.cuda.synchronize()
        times.append(s.elapsed_time(e))
        del out
    peak = torch.cuda.max_memory_allocated() - base
    times.sort()
    return {"median_ms": round(times[len(times) // 2], 3), "min_ms": round(times[0], 3), "max_ms": round(times[-1], 3),
            "peak_extra_gb": round(peak / 1e9, 3)}


def crop_bytes(t, h, w, h2, w2, fused):
    """(algorithmic, kernel-level) bytes: one read of the movie and one write of the output; and that plus the
    complex64 intermediates each pass writes and the next reads: rows -> columns at h rows on whole frame pairs, then
    the (h2, kx) columns once with the fused column kernel, or the ky box and the box after the inverse column pass"""
    kx = w2 // 2 + 1
    planes = 2 * ((t + 1) // 2)
    algorithmic = 4 * t * (h * w + h2 * w2)
    intermediate = 8 * planes * h * kx + 8 * t * h2 * kx + (0 if fused else 8 * planes * h2 * kx)
    return algorithmic, algorithmic + 2 * intermediate


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--frames", type=int, default=40)
    ap.add_argument("--hbm-gbps", type=float, default=6535.0, help="measured HBM read+write rate the passes are held to")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    print(json.dumps({"card": card}), flush=True)
    t = args.frames
    default_chunk = _fourier.CHUNK_BYTES
    g = torch.Generator(device=dev).manual_seed(0)
    for h, w in ((8192, 8192), (11520, 8184), (5760, 4092)):
        movie = torch.randn((t, h, w), generator=g, device=dev)
        h2, w2 = fourier_crop_shape((h, w), 2)
        r = timed(lambda: tmc.fourier_crop(movie, 2), args.reps)
        algorithmic, kernel = crop_bytes(t, h, w, h2, w2, fused=(h & (h - 1)) == 0)
        s = r["median_ms"] * 1e-3
        _lib.kernel_timing(True)
        tmc.fourier_crop(movie, 2)
        torch.cuda.synchronize()
        kernels = {k: round(ms, 3) for k, (_, ms) in _lib.kernel_timing_report().items()}
        _lib.kernel_timing(False)
        print(json.dumps({"shape": [t, h, w], "out": [h2, w2], "what": "fourier_crop", **r,
                          "algorithmic_gb": round(algorithmic / 1e9, 2),
                          "algorithmic_share_of_measured_hbm": round(algorithmic / s / 1e9 / args.hbm_gbps, 3),
                          "algorithmic_floor_ms": round(algorithmic / (args.hbm_gbps * 1e9) * 1e3, 3),
                          "kernel_gb": round(kernel / 1e9, 2),
                          "kernel_share_of_measured_hbm": round(kernel / s / 1e9 / args.hbm_gbps, 3),
                          "kernel_ms_one_call": kernels}), flush=True)
        if h == 8192:
            ab = {}
            for _ in range(3):  # rounds: every chunk size runs between the others
                for chunk in (1 << 30, 8 << 30):
                    _fourier.CHUNK_BYTES = chunk
                    ab.setdefault(chunk, []).append(timed(lambda: tmc.fourier_crop(movie, 2), args.reps)["median_ms"])
            for chunk, meds in ab.items():
                _fourier.CHUNK_BYTES = chunk
                _lib.kernel_timing(True)
                tmc.fourier_crop(movie, 2)
                torch.cuda.synchronize()
                kernels = {k: round(ms, 3) for k, (_, ms) in _lib.kernel_timing_report().items()}
                _lib.kernel_timing(False)
                print(json.dumps({"shape": [t, h, w], "what": "fourier_crop chunk sizes", "chunk_bytes": chunk,
                                  "round_medians_ms": meds, "kernel_ms_one_call": kernels}), flush=True)
            _fourier.CHUNK_BYTES = default_chunk
        del movie
        torch.cuda.empty_cache()

    px = 0.415
    movie = torch.randn((t, 8192, 8192), generator=g, device=dev)
    for label, b in (("motion_correct(fourier_bin=2)", 2), ("motion_correct", None)):
        r = timed(lambda: tmc.motion_correct(movie, px, fourier_bin=b), max(2, args.reps // 3))
        print(json.dumps({"shape": [t, 8192, 8192], "what": label, **r,
                          "stack_gb": round(movie.numel() * 4 / 1e9, 3)}), flush=True)


if __name__ == "__main__":
    main()
