"""Time and peak device memory of the frame sums of a corrected movie: correct_motion_sum, correct_motion_sums with the
dose-weighted sum (and with half sets too), and the materialising route correct_motion + dose_weight.

CUDA events around each call after warm-up; every movie is larger than the 126 MB L2.  Prints the card and its power
limit, then one JSON line per (workload, route).  Usage: python tools/time_sums.py [--reps N]"""

import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

import torch_motion_correction_b200 as tmc  # noqa: E402

# (name, frames, side, Angstrom / px, e / A^2 / frame)
WORKLOADS = [("c2", 40, 4096, 0.83, 1.0), ("400x4096", 400, 4096, 0.83, 0.1)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    print(json.dumps({"card": card}), flush=True)
    routes = {
        "correct_motion_sum": lambda m, f, px, d: tmc.correct_motion_sum(m, f, px, grid_type="bspline"),
        "correct_motion_sums(dose)": lambda m, f, px, d: tmc.correct_motion_sums(m, f, px, "bspline", dose_per_frame=d),
        "correct_motion_sums(dose, half_sets)": lambda m, f, px, d: tmc.correct_motion_sums(
            m, f, px, "bspline", dose_per_frame=d, half_sets=True),
        "correct_motion + dose_weight": lambda m, f, px, d: tmc.dose_weight(
            tmc.correct_motion(m, f, px, grid_type="bspline"), px, dose_per_frame=d),
    }
    for name, t, side, px, dose in WORKLOADS:
        g = torch.Generator(device=dev).manual_seed(0)
        movie = torch.randn((t, side, side), generator=g, device=dev)
        field = 3.0 * torch.randn((2, 3, 5, 5), generator=g, device=dev)
        for route, fn in routes.items():
            fn(movie, field, px, dose)  # warm-up: module load, plans, host tables
            torch.cuda.synchronize()
            base = torch.cuda.memory_allocated()
            torch.cuda.reset_peak_memory_stats()
            times = []
            for _ in range(args.reps):
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                out = fn(movie, field, px, dose)
                e.record()
                torch.cuda.synchronize()
                times.append(s.elapsed_time(e))
                del out
            peak = torch.cuda.max_memory_allocated() - base
            times.sort()
            print(json.dumps({"workload": name, "shape": [t, side, side], "route": route, "median_ms": round(times[len(times) // 2], 2),
                              "min_ms": round(times[0], 2), "max_ms": round(times[-1], 2),
                              "peak_extra_gb": round(peak / 1e9, 3), "stack_gb": round(movie.numel() * 4 / 1e9, 3)}), flush=True)
        del movie
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
