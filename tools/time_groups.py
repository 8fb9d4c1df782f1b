"""Time of frame grouping at 400 x 4096^2, G = 10: the group_frames kernel (and its HBM rate), estimate_motion on the
group sums against estimate_motion on the raw frames, and motion_correct(dose_per_frame=0.1, frame_group=10) end to end
with its peak extra device memory.

CUDA events around each call after warm-up; the movie (26.8 GB) is far larger than the 126 MB L2.  Prints the card and
its power limit, then one JSON line per measurement.  Usage: python tools/time_groups.py [--reps N] [--frames T]"""

import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

import torch_motion_correction_b200 as tmc  # noqa: E402


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--frames", type=int, default=400)
    ap.add_argument("--side", type=int, default=4096)
    ap.add_argument("--group", type=int, default=10)
    ap.add_argument("--hbm-gbps", type=float, default=6535.0, help="measured HBM read+write rate the kernel is held to")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    print(json.dumps({"card": card}), flush=True)
    t, side, group, px, dose = args.frames, args.side, args.group, 0.83, 0.1
    shape = [t, side, side]
    g = torch.Generator(device=dev).manual_seed(0)
    movie = torch.randn((t, side, side), generator=g, device=dev)

    n_bytes = (t + t // group) * side * side * 4  # one read of the movie + one write of the group sums
    r = timed(lambda: tmc.group_frames(movie, group), 4 * args.reps)
    gbps = n_bytes / (r["median_ms"] * 1e-3) / 1e9
    print(json.dumps({"shape": shape, "group": group, "what": "group_frames", **r, "gb_moved": round(n_bytes / 1e9, 2),
                      "gbps": round(gbps, 1), "share_of_measured_hbm": round(gbps / args.hbm_gbps, 3),
                      "floor_ms": round(n_bytes / (args.hbm_gbps * 1e9) * 1e3, 3)}), flush=True)

    for label, fg in (("estimate_motion grouped", group), ("estimate_motion ungrouped", None)):
        try:
            r = timed(lambda: tmc.estimate_motion(movie, px, dose_per_frame=dose, frame_group=fg), args.reps)
        except torch.cuda.OutOfMemoryError as e:
            r = {"error": str(e).splitlines()[0]}
            torch.cuda.empty_cache()
        print(json.dumps({"shape": shape, "group": fg, "what": label, **r}), flush=True)

    r = timed(lambda: tmc.motion_correct(movie, px, dose_per_frame=dose, frame_group=group), args.reps)
    print(json.dumps({"shape": shape, "group": group, "what": "motion_correct(dose_per_frame=0.1) grouped", **r,
                      "stack_gb": round(movie.numel() * 4 / 1e9, 3)}), flush=True)


if __name__ == "__main__":
    main()
