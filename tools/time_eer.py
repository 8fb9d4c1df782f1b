"""Time of rendering a full-size EER movie on the device, and of EER input end to end.

A synthetic EER movie (tests/eer_synth.py) of 4096^2 frames: --frames hardware frames at --rate electrons per pixel per
frame, codec --codec, rendered in fractions of --F frames (1100 x 0.025 e-/px, F = 27: 40 fractions of 0.675 e-/px).
Prints the card and its power limit, then one JSON line per measurement:

* render: median of --reps tmc_eer_render calls after warm-up (CUDA events; payload already on the device), with the
  payload and counts bytes against the HBM floor, and the median host-to-device copy of the payload from pinned memory
  (the bound EER input should be held to: rendering faster than the copy leaves the copy as the limit);
* pipeline: motion_correct_many over --files copies of the movie (EER payload across PCIe, rendered on the device)
  against the same counts as uint8 MRC stacks through mrc_movies (40 x 4096^2 bytes across PCIe), alternating in
  --rounds rounds, host clock around the whole generator.

Usage: python tools/time_eer.py [--frames 1100] [--rate 0.025] [--F 27] [--codec 65001] [--reps 20] [--files 3]"""

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import eer_synth as es  # noqa: E402
import torch_motion_correction_b200 as tmc  # noqa: E402
from torch_motion_correction_b200 import movie_io, prepare  # noqa: E402

HBM_BYTES_PER_S = 7.7e12  # HGX B200 data sheet, one GPU


def median_ms(fn, reps):
    times = []
    for _ in range(reps):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        torch.cuda.synchronize()
        times.append(s.elapsed_time(e))
    times.sort()
    return times[len(times) // 2], times[0], times[-1]


def write_uint8_mrc(path, counts):
    """uint8 MRC: mode 0 with the IMOD flag word saying the bytes are unsigned."""
    tmc.write_mrc(path, counts.view(torch.int8))
    with open(path, "r+b") as f:
        f.seek(152)
        f.write(np.array([1146047817, 0], dtype="<i4").tobytes())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1100)
    ap.add_argument("--rate", type=float, default=0.025)
    ap.add_argument("--F", type=int, default=27)
    ap.add_argument("--codec", type=int, default=65001)
    ap.add_argument("--size", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--files", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=2)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    print(json.dumps({"card": card}), flush=True)
    n = args.size
    with tempfile.TemporaryDirectory() as tmp:
        t0 = time.perf_counter()
        rng = np.random.default_rng(0)
        frames = es.random_frames(rng, args.frames, n * n, args.rate)
        path = os.path.join(tmp, "movie.eer")
        es.write_eer(path, frames, n, n, compression=args.codec, bigtiff=True)
        del frames
        build_s = time.perf_counter() - t0
        t0 = time.perf_counter()
        eer = movie_io.read_eer(path)
        read_s = time.perf_counter() - t0
        nf, dtype = prepare.eer_fractions(eer, args.F)
        used = nf * args.F
        payload = eer.payload[:int(eer.frame_offsets[used])]
        payload_dev = payload.to(dev)
        offsets_dev = eer.frame_offsets[:used + 1].to(dev)
        counts = prepare.eer_counts_buffer((nf, n, n), dtype, dev)
        status = torch.empty((used,), dtype=torch.int32, device=dev)

        def render():
            prepare.render_eer_into(payload_dev, offsets_dev, eer, args.F, counts, status)

        render()
        torch.cuda.synchronize()
        assert int(status.abs().sum()) == 0
        ms, lo, hi = median_ms(render, args.reps)
        copy_ms, _, _ = median_ms(lambda: payload_dev.copy_(payload, non_blocking=True), max(5, args.reps // 2))
        counts_bytes = counts.numel() * counts.element_size()
        floor_ms = 1e3 * (payload.numel() + 2 * counts_bytes) / HBM_BYTES_PER_S  # payload read, counts zeroed + written
        print(json.dumps({
            "what": "render_eer", "frames": used, "size": n, "codec": args.codec, "F": args.F, "fractions": nf,
            "electrons_per_px_per_frame": args.rate, "payload_bytes": int(payload.numel()), "counts_bytes": counts_bytes,
            "median_ms": round(ms, 3), "min_ms": round(lo, 3), "max_ms": round(hi, 3),
            "hbm_floor_ms": round(floor_ms, 3), "payload_h2d_ms": round(copy_ms, 3),
            "payload_h2d_gbps": round(payload.numel() / copy_ms / 1e6, 1),
            "render_over_copy": round(ms / copy_ms, 3), "synth_build_s": round(build_s, 1), "read_eer_s": round(read_s, 2),
        }), flush=True)

        # end to end: the same movie through motion_correct_many as EER and as uint8 MRC
        mrc = os.path.join(tmp, "movie.mrc")
        write_uint8_mrc(mrc, counts.cpu())
        del payload_dev, offsets_dev, counts, status
        eer_paths, mrc_paths = [path] * args.files, [mrc] * args.files
        runs = {"eer": [], "mrc": []}

        def run(kind):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            if kind == "eer":
                out = list(tmc.motion_correct_many(tmc.eer_movies(eer_paths), 1.0, device=dev, eer_frames_per_fraction=args.F))
            else:
                out = list(tmc.motion_correct_many(tmc.mrc_movies(mrc_paths), 1.0, device=dev))
            torch.cuda.synchronize()
            return (time.perf_counter() - t0) * 1e3 / args.files, out

        _, a = run("eer")  # warm-up of both routes; and they must agree
        _, b = run("mrc")
        same = all(torch.equal(x[0], y[0]) for x, y in zip(a, b))
        for _ in range(args.rounds):
            for kind in ("eer", "mrc"):
                runs[kind].append(run(kind)[0])
        for kind in ("eer", "mrc"):
            print(json.dumps({"what": f"motion_correct_many_{kind}", "files": args.files,
                              "ms_per_movie": [round(v, 1) for v in runs[kind]], "sums_equal": same,
                              "pcie_bytes_per_movie": int(eer.frame_offsets[used]) if kind == "eer" else nf * n * n}),
                  flush=True)


if __name__ == "__main__":
    main()
