"""Time of decoding full-size LZW TIFF movies on the device, and of LZW TIFF input end to end.

Two movies written by OpenCV (libtiff, LZW with its default Predictor 2): a K3 counting movie (40 x 4092 x 5760 uint8,
Poisson 0.8 e-/px) and a super-resolution movie (40 x 8184 x 11520 uint8, Poisson 0.2), each in three strip layouts:
one row per strip, 64 rows per strip and one strip per frame.  Prints the card and its power limit, then one JSON line
per measurement:

* decode: median of --reps tmc_tiff_lzw_decode calls after warm-up (CUDA events; payload already on the device), the
  payload and stack bytes against the HBM floor, the per-kernel split, and in the same run the median host-to-device
  copy from pinned memory of the payload and of the uncompressed uint8 stack (the target: decoding faster than the
  uncompressed copy, so a TIFF is never slower to ingest than pre-decoded counts);
* pipeline (--e2e): motion_correct_many over --files copies of the TIFF against the same frames as uint8 MRC stacks,
  alternating in --rounds rounds, host clock around the whole generator.

Usage: python tools/time_tiff.py [--movies k3,sr] [--layouts row,64,frame] [--reps 10] [--e2e] [--files 3]"""

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import torch_motion_correction_b200 as tmc  # noqa: E402
from torch_motion_correction_b200 import _lib, movie_io, prepare  # noqa: E402
from time_eer import HBM_BYTES_PER_S, median_ms, write_uint8_mrc  # noqa: E402

MOVIES = {"k3": (4092, 5760, 0.8), "sr": (8184, 11520, 0.2)}


def main():
    import cv2

    ap = argparse.ArgumentParser()
    ap.add_argument("--movies", default="k3,sr")
    ap.add_argument("--layouts", default="row,64,frame")
    ap.add_argument("--frames", type=int, default=40)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--e2e", action="store_true")
    ap.add_argument("--files", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=2)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    print(json.dumps({"card": card}), flush=True)
    for name in args.movies.split(","):
        h, w, rate = MOVIES[name]
        rng = np.random.default_rng(0)
        t0 = time.perf_counter()
        frames = rng.poisson(rate, size=(args.frames, h, w)).astype(np.uint8)
        host = torch.from_numpy(frames).pin_memory()
        stack_dev = torch.empty_like(host, device=dev)
        raw_ms, _, _ = median_ms(lambda: stack_dev.copy_(host, non_blocking=True), 5)
        for layout in args.layouts.split(","):
            rps = {"row": 1, "frame": h}.get(layout) or int(layout)
            with tempfile.TemporaryDirectory() as tmp:
                path = os.path.join(tmp, "movie.tif")
                t0 = time.perf_counter()
                assert cv2.imwritemulti(path, list(frames), [cv2.IMWRITE_TIFF_COMPRESSION, 5,
                                                             cv2.IMWRITE_TIFF_ROWSPERSTRIP, rps])
                write_s = time.perf_counter() - t0
                movie = movie_io.read_tiff_movie(path)
                payload_dev = movie.payload.to(dev)
                tables = [movie.strip_offsets.to(dev), movie.out_offsets.to(dev)]
                ws = torch.empty((prepare.tiff_workspace_bytes(movie),), dtype=torch.uint8, device=dev)
                status = torch.empty((movie.n_strips,), dtype=torch.int32, device=dev)
                out = torch.empty(movie.shape, dtype=movie.dtype, device=dev)

                def decode():
                    prepare.decode_tiff_into(payload_dev, tables[0], tables[1], movie, out, ws, status)

                decode()
                torch.cuda.synchronize()
                exact = int(status.abs().sum()) == 0 and torch.equal(out, stack_dev)
                ms, lo, hi = median_ms(decode, args.reps)
                _lib.kernel_timing(True)
                decode()
                torch.cuda.synchronize()
                kernels = {k: round(v[1], 3) for k, v in _lib.kernel_timing_report().items() if k.startswith("lzw")}
                _lib.kernel_timing(False)
                copy_ms, _, _ = median_ms(lambda: payload_dev.copy_(movie.payload, non_blocking=True), 5)
                stack_bytes = out.numel()
                floor_ms = 1e3 * (payload_dev.numel() + stack_bytes * (3 if movie.predictor == 2 else 1)) / HBM_BYTES_PER_S
                print(json.dumps({
                    "what": "decode_tiff", "movie": name, "frames": args.frames, "h": h, "w": w, "rate": rate,
                    "rows_per_strip": rps, "strips": movie.n_strips, "predictor": movie.predictor, "exact": exact,
                    "payload_bytes": int(payload_dev.numel()), "stack_bytes": stack_bytes,
                    "ratio": round(payload_dev.numel() / stack_bytes, 3), "median_ms": round(ms, 3),
                    "min_ms": round(lo, 3), "max_ms": round(hi, 3), "kernels_ms": kernels,
                    "hbm_floor_ms": round(floor_ms, 3), "floor_fraction": round(floor_ms / ms, 3),
                    "payload_h2d_ms": round(copy_ms, 3), "uint8_stack_h2d_ms": round(raw_ms, 3),
                    "decode_over_uint8_copy": round(ms / raw_ms, 3), "opencv_write_s": round(write_s, 1),
                }), flush=True)
                del payload_dev, tables, ws, status, out
                if not args.e2e:
                    continue
                mrc = os.path.join(tmp, "movie.mrc")
                write_uint8_mrc(mrc, host)
                runs = {"tiff": [], "mrc": []}

                def run(kind):
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    src = tmc.tiff_movies([path] * args.files) if kind == "tiff" else tmc.mrc_movies([mrc] * args.files)
                    res = [(s.clone(), f) for s, f in tmc.motion_correct_many(src, 1.0, device=dev)]
                    torch.cuda.synchronize()
                    return (time.perf_counter() - t0) * 1e3 / args.files, res

                _, a = run("tiff")
                _, b = run("mrc")
                same = all(torch.equal(x[0], y[0]) for x, y in zip(a, b))
                del a, b
                for _ in range(args.rounds):
                    for kind in ("tiff", "mrc"):
                        runs[kind].append(run(kind)[0])
                for kind in ("tiff", "mrc"):
                    print(json.dumps({"what": f"motion_correct_many_{kind}", "movie": name, "rows_per_strip": rps,
                                      "files": args.files, "ms_per_movie": [round(v, 1) for v in runs[kind]],
                                      "sums_equal": same}), flush=True)
        del host, stack_dev


if __name__ == "__main__":
    main()
