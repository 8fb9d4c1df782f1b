"""Device times and live row blocks of the C2 peak searches (tmc_xc_peaks) on the benchmark movie:
python tools/time_peaks.py [frame size, default 4096]

Builds the two searches of a motion_correct step from bench.py's seeded movie (40 frames, 0.83 A/px, 300-10 A band):
the whole-frame products against the middle frame and the leave-one-out products of the 1024-px patches.  Prints one
JSON line per search: CUDA-event ms per search (median of 10), per-kernel ms of one search (library timing), the coarse
groups the coarse bound samples (one seed group per item: count, total, fraction) and the live row blocks left by the
row L1 norms and the seed's bound (count, total, fraction)."""
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import bench  # noqa: E402
from torch_motion_correction_b200 import _fourier, _lib, _ops  # noqa: E402
from torch_motion_correction_b200.estimate_motion_xc import (global_spectra, mean_except_current_spectra,  # noqa: E402
                                                             patch_xc_geometry)

dev = torch.device("cuda:0")
size = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
movie, _ = bench.synthetic_movie_gpu(40, size, size, 4040, dev)
t = movie.shape[0]
stats = _ops.stack_stats(movie)

plan_g, spec_g = global_spectra(movie, stats, 0.83, 500, (300, 10))
cur = torch.arange(t, dtype=torch.int32, device=dev)
ref = torch.full((t,), t // 2, dtype=torch.int32, device=dev)
prod_g = _fourier.pair_products(spec_g, ref, cur, plan_g.plane_elems).view(t, plan_g.ky, plan_g.kx, 2)

_, origins, plan_p, mask, _ = patch_xc_geometry(movie.shape, 1024, 0.83, 500, (300, 10), None, dev)
g = len(origins)
_, spec_p = mean_except_current_spectra(movie, stats, plan_p, mask, 1024, origins, None)
offsets = torch.zeros((t + 1,), dtype=torch.int32, device=dev)
deltas = torch.zeros((1,), dtype=torch.int32, device=dev)
prod_p = _fourier.leave_one_out_products(spec_p, t, g, plan_p.plane_elems, offsets, deltas).view(t * g, plan_p.ky, plan_p.kx, 2)
del movie, spec_g, spec_p
# rows of a coarse group: the row block of rows_coarse_bound_p2<nx / 4>
GROUP_ROWS = {1024: 128, 4096: 32, 8192: 16}
power_limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True).stdout.strip()

for name, plan, prod in (("whole_frame", plan_g, prod_g), ("patches", plan_p, prod_p)):
    for _ in range(3):
        plan.peaks(prod, sub_pixel=name == "patches")
    times = []
    for _ in range(10):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        plan.peaks(prod, sub_pixel=name == "patches")
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    _lib.kernel_timing(True)
    ws = []
    plan.peaks(prod, sub_pixel=name == "patches", workspace_out=ws)
    torch.cuda.synchronize()
    kernels = {k: round(ms, 4) for k, (n, ms) in _lib.kernel_timing_report().items()}
    _lib.kernel_timing(False)
    total = prod.shape[0] * _lib.query("tmc_xc_peak_partials", plan.ny, plan.nx)
    live, sampled = ws[0][:8].view(torch.int32).tolist()
    all_groups = prod.shape[0] * -(-plan.ny // GROUP_ROWS[plan.nx])
    print(json.dumps({"search": name, "items": prod.shape[0], "shape": [plan.ny, plan.nx], "kx": plan.kx,
                      "ms_per_search": round(sorted(times)[len(times) // 2], 4), "kernels_ms": kernels,
                      "coarse_groups": sampled, "groups": all_groups, "coarse_fraction": round(sampled / all_groups, 5),
                      "live_blocks": live, "row_blocks": total, "live_fraction": round(live / total, 5),
                      "gpu": torch.cuda.get_device_name(dev), "power_limit": power_limit}))
