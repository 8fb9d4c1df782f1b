"""Device time per iteration of the spline optimiser on the benchmark movie (diagnostic): python tools/time_optimiser.py"""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch, bench
import torch_motion_correction_b200 as tmc

dev = torch.device("cuda:0")
movie, _ = bench.synthetic_movie_gpu(40, 4096, 4096, 1000, dev)
f0, c = tmc.estimate_motion_cross_correlation_patches(movie, 0.83, patch_sidelength=1024)
res = {}
for n in (100, 500):
    for rep in range(2):
        torch.cuda.synchronize(); t0 = time.perf_counter()
        tmc.estimate_local_motion(movie, 0.83, (1024, 1024), (3, 5, 5), f0, n_iterations=n, grid_type="bspline")
        torch.cuda.synchronize(); res[n] = (time.perf_counter() - t0) * 1e3
print(f"{(res[500] - res[100]) / 400 * 1e3:.2f} us per iteration")
