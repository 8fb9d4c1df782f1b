"""Device time of the fused warp-and-sum's kernels at the benchmark size (diagnostic): python tools/warp_time.py [t h w]."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch_motion_correction_b200 as tmc
from torch_motion_correction_b200 import _lib

t, h, w = (int(v) for v in sys.argv[1:4]) if len(sys.argv) > 3 else (40, 4096, 4096)
dev = torch.device("cuda:0")
g = torch.Generator(device=dev).manual_seed(21)
img = torch.randn((t, h, w), generator=g, device=dev)
field = (torch.randn((2, 3, 5, 5), generator=g, device=dev) * 2.0)
for _ in range(2):
    tmc.correct_motion_sum(img, field, 0.83, grid_type="bspline")
torch.cuda.synchronize()
_lib.kernel_timing(True)
for _ in range(5):
    tmc.correct_motion_sum(img, field, 0.83, grid_type="bspline")
torch.cuda.synchronize()
rep = _lib.kernel_timing_report()
_lib.kernel_timing(False)
print({k: round(ms / n, 4) for k, (n, ms) in rep.items() if "warp" in k or "lattice" in k})
