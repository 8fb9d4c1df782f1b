"""Which warp kernel serves a movie: the TMA-staged tile kernel takes frames with 16-byte aligned rows, the global-memory
kernel the rest.  Helpers that select each by its input and report which one ran."""

import torch

from torch_motion_correction_b200 import _lib


def at_offset(x):
    """A copy of ``x`` that starts one float into its allocation: its rows are not 16-byte aligned, so the warp runs on
    the global-memory kernel instead of the TMA-staged one."""
    buf = torch.empty(x.numel() + 1, dtype=x.dtype, device=x.device)
    v = buf[1:].view(x.shape)
    v.copy_(x)
    return v


def warp_kernels_ran():
    """The warp kernels launched since ``_lib.kernel_timing(True)``, as their name's prefix; switches the timing off."""
    torch.cuda.synchronize()
    names = _lib.kernel_timing_report()
    _lib.kernel_timing(False)
    return {p for p in ("warp_tma_kernel", "warp_lattice_kernel") if any(k.startswith(p) for k in names)}
