"""Tensor-level wrappers over the C ABI (one function per entry point)."""

from __future__ import annotations

import torch

from . import _lib
from ._lib import call, ptr, query, stream_ptr


def _f32(shape, like: torch.Tensor) -> torch.Tensor:
    return torch.empty(shape, dtype=torch.float32, device=like.device)


def stack_stats(image: torch.Tensor, frac_low: float = 0.25, frac_high: float = 0.75) -> torch.Tensor:
    """Device float[2] = (mean, unbiased std) of the central box (reference utils.py:72-80)."""
    t, h, w = image.shape
    y0, y1 = int(frac_low * h), int(frac_high * h)
    x0, x1 = int(frac_low * w), int(frac_high * w)
    out = _f32((2,), image)
    ws = torch.empty(query("tmc_stack_stats_workspace_doubles"), dtype=torch.float64, device=image.device)
    with torch.cuda.device(image.device):
        call("tmc_stack_stats", ptr(image), t, h, w, y0, y1, x0, x1, ptr(out), ptr(ws), stream_ptr(image.device))
    return out


def stack_moments(image: torch.Tensor, frac_low: float = 0.25, frac_high: float = 0.75) -> torch.Tensor:
    """Device double[3] = (sum, sum of squares, count) of the central box of the local frames."""
    t, h, w = image.shape
    y0, y1 = int(frac_low * h), int(frac_high * h)
    x0, x1 = int(frac_low * w), int(frac_high * w)
    out = torch.empty((3,), dtype=torch.float64, device=image.device)
    ws = torch.empty(query("tmc_stack_stats_workspace_doubles"), dtype=torch.float64, device=image.device)
    with torch.cuda.device(image.device):
        call("tmc_stack_moments", ptr(image), t, h, w, y0, y1, x0, x1, ptr(out), ptr(ws), stream_ptr(image.device))
    return out


def moments_to_mean_std(moments: torch.Tensor) -> torch.Tensor:
    out = torch.empty((2,), dtype=torch.float32, device=moments.device)
    with torch.cuda.device(moments.device):
        call("tmc_moments_to_mean_std", ptr(moments), ptr(out), stream_ptr(moments.device))
    return out


def xc_postprocess(shifts, field, pixel_spacing, skip_frame, outlier_rejection, outlier_threshold, temporal_smoothing,
                   smoothing_window_size) -> None:
    """In place on ``field`` (2, t, gh, gw) Angstrom: outlier rejection of the (t, gh gw, 2) px ``shifts``, accumulation
    onto the field, Savitzky-Golay smoothing and one joint mean removed (``skip_frame`` -1: none skipped)."""
    _, t, gh, gw = field.shape
    scratch = torch.empty_like(field)
    with torch.cuda.device(field.device):
        call("tmc_xc_postprocess", ptr(shifts), t, gh * gw, float(pixel_spacing), int(skip_frame), int(bool(outlier_rejection)),
             float(outlier_threshold), int(bool(temporal_smoothing)), int(smoothing_window_size), 1, ptr(field), ptr(scratch),
             stream_ptr(field.device))


def global_shifts_to_field(shifts: torch.Tensor, pixel_spacing, reference_frame: int) -> torch.Tensor:
    """(t, 2) px shifts -> (2, t, 1, 1) Angstrom field, zero at ``reference_frame``."""
    t = shifts.shape[0]
    field = _f32((2, t, 1, 1), shifts)
    with torch.cuda.device(shifts.device):
        call("tmc_global_shifts_to_field", ptr(shifts), t, float(pixel_spacing), int(reference_frame), ptr(field),
             stream_ptr(shifts.device))
    return field


def subtract_mean(data: torch.Tensor) -> None:
    """In place: ``data`` (contiguous float32) -= its mean, one joint scalar."""
    with torch.cuda.device(data.device):
        call("tmc_subtract_mean", ptr(data), data.numel(), stream_ptr(data.device))


def spline_eval(coeffs: torch.Tensor, kind: int, tyx: torch.Tensor, out=None, ws=None) -> torch.Tensor:
    """``out`` (n, c) / ``ws`` (tmc_spline_workspace_floats) may be preallocated (allocation-free replays)."""
    c, n0, n1, n2 = coeffs.shape
    lead = tyx.shape[:-1]
    pts = tyx.reshape(-1, 3).contiguous()
    n = pts.shape[0]
    if out is None:
        out = _f32((n, c), coeffs)
    if ws is None:
        ws = _f32((query("tmc_spline_workspace_floats", c, n0, n1, n2),), coeffs)
    with torch.cuda.device(coeffs.device):
        call("tmc_spline_eval", ptr(coeffs), c, n0, n1, n2, kind, ptr(pts), n, ptr(out), ptr(ws), stream_ptr(coeffs.device))
    return out.reshape(*lead, c)


def spline_eval_backward(shape, kind: int, tyx: torch.Tensor, grad_out: torch.Tensor, scale: float = 1.0, out=None,
                         ws=None) -> torch.Tensor:
    c, n0, n1, n2 = shape
    pts = tyx.reshape(-1, 3).contiguous()
    go = grad_out.reshape(-1, c).contiguous()
    n = pts.shape[0]
    grad = _f32((c, n0, n1, n2), pts) if out is None else out
    if ws is None:
        ws = _f32((query("tmc_spline_workspace_floats", c, n0, n1, n2),), pts)
    with torch.cuda.device(pts.device):
        call("tmc_spline_eval_backward", c, n0, n1, n2, kind, ptr(pts), n, ptr(go), float(scale), ptr(grad), ptr(ws),
             stream_ptr(pts.device))
    return grad


def spline_lattice(coeffs, kind, n_frames, lh, lw, coeffs2=None, kind2=0, frame_offset=0, total_frames=None, times=None):
    """(n_frames, c, lh, lw) lattice of the field at t = linspace(0,1,total)[offset + f], or at t = times[f] when
    ``times`` (device float32 (n_frames,)) is given."""
    c, n0, n1, n2 = coeffs.shape
    total = n_frames if total_frames is None else total_frames
    n_ws = query("tmc_spline_workspace_floats", c, n0, n1, n2)
    m0 = m1 = m2 = 1
    if coeffs2 is not None:
        _, m0, m1, m2 = coeffs2.shape
        n_ws += query("tmc_spline_workspace_floats", c, m0, m1, m2)
    ws = _f32((n_ws,), coeffs)
    lattice = _f32((n_frames, c, lh, lw), coeffs)
    with torch.cuda.device(coeffs.device):
        if times is None:
            call("tmc_spline_lattice", ptr(coeffs), c, n0, n1, n2, kind, ptr(coeffs2), m0, m1, m2, kind2, n_frames,
                 frame_offset, total, lh, lw, ptr(lattice), ptr(ws), stream_ptr(coeffs.device))
        else:
            if times.shape != (n_frames,) or times.dtype != torch.float32 or times.device != coeffs.device or \
                    not times.is_contiguous():
                raise ValueError(f"times must be a contiguous float32 ({n_frames},) tensor on {coeffs.device}")
            call("tmc_spline_lattice_times", ptr(coeffs), c, n0, n1, n2, kind, ptr(coeffs2), m0, m1, m2, kind2, n_frames,
                 ptr(times), lh, lw, ptr(lattice), ptr(ws), stream_ptr(coeffs.device))
    return lattice


def group_frames(movie, frame_group):
    """(n_groups, h, w) sums of frame_group consecutive frames of a contiguous fp32 device movie (tmc_group_frames)."""
    t, h, w = movie.shape
    out = _f32((t // frame_group, h, w), movie)
    with torch.cuda.device(movie.device):
        call("tmc_group_frames", ptr(movie), t, h, w, int(frame_group), ptr(out), stream_ptr(movie.device))
    return out


def warp_lattice(image, lattice, pixel_spacing, mean_std=None, out_stack=None, out_sum=None, accumulate_sum=False):
    t, h, w = image.shape
    _, _, lh, lw = lattice.shape
    ws = _f32((query("tmc_warp_workspace_floats", t, w, lh),), image)
    with torch.cuda.device(image.device):
        call("tmc_warp_lattice", ptr(image), t, h, w, ptr(lattice), lh, lw, float(pixel_spacing), ptr(mean_std),
             ptr(out_stack), ptr(out_sum), int(accumulate_sum), ptr(ws), stream_ptr(image.device))


def pixel_shifts(lattice, h, w, pixel_spacing):
    _, lh, lw = lattice.shape
    out = _f32((h, w, 2), lattice)
    with torch.cuda.device(lattice.device):
        call("tmc_pixel_shifts", ptr(lattice), lh, lw, h, w, float(pixel_spacing), ptr(out), stream_ptr(lattice.device))
    return out


def warp_dense_shifts(image, shifts):
    t, h, w = image.shape
    out = torch.empty_like(image)
    with torch.cuda.device(image.device):
        call("tmc_warp_dense_shifts", ptr(image), t, h, w, ptr(shifts), ptr(out), stream_ptr(image.device))
    return out


def pixel_tyx(h, w, t, device, frame_offset=0, total_frames=None):
    total = t if total_frames is None else total_frames
    out = torch.empty((t, h, w, 3), dtype=torch.float32, device=device)
    with torch.cuda.device(device):
        call("tmc_pixel_tyx", h, w, t, frame_offset, total, ptr(out), stream_ptr(device))
    return out
