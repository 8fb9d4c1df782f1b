"""Motion correction with a deformation field (mirror of the reference's ``correct_motion.py``).

All arithmetic runs in hand-written sm_100a kernels behind the C ABI (``csrc/warp.cu``,
``csrc/spline.cu``, ``csrc/fourier.cu``); this file only validates arguments and owns tensors.
"""

from __future__ import annotations

import numpy as np
import torch

from . import _ops
from ._common import as_f32, grid_kind, resolve_device
from .frame_groups import frame_groups


def _movie(image: torch.Tensor, dev: torch.device) -> torch.Tensor:
    if image.ndim != 3:
        raise ValueError(f"image must be (t, h, w), got {tuple(image.shape)}")
    return as_f32(image, dev)


def _field(deformation_grid: torch.Tensor, dev: torch.device) -> torch.Tensor:
    if deformation_grid.ndim != 4 or deformation_grid.shape[0] != 2:
        raise ValueError(f"deformation_grid must be (2, nt, nh, nw), got {tuple(deformation_grid.shape)}")
    return as_f32(deformation_grid, dev)


def _frame_times(frame_group, total, first, stop, dev):
    """Device float32 time of each of the frames first .. stop - 1 of a ``total``-frame movie on the time axis of a field
    estimated with ``estimate_motion(..., frame_group=...)`` (``frame_groups``); None without grouping (None or 1)."""
    if frame_group is None:
        return None
    groups = frame_groups(total, frame_group)
    if groups.group_size == 1:
        return None
    if not 0 <= first < stop <= total:
        raise ValueError(f"frames [{first}, {stop}) outside a movie of {total}")
    return torch.from_numpy(groups.times[first:stop]).to(dev)


def _lattice(field, kind, n_frames, frame_offset=0, total_frames=None, frame_group=None):
    """The warp's (n_frames, 2, 10 gh, 10 gw) lattice for frames frame_offset .. of a total_frames movie."""
    gh, gw = field.shape[-2:]
    total = n_frames if total_frames is None else total_frames
    times = _frame_times(frame_group, total, frame_offset, frame_offset + n_frames, field.device)
    return _ops.spline_lattice(field, kind, n_frames, 10 * gh, 10 * gw, frame_offset=frame_offset, total_frames=total,
                               times=times)


def correct_motion(
    image: torch.Tensor,
    deformation_grid: torch.Tensor,
    pixel_spacing: float,
    grad: bool = False,
    grid_type: str = "catmull_rom",
    device: torch.device = None,
    _mean_std: torch.Tensor | None = None,
    *,
    frame_group: int | None = None,
) -> torch.Tensor:
    """(t, h, w) movie warped by a (yx, nt, nh, nw) Angstrom field -> (t, h, w).

    Reference: correct_motion.py:18-78 (spline -> 10x lattice -> bicubic lattice lookup ->
    bicubic frame gather; quirk Q17).  ``grad`` is accepted for signature compatibility; like
    the reference the result is detached.

    ``frame_group=G``: the field was estimated with ``estimate_motion(..., frame_group=G)`` on this movie, so its time
    axis runs over the group sums; every raw frame is corrected at its place on that axis (``frame_groups``).
    """
    dev = resolve_device(image, device)
    movie = _movie(image, dev)
    field = _field(deformation_grid, dev)
    lattice = _lattice(field, grid_kind(grid_type), movie.shape[0], frame_group=frame_group)
    out = torch.empty_like(movie)
    # _mean_std (internal): warp the normalised movie (image - mean) / std without materialising it
    _ops.warp_lattice(movie, lattice, pixel_spacing, mean_std=_mean_std, out_stack=out)
    return out


def correct_motion_fast(
    image: torch.Tensor,
    deformation_grid: torch.Tensor,
    device: torch.device = None,
    _mean_std: torch.Tensor | None = None,
) -> torch.Tensor:
    """Rigid per-frame Fourier phase shift for a (2, t, 1, 1) field.

    Reference: correct_motion.py:430-498, including quirk Q2: the field is NEGATED IN PLACE (the
    reference's ``shifts`` is a view of the caller's tensor) and its values are used as pixels."""
    from . import _fourier
    from ._lib import call, ptr, stream_ptr

    if tuple(deformation_grid.shape[-2:]) != (1, 1):
        raise ValueError(
            f"Expected single patch deformation field with shape (2, t, 1, 1), "
            f"but got shape {tuple(deformation_grid.shape)}. "
            f"Final two dimensions must be (1, 1) for single patch correction."
        )
    dev = resolve_device(image, device)
    movie = _movie(image, dev)
    t, h, w = movie.shape
    moved = deformation_grid.to(dev)
    moved *= -1  # Q2: the reference negates the caller's tensor in place ...
    if moved.data_ptr() != deformation_grid.data_ptr():
        with torch.no_grad():
            deformation_grid.mul_(-1)  # ... also when .to() had to copy it to the device (CPU callers)
    field = moved.detach().to(torch.float32).contiguous()
    plan = _fourier.BandPlan(h, w, dev, full=True)
    if _fourier.query("tmc_fourier_shift_frames_supported", h, w):
        return plan.shift_frames(movie, _mean_std, field)
    spec = plan.forward(movie, _mean_std, None, 0, h, _fourier.frame_pair_jobs(t, dev), job_mode=2)
    with torch.cuda.device(dev):
        call("tmc_fourier_shift", ptr(spec), t, h, w, ptr(field), 1.0, stream_ptr(dev))
    out = torch.empty_like(movie)
    plan.inverse_full(spec[:t], out)
    return out


def correct_motion_sum(
    image: torch.Tensor,
    deformation_grid: torch.Tensor,
    pixel_spacing: float,
    grid_type: str = "catmull_rom",
    device: torch.device = None,
    out: torch.Tensor | None = None,
    accumulate: bool = False,
    frame_offset: int = 0,
    total_frames: int | None = None,
    *,
    frame_group: int | None = None,
) -> torch.Tensor:
    """Fused ``correct_motion(...).sum(dim=0)`` that never materialises the warped stack.

    New (additive) entry point: the reference leaves the frame sum to the caller
    (``examples/ttMotion.py:398``).  ``frame_offset``/``total_frames`` let one rank warp a
    contiguous block of frames of a larger movie (frame-split multi-GPU).  ``frame_group``: as for
    ``correct_motion``; the groups are those of the whole ``total_frames`` movie."""
    dev = resolve_device(image, device)
    movie = _movie(image, dev)
    field = _field(deformation_grid, dev)
    t, h, w = movie.shape
    lattice = _lattice(field, grid_kind(grid_type), t, frame_offset, total_frames, frame_group)
    if out is None:
        out = torch.empty((h, w), dtype=torch.float32, device=dev)
        accumulate = False
    _ops.warp_lattice(movie, lattice, pixel_spacing, out_sum=out, accumulate_sum=accumulate)
    return out


#: weighted sums per launch of tmc_warp_lattice_sums (larger requests run in passes over the movie)
_MAX_SUMS_PER_PASS = 19
#: bit of each dose-weighted output in the plane masks of tmc_dose_lowrank_combine
_DOSE_OUTPUTS = ("dose_weighted", "dose_weighted_even", "dose_weighted_odd")


def check_sums_arguments(shape, frame_range, dose_per_frame) -> tuple[int, int]:
    """Validate the host-side arguments of correct_motion_sums (no CUDA call); returns (first, stop)."""
    if len(shape) != 3:
        raise ValueError(f"image must be (t, h, w), got {tuple(shape)}")
    t, h, w = shape
    first, stop = (0, t) if frame_range is None else (int(frame_range[0]), int(frame_range[1]))
    if not 0 <= first < stop <= t:
        raise ValueError(f"frame_range must satisfy 0 <= first < stop <= {t} frames, got {frame_range}")
    if dose_per_frame is not None:
        if not dose_per_frame > 0:
            raise ValueError(f"dose_per_frame must be > 0, got {dose_per_frame}")
        from ._fourier import unsupported_lengths

        msg = unsupported_lengths(h, w, True)
        if msg:
            raise ValueError(msg)
    return first, stop


def warp_sums(movie, field, pixel_spacing, kind, frame_offset, total_frames, half_sets, lowrank, pixel_size=None,
              voltage=300.0, times=None) -> dict:
    """Frame sums of ``movie`` (frames frame_offset .. of a movie of total_frames) in one pass of the weighted-sum warp
    (two or more beyond 19 sums), plus the low-rank dose-weighted sums of ``lowrank`` (exposure_filter_lowrank).  Every
    output is linear in the frames, so sums over blocks of one movie add up to the sums over the movie.  ``times``
    (device float32 (t,), optional): the field's time at each frame, instead of its place in linspace(0, 1, total)."""
    from . import _fourier
    from ._lib import call, ptr, query, stream_ptr

    dev = movie.device
    t, h, w = movie.shape
    frames = np.arange(frame_offset, frame_offset + t)
    rows, names = [np.ones(t)], ["sum"]
    if half_sets:
        rows += [(frames % 2 == 0).astype(np.float64), (frames % 2 == 1).astype(np.float64)]
        names += ["sum_even", "sum_odd"]
    n_plain = len(rows)
    dose_names, masks, tables = [], [], []
    if lowrank is not None:
        dose_names = list(_DOSE_OUTPUTS if half_sets else _DOSE_OUTPUTS[:1])
        for name, g in lowrank.groups.items():
            mask = {"all": 1, "even": 1 | 2, "odd": 1 | 4}[name]  # the half sets add up to the whole
            local = g.frames - frame_offset
            keep = (local >= 0) & (local < t)
            for r in range(g.basis.shape[1]):
                row = np.zeros(t)
                row[local[keep]] = g.basis[keep, r]
                rows.append(row)
                masks.append(mask)
                tables.append(g.table[r])
    weights = torch.from_numpy(np.stack(rows).astype(np.float32)).to(dev)
    n_sums = weights.shape[0]
    gh, gw = field.shape[-2:]
    lattice = _ops.spline_lattice(field, kind, t, 10 * gh, 10 * gw, frame_offset=frame_offset, total_frames=total_frames,
                                  times=times)
    lh, lw = lattice.shape[-2:]
    ws = torch.empty((query("tmc_warp_workspace_floats", t, w, lh),), dtype=torch.float32, device=dev)
    sums = torch.empty((n_sums, h, w), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        for s0 in range(0, n_sums, _MAX_SUMS_PER_PASS):
            n = min(_MAX_SUMS_PER_PASS, n_sums - s0)
            call("tmc_warp_lattice_sums", ptr(movie), t, h, w, ptr(lattice), lh, lw, float(pixel_spacing),
                 weights.data_ptr() + s0 * t * 4, n, sums.data_ptr() + s0 * h * w * 4, ptr(ws), stream_ptr(dev))
    # the plain sums are copied out so that the dose planes' memory is freed with `sums`
    plain = sums[:n_plain].clone() if n_sums > n_plain else sums
    out = {name: plain[i] for i, name in enumerate(names)}
    if dose_names:
        n_planes = n_sums - n_plain
        plan = _fourier.BandPlan(h, w, dev, full=True)
        dw = torch.zeros((len(dose_names), h, w), dtype=torch.float32, device=dev)
        if n_planes:  # no planes: this block holds none of the frames of the filter
            spec = plan.forward(sums[n_plain:], None, None, 0, h, _fourier.frame_pair_jobs(n_planes, dev), job_mode=2)
            table = torch.from_numpy(np.stack(tables).astype(np.float32)).to(dev)
            plane_outputs = torch.tensor(masks, dtype=torch.int32).to(dev)
            combined = torch.empty((len(dose_names), h, w // 2 + 1, 2), dtype=torch.float32, device=dev)
            with torch.cuda.device(dev):
                call("tmc_dose_lowrank_combine", ptr(spec), n_planes, h, w, float(pixel_size), float(voltage), ptr(table),
                     table.shape[1], float(lowrank.x_max), ptr(plane_outputs), len(dose_names), ptr(combined),
                     stream_ptr(dev))
            del spec
            plan.inverse_full(combined, dw)
        out.update({name: dw[i] for i, name in enumerate(dose_names)})
    return out


def correct_motion_sums(
    image: torch.Tensor,
    deformation_grid: torch.Tensor,
    pixel_spacing: float,
    grid_type: str = "catmull_rom",
    device: torch.device = None,
    *,
    dose_per_frame: float | None = None,
    pre_exposure: float = 0.0,
    voltage: float = 300.0,
    half_sets: bool = False,
    frame_range: tuple[int, int] | None = None,
    frame_group: int | None = None,
) -> dict[str, torch.Tensor]:
    """Frame sums of the motion-corrected movie, never materialising the corrected stack: {name: (h, w) fp32}.

    * ``"sum"``: ``correct_motion(...).sum(0)``, bit for bit the output of ``correct_motion_sum``;
    * ``half_sets``: ``"sum_even"`` / ``"sum_odd"`` over the frames of even / odd (0-based, global) index -- the half
      sets denoisers train on and resolution estimates compare;
    * ``dose_per_frame`` (e/A^2): ``"dose_weighted"``, the sum ``dose_weight`` forms from the corrected stack (Grant &
      Grigorieff exposure filter, N_t = pre_exposure + (t + 1) dose_per_frame for global frame index t, the same N_e and
      200 kV scaling), and with ``half_sets`` also ``"dose_weighted_even"`` / ``"dose_weighted_odd"``.  The halves use
      the normalisation of all included frames, so dose_weighted_even + dose_weighted_odd == dose_weighted.

    The exposure weights are applied through a low-rank factorisation (``dose_weight.exposure_filter_lowrank``: worst
    residual 1e-6 per frequency, R <= 8 components for real exposures): R frame-weighted sums formed while warping, R
    full-frame transforms and one inverse per output, independent of the number of frames.

    ``frame_range=(first, stop)`` restricts every sum to frames first .. stop - 1: only those frames are read, the field
    is evaluated at their place in the whole movie, exposure still counts all earlier frames and the dose
    normalisation runs over the included frames.

    ``frame_group=G``: the field was estimated with ``estimate_motion(..., frame_group=G)`` on this movie; every raw frame
    is warped at its time on the group axis (``frame_groups``), while half sets and exposures stay those of the raw
    frames."""
    first, stop = check_sums_arguments(image.shape, frame_range, dose_per_frame)
    kind = grid_kind(grid_type)
    dev = resolve_device(image, device)
    total = image.shape[0]
    times = _frame_times(frame_group, total, first, stop, dev)
    movie = _movie(image[first:stop], dev)
    field = _field(deformation_grid, dev)
    lowrank = None
    if dose_per_frame is not None:
        from .dose_weight import exposure_filter_lowrank

        h, w = movie.shape[-2:]
        lowrank = exposure_filter_lowrank(h, w, pixel_spacing, range(first, stop), dose_per_frame, pre_exposure,
                                          voltage, half_sets)
    return warp_sums(movie, field, pixel_spacing, kind, first, total, half_sets, lowrank, pixel_spacing, voltage, times)


def get_pixel_shifts(
    frame: torch.Tensor,
    pixel_spacing: float,
    frame_deformation_grid: torch.Tensor,
    pixel_grid: torch.Tensor = None,
) -> torch.Tensor:
    """(h, w, yx) px shifts from a (yx, gh, gw) Angstrom lattice.  Reference: correct_motion.py:132-185.

    ``pixel_grid`` is accepted for signature compatibility (the kernel derives the integer pixel
    coordinates from thread indices)."""
    dev = resolve_device(frame, None)
    h, w = frame.shape[-2:]
    lattice = as_f32(frame_deformation_grid, dev)
    return _ops.pixel_shifts(lattice, h, w, pixel_spacing)


def correct_motion_slow(
    image: torch.Tensor,
    deformation_grid: torch.Tensor,
    grad: bool = False,
    device: torch.device = None,
) -> torch.Tensor:
    """Exact per-pixel Catmull-Rom evaluation of the field (no lattice, no /pixel_spacing).

    Reference: correct_motion.py:320-427."""
    dev = resolve_device(image, device)
    movie = _movie(image, dev)
    field = _field(deformation_grid, dev)
    t, h, w = movie.shape
    out = torch.empty_like(movie)
    # one frame at a time bounds the (h, w, 3) + (h, w, 2) temporaries
    for f in range(t):
        tyx = _ops.pixel_tyx(h, w, 1, dev, frame_offset=f, total_frames=t)
        shifts = _ops.spline_eval(field, 0, tyx)  # (1, h, w, 2)
        out[f : f + 1] = _ops.warp_dense_shifts(movie[f : f + 1], shifts)
    return out


def _grid_data(grid) -> tuple[torch.Tensor, int]:
    """Accept a spline-grid module (anything with ``.data`` of shape (2, nt, nh, nw)) or a tensor."""
    data = grid.data if hasattr(grid, "data") and not isinstance(grid, torch.Tensor) else grid
    kind = getattr(grid, "grid_kind", None)
    if kind is None:
        name = type(grid).__name__.lower()
        kind = 1 if "bspline" in name else 0
    return data, kind


def correct_motion_two_grids(
    image: torch.Tensor,
    new_deformation_grid,
    base_deformation_grid,
    pixel_spacing: float,
    grad: bool = True,
    device: torch.device = None,
) -> torch.Tensor:
    """Warp with shifts = new(tyx) + base(tyx).  Reference: correct_motion.py:188-317.

    With ``grad=True`` the result carries a graph to ``new_deformation_grid``'s coefficients
    (see ``_autograd.WarpTwoGrids``)."""
    dev = resolve_device(image, device)
    movie = _movie(image, dev)
    new_data, new_kind = _grid_data(new_deformation_grid)
    base_data, base_kind = _grid_data(base_deformation_grid)
    if grad and torch.is_tensor(new_data) and new_data.requires_grad:
        from ._autograd import WarpTwoGrids

        return WarpTwoGrids.apply(new_data, movie, as_f32(base_data, dev), float(pixel_spacing), new_kind, base_kind)
    new_f, base_f = as_f32(new_data, dev), as_f32(base_data, dev)
    t = movie.shape[0]
    gh, gw = new_f.shape[-2:]
    lattice = _ops.spline_lattice(new_f, new_kind, t, 10 * gh, 10 * gw, coeffs2=base_f, kind2=base_kind)
    out = torch.empty_like(movie)
    _ops.warp_lattice(movie, lattice, pixel_spacing, out_stack=out)
    return out
