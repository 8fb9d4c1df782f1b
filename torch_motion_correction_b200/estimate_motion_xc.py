"""Cross-correlation motion estimators (mirror of the reference's ``estimate_motion_xc.py``).

Host code only plans the work (patch geometry, the cache-aliasing schedule of quirk Q1, job
lists); every arithmetic step runs in ``csrc/fourier.cu`` / ``csrc/postprocess.cu``.  No step
synchronises with the host."""

from __future__ import annotations

import torch

from . import _fourier, _ops
from ._common import as_f32, cached_device_tensor, resolve_device
from .correct_motion import correct_motion, correct_motion_fast
from .deformation_field_utils import resample_deformation_field
from .patch_grid import patch_grid_centers


def estimate_global_motion(
    image: torch.Tensor,
    pixel_spacing: float,
    reference_frame: int | None = None,
    b_factor: float = 500,
    frequency_range: tuple[float, float] = (300, 10),
    device: torch.device = None,
    _stats: torch.Tensor | None = None,
) -> torch.Tensor:
    """Integer-pixel whole-frame cross-correlation against one frame -> (2, t, 1, 1) Angstrom field.

    Reference: estimate_motion_xc.py:21-135 (quirk Q5: integer shifts, reference frame t // 2)."""
    dev = resolve_device(image, device)
    movie = as_f32(image, dev)
    t, h, w = movie.shape
    if reference_frame is None:
        reference_frame = t // 2
    stats = _stats if _stats is not None else _ops.stack_stats(movie)  # _stats: the pipeline computes them once per movie
    plan, spec = global_spectra(movie, stats, pixel_spacing, b_factor, frequency_range)
    cur = torch.arange(t, dtype=torch.int32, device=dev)
    ref = torch.full((t,), int(reference_frame), dtype=torch.int32, device=dev)
    prod = _fourier.pair_products(spec, ref, cur, plan.plane_elems)
    shifts = plan.peaks(prod.view(t, plan.ky, plan.kx, 2), sub_pixel=False)
    return _ops.global_shifts_to_field(shifts, pixel_spacing, reference_frame)


def global_spectra(frames: torch.Tensor, stats, pixel_spacing, b_factor, frequency_range):
    """(plan, band-limited whole-frame spectra of ``frames`` (plane k = frame k)) under the soft disc of the whole-frame
    cross-correlation."""
    t, h, w = frames.shape
    dev = frames.device
    plan = _fourier.BandPlan(h, w, dev, pixel_spacing, b_factor, frequency_range)
    mask, ylo, yhi = _fourier.soft_disc_mask((h, w), min(h, w) / 4, min(h, w) / 8, dev)
    return plan, plan.forward(frames, stats, mask, ylo, yhi, _fourier.frame_pair_jobs(t, dev), job_mode=2)


class _CacheModel:
    """Which frames the reference's ``LazyPatchGrid`` cache holds, and how many times each cached
    frame has been multiplied by the mask in place (quirk Q1).

    Mirrors the observable behaviour of patch_grid/_patch_grid.py:264-347: a dict plus a set of
    keys, more than 50 entries => the first half of ``list(keys)`` is dropped.  Using the same
    container types keeps the eviction order identical."""

    def __init__(self, limit: int = 50):
        self.limit = limit
        self.masked: dict[int, int] = {}
        self.keys: set[int] = set()

    def get(self, frame: int) -> int:
        if frame in self.masked:
            return self.masked[frame]
        self.masked[frame] = 0
        self.keys.add(frame)
        if len(self.masked) > self.limit:
            for victim in list(self.keys)[: len(self.keys) // 2]:
                self.masked.pop(victim, None)
                self.keys.discard(victim)
        return 0

    def mask(self, frame: int) -> None:
        if frame in self.masked:  # an entry evicted at creation is mutated outside the cache
            self.masked[frame] += 1


def _aliasing_schedule(t: int, strategy: str, reference_frame: int):
    """For ``mean_except_current``: (delta_offsets, deltas) describing, frame by frame, which other
    frames are already masked in the cache; for ``middle_frame``: the mask power carried by the
    reference frame when each frame is processed (list of length t, 0 for the reference itself)."""
    cache = _CacheModel()
    if strategy == "middle_frame":
        power = [0] * t
        for k in range(t):
            if k == reference_frame:
                continue
            power[k] = cache.get(reference_frame) + 1
            cache.mask(reference_frame)
            cache.get(k)
            cache.mask(k)
        return power
    offsets, deltas, prev = [0], [], [0] * t
    for k in range(t):
        row = [0] * t
        for j in range(t):
            if j != k:
                row[j] = cache.get(j)
        cache.get(k)
        cache.mask(k)
        for j in range(t):
            if row[j] != prev[j]:
                deltas.append((j + 1) if row[j] else -(j + 1))
        offsets.append(len(deltas))
        prev = row
    return offsets, deltas


def patch_xc_geometry(shape, p: int, pixel_spacing, b_factor, frequency_range, base_field, dev):
    """Patch grid of the cross-correlation of a (t, h, w) movie with p x p patches at 50 % overlap: (device centres
    (t, gh, gw, 3), window origins [y0, x0] of every patch, plan, (mask, ylo, yhi), initial (2, t, gh, gw) field: zeros,
    or ``base_field`` resampled onto the grid)."""
    t, h, w = shape
    centers = patch_grid_centers((t, h, w), (1, p, p), (1, p // 2, p // 2), distribute_patches=True)
    gh, gw = centers.shape[1:3]
    origins = (centers[0, :, :, 1:] - p // 2).reshape(-1, 2).tolist()
    plan = _fourier.BandPlan(p, p, dev, pixel_spacing, b_factor, frequency_range)
    mask = _fourier.soft_disc_mask((p, p), p / 4, p / 8, dev)
    if base_field is None:
        field = torch.zeros((2, t, gh, gw), dtype=torch.float32, device=dev)
    else:
        field = resample_deformation_field(base_field, (t, gh, gw))
    return cached_device_tensor(("patch_centres", (t, h, w, p)), lambda: centers, dev), origins, plan, mask, field


def mean_except_current_spectra(source, source_stats, plan, mask, p: int, origins, frame_shifts):
    """(jobs, spectra) of every (frame, patch) of ``source`` under mask powers 1 and 2 (quirk Q1), frame-major: planes
    (frame, patch, power)."""
    t, h, w = source.shape
    jobs = cached_device_tensor(
        ("xc_jobs_mean", (t, h, w, p)),
        lambda: torch.tensor([[k, 1, k, 2, y0, x0] for k in range(t) for (y0, x0) in origins], dtype=torch.int32),
        source.device)
    return jobs, plan.forward(source, source_stats, *mask, jobs, job_mode=1, frame_shifts=frame_shifts)


def leave_one_out_shifts(spec: torch.Tensor, t: int, g: int, plan, sub_pixel) -> torch.Tensor:
    """(t * g, 2) px peak shifts of every (frame, patch) against the sum of the other frames, from the frame-major
    spectra of both mask powers of ALL t frames (``mean_except_current``; the mask powers of the leave-one-out
    references follow the reference's patch cache, quirk Q1)."""
    dev = spec.device

    def schedule(part):
        offsets, deltas = _aliasing_schedule(t, "mean_except_current", t // 2)
        return torch.tensor(offsets if part == 0 else (deltas if deltas else [0]), dtype=torch.int32)

    d_off = cached_device_tensor(("xc_delta_offsets", t), lambda: schedule(0), dev)
    d_val = cached_device_tensor(("xc_deltas", t), lambda: schedule(1), dev)
    prod = _fourier.leave_one_out_products(spec, t, g, plan.plane_elems, d_off, d_val)
    return plan.peaks(prod.view(t * g, plan.ky, plan.kx, 2), sub_pixel=bool(sub_pixel))


def estimate_motion_cross_correlation_patches(
    image: torch.Tensor,
    pixel_spacing: float,
    reference_frame: int | None = None,
    reference_strategy: str = "mean_except_current",
    b_factor: float = 500,
    frequency_range: tuple[float, float] = (300, 10),
    patch_sidelength: int = 1024,
    sub_pixel_refinement: bool = True,
    temporal_smoothing: bool = True,
    smoothing_window_size: int = 5,
    deformation_field: torch.Tensor = None,
    outlier_rejection: bool = True,
    outlier_threshold: float = 3.0,
    device: torch.device = None,
    dose_per_frame: float | None = None,
    pre_exposure: float = 0.0,
    voltage: float = 300.0,
    _stats: torch.Tensor | None = None,
    _whole_pixel_field: bool | None = None,
) -> tuple[torch.Tensor, torch.Tensor]:
    """Patch-wise Fourier cross-correlation -> ((2, t, gh, gw) Angstrom field, (t, gh, gw, 3) centres).

    ``dose_per_frame`` (additive, default off = the reference's behaviour): every frame's patch spectra are also
    multiplied by the exposure filter ``q_t / sqrt(sum_t q_t^2)`` (Grant & Grigorieff; the filter the reference's
    example applies to the corrected stack) before the leave-one-out sums and the cross-correlation.

    Reference: estimate_motion_xc.py:138-411, including the result-changing quirks Q1 (cached patches
    are masked in place, so earlier frames enter later references double-masked), Q2/Q3 (rigid
    pre-correction negates the caller's field in place and uses Angstrom as px; full pre-correction
    uses the B-spline, resampling uses Catmull-Rom), Q4, Q6-Q9.

    A rigid (2, t, 1, 1) field whose values are whole numbers (the integer estimate of ``estimate_global_motion``, quirk
    Q5, handed over in pixels) needs no pre-correction pass: an integer Fourier shift is a circular roll, so every
    frame's patch windows are simply read at origins moved by that frame's shift (wrapping around the frame edges).  The
    check costs one host synchronisation; ``_whole_pixel_field`` (internal) vouches for it (True) or forces the
    Fourier-shift pass (False)."""
    dev = resolve_device(image, device)
    movie = as_f32(image, dev)
    t, h, w = movie.shape
    if reference_frame is None:
        reference_frame = t // 2
    if reference_strategy not in ("middle_frame", "mean_except_current"):
        raise ValueError(f"Unknown reference_strategy: {reference_strategy}")
    if reference_strategy == "mean_except_current" and t < 2:
        raise ValueError("mean_except_current needs at least two frames")
    stats = _stats if _stats is not None else _ops.stack_stats(movie)  # _stats: the pipeline computes them once per movie

    source, source_stats = movie, stats  # patches are read from here, normalised on load
    frame_shifts = None
    if deformation_field is not None:
        callers_field = deformation_field
        deformation_field = deformation_field.to(dev)
        if tuple(deformation_field.shape[-2:]) == (1, 1):
            if deformation_field.shape[1] != t:
                raise ValueError(f"deformation_field has {deformation_field.shape[1]} frames, the movie {t}")
            whole = _whole_pixel_field
            if whole is not False:
                shifts, not_whole = _fourier.integer_shifts(deformation_field)
                if whole is None:
                    whole = int(not_whole.item()) == 0  # the one host synchronisation of this function
            if whole:
                frame_shifts = shifts
                deformation_field *= -1  # quirk Q2: correct_motion_fast negates the caller's field in place
                if deformation_field.data_ptr() != callers_field.data_ptr():
                    with torch.no_grad():
                        callers_field.mul_(-1)  # a CPU caller's tensor was copied to the device: negate the original too
            else:
                source = correct_motion_fast(movie, deformation_field, device=dev, _mean_std=stats)
                source_stats = None
                if deformation_field.data_ptr() != callers_field.data_ptr():
                    with torch.no_grad():
                        callers_field.mul_(-1)  # quirk Q2 for a CPU caller's tensor (negated on the device copy above)
        else:
            source = correct_motion(movie, deformation_field, pixel_spacing, grid_type="bspline", device=dev, _mean_std=stats)
            source_stats = None

    p = int(patch_sidelength)
    centres, origins, plan, mask, field = patch_xc_geometry((t, h, w), p, pixel_spacing, b_factor, frequency_range,
                                                            deformation_field, dev)
    n_patches = len(origins)

    skip = -1
    if reference_strategy == "mean_except_current":
        jobs, spec = mean_except_current_spectra(source, source_stats, plan, mask, p, origins, frame_shifts)
        if dose_per_frame is not None:
            plan.dose_filter(spec, jobs, t, pixel_spacing, pre_exposure, dose_per_frame, voltage)
        shifts = leave_one_out_shifts(spec, t, n_patches, plan, sub_pixel_refinement)
    else:
        skip = int(reference_frame)

        def middle_jobs():
            power = _aliasing_schedule(t, reference_strategy, reference_frame)
            return torch.tensor(
                [[k, 1, reference_frame, max(power[k], 1), y0, x0] for k in range(t) for (y0, x0) in origins], dtype=torch.int32
            )

        jobs = cached_device_tensor(("xc_jobs_middle", (t, h, w, p), int(reference_frame)), middle_jobs, dev)
        spec = plan.forward(source, source_stats, *mask, jobs, frame_shifts=frame_shifts)
        if dose_per_frame is not None:
            plan.dose_filter(spec, jobs, t, pixel_spacing, pre_exposure, dose_per_frame, voltage)
        items = torch.arange(t * n_patches, dtype=torch.int32, device=dev)
        prod = _fourier.pair_products(spec, 2 * items + 1, 2 * items, plan.plane_elems)
        shifts = plan.peaks(prod.view(t * n_patches, plan.ky, plan.kx, 2), sub_pixel=bool(sub_pixel_refinement))

    _ops.xc_postprocess(shifts, field, pixel_spacing, skip, outlier_rejection, outlier_threshold, temporal_smoothing,
                        smoothing_window_size)
    return field, centres.clone()
