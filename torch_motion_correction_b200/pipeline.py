"""End-to-end drivers built from the reference-compatible entry points (additive API).

``estimate_motion`` = global (whole-frame XC) -> patch XC on the rigidly pre-corrected movie ->
optional spline-coefficient optimisation; ``motion_correct`` = estimate + fused warp-and-sum.
This is the workflow the reference sketches in ``examples/ttMotion.py:287-329,383-398``."""

from __future__ import annotations

import torch

from .correct_motion import correct_motion_sum
from .estimate_motion_xc import estimate_global_motion, estimate_motion_cross_correlation_patches


def cumulative_patch_field(global_field: torch.Tensor, pixel_spacing: float, patch_estimator, smoothing_window_size: int = 5):
    """Patch cross-correlation on top of a rigid (2, t, 1, 1) Angstrom field, composed so that the result is
    ``smooth(global + patch residuals)``.

    The reference-compatible estimator takes the rigid field through ``correct_motion_fast``, which uses Angstrom values
    as pixels and negates the caller's tensor in place, and then accumulates the patch shifts onto the NEGATED field
    (quirk Q2; the reference's own example loop, ``examples/ttMotion.py:287-329``, only recovers from that in its later
    iterations).  Here the estimator is handed ``global / pixel_spacing`` -- so the pre-correction moves every frame by
    exactly minus its shift in pixels -- WITHOUT temporal smoothing; the base it accumulated on is swapped for the true
    global field, and only then the Savitzky-Golay filter and the single joint mean subtraction (quirks Q9, Q4) are applied
    to the composed field.  (Smoothing before the swap would leave the smoothing residual of the integer-quantised
    global track, quirk Q5, in the result.)
    ``patch_estimator(pre)`` must return ``(field (2, t, gh, gw), centres)`` computed with ``temporal_smoothing=False``
    and may negate ``pre`` in place or not."""
    from . import _ops
    from .deformation_field_utils import resample_deformation_field

    pre = global_field / float(pixel_spacing)
    handed = pre.clone()
    xc_field, centres = patch_estimator(pre)
    t, gh, gw = xc_field.shape[1:]
    used_base = resample_deformation_field(-handed, (t, gh, gw))  # what the estimator accumulated the patch shifts on
    field = (xc_field - used_base + resample_deformation_field(global_field, (t, gh, gw))).contiguous()
    zero_shifts = torch.zeros((t, gh * gw, 2), dtype=torch.float32, device=field.device)
    # smoothing + one joint mean (quirk Q4) of the composed field: the estimator's own tail with nothing to add
    _ops.xc_postprocess(zero_shifts, field, pixel_spacing, -1, False, 0.0, True, smoothing_window_size)
    return field, centres


def estimate_motion(
    image: torch.Tensor,
    pixel_spacing: float,
    patch_sidelength: int = 1024,
    deformation_field_resolution: tuple[int, int, int] | None = None,
    n_iterations: int = 0,
    b_factor: float = 500,
    frequency_range: tuple[float, float] = (300, 10),
    grid_type: str = "bspline",
    optimizer_kwargs: dict | None = None,
    device: torch.device = None,
    dose_per_frame: float | None = None,
    pre_exposure: float = 0.0,
    voltage: float = 300.0,
    n_refinements: int = 0,
    refinement_tolerance: float = 1e-3,
    return_history: bool = False,
    frame_group: int | None = None,
):
    """Returns ``(field (2, nt, nh, nw) Angstrom, patch_centres)`` (and the refinement history with ``return_history``).

    ``frame_group=G`` (int >= 2; None or 1: off) estimates on the sums of G consecutive frames (``group_frames``: the
    last group also takes the t % G leftover frames) instead of on single frames -- MotionCor2's ``-Group``, for finely
    fractionated movies whose single frames hold too few electrons for a usable cross-correlation peak.  Everything
    below runs unchanged on the t // G group sums, so the returned field's time axis runs over the GROUPS: correct
    the raw frames with ``correct_motion*(..., frame_group=G)``, which evaluate it at each frame's place between the
    group centres (``frame_groups``).  The patch-XC exposure pre-filter treats a group as one frame of G *
    ``dose_per_frame``, so group g is filtered at the exposure at the end of its last frame; for a last group with
    leftover frames that under-counts its exposure by t % G frames.

    ``dose_per_frame`` switches on the exposure pre-filter of the patch cross-correlation.

    ``n_refinements > 0``: the iterative refinement the reference sketches in ``examples/ttMotion.py:287-329`` -- up to
    that many further passes of the patch cross-correlation, each on the movie pre-corrected with the cumulative field
    of the pass before (``deformation_field=`` route: B-spline warp, residual shifts accumulated on the field, smoothed).
    It stops early when the mean absolute change of the field drops below ``refinement_tolerance`` Angstrom (the
    criterion the example prints and leaves commented out, ``:311-316``; one host synchronisation per pass).

    With ``n_iterations > 0`` the patch-XC field initialises ``estimate_local_motion`` on a
    ``deformation_field_resolution`` spline grid (default (3, 5, 5), BASELINE config 2)."""
    # normalisation statistics of the movie: computed once, shared by the three estimators (the reference's
    # normalize_image recomputes them in each, utils.py:49-84)
    from . import _ops
    from ._common import as_f32, resolve_device

    if frame_group is not None:
        from .frame_groups import frame_groups
        from .prepare import group_frames

        group_size = frame_groups(image.shape[0], frame_group).group_size
        if group_size > 1:
            image = group_frames(image, group_size, device=device)  # freed when this call returns
            if dose_per_frame is not None:
                dose_per_frame = dose_per_frame * group_size
    stats = _ops.stack_stats(as_f32(image, resolve_device(image, device)))
    global_field = estimate_global_motion(
        image, pixel_spacing, b_factor=b_factor, frequency_range=frequency_range, device=device, _stats=stats
    )
    field, centres = cumulative_patch_field(
        global_field, pixel_spacing,
        lambda pre: estimate_motion_cross_correlation_patches(
            image, pixel_spacing, b_factor=b_factor, frequency_range=frequency_range, patch_sidelength=patch_sidelength,
            deformation_field=pre, device=device, dose_per_frame=dose_per_frame, pre_exposure=pre_exposure, voltage=voltage,
            temporal_smoothing=False, _stats=stats,
            _whole_pixel_field=True,  # estimate_global_motion returns whole pixels (quirk Q5): no pre-correction pass, no sync
        ),
    )
    history = []
    for _ in range(int(n_refinements)):
        refined, _ = estimate_motion_cross_correlation_patches(
            image, pixel_spacing, b_factor=b_factor, frequency_range=frequency_range, patch_sidelength=patch_sidelength,
            deformation_field=field.clone(), device=device, dose_per_frame=dose_per_frame, pre_exposure=pre_exposure,
            voltage=voltage, _stats=stats,
        )
        change = float((refined - field).abs().mean())
        history.append(change)
        field = refined
        if change < refinement_tolerance:
            break
    if n_iterations > 0:
        from .estimate_motion_optimizer import estimate_local_motion

        resolution = deformation_field_resolution or (3, 5, 5)
        field = estimate_local_motion(
            image, pixel_spacing, (patch_sidelength, patch_sidelength), resolution, field, device=device,
            n_iterations=n_iterations, b_factor=b_factor, frequency_range=frequency_range, grid_type=grid_type,
            optimizer_kwargs=optimizer_kwargs, _stats=stats,
        )
    if return_history:
        return field, centres, history
    return field, centres


def motion_correct(image: torch.Tensor, pixel_spacing: float, grid_type: str = "bspline", device=None,
                   dose_per_frame: float | None = None, pre_exposure: float = 0.0, voltage: float = 300.0,
                   frame_group: int | None = None, fourier_bin: float | None = None, **estimate_kwargs):
    """Estimate + correct: returns ``(aligned frame sum (h, w), field)``.

    With ``dose_per_frame`` (e-/A^2 per frame) the patch cross-correlation is exposure pre-filtered and the sum is dose
    weighted (``examples/ttMotion.py:331-351,383-398``: correct -> per-frame exposure filter -> sum), which needs the
    corrected stack instead of the fused sum.

    ``frame_group=G``: estimate on the sums of G consecutive frames (``estimate_motion``), then correct every raw frame
    with that field.  The dose-weighted sum is then formed without materialising the corrected stack
    (``correct_motion_sums``), since grouping is meant for movies of hundreds of frames.

    ``fourier_bin=b`` (real >= 1; None or 1: off) Fourier-crops the movie by b first (``fourier_crop``: MotionCor2's
    ``-FtBin``, for super-resolution movies) and runs everything on the cropped movie at ``b * pixel_spacing``:
    estimation, frame grouping, the exposure pre-filter and the (dose-weighted) sum.  The sum is returned binned,
    (h / b, w / b), and the field in Angstrom as always; ``patch_sidelength`` and the other keywords given in pixels are
    then binned pixels.  To estimate binned but correct at full resolution, pass the field with the original movie and
    pixel spacing to ``correct_motion_sums`` and crop the result (see ``fourier_crop``)."""
    if fourier_bin is not None:
        from .prepare import fourier_crop

        binned = fourier_crop(image, fourier_bin, device=device)  # checks fourier_bin; factor 1 returns image itself
        if binned is not image:
            image, pixel_spacing = binned, fourier_bin * pixel_spacing  # the binned movie is freed when this call returns
    field, _ = estimate_motion(image, pixel_spacing, grid_type=grid_type, device=device, dose_per_frame=dose_per_frame,
                               pre_exposure=pre_exposure, voltage=voltage, frame_group=frame_group, **estimate_kwargs)
    if dose_per_frame is None:
        total = correct_motion_sum(image, field, pixel_spacing, grid_type=grid_type, device=device, frame_group=frame_group)
    elif frame_group is not None and frame_group != 1:
        from .correct_motion import correct_motion_sums

        total = correct_motion_sums(image, field, pixel_spacing, grid_type, device, dose_per_frame=dose_per_frame,
                                    pre_exposure=pre_exposure, voltage=voltage, frame_group=frame_group)["dose_weighted"]
    else:
        from .correct_motion import correct_motion
        from .dose_weight import dose_weight

        corrected = correct_motion(image, field, pixel_spacing, grid_type=grid_type, device=device)
        total = dose_weight(corrected, pixel_spacing, pre_exposure, dose_per_frame, voltage, device=device)
    return total, field


def motion_correct_many(host_movies, pixel_spacing: float, device=None, out_host=None, gain=None, hot_pixel_threshold=None,
                        zero_frame_means=False, eer_frames_per_fraction: int | None = None, **kwargs):
    """Align a sequence of movies held in (ideally pinned) HOST memory; yields ``(sum_host, field)``.

    Movies may arrive in their detector-native type (uint8 / int8 / uint16 / int16 / float16, or float32): they cross PCIe as
    they are (1-2 bytes per pixel instead of 4) and are converted on the device, together with the optional preparation of
    ``prepare_movie`` (``gain`` multiply, hot-pixel replacement, per-frame mean removal; examples/ttMotion.py:90-202).

    The H2D copy of movie i+1 runs on a side stream while movie i is being estimated and corrected
    (two device buffers), and each result is copied back asynchronously: dataset-scale processing
    is bounded by max(PCIe, compute) instead of their sum (SURVEY.md §8f rank 2).

    The result of movie i is yielded only after movie i+1 has been enqueued and after the device-to-host copy of its sum
    has completed (a CUDA event is waited for), so ``sum_host`` is always safe to read; the overlap is kept because the
    GPU is already busy with movie i+1 while the host waits.  With ``out_host`` the same buffer is reused for every
    movie: consume it before advancing the generator.

    Items may also be EER movies (``read_eer`` / ``eer_movies``), which need ``eer_frames_per_fraction=F``: only their
    compressed payload and frame table cross PCIe, into staging buffers that grow to the largest payload seen; they are
    rendered on the device into a reused counts buffer (``render_eer``: n_frames // F fractions, the trailing frames
    dropped) and go on as uint8 / uint16 movies.  ``dose_per_frame`` is then the dose of one fraction.  A movie with
    malformed frames raises ``ValueError`` when its result would be handed out."""
    from .movie_io import EerMovie

    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    movies = iter(host_movies)
    copy_stream = torch.cuda.Stream(device=dev)
    main = torch.cuda.current_stream(dev)
    buffers = [None, None]
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]

    prepared = [None]  # one fp32 buffer: movie i is prepared into it while movie i + 1 is still in flight over PCIe
    gain_dev = gain.to(device=dev, dtype=torch.float32).contiguous() if gain is not None else None

    eer_items = [None, None]  # the EerMovie staged in each slot (None: a tensor in buffers[slot])
    eer_stage = [[None, None], [None, None]]  # per slot: device payload and frame-table buffers, grown, never shrunk
    counts = [None]  # rendered EER counts of the current movie

    def start_eer_copy(slot, eer):
        from .prepare import eer_fractions

        if eer_frames_per_fraction is None:
            raise ValueError("motion_correct_many: EER movies need eer_frames_per_fraction=")
        n, _ = eer_fractions(eer, eer_frames_per_fraction)
        used = n * eer_frames_per_fraction
        nbytes = int(eer.frame_offsets[used])
        stage = eer_stage[slot]
        grown = False
        if stage[0] is None or stage[0].numel() < nbytes:
            stage[0] = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
            grown = True
        if stage[1] is None or stage[1].numel() < used + 1:
            stage[1] = torch.empty((used + 1,), dtype=torch.int64, device=dev)
            grown = True
        eer_items[slot] = eer
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[slot])
            if grown:  # fresh memory from the main stream's pool: its earlier users must be done with it
                copy_stream.wait_stream(main)
            stage[0][:nbytes].copy_(eer.payload[:nbytes], non_blocking=True)
            stage[1][:used + 1].copy_(eer.frame_offsets[:used + 1], non_blocking=True)
            ready[slot].record(copy_stream)

    def start_copy(slot, host):
        if isinstance(host, EerMovie):
            start_eer_copy(slot, host)
            return
        eer_items[slot] = None
        if buffers[slot] is None or buffers[slot].shape != host.shape or buffers[slot].dtype != host.dtype:
            buffers[slot] = torch.empty(host.shape, dtype=host.dtype, device=dev)
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[slot])  # the previous occupant of this buffer has been processed
            buffers[slot].copy_(host, non_blocking=True)
            ready[slot].record(copy_stream)

    try:
        nxt = next(movies)
    except StopIteration:
        return
    consumed[0].record(main)
    consumed[1].record(main)
    start_copy(0, nxt)
    slot = 0
    pending = None  # (host sum, field, event after its D2H copy) of the previous movie
    d2h_stream = torch.cuda.Stream(device=dev)
    while nxt is not None:
        try:
            upcoming = next(movies)
        except StopIteration:
            upcoming = None
        if upcoming is not None:
            start_copy(1 - slot, upcoming)
        main.wait_event(ready[slot])
        status = None
        if eer_items[slot] is not None:
            from .prepare import eer_counts_buffer, eer_fractions, render_eer_into

            eer = eer_items[slot]
            n, dtype = eer_fractions(eer, eer_frames_per_fraction)
            if counts[0] is None or counts[0].shape != (n, eer.h, eer.w) or counts[0].dtype != dtype:
                counts[0] = eer_counts_buffer((n, eer.h, eer.w), dtype, dev)
            used = n * eer_frames_per_fraction
            status = torch.empty((used,), dtype=torch.int32, device=dev)
            with torch.cuda.device(dev):
                render_eer_into(eer_stage[slot][0][:int(eer.frame_offsets[used])], eer_stage[slot][1][:used + 1], eer,
                                eer_frames_per_fraction, counts[0], status)
            consumed[slot].record(main)  # the staging buffers are free as soon as the movie has been rendered
            movie = counts[0]
        else:
            movie = buffers[slot]
        if movie.dtype != torch.float32 or gain_dev is not None or hot_pixel_threshold is not None or zero_frame_means:
            from .prepare import prepare_movie

            if prepared[0] is None or prepared[0].shape != movie.shape:
                prepared[0] = torch.empty(movie.shape, dtype=torch.float32, device=dev)
            movie = prepare_movie(movie, gain=gain_dev, hot_pixel_threshold=hot_pixel_threshold,
                                  zero_frame_means=zero_frame_means, device=dev, out=prepared[0])
            consumed[slot].record(main)  # the staging buffer is free as soon as it has been converted
            total, field = motion_correct(movie, pixel_spacing, device=dev, **kwargs)
        else:
            total, field = motion_correct(movie, pixel_spacing, device=dev, **kwargs)
            consumed[slot].record(main)
        if pending is not None and out_host is not None:
            yield _hand_out(pending)  # one shared host buffer: hand the previous result out before overwriting it
            pending = None
        host_sum = out_host if out_host is not None else torch.empty(total.shape, dtype=torch.float32, pin_memory=True)
        host_status = torch.empty(status.shape, dtype=torch.int32, pin_memory=True) if status is not None else None
        done = torch.cuda.Event()
        d2h_stream.wait_stream(main)
        with torch.cuda.stream(d2h_stream):
            host_sum.copy_(total, non_blocking=True)
            if status is not None:
                host_status.copy_(status, non_blocking=True)
            done.record(d2h_stream)
        total.record_stream(d2h_stream)
        if status is not None:
            status.record_stream(d2h_stream)
        if pending is not None:
            yield _hand_out(pending)
        pending = (host_sum, field, done, host_status)
        nxt, slot = upcoming, 1 - slot
    if pending is not None:
        yield _hand_out(pending)


def _hand_out(pending):
    """Wait for a result's device-to-host copy; raise if its EER render reported malformed frames."""
    host_sum, field, done, host_status = pending
    done.synchronize()
    if host_status is not None:
        from .prepare import check_eer_status

        check_eer_status(host_status)
    return host_sum, field
