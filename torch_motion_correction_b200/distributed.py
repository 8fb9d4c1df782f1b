"""Multi-GPU sharding of the hot path (one process per GPU, ``torch.distributed`` plumbing).

Two levels (SURVEY.md §8e):

* independent movies -> one movie per rank, no data-path collective (``bench.py --gpus N``);
* ONE large movie split into contiguous frame blocks (``motion_correct_frame_split``).  The only
  bandwidth-relevant collective is the all-reduce of the (h, w) frame sum; the estimators exchange
  three double-precision moments, the band-limited patch spectra (a few % of the movie) and a few
  KB of shifts.  Every rank ends up with the same field and the full frame sum.

Nothing here reshapes data for the network: spectra are gathered exactly as the kernels produce
them.  With ``group=None`` and no initialised process group the functions degenerate to the
single-GPU path (world size 1), which is how the ``-m gpu`` tests exercise the bookkeeping.
"""

from __future__ import annotations

import os

import torch
import torch.distributed as dist

from . import _fourier, _ops
from ._common import as_f32, cached_device_tensor, grid_kind, resolve_device
from ._lib import call, ptr, stream_ptr
from .correct_motion import correct_motion_fast
from .estimate_motion_xc import global_spectra, leave_one_out_shifts, mean_except_current_spectra, patch_xc_geometry


def frame_range(total_frames: int, rank: int, world: int) -> tuple[int, int]:
    """Contiguous block [f0, f1) of rank ``rank``: the first ``total % world`` ranks hold one more."""
    base, extra = divmod(total_frames, world)
    f0 = rank * base + min(rank, extra)
    return f0, f0 + base + (1 if rank < extra else 0)


def _world(group):
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(group), dist.get_world_size(group)
    return 0, 1


def all_gather_frames(local: torch.Tensor, total_frames: int, group=None, dim: int = 0) -> torch.Tensor:
    """Concatenate per-rank blocks ``local`` along ``dim`` (rank order == index order; rank r holds the entries
    ``frame_range(total_frames, r, world)``) into ``total_frames`` entries on every rank.  Blocks may differ by one
    entry: pad, gather, trim."""
    _, world = _world(group)
    if world == 1:
        return local
    shape = list(local.shape)
    shape[dim] = -(-total_frames // world)
    padded = torch.zeros(shape, dtype=local.dtype, device=local.device)
    padded.narrow(dim, 0, local.shape[dim]).copy_(local)
    parts = [torch.empty_like(padded) for _ in range(world)]
    dist.all_gather(parts, padded, group=group)
    out = []
    for r in range(world):
        f0, f1 = frame_range(total_frames, r, world)
        out.append(parts[r].narrow(dim, 0, f1 - f0))
    return torch.cat(out, dim=dim)


def _reshard_frames_to_patches(spec, spec_sub, t, g, words, rank, world, group, frame_major=False):
    """spec (t_local, G, words): every patch of this rank's frames -> every frame of this rank's patches, written to
    spec_sub[:, :t] (G_r, T, words) or, ``frame_major``, to spec_sub[:t, :G_r] (T, G_r, words).  An all-to-all: every rank
    sends each peer only the planes of that peer's patches (1/world of what an all-gather would deliver to everybody);
    falls back to the all-gather where the backend has no all-to-all."""
    g0, g1 = frame_range(g, rank, world)

    def put(f0, f1, block):  # block (f1 - f0, G_r, words)
        if frame_major:
            spec_sub[f0:f1, : g1 - g0] = block
        else:
            spec_sub[: g1 - g0, f0:f1] = block.permute(1, 0, 2)

    if world == 1:
        if g1 > g0:
            put(0, t, spec)
        return
    t_local = spec.shape[0]
    frames_of = [frame_range(t, r, world) for r in range(world)]
    patches_of = [frame_range(g, r, world) for r in range(world)]
    try:
        send = torch.cat([spec[:, a:b].reshape(-1) for a, b in patches_of]) if t_local > 0 else spec.reshape(-1)
        in_splits = [t_local * (b - a) * words for a, b in patches_of]
        out_splits = [(f1 - f0) * (g1 - g0) * words for f0, f1 in frames_of]
        recv = torch.empty((sum(out_splits),), dtype=spec.dtype, device=spec.device)
        dist.all_to_all_single(recv, send, out_splits, in_splits, group=group)
        offset = 0
        for (f0, f1), n in zip(frames_of, out_splits):
            if n:
                put(f0, f1, recv[offset : offset + n].view(f1 - f0, g1 - g0, words))
            offset += n
    except (RuntimeError, NotImplementedError):
        full = all_gather_frames(spec, t, group)  # (T, G, words) on every rank
        if g1 > g0:
            put(0, t, full[:, g0:g1])


def stack_stats_frame_split(local_frames: torch.Tensor, group=None) -> torch.Tensor:
    """normalize_image statistics of the WHOLE movie from per-rank moments (24 bytes all-reduced)."""
    moments = _ops.stack_moments(local_frames)
    _, world = _world(group)
    if world > 1:
        dist.all_reduce(moments, op=dist.ReduceOp.SUM, group=group)
    return _ops.moments_to_mean_std(moments)


def correct_motion_sum_frame_split(local_frames, deformation_grid, pixel_spacing, frame_offset, total_frames,
                                   grid_type="catmull_rom", group=None, reduce=True) -> torch.Tensor:
    """Warp the local frame block, sum it, and all-reduce the (h, w) partial sums (NCCL over NVLink)."""
    from .correct_motion import correct_motion_sum

    total = correct_motion_sum(
        local_frames, deformation_grid, pixel_spacing, grid_type=grid_type, frame_offset=frame_offset, total_frames=total_frames
    )
    _, world = _world(group)
    if world > 1 and reduce:
        dist.all_reduce(total, op=dist.ReduceOp.SUM, group=group)
    return total


def correct_motion_sums_frame_split(local_frames, deformation_grid, pixel_spacing, frame_offset, total_frames,
                                    grid_type="catmull_rom", *, dose_per_frame=None, pre_exposure=0.0, voltage=300.0,
                                    half_sets=False, group=None, device=None) -> dict:
    """``correct_motion_sums`` of a movie whose frames [frame_offset, frame_offset + t_local) live on this rank: every
    rank forms its frames' sums with the exposure filter of the WHOLE movie (factorised on the first rank of ``group``
    and broadcast, so that all ranks use the same tables) and the (h, w) outputs are all-reduced.  Every output is linear
    in the frames, so the partial sums add up to the single-process result."""
    from .correct_motion import _field, _movie, check_sums_arguments, warp_sums
    from .dose_weight import exposure_filter_lowrank

    dev = resolve_device(local_frames, device)
    check_sums_arguments(local_frames.shape, None, dose_per_frame)
    if not (0 <= frame_offset and frame_offset + local_frames.shape[0] <= total_frames):
        raise ValueError(f"frames [{frame_offset}, {frame_offset + local_frames.shape[0]}) outside a movie of {total_frames}")
    movie = _movie(local_frames, dev)
    field = _field(deformation_grid, dev)
    rank, world = _world(group)
    lowrank = None
    if dose_per_frame is not None:
        if rank == 0:
            h, w = movie.shape[-2:]
            lowrank = exposure_filter_lowrank(h, w, pixel_spacing, range(total_frames), dose_per_frame, pre_exposure,
                                              voltage, half_sets)
        if world > 1:
            box = [lowrank]
            dist.broadcast_object_list(box, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
            lowrank = box[0]
    out = warp_sums(movie, field, pixel_spacing, grid_kind(grid_type), frame_offset, total_frames, half_sets, lowrank,
                    pixel_spacing, voltage)
    if world > 1:
        for name in sorted(out):
            dist.all_reduce(out[name], op=dist.ReduceOp.SUM, group=group)
    return out


def estimate_global_motion_frame_split(local_frames, pixel_spacing, frame_offset, total_frames, mean_std,
                                       reference_frame=None, b_factor=500, frequency_range=(300, 10), group=None):
    """``estimate_global_motion`` for a frame-split movie: the owner of the reference frame
    broadcasts its band-limited spectrum (a few MB); shifts are all-gathered."""
    rank, world = _world(group)
    dev = local_frames.device
    t_local = local_frames.shape[0]
    if reference_frame is None:
        reference_frame = total_frames // 2
    plan, spec = global_spectra(local_frames, mean_std, pixel_spacing, b_factor, frequency_range)
    ref_spec = torch.empty((1, plan.ky, plan.kx, 2), dtype=torch.float32, device=dev)
    owner = next(r for r in range(world) if frame_range(total_frames, r, world)[0] <= reference_frame < frame_range(total_frames, r, world)[1])
    if rank == owner:
        ref_spec.copy_(spec[reference_frame - frame_offset : reference_frame - frame_offset + 1])
    if world > 1:
        dist.broadcast(ref_spec, src=dist.get_global_rank(group, owner) if group is not None else owner, group=group)
    both = torch.cat([spec[:t_local], ref_spec], dim=0)
    cur = torch.arange(t_local, dtype=torch.int32, device=dev)
    ref = torch.full((t_local,), t_local, dtype=torch.int32, device=dev)
    prod = _fourier.pair_products(both, ref, cur, plan.plane_elems)
    shifts = plan.peaks(prod.view(t_local, plan.ky, plan.kx, 2), sub_pixel=False)
    shifts = all_gather_frames(shifts, total_frames, group)
    return _ops.global_shifts_to_field(shifts, pixel_spacing, reference_frame)


def estimate_patch_motion_frame_split(local_frames, pixel_spacing, frame_offset, total_frames, mean_std,
                                      deformation_field=None, b_factor=500, frequency_range=(300, 10), patch_sidelength=1024,
                                      sub_pixel_refinement=True, temporal_smoothing=True, smoothing_window_size=5,
                                      outlier_rejection=True, outlier_threshold=3.0, group=None, whole_pixel_field=False):
    """``estimate_motion_cross_correlation_patches`` (``mean_except_current``) for a frame-split movie.

    Each rank transforms the patches of its own frames; the band-limited spectra (both mask powers, quirk Q1) are
    re-sharded by patch (all-to-all) so that every rank forms the leave-one-out references and peaks of ALL frames of its
    share of the patches; the shifts are all-gathered."""
    rank, world = _world(group)
    dev = local_frames.device
    t_local, h, w = local_frames.shape
    t = total_frames
    if t < 2:
        raise ValueError("mean_except_current needs at least two frames")
    source, source_stats = local_frames, mean_std
    frame_shifts = None
    if deformation_field is not None:
        deformation_field = deformation_field.to(dev)
        if tuple(deformation_field.shape[-2:]) != (1, 1):
            raise NotImplementedError("frame-split pre-correction supports the rigid (2, t, 1, 1) field")
        local_field = deformation_field[:, frame_offset : frame_offset + t_local].clone()
        if whole_pixel_field:
            # whole-pixel rigid field (estimate_global_motion, quirk Q5): the integer Fourier shift is a circular roll,
            # i.e. patch windows read at origins moved by each frame's shift -- no pre-correction pass
            frame_shifts, _ = _fourier.integer_shifts(local_field)
        else:
            source = correct_motion_fast(local_frames, local_field, device=dev, _mean_std=mean_std)
            source_stats = None
        deformation_field = deformation_field * -1  # the reference negates the caller's field in place (Q2)
    p = int(patch_sidelength)
    centres, origins, plan, mask, field = patch_xc_geometry((t, h, w), p, pixel_spacing, b_factor, frequency_range,
                                                            deformation_field, dev)
    g = len(origins)
    words = 2 * plan.plane_elems * 2  # both mask powers of one (frame, patch), float32 words
    _, spec_local = mean_except_current_spectra(source, source_stats, plan, mask, p, origins, frame_shifts)
    # frames for the transforms, patches for the cross-correlation: every rank receives ALL frames of ITS share of the
    # patches (all-to-all, 1/world of an all-gather), forms their leave-one-out references and peaks, and the shifts
    # (KBs) are gathered
    g0, g1 = frame_range(g, rank, world)
    g_sub = g1 - g0
    gs = max(g_sub, 1)
    spec_sub = torch.zeros((t, gs, words), dtype=torch.float32, device=dev)
    _reshard_frames_to_patches(spec_local.view(t_local, g, words), spec_sub, t, g, words, rank, world, group, frame_major=True)
    del spec_local
    shifts = leave_one_out_shifts(spec_sub, t, gs, plan, sub_pixel_refinement)
    shifts = all_gather_frames(shifts.view(t, gs, 2)[:, :g_sub], g, group, dim=1).contiguous()
    _ops.xc_postprocess(shifts, field, pixel_spacing, -1, outlier_rejection, outlier_threshold, temporal_smoothing,
                        smoothing_window_size)
    return field, centres.clone()


def estimate_local_motion_frame_split(local_frames, pixel_spacing, patch_shape, deformation_field_resolution,
                                      initial_deformation_field, frame_offset, total_frames, mean_std, n_iterations=100,
                                      b_factor=500, frequency_range=(300, 10), grid_type="catmull_rom", loss_type="mse",
                                      optimizer_kwargs=None, group=None, return_losses=False):
    """``estimate_local_motion`` (Adam; "mse" / "cc" losses) for a frame-split movie.

    Frames for the transforms, patches for the optimiser: every rank transforms the patches of its own frames once, the
    band-limited spectra (a few % of the movie) are exchanged so that every rank holds ALL frames of ITS share of the
    patches, and the iterations run on the single-GPU kernels (``tmc_local_steps``).  ``Sigma = sum_t S_t``, the only
    coupling between frames (estimate_motion_optimizer.py:391-399), is then local to a rank; per iteration only the
    coefficient gradient (2 nt nh nw floats) is all-reduced, and the Adam update is replicated.  The shuffled mini-batch
    weighting (quirks Q10 / Q11) is drawn on rank 0 and broadcast, so the result equals the single-GPU run with the same
    ``random`` state up to the order of the fp32 sums.  Returns the (2, nt, nh, nw) field (identical on all ranks)."""
    from .estimate_motion_optimizer import (LOSS_TYPES, LocalMotionProblem, _shuffled_batches, base_grid, fused_adam_state,
                                            local_patches, local_spectra, normalised_centres, patch_scales)

    rank, world = _world(group)
    dev = local_frames.device
    frames = as_f32(local_frames, dev)
    t_local, h, w = frames.shape
    t = int(total_frames)
    ph, pw = patch_shape
    if loss_type not in ("mse", "cc"):
        raise NotImplementedError("the frame-split optimiser covers the 'mse' and 'cc' losses")
    lt = LOSS_TYPES[loss_type]
    kind = grid_kind(grid_type)
    resolution = tuple(int(r) for r in deformation_field_resolution)
    kw = dict(optimizer_kwargs) if optimizer_kwargs is not None else {}

    centers, origins = local_patches((t, h, w), patch_shape)
    g = len(origins[0])
    base = base_grid(initial_deformation_field, resolution, dev)

    # spectra of the local frames: one plane per (frame, patch), frame-major (t_local, G, KY, KX)
    plan = _fourier.BandPlan(ph, pw, dev, float(pixel_spacing), b_factor, frequency_range)
    words = plan.plane_elems * 2
    if t_local > 0:
        pairs = (t_local + 1) // 2
        spec = local_spectra(frames, mean_std, plan, patch_shape, origins, True)  # planes [pair][patch][frame of the pair]
        spec = spec.view(pairs, g, 2, words).permute(0, 2, 1, 3).reshape(2 * pairs, g, words)[:t_local].contiguous()
    else:
        spec = torch.zeros((0, g, words), dtype=torch.float32, device=dev)
    # this rank's share of the patches, all frames: (G_r, tp, KY, KX)
    g0, g1 = frame_range(g, rank, world)
    g_sub = g1 - g0
    tp = 2 * ((t + 1) // 2)
    spec_sub = torch.zeros((max(g_sub, 1), tp, words), dtype=torch.float32, device=dev)
    _reshard_frames_to_patches(spec, spec_sub, t, g, words, rank, world, group)
    del spec

    centres_sub = cached_device_tensor(("split_centres", (t, h, w, ph, pw), g0, g1),
                                       lambda: normalised_centres(centers, (t, h, w))[:, g0:max(g1, g0 + 1)].contiguous(), dev)
    problem = LocalMotionProblem.from_spectra(spec_sub, False, centres_sub, base, plan, patch_shape, kind, lt, pixel_spacing)

    # the mini-batch weighting of every iteration: drawn once (rank 0) and broadcast; each rank uses its patches' columns
    n_iterations = int(n_iterations)
    scales = torch.zeros((max(n_iterations, 1), g), dtype=torch.float32)
    if rank == 0:
        for i in range(n_iterations):
            scales[i] = torch.tensor(patch_scales(_shuffled_batches(g, 8), g, t, ph, pw, lt), dtype=torch.float32)
    scales = scales.to(dev)
    if world > 1:
        dist.broadcast(scales, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
    scales_sub = scales[:, g0:max(g1, g0 + 1)].contiguous()
    if g_sub == 0:
        scales_sub.zero_()  # a rank without patches contributes nothing

    new = torch.zeros((2, *resolution), dtype=torch.float32, device=dev)
    adam = fused_adam_state(new, kw)
    exp_avg, exp_avg_sq, lr, b1, b2, eps, wd = adam
    steps = torch.arange(max(n_iterations, 1), dtype=torch.int32, device=dev)  # Adam's step number - 1 of every iteration
    losses = []
    def reduce_gradient(loss, grad):
        if world > 1:
            dist.all_reduce(grad, op=dist.ReduceOp.SUM, group=group)
        if return_losses:
            total = loss.clone()
            if world > 1:
                dist.all_reduce(total, op=dist.ReduceOp.SUM, group=group)
            losses.append(total)

    with torch.cuda.device(dev):
        stream = stream_ptr(dev)
        if problem.fused:
            # three launches and one all-reduce per iteration: [Adam on the reduced gradient + next shifts] -> loss /
            # gradient kernel -> backward to the coefficient gradient (tmc_local_steps modes 1, 2, 3)
            for i in range(n_iterations):
                problem.fused_steps(new, scales_sub, i, 1, 1 if i == 0 else 2, problem.loss, adam=adam)
                reduce_gradient(problem.loss, problem.grad)
            if n_iterations > 0:
                problem.fused_steps(new, scales_sub, n_iterations, 1, 3, problem.loss, adam=adam)
        else:
            for i in range(n_iterations):
                loss, grad = problem.loss_and_grad(new, scales_sub[i])
                reduce_gradient(loss, grad)
                call("tmc_adam_step", ptr(new), ptr(grad), ptr(exp_avg), ptr(exp_avg_sq), new.numel(), lr, b1, b2, eps, wd,
                     steps.data_ptr() + 4 * i, stream)
    final = (new + base).contiguous()
    _ops.subtract_mean(final)
    if return_losses:
        return final, [float(l) for l in losses]
    return final


def motion_correct_frame_split(local_frames: torch.Tensor, pixel_spacing: float, frame_offset: int, total_frames: int,
                               patch_sidelength: int = 1024, b_factor: float = 500, frequency_range=(300, 10),
                               grid_type: str = "bspline", group=None, device=None, n_iterations: int = 0,
                               deformation_field_resolution=None, optimizer_kwargs=None):
    """Estimate (global + patch XC [+ ``n_iterations`` of the spline optimiser]) and correct ONE movie whose frames are
    split across the ranks of ``group``.  Returns ``(frame sum (h, w) on every rank, field)``; the field is
    (2, t, gh, gw) without the optimiser and (2, nt, nh, nw) with it."""
    dev = resolve_device(local_frames, device)
    frames = as_f32(local_frames, dev)
    grid_kind(grid_type)
    stats = stack_stats_frame_split(frames, group)
    global_field = estimate_global_motion_frame_split(
        frames, pixel_spacing, frame_offset, total_frames, stats, b_factor=b_factor, frequency_range=frequency_range, group=group
    )
    from .pipeline import cumulative_patch_field

    field, _ = cumulative_patch_field(
        global_field, pixel_spacing,
        lambda pre: estimate_patch_motion_frame_split(
            frames, pixel_spacing, frame_offset, total_frames, stats, deformation_field=pre, b_factor=b_factor,
            frequency_range=frequency_range, patch_sidelength=patch_sidelength, group=group, temporal_smoothing=False,
            whole_pixel_field=True,
        ),
    )
    if n_iterations > 0:
        field = estimate_local_motion_frame_split(
            frames, pixel_spacing, (patch_sidelength, patch_sidelength), deformation_field_resolution or (3, 5, 5), field,
            frame_offset, total_frames, stats, n_iterations=n_iterations, b_factor=b_factor, frequency_range=frequency_range,
            grid_type=grid_type, optimizer_kwargs=optimizer_kwargs, group=group,
        )
    total = correct_motion_sum_frame_split(frames, field, pixel_spacing, frame_offset, total_frames, grid_type, group)
    return total, field
