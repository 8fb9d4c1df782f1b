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
from .deformation_field_utils import resample_deformation_field
from .estimate_motion_xc import _aliasing_schedule
from .patch_grid import patch_grid_centers


def frame_range(total_frames: int, rank: int, world: int) -> tuple[int, int]:
    """Contiguous block [f0, f1) of rank ``rank``: the first ``total % world`` ranks hold one more."""
    base, extra = divmod(total_frames, world)
    f0 = rank * base + min(rank, extra)
    return f0, f0 + base + (1 if rank < extra else 0)


def _world(group):
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(group), dist.get_world_size(group)
    return 0, 1


def all_gather_frames(local: torch.Tensor, total_frames: int, group=None) -> torch.Tensor:
    """Concatenate per-rank blocks ``local (t_local, ...)`` (rank order == frame order) into
    ``(total_frames, ...)`` on every rank.  Blocks may differ by one frame: pad, gather, trim."""
    rank, world = _world(group)
    if world == 1:
        return local
    t_max = -(-total_frames // world)
    padded = local
    if local.shape[0] < t_max:
        pad = torch.zeros((t_max - local.shape[0], *local.shape[1:]), dtype=local.dtype, device=local.device)
        padded = torch.cat([local, pad], dim=0)
    padded = padded.contiguous()
    parts = [torch.empty_like(padded) for _ in range(world)]
    dist.all_gather(parts, padded, group=group)
    out = []
    for r in range(world):
        f0, f1 = frame_range(total_frames, r, world)
        out.append(parts[r][: f1 - f0])
    return torch.cat(out, dim=0)


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


def _all_gather_patches(local, g, rank, world, group):
    """(t, G_r, c) blocks of consecutive patch ranges (frame_range(g, r, world)) -> (t, G, c) on every rank."""
    if world == 1:
        return local
    g_max = -(-g // world)
    padded = torch.zeros((local.shape[0], g_max, local.shape[2]), dtype=local.dtype, device=local.device)
    padded[:, : local.shape[1]] = local
    parts = [torch.empty_like(padded) for _ in range(world)]
    dist.all_gather(parts, padded, group=group)
    out = []
    for r in range(world):
        a, b = frame_range(g, r, world)
        out.append(parts[r][:, : b - a])
    return torch.cat(out, dim=1)


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
    t_local, h, w = local_frames.shape
    if reference_frame is None:
        reference_frame = total_frames // 2
    plan = _fourier.BandPlan(h, w, dev, pixel_spacing, b_factor, frequency_range)
    mask, ylo, yhi = _fourier.soft_disc_mask((h, w), min(h, w) / 4, min(h, w) / 8, dev)
    spec = plan.forward(local_frames, mean_std, mask, ylo, yhi, _fourier.frame_pair_jobs(t_local, dev), job_mode=2)
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
    field = torch.empty((2, total_frames, 1, 1), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        call("tmc_global_shifts_to_field", ptr(shifts), total_frames, float(pixel_spacing), int(reference_frame), ptr(field),
             stream_ptr(dev))
    return field


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
    centers = patch_grid_centers((t, h, w), (1, p, p), (1, p // 2, p // 2), distribute_patches=True)
    gh, gw = centers.shape[1:3]
    g = gh * gw
    origins = (centers[0, :, :, 1:] - p // 2).reshape(-1, 2).tolist()
    plan = _fourier.BandPlan(p, p, dev, pixel_spacing, b_factor, frequency_range)
    mask, ylo, yhi = _fourier.soft_disc_mask((p, p), p / 4, p / 8, dev)
    if deformation_field is None:
        field = torch.zeros((2, t, gh, gw), dtype=torch.float32, device=dev)
    else:
        field = resample_deformation_field(deformation_field, (t, gh, gw))
    # planning tensors are pure functions of the geometry: built once per device (no host-blocking copies per call)
    jobs = cached_device_tensor(
        ("split_xc_jobs", (t_local, h, w, p)),
        lambda: torch.tensor([[k, 1, k, 2, y0, x0] for k in range(t_local) for (y0, x0) in origins], dtype=torch.int32), dev)
    words = 2 * plan.plane_elems * 2  # both mask powers of one (frame, patch), float32 words
    spec_local = plan.forward(source, source_stats, mask, ylo, yhi, jobs, job_mode=1, frame_shifts=frame_shifts).view(t_local, g, words)
    # frames for the transforms, patches for the cross-correlation: every rank receives ALL frames of ITS share of the
    # patches (all-to-all, 1/world of an all-gather), forms their leave-one-out references and peaks, and the shifts
    # (KBs) are gathered
    g0, g1 = frame_range(g, rank, world)
    g_sub = g1 - g0
    spec_sub = torch.zeros((t, max(g_sub, 1), words), dtype=torch.float32, device=dev)
    _reshard_frames_to_patches(spec_local, spec_sub, t, g, words, rank, world, group, frame_major=True)
    del spec_local

    def schedule(part):
        offsets, deltas = _aliasing_schedule(t, "mean_except_current", t // 2)
        return torch.tensor(offsets if part == 0 else (deltas if deltas else [0]), dtype=torch.int32)

    d_off = cached_device_tensor(("xc_delta_offsets", t), lambda: schedule(0), dev)  # same keys as estimate_motion_xc
    d_val = cached_device_tensor(("xc_deltas", t), lambda: schedule(1), dev)
    gs = max(g_sub, 1)
    prod = _fourier.leave_one_out_products(spec_sub, t, gs, plan.plane_elems, d_off, d_val)
    shifts = plan.peaks(prod.view(t * gs, plan.ky, plan.kx, 2), sub_pixel=bool(sub_pixel_refinement))
    shifts = _all_gather_patches(shifts.view(t, gs, 2)[:, :g_sub], g, rank, world, group).contiguous()
    scratch = torch.empty_like(field)
    with torch.cuda.device(dev):
        call("tmc_xc_postprocess", ptr(shifts), t, g, float(pixel_spacing), -1, int(bool(outlier_rejection)),
             float(outlier_threshold), int(bool(temporal_smoothing)), int(smoothing_window_size), 1, ptr(field), ptr(scratch),
             stream_ptr(dev))
    return field, cached_device_tensor(("patch_centres", (t, h, w, p)), lambda: centers, dev).clone()


def _make_patch_shard_problem(spec_sub, centres_norm_sub, base, kind, loss_code, px, t, ph, pw, resolution, plan, dev):
    """A ``LocalMotionProblem`` (estimate_motion_optimizer.py) for a subset of the patches with ALL frames, built from
    spectra ``spec_sub`` (G_r, tp, KY, KX) that are already on the device."""
    from .estimate_motion_optimizer import LocalMotionProblem, fused_steps_apply
    from ._lib import query

    prob = LocalMotionProblem.__new__(LocalMotionProblem)
    g = spec_sub.shape[0]
    prob.kind, prob.loss_type, prob.dev, prob.px = kind, loss_code, dev, px
    prob.t, prob.ph, prob.pw = t, ph, pw
    prob.resolution = resolution
    prob.g = g
    prob.base = base
    prob.plan = plan
    prob.tp = spec_sub.shape[1]
    prob.fused = fused_steps_apply(loss_code, g, t, resolution, plan)
    prob.frame_major = False  # (G, tp, KY, KX): patch-major
    prob.spec = spec_sub
    prob.norms = torch.empty((g, t, 2), dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        call("tmc_local_spectra_norms", ptr(spec_sub), g, t, prob.tp, ph, pw, plan.ky, plan.kx, plan.ky_start, 0, ptr(prob.norms),
             stream_ptr(dev))
    prob.centres_norm = centres_norm_sub  # (T, g, 3)
    prob.eval_base = _ops.spline_eval(base, kind, centres_norm_sub)
    ws_bytes = query("tmc_local_loss_workspace_bytes", g, t, plan.ky, plan.kx)
    prob.workspace = torch.empty(((ws_bytes + 7) // 8,), dtype=torch.float64, device=dev)
    prob.loss = torch.zeros((1,), dtype=torch.float64, device=dev)
    prob.grad_eval = torch.empty((t, g, 2), dtype=torch.float32, device=dev)
    prob.eval_new = torch.empty((t, g, 2), dtype=torch.float32, device=dev)
    prob.grad = torch.empty((2, *resolution), dtype=torch.float32, device=dev)
    n_ws = query("tmc_spline_workspace_floats", 2, *resolution)
    prob.ws_eval = torch.empty((n_ws,), dtype=torch.float32, device=dev)
    prob.ws_back = torch.empty((n_ws,), dtype=torch.float32, device=dev)
    if prob.fused:
        prob._setup_fused_steps()
    return prob


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
    from .estimate_motion_optimizer import LOSS_TYPES, _shuffled_batches

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
    px = float(pixel_spacing)
    kw = dict(optimizer_kwargs) if optimizer_kwargs is not None else {}

    centers = patch_grid_centers((t, h, w), (1, ph, pw), (1, ph // 2, pw // 2), distribute_patches=True)
    gh, gw = centers.shape[1:3]
    g = gh * gw
    flat = centers[0].reshape(-1, 3)
    y0 = (flat[:, 1] - ph // 2).tolist()
    x0 = (flat[:, 2] - pw // 2).tolist()
    if min(y0) < 0 or min(x0) < 0 or max(y0) + ph > h or max(x0) + pw > w:
        raise AssertionError(f"Patch size {tuple(patch_shape)} too large for control points in image of shape {(t, h, w)}")

    if initial_deformation_field is None:
        base = torch.zeros((2, *resolution), dtype=torch.float32, device=dev)
    else:
        base = resample_deformation_field(as_f32(initial_deformation_field, dev), resolution)
        with torch.cuda.device(dev):
            call("tmc_subtract_mean", ptr(base), base.numel(), stream_ptr(dev))

    # spectra of the local frames: one plane per (frame, patch), frame-major (t_local, G, KY, KX)
    plan = _fourier.BandPlan(ph, pw, dev, px, b_factor, frequency_range)
    mask, ylo, yhi = _fourier.soft_disc_mask((ph, pw), pw / 4, pw / 4, dev)  # quirk Q18
    words = plan.plane_elems * 2
    if t_local > 0:
        jobs = cached_device_tensor(
            ("split_local_jobs", (t_local, h, w, ph, pw)),
            lambda: torch.tensor([[i, 1, i + 1 if i + 1 < t_local else -1, 1, y0[gi], x0[gi]] for i in range(0, t_local, 2)
                                  for gi in range(g)], dtype=torch.int32), dev)
        pairs = (t_local + 1) // 2
        spec = plan.forward(frames, mean_std, mask, ylo, yhi, jobs, job_mode=2)  # planes [pair][patch][frame of the pair]
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

    # normalised (t, y, x) centres of this rank's patches, time-major (T, G_r, 3)
    norm = centers.clone().float()
    norm[..., 0] /= float(t - 1) if t > 1 else float("nan")
    norm[..., 1] /= float(h - 1)
    norm[..., 2] /= float(w - 1)
    centres_sub = cached_device_tensor(("split_centres", (t, h, w, ph, pw), g0, g1),
                                       lambda: norm.reshape(t, g, 3)[:, g0:max(g1, g0 + 1)].contiguous(), dev)
    problem = _make_patch_shard_problem(spec_sub, centres_sub, base, kind, lt, px, t, ph, pw, resolution, plan, dev)

    # the mini-batch weighting of every iteration: drawn once (rank 0) and broadcast; each rank uses its patches' columns
    def patch_scales(batches):
        scale = [0.0] * g
        for batch in batches:
            b = len(batch)
            sc = 1.0 / (b * t * ph * (pw // 2 + 1)) / (ph * pw) if lt == 0 else 1.0 / (b * t)
            for gi in batch:
                scale[gi] = sc
        return scale

    n_iterations = int(n_iterations)
    scales = torch.zeros((max(n_iterations, 1), g), dtype=torch.float32)
    if rank == 0:
        for i in range(n_iterations):
            scales[i] = torch.tensor(patch_scales(_shuffled_batches(g, 8)), dtype=torch.float32)
    scales = scales.to(dev)
    if world > 1:
        dist.broadcast(scales, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
    scales_sub = scales[:, g0:max(g1, g0 + 1)].contiguous()
    if g_sub == 0:
        scales_sub.zero_()  # a rank without patches contributes nothing

    new = torch.zeros((2, *resolution), dtype=torch.float32, device=dev)
    exp_avg, exp_avg_sq = torch.zeros_like(new), torch.zeros_like(new)
    lr, (b1, b2) = float(kw.get("lr", 0.01)), kw.get("betas", (0.9, 0.999))
    eps, wd = float(kw.get("eps", 1e-08)), float(kw.get("weight_decay", 0))
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
            adam = (exp_avg, exp_avg_sq, lr, float(b1), float(b2), eps, wd)
            for i in range(n_iterations):
                problem.fused_steps(new, scales_sub, i, 1, 1 if i == 0 else 2, problem.loss, adam=adam)
                reduce_gradient(problem.loss, problem.grad)
            if n_iterations > 0:
                problem.fused_steps(new, scales_sub, n_iterations, 1, 3, problem.loss, adam=adam)
        else:
            for i in range(n_iterations):
                loss, grad = problem.loss_and_grad(new, scales_sub[i])
                reduce_gradient(loss, grad)
                call("tmc_adam_step", ptr(new), ptr(grad), ptr(exp_avg), ptr(exp_avg_sq), new.numel(), lr, float(b1), float(b2), eps,
                     wd, steps.data_ptr() + 4 * i, stream)
    final = (new + base).contiguous()
    with torch.cuda.device(dev):
        call("tmc_subtract_mean", ptr(final), final.numel(), stream_ptr(dev))
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
