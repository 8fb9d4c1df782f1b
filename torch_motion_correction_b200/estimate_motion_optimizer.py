"""Spline-coefficient optimisation of local motion (mirror of the reference's
``estimate_motion_optimizer.py``).

The forward model and its gradient are closed-form CUDA kernels (``csrc/optimizer.cu``): the
masked patch spectra are transformed ONCE (the reference re-does the FFTs every iteration, quirk
Q19) and only their pass band is kept; each iteration evaluates the two spline grids at the patch
centres, the loss, dL/d(shifts) and scatters that back onto the coefficients.  ``torch.optim``
drives the coefficient update exactly as in the reference (same defaults)."""

from __future__ import annotations

import os
import random
from typing import Any, cast

import torch

from . import _fourier, _ops
from ._common import as_f32, cached_device_tensor, grid_kind, resolve_device, to_device_async
from ._lib import call, ptr, query, stream_ptr
from .deformation_field_utils import resample_deformation_field
from .optimization_state import OptimizationTracker
from .patch_grid import patch_grid_centers

LOSS_TYPES = {"mse": 0, "cc": 1, "ncc": 2}

#: use the one-kernel iteration (csrc/optimizer_tiled.cu) for the "mse" / "cc" losses when the frame count fits
FUSED_STEPS = os.environ.get("TMC_FUSED_STEPS", "1") != "0"


def fused_steps_apply(loss_type: int, g: int, t: int, resolution, plan) -> bool:
    """Whether the one-kernel iteration runs this problem: "mse" / "cc" at a size it supports, and for "cc" a band
    without weight on the self-paired Nyquist bins (``_fourier.self_paired_weight``; the generic kernels take those)."""
    if not FUSED_STEPS or loss_type == 2:
        return False
    if loss_type == 1 and _fourier.self_paired_weight(plan):
        return False
    return bool(query("tmc_local_steps_supported", g, t, resolution[0], resolution[1] * resolution[2]))


def _setup_optimizer(optimizer_type: str, parameters, **kwargs: Any) -> torch.optim.Optimizer:
    """Same optimisers and defaults as the reference (estimate_motion_optimizer.py:513-608)."""
    name = optimizer_type.lower()
    if name == "adam":
        return torch.optim.Adam(
            parameters, lr=kwargs.get("lr", 0.01), betas=kwargs.get("betas", (0.9, 0.999)), eps=kwargs.get("eps", 1e-08),
            weight_decay=kwargs.get("weight_decay", 0), amsgrad=kwargs.get("amsgrad", False), capturable=True,
        )
    if name == "sgd":
        return torch.optim.SGD(
            parameters, lr=kwargs.get("lr", 0.01), momentum=kwargs.get("momentum", 0.9),
            weight_decay=kwargs.get("weight_decay", 0), dampening=kwargs.get("dampening", 0), nesterov=kwargs.get("nesterov", True),
        )
    if name == "rmsprop":
        return torch.optim.RMSprop(
            parameters, lr=kwargs.get("lr", 0.01), alpha=kwargs.get("alpha", 0.99), eps=kwargs.get("eps", 1e-08),
            weight_decay=kwargs.get("weight_decay", 0), momentum=kwargs.get("momentum", 0), centered=kwargs.get("centered", False),
            capturable=True,
        )
    if name == "lbfgs":
        max_iter = cast(int, kwargs.get("max_iter", 1))
        max_eval = kwargs.get("max_eval", None)
        if max_eval is None:
            max_eval = max(1, int(max_iter * 1.25))
        return torch.optim.LBFGS(
            parameters, lr=kwargs.get("lr", 1), max_iter=max_iter, max_eval=max_eval,
            tolerance_grad=kwargs.get("tolerance_grad", 1e-11), tolerance_change=kwargs.get("tolerance_change", 1e-11),
            history_size=kwargs.get("history_size", 5), line_search_fn=kwargs.get("line_search_fn", "strong_wolfe"),
        )
    raise ValueError(f"Unsupported optimizer: {optimizer_type}. Choose 'adam', 'sgd', 'rmsprop', or 'lbfgs'.")


def local_patches(shape, patch_shape):
    """Patch grid of the optimiser on a (t, h, w) movie: (centres (t, gh, gw, 3), window origins (y0 list, x0 list)).
    Patch window = floor(centre) - p // 2, no clipping (patch_utils.py:117-120,173-183; quirk Q20)."""
    t, h, w = shape
    ph, pw = patch_shape
    centers = patch_grid_centers((t, h, w), (1, ph, pw), (1, ph // 2, pw // 2), distribute_patches=True)
    flat = centers[0].reshape(-1, 3)
    y0 = (flat[:, 1] - ph // 2).tolist()
    x0 = (flat[:, 2] - pw // 2).tolist()
    if min(y0) < 0 or min(x0) < 0 or max(y0) + ph > h or max(x0) + pw > w:
        raise AssertionError(f"Patch size {tuple(patch_shape)} too large for control points in image of shape {(t, h, w)}")
    return centers, (y0, x0)


def normalised_centres(centers: torch.Tensor, shape) -> torch.Tensor:
    """Normalised (t, y, x) patch centres, (T, G, 3) time-major (patch_utils.py:88-93,157-172; quirk Q10)."""
    t, h, w = shape
    norm = centers.clone().float()
    norm[..., 0] /= float(t - 1) if t > 1 else float("nan")
    norm[..., 1] /= float(h - 1)
    norm[..., 2] /= float(w - 1)
    return norm.reshape(t, -1, 3).contiguous()


def base_grid(initial_field, resolution, dev) -> torch.Tensor:
    """Frozen base grid (estimate_motion_optimizer.py:135-158): zeros, or the initial field resampled onto the spline
    grid with its mean removed."""
    if initial_field is None:
        return torch.zeros((2, *resolution), dtype=torch.float32, device=dev)
    base = resample_deformation_field(as_f32(initial_field, dev), resolution)
    _ops.subtract_mean(base)
    return base


def local_spectra(movie, stats, plan, patch_shape, origins, frame_major: bool) -> torch.Tensor:
    """Spectra FW[g][t] = rfft2(mask * patch) * band * envelope on the pass-band box of every patch and frame of
    ``movie``, frames packed in pairs: (g * tp, KY, KX, 2) planes, patch by patch or, ``frame_major``, frame pair by
    frame pair (the two layouts the optimiser kernels read)."""
    t, h, w = movie.shape
    ph, pw = patch_shape
    y0, x0 = origins
    g = len(y0)
    mask, ylo, yhi = _fourier.soft_disc_mask((ph, pw), pw / 4, pw / 4, movie.device)  # quirk Q18: smoothing pw/4

    def build_jobs():
        pairs = [(i, i + 1 if i + 1 < t else -1) for i in range(0, t, 2)]
        order = [(pair, gi) for pair in pairs for gi in range(g)] if frame_major else \
            [(pair, gi) for gi in range(g) for pair in pairs]
        return torch.tensor([[a, 1, b, 1, y0[gi], x0[gi]] for (a, b), gi in order], dtype=torch.int32)

    jobs = cached_device_tensor(("local_jobs", (t, h, w, ph, pw), frame_major), build_jobs, movie.device)
    return plan.forward(movie, stats, mask, ylo, yhi, jobs, job_mode=2)


def patch_scales(batches, g: int, t: int, ph: int, pw: int, loss_type: int) -> list:
    """Per-patch weight reproducing the reference's per-mini-batch ``mean`` (quirk Q11): the gradient is the SUM over
    mini-batches of each batch's mean-reduced loss."""
    scale = [0.0] * g
    for batch in batches:
        b = len(batch)
        if loss_type == 0:
            s = 1.0 / (b * t * ph * (pw // 2 + 1)) / (ph * pw)
        else:
            s = 1.0 / (b * t)
        for gi in batch:
            scale[gi] = s
    return scale


def fused_adam_state(coef: torch.Tensor, optimizer_kwargs: dict) -> tuple:
    """State and hyper-parameters of the fused Adam update of ``coef``: (exp_avg, exp_avg_sq, lr, b1, b2, eps,
    weight_decay), torch.optim.Adam's defaults unless ``optimizer_kwargs`` sets them."""
    b1, b2 = optimizer_kwargs.get("betas", (0.9, 0.999))
    return (torch.zeros_like(coef), torch.zeros_like(coef), float(optimizer_kwargs.get("lr", 0.01)), float(b1), float(b2),
            float(optimizer_kwargs.get("eps", 1e-08)), float(optimizer_kwargs.get("weight_decay", 0)))


class LocalMotionProblem:
    """Device-resident state of one ``estimate_local_motion`` call: band-limited patch spectra,
    their norms, normalised patch centres and the frozen base grid's values at the centres."""

    def __init__(self, image, pixel_spacing, patch_shape, resolution, initial_field, dev, b_factor, frequency_range,
                 grid_type, loss_type, stats=None):
        if loss_type not in LOSS_TYPES:
            raise ValueError(f"Invalid loss type: {loss_type}. Must be 'mse', 'cc' or 'ncc'.")
        kind = grid_kind(grid_type)
        movie = as_f32(image, dev)
        t, h, w = movie.shape
        ph, pw = patch_shape
        resolution = tuple(int(r) for r in resolution)
        if stats is None:
            stats = _ops.stack_stats(movie)
        centers, origins = local_patches((t, h, w), patch_shape)
        base = base_grid(initial_field, resolution, dev)
        plan = _fourier.BandPlan(ph, pw, dev, pixel_spacing, b_factor, frequency_range)
        # for the tiled path the jobs are listed frame pair by frame pair, so the 50 %-overlapping patches of a pair run
        # back to back and every frame comes from HBM once (patch-major order re-read it 2.3x: ncu); _init_state takes
        # the same decision
        frame_major = fused_steps_apply(LOSS_TYPES[loss_type], len(origins[0]), t, resolution, plan)
        spec = local_spectra(movie, stats, plan, patch_shape, origins, frame_major)
        geometry = (t, h, w, ph, pw)
        centres_norm = cached_device_tensor(("local_centres", geometry), lambda: normalised_centres(centers, (t, h, w)), dev)
        self._init_state(spec, frame_major, centres_norm, base, plan, patch_shape, kind, LOSS_TYPES[loss_type],
                         pixel_spacing, geometry)

    @classmethod
    def from_spectra(cls, spec, frame_major, centres_norm, base, plan, patch_shape, kind, loss_type, pixel_spacing):
        """A problem over spectra that are already on the device (the frame-split optimiser's share of the patches, with
        ALL frames): spec / centres_norm laid out as ``local_spectra`` / ``normalised_centres`` make them.  Not entered
        in the separable-weights cache, since its centres are no function of a movie geometry."""
        problem = cls.__new__(cls)
        problem._init_state(spec, frame_major, centres_norm, base, plan, patch_shape, kind, loss_type, pixel_spacing, None)
        return problem

    def _init_state(self, spec, frame_major, centres_norm, base, plan, patch_shape, kind, loss_type, pixel_spacing,
                    geometry):
        """Everything an iteration reads or writes, from the spectra (g * tp planes in ``frame_major`` order), the
        (T, G, 3) normalised centres and the (2, nt, nh, nw) base grid.  ``geometry`` (t, h, w, ph, pw), which the
        centres are a function of, keys the cache of the separable spline weights; None: not cached."""
        self.spec, self.frame_major, self.centres_norm, self.base, self.plan = spec, frame_major, centres_norm, base, plan
        self.kind, self.loss_type, self.px = kind, loss_type, float(pixel_spacing)
        dev = spec.device
        t, g = centres_norm.shape[:2]
        self.dev, self.t, self.g = dev, t, g
        self.ph, self.pw = patch_shape
        self.tp = 2 * ((t + 1) // 2)
        self.resolution = tuple(base.shape[1:])
        self.fused = fused_steps_apply(loss_type, g, t, self.resolution, plan)
        self.norms = torch.empty((g, t, 2), dtype=torch.float64, device=dev)
        p = plan
        with torch.cuda.device(dev):
            call("tmc_local_spectra_norms", ptr(spec), g, t, self.tp, self.ph, self.pw, p.ky, p.kx, p.ky_start,
                 int(frame_major), ptr(self.norms), stream_ptr(dev))
        self.eval_base = _ops.spline_eval(base, kind, centres_norm)  # (T, G, 2)
        ws_bytes = query("tmc_local_loss_workspace_bytes", g, t, p.ky, p.kx)
        self.workspace = torch.empty(((ws_bytes + 7) // 8,), dtype=torch.float64, device=dev)
        self.loss = torch.zeros((1,), dtype=torch.float64, device=dev)
        self.grad_eval = torch.empty((t, g, 2), dtype=torch.float32, device=dev)
        # everything an iteration touches is allocated once: a captured step allocates nothing
        self.eval_new = torch.empty((t, g, 2), dtype=torch.float32, device=dev)
        self.grad = torch.empty((2, *self.resolution), dtype=torch.float32, device=dev)
        n_ws = query("tmc_spline_workspace_floats", 2, *self.resolution)
        self.ws_eval = torch.empty((n_ws,), dtype=torch.float32, device=dev)
        self.ws_back = torch.empty((n_ws,), dtype=torch.float32, device=dev)
        if self.fused:
            self._setup_fused_steps(geometry)

    def _setup_fused_steps(self, geometry):
        """State of the one-kernel iteration (csrc/optimizer_tiled.cu): tiled spectra, the separable dense spline
        weights of the patch centres, accumulators.  The (g * tp, KY, KX) spectra are released."""
        dev, t, p = self.dev, self.t, self.plan
        nt, nh, nw = self.resolution
        self.tiles = _fourier.band_tiles(p)
        n_tiles = self.tiles.shape[0]
        self.tiled = torch.empty((self.g, n_tiles, t, 2, 128), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            call("tmc_local_tile_spectra", ptr(self.spec), self.g, t, self.tp, p.ky, p.kx, ptr(self.tiles), n_tiles,
                 int(self.frame_major), ptr(self.tiled), stream_ptr(dev))
        self.spec = None
        self.sum_norms = self.norms[:, :, 0 if self.loss_type == 0 else 1].sum(dim=1).contiguous()
        # the patch centres are a product grid (frame) x (patch): the 64-tap spline weights factor into a dense
        # (T, nt) time matrix and a dense (G, nh nw) spatial matrix, phantom nodes folded in (spline of unit grids)
        # keyed by the geometry the centres are a function of (never by a device pointer); problems built from ad-hoc
        # centres (frame-split patch shards) carry no geometry key and are not cached
        key = ("local_weights", (dev.type, dev.index), self.kind, self.resolution, geometry) if geometry is not None else None
        hit = _separable_weights.get(key) if key is not None else None
        if hit is None:
            while len(_separable_weights) > 64:
                _separable_weights.pop(next(iter(_separable_weights)))
            cn = self.centres_norm
            pts_t = torch.zeros((t, 3), dtype=torch.float32, device=dev)
            pts_t[:, 0] = cn[:, 0, 0]
            pts_s = cn[0].clone()
            pts_s[:, 0] = 0.0
            eye_t = torch.eye(nt, dtype=torch.float32, device=dev).reshape(nt, nt, 1, 1).contiguous()
            eye_s = torch.eye(nh * nw, dtype=torch.float32, device=dev).reshape(nh * nw, 1, nh, nw).contiguous()
            hit = (_ops.spline_eval(eye_t, self.kind, pts_t).contiguous(), _ops.spline_eval(eye_s, self.kind, pts_s).contiguous())
            if key is not None:
                _separable_weights[key] = hit
        self.w_t, self.w_sp = hit[0], hit[1]
        ws_bytes = query("tmc_local_steps_workspace_bytes", self.g, t, nt)
        self.step_ws = torch.empty(((ws_bytes + 7) // 8,), dtype=torch.float64, device=dev)

    def fused_steps(self, coef, scales, first_row, n_steps, mode, loss_out, adam=None):
        """``n_steps`` iterations (loss/gradient kernel + coefficient kernel each).  mode 0: Adam (``adam`` = (exp_avg,
        exp_avg_sq, lr, b1, b2, eps, wd)) updating ``coef`` in place; mode 1: gradient into ``self.grad`` and loss into
        ``loss_out[0]``.  ``scales`` (rows, G): step i uses row ``first_row + i``."""
        p = self.plan
        nt, nh, nw = self.resolution
        exp_avg, exp_avg_sq, lr, b1, b2, eps, wd = adam if adam is not None else (None, None, 0.0, 0.0, 0.0, 0.0, 0.0)
        with torch.cuda.device(self.dev):
            call("tmc_local_steps", ptr(self.tiled), ptr(self.tiles), self.tiles.shape[0], self.g, self.t, self.ph, self.pw,
                 p.ky, p.kx, p.ky_start, ptr(self.sum_norms), ptr(self.eval_base), ptr(self.w_t), ptr(self.w_sp), nt, nh * nw,
                 ptr(scales), self.px, self.loss_type, ptr(coef), ptr(exp_avg), ptr(exp_avg_sq), float(lr), float(b1),
                 float(b2), float(eps), float(wd), int(first_row), int(mode), int(n_steps), ptr(loss_out), ptr(self.grad),
                 ptr(self.step_ws), stream_ptr(self.dev))

    def patch_scales(self, batches) -> list:
        return patch_scales(batches, self.g, self.t, self.ph, self.pw, self.loss_type)

    def loss_and_grad(self, new_data: torch.Tensor, scale: torch.Tensor, iteration: torch.Tensor | None = None, row: int = 0):
        """Sum over mini-batches of the batch losses (device float64 (1,)) and d/d new_data.

        ``scale`` is (G,) or (n, G) with the row picked by ``row`` (host int; tiled two-kernel path) or by
        ``iteration`` (device int32 counter; generic mse / cc path inside a captured graph)."""
        if self.fused:
            self.fused_steps(new_data, scale, row, 1, 1, self.loss)
            return self.loss, self.grad
        eval_new = _ops.spline_eval(new_data, self.kind, self.centres_norm, out=self.eval_new.view(-1, 2), ws=self.ws_eval)
        p = self.plan
        with torch.cuda.device(self.dev):
            call("tmc_local_loss_grad", ptr(self.spec), ptr(self.norms), ptr(eval_new), ptr(self.eval_base), ptr(scale),
                 ptr(iteration), self.g, self.t, self.tp, self.ph, self.pw, p.ky, p.kx, p.ky_start, self.px, self.loss_type,
                 ptr(self.loss), ptr(self.grad_eval), ptr(self.workspace), stream_ptr(self.dev))
        grad = _ops.spline_eval_backward(
            (2, *self.resolution), self.kind, self.centres_norm, self.grad_eval, out=self.grad, ws=self.ws_back
        )
        return self.loss, grad


_separable_weights: dict = {}


def _graph_capable(optimizer: torch.optim.Optimizer) -> bool:
    """Optimisers whose step can be captured in a CUDA graph (no host-side state in the step)."""
    if isinstance(optimizer, torch.optim.SGD):
        return True
    return bool(optimizer.defaults.get("capturable", False))


def _run_captured(one_step, n_iterations: int, dev: torch.device) -> int:
    """Run ``n_iterations`` optimiser steps as one eager warm-up + CUDA-graph replays (launch-bound
    inner loop: ~15 tiny kernels per step).  Returns the number of steps performed (0 if capture
    is not possible here, e.g. when already capturing)."""
    if torch.cuda.is_current_stream_capturing():
        return 0
    main = torch.cuda.current_stream(dev)
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(main)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        one_step(0)  # lazily creates the optimiser state outside the capture
        # capture_begin / capture_end directly: the torch.cuda.graph() context manager would
        # synchronise the device and empty the caching allocator (every later call would then pay
        # cudaMalloc for its multi-GB workspaces again)
        try:
            launches_before = query("tmc_launch_count")
            graph.capture_begin()  # the step allocates nothing (buffers live in LocalMotionProblem)
            try:
                one_step(1)
            finally:
                graph.capture_end()
            kernels_per_step = query("tmc_launch_count") - launches_before
        except Exception as exc:  # pragma: no cover - capture refused: finish eagerly
            import os
            import warnings

            if os.environ.get("TMC_DEBUG"):
                raise
            warnings.warn(f"CUDA-graph capture of the optimiser step failed ({exc}); running eagerly", stacklevel=2)
            main.wait_stream(side)
            return 1
    main.wait_stream(side)
    from . import _lib

    timing = _lib.TIMING
    if timing is not None:  # bench.py: the replayed kernels are invisible to the per-call timers
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
    for _ in range(n_iterations - 1):
        graph.replay()
    _lib.GRAPH_LAUNCHES += kernels_per_step * (n_iterations - 2)  # the capture pass itself was already counted
    if timing is not None:
        end.record()
        timing.setdefault("graph:optimiser_steps", []).append((start, end))
    return n_iterations


def _shuffled_batches(n_patches: int, batch_size: int):
    """``ImagePatchIterator.get_iterator`` order: ``random.shuffle`` of the flat patch indices
    (patch_utils.py:157-172); seed ``random`` to make runs repeatable, as with the reference."""
    order = list(range(n_patches))
    random.shuffle(order)
    return [order[i : i + batch_size] for i in range(0, n_patches, batch_size)]


def estimate_local_motion(
    image: torch.Tensor,
    pixel_spacing: float,
    patch_shape: tuple[int, int],
    deformation_field_resolution: tuple[int, int, int],
    initial_deformation_field: torch.Tensor | None,
    device: torch.device = None,
    n_iterations: int = 100,
    b_factor: float = 500,
    frequency_range: tuple[float, float] = (300, 10),
    optimizer_type: str = "adam",
    grid_type: str = "catmull_rom",
    loss_type: str = "mse",
    optimizer_kwargs: dict | None = None,
    return_trajectory: bool = False,
    trajectory_kwargs: dict | None = None,
    _stats: torch.Tensor | None = None,
) -> torch.Tensor | tuple[torch.Tensor, OptimizationTracker]:
    """Optimise a learnable (2, nt, nh, nw) spline grid added to a frozen base grid so that the
    Fourier-shifted patches of every frame agree with the mean of the other frames.

    Reference: estimate_motion_optimizer.py:28-439.  Returns the (2, nt, nh, nw) Angstrom field
    (and an ``OptimizationTracker`` when ``return_trajectory``)."""
    dev = resolve_device(image, device)
    if return_trajectory:
        trajectory_kwargs = trajectory_kwargs if trajectory_kwargs is not None else {}
        trajectory_kwargs.setdefault("sample_every_n_steps", 1)
        trajectory_kwargs.setdefault("total_steps", n_iterations)
        trajectory = OptimizationTracker(**trajectory_kwargs)
    problem = LocalMotionProblem(
        image, pixel_spacing, patch_shape, deformation_field_resolution, initial_deformation_field, dev, b_factor,
        frequency_range, grid_type, loss_type, stats=_stats,
    )
    kwargs = dict(optimizer_kwargs) if optimizer_kwargs is not None else {}
    new = torch.nn.Parameter(torch.zeros((2, *problem.resolution), dtype=torch.float32, device=dev))
    optimizer = _setup_optimizer(optimizer_type, [new], **kwargs)
    is_lbfgs = optimizer_type.lower() == "lbfgs"
    subsample = kwargs.get("lbfgs_patch_subsample", None) if is_lbfgs else None

    if is_lbfgs:
        for iter_idx in range(n_iterations):
            state = {}

            def closure():
                optimizer.zero_grad()
                batches = _shuffled_batches(problem.g, 1)
                if subsample is not None:
                    batches = batches[:subsample]
                if not batches:
                    return torch.tensor(0.0, device=dev, requires_grad=True)
                scale = [s / len(batches) for s in problem.patch_scales(batches)]
                loss, grad = problem.loss_and_grad(new.data, torch.tensor(scale, dtype=torch.float32).to(dev))
                new.grad = grad
                state["loss"] = loss.to(torch.float32).reshape(())
                return state["loss"]

            step_loss = optimizer.step(closure)
            if return_trajectory and trajectory.sample_this_step(iter_idx):
                trajectory.add_checkpoint(deformation_field=new.data, loss=float(step_loss), step=iter_idx)
    elif n_iterations > 0:
        # the mini-batch weighting of every iteration, uploaded once (same random.shuffle stream as the reference)
        all_batches = [_shuffled_batches(problem.g, 8) for _ in range(n_iterations)]
        scales = to_device_async(torch.tensor([problem.patch_scales(b) for b in all_batches], dtype=torch.float32), dev)
        counter = torch.zeros((1,), dtype=torch.int32, device=dev)
        fused = problem.loss_type != 2  # mse / cc: the kernel picks the row from the device-side counter

        # default optimiser: the Adam update is one fused kernel reading the device-side step counter
        # (torch.optim.Adam's foreach path costs ~15 launches for these <= few hundred parameters)
        fused_adam = optimizer_type.lower() == "adam" and not kwargs.get("amsgrad", False)
        if fused_adam:
            adam = fused_adam_state(new.data, kwargs)
            exp_avg, exp_avg_sq, lr, b1, b2, eps, wd = adam

        def one_step(i: int):
            if problem.fused:
                loss, grad = problem.loss_and_grad(new.data, scales, row=i)
            elif fused:
                loss, grad = problem.loss_and_grad(new.data, scales, counter)
            else:
                loss, grad = problem.loss_and_grad(new.data, scales[i])
            if fused_adam:
                with torch.cuda.device(dev):
                    call("tmc_adam_step", ptr(new.data), ptr(grad), ptr(exp_avg), ptr(exp_avg_sq), new.numel(), lr, b1, b2,
                         eps, wd, ptr(counter), stream_ptr(dev))
            else:
                new.grad = grad
                optimizer.step()
            with torch.cuda.device(dev):
                call("tmc_advance_counter", ptr(counter), stream_ptr(dev))
            return loss

        done = 0
        if problem.fused and fused_adam and not return_trajectory:
            losses = torch.empty((n_iterations,), dtype=torch.float64, device=dev)
            problem.fused_steps(new.data, scales, 0, n_iterations, 0, losses, adam)
            done = n_iterations
        elif fused and not problem.fused and not return_trajectory and n_iterations >= 4 and (fused_adam or _graph_capable(optimizer)):
            done = _run_captured(one_step, n_iterations, dev)
        for iter_idx in range(done, n_iterations):
            loss = one_step(iter_idx)
            if return_trajectory and trajectory.sample_this_step(iter_idx):
                trajectory.add_checkpoint(
                    deformation_field=new.data, loss=float(loss) / len(all_batches[iter_idx]), step=iter_idx
                )

    final = (new.data + problem.base).contiguous()
    _ops.subtract_mean(final)
    if return_trajectory:
        return final, trajectory
    return final
