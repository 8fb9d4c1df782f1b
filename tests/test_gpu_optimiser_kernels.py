"""Spline-optimiser kernels against a float64 reference, at the shapes and settings where they can go wrong.

Every case evaluates one loss and gradient with ``LocalMotionProblem.loss_and_grad`` twice: on the tiled two-kernel
iteration (csrc/optimizer_tiled.cu) and on the generic kernels (csrc/optimizer.cu), and compares both with
``rp.loss_and_grad`` run in float64 (autograd through the reference's own ``irfftn`` path).  The Adam tests pin the
fused optimiser update (tmc_local_steps modes 0, 2, 3) against ``torch.optim.Adam`` and the reference loss.

Worst cases measured on a B200 (1000 W power limit) are listed in the comments beside the tolerances."""

import random
from dataclasses import dataclass

import pytest
import torch

from oracle import reference_path as rp
from torch_motion_correction_b200 import _lib
from torch_motion_correction_b200 import estimate_motion_optimizer as emo
from torch_motion_correction_b200.estimate_motion_optimizer import LocalMotionProblem

pytestmark = pytest.mark.gpu

# The spectra and the per-bin arithmetic are float32, the loss sums are float64.  Measured worst cases over all
# cases and both paths: loss 1.2e-6 (mse, T = 3; the tiled path's float32 Sigma), gradient 6.5e-6 (the widest grid);
# the generic kernels before they formed the Hermitian part of the Nyquist bins: loss 8e-5 .. 1.6e-4 on nyquist_*.
LOSS_RTOL = 1e-5
GRAD_TOL = 2e-4  # max-abs error / max |reference gradient|

# band settings: name -> (b_factor, frequency_range as a function of the pixel spacing)
BANDS = {
    "default": lambda px: (500, (300, 10)),
    # cut-on close to the cutoff: the tiles inside the inner radius hold no pass-band bin and are dropped
    "annular": lambda px: (0, (4 * px, 3 * px)),
    # cutoff at 2 px: the band box holds every ky (ky_start = -(ny // 2))
    "full_ky": lambda px: (500, (300, 2 * px)),
    # as full_ky with no B-factor: non-zero weight on the Nyquist column and on the ky = -ny/2 bin of the DC column
    "nyquist": lambda px: (0, (300, 2 * px)),
    # a band box of several 8 x 16 tiles in both directions
    "multi_tile": lambda px: (500, (300, 3)),
}


@dataclass(frozen=True)
class Case:
    branch: str  # what the case exists for
    t: int
    frame: tuple
    patch: tuple
    res: tuple
    loss: str = "mse"
    grid: str = "catmull_rom"
    band: str = "default"
    px: float = 1.0
    large_shifts: bool = False  # initial field of +-40 px: the phase range reduction of fast_cis
    subset: bool = False  # only some patches weighted, the others have patch_scale 0
    noise: bool = False  # noise-dominated content (sigma_f 0.3): power up to the Nyquist bins
    tiled: bool = True  # False: the tiled iteration must refuse the problem


def _max_grid_supported(g: int, t: int, nt: int) -> int:
    """Largest nh * nw that tmc_local_steps accepts for this problem."""
    n = 1
    while _lib.query("tmc_local_steps_supported", g, t, nt, n + 1):
        n += 1
    return n


CASES = {
    "t2_leave_one_out_factor_2": Case("T = 2: a = T / (T - 1) = 2", 2, (96, 96), (32, 32), (2, 3, 3), loss="cc"),
    "t3_odd_frames_grid_1": Case("odd T: empty half-warp in pass 2, empty second slot of the frame-pair jobs; (1, 1, 1) grid",
                                 3, (96, 96), (32, 32), (1, 1, 1), grid="bspline", px=0.83),
    "t8_one_full_chunk_bluestein": Case("T = 8: one full 8-frame chunk; 48-px (Bluestein) patches; a subset of patches",
                                        8, (144, 144), (48, 48), (3, 3, 3), loss="cc", grid="bspline", subset=True),
    "t9_partial_chunk_non_square": Case("T = 9: a last chunk of one frame; 64 x 48 patches; (T, 2, 2) grid; +-40 px",
                                        9, (128, 120), (64, 48), (9, 2, 2), px=0.83, large_shifts=True),
    "t17_odd_side_full_ky": Case("T = 17: partial chunk; odd 33-px side; every ky in the band box", 17, (99, 99), (33, 33),
                                 (3, 3, 3), loss="cc", band="full_ky"),
    "t40_annular_band": Case("annular band: tiles without pass-band bins dropped; 128-px patches", 40, (256, 256), (128, 128),
                             (3, 2, 2), grid="bspline", band="annular"),
    "t61_multi_tile_band_box": Case("T = 61; frequency_range (300, 3): a multi-tile band box; +-40 px; a subset of patches",
                                    61, (256, 256), (128, 128), (3, 3, 3), loss="cc", band="multi_tile", px=0.83,
                                    large_shifts=True, subset=True),
    "t157_largest_tiled": Case("T = 157: the largest frame count of the tiled iteration (200 KB tile)", 157, (64, 64),
                               (32, 32), (3, 2, 2), grid="bspline"),
    "t158_generic_fallback": Case("T = 158: the first frame count the tiled iteration refuses", 158, (64, 64), (32, 32),
                                  (3, 2, 2), loss="cc", tiled=False),
    "nyquist_mse_even_full_ky": Case("even side, full ky, weight on the Nyquist bins: 'mse' stays on the tiled path", 6,
                                     (96, 96), (32, 32), (3, 3, 3), band="nyquist", noise=True),
    "nyquist_cc": Case("'cc' with weight on the Nyquist bins: irfftn keeps only their Hermitian part", 6, (96, 96),
                       (32, 32), (3, 3, 3), loss="cc", band="nyquist", noise=True, tiled=False),
    "nyquist_cc_odd_nyquist_column": Case("'cc', Nyquist column kx = 15 on an odd tile column (30-px side), 0.83 A", 5,
                                          (90, 90), (30, 30), (2, 2, 2), loss="cc", band="nyquist", noise=True, px=0.83,
                                          tiled=False),
    "nyquist_ncc": Case("'ncc' with weight on the Nyquist bins", 6, (96, 96), (32, 32), (3, 3, 3), loss="ncc",
                        grid="bspline", band="nyquist", noise=True, tiled=False),
    "ncc_default": Case("'ncc' (generic kernels only), default band, +-40 px", 9, (96, 96), (32, 32), (3, 3, 3),
                        loss="ncc", large_shifts=True, tiled=False),
    "grid_at_limit": Case("the largest nh * nw the coefficient kernel's 160 KB shared memory takes", 3, (96, 96), (32, 32),
                          (3, 0, 0), grid="bspline"),
    "grid_past_limit": Case("one past that grid size: generic kernels", 3, (96, 96), (32, 32), (3, 0, 1), loss="cc",
                            tiled=False),
    "t40_production_1024": Case("1024-px patches at T = 40, 2 patches per frame: the production band box (~22 x 6 tiles)",
                                40, (1024, 1537), (1024, 1024), (3, 1, 2)),
}


def _resolution(case: Case, g: int):
    """(nt, 0, 0): nh * nw at the tiled iteration's limit; (nt, 0, 1): one column of nodes past it."""
    nt, nh, nw = case.res
    if nh != 0:
        return case.res
    limit = _max_grid_supported(g, case.t, nt)
    nh = next((d for d in range(2, 9) if limit % d == 0), 2)
    return (nt, nh, limit // nh + nw)


def _movie(case: Case, seed: int) -> torch.Tensor:
    """Band-limited specimen moved by a whole-pixel random walk, plus white noise (float64)."""
    gen = torch.Generator().manual_seed(seed)
    t, (h, w) = case.t, case.frame
    sigma_f, noise = (0.3, 1.0) if case.noise else (0.08, 0.3)
    white = torch.randn((h + 16, w + 16), generator=gen, dtype=torch.float64)
    fy = torch.fft.fftfreq(h + 16, dtype=torch.float64)[:, None]
    fx = torch.fft.rfftfreq(w + 16, dtype=torch.float64)[None, :]
    spec = torch.fft.irfftn(torch.fft.rfftn(white) * torch.exp(-(fy**2 + fx**2) / (2 * sigma_f**2)), s=white.shape)
    spec = spec / spec.std()
    walk = torch.cumsum(torch.randint(-1, 2, (t, 2), generator=gen), dim=0).clamp(-8, 8) + 8
    frames = [spec[int(dy) : int(dy) + h, int(dx) : int(dx) + w] for dy, dx in walk.tolist()]
    movie = torch.stack(frames) + noise * torch.randn((t, h, w), generator=gen, dtype=torch.float64)
    # float32 values: the kernels and the reference see the same movie
    return movie.float().double()


def _batches(g: int, subset: bool, seed: int):
    """Ragged mini-batches (8, 5, rest) of a shuffled patch order, or (subset) a few patches of it."""
    order = list(range(g))
    random.Random(seed).shuffle(order)
    if subset:
        return [order[: max(1, g // 2)]]
    out = [order[:8], order[8:13], order[13:]]
    return [b for b in out if b]


_REFERENCE: dict = {}


def _problem_inputs(name: str):
    case = CASES[name]
    seed = sum(map(ord, name))
    movie = _movie(case, seed)
    ph, pw = case.patch
    centers = rp.patch_grid_centers((case.t, *case.frame), (1, ph, pw), (1, ph // 2, pw // 2))
    g = centers.shape[1] * centers.shape[2]
    res = _resolution(case, g)
    gen = torch.Generator().manual_seed(seed + 1)
    if case.large_shifts:
        init = (torch.rand((2, 3, 3, 3), generator=gen, dtype=torch.float64) * 80 - 40) * case.px
    else:
        init = torch.randn((2, 3, 3, 3), generator=gen, dtype=torch.float64) * 0.3
    new = torch.randn((2, *res), generator=gen, dtype=torch.float64) * 0.3
    batches = [[i] for i in range(g)] if ph >= 1024 else _batches(g, case.subset, seed)
    b_factor, fr = BANDS[case.band](case.px)
    return case, movie, res, init, new, batches, b_factor, fr


def _reference(name: str):
    if name not in _REFERENCE:
        case, movie, res, init, new, batches, b_factor, fr = _problem_inputs(name)
        loss, grad = rp.loss_and_grad(movie, case.px, case.patch, res, init, new, batches, b_factor=b_factor,
                                      frequency_range=fr, grid_type=case.grid, loss_type=case.loss)
        assert grad.dtype == torch.float64
        _REFERENCE[name] = (loss, grad)
    return _REFERENCE[name]


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


PATHS = [(n, p) for n in CASES for p in (("tiled", "generic") if CASES[n].tiled else ("generic",))]


@pytest.mark.parametrize("name,path", PATHS, ids=[f"{n}-{p}" for n, p in PATHS])
def test_loss_and_gradient_match_float64_reference(dev, monkeypatch, record_property, name, path):
    case, movie, res, init, new, batches, b_factor, fr = _problem_inputs(name)
    if path == "generic":
        monkeypatch.setattr(emo, "FUSED_STEPS", False)
    prob = LocalMotionProblem(movie.float().to(dev), case.px, case.patch, res, init.float().to(dev), dev, b_factor, fr,
                              case.grid, case.loss)
    if path == "tiled":
        assert prob.fused
    if not case.tiled:
        monkeypatch.setattr(emo, "FUSED_STEPS", True)
        refused = LocalMotionProblem(movie.float().to(dev), case.px, case.patch, res, init.float().to(dev), dev, b_factor,
                                     fr, case.grid, case.loss)
        assert not refused.fused, "the tiled iteration must not take this problem"
    scale = torch.tensor(prob.patch_scales(batches), dtype=torch.float32).to(dev)
    loss, grad = prob.loss_and_grad(new.float().to(dev), scale)
    loss, grad = float(loss), grad.double().cpu()
    want_loss, want_grad = _reference(name)
    loss_err = abs(loss - want_loss) / abs(want_loss)
    grad_scale = float(want_grad.abs().max())
    if res[0] == 1:
        # one node in time moves every frame alike: the leave-one-out losses do not depend on it, the reference
        # gradient is round-off (~1e-10); bound the kernels' round-off by the loss per Angstrom instead (measured 6.5e-5)
        grad_scale = max(grad_scale, 1e-3 * abs(want_loss))
    grad_err = float((grad - want_grad).abs().max()) / grad_scale
    record_property("loss_rel_err", loss_err)
    record_property("grad_rel_err", grad_err)
    assert loss_err <= LOSS_RTOL, (loss, want_loss, loss_err)
    assert grad_err <= GRAD_TOL, grad_err


# ---- Adam ---------------------------------------------------------------------------------------------------------------

ADAM = dict(lr=0.05, betas=(0.8, 0.99), eps=1e-6, weight_decay=0.01)
N_STEPS = 5


@pytest.fixture(scope="module")
def adam_problem():
    """A cc problem on the tiled path with the mini-batch rows of N_STEPS iterations."""
    case = Case("Adam", 7, (96, 96), (32, 32), (3, 3, 3), loss="cc", grid="bspline", px=0.83)
    movie = _movie(case, 5)
    init = torch.randn((2, 3, 3, 3), generator=torch.Generator().manual_seed(6), dtype=torch.float64) * 0.5
    return case, movie, init


def _scales(prob, n_patches: int):
    rows = [_batches(n_patches, False, 100 + i) for i in range(N_STEPS)]
    return rows, torch.tensor([prob.patch_scales(b) for b in rows], dtype=torch.float32).to(prob.dev)


def test_fused_adam_matches_torch_adam_and_reference_loss(dev, adam_problem, record_property):
    case, movie, init = adam_problem
    prob = LocalMotionProblem(movie.float().to(dev), case.px, case.patch, case.res, init.float().to(dev), dev, 500, (300, 10),
                              case.grid, case.loss)
    assert prob.fused
    rows, scales = _scales(prob, prob.g)
    lr, (b1, b2), eps, wd = ADAM["lr"], ADAM["betas"], ADAM["eps"], ADAM["weight_decay"]
    adam_args = lambda ea, eas: (ea, eas, lr, b1, b2, eps, wd)  # noqa: E731

    # mode 0, all steps in one call (the estimate_local_motion path)
    coef = torch.zeros((2, *case.res), dtype=torch.float32, device=dev)
    ea, eas = torch.zeros_like(coef), torch.zeros_like(coef)
    losses = torch.zeros((N_STEPS,), dtype=torch.float64, device=dev)
    prob.fused_steps(coef, scales, 0, N_STEPS, 0, losses, adam_args(ea, eas))

    # mode 0, one step per call: the coefficients each row's loss was evaluated at
    step = torch.zeros_like(coef)
    sea, seas = torch.zeros_like(coef), torch.zeros_like(coef)
    step_losses = torch.zeros((N_STEPS,), dtype=torch.float64, device=dev)
    before = []
    for i in range(N_STEPS):
        before.append(step.double().cpu())
        prob.fused_steps(step, scales, i, 1, 0, step_losses, adam_args(sea, seas))
    assert float((step - coef).abs().max()) <= 1e-6 * max(1.0, float(coef.abs().max()))

    # (a) mode-1 gradients of the same kernel, fed to a float32 torch.optim.Adam
    param = torch.nn.Parameter(torch.zeros_like(coef))
    opt = torch.optim.Adam([param], **ADAM)
    worst = 0.0
    for i in range(N_STEPS):
        loss, grad = prob.loss_and_grad(param.data, scales, row=i)
        param.grad = grad.clone()
        opt.step()
        # a few float32 ulp per step (the gradient is the same kernel's; Adam's arithmetic order differs): measured 8.9e-8
        err = float((param.data - before[i + 1].float().to(dev) if i + 1 < N_STEPS else param.data - coef).abs().max())
        worst = max(worst, err)
        assert err <= 4 * (i + 1) * 2.0**-23 * max(lr, float(coef.abs().max())), (i, err)
    record_property("adam_vs_torch_max_abs", worst)

    # (b) every row's loss against the float64 reference at the same coefficients
    worst = 0.0
    for i in range(N_STEPS):
        want, _ = rp.loss_and_grad(movie, case.px, case.patch, case.res, init, before[i], rows[i], b_factor=500,
                                   frequency_range=(300, 10), grid_type=case.grid, loss_type=case.loss)
        for got in (float(losses[i]), float(step_losses[i])):
            err = abs(got - want) / abs(want)
            worst = max(worst, err)
            assert err <= LOSS_RTOL, (i, got, want)
    record_property("adam_loss_rel_err", worst)


def test_frame_split_adam_modes_match_one_call(dev, adam_problem, record_property):
    """Modes 1 -> 2 ... -> 3 of tmc_local_steps (the frame-split optimiser, world size 1) against mode 0."""
    from torch_motion_correction_b200 import _ops
    from torch_motion_correction_b200.distributed import estimate_local_motion_frame_split
    import torch_motion_correction_b200 as tmc

    case, movie, init = adam_problem
    m, i0 = movie.float().to(dev), init.float().to(dev)
    kw = dict(n_iterations=N_STEPS, b_factor=500, frequency_range=(300, 10), grid_type=case.grid, loss_type=case.loss,
              optimizer_kwargs=ADAM)
    random.seed(21)
    want = tmc.estimate_local_motion(m, case.px, case.patch, case.res, i0, **kw)
    random.seed(21)
    got = estimate_local_motion_frame_split(m, case.px, case.patch, case.res, i0, 0, case.t, _ops.stack_stats(m), **kw)
    err = float((got - want).abs().max())
    record_property("split_vs_mode0_max_abs", err)
    # the same kernels on patch-major instead of frame-pair-major spectra: float32 sums in another order (measured 1.2e-7)
    assert err <= 1e-5 * max(1.0, float(want.abs().max())), err
