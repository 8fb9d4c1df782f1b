"""CUDA warp / spline / statistics kernels against the CPU oracle and the golden vectors."""

import numpy as np
import pytest
import torch

import torch_motion_correction_b200 as tmc
from oracle import deps
from oracle import reference_path as rp
from torch_motion_correction_b200 import _lib, _ops
from warp_kernels import at_offset, warp_kernels_ran

pytestmark = pytest.mark.gpu

# north-star tolerances
REL_L2 = 1e-4  # corrected frames / frame sums, fp32
SHIFT_PX = 0.01  # shifts


def rel_l2(a, b):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return float(torch.linalg.norm(a - b) / torch.linalg.norm(b))


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def small(golden_small):
    g = golden_small
    return g, torch.as_tensor(g["movie"]), float(g["pixel_spacing"])


def test_stack_stats(dev):
    g = torch.Generator().manual_seed(0)
    for shape in [(5, 64, 64), (3, 130, 77), (2, 512, 1024)]:
        img = torch.randn(shape, generator=g) * 3.0 + 10.0
        t, h, w = shape
        box = img[:, int(0.25 * h) : int(0.75 * h), int(0.25 * w) : int(0.75 * w)]
        std, mean = torch.std_mean(box)
        got = _ops.stack_stats(img.to(dev)).cpu()
        assert abs(float(got[0] - mean)) <= 1e-5 * abs(float(mean))
        assert abs(float(got[1] - std)) <= 1e-5 * float(std)


@pytest.mark.parametrize("grid_type", ["catmull_rom", "bspline"])
@pytest.mark.parametrize("shape", [(3, 4, 4), (6, 1, 1), (2, 2, 5), (1, 3, 3), (40, 6, 6)])
def test_spline_eval(dev, grid_type, shape):
    g = torch.Generator().manual_seed(4)
    field = torch.randn((2, *shape), generator=g)
    tyx = torch.rand((1000, 3), generator=g)
    tyx[0] = 0.0
    tyx[1] = 1.0
    want = rp.evaluate_deformation_field(field, tyx, grid_type)
    got = tmc.evaluate_deformation_field(field.to(dev), tyx.to(dev), grid_type).cpu()
    assert float((got - want).abs().max()) <= 2e-6 * max(1.0, float(want.abs().max()))


def test_spline_eval_golden(dev, small):
    g, _, _ = small
    field = torch.as_tensor(g["field_344"]).to(dev)
    tyx = torch.as_tensor(g["tyx"]).to(dev)
    for name, kind in (("eval_catmull", "catmull_rom"), ("eval_bspline", "bspline")):
        got = tmc.evaluate_deformation_field(field, tyx, kind).cpu()
        assert float((got - torch.as_tensor(g[name])).abs().max()) <= 5e-6
    got = tmc.evaluate_deformation_field(torch.as_tensor(g["field_611"]).to(dev), tyx, "catmull_rom").cpu()
    assert float((got - torch.as_tensor(g["eval_611_catmull"])).abs().max()) <= 5e-6
    got = tmc.resample_deformation_field(field, (5, 3, 4)).cpu()
    assert float((got - torch.as_tensor(g["resample_to_534"])).abs().max()) <= 5e-6
    lat = tmc.evaluate_deformation_field_at_t(field, 0.4, (40, 40), "bspline").cpu()
    assert float((lat - torch.as_tensor(g["lattice_t04_bspline"])).abs().max()) <= 5e-6


@pytest.mark.parametrize("grid_type", ["catmull_rom", "bspline"])
def test_spline_backward_is_transpose(dev, grid_type):
    g = torch.Generator().manual_seed(5)
    shape = (2, 3, 5, 4)
    tyx = torch.rand((333, 3), generator=g)
    go = torch.randn((333, 2), generator=g)
    coeffs = torch.randn(shape, generator=g, requires_grad=True)
    kind = 0 if grid_type == "catmull_rom" else 1
    out = deps.evaluate_cubic_grid_3d(coeffs, tyx, rp._matrix(grid_type))
    (out * go).sum().backward()
    got = _ops.spline_eval_backward(shape, kind, tyx.to(dev), go.to(dev), scale=-0.5).cpu()
    assert float((got - (-0.5) * coeffs.grad).abs().max()) <= 1e-4 * float(coeffs.grad.abs().max())
    # singleton axes
    shape = (2, 4, 1, 1)
    coeffs = torch.randn(shape, generator=g, requires_grad=True)
    out = deps.evaluate_cubic_grid_3d(coeffs, tyx, rp._matrix(grid_type))
    (out * go).sum().backward()
    got = _ops.spline_eval_backward(shape, kind, tyx.to(dev), go.to(dev)).cpu()
    assert float((got - coeffs.grad).abs().max()) <= 1e-4 * float(coeffs.grad.abs().max())


def test_pixel_shifts_golden(dev, small):
    g, movie, px = small
    lat = torch.as_tensor(g["lattice_t04_bspline"]).to(dev)
    got = tmc.get_pixel_shifts(movie[0].to(dev), px, lat, None).cpu()
    assert float((got - torch.as_tensor(g["pixel_shifts"])).abs().max()) <= 1e-5


def test_correct_motion_golden(dev, small):
    g, movie, px = small
    m = movie.to(dev)
    field = torch.as_tensor(g["field_344"]).to(dev)
    # the corrected stacks are stored for every other row
    assert rel_l2(tmc.correct_motion(m, field, px)[:, ::2], g["correct_catmull"]) <= REL_L2
    assert rel_l2(tmc.correct_motion(m, field, px, grid_type="bspline")[:, ::2], g["correct_bspline"]) <= REL_L2
    f1 = torch.as_tensor(g["field_611"]).to(dev)
    assert rel_l2(tmc.correct_motion(m, f1, px)[:, ::2], g["correct_611_catmull"]) <= REL_L2
    assert rel_l2(tmc.correct_motion_slow(m, field)[:, ::2], g["correct_slow"]) <= REL_L2
    new = torch.as_tensor(g["two_grids_new"]).to(dev)
    assert rel_l2(tmc.correct_motion_two_grids(m, new, field, px, grad=False)[:, ::2], g["correct_two_grids"]) <= REL_L2
    s = tmc.correct_motion_sum(m, field, px, grid_type="bspline")
    assert rel_l2(s[::2], torch.as_tensor(g["correct_bspline"]).sum(dim=0)) <= REL_L2


def test_zero_field_is_identity(dev):
    """The reference's only numeric assertions (tests/test_correct_motion.py:132-145,241-252)."""
    g = torch.Generator().manual_seed(2)
    img = torch.randn((5, 64, 64), generator=g).to(dev)
    zero = torch.zeros((2, 5, 2, 2), device=dev)
    assert torch.allclose(tmc.correct_motion(img, zero, 1.0), img, atol=1e-4)
    assert torch.allclose(tmc.correct_motion_slow(img, zero), img, atol=1e-4)


@pytest.mark.parametrize("shape", [(4, 130, 77), (3, 257, 300)])
def test_correct_motion_ragged_sizes_and_big_shifts(dev, shape):
    """Odd sizes, shifts that push samples outside the frame (zero fill) and across borders."""
    t, h, w = shape
    g = torch.Generator().manual_seed(8)
    img = torch.randn(shape, generator=g)
    field = torch.randn((2, 3, 3, 4), generator=g) * 12.0
    want = rp.correct_motion(img, field, 0.9, "bspline")
    got = tmc.correct_motion(img.to(dev), field.to(dev), 0.9, grid_type="bspline")
    assert rel_l2(got, want) <= REL_L2
    assert float((want == 0).float().mean()) > 0.01  # the case really exercises the zero fill


@pytest.mark.parametrize("layout", ["aligned", "offset"])
@pytest.mark.parametrize("amplitude", [2.0, 40.0])
@pytest.mark.parametrize("shape,grid", [((5, 300, 388), (3, 4, 5)), ((3, 331, 260), (3, 2, 2)), ((41, 64, 128), (41, 1, 1))])
def test_correct_motion_tma_tiles(dev, shape, grid, amplitude, layout):
    """Images with 16-byte aligned rows run on the TMA-staged tile kernel (one float off: the global-memory kernel):
    smooth fields (taps inside the staged boxes), a wild field (boxes hang over the frame edge, taps leave the boxes:
    per-pixel fall-backs, zero fill outside the frame), ragged tile edges, more frames than pipeline stages, stack
    output and fused sum, accumulation into an existing sum."""
    g = torch.Generator().manual_seed(21)
    img = torch.randn(shape, generator=g)
    field = torch.randn((2, *grid), generator=g) * amplitude
    want = rp.correct_motion(img, field, 1.1, "bspline")
    m = img.to(dev) if layout == "aligned" else at_offset(img.to(dev))
    _lib.kernel_timing(True)
    got = tmc.correct_motion(m, field.to(dev), 1.1, grid_type="bspline")
    assert rel_l2(got, want) <= REL_L2
    total = tmc.correct_motion_sum(m, field.to(dev), 1.1, grid_type="bspline")
    assert rel_l2(total, want.sum(dim=0)) <= REL_L2
    # accumulate into an existing sum (frame blocks of one movie)
    again = total.clone()
    tmc.correct_motion_sum(m, field.to(dev), 1.1, grid_type="bspline", out=again, accumulate=True)
    assert rel_l2(again, 2 * want.sum(dim=0)) <= REL_L2
    assert warp_kernels_ran() == {"warp_tma_kernel" if layout == "aligned" else "warp_lattice_kernel"}


def test_tma_and_global_memory_kernels_agree(dev):
    """Same arithmetic up to the evaluation order of the Keys weights: 2048^2, shifts of a few pixels plus one corner
    pushed far outside, normalised output.  The frames one float off their allocation run on the global-memory kernel."""
    g = torch.Generator().manual_seed(5)
    img = torch.randn((7, 2048, 2048), generator=g).to(dev)
    field = torch.randn((2, 3, 5, 5), generator=g) * 4.0
    field[:, :, 0, 0] = 90.0
    field = field.to(dev)
    from torch_motion_correction_b200 import _ops
    from torch_motion_correction_b200._common import grid_kind

    stats = _ops.stack_stats(img)
    lattice = _ops.spline_lattice(field, grid_kind("bspline"), 7, 50, 50)
    outs = {}
    for tma, frames, kernel in (("1", img, "warp_tma_kernel"), ("0", at_offset(img), "warp_lattice_kernel")):
        stack, total = torch.empty_like(img), torch.empty_like(img[0])
        _lib.kernel_timing(True)
        _ops.warp_lattice(frames, lattice, 0.83, mean_std=stats, out_stack=stack, out_sum=total)
        assert warp_kernels_ran() == {kernel}
        outs[tma] = (stack, total)
    # the kernels evaluate the Keys weights in different (equivalent) orders: ~1e-7 per weight, 16 taps
    assert rel_l2(outs["1"][0], outs["0"][0]) <= 5e-6
    assert rel_l2(outs["1"][1], outs["0"][1]) <= 5e-6
    assert rel_l2(outs["1"][1], outs["1"][0].sum(dim=0)) <= 1e-6


def test_frame_split_sum_matches_whole(dev):
    """Frame-split (multi-GPU style) partial sums add up to the whole-movie sum."""
    movie, _ = rp.synthetic_movie(8, 128, 128, seed=5)
    g = torch.Generator().manual_seed(3)
    field = (torch.randn((2, 4, 3, 3), generator=g) * 2).to(dev)
    m = movie.to(dev)
    whole = tmc.correct_motion_sum(m, field, 1.1, grid_type="bspline")
    part = tmc.correct_motion_sum(m[:3], field, 1.1, grid_type="bspline", frame_offset=0, total_frames=8)
    part = tmc.correct_motion_sum(m[3:], field, 1.1, grid_type="bspline", out=part, accumulate=True, frame_offset=3, total_frames=8)
    assert rel_l2(part, whole) <= 1e-6
    want = rp.correct_motion(movie, field.cpu(), 1.1, "bspline").sum(dim=0)
    assert rel_l2(whole, want) <= REL_L2


@pytest.mark.parametrize("grid_type", ["catmull_rom", "bspline"])
def test_two_grids_gradient_matches_autograd(dev, grid_type):
    """d(sum w * corrected) / d(new grid coefficients): CUDA backward kernels vs autograd through the oracle."""
    from torch_motion_correction_b200.spline_grids import CubicBSplineGrid3d, CubicCatmullRomGrid3d

    movie, _ = rp.synthetic_movie(4, 96, 80, seed=6, noise=0.2, sigma_f=0.05)
    g = torch.Generator().manual_seed(12)
    new = (torch.randn((2, 3, 3, 2), generator=g) * 1.5).requires_grad_(True)
    base = torch.randn((2, 3, 3, 2), generator=g) * 1.5
    weights = torch.randn(movie.shape, generator=g)
    out = rp.correct_motion_two_grids(movie, new, base, 1.2, grid_type)
    (out * weights).sum().backward()
    cls = CubicBSplineGrid3d if grid_type == "bspline" else CubicCatmullRomGrid3d
    new_mod = cls.from_grid_data(new.detach()).to(dev)
    base_mod = cls.from_grid_data(base).to(dev)
    got = tmc.correct_motion_two_grids(movie.to(dev), new_mod, base_mod, 1.2, grad=True)
    assert got.requires_grad and rel_l2(got.detach(), out.detach()) <= REL_L2
    (got * weights.to(dev)).sum().backward()
    grad = new_mod.data.grad.cpu()
    assert float((grad - new.grad).abs().max()) <= 2e-3 * float(new.grad.abs().max())
