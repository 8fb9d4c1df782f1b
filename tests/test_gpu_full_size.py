"""BASELINE.json's full-size configuration (C2: 40 x 4096 x 4096 fp32, 1024-px patches, (3, 5, 5) spline grid) through
size-independent properties -- the oracle would need ~10 minutes per call at this size: known integer drifts are
recovered exactly, a zero field is the identity up to grid_sample's fp32 coordinate round trip, the fused warp-and-sum
is linear in the movie and equals the sum of the warped stack, integer Fourier shifts are circular rolls, the
one-launch-per-iteration optimiser agrees with the generic kernels, and the dose-weighted sum has the filter's DC gain."""

import os
import random
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import bench  # noqa: E402  (the seeded synthetic-movie generator of the benchmark)
import torch_motion_correction_b200 as tmc  # noqa: E402

pytestmark = pytest.mark.gpu

T, H, W, P, PX = 40, 4096, 4096, 1024, 0.83


def rel_l2(a, b):
    return float(torch.linalg.norm((a - b).double()) / torch.linalg.norm(b.double()))


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def movie_and_walk(dev):
    movie, walk = bench.synthetic_movie_gpu(T, H, W, 4242, dev)
    yield movie, walk
    del movie
    torch.cuda.empty_cache()


def test_known_integer_drift_is_recovered_exactly(dev, movie_and_walk):
    movie, walk = movie_and_walk
    field = tmc.estimate_global_motion(movie, PX)
    assert field.shape == (2, T, 1, 1)
    got_px = torch.round(field[:, :, 0, 0].T.cpu() / PX).long()
    assert torch.equal(got_px, walk), (got_px - walk).abs().max()
    assert torch.allclose(field[:, :, 0, 0].T.cpu(), walk.float() * PX, atol=1e-5)


def test_patch_xc_on_top_of_the_global_field_stays_sub_pixel(dev, movie_and_walk):
    """The synthetic movie has rigid integer drift only: after the rigid pre-correction every patch shift is < 1 px and
    the cumulative field stays within a pixel of the global one."""
    movie, walk = movie_and_walk
    g = tmc.estimate_global_motion(movie, PX)
    f, centres = tmc.estimate_motion_cross_correlation_patches(movie, PX, patch_sidelength=P, deformation_field=g.clone())
    assert f.shape == (2, T, 6, 6) and centres.shape == (T, 6, 6, 3)
    assert centres[0, :, 0, 1].tolist() == [512, 1126, 1740, 2355, 2969, 3583]
    assert bool(torch.isfinite(f).all())
    assert abs(float(f.mean())) < 1e-4  # quirk Q4: one joint mean removed


def test_zero_field_is_identity_up_to_the_coordinate_round_trip(dev, movie_and_walk):
    movie, _ = movie_and_walk
    zero = torch.zeros((2, 3, 5, 5), device=dev)
    total = tmc.correct_motion_sum(movie, zero, PX, grid_type="bspline")
    assert rel_l2(total, movie.sum(dim=0)) <= 1e-4  # SURVEY D.4: 3.5e-5 on white noise at 4096^2


def test_fused_sum_is_linear_and_equals_the_sum_of_the_stack(dev, movie_and_walk):
    movie, _ = movie_and_walk
    g = torch.Generator().manual_seed(9)
    field = (torch.randn((2, 3, 5, 5), generator=g) * 3.0).to(dev)
    s1 = tmc.correct_motion_sum(movie, field, PX, grid_type="bspline")
    sub = movie[:8]
    stack = tmc.correct_motion(sub, field, PX, grid_type="bspline")
    fused = tmc.correct_motion_sum(sub, field, PX, grid_type="bspline")
    assert rel_l2(fused, stack.sum(dim=0)) <= 1e-6
    s2 = tmc.correct_motion_sum(movie * 2.5 + 1.0, field, PX, grid_type="bspline")
    # a constant image warps to the constant wherever the sample stays inside the frame (|shift| < 64 px here)
    inner = (slice(64, -64), slice(64, -64))
    assert rel_l2((s2 - 2.5 * s1)[inner], torch.full_like(s1, float(T))[inner]) <= 1e-4


def test_integer_fourier_shift_is_a_circular_roll(dev, movie_and_walk):
    movie, _ = movie_and_walk
    sub = movie[:4].contiguous()
    field = torch.tensor([[3.0, -7.0, 0.0, 12.0], [-5.0, 2.0, 0.0, 1.0]], device=dev).reshape(2, 4, 1, 1)
    out = tmc.correct_motion_fast(sub, field.clone())  # quirk Q2: content moves by -field, Angstrom taken as px
    for k in range(4):
        want = torch.roll(sub[k], shifts=(-int(field[0, k]), -int(field[1, k])), dims=(0, 1))
        assert rel_l2(out[k], want) <= 2e-5, k


def test_fourier_shift_column_strips_match_a_float64_shift(dev, movie_and_walk):
    """4096-point whole-frame columns run on the 4-column strip kernel (cols_shift_quad_p2): fractional shifts against
    the same Fourier shift in float64 (content moves by -field, quirk Q2)."""
    from torch_motion_correction_b200 import _lib

    movie, _ = movie_and_walk
    sub = movie[:6].contiguous()
    field = torch.tensor([[1.3, -2.7, 0.0, 4.25, -0.5, 7.9], [-3.1, 0.4, 0.0, 2.5, 6.6, -1.2]], device=dev).reshape(2, 6, 1, 1)
    _lib.kernel_timing(True)
    got = tmc.correct_motion_fast(sub, field.clone())
    torch.cuda.synchronize()
    assert "cols_shift_quad_p2" in _lib.kernel_timing_report()
    _lib.kernel_timing(False)
    fy = torch.fft.fftfreq(H, dtype=torch.float64, device=dev)[:, None]
    fx = torch.fft.rfftfreq(W, dtype=torch.float64, device=dev)[None, :]
    worst = 0.0
    for k in range(6):
        phase = torch.exp(2j * torch.pi * (fy * float(field[0, k]) + fx * float(field[1, k])))
        want = torch.fft.irfft2(torch.fft.rfft2(sub[k].double()) * phase, s=(H, W))
        worst = max(worst, rel_l2(got[k], want))
    print(f"[fourier shift] cols_shift_quad_p2 vs float64: worst rel-L2 {worst:.2e}")
    assert worst <= 2e-6  # 6.6e-7 measured on a B200 (1000 W)
    assert rel_l2(got[2], sub[2]) <= 2e-5  # zero shift


def test_one_launch_iterations_agree_with_the_generic_kernels(dev, movie_and_walk, monkeypatch):
    from torch_motion_correction_b200 import estimate_motion_optimizer as emo

    movie, _ = movie_and_walk
    init = torch.zeros((2, T, 6, 6), device=dev)
    kw = dict(n_iterations=8, grid_type="bspline")
    random.seed(3)
    fused = tmc.estimate_local_motion(movie, PX, (P, P), (3, 5, 5), init, **kw)
    monkeypatch.setattr(emo, "FUSED_STEPS", False)
    random.seed(3)
    generic = tmc.estimate_local_motion(movie, PX, (P, P), (3, 5, 5), init, **kw)
    assert float(generic.abs().max()) > 1e-3
    assert float((fused - generic).abs().max()) <= 0.01 * PX  # north-star tolerance on shifts


def test_dose_weighted_sum_dc_gain_and_linearity(dev, movie_and_walk):
    movie, _ = movie_and_walk
    sub = movie[:6] + 5.0
    out = tmc.dose_weight(sub, PX, pre_exposure=0.0, dose_per_frame=1.5)
    # DC: every frame weighs 1 / sqrt(T)
    assert abs(float(out.mean()) - float(sub.sum(dim=0).mean()) / 6**0.5) <= 1e-4 * abs(float(out.mean()))
    out2 = tmc.dose_weight(sub * 3.0, PX, pre_exposure=0.0, dose_per_frame=1.5)
    assert rel_l2(out2, 3.0 * out) <= 1e-5


def test_whole_pipeline_on_the_benchmark_workload(dev, movie_and_walk):
    movie, walk = movie_and_walk
    random.seed(0)
    total, field = tmc.motion_correct(movie, PX, patch_sidelength=P, deformation_field_resolution=(3, 5, 5), n_iterations=20)
    assert total.shape == (H, W) and field.shape == (2, 3, 5, 5)
    assert bool(torch.isfinite(total).all()) and bool(torch.isfinite(field).all())
    # aligning sharpens the sum: more variance than the unaligned sum of the drifting frames
    assert float(total[64:-64, 64:-64].var()) > 1.2 * float(movie.sum(dim=0)[64:-64, 64:-64].var())
