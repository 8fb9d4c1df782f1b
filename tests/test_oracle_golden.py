"""The CPU oracle (``oracle.reference_path``) against the committed golden vectors that the
UNMODIFIED reference produced (``tests/golden/make_golden.py``).  CPU only."""

import random

import numpy as np
import pytest
import torch

from oracle import deps
from oracle import reference_path as rp

# the oracle follows the reference op-for-op on the CPU, so the match is (near) bit-exact
TOL = 1e-6


def close(a, b, tol=TOL):
    a = torch.as_tensor(a)
    b = torch.as_tensor(b)
    assert a.shape == b.shape
    assert float((a - b).abs().max()) <= tol * max(1.0, float(b.abs().max()))


@pytest.fixture(scope="module")
def small(golden_small):
    g = golden_small
    return g, torch.as_tensor(g["movie"]), float(g["pixel_spacing"]), tuple(float(v) for v in g["frequency_range"])


def test_global_motion(small):
    g, movie, px, fr = small
    close(rp.estimate_global_motion(movie, px, frequency_range=fr), g["global_field"])
    close(
        rp.estimate_global_motion(movie, px, reference_frame=0, b_factor=1000, frequency_range=fr),
        g["global_field_ref0_b1000"],
    )


@pytest.mark.parametrize("strategy", ["mean_except_current", "middle_frame"])
def test_xc_patches(small, strategy):
    g, movie, px, fr = small
    f, pos = rp.estimate_motion_cross_correlation_patches(
        movie, px, reference_strategy=strategy, patch_sidelength=32, frequency_range=fr, smooth=False, reject_outliers=False
    )
    close(f, g[f"xc_raw_{strategy}"])
    f, pos = rp.estimate_motion_cross_correlation_patches(
        movie, px, reference_strategy=strategy, patch_sidelength=32, frequency_range=fr,
        smoothing_window_size=3, outlier_threshold=1.5,
    )
    close(f, g[f"xc_full_{strategy}"])
    assert np.array_equal(pos.numpy(), g["xc_positions"])


def test_xc_integer_and_cumulative(small):
    g, movie, px, fr = small
    f, _ = rp.estimate_motion_cross_correlation_patches(
        movie, px, patch_sidelength=32, frequency_range=fr, sub_pixel=False, smooth=False, reject_outliers=False
    )
    close(f, g["xc_integer"])
    g0 = torch.as_tensor(g["global_field"]).clone()
    f, _ = rp.estimate_motion_cross_correlation_patches(movie, px, patch_sidelength=32, frequency_range=fr, deformation_field=g0)
    close(f, g["xc_cumulative_global"])
    close(g0, g["xc_cumulative_global_field_after"])  # Q2: caller's field negated in place
    f, _ = rp.estimate_motion_cross_correlation_patches(
        movie, px, patch_sidelength=32, frequency_range=fr,
        deformation_field=torch.as_tensor(g["xc_cumulative_full_in"]).clone(),
    )
    close(f, g["xc_cumulative_full"])


def test_correction(small):
    g, movie, px, _ = small
    field = torch.as_tensor(g["field_344"])
    field1 = torch.as_tensor(g["field_611"])
    # the corrected stacks are stored for every other row
    close(rp.correct_motion(movie, field, px)[:, ::2], g["correct_catmull"])
    close(rp.correct_motion(movie, field, px, "bspline")[:, ::2], g["correct_bspline"])
    close(rp.correct_motion(movie, field1, px)[:, ::2], g["correct_611_catmull"])
    fast_in = field1.clone()
    close(rp.correct_motion_fast(movie, fast_in)[:, ::2], g["correct_fast"], 1e-5)
    close(fast_in, g["correct_fast_field_after"])
    close(rp.correct_motion_slow(movie, field)[:, ::2], g["correct_slow"])
    close(rp.correct_motion_two_grids(movie, torch.as_tensor(g["two_grids_new"]), field, px)[:, ::2], g["correct_two_grids"])
    with pytest.raises(ValueError, match="Expected single patch deformation field"):
        rp.correct_motion_fast(movie, field.clone())


def test_field_utils(small):
    g, movie, px, _ = small
    field = torch.as_tensor(g["field_344"])
    field1 = torch.as_tensor(g["field_611"])
    lat = rp.evaluate_deformation_field_at_t(field, 0.4, (40, 40), "bspline")
    close(lat, g["lattice_t04_bspline"])
    close(rp.get_pixel_shifts(movie[0], px, lat, deps.coordinate_grid((96, 96))), g["pixel_shifts"])
    tyx = torch.as_tensor(g["tyx"])
    close(rp.evaluate_deformation_field(field, tyx), g["eval_catmull"])
    close(rp.evaluate_deformation_field(field, tyx, "bspline"), g["eval_bspline"])
    close(rp.evaluate_deformation_field(field1, tyx), g["eval_611_catmull"])
    close(rp.resample_deformation_field(field, (5, 3, 4)), g["resample_to_534"])


LOCAL_CASES = {
    "adam_catmull_mse": dict(optimizer_type="adam", grid_type="catmull_rom", loss_type="mse"),
    "adam_bspline_mse": dict(optimizer_type="adam", grid_type="bspline", loss_type="mse"),
    "sgd_bspline_ncc": dict(optimizer_type="sgd", grid_type="bspline", loss_type="ncc"),
    "rmsprop_catmull_cc": dict(optimizer_type="rmsprop", grid_type="catmull_rom", loss_type="cc", optimizer_kwargs={"lr": 0.001}),
    "lbfgs_bspline_mse": dict(optimizer_type="lbfgs", grid_type="bspline", loss_type="mse"),
}


@pytest.mark.parametrize("name", list(LOCAL_CASES))
def test_local_motion(small, name):
    g, movie, px, fr = small
    init = torch.as_tensor(g["xc_full_mean_except_current"])
    random.seed(1234)
    res, losses = rp.estimate_local_motion(
        movie, px, (32, 32), (3, 3, 3), init.clone(), n_iterations=6, frequency_range=fr, return_losses=True,
        **LOCAL_CASES[name],
    )
    close(res, g[f"local_{name}"], 1e-5)
    assert np.allclose(np.asarray(losses), g[f"local_{name}_losses"], rtol=1e-5, atol=1e-7)


def test_local_motion_no_initial_field(small):
    g, movie, px, fr = small
    random.seed(77)
    res = rp.estimate_local_motion(movie, px, (48, 48), (2, 2, 2), None, n_iterations=4, frequency_range=fr)
    close(res, g["local_noinit_p48"], 1e-5)


@pytest.mark.parametrize("strategy", ["mean_except_current", "middle_frame"])
def test_eviction_regime(golden_eviction, strategy):
    """T = 60 > 50 cached frames: Q1's irregular double-masking pattern (SURVEY Appendix D.5)."""
    g = golden_eviction
    movie = torch.as_tensor(g["movie"].astype(np.float32))
    fr = tuple(float(v) for v in g["frequency_range"])
    f, _ = rp.estimate_motion_cross_correlation_patches(
        movie, 1.0, reference_strategy=strategy, patch_sidelength=32, frequency_range=fr, smooth=False, reject_outliers=False
    )
    close(f, g[f"xc_raw_{strategy}"])


def test_q1_schedule_structure():
    """T <= 50: frame k's reference holds exactly the k earlier frames double-masked."""
    sched = rp.q1_schedule(12, "mean_except_current", 6)
    for k, row in sched.items():
        assert row == [1 if j < k else 0 for j in range(12)]
    sched = rp.q1_schedule(12, "middle_frame", 6)
    assert [sched[k] for k in sorted(sched)] == list(range(1, 12))
    # T > 50 is irregular
    sched = rp.q1_schedule(60, "mean_except_current", 30)
    assert any(sum(row) != k for k, row in sched.items())


def test_c1_known_answer(golden_c1):
    """BASELINE config 1: 10x512x512 with known integer drifts (SURVEY Appendix D.3)."""
    g = golden_c1
    movie, walk = rp.synthetic_movie(10, 512, 512, seed=0, noise=1.0, drift=6.0, integer_shifts=True, sigma_f=0.08)
    assert np.array_equal(walk.numpy(), g["true_shifts"])
    gf = rp.estimate_global_motion(movie, 1.0)
    close(gf, g["global_field"])
    # reference recovers the integer drift exactly (relative to the middle frame)
    assert torch.equal(gf[:, :, 0, 0].T, walk)
    f, pos = rp.estimate_motion_cross_correlation_patches(movie, 1.0, patch_sidelength=128)
    close(f, g["xc_field"])
    assert np.array_equal(pos.numpy(), g["xc_positions"])
    s = rp.correct_motion(movie, f, 1.0, "bspline").sum(dim=0)
    close(s[192:320, 192:320], g["corrected_sum_crop"], 1e-5)
    close(s[::64, :], g["corrected_sum_rows"], 1e-5)
