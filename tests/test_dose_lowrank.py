"""Low-rank factorisation of the exposure filter behind ``correct_motion_sums`` (float64 host code), and the argument
checks of ``correct_motion_sums`` and of its C-ABI entry points (no CUDA call: runs without a GPU)."""

import importlib

import numpy as np
import pytest
import torch

from torch_motion_correction_b200 import _build, _lib
from torch_motion_correction_b200.correct_motion import correct_motion_sums

dw = importlib.import_module("torch_motion_correction_b200.dose_weight")  # the package's `dose_weight` is the function


@pytest.fixture(scope="module", autouse=True)
def library():
    _build.build()  # the size checks query the library (host function, no GPU)


# (frames, A/px, e/A^2/frame, kV): C2, C3, C4, few high-dose frames, super-resolution, 400 and 2000 low-dose fractions
CONFIGS = [(40, 0.83, 1.0, 300), (60, 0.83, 1.0, 300), (40, 0.415, 1.0, 300), (10, 0.83, 5.0, 300), (20, 0.3, 2.0, 300),
           (400, 0.83, 0.1, 300), (2000, 0.83, 0.02, 300), (40, 0.83, 1.0, 200)]


@pytest.mark.parametrize("t,px,dose,kv", CONFIGS)
def test_rank_of_real_exposures_is_at_most_8(t, px, dose, kv):
    for half in (False, True):
        f = dw.exposure_filter_lowrank(4096, 4096, px, range(t), dose, voltage=kv, half_sets=half)
        for name, g in f.groups.items():
            assert 1 <= g.basis.shape[1] <= 8, (name, g.basis.shape)
            assert g.residual <= dw.LOWRANK_TOLERANCE
            np.testing.assert_allclose(g.basis.T @ g.basis, np.eye(g.basis.shape[1]), atol=1e-12)


def _worst_bin_residual(f, ny, nx, px, exposures, frames, kv):
    """max over every bin of the (ny, nx) rfft grid of || w(k) - sum_groups U v(x(k)) ||_2 over the frames"""
    x = dw.rfft_grid_x(ny, nx, px, kv).ravel()
    nodes = np.linspace(0.0, f.x_max, dw.LOWRANK_TABLE_NODES)
    worst = 0.0
    for c0 in range(0, x.size, 1 << 16):
        xc = x[c0 : c0 + (1 << 16)]
        err = dw.exposure_weights(xc, exposures)
        for g in f.groups.values():
            v = np.stack([np.interp(xc, nodes, row) for row in g.table])
            err[np.searchsorted(frames, g.frames)] -= g.basis @ v
        worst = max(worst, float(np.sqrt((err * err).sum(0)).max()))
    return worst


@pytest.mark.parametrize("ny,nx", [(256, 384), (600, 5000), (255, 97)])
@pytest.mark.parametrize("px", [0.83, 1.0])
@pytest.mark.parametrize("half", [False, True])
def test_residual_at_every_bin_of_real_grids(ny, nx, px, half):
    frames = np.arange(40)
    exposures = 0.5 + (frames + 1) * 1.0
    f = dw.exposure_filter_lowrank(ny, nx, px, range(40), 1.0, pre_exposure=0.5, half_sets=half)
    assert _worst_bin_residual(f, ny, nx, px, exposures, frames, 300) <= dw.LOWRANK_TOLERANCE


def test_frame_range_keeps_global_exposure_and_normalises_over_included_frames():
    frames = np.arange(7, 23)
    f = dw.exposure_filter_lowrank(128, 128, 1.0, range(7, 23), 2.0, pre_exposure=1.0, half_sets=True)
    assert sorted(np.concatenate([g.frames for g in f.groups.values()]).tolist()) == frames.tolist()
    assert (f.groups["even"].frames % 2 == 0).all() and (f.groups["odd"].frames % 2 == 1).all()
    exposures = 1.0 + (frames + 1) * 2.0
    assert _worst_bin_residual(f, 128, 128, 1.0, exposures, frames, 300) <= dw.LOWRANK_TOLERANCE


def test_factorisation_is_deterministic():
    a = dw.exposure_filter_lowrank(512, 512, 0.83, range(40), 1.0, half_sets=True)
    dw._exposure_filter_lowrank.cache_clear()
    b = dw.exposure_filter_lowrank(512, 512, 0.83, range(40), 1.0, half_sets=True)
    assert a is not b
    assert a.x_max == b.x_max
    for name in a.groups:
        assert np.array_equal(a.groups[name].table, b.groups[name].table)
        assert np.array_equal(a.groups[name].basis, b.groups[name].basis)


def test_rank_cap_is_a_clear_error(monkeypatch):
    monkeypatch.setattr(dw, "LOWRANK_MAX_RANK", 3)
    dw._exposure_filter_lowrank.cache_clear()
    with pytest.raises(ValueError, match="more than 3 low-rank components"):
        dw.exposure_filter_lowrank(512, 512, 0.83, range(40), 1.0)


def test_inverse_critical_exposure_matches_the_oracle():
    from oracle import deps

    k = np.array([0.0, 1e-3, 0.05, 0.3, 0.85, 2.4])
    for kv in (300.0, 200.0):
        want = 1.0 / deps.critical_exposure(torch.from_numpy(k), kv).numpy()
        np.testing.assert_allclose(dw.inverse_critical_exposure(k, kv), want, rtol=1e-12)


def _args(t=6, h=64, w=64):
    return torch.zeros((t, h, w)), torch.zeros((2, 3, 2, 2)), 1.0


@pytest.mark.parametrize("frame_range", [(3, 3), (4, 2), (-1, 3), (0, 7), (6, 7)])
def test_bad_frame_range_is_rejected(frame_range):
    with pytest.raises(ValueError, match="frame_range"):
        correct_motion_sums(*_args(), frame_range=frame_range)


@pytest.mark.parametrize("dose", [0.0, -1.0, float("nan")])
def test_bad_dose_is_rejected(dose):
    with pytest.raises(ValueError, match="dose_per_frame"):
        correct_motion_sums(*_args(), dose_per_frame=dose)
    with pytest.raises(ValueError, match="dose_per_frame"):
        dw.exposure_filter_lowrank(64, 64, 1.0, range(6), dose)


def test_frame_size_without_full_spectrum_transform_is_rejected():
    # 13000 = 4 x 3250: band-limited transforms only; the plain sums need no transform and are not checked
    with pytest.raises(ValueError, match="transform length 13000 is not supported"):
        correct_motion_sums(*_args(2, 64, 13000), dose_per_frame=1.0)


def test_bad_arguments_of_the_entry_points_are_reported_not_crashed():
    fake = 256  # never dereferenced: validation happens before any CUDA call
    with pytest.raises(ValueError, match="null pointer"):
        _lib.call("tmc_warp_lattice_sums", fake, 4, 64, 64, fake, 30, 30, 1.0, None, 3, fake, fake, None)
    with pytest.raises(ValueError, match="n_sums=20"):
        _lib.call("tmc_warp_lattice_sums", fake, 4, 64, 64, fake, 30, 30, 1.0, fake, 20, fake, fake, None)
    with pytest.raises(ValueError, match="n_sums=0"):
        _lib.call("tmc_warp_lattice_sums", fake, 4, 64, 64, fake, 30, 30, 1.0, fake, 0, fake, fake, None)
    with pytest.raises(ValueError, match="pixel_spacing"):
        _lib.call("tmc_warp_lattice_sums", fake, 4, 64, 64, fake, 30, 30, 0.0, fake, 3, fake, fake, None)
    with pytest.raises(ValueError, match="null pointer"):
        _lib.call("tmc_dose_lowrank_combine", None, 7, 64, 64, 1.0, 300.0, fake, 4096, 0.3, fake, 1, fake, None)
    with pytest.raises(ValueError, match="n_out=4"):
        _lib.call("tmc_dose_lowrank_combine", fake, 7, 64, 64, 1.0, 300.0, fake, 4096, 0.3, fake, 4, fake, None)
    with pytest.raises(ValueError, match="x_max"):
        _lib.call("tmc_dose_lowrank_combine", fake, 7, 64, 64, 1.0, 300.0, fake, 4096, 0.0, fake, 1, fake, None)
