"""The tail of the patch estimator (tmc_xc_postprocess: per-frame outlier rejection, accumulation onto the base field,
Savitzky-Golay smoothing, one joint mean removed) against a float64 restatement of estimate_motion_xc.py."""

import numpy as np
import pytest
import scipy.signal
import torch

from torch_motion_correction_b200 import _lib, _ops

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def reference(shifts, base, px, skip_frame, reject, threshold, smooth, window):
    """shifts (t, g, 2) px, base (2, t, g) Angstrom -> (2, t, g) float64.  Lower median, unbiased std (NaN for one
    patch: nothing rejected), rejected patches replaced by the mean of the kept ones (the median if none is kept);
    savgol_filter(polyorder=1, mode="interp") with the window made odd and capped at t (an even t caps it at an even
    value, quirk Q9), skipped below 3; one joint mean removed."""
    t, g, _ = shifts.shape
    field = base.astype(np.float64).copy()
    for k in range(t):
        if k == skip_frame:
            continue
        v = shifts[k].astype(np.float64).T.copy()  # (2, g)
        if reject:
            med = np.sort(v, axis=1)[:, (g - 1) // 2]
            with np.errstate(invalid="ignore", divide="ignore"):
                sd = v.std(axis=1, ddof=1) if g > 1 else np.full(2, np.nan)
                sd = np.where(np.isnan(sd), sd, np.maximum(sd, 1e-6))
                z = np.abs(v - med[:, None]) / sd[:, None]
            bad = (z > threshold).any(axis=0)
            fill = v[:, ~bad].mean(axis=1) if (~bad).any() else med
            v[:, bad] = fill[:, None]
        field[:, k] += v * px
    if smooth:
        w = window + 1 if window % 2 == 0 else window
        w = min(w, t)
        if w >= 3:
            field = scipy.signal.savgol_filter(field, w, 1, axis=1, mode="interp")
    return field - field.mean()


def run(dev, shifts, base, px, skip_frame=-1, reject=True, threshold=1.5, smooth=True, window=5):
    t, g, _ = shifts.shape
    field = torch.as_tensor(base, dtype=torch.float32).reshape(2, t, g, 1).to(dev).contiguous()
    _ops.xc_postprocess(torch.as_tensor(shifts, dtype=torch.float32).to(dev).contiguous(), field, px, skip_frame, reject,
                        threshold, smooth, window)
    got = field.cpu().double().numpy().reshape(2, t, g)
    want = reference(shifts, base, px, skip_frame, reject, threshold, smooth, window)
    scale = max(1.0, float(np.abs(want).max()))
    assert np.abs(got - want).max() <= 2e-6 * scale, (np.abs(got - want).max(), scale)
    return got


def random_case(t, g, seed):
    rng = np.random.default_rng(seed)
    shifts = rng.normal(0.0, 1.0, (t, g, 2)).astype(np.float32)
    shifts[:, : max(1, g // 10)] *= 6.0  # a few outliers per frame
    base = rng.normal(0.0, 2.0, (2, t, g)).astype(np.float32)
    return shifts, base


@pytest.mark.parametrize("t,window", [(6, 5), (4, 5), (8, 7), (4, 3), (6, 9), (7, 9), (5, 4), (9, 6), (2, 5), (1, 5),
                                      (3, 3), (12, 3)])
def test_windows(dev, t, window):
    """Even windows capped by an even frame count, requests of at least t, even requests (made odd), and t = 1, 2
    where the capped window is below 3 and nothing is smoothed."""
    shifts, base = random_case(t, 20, 100 * t + window)
    run(dev, shifts, base, 1.3, window=window)
    run(dev, shifts, base, 1.3, window=window, reject=False)


@pytest.mark.parametrize("g", [1, 2, 3, 127, 128, 129, 300])
def test_patch_counts(dev, g):
    """g = 1: NaN std, nothing rejected; g > 128: several strides of the 128-thread CTA."""
    shifts, base = random_case(7, g, g)
    run(dev, shifts, base, 0.83)
    run(dev, shifts, base, 0.83, threshold=0.5, smooth=False)


def test_ties_at_the_median(dev):
    t, g = 5, 9
    shifts = np.tile(np.array([2.0, 2.0, 2.0, 2.0, 5.0, -1.0, 2.0, 2.0, 9.0], np.float32)[:, None], (t, 1, 2))
    shifts[:, :, 1] = np.array([0.5, 0.5, -3.0, 0.5, 0.5, 4.0, 0.5, 0.25, 0.5], np.float32)
    shifts += np.arange(t, dtype=np.float32)[:, None, None]
    base = np.zeros((2, t, g), np.float32)
    run(dev, shifts, base, 1.0, threshold=1.0)
    run(dev, shifts, base, 1.0, threshold=0.1, smooth=False)


def test_values_exactly_at_the_threshold(dev):
    """Values -1, -1, 0, 1, 1: lower median 0, unbiased std exactly 1, z = 1 for four of them.  z > threshold
    rejects, z == threshold keeps."""
    t, g = 3, 5
    row = np.array([-1.0, 1.0, 0.0, 1.0, -1.0], np.float32)
    shifts = np.stack([np.tile(row, (t, 1)), np.tile(row[::-1], (t, 1))], axis=2) * 4.0
    base = np.zeros((2, t, g), np.float32)
    kept = run(dev, shifts, base, 1.0, threshold=1.0, smooth=False)
    assert np.ptp(kept[:, 0]) > 0  # nothing replaced
    rejected = run(dev, shifts, base, 1.0, threshold=np.nextafter(np.float32(1.0), np.float32(0.0)), smooth=False)
    assert np.ptp(rejected[:, 0]) == 0  # all four replaced by the mean of the middle value


def test_negative_threshold_replaces_every_patch_by_the_median(dev):
    shifts, base = random_case(6, 11, 4)
    got = run(dev, shifts, np.zeros_like(base), 1.0, threshold=-1.0, smooth=False)
    assert np.ptp(got[0, 2]) == 0 and np.ptp(got[1, 4]) == 0
    run(dev, shifts, base, 1.0, threshold=-1.0)


@pytest.mark.parametrize("skip_frame", [0, 3, 6])
def test_skip_frame(dev, skip_frame):
    shifts, base = random_case(7, 16, 10 + skip_frame)
    run(dev, shifts, base, 1.1, skip_frame=skip_frame)
    run(dev, shifts, base, 1.1, skip_frame=skip_frame, reject=False, smooth=False)


def test_launch_count_without_smoothing_or_mean(dev):
    """Only the rejection kernel runs when smoothing and the mean removal are off."""
    shifts = torch.zeros((4, 3, 2), dtype=torch.float32, device=dev)
    field = torch.zeros((2, 4, 3), dtype=torch.float32, device=dev)
    scratch = torch.empty_like(field)
    before = _lib.query("tmc_launch_count")
    with torch.cuda.device(dev):
        _lib.call("tmc_xc_postprocess", _lib.ptr(shifts), 4, 3, 1.0, -1, 1, 1.5, 0, 5, 0, _lib.ptr(field), _lib.ptr(scratch),
                  _lib.stream_ptr(dev))
    assert _lib.query("tmc_launch_count") - before == 1
