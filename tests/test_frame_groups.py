"""Frame grouping without a GPU: the group layout and the time table tau of frame_groups, the argument checks of the
Python entry points, and the argument checks of tmc_group_frames / tmc_spline_lattice_times (made before any CUDA
call)."""

import numpy as np
import pytest
import torch

from torch_motion_correction_b200 import _lib
from torch_motion_correction_b200.frame_groups import frame_groups

FRAMES = [2, 3, 10, 41, 400, 401]


def _cases():
    for t in FRAMES:
        for g in sorted({1, 2, 10, t // 2}):
            yield t, g


@pytest.mark.parametrize("t,g", list(_cases()))
def test_layout_and_times(t, g):
    if g < 1 or t // g < 2:
        with pytest.raises(ValueError):
            frame_groups(t, g)
        return
    fg = frame_groups(t, g)
    n = t // g
    assert fg.n_groups == n and fg.group_size == g
    # every frame in exactly one group, groups contiguous and in order, the last one taking the leftovers
    member = np.concatenate([np.full(c, i) for i, c in enumerate(fg.counts)])
    assert len(member) == t
    assert np.array_equal(member, fg.group_of(np.arange(t)))
    assert np.array_equal(fg.starts, np.concatenate([[0], np.cumsum(fg.counts)[:-1]]))
    assert np.all(fg.counts[:-1] == g) and fg.counts[-1] == g + t % g
    assert np.array_equal(fg.centres, fg.starts + (fg.counts - 1) / 2)
    # tau(c_g) = g / (n - 1)
    assert np.array_equal(fg.time_at(fg.centres), np.arange(n) / (n - 1))
    tau = fg.times
    assert tau.dtype == np.float32 and tau.shape == (t,)
    assert np.all(np.diff(tau.astype(np.float64)) > 0)
    # rounded once from float64
    assert np.array_equal(tau, fg.time_at(np.arange(t)).astype(np.float32))
    # linear beyond the outer centres: the first and last segments extended
    f = np.arange(t, dtype=np.float64)
    slope0 = 1 / ((n - 1) * (fg.centres[1] - fg.centres[0]))
    slope1 = 1 / ((n - 1) * (fg.centres[-1] - fg.centres[-2]))
    lo, hi = f <= fg.centres[0], f >= fg.centres[-1]
    assert np.allclose(fg.time_at(f[lo]), (f[lo] - fg.centres[0]) * slope0, rtol=0, atol=1e-12)
    assert np.allclose(fg.time_at(f[hi]), 1 + (f[hi] - fg.centres[-1]) * slope1, rtol=0, atol=1e-12)
    if g == 1:
        assert np.allclose(tau, torch.linspace(0, 1, t).numpy(), rtol=0, atol=2.0**-24)
        assert tau[0] == 0 and tau[-1] == 1
    else:
        assert tau[0] < 0 and tau[-1] > 1  # the outer half groups lie outside [0, 1]: not clamped


@pytest.mark.parametrize("t,g", [(10, 0), (10, -2), (10, 6), (401, 201), (1, 1), (5, 2.0), (5, "2"), (5, True), (5, None)])
def test_bad_group_sizes_raise(t, g):
    with pytest.raises(ValueError):
        frame_groups(t, g)


def test_numpy_integers_are_accepted():
    assert frame_groups(10, np.int64(3)).n_groups == 3


def test_entry_points_reject_bad_frame_group_without_a_gpu():
    """the layout is checked on the host before any device work"""
    import torch_motion_correction_b200 as tmc

    one_frame = torch.zeros((1, 8, 8))
    field = torch.zeros((2, 1, 1, 1))
    movie = torch.zeros((10, 8, 8))
    for call in (
        lambda: tmc.group_frames(one_frame, 1),
        lambda: tmc.group_frames(movie, 0),
        lambda: tmc.group_frames(movie, 6),
        lambda: tmc.estimate_motion(one_frame, 1.0, frame_group=2),
        lambda: tmc.motion_correct(movie, 1.0, frame_group=2.5),
    ):
        with pytest.raises(ValueError):
            call()
    if not torch.cuda.is_available():
        return
    for call in (  # these resolve the device first
        lambda: tmc.correct_motion(movie, field, 1.0, frame_group=6),
        lambda: tmc.correct_motion_sum(movie, field, 1.0, frame_group=0),
        lambda: tmc.correct_motion_sums(movie, field, 1.0, frame_group=11),
    ):
        with pytest.raises(ValueError):
            call()


def test_c_abi_rejects_bad_arguments_before_any_cuda_call():
    fake = 1 << 20  # never dereferenced: validation fails first
    bad_group_frames = [
        ((None, 10, 8, 8, 2, fake, None), "null pointer"),
        ((fake, 10, 8, 8, 2, None, None), "null pointer"),
        ((fake, 0, 8, 8, 2, fake, None), "bad movie shape"),
        ((fake, 10, 8, 0, 2, fake, None), "bad movie shape"),
        ((fake, 10, 8, 8, 0, fake, None), "frame_group must be >= 1"),
        ((fake, 10, 8, 8, 6, fake, None), "give 1 groups"),
        ((fake, 1, 8, 8, 1, fake, None), "give 1 groups"),
    ]
    for args, msg in bad_group_frames:
        with pytest.raises(ValueError, match=msg):
            _lib.call("tmc_group_frames", *args)
    # coeffs, c, n0, n1, n2, kind, coeffs2, m0, m1, m2, kind2, n_frames, times, lh, lw, lattice, workspace, stream
    good = [fake, 2, 3, 4, 4, 1, None, 1, 1, 1, 0, 5, fake, 40, 40, fake, fake, None]
    bad_lattice = [
        ({0: None}, "null coefficient pointer"),
        ({12: None}, "null pointer"),
        ({15: None}, "null pointer"),
        ({16: None}, "null pointer"),
        ({11: 0}, "bad sizes"),
        ({13: 0}, "bad sizes"),
        ({5: 3}, "kind must be"),
        ({6: fake, 7: 0}, "bad grid shape"),
    ]
    for change, msg in bad_lattice:
        args = list(good)
        for i, v in change.items():
            args[i] = v
        with pytest.raises(ValueError, match=msg):
            _lib.call("tmc_spline_lattice_times", *args)
