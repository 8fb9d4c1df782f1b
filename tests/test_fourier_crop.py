"""Fourier cropping without a GPU: the shape rule of fourier_crop_shape, the errors fourier_crop raises before any CUDA
call, and the argument checks of tmc_fourier_crop (made before any CUDA call)."""

import numpy as np
import pytest
import torch

import torch_motion_correction_b200 as tmc
from torch_motion_correction_b200 import _lib
from torch_motion_correction_b200.prepare import fourier_crop_shape

SIDES = [(4096, 4096), (8192, 8192), (5760, 4092), (11520, 8184), (1024, 768)]
FACTORS = [1, 1.5, 2, 3, 4]

# (h, w), factor -> expected output, worked out by hand
EXPECTED = {
    ((4096, 4096), 2): (2048, 2048),
    ((4096, 4096), 4): (1024, 1024),
    ((8192, 8192), 2): (4096, 4096),
    ((8192, 8192), 4): (2048, 2048),
    ((5760, 4092), 2): (2880, 2046),
    ((5760, 4092), 1.5): (3840, 2728),
    ((5760, 4092), 3): (1920, 1364),
    ((11520, 8184), 1.5): (7680, 5456),
    ((11520, 8184), 2): (5760, 4092),
    ((11520, 8184), 3): (3840, 2728),
    ((11520, 8184), 4): (2880, 2046),
    ((1024, 768), 2): (512, 384),
    ((1024, 768), 4): (256, 192),
}


@pytest.mark.parametrize("sides", SIDES)
@pytest.mark.parametrize("factor", FACTORS)
def test_shape_rule(sides, factor):
    if factor == 1:
        assert fourier_crop_shape(sides, factor) == sides
        return
    want = EXPECTED.get((sides, factor))
    if want is None:  # some side divided by the factor is not an even whole number
        with pytest.raises(ValueError, match="not an even whole number"):
            fourier_crop_shape(sides, factor)
        return
    assert fourier_crop_shape(sides, factor) == want
    assert fourier_crop_shape(sides, float(factor)) == want
    assert fourier_crop_shape(sides, np.float32(factor)) == want


def test_factors_that_miss_a_whole_number_by_rounding_only():
    # 5760 / (5760 / 3840) is 3840 to within float rounding
    assert fourier_crop_shape((5760, 4092), 5760 / 3840) == (3840, 2728)
    with pytest.raises(ValueError, match="not an even whole number"):
        fourier_crop_shape((4096, 4096), 2.0001)


@pytest.mark.parametrize("factor", [0.5, 0, -2, float("nan"), float("inf"), True, "2", None, 2 + 0j])
def test_factor_must_be_a_real_number_of_at_least_one(factor):
    with pytest.raises(ValueError, match="factor must be a real number >= 1"):
        fourier_crop_shape((1024, 1024), factor)


@pytest.mark.parametrize("sides,factor", [((1023, 1024), 2), ((1024, 1022), 2), ((1024, 1024), 1024),
                                          ((1024, 1024), 1024 / 3), ((96, 96), 2 * 48 / 47)])
def test_sides_must_be_even_before_and_after(sides, factor):
    with pytest.raises(ValueError):
        fourier_crop_shape(sides, factor)


def test_odd_sides_are_fine_at_factor_one():
    assert fourier_crop_shape((1023, 1025), 1) == (1023, 1025)


def test_lengths_without_full_spectrum_transforms_are_not_implemented():
    assert _lib.query("tmc_fft_supported_length", 16392) == 2 and _lib.query("tmc_fft_supported_length", 8196) == 1
    with pytest.raises(NotImplementedError, match="transform length 16392 is not supported"):
        fourier_crop_shape((16392, 16392), 2)  # the input
    assert _lib.query("tmc_fft_supported_length", 16384) == 1 and _lib.query("tmc_fft_supported_length", 13000) == 2
    with pytest.raises(NotImplementedError, match="transform length 13000 is not supported"):
        fourier_crop_shape((16384, 16384), 16384 / 13000)  # the output


@pytest.mark.parametrize("shape,factor,error", [((4, 64, 64), 0.5, ValueError), ((4, 63, 64), 2, ValueError),
                                                ((4, 64, 64), 3, ValueError), ((64,), 2, ValueError),
                                                ((2, 2, 64, 64), 2, ValueError), ((0, 64, 64), 2, ValueError),
                                                ((2, 16392, 16392), 2, NotImplementedError)])
def test_fourier_crop_raises_before_any_cuda_call(shape, factor, error):
    image = torch.empty(shape, dtype=torch.float32, device="meta")  # no data: the checks must come first
    with pytest.raises(error):
        tmc.fourier_crop(image, factor)


def test_factor_one_returns_the_input_itself():
    image = torch.zeros((3, 7, 9))
    assert tmc.fourier_crop(image, 1) is image
    assert tmc.fourier_crop(image, 1.0) is image
    frame = image[0]
    assert tmc.fourier_crop(frame, 1) is frame


def _crop_args(**kw):
    args = dict(image=16, t=2, h=64, w=64, out_h=32, out_w=32, jobs=16, njobs=1, plan_x=16, plan_y=16, plan_x_out=16,
                plan_y_out=16, workspace=16, out=16, stream=None)
    args.update(kw)
    return list(args.values())


@pytest.mark.parametrize("kw,match", [
    (dict(image=None), "null pointer"), (dict(jobs=None), "null pointer"), (dict(plan_y_out=None), "null pointer"),
    (dict(workspace=None), "null pointer"), (dict(out=None), "null pointer"),
    (dict(njobs=0), "jobs do not cover"), (dict(t=5, njobs=2), "jobs do not cover"), (dict(njobs=2), "jobs do not cover"),
    (dict(h=63), "sides must be even"), (dict(out_w=31), "sides must be even"), (dict(out_h=0), "sides must be even"),
    (dict(out_h=128), "larger than the input"), (dict(out_w=66), "larger than the input"),
])
def test_entry_point_rejects_bad_arguments(kw, match):
    with pytest.raises(ValueError, match=match):
        _lib.call("tmc_fourier_crop", *_crop_args(**kw))


def test_entry_point_reports_unsupported_lengths():
    with pytest.raises(NotImplementedError, match="transform length 16392"):
        _lib.call("tmc_fourier_crop", *_crop_args(h=16392, w=16392, out_h=8196, out_w=8196))


def test_workspace_query():
    q = lambda *a: _lib.query("tmc_fourier_crop_workspace_bytes", *a)
    assert q(40, 8192, 8192, 4096, 4096) == 40 * (8192 + 4096) * 2049 * 8
    assert q(3, 64, 64, 32, 32) == 4 * (64 + 32) * 17 * 8  # an odd frame count rounds up to whole frame pairs
    assert q(0, 64, 64, 32, 32) == -1
