"""Parity of the CUDA path with the UNMODIFIED reference on the benchmarked code paths: 1024-px patches (polyphase row
transforms, tiled optimiser kernels), T = 40 / 60 (the Q1 cache schedule, with eviction for T > 50), 4096-point
whole-frame transforms, (3, 5, 5) / (5, 6, 6) spline grids -- at half size (2048^2) and at BASELINE's full size (4096^2),
plus config 4's frame size (8192^2: 8192-point whole-frame transforms, 15 x 15 / 14 x 14 patch grids) on 10 frames.

The golden vectors were produced in the build container by ``tests/golden/make_golden.py`` (verbatim reference source
on the CPU); only fields, crops and norms are stored.  The movies are regenerated here from their seeds with the same
generator (``oracle.reference_path.synthetic_movie_large`` / ``synthetic_movie``) and checked against a stored probe.

Tolerances (BASELINE.json north star): shifts <= 0.01 px, corrected sums <= 1e-4 relative L2."""

import os
import random

import numpy as np
import pytest
import torch

import torch_motion_correction_b200 as tmc
from oracle import reference_path as rp

from conftest import GOLDEN, load_golden

pytestmark = pytest.mark.gpu

SHIFT_PX = 0.01
SUM_REL = 1e-4
P = 1024


def rel_l2(a, b):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return float(torch.linalg.norm(a - b) / torch.linalg.norm(b))


def sum_samples(s):
    h, w = s.shape
    return {
        "sum_centre": s[h // 2 - 96 : h // 2 + 96, w // 2 - 96 : w // 2 + 96],
        "sum_corner": s[:96, :96],
        "sum_rows": s[:: h // (16 if h <= 4096 else 8), :],  # 8 rows of 8192^2: keeps each golden file under 1 MB
    }


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


CASES = ["c2half", "c3half", "c2full", "c3full", "c4short"]


@pytest.fixture(scope="module", params=CASES)
def case(request, dev):
    """(name, golden dict, movie on the device, pixel spacing); module scope: pytest groups the tests by case, so every
    movie is generated once."""
    name = request.param
    path = os.path.join(GOLDEN, name + ".npz")
    if not os.path.exists(path):
        pytest.skip(f"{name}.npz not generated")
    g = load_golden(name + ".npz")
    t, n = int(g["t"]), int(g["size"])
    movie, walk = rp.synthetic_movie_large(t, n, n, seed=int(g["seed"]), noise=1.0, drift=6.0, local=1.5)
    probe = movie[:: max(t // 4, 1), ::257, ::263].numpy()
    # the generator must reproduce the movie the golden vectors were computed from
    assert np.allclose(probe, g["movie_probe"], atol=2e-5), float(np.abs(probe - g["movie_probe"]).max())
    assert abs(float(movie.double().sum()) - float(g["movie_checksum"])) <= 1e-6 * movie.numel()
    yield name, g, movie.to(dev), float(g["pixel_spacing"])
    torch.cuda.empty_cache()


def test_global_and_patch_cross_correlation(dev, case):
    name, g, movie, px = case
    field = tmc.estimate_global_motion(movie, px)
    assert float((field.cpu() - torch.as_tensor(g["global_field"])).abs().max()) <= 1e-5
    f, pos = tmc.estimate_motion_cross_correlation_patches(movie, px, patch_sidelength=P)
    assert torch.equal(pos.cpu(), torch.as_tensor(g["xc_positions"]))
    err = float((f.cpu() - torch.as_tensor(g["xc_field"])).abs().max())
    assert err <= SHIFT_PX * px, err
    fraw, _ = tmc.estimate_motion_cross_correlation_patches(
        movie, px, patch_sidelength=P, temporal_smoothing=False, outlier_rejection=False)
    err = float((fraw.cpu() - torch.as_tensor(g["xc_raw"])).abs().max())
    assert err <= SHIFT_PX * px, err


def test_patch_cross_correlation_on_a_rigid_pre_field(dev, case):
    """(2, t, 1, 1) field handed over in pixels (the route the pipeline drives): quirk Q2 -- used as px by the rigid
    pre-correction, negated in place, patch shifts accumulated on the negated field."""
    name, g, movie, px = case
    if not name.startswith("c2"):
        pytest.skip("stored for the C2 cases only")
    for key, kw in (("xc_pre_nosmooth", dict(temporal_smoothing=False)), ("xc_pre", {})):
        pre = (torch.as_tensor(g["global_field"]) / px).to(dev)
        f, _ = tmc.estimate_motion_cross_correlation_patches(movie, px, patch_sidelength=P, deformation_field=pre, **kw)
        err = float((f.cpu() - torch.as_tensor(g[key])).abs().max())
        assert err <= SHIFT_PX * px, (key, err)
        assert torch.allclose(pre.cpu(), torch.as_tensor(g["xc_pre_field_after"]), atol=1e-6)


def test_spline_optimiser(dev, case):
    name, g, movie, px = case
    init = torch.as_tensor(g["xc_field"]).to(dev)
    want = torch.as_tensor(g["local_field"])
    random.seed(2024)
    res, traj = tmc.estimate_local_motion(
        movie, px, (P, P), tuple(want.shape[1:]), init, n_iterations=len(g["local_losses"]), grid_type="bspline",
        return_trajectory=True,
    )
    err = float((res.cpu() - want).abs().max())
    assert err <= SHIFT_PX * px, err
    losses = np.asarray([c.loss for c in traj.checkpoints])
    assert np.allclose(losses, g["local_losses"], rtol=2e-3), (losses, g["local_losses"])
    # the one-launch-per-iteration Adam path (no trajectory) must land on the same field
    random.seed(2024)
    fused = tmc.estimate_local_motion(
        movie, px, (P, P), tuple(want.shape[1:]), init, n_iterations=len(g["local_losses"]), grid_type="bspline")
    err = float((fused.cpu() - want).abs().max())
    assert err <= SHIFT_PX * px, err


def test_corrected_sum(dev, case):
    name, g, movie, px = case
    if "sum_norm" not in g:
        pytest.skip("stored for the C2 / C4 cases only")
    field = torch.as_tensor(g["local_field"]).to(dev)
    total = tmc.correct_motion_sum(movie, field, px, grid_type="bspline")
    for key, got in sum_samples(total).items():
        assert rel_l2(got, g[key]) <= SUM_REL, (key, rel_l2(got, g[key]))
    assert abs(float(torch.linalg.norm(total.double())) - float(g["sum_norm"])) <= SUM_REL * float(g["sum_norm"])
    if "xcfield_sum_centre" not in g:
        return
    # the drop-in stack output, summed, and a (2, t, gh, gw) field under the Catmull-Rom default
    stack = tmc.correct_motion(movie[:6], torch.as_tensor(g["xc_field"])[:, :6].contiguous().to(dev), px)
    for key, got in sum_samples(stack.sum(dim=0)).items():
        assert rel_l2(got, g["xcfield_" + key]) <= SUM_REL, (key, rel_l2(got, g["xcfield_" + key]))


@pytest.mark.parametrize("n", [4096, 8192])
def test_whole_frame_transforms(dev, n):
    """n-point row and column transforms: global estimate and rigid Fourier-shift correction of 4 frames."""
    if not os.path.exists(os.path.join(GOLDEN, f"whole{n}.npz")):
        pytest.skip(f"whole{n}.npz not generated")
    g = load_golden(f"whole{n}.npz")
    movie, walk = rp.synthetic_movie(4, n, n, seed=int(g["seed"]), noise=1.0, drift=9.0, integer_shifts=True, sigma_f=0.08)
    assert torch.equal(walk, torch.as_tensor(g["true_shifts"]))
    movie = movie.to(dev)
    px = 0.83
    field = tmc.estimate_global_motion(movie, px)
    assert float((field.cpu() - torch.as_tensor(g["global_field"])).abs().max()) <= 1e-5
    shift = torch.as_tensor(g["fast_field"]).to(dev)
    out = tmc.correct_motion_fast(movie, shift)
    assert rel_l2(out[:, n // 2 - 64 : n // 2 + 64, n // 2 - 64 : n // 2 + 64], g["fast_centre"]) <= SUM_REL
    assert rel_l2(out[:, :64, :64], g["fast_corner"]) <= SUM_REL
    assert rel_l2(out[:, :: n // (8 if n <= 4096 else 4), :], g["fast_rows"]) <= SUM_REL  # 4 rows of 8192^2 frames
    assert abs(float(torch.linalg.norm(out.double())) - float(g["fast_norm"])) <= SUM_REL * float(g["fast_norm"])
