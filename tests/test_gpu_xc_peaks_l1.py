"""The L1 tier of the peak search (rows_l1_bound + rows_l1_seeds): every row is bounded by the L1 norm of its
coefficients, the coarse bound runs on each surface's seed group (the group of its row with the largest norm) alone, and
a row block stays live only if its norm bound reaches the seed's best lower bound.  The result must be what the full
search returns; checked against the float64 reference of test_gpu_xc_peaks_coarse on surfaces where the seed is not the
peak's group, peaks in the last partial group, surfaces pruned to the seed and surfaces with every block live (ties),
non-finite and oversized norms, bench-like products, and calls split over more than 65535 items."""

import numpy as np
import pytest
import torch

from torch_motion_correction_b200 import _fourier, _lib, _ops
from torch_motion_correction_b200.estimate_motion_xc import global_spectra, mean_except_current_spectra, patch_xc_geometry
from test_gpu_xc_peaks import Case, wrap
from test_gpu_xc_peaks_coarse import (COARSE, SHAPES, as_prod, bench_like_movie, check_against_reference, ramp_box,
                                      reference_case, shape_id)

pytestmark = pytest.mark.gpu

# rows of a coarse group (the row block of rows_coarse_bound_p2<nx / 4>) and of a fine row block (polyphase 1024-point,
# half-length 4096- and 8192-point kernels)
GROUP_ROWS = {1024: 128, 4096: 32, 8192: 16}
FINE_ROWS = {1024: 32, 4096: 8, 8192: 4}


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def search(case, prod):
    """(shifts, live row blocks, all row blocks) of one call."""
    _lib.kernel_timing(True)
    ws = []
    got = case.plan.peaks(prod, sub_pixel=False, workspace_out=ws)
    torch.cuda.synchronize()
    ran = set(_lib.kernel_timing_report())
    _lib.kernel_timing(False)
    assert COARSE in "".join(ran) and "rows_l1_bound" in ran, ran
    fine, seeds = ws[0][:8].view(torch.int32).tolist()
    n = prod.shape[0]
    assert seeds == n
    return got.cpu().double().numpy(), fine, n * _lib.query("tmc_xc_peak_partials", case.ny, case.nx)


def column_rows(case, box):
    """float64 rows c_k(y) after the column pass of a (KY, KX) box."""
    full = np.zeros((case.ny, case.plan.kx), dtype=np.complex128)
    full[case.kyi] = box
    return np.fft.ifft(full, axis=0) * case.ny


def row_l1(case, box):
    c = column_rows(case, box)
    return np.abs(c[:, 0].real) + 2 * np.abs(c[:, 1:]).sum(1)


def decoy_box(case, y, scale, seed=0):
    """A row y of random-phase coefficients: its L1 norm is scale, its largest value about a third of that (KX ~ 86)."""
    rng = np.random.default_rng(seed)
    u = np.exp(2j * np.pi * rng.random(case.plan.kx))
    u[0] = 1.0
    ky = (np.arange(case.plan.ky) + case.plan.ky_start)[:, None]
    box = np.exp(-2j * np.pi * (ky * y % case.ny) / case.ny) * u[None, :] / case.ny
    return box * scale / row_l1(case, box).max()


@pytest.mark.parametrize("c", SHAPES, ids=shape_id)
def test_seed_is_not_the_peak_group(dev, c):
    """The row with the largest L1 norm is a random-phase decoy far from the peak: the seed's coarse samples are lower
    than the peak's, the peak's group must stay live and the search returns the peak."""
    case = Case(dev, *c)
    ny, nx = case.ny, case.nx
    rows = GROUP_ROWS[nx]
    ya, xa = 3, 4 * (nx // 8) + 1
    yb = ya + ny // 2
    peak = case.ps * ramp_box(case, ya, xa)
    box = peak + decoy_box(case, yb, 1.3 * row_l1(case, peak).max())
    l1 = row_l1(case, box)
    s = case.surface(box)
    assert int(l1.argmax()) // rows != ya // rows  # the seed is another group
    assert divmod(int(s.argmax()), nx) == (ya, xa)
    got, fine, fine_total = search(case, as_prod([box], dev))
    assert (int(got[0, 0]) % ny, int(got[0, 1]) % nx) == (ya, xa)
    assert fine < fine_total
    check_against_reference(case, [box.astype(np.complex64)], got)


# ny not a multiple of the coarse group (128 / 32 rows): a short last group
PARTIAL_SHAPES = [(1001, 1024, 86, 171), (77, 4096, 341, 41)]


@pytest.mark.parametrize("c", PARTIAL_SHAPES, ids=shape_id)
def test_peak_in_the_last_partial_group(dev, c):
    """Peaks on the last rows (the unpaired last row included) with the largest-norm row in the middle of the surface."""
    case = Case(dev, *c)
    ny, nx = case.ny, case.nx
    boxes = []
    for i, y in enumerate([ny - 1, ny - 2, ny - 3]):
        peak = case.ps * ramp_box(case, y, 4 * (37 * i + 5) + 2)
        boxes.append(peak + decoy_box(case, ny // 2, 1.3 * row_l1(case, peak).max(), seed=i))
        assert int(row_l1(case, boxes[-1]).argmax()) // GROUP_ROWS[nx] != y // GROUP_ROWS[nx]
    got, fine, fine_total = search(case, as_prod(boxes, dev))
    assert fine < fine_total
    check_against_reference(case, [b.astype(np.complex64) for b in boxes], got)
    assert np.array_equal(got[:, 0], wrap(np.array([ny - 1, ny - 2, ny - 3]), ny))


@pytest.mark.parametrize("c", SHAPES, ids=shape_id)
def test_pruned_to_the_seed_beside_all_live(dev, c):
    """Two surfaces in one call: a single peak in the middle of a group, where the tier drops every group but the seed
    (the other groups' finite hi and lo must leave the surface finite: only blocks of the seed group stay live), and a
    product only in the ky = 0 row, whose rows are all equal (ties: every block stays live, the peak is on row 0)."""
    case = Case(dev, *c)
    ny, nx = case.ny, case.nx
    rows = GROUP_ROWS[nx]
    ya, xa = min(ny - 1, rows + rows // 2), 4 * (nx // 16) + 3
    peak = case.ps * ramp_box(case, ya, xa)
    l1 = row_l1(case, peak)
    outside = np.delete(l1, np.arange(ya // rows * rows, min(ny, ya // rows * rows + rows)))
    assert outside.max() < 0.9 * case.surface(peak).max()  # every other group is below the seed's samples
    rng = np.random.default_rng(5)
    flat = np.zeros((case.plan.ky, case.plan.kx), dtype=np.complex128)
    flat[-case.plan.ky_start, :] = rng.standard_normal(case.plan.kx) + 1j * rng.standard_normal(case.plan.kx)
    boxes = [peak.astype(np.complex64), flat.astype(np.complex64)]
    got, fine, fine_total = search(case, as_prod(boxes, dev))
    per_item = fine_total // 2
    assert per_item < fine <= per_item + rows // FINE_ROWS[nx]  # every block of the flat surface, the seed's of the peak
    assert (int(got[0, 0]) % ny, int(got[0, 1]) % nx) == (ya, xa)
    assert got[1, 0] == 0, got
    check_against_reference(case, boxes, got)


@pytest.mark.parametrize("c", SHAPES, ids=shape_id)
def test_non_finite_and_oversized_norms_keep_every_group(dev, c):
    """A NaN bin reaches every row through the column pass: every group and block stays live and the search returns
    what the full search returns (index INT_MAX).  A surface pruned to its seed when small, scaled so that its largest
    row norm passes 1e36: every group stays live and the peak is found."""
    case = Case(dev, *c)
    ny, nx = case.ny, case.nx
    rows = GROUP_ROWS[nx]
    ya, xa = min(ny - 1, rows + rows // 2), 4 * (nx // 16) + 3
    peak = case.ps * ramp_box(case, ya, xa)
    nan = peak.astype(np.complex64)
    nan[0, 1] = np.nan
    big = (peak * (4e36 / row_l1(case, peak).max())).astype(np.complex64)
    small = peak.astype(np.complex64)
    got, fine, fine_total = search(case, as_prod([nan, big, small], dev))
    per_item = fine_total // 3
    assert 2 * per_item < fine <= 2 * per_item + rows // FINE_ROWS[nx]  # all of the first two, the seed's of the third
    big_idx = 0x7FFFFFFF
    want = np.array([big_idx // nx, big_idx % nx], dtype=np.float32)
    want = np.where(want <= np.array([ny // 2, nx // 2], dtype=np.float32), want, want - np.array([ny, nx], dtype=np.float32))
    assert np.array_equal(got[0], want.astype(np.float64)), got[0]
    for i in (1, 2):
        assert (int(got[i, 0]) % ny, int(got[i, 1]) % nx) == (ya, xa), got[i]


# ---- bench-like products ---------------------------------------------------------------------------------------------


def check_bench_like(dev, plan, prod, most):
    case = reference_case(plan, dev)
    got, fine, fine_total = search(case, prod)
    print(f"[l1] {plan.ny}x{plan.nx} kx={plan.kx}: {fine} of {fine_total} row blocks live ({100 * fine / fine_total:.2f} %)")
    assert 0 < fine <= most * fine_total
    boxes = torch.view_as_complex(prod.cpu()).numpy()
    check_against_reference(case, boxes, got)


def test_bench_like_patch_products(dev):
    """Leave-one-out patch products of a bench-like movie at C2's patch size, pixel size and band."""
    movie = bench_like_movie(8, 2048, 2048, 4040, dev)
    stats = _ops.stack_stats(movie)
    _, origins, plan, mask, _ = patch_xc_geometry(movie.shape, 1024, 0.83, 500, (300, 10), None, dev)
    t, g = movie.shape[0], len(origins)
    _, spec = mean_except_current_spectra(movie, stats, plan, mask, 1024, origins, None)
    offsets = torch.tensor([0] * (t + 1), dtype=torch.int32, device=dev)
    deltas = torch.zeros((1,), dtype=torch.int32, device=dev)
    loo = _fourier.leave_one_out_products(spec, t, g, plan.plane_elems, offsets, deltas)
    check_bench_like(dev, plan, loo.view(t * g, plan.ky, plan.kx, 2), 0.08)


def test_bench_like_whole_frame_products(dev):
    """Whole-frame products against the middle frame of a bench-like 4096^2 movie at C2's pixel size and band."""
    movie = bench_like_movie(6, 4096, 4096, 4041, dev)
    stats = _ops.stack_stats(movie)
    plan, spec = global_spectra(movie, stats, 0.83, 500, (300, 10))
    t = movie.shape[0]
    cur = torch.arange(t, dtype=torch.int32, device=dev)
    ref = torch.full((t,), t // 2, dtype=torch.int32, device=dev)
    prod = _fourier.pair_products(spec, ref, cur, plan.plane_elems)
    check_bench_like(dev, plan, prod.view(t, plan.ky, plan.kx, 2), 0.01)


# ---- repeat calls and calls over more than 65535 items ---------------------------------------------------------------


def test_repeat_and_split_calls_are_bitwise_equal(dev):
    """70000 items of 64 x 4096 surfaces (two coarse groups each) in one call, which the search splits at 65535 items,
    bitwise equal to three calls under the limit and to a repeat of the call."""
    case = Case(dev, 64, 4096, 16, 41)
    g = torch.Generator(device=dev).manual_seed(9)
    n = 70000
    ys = torch.randint(0, 64, (16,), generator=g, device=dev).cpu().numpy()
    xs = torch.randint(0, 4096, (16,), generator=g, device=dev).cpu().numpy()
    base = case.ramp(ys, xs).repeat(n // 16 + 1, 1, 1, 1)[:n]
    prod = base + 0.01 * float(case.ps.max()) * torch.randn(base.shape, generator=g, device=dev)
    whole = case.plan.peaks(prod, sub_pixel=True).clone()
    again = case.plan.peaks(prod, sub_pixel=True)
    torch.cuda.synchronize()
    bounds = np.linspace(0, n, 4).astype(int)
    split = torch.cat([case.plan.peaks(prod[a:b].contiguous(), sub_pixel=True) for a, b in zip(bounds[:-1], bounds[1:])])
    assert torch.equal(whole, again)
    assert torch.equal(whole, split)
