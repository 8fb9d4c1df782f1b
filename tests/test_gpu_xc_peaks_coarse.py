"""The coarse bound of the peak search (rows_coarse_bound_p2 + rows_select_live): where the band fits a quarter-length
row transform, every row is bounded from its samples at x = 4m and the full-length row kernels run only on the row
blocks that can hold the maximum.  The result must be what the full search returns; checked here against the float64
irfft2 reference of test_gpu_xc_peaks at the C2 and config-4 row lengths and bands (1024 / KX 86, 4096 / KX 341,
8192 / KX 341) on surfaces that stress the bound: maxima between coarse samples, coarse samples ranking two peaks the
wrong way round, constant rows and columns (ties), all-zero and NaN products, and bench-like products, where the
bound must also drop most row blocks."""

import numpy as np
import pytest
import torch

from torch_motion_correction_b200 import _fourier, _lib, _ops
from torch_motion_correction_b200.estimate_motion_xc import global_spectra, mean_except_current_spectra, patch_xc_geometry
from test_gpu_xc_peaks import Case, wrap

pytestmark = pytest.mark.gpu

COARSE = "rows_coarse_bound_p2"
# (ny, nx, kx, ky): C2 patches (1024 px, 0.83 A/px, 10 A cut-off), C2 whole frames, config-4 whole frames (rows only:
# the column length does not enter the bound, so a short surface keeps the float64 reference cheap)
SHAPES = [(1024, 1024, 86, 171), (64, 4096, 341, 41), (64, 8192, 341, 41)]


def shape_id(c):
    return f"{c[0]}x{c[1]}-kx{c[2]}"


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def live_blocks(case, prod):
    """(shifts, kernels that ran, live row blocks, all row blocks) of one search."""
    _lib.kernel_timing(True)
    ws = []
    got = case.plan.peaks(prod, sub_pixel=False, workspace_out=ws)
    torch.cuda.synchronize()
    ran = set(_lib.kernel_timing_report())
    _lib.kernel_timing(False)
    count = int(ws[0][:4].view(torch.int32).item()) if ws[0] is not None else None
    total = prod.shape[0] * _lib.query("tmc_xc_peak_partials", case.ny, case.nx)
    return got.cpu().double().numpy(), ran, count, total


def check_against_reference(case, boxes, got):
    """Integer peaks of complex64 boxes (n, KY, KX) against the float64 surfaces."""
    ny, nx = case.ny, case.nx
    for i, box in enumerate(boxes):
        s = case.surface(box.astype(np.complex128))
        bound = case.value_bound(box)
        flat = s.ravel()
        top2 = np.partition(flat, -2)[-2:]
        gy, gx = int(got[i, 0]) % ny, int(got[i, 1]) % nx
        if top2[1] - top2[0] > bound:
            assert (gy, gx) == divmod(int(flat.argmax()), nx), (i, got[i])
        else:
            assert s[gy, gx] >= top2[1] - bound, (i, got[i])


def as_prod(boxes, dev):
    return torch.view_as_real(torch.as_tensor(np.stack(boxes).astype(np.complex64))).to(dev).contiguous()


def ramp_box(case, y0, x0):
    ky = (np.arange(case.plan.ky) + case.plan.ky_start)[:, None]
    kx = np.arange(case.plan.kx)[None, :]
    return np.exp(-2j * np.pi * ((ky * y0 % case.ny) / case.ny + (kx * x0 % case.nx) / case.nx))


@pytest.mark.parametrize("c", SHAPES, ids=shape_id)
def test_maxima_between_coarse_samples(dev, c):
    """Sharp peaks at x = 1, 2, 3 (mod 4) on rows spread over the surface: the coarse samples miss every one of them."""
    case = Case(dev, *c)
    ny, nx = case.ny, case.nx
    ys = np.array([(97 * i + 5) % ny for i in range(12)])
    xs = np.array([4 * ((1009 * i) % (nx // 4)) + 1 + i % 3 for i in range(12)])
    got, ran, _, _ = live_blocks(case, case.ramp(ys, xs))
    assert COARSE in "".join(ran), ran
    assert case.gap > case.bound
    assert np.array_equal(got[:, 0], wrap(ys, ny)) and np.array_equal(got[:, 1], wrap(xs, nx))


@pytest.mark.parametrize("c", SHAPES, ids=shape_id)
def test_coarse_samples_rank_two_peaks_the_wrong_way(dev, c):
    """Peak A between coarse samples (x = 4m + 2) and a slightly lower peak B on a coarse sample, on distant rows: the
    coarse samples rank B first, the full search returns A."""
    case = Case(dev, *c)
    ny, nx = case.ny, case.nx
    s0 = case.s0
    ratio = s0[:, 2::4].max() / s0[0, 0]  # A's best coarse sample (x - xa = 2 mod 4) relative to its peak
    b = 0.5 * (1.0 + ratio)      # B's height: above A's coarse samples, below A
    ya, xa, yb, xb = 3, 4 * (nx // 8) + 2, ny // 2 + 7, 4 * (nx // 16)
    box = case.ps * (ramp_box(case, ya, xa) + b * ramp_box(case, yb, xb))
    s = case.surface(box)
    coarse = s[:, ::4]
    assert divmod(int(coarse.argmax()), coarse.shape[1])[0] == yb  # the coarse samples rank B first
    assert divmod(int(s.argmax()), nx) == (ya, xa)
    got, ran, _, _ = live_blocks(case, as_prod([box], dev))
    assert COARSE in "".join(ran), ran
    assert (int(got[0, 0]) % ny, int(got[0, 1]) % nx) == (ya, xa)
    check_against_reference(case, [box.astype(np.complex64)], got)


@pytest.mark.parametrize("c", SHAPES, ids=shape_id)
def test_constant_rows_and_columns(dev, c):
    """A product only in the kx = 0 column makes every row constant (ties along x: x = 0); one only in the ky = 0 row
    makes every column constant (ties along y: row 0)."""
    case = Case(dev, *c)
    ny, nx = case.ny, case.nx
    rng = np.random.default_rng(11)
    col = np.zeros((case.plan.ky, case.plan.kx), dtype=np.complex128)
    col[:, 0] = rng.standard_normal(case.plan.ky) + 1j * rng.standard_normal(case.plan.ky)
    row = np.zeros_like(col)
    row[-case.plan.ky_start, :] = rng.standard_normal(case.plan.kx) + 1j * rng.standard_normal(case.plan.kx)
    boxes = [col.astype(np.complex64), row.astype(np.complex64)]
    got, ran, _, _ = live_blocks(case, as_prod(boxes, dev))
    assert COARSE in "".join(ran), ran
    assert got[0, 1] == 0 and got[1, 0] == 0, got
    check_against_reference(case, boxes, got)


@pytest.mark.parametrize("c", SHAPES, ids=shape_id)
def test_zero_and_nan_products(dev, c):
    """All-zero products peak at (0, 0); a NaN bin turns the whole surface to NaN, where no sample compares greater and
    the search returns what it returns without the bound (index INT_MAX).  Items beside them are unaffected."""
    case = Case(dev, *c)
    ny, nx = case.ny, case.nx
    prod = torch.cat([torch.zeros((1, case.plan.ky, case.plan.kx, 2), device=dev), case.ramp([5], [4 * 7 + 3])])
    prod = torch.cat([prod, prod[:1].clone()])
    prod[2, 0, 1, 0] = float("nan")
    got, ran, _, _ = live_blocks(case, prod)
    assert COARSE in "".join(ran), ran
    assert np.array_equal(got[0], [0, 0]) and np.array_equal(got[1], [5, 31]), got
    big = 0x7FFFFFFF
    want = np.array([big // nx, big % nx], dtype=np.float32)
    want = np.where(want <= np.array([ny // 2, nx // 2], dtype=np.float32), want, want - np.array([ny, nx], dtype=np.float32))
    assert np.array_equal(got[2], want.astype(np.float64)), got[2]


# ny not a multiple of the coarse CTA (128 / 32 rows), of the fine row block (32 / 8 rows) nor of 2: a short last coarse
# CTA, a partial last fine block and a last row pair without its second row
PARTIAL_SHAPES = [(1001, 1024, 86, 171), (77, 4096, 341, 41)]


@pytest.mark.parametrize("c", PARTIAL_SHAPES, ids=shape_id)
def test_partial_last_blocks(dev, c):
    """Peaks on the last rows (the unpaired last row included), between coarse samples, and on the first rows."""
    case = Case(dev, *c)
    ny, nx = case.ny, case.nx
    ys = np.array([ny - 1, ny - 2, ny - 3, ny - 5, ny - 9, 0, 1, ny // 2])
    xs = np.array([4 * ((613 * i) % (nx // 4)) + i % 4 for i in range(len(ys))])
    got, ran, count, total = live_blocks(case, case.ramp(ys, xs))
    assert COARSE in "".join(ran), ran
    assert 0 < count < total
    assert case.gap > case.bound
    assert np.array_equal(got[:, 0], wrap(ys, ny)) and np.array_equal(got[:, 1], wrap(xs, nx))


def test_wide_band_runs_the_full_search(dev):
    """2 KX - 1 > nx / 4: the half-length kernel searches every row, without a workspace."""
    case = Case(dev, 64, 4096, 600, 41)
    assert _lib.query("tmc_xc_peaks_workspace_bytes", 1, 64, 4096, 600) == 0
    assert _lib.query("tmc_xc_peaks_workspace_bytes", 1, 64, 4096, 341) > 0
    ys, xs = np.array([0, 17, 63, 40]), np.array([1, 2050, 4095, 3])
    got, ran, count, _ = live_blocks(case, case.ramp(ys, xs))
    assert COARSE not in "".join(ran) and "rows_inverse_argmax_real2n<2048>" in ran, ran
    assert count is None
    assert np.array_equal(got[:, 0], wrap(ys, 64)) and np.array_equal(got[:, 1], wrap(xs, 4096))


# ---- bench-like products ---------------------------------------------------------------------------------------------


def bench_like_movie(t, h, w, seed, dev):
    """Band-limited random specimen (unit variance), integer drift, unit Gaussian noise: bench.py's synthetic movie."""
    g = torch.Generator(device=dev).manual_seed(seed)
    spec = torch.fft.rfftn(torch.randn((h + 32, w + 32), generator=g, device=dev))
    fy = torch.fft.fftfreq(h + 32, device=dev)[:, None]
    fx = torch.fft.rfftfreq(w + 32, device=dev)[None, :]
    specimen = torch.fft.irfftn(spec * torch.exp(-(fy**2 + fx**2) / (2 * 0.08**2)), s=(h + 32, w + 32))
    specimen = specimen / specimen.std()
    walk = np.round(np.cumsum(np.random.default_rng(seed).standard_normal((t, 2)), axis=0) * 2).astype(int)
    walk = np.clip(walk - walk[t // 2], -12, 12)
    movie = torch.empty((t, h, w), device=dev)
    for k in range(t):
        sy, sx = walk[k]
        movie[k] = specimen[16 - sy : 16 - sy + h, 16 - sx : 16 - sx + w] + torch.randn((h, w), generator=g, device=dev)
    return movie


def reference_case(plan, dev):
    """A Case whose reference helpers (surface, value_bound) serve ``plan``'s geometry."""
    case = Case.__new__(Case)
    case.ny, case.nx, case.dev, case.plan = plan.ny, plan.nx, dev, plan
    case.kyi = (np.arange(plan.ky) + plan.ky_start) % plan.ny
    return case


def check_bench_like(dev, plan, prod):
    case = reference_case(plan, dev)
    got, ran, count, total = live_blocks(case, prod)
    assert COARSE in "".join(ran), ran
    print(f"[coarse] {plan.ny}x{plan.nx} kx={plan.kx}: {count} of {total} row blocks live ({100 * count / total:.2f} %)")
    assert 0 < count < 0.1 * total
    boxes = torch.view_as_complex(prod.cpu()).numpy()
    check_against_reference(case, boxes, got)


def test_bench_like_patch_products(dev):
    """Leave-one-out and middle-frame patch products of a bench-like movie at C2's patch size, pixel size and band."""
    movie = bench_like_movie(8, 2048, 2048, 4040, dev)
    stats = _ops.stack_stats(movie)
    _, origins, plan, mask, _ = patch_xc_geometry(movie.shape, 1024, 0.83, 500, (300, 10), None, dev)
    assert (plan.nx, plan.kx) == (1024, 85)
    t, g = movie.shape[0], len(origins)
    jobs, spec = mean_except_current_spectra(movie, stats, plan, mask, 1024, origins, None)
    offsets = torch.tensor([0] * (t + 1), dtype=torch.int32, device=dev)
    deltas = torch.zeros((1,), dtype=torch.int32, device=dev)
    loo = _fourier.leave_one_out_products(spec, t, g, plan.plane_elems, offsets, deltas)
    check_bench_like(dev, plan, loo.view(t * g, plan.ky, plan.kx, 2))
    items = torch.arange(t * g, dtype=torch.int32, device=dev)
    ref = (2 * ((t // 2) * g + items % g)).to(torch.int32)
    pair = _fourier.pair_products(spec, ref, 2 * items, plan.plane_elems)
    check_bench_like(dev, plan, pair.view(t * g, plan.ky, plan.kx, 2))


def test_bench_like_whole_frame_products(dev):
    """Whole-frame products against the middle frame of a bench-like 4096^2 movie at C2's pixel size and band."""
    movie = bench_like_movie(6, 4096, 4096, 4041, dev)
    stats = _ops.stack_stats(movie)
    plan, spec = global_spectra(movie, stats, 0.83, 500, (300, 10))
    assert (plan.nx, plan.kx) == (4096, 340)
    t = movie.shape[0]
    cur = torch.arange(t, dtype=torch.int32, device=dev)
    ref = torch.full((t,), t // 2, dtype=torch.int32, device=dev)
    prod = _fourier.pair_products(spec, ref, cur, plan.plane_elems)
    check_bench_like(dev, plan, prod.view(t, plan.ky, plan.kx, 2))
