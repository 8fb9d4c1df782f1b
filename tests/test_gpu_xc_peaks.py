"""The cross-correlation peak search (tmc_xc_peaks: inverse transform of a band-limited product, argmax, 3-point
parabola, wrap) against a float64 reference, kernel by kernel.

Reference: the band box of a product is zero-padded to (ny, nx/2+1) and inverted with numpy's float64 irfft2, which
keeps only the real part of the self-paired DC / Nyquist columns as the kernels do.  The kernels get the same box
rounded to complex64; the reference starts from that rounded box.  Integer peaks are placed by an exact phase ramp on
a non-negative spectrum (|FA|^2 times a Gaussian weight): its surface is the autocorrelation S0 rolled to the peak,
so one irfft2 per shape serves every item.

Error bound on one sample of the unnormalised fp32 surface (``value_bound``): every sample is a sum of terms of
magnitude <= 2 |P_k|, and each butterfly stage of the row and column transforms (Bluestein: three transforms of
M >= 2n - 1 points; decimated axes: R twiddled sub-transforms summed) rounds partial sums bounded by sum 2 |P_k|
with a relative error of a few eps32.  Where the float64 maximum beats the runner-up by more than the bound, the
index must be exact; otherwise the chosen sample must lie within the bound of the maximum.

Sub-pixel: the kernel's refined shift is compared with the float64 parabola at the kernel's integer peak, modulo the
axis length.  Worst error measured on a B200 (1000 W), over both the sweeps and the fractional shifts with noise;
``SUBPX_BOUND`` (1e-3 px) is about 3x the largest and 10x below the 0.01 px target:
  rows_inverse_argmax_kernel (generic, Bluestein, decimated) ........ 3.0e-4 px (9000 x 16, 64 x 12288)
  rows_inverse_argmax_p2 / p2<1024> / p2<4096> ....................... 1.3e-4 / 2.6e-5 / 1.1e-4 px
  rows_inverse_argmax_poly ........................................... 1.6e-5 px
  rows_inverse_argmax_real2n<2048> / <4096> .......................... 1.1e-4 / 9.2e-6 px
The fractional cases are the larger ones; on the integer sweeps the symmetric surfaces leave at most 2e-6 px.
"""

import math

import numpy as np
import pytest
import torch

import torch_motion_correction_b200 as tmc
from torch_motion_correction_b200 import _fourier, _lib
from oracle import reference_path as rp

pytestmark = pytest.mark.gpu

EPS32 = float(np.finfo(np.float32).eps)
SUBPX_BOUND = 1e-3  # px: ~3x the worst measured, 10x below the 0.01 px north star

GEN, POLY = "rows_inverse_argmax_kernel", "rows_inverse_argmax_poly"
P2, P2_1024, P2_4096 = "rows_inverse_argmax_p2", "rows_inverse_argmax_p2<1024>", "rows_inverse_argmax_p2<4096>"
R2N_2048, R2N_4096 = "rows_inverse_argmax_real2n<2048>", "rows_inverse_argmax_real2n<4096>"


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def _pow2(n):
    """A power of two the shared-memory transforms take whole (16384 = 4 x 4096 is decimated)."""
    return 16 <= n <= 8192 and n & (n - 1) == 0


def row_kernel(nx, kx, real2n=True):
    """Name of the row kernel tmc_xc_peaks runs for rows of nx points with kx_count = kx."""
    if _pow2(nx) and nx >= 256:
        if nx in (4096, 8192) and kx <= nx // 4 and real2n:
            return f"rows_inverse_argmax_real2n<{nx // 2}>"
        if nx == 1024 and kx <= 128:
            return POLY
        return {1024: P2_1024, 4096: P2_4096}.get(nx, P2)
    return GEN


def col_kernel(ny):
    if _pow2(ny) and ny >= 256:
        return {1024: "cols_inverse_p2<1024>", 4096: "cols_inverse_p2<4096>"}.get(ny, "cols_inverse_p2")
    return "cols_inverse_kernel"


# (ny, nx, kx_count, ky_count or None for every row); a full box is (ny, nx, nx // 2 + 1, None)
ROW_CASES = [
    (32, 16, 5, 13), (32, 64, 20, 17), (48, 128, 40, 25),  # generic power of two
    (32, 256, 60, 21), (32, 512, 100, 21), (16, 2048, 300, 13),  # p2
    (64, 1024, 100, 41), (64, 1024, 300, 41),  # polyphase, p2<1024>
    (32, 4096, 1000, 21), (16, 8192, 2000, 13), (32, 4096, 1500, 21), (16, 8192, 3000, 13),  # real2n, p2
    (32, 96, 30, 21), (33, 97, 30, 21), (16, 927, 200, 13), (16, 4092, 800, 13),  # Bluestein
    (16, 5000, 800, 13), (16, 9000, 1500, 13),  # decimated Bluestein: 2 x 2500, 3 x 3000
    (64, 12288, 1500, 41), (64, 16384, 2000, 41),  # decimated onto 4096-point transforms: 3 x, 4 x
]
COL_CASES = [
    (64, 16, 5, 41), (97, 16, 5, 61), (128, 16, 5, 61), (256, 16, 5, 101), (927, 16, 5, 301), (1024, 16, 5, 301),
    (2048, 16, 5, 401), (4092, 16, 5, 801), (4096, 16, 5, 801), (5000, 16, 5, 801), (5760, 96, 30, 601),
    (8192, 16, 5, 1001), (9000, 16, 5, 1201), (12288, 32, 10, 1201), (16384, 64, 20, 2001),
]
FULL_LENGTHS = [16, 64, 96, 97, 128, 256, 512, 927, 1024, 2048, 4092, 4096, 5000, 5760, 8192, 9000, 12288, 16384]
FULL_CASES = [(16, n, n // 2 + 1, None) for n in FULL_LENGTHS] + [(n, 16, 9, None) for n in FULL_LENGTHS if n > 16]


def case_id(c):
    ny, nx, kx, ky = c
    return f"{ny}x{nx}-kx{kx}-" + ("full" if ky is None else f"ky{ky}")


class Case:
    """A band box of one transform size, a non-negative spectrum on it and the float64 autocorrelation surface."""

    def __init__(self, dev, ny, nx, kx, ky, seed=0):
        assert _fourier.unsupported_lengths(ny, nx, True) is None
        self.ny, self.nx, self.dev = ny, nx, dev
        plan = _fourier.BandPlan(ny, nx, dev, full=True)
        plan.kx = kx
        plan.ky, plan.ky_start = (ny, -(ny // 2)) if ky is None else (ky, -(ky // 2))
        self.plan = plan
        self.kyi = (np.arange(plan.ky) + plan.ky_start) % ny  # box row -> spectrum row
        rng = np.random.default_rng(seed + 7 * ny + nx)
        self.fa = np.fft.rfft2(rng.standard_normal((ny, nx)))[self.kyi][:, :kx]
        fy = (np.arange(plan.ky) + plan.ky_start) / (plan.ky / 2 + 1)
        fx = np.arange(kx) / (kx + 1)
        self.weight = np.exp(-(fy[:, None] ** 2 + fx[None, :] ** 2))
        ps = (np.abs(self.fa) ** 2 * self.weight).astype(np.complex64).real.astype(np.float64)
        self.ps = ps  # exactly representable in complex64
        self.s0 = self.surface(ps)
        top2 = np.partition(self.s0.ravel(), -2)[-2:]
        self.gap = float(top2[1] - top2[0])
        assert self.s0[0, 0] == self.s0.max()
        self.bound = self.value_bound(ps)

    def value_bound(self, box):
        l1 = 2.0 * float(np.abs(box).sum())
        return 16.0 * EPS32 * (math.log2(self.ny) + math.log2(self.nx) + 8.0) * l1

    def surface(self, box):
        """Unnormalised float64 inverse of the zero-padded box."""
        full = np.zeros((self.ny, self.nx // 2 + 1), dtype=np.complex128)
        full[self.kyi, : self.plan.kx] = box
        return np.fft.irfft2(full, s=(self.ny, self.nx)) * (self.ny * self.nx)

    def ramp(self, y0, x0):
        """(n, KY, KX) complex64 products ps * exp(-2 pi i (ky y0 / ny + kx x0 / nx)): surfaces S0 rolled to (y0, x0)."""
        ky = torch.as_tensor((np.arange(self.plan.ky) + self.plan.ky_start), dtype=torch.int64, device=self.dev)
        kx = torch.arange(self.plan.kx, dtype=torch.int64, device=self.dev)
        ps = torch.as_tensor(self.ps, device=self.dev)
        out = torch.empty((len(y0), self.plan.ky, self.plan.kx, 2), dtype=torch.float32, device=self.dev)
        yy = torch.as_tensor(y0, dtype=torch.int64, device=self.dev)
        xx = torch.as_tensor(x0, dtype=torch.int64, device=self.dev)
        for i0 in range(0, len(y0), 64):
            ay = ((ky[None, :] * yy[i0 : i0 + 64, None]) % self.ny).double() / self.ny
            ax = ((kx[None, :] * xx[i0 : i0 + 64, None]) % self.nx).double() / self.nx
            ang = -2.0 * math.pi * (ay[:, :, None] + ax[:, None, :])
            out[i0 : i0 + 64] = torch.view_as_real(torch.polar(ps.expand_as(ang), ang)).float()
        return out

    def peaks(self, prod, sub_pixel):
        _lib.kernel_timing(True)
        got = self.plan.peaks(prod, sub_pixel=sub_pixel)
        torch.cuda.synchronize()
        ran = set(_lib.kernel_timing_report())
        _lib.kernel_timing(False)
        return got.cpu().double().numpy(), ran


def wrap(v, n):
    return np.where(v <= n // 2, v, v - n)


def parabola(value, y, x, ny, nx):
    """estimate_motion_xc.py's 3-point refinement (oracle.reference_path.sub_pixel_refinement) in float64, then the
    wrap; ``value(yy, xx)`` reads the float64 surface."""
    py, px = float(y), float(x)
    if 1 <= y < ny - 1 and 1 <= x < nx - 1:
        a, b, c = value(y - 1, x), value(y, x), value(y + 1, x)
        if c != a:
            py += 0.5 * (a - c) / (a - 2 * b + c)
        a, b, c = value(y, x - 1), value(y, x), value(y, x + 1)
        if c != a:
            px += 0.5 * (a - c) / (a - 2 * b + c)
    return float(wrap(np.float64(py), ny)), float(wrap(np.float64(px), nx))


def circular_err(got, want, n):
    return abs((got - want + n / 2) % n - n / 2)


def sweep_positions(ny, nx):
    """Peak positions covering every row (or every 16th row: each CTA of every row kernel owns >= 32 rows of such
    tall surfaces) and spread over the columns, plus the wrap and border positions."""
    step = 1 if ny <= 64 else 16
    ys = list(range(0, ny, step))
    xs = [(7919 * i + 3) % nx for i in range(len(ys))]
    edges = [(0, 0), (0, nx - 1), (ny - 1, 0), (ny - 1, nx - 1), (ny // 2, nx // 2), (ny // 2 + 1, nx // 2 + 1),
             (1, nx // 2), (ny // 2, 1), (ny - 2, nx - 2)]
    for y, x in edges:
        ys.append(y % ny)
        xs.append(x % nx)
    return np.array(ys), np.array(xs)


def check_sweep(case, real2n=True, monkeypatch=None):
    ny, nx = case.ny, case.nx
    ys, xs = sweep_positions(ny, nx)
    prod = case.ramp(ys, xs)
    got, ran = case.peaks(prod, sub_pixel=False)
    assert row_kernel(nx, case.plan.kx, real2n) in ran, ran
    assert col_kernel(ny) in ran, ran
    # integer peak: the surface of item i is S0 rolled to (ys[i], xs[i])
    gy, gx = got[:, 0].astype(np.int64) % ny, got[:, 1].astype(np.int64) % nx
    assert np.array_equal(got, np.rint(got)), "integer search returned a fraction"
    dy, dx = (gy - ys) % ny, (gx - xs) % nx
    if case.gap > case.bound:
        bad = np.nonzero((dy != 0) | (dx != 0))[0]
        assert len(bad) == 0, f"{len(bad)} of {len(ys)} peaks missed, e.g. item {bad[:5]}: want {ys[bad[:5]]},{xs[bad[:5]]} got {got[bad[:5]]}"
        assert np.array_equal(got[:, 0], wrap(ys, ny)) and np.array_equal(got[:, 1], wrap(xs, nx))
    else:
        assert (case.s0[dy, dx] >= case.s0.max() - case.bound).all()
    # sub-pixel at the same integer peaks
    sub, _ = case.peaks(prod, sub_pixel=True)
    worst = 0.0
    for i in range(len(ys)):
        value = lambda yy, xx, i=i: case.s0[(yy - ys[i]) % ny, (xx - xs[i]) % nx]
        wy, wx = parabola(value, int(gy[i]), int(gx[i]), ny, nx)
        worst = max(worst, circular_err(sub[i, 0], wy, ny), circular_err(sub[i, 1], wx, nx))
        if not (1 <= gy[i] < ny - 1 and 1 <= gx[i] < nx - 1):  # border: no refinement, same value as without
            assert sub[i, 0] == got[i, 0] and sub[i, 1] == got[i, 1]
    print(f"[subpx] {row_kernel(nx, case.plan.kx, real2n)} {ny}x{nx} kx={case.plan.kx}: sweep {worst:.2e} px")
    assert worst <= SUBPX_BOUND, worst
    return got


@pytest.mark.parametrize("c", ROW_CASES + COL_CASES + FULL_CASES, ids=case_id)
def test_peak_sweep_every_row_block(dev, c):
    """One batch of items whose peaks sweep the rows and columns, so every CTA's share of the surface holds a peak in
    some item; the wrap (<= n // 2) and border (no refinement) positions; exact against the float64 surface."""
    check_sweep(Case(dev, *c))


@pytest.mark.parametrize("c", [(32, 4096, 1000, 21), (16, 8192, 2000, 13)], ids=case_id)
def test_peak_sweep_without_half_length_rows(dev, c, monkeypatch):
    """TMC_FFT_REAL2N=0 (read per call) takes the full-length p2 row kernels where real2n would run."""
    monkeypatch.setenv("TMC_FFT_REAL2N", "0")
    check_sweep(Case(dev, *c), real2n=False)


FRACTIONAL_CASES = [c for c in ROW_CASES + COL_CASES if c[0] * c[1] <= 1 << 20]


@pytest.mark.parametrize("c", FRACTIONAL_CASES, ids=case_id)
def test_fractional_shifts_with_noise(dev, c):
    """B = A Fourier-shifted by a fractional amount plus noise: the product conj(FA) (FA e^{-i theta} + FN) W.  Integer
    peak and parabola against numpy's float64 irfft2 of each item."""
    case = Case(dev, *c)
    ny, nx = case.ny, case.nx
    rng = np.random.default_rng(ny * 31 + nx)
    n = 6
    shifts = np.stack([rng.uniform(-ny / 4, ny / 4, n), rng.uniform(-nx / 4, nx / 4, n)], axis=1)
    shifts[0] = (0.5 + 0.25, -0.3)  # near the origin
    fy = (np.arange(case.plan.ky) + case.plan.ky_start) / ny
    fx = np.arange(case.plan.kx) / nx
    boxes = []
    for sy, sx in shifts:
        fn = np.fft.rfft2(0.3 * rng.standard_normal((ny, nx)))[case.kyi][:, : case.plan.kx]
        fb = case.fa * np.exp(-2j * np.pi * (fy[:, None] * sy + fx[None, :] * sx)) + fn
        boxes.append((np.conj(case.fa) * fb * case.weight).astype(np.complex64))
    prod = torch.view_as_real(torch.as_tensor(np.stack(boxes))).to(dev).contiguous()
    got, ran = case.peaks(prod, sub_pixel=False)
    sub, _ = case.peaks(prod, sub_pixel=True)
    assert row_kernel(nx, case.plan.kx) in ran and col_kernel(ny) in ran, ran
    worst = 0.0
    for i, box in enumerate(boxes):
        s = case.surface(box.astype(np.complex128))
        bound = case.value_bound(box)
        flat = s.ravel()
        top2 = np.partition(flat, -2)[-2:]
        gy, gx = int(got[i, 0]) % ny, int(got[i, 1]) % nx
        if top2[1] - top2[0] > bound:
            wy, wx = divmod(int(flat.argmax()), nx)
            assert (gy, gx) == (wy, wx), (i, shifts[i], got[i], (wy, wx))
        else:
            assert s[gy, gx] >= top2[1] - bound
        wy, wx = parabola(lambda yy, xx: s[yy, xx], gy, gx, ny, nx)
        worst = max(worst, circular_err(sub[i, 0], wy, ny), circular_err(sub[i, 1], wx, nx))
        # the estimate lands on the applied shift (noise and the band limit move it by far less than a pixel)
        assert circular_err(sub[i, 0], shifts[i, 0], ny) < 0.5 and circular_err(sub[i, 1], shifts[i, 1], nx) < 0.5
    print(f"[subpx] {row_kernel(nx, case.plan.kx)} {ny}x{nx} kx={case.plan.kx}: fractional {worst:.2e} px")
    assert worst <= SUBPX_BOUND, worst


@pytest.mark.parametrize("c", [(32, 16, 5, 13), (64, 1024, 100, 41), (32, 4096, 1000, 21), (33, 97, 30, 21),
                               (64, 16384, 2000, 41), (16, 5000, 2501, None), (5760, 96, 30, 601)], ids=case_id)
def test_degenerate_products(dev, c):
    """An all-zero product gives (0, 0) with and without refinement (argmax of a constant surface is sample 0, a border
    sample), as the reference does; a real image against itself peaks at the origin."""
    case = Case(dev, *c)
    zero = torch.zeros((3, case.plan.ky, case.plan.kx, 2), dtype=torch.float32, device=dev)
    for sub_pixel in (False, True):
        got, _ = case.peaks(zero, sub_pixel)
        assert np.array_equal(got, np.zeros((3, 2))), got
        got, _ = case.peaks(case.ramp([0], [0]), sub_pixel)
        assert np.array_equal(got, np.zeros((1, 2))), got


def test_chunked_peaks_are_bitwise_equal(dev, monkeypatch):
    """Items split over several launches (a small CHUNK_BYTES) give bitwise the same shifts as one launch."""
    case = Case(dev, 64, 16384, 2000, 41)
    ys, xs = sweep_positions(64, 16384)
    prod = case.ramp(ys, xs)
    one = case.plan.peaks(prod, sub_pixel=True).clone()
    monkeypatch.setattr(_fourier, "CHUNK_BYTES", 3 * case.ny * case.plan.kx * 8)
    split = case.plan.peaks(prod, sub_pixel=True)
    assert torch.equal(one, split)


def test_cases_cover_every_row_kernel():
    names = {row_kernel(nx, kx) for _, nx, kx, _ in ROW_CASES + FULL_CASES} | {row_kernel(4096, 1000, False)}
    assert names == {GEN, POLY, P2, P2_1024, P2_4096, R2N_2048, R2N_4096}


# ---- launches with more than 65535 jobs / items on the grid's y axis ---------------------------------------------------


def _split(fn, n, parts):
    bounds = np.linspace(0, n, parts + 1).astype(int)
    return torch.cat([fn(int(a), int(b)) for a, b in zip(bounds[:-1], bounds[1:])])


def test_forward_more_than_32768_jobs(dev):
    """2 njobs > 65535 column planes in one tmc_rfft2_band call, bitwise equal to calls under the limit."""
    g = torch.Generator().manual_seed(3)
    img = torch.randn((4, 48, 48), generator=g).to(dev)
    plan = _fourier.BandPlan(32, 32, dev, 1.0, 500.0, (60, 4))
    mask, ylo, yhi = _fourier.soft_disc_mask((32, 32), 8.0, 4.0, dev)
    njobs = 33000
    fa = torch.randint(0, 4, (njobs,), generator=g)
    jobs = torch.stack([fa, torch.ones_like(fa), (fa + 1) % 4, torch.ones_like(fa), torch.randint(0, 17, (njobs,), generator=g),
                        torch.randint(0, 17, (njobs,), generator=g)], dim=1).to(torch.int32).to(dev)
    whole = plan.forward(img, None, mask, ylo, yhi, jobs, job_mode=2)
    torch.cuda.synchronize()
    split = _split(lambda a, b: plan.forward(img, None, mask, ylo, yhi, jobs[a:b].contiguous(), job_mode=2), njobs, 3)
    assert torch.equal(whole, split)


def test_peaks_more_than_65535_items(dev):
    g = torch.Generator().manual_seed(4)
    plan = _fourier.BandPlan(32, 32, dev, 1.0, 500.0, (60, 4))
    n = 70000
    prod = torch.randn((n, plan.ky, plan.kx, 2), generator=g).to(dev)
    whole = plan.peaks(prod, sub_pixel=True)
    torch.cuda.synchronize()
    split = _split(lambda a, b: plan.peaks(prod[a:b].contiguous(), sub_pixel=True), n, 3)
    assert torch.equal(whole, split)


def test_pair_products_more_than_65535_items(dev):
    g = torch.Generator().manual_seed(5)
    planes, elems, n = 100, 64 * 33, 70000
    spec = torch.randn((planes, elems, 2), generator=g).to(dev)
    ref = torch.randint(0, planes, (n,), generator=g, dtype=torch.int32).to(dev)
    cur = torch.randint(0, planes, (n,), generator=g, dtype=torch.int32).to(dev)
    whole = _fourier.pair_products(spec, ref, cur, elems)
    torch.cuda.synchronize()
    split = _split(lambda a, b: _fourier.pair_products(spec, ref[a:b].contiguous(), cur[a:b].contiguous(), elems), n, 3)
    assert torch.equal(whole, split)


@pytest.fixture(scope="module")
def movie_40x1024():
    movie, _ = rp.synthetic_movie(40, 1024, 1024, seed=9, noise=1.0, drift=3.0, sigma_f=0.08)
    return movie


@pytest.mark.parametrize("strategy", ["mean_except_current", "middle_frame"])
def test_small_patches_of_a_long_movie(dev, movie_40x1024, strategy, monkeypatch):
    """40 x 1024^2 frames at patch_sidelength=64: 900 patches, 36000 jobs in one chunk.  The field is bitwise the same
    when the chunking splits the work into many small launches."""
    m = movie_40x1024.to(dev)
    kw = dict(patch_sidelength=64, reference_strategy=strategy)
    f_one, _ = tmc.estimate_motion_cross_correlation_patches(m, 1.0, **kw)
    f_one = f_one.clone()
    assert bool(torch.isfinite(f_one).all())
    monkeypatch.setattr(_fourier, "CHUNK_BYTES", 1 << 22)
    f_split, _ = tmc.estimate_motion_cross_correlation_patches(m, 1.0, **kw)
    assert torch.equal(f_one, f_split)
