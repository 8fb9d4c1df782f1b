"""FFT building blocks, tables and the cross-correlation estimators against the oracle / goldens."""

import numpy as np
import pytest
import torch

import torch_motion_correction_b200 as tmc
from oracle import deps
from oracle import reference_path as rp
from torch_motion_correction_b200 import _fourier, _ops

pytestmark = pytest.mark.gpu

SHIFT_PX = 0.01  # north-star tolerance on estimated shifts (px)


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def as_complex(t):
    return torch.view_as_complex(t.contiguous())


@pytest.mark.parametrize(
    "shape",
    [(16, 16), (32, 32), (64, 128), (128, 64), (256, 256), (512, 1024), (2048, 2048),
     # arbitrary lengths run as Bluestein chirp-z transforms on the same FFT core
     (96, 96), (48, 80), (100, 36), (959, 927), (30, 4092),
     # axes beyond the shared-memory transforms: decimated by R (5000 = 2 x 2500, 5760 = 2 x 2880, 9000 = 3 x 3000,
     # 11520 = 3 x 3840, 12288 = 3 x 4096, 16384 = 4 x 4096), every output bin sums R aliased sources
     (5000, 48), (64, 5760), (4100, 5000), (9000, 40), (32, 11520), (12288, 32), (48, 16384)],
)
def test_full_rfft2_and_irfft2_match_torch(dev, shape):
    ny, nx = shape
    g = torch.Generator().manual_seed(ny + nx)
    t = 3
    img = torch.randn((t, ny, nx), generator=g).to(dev)
    plan = _fourier.BandPlan(ny, nx, dev, full=True)
    spec = plan.forward(img, None, None, 0, ny, _fourier.frame_pair_jobs(t, dev), job_mode=2)[:t]
    want = torch.fft.rfftn(img.double(), dim=(-2, -1))
    err = (as_complex(spec).to(torch.complex128) - want).abs().max() / want.abs().max()
    assert float(err) < 2e-6
    back = torch.empty_like(img)
    plan.inverse_full(spec, back)
    assert float((back - img).abs().max()) < 1e-5 * float(img.abs().max()) * np.log2(ny * nx)


@pytest.mark.parametrize("p,radius,smooth", [(32, 8.0, 4.0), (128, 32.0, 16.0), (128, 32.0, 32.0), (64, 16.0, 0.0)])
def test_soft_disc_mask_matches_circle(dev, p, radius, smooth):
    want = deps.circle(radius, (p, p), smoothing_radius=smooth)
    got, ylo, yhi = _fourier.soft_disc_mask((p, p), radius, smooth, dev)
    assert float((got.cpu() - want).abs().max()) < 1e-6
    rows = (want != 0).any(dim=1).nonzero().flatten()
    assert ylo <= int(rows[0]) and int(rows[-1]) < yhi


def test_soft_disc_mask_non_square(dev):
    want = deps.circle(20.0, (64, 96), smoothing_radius=10.0)
    got, _, _ = _fourier.soft_disc_mask((64, 96), 20.0, 10.0, dev)
    assert float((got.cpu() - want).abs().max()) < 1e-6


@pytest.mark.parametrize("n,px,fr,b", [(128, 1.0, (300, 10), 500), (64, 1.3, (120, 6), 500), (32, 1.3, (120, 6), 1000), (256, 0.83, (300, 10), 500)])
def test_band_weights_match_reference_filters(dev, n, px, fr, b):
    band, env = rp.fourier_weight((n, n), px, b, fr)
    want = band * env  # (n, n//2+1)
    plan = _fourier.BandPlan(n, n, dev, px, b, fr)
    got = plan.weight.cpu()
    ky = (torch.arange(plan.ky) + plan.ky_start) % n
    box = want[ky][:, : plan.kx]
    assert float((got - box).abs().max()) < 1e-6
    # nothing of the pass band lies outside the kept box
    outside = want.clone()
    outside[ky[:, None], torch.arange(plan.kx)[None, :]] = 0
    assert float(outside.abs().max()) == 0.0
    assert int((got != 0).sum()) == int((want != 0).sum())


def test_band_limited_patch_spectra(dev):
    """rows+cols forward kernels vs torch: rfft2(mask^e * normalised patch) * W on the band box."""
    movie, _ = rp.synthetic_movie(4, 160, 192, seed=4)
    p, px, fr = 64, 1.1, (100, 5)
    m = movie.to(dev)
    stats = _ops.stack_stats(m)
    plan = _fourier.BandPlan(p, p, dev, px, 500, fr)
    mask, ylo, yhi = _fourier.soft_disc_mask((p, p), p / 4, p / 8, dev)
    jobs = torch.tensor([[0, 1, 0, 2, 10, 20], [2, 1, 3, 3, 96, 128], [1, 2, -1, 1, 50, 7]], dtype=torch.int32).to(dev)
    spec = as_complex(plan.forward(m, stats, mask, ylo, yhi, jobs)).cpu()
    norm = rp.normalize_image(movie)
    mk = deps.circle(p / 4, (p, p), smoothing_radius=p / 8)
    band, env = rp.fourier_weight((p, p), px, 500, fr)
    ky = (torch.arange(plan.ky) + plan.ky_start) % p
    for j, (fa, ea, fb, eb, y0, x0) in enumerate(jobs.cpu().tolist()):
        for part, (f, e) in enumerate(((fa, ea), (fb, eb))):
            if f < 0:
                continue
            want = torch.fft.rfftn(norm[f, y0 : y0 + p, x0 : x0 + p] * mk**e, dim=(-2, -1)) * band * env
            want = want[ky][:, : plan.kx]
            err = (spec[2 * j + part] - want).abs().max() / want.abs().max()
            assert float(err) < 5e-6, (j, part, float(err))


def test_global_motion_golden(dev, golden_small, golden_c1):
    g = golden_small
    movie = torch.as_tensor(g["movie"]).to(dev)
    px, fr = float(g["pixel_spacing"]), tuple(float(v) for v in g["frequency_range"])
    got = tmc.estimate_global_motion(movie, px, frequency_range=fr)
    assert got.shape == (2, 6, 1, 1)
    assert float((got.cpu() - torch.as_tensor(g["global_field"])).abs().max()) <= SHIFT_PX * px
    got = tmc.estimate_global_motion(movie, px, reference_frame=0, b_factor=1000, frequency_range=fr)
    assert float((got.cpu() - torch.as_tensor(g["global_field_ref0_b1000"])).abs().max()) <= SHIFT_PX * px
    # BASELINE config 1: known integer drifts are recovered exactly
    movie, walk = rp.synthetic_movie(10, 512, 512, seed=0, noise=1.0, drift=6.0, integer_shifts=True, sigma_f=0.08)
    got = tmc.estimate_global_motion(movie.to(dev), 1.0).cpu()
    assert torch.equal(got, torch.as_tensor(golden_c1["global_field"]))
    assert torch.equal(got[:, :, 0, 0].T, walk)


@pytest.mark.parametrize("strategy", ["mean_except_current", "middle_frame"])
def test_xc_patches_golden(dev, golden_small, strategy):
    g = golden_small
    movie = torch.as_tensor(g["movie"]).to(dev)
    px, fr = float(g["pixel_spacing"]), tuple(float(v) for v in g["frequency_range"])
    f, pos = tmc.estimate_motion_cross_correlation_patches(
        movie, px, reference_strategy=strategy, patch_sidelength=32, frequency_range=fr,
        temporal_smoothing=False, outlier_rejection=False,
    )
    assert np.array_equal(pos.cpu().numpy(), g["xc_positions"])
    assert float((f.cpu() - torch.as_tensor(g[f"xc_raw_{strategy}"])).abs().max()) <= SHIFT_PX * px
    f, _ = tmc.estimate_motion_cross_correlation_patches(
        movie, px, reference_strategy=strategy, patch_sidelength=32, frequency_range=fr,
        smoothing_window_size=3, outlier_threshold=1.5,
    )
    assert float((f.cpu() - torch.as_tensor(g[f"xc_full_{strategy}"])).abs().max()) <= SHIFT_PX * px


def test_xc_patches_integer_and_cumulative_golden(dev, golden_small):
    g = golden_small
    movie = torch.as_tensor(g["movie"]).to(dev)
    px, fr = float(g["pixel_spacing"]), tuple(float(v) for v in g["frequency_range"])
    f, _ = tmc.estimate_motion_cross_correlation_patches(
        movie, px, patch_sidelength=32, frequency_range=fr, sub_pixel_refinement=False,
        temporal_smoothing=False, outlier_rejection=False,
    )
    assert float((f.cpu() - torch.as_tensor(g["xc_integer"])).abs().max()) <= 1e-5
    g0 = torch.as_tensor(g["global_field"]).to(dev)
    f, _ = tmc.estimate_motion_cross_correlation_patches(movie, px, patch_sidelength=32, frequency_range=fr, deformation_field=g0)
    assert float((f.cpu() - torch.as_tensor(g["xc_cumulative_global"])).abs().max()) <= SHIFT_PX * px
    assert torch.equal(g0.cpu(), torch.as_tensor(g["xc_cumulative_global_field_after"]))  # Q2
    f0 = torch.as_tensor(g["xc_cumulative_full_in"]).to(dev)
    f, _ = tmc.estimate_motion_cross_correlation_patches(movie, px, patch_sidelength=32, frequency_range=fr, deformation_field=f0)
    assert float((f.cpu() - torch.as_tensor(g["xc_cumulative_full"])).abs().max()) <= SHIFT_PX * px


@pytest.mark.parametrize("strategy", ["mean_except_current", "middle_frame"])
def test_xc_patches_eviction_regime(dev, golden_eviction, strategy):
    """T = 60 > 50: the cache-eviction regime of quirk Q1."""
    g = golden_eviction
    movie = torch.as_tensor(g["movie"].astype(np.float32)).to(dev)
    fr = tuple(float(v) for v in g["frequency_range"])
    f, _ = tmc.estimate_motion_cross_correlation_patches(
        movie, 1.0, reference_strategy=strategy, patch_sidelength=32, frequency_range=fr,
        temporal_smoothing=False, outlier_rejection=False,
    )
    assert float((f.cpu() - torch.as_tensor(g[f"xc_raw_{strategy}"])).abs().max()) <= SHIFT_PX


def test_xc_patches_c1_golden(dev, golden_c1):
    g = golden_c1
    movie, _ = rp.synthetic_movie(10, 512, 512, seed=0, noise=1.0, drift=6.0, integer_shifts=True, sigma_f=0.08)
    f, pos = tmc.estimate_motion_cross_correlation_patches(movie.to(dev), 1.0, patch_sidelength=128)
    assert np.array_equal(pos.cpu().numpy(), g["xc_positions"])
    assert float((f.cpu() - torch.as_tensor(g["xc_field"])).abs().max()) <= SHIFT_PX
    s = tmc.correct_motion_sum(movie.to(dev), f, 1.0, grid_type="bspline").cpu()
    want = torch.as_tensor(g["corrected_sum_rows"])
    assert float(torch.linalg.norm(s[::64] - want) / torch.linalg.norm(want)) <= 1e-4


def test_correct_motion_fast_golden(dev, golden_small):
    g = golden_small
    movie = torch.as_tensor(g["movie"]).to(dev)
    field = torch.as_tensor(g["field_611"]).to(dev)
    out = tmc.correct_motion_fast(movie, field)
    want = torch.as_tensor(g["correct_fast"])  # every other row
    assert float(torch.linalg.norm(out.cpu()[:, ::2] - want) / torch.linalg.norm(want)) <= 1e-4
    assert torch.equal(field.cpu(), torch.as_tensor(g["correct_fast_field_after"]))  # Q2: negated in place
    with pytest.raises(ValueError, match="Expected single patch deformation field"):
        tmc.correct_motion_fast(movie, torch.zeros((2, 6, 2, 2), device=dev))
    zero = torch.zeros((2, 6, 1, 1), device=dev)
    assert torch.allclose(tmc.correct_motion_fast(movie, zero), movie, atol=1e-5)


def test_unsupported_length_raises(dev):
    # 8198 = 2 x 4099 (prime): no decimation into lengths the shared-memory transforms cover
    with pytest.raises(NotImplementedError):
        tmc.estimate_global_motion(torch.zeros((2, 8198, 64), device=dev), 1.0)
    # full (not band-limited) transforms of a decimated length whose accumulators do not fit in shared memory
    assert _ops.query("tmc_fft_supported_length", 13000) == 2
    with pytest.raises(NotImplementedError):
        tmc.correct_motion_fast(torch.zeros((2, 13000, 64), device=dev), torch.zeros((2, 2, 1, 1), device=dev))


def test_correct_motion_fast_k3_frame_size(dev):
    """correct_motion_fast (full-spectrum Fourier shift) on K3-sized frames, 5760 = 2 x 2880 columns, against the oracle."""
    movie, _ = rp.synthetic_movie(3, 4092, 5760, seed=5, noise=1.0, drift=3.0, sigma_f=0.08)
    field = torch.tensor([[0.0, 1.7, -2.4], [0.0, -3.2, 5.5]]).reshape(2, 3, 1, 1)
    want = rp.correct_motion_fast(movie, field.clone())
    got = tmc.correct_motion_fast(movie.to(dev), field.clone().to(dev))
    assert float(torch.linalg.norm(got.cpu() - want) / torch.linalg.norm(want)) <= 1e-4


@pytest.mark.parametrize("shape", [(5000, 4100), (5760, 4092), (600, 9000), (11520, 96), (16384, 128)])
def test_band_limited_spectra_of_long_axes(dev, shape):
    """Axes beyond the shared-memory transforms (> 4096, not a power of two <= 8192) are decimated, n = R n': the R
    sub-transforms are combined on the band (forward) / the twiddled band is inverted per sub-sequence (inverse)."""
    ny, nx = shape
    g = torch.Generator().manual_seed(ny + nx)
    img = torch.randn((3, ny, nx), generator=g).to(dev)
    px = 1.0
    plan = _fourier.BandPlan(ny, nx, dev, px, 500.0, (300, 10))
    mask, ylo, yhi = _fourier.soft_disc_mask((ny, nx), min(ny, nx) / 4, min(ny, nx) / 8, dev)
    spec = plan.forward(img, None, mask, ylo, yhi, _fourier.frame_pair_jobs(3, dev), job_mode=2)[:3]
    full = torch.fft.rfftn((img * mask).double(), dim=(-2, -1))
    ky = (torch.arange(plan.ky, device=dev) + plan.ky_start) % ny
    want = full[:, ky][:, :, : plan.kx] * plan.weight.double()
    err = (as_complex(spec).to(torch.complex128) - want).abs().max() / want.abs().max()
    assert float(err) < 5e-6, float(err)
    # inverse + argmax: the cross-correlation of frame 0 with a rolled copy of itself peaks at the roll
    sy, sx = min(37, ny // 16), -min(21, nx // 16)  # well inside the mask of the narrow shapes
    pair = torch.stack([img[0], torch.roll(img[0], (sy, sx), dims=(0, 1))])
    sp = plan.forward(pair, None, mask, ylo, yhi, _fourier.frame_pair_jobs(2, dev), job_mode=2)
    prod = _fourier.pair_products(sp, torch.tensor([0], dtype=torch.int32, device=dev), torch.tensor([1], dtype=torch.int32, device=dev),
                                  plan.plane_elems)
    shifts = plan.peaks(prod.view(1, plan.ky, plan.kx, 2), sub_pixel=False)
    assert shifts.cpu().tolist() == [[float(sy), float(sx)]]


def test_global_motion_k3_frame_size(dev):
    """K3-sized frames (5760 x 4092) through estimate_global_motion against the oracle."""
    movie, walk = rp.synthetic_movie(4, 4092, 5760, seed=3, noise=1.0, drift=7.0, integer_shifts=True, sigma_f=0.08)
    want = rp.estimate_global_motion(movie, 0.83)
    got = tmc.estimate_global_motion(movie.to(dev), 0.83)
    assert torch.equal(torch.round(got[:, :, 0, 0].T.cpu() / 0.83), walk)
    assert float((got.cpu() - want).abs().max()) <= 1e-5


def test_half_length_row_transforms_agree_with_the_full_length_kernels(dev, monkeypatch):
    """4096-point rows of frame pairs: two 2048-point transforms of pixel pairs (rows_forward_real2n, the default) against
    one 4096-point transform of the packed pair (TMC_FFT_REAL2N=0) and against torch.fft; odd window origins take the
    4-byte load path, an odd frame count the single-frame job."""
    n = 4096
    g = torch.Generator().manual_seed(23)
    movie = (torch.randn((3, 700, n + 8), generator=g) * 2.0 + 1.0).to(dev)
    plan = _fourier.BandPlan(512, n, dev, 0.83, 500, (300, 10))
    mask, ylo, yhi = _fourier.soft_disc_mask((512, n), 128.0, 64.0, dev)
    jobs = torch.tensor([[0, 1, 1, 1, 100, 4], [2, 1, -1, 1, 37, 5]], dtype=torch.int32).to(dev)
    out = {}
    for flag in ("1", "0"):
        monkeypatch.setenv("TMC_FFT_REAL2N", flag)
        out[flag] = as_complex(plan.forward(movie, None, mask, ylo, yhi, jobs, job_mode=2)).clone()
    scale = float(out["0"][:3].abs().max())  # plane 3 (no second frame in the last job) is never written
    assert float((out["1"][:3] - out["0"][:3]).abs().max()) <= 5e-6 * scale
    ky = (torch.arange(plan.ky, device=dev) + plan.ky_start) % 512
    for plane, (f, y0, x0) in ((0, (0, 100, 4)), (1, (1, 100, 4)), (2, (2, 37, 5))):
        want = torch.fft.rfftn((movie[f, y0 : y0 + 512, x0 : x0 + n] * mask).double(), dim=(-2, -1))[ky][:, : plan.kx]
        want = want * plan.weight.double()
        err = (out["1"][plane].to(torch.complex128) - want).abs().max() / want.abs().max()
        assert float(err) < 5e-6, (plane, float(err))


def test_global_motion_non_power_of_two_frames(dev):
    """96x80 frames (Bluestein on both axes) recover known integer drifts exactly."""
    movie, walk = rp.synthetic_movie(6, 96, 80, seed=2, noise=0.3, drift=4.0, integer_shifts=True, sigma_f=0.1)
    want = rp.estimate_global_motion(movie, 1.0, frequency_range=(60, 4))
    got = tmc.estimate_global_motion(movie.to(dev), 1.0, frequency_range=(60, 4)).cpu()
    assert torch.equal(got, want)
    assert torch.equal(got[:, :, 0, 0].T, walk)


@pytest.mark.parametrize("job_mode,x0", [(1, 36), (2, 36), (2, 37)])
def test_polyphase_rows_1024_patch_spectra(dev, job_mode, x0):
    """1024-px patches run the polyphase row kernel (four 256-point warp FFTs per row, csrc/fourier_poly.cuh):
    rfft2(mask^e * normalised patch) * W on the band box against torch.fft in float64; x0 = 37 exercises the
    misaligned (scalar-load) path."""
    g = torch.Generator().manual_seed(11)
    movie = torch.randn((3, 1100, 1100), generator=g) * 2.0 + 1.0
    p, px, fr = 1024, 0.9, (300, 10)
    m = movie.to(dev)
    stats = _ops.stack_stats(m)
    plan = _fourier.BandPlan(p, p, dev, px, 500, fr)
    assert plan.kx <= 128
    mask, ylo, yhi = _fourier.soft_disc_mask((p, p), p / 4, p / 8, dev)
    if job_mode == 1:
        jobs = [[0, 1, 0, 2, 40, x0], [2, 1, 2, 2, 3, 5]]
    else:
        jobs = [[0, 1, 1, 1, 40, x0], [2, 1, -1, 1, 3, 5]]
    jobs_dev = torch.tensor(jobs, dtype=torch.int32).to(dev)
    spec = as_complex(plan.forward(m, stats, mask, ylo, yhi, jobs_dev, job_mode=job_mode)).cpu()
    norm = rp.normalize_image(movie).double()
    mk = deps.circle(p / 4, (p, p), smoothing_radius=p / 8).double()
    band, env = rp.fourier_weight((p, p), px, 500, fr)
    ky = (torch.arange(plan.ky) + plan.ky_start) % p
    for j, (fa, ea, fb, eb, y0, xx) in enumerate(jobs):
        for part, (f, e) in enumerate(((fa, ea), (fb, eb))):
            if f < 0:
                continue
            want = torch.fft.rfftn(norm[f, y0 : y0 + p, xx : xx + p] * mk**e, dim=(-2, -1)) * (band * env).double()
            want = want[ky][:, : plan.kx]
            err = (spec[2 * j + part].to(torch.complex128) - want).abs().max() / want.abs().max()
            assert float(err) < 5e-6, (j, part, float(err))


def test_polyphase_rows_1024_peaks(dev):
    """Inverse polyphase rows + argmax on 1024 x 1024 surfaces: a band-limited product whose correlation peak
    sits at a known integer position, plus agreement with torch.fft.irfftn's argmax on random band-limited data."""
    p, px, fr = 1024, 1.0, (300, 10)
    plan = _fourier.BandPlan(p, p, dev, px, 500, fr)
    ky = ((torch.arange(plan.ky) + plan.ky_start) % p).to(dev)
    g = torch.Generator().manual_seed(5)
    n = 5
    # band-limit the spectrum of a REAL random image: Hermitian-consistent input, as the products of real patches are
    img = torch.randn((n, p, p), generator=g).to(dev)
    spec = torch.fft.rfftn(img, dim=(-2, -1))
    kxs = torch.arange(plan.kx, device=dev)
    box = torch.view_as_real(spec[:, ky[:, None], kxs[None, :]].contiguous()) * (plan.weight != 0)[None, :, :, None]
    full = torch.zeros((n, p, p // 2 + 1), dtype=torch.complex64, device=dev)
    full[:, ky[:, None], kxs[None, :]] = torch.view_as_complex(box.contiguous())
    surf = torch.fft.irfftn(full, s=(p, p), dim=(-2, -1))
    want = surf.reshape(n, -1).argmax(dim=1)
    wy, wx = (want // p).float(), (want % p).float()
    wy = torch.where(wy > p // 2, wy - p, wy)
    wx = torch.where(wx > p // 2, wx - p, wx)
    got = plan.peaks(box.contiguous(), sub_pixel=False)
    # the argmax itself, up to fp32 near-ties of the band-limited (smooth) surface between the two transforms
    gy, gx = got[:, 0].long() % p, got[:, 1].long() % p
    picked = surf[torch.arange(n, device=dev), gy, gx]
    top = surf.reshape(n, -1).max(dim=1).values
    assert bool((picked >= top - 1e-4 * top.abs()).all()), (got, wy, wx, picked, top)
    assert int(((gy == want // p) & (gx == want % p)).sum()) >= n - 1


@pytest.mark.parametrize("shape,voltage", [((6, 96, 128), 300.0), ((5, 300, 256), 200.0), ((7, 64, 90), 300.0),
                                           ((3, 600, 5000), 300.0)])  # 5000 = 2 x 2500: decimated full-spectrum rows
def test_dose_weighted_sum_matches_oracle(dev, shape, voltage, monkeypatch):
    """tmc.dose_weight (full rfft2 of every frame, exposure-filtered sum in Fourier space, ONE inverse transform)
    against the example script's per-frame filter + irfft2 + sum; frame blocks accumulate (forced small blocks)."""
    import sys

    dw_mod = sys.modules["torch_motion_correction_b200.dose_weight"]  # the package attribute of that name is the function
    g = torch.Generator().manual_seed(31)
    movie = torch.randn(shape, generator=g) + 3.0
    want = rp.dose_weight(movie, 0.936, pre_exposure=1.5, dose_per_frame=1.2, voltage=voltage)
    got = tmc.dose_weight(movie.to(dev), 0.936, pre_exposure=1.5, dose_per_frame=1.2, voltage=voltage).cpu()
    assert float(torch.linalg.norm(got - want) / torch.linalg.norm(want)) <= 1e-5
    monkeypatch.setattr(dw_mod, "_BLOCK_BYTES", 2 * shape[1] * (shape[2] // 2 + 1) * 8)
    blocked = tmc.dose_weight(movie.to(dev), 0.936, pre_exposure=1.5, dose_per_frame=1.2, voltage=voltage).cpu()
    assert float(torch.linalg.norm(blocked - want) / torch.linalg.norm(want)) <= 1e-5


@pytest.mark.parametrize("strategy", ["mean_except_current", "middle_frame"])
def test_xc_patches_exposure_prefilter(dev, golden_small, strategy):
    """Additive option: per-frame exposure (dose) weights on the patch spectra before the leave-one-out sums and the
    cross-correlation, against the oracle restatement with the same filter; the filter really changes the estimate."""
    g = golden_small
    movie = torch.as_tensor(g["movie"])
    px, fr = float(g["pixel_spacing"]), tuple(float(v) for v in g["frequency_range"])
    kw = dict(reference_strategy=strategy, patch_sidelength=32, frequency_range=fr)
    want, _ = rp.estimate_motion_cross_correlation_patches(movie, px, smooth=False, reject_outliers=False, dose=(0.5, 4.0, 300.0), **kw)
    got, _ = tmc.estimate_motion_cross_correlation_patches(
        movie.to(dev), px, temporal_smoothing=False, outlier_rejection=False, dose_per_frame=4.0, pre_exposure=0.5, **kw
    )
    assert float((got.cpu() - want).abs().max()) <= SHIFT_PX * px
    plain = torch.as_tensor(g[f"xc_raw_{strategy}"])
    assert float((want - plain).abs().max()) > 1e-4
