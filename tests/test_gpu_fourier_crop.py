"""Fourier cropping on the GPU: against a float64 rfft2 / box / irfft2 reference on both column paths, against an
analytic band-limited image, on the self-paired Nyquist columns of the box, bit for bit between calls, and through
motion_correct(fourier_bin=...) down to a known drift."""

import numpy as np
import pytest
import torch

import torch_motion_correction_b200 as tmc
from oracle import reference_path as rp

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")


def _reference(image, h2, w2):
    """float64 rfft2, the box ky in [-h2/2, h2/2), kx in [0, w2/2], irfft2 at (h2, w2), times h2 w2 / (h w), on the CPU:
    pocketfft's c2r (as numpy's) takes the Hermitian part of the box's self-paired columns, which is the documented
    meaning of irfft2 on a box that is not Hermitian there"""
    h, w = image.shape[-2:]
    X = torch.fft.rfft2(image.double().cpu())
    box = torch.cat([X[..., : h2 // 2, : w2 // 2 + 1], X[..., h - h2 // 2 :, : w2 // 2 + 1]], dim=-2)
    return torch.fft.irfft2(box, s=(h2, w2)) * (h2 * w2) / (h * w)


def _worst_rel(got, want):
    """largest per-frame relative L2 error"""
    got, want = got.reshape(-1, *got.shape[-2:]).double().cpu(), want.reshape(-1, *want.shape[-2:]).double().cpu()
    return max(float(torch.linalg.norm(g - r) / torch.linalg.norm(r)) for g, r in zip(got, want))


def _noise(shape, seed):
    return torch.randn(shape, generator=torch.Generator(device=DEV).manual_seed(seed), device=DEV)


CASES = [  # (t, h, w), factor; power-of-two heights halved or quartered run the fused column kernel
    ((2, 1024, 1024), 2),
    ((3, 4096, 4096), 2),
    ((2, 8192, 8192), 2),
    ((3, 4096, 4096), 4),
    ((2, 512, 1024), 2),  # rectangular powers of two
    ((3, 5760, 4092), 2),  # K3: decimated columns, Bluestein rows
    ((2, 11520, 8184), 2),  # K3 super-resolution
    ((3, 5760, 4092), 1.5),
    ((5, 1024, 768), 4),
    ((1, 256, 256), 2),
]


@pytest.mark.parametrize("shape,factor", CASES)
def test_matches_the_float64_reference(shape, factor):
    image = _noise(shape, seed=shape[1] + shape[0])
    h2, w2 = tmc.prepare.fourier_crop_shape(shape[1:], factor)
    got = tmc.fourier_crop(image, factor)
    assert got.shape == (shape[0], h2, w2) and got.dtype == torch.float32
    rel = _worst_rel(got, _reference(image, h2, w2))
    print(f"[fourier_crop] {shape} / {factor}: worst per-frame rel L2 {rel:.2e}")
    assert rel <= 1e-5, rel


def test_a_single_image():
    image = _noise((1024, 768), seed=3)
    got = tmc.fourier_crop(image, 2)
    assert got.shape == (512, 384)
    assert _worst_rel(got, _reference(image, 512, 384)) <= 1e-5
    assert torch.equal(got, tmc.fourier_crop(image[None], 2)[0])


def test_other_input_types_are_converted():
    image = _noise((2, 256, 256), seed=4)
    assert torch.equal(tmc.fourier_crop(image.half(), 2), tmc.fourier_crop(image.half().float(), 2))
    assert torch.equal(tmc.fourier_crop(image.cpu(), 2), tmc.fourier_crop(image, 2))


@pytest.mark.parametrize("h,w,factor", [(1024, 1024, 2), (4096, 2048, 4), (1152, 768, 1.5)])
def test_band_limited_cosines_are_sampled_exactly(h, w, factor):
    """Known answer independent of FFT conventions: a sum of cosines inside the box is the band-limited image itself,
    so the crop is that function sampled at (factor i, factor j)."""
    h2, w2 = tmc.prepare.fourier_crop_shape((h, w), factor)
    rng = np.random.default_rng(h + w)
    waves = [(int(rng.integers(-h2 // 2 + 1, h2 // 2)), int(rng.integers(0, w2 // 2)), rng.uniform(0.5, 2), rng.uniform(0, 2 * np.pi))
             for _ in range(6)] + [(0, 0, 3.0, 0.0), (h2 // 2 - 1, w2 // 2 - 1, 1.0, 0.3)]

    def field(y, x):
        return sum(a * torch.cos(2 * np.pi * (ky * y / h + kx * x / w) + p) for ky, kx, a, p in waves)

    y = torch.arange(h, dtype=torch.float64, device=DEV)[:, None]
    x = torch.arange(w, dtype=torch.float64, device=DEV)[None, :]
    image = field(y, x).float()
    want = field(factor * torch.arange(h2, dtype=torch.float64, device=DEV)[:, None],
                 factor * torch.arange(w2, dtype=torch.float64, device=DEV)[None, :])
    got = tmc.fourier_crop(image, factor).double()
    err = float((got - want).abs().max())
    print(f"[fourier_crop] cosines {h} x {w} / {factor}: max |error| {err:.2e}")
    assert err <= 2e-5 * sum(a for _, _, a, _ in waves), err


@pytest.mark.parametrize("shape,factor", [((2, 1024, 1024), 2), ((3, 5760, 4092), 2)])
def test_self_paired_columns_enter_through_their_hermitian_part(shape, factor):
    """Energy only at ky = h'/2 and kx = w'/2: the box holds ky = -h'/2 without its partner +h'/2, and its columns
    kx = 0 and kx = w'/2 are not Hermitian.  irfft2 takes those columns' Hermitian part; so must the crop."""
    t, h, w = shape
    h2, w2 = tmc.prepare.fourier_crop_shape((h, w), factor)
    y = torch.arange(h, dtype=torch.float64, device=DEV)[:, None]
    x = torch.arange(w, dtype=torch.float64, device=DEV)[None, :]
    frames = []
    for f in range(t):
        p = 0.7 + f
        frames.append(torch.cos(2 * np.pi * (h2 // 2) * y / h + p) + torch.cos(2 * np.pi * (w2 // 2) * x / w + 2 * p)
                      + torch.cos(2 * np.pi * ((h2 // 2) * y / h + (w2 // 2) * x / w) + 3 * p)
                      + torch.cos(2 * np.pi * ((h2 // 2) * y / h - 5 * x / w) + p))
    image = torch.stack(frames).float()
    want = _reference(image, h2, w2)
    assert float(want.abs().max()) > 0.1  # the case has something to get right
    rel = _worst_rel(tmc.fourier_crop(image, factor), want)
    print(f"[fourier_crop] Nyquist-only {shape} / {factor}: worst per-frame rel L2 {rel:.2e}")
    assert rel <= 1e-5, rel


@pytest.mark.parametrize("shape,factor", [((3, 8192, 8192), 2), ((3, 1024, 1024), 4), ((5, 2048, 768), 2)])
def test_fused_and_composed_column_passes_agree(shape, factor, monkeypatch):
    image = _noise(shape, seed=shape[1] + 7)
    fused = tmc.fourier_crop(image, factor)
    monkeypatch.setenv("TMC_FFT_CROP_FUSED", "0")
    composed = tmc.fourier_crop(image, factor)
    rel = _worst_rel(fused, composed.double())
    print(f"[fourier_crop] fused vs composed {shape} / {factor}: worst per-frame rel L2 {rel:.2e}, "
          f"bitwise {torch.equal(fused, composed)}")
    assert rel <= 1e-6, rel


def test_calls_are_bitwise_repeatable_and_factor_one_is_the_input():
    image = _noise((5, 2048, 2048), seed=9)
    a = tmc.fourier_crop(image, 2)
    b = tmc.fourier_crop(image, 2)
    assert torch.equal(a, b)
    assert tmc.fourier_crop(image, 1) is image


def test_chunked_calls_match_one_call(monkeypatch):
    from torch_motion_correction_b200 import _fourier

    image = _noise((7, 512, 512), seed=11)
    whole = tmc.fourier_crop(image, 2)
    monkeypatch.setattr(_fourier, "CHUNK_BYTES", 1)  # one frame pair per call
    assert torch.equal(tmc.fourier_crop(image, 2), whole)


# ---- the pipeline ---------------------------------------------------------------------------------------------------

PIPE = dict(patch_sidelength=96, frequency_range=(120.0, 6.0))


def _pipeline_movie():
    movie, _ = rp.synthetic_movie_large(16, 512, 512, seed=6, noise=1.0, drift=4.0, local=0.5, sigma_f=0.04)
    return movie.to(DEV)


@pytest.mark.parametrize("kw", [dict(), dict(dose_per_frame=0.3), dict(frame_group=2), dict(frame_group=2, dose_per_frame=0.3)])
def test_motion_correct_runs_on_the_cropped_movie(kw):
    movie = _pipeline_movie()
    px = 0.5
    total, field = tmc.motion_correct(movie, px, fourier_bin=2, **kw, **PIPE)
    want_total, want_field = tmc.motion_correct(tmc.fourier_crop(movie, 2), 2 * px, **kw, **PIPE)
    assert total.shape == (256, 256)
    assert torch.equal(field, want_field) and torch.equal(total, want_total)


def test_no_binning_is_todays_result():
    movie = _pipeline_movie()
    px = 0.5
    ref_total, ref_field = tmc.motion_correct(movie, px, **PIPE)
    for b in (None, 1, 1.0):
        total, field = tmc.motion_correct(movie, px, fourier_bin=b, **PIPE)
        assert torch.equal(field, ref_field) and torch.equal(total, ref_total), b


def test_motion_correct_many_bins_each_movie():
    movie = _pipeline_movie()
    px = 0.5
    host = [movie.half().cpu().pin_memory(), (movie.flip(1) * 0.5).half().cpu().pin_memory()]  # prepared on the device
    out_host = torch.empty((256, 256), dtype=torch.float32, pin_memory=True)  # the binned sum's size, reused
    got = [(s.clone(), f) for s, f in tmc.motion_correct_many(host, px, out_host=out_host, fourier_bin=2, **PIPE)]
    assert len(got) == 2
    for (s, f), m in zip(got, host):
        want_s, want_f = tmc.motion_correct(tmc.prepare_movie(m.to(DEV)), px, fourier_bin=2, **PIPE)
        assert torch.equal(f, want_f) and torch.equal(s.to(DEV), want_s)


# ---- known answer: a super-resolution movie with a known drift ---------------------------------------------------------

KNOWN_PX = 0.5  # Angstrom per super-resolution pixel
# Angstrom; on a B200 (1000 W) this case measures 0.111 A binned by 2 and 0.066 A at full resolution, on a track of RMS
# 1.52 A (a pixel spacing off by the binning factor would be about the whole track off)
KNOWN_RMS_BOUND = 0.2


def known_answer_rms(fourier_bin, t=24, n=1024, seed=8, drift=8.0):
    """RMS over frames of |mean field of frame k - true shift of frame k| in Angstrom (means over frames removed) for a
    rigidly drifting movie whose specimen lies below the binned Nyquist.  The estimators smooth the field over time with a
    5-frame Savitzky-Golay filter of order 1 (tmc_xc_postprocess), so the truth is the walk smoothed the same way: on this
    24-frame random walk of 4 A the smoothing alone moves it 0.62 A RMS."""
    from scipy.signal import savgol_filter

    movie, walk = rp.synthetic_movie_large(t, n, n, seed=seed, noise=1.0, drift=drift, local=0.0, sigma_f=0.04)
    _, field = tmc.motion_correct(movie.to(DEV), KNOWN_PX, fourier_bin=fourier_bin,
                                  patch_sidelength=256 // (fourier_bin or 1))
    est = field.mean(dim=(-2, -1)).T.cpu().double().numpy()  # (t, 2) Angstrom
    truth = savgol_filter(walk.double().numpy() * KNOWN_PX, 5, 1, axis=0, mode="interp")
    est, truth = est - est.mean(0), truth - truth.mean(0)
    return float(np.sqrt(((est - truth) ** 2).sum(-1).mean()))


def test_binned_estimate_tracks_a_known_drift():
    binned, full = known_answer_rms(2), known_answer_rms(None)
    print(f"[fourier_crop] known drift: RMS error {binned:.3f} A binned by 2, {full:.3f} A at full resolution")
    assert binned <= KNOWN_RMS_BOUND, (binned, full)
