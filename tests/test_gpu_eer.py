"""EER rendering on the device (prepare.render_eer, csrc/eer.cu): counts bitwise equal to np.add.at over the electron
lists the movies were written from (tests/eer_synth.py, which follows the format rules, not the decoder); malformed
frames reported by index; EER movies through motion_correct_many; drift recovered from rendered fractions."""

import numpy as np
import pytest
import torch

import eer_synth as es
import torch_motion_correction_b200 as tmc
from torch_motion_correction_b200 import movie_io, prepare

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda", 0)
CODECS = [(65000, None), (65001, None), (65002, (6, 2, 1))]


def rle_of(compression, codec):
    return codec[0] if compression == 65002 else es.CODECS[compression][0]


def render_written(tmp_path, frames, h, w, F, compression=65001, codec=None, name="m.eer", **kw):
    path = tmp_path / name
    es.write_eer(path, frames, h, w, compression=compression, codec=codec, **kw)
    return tmc.render_eer(movie_io.read_eer(path), F, device=DEV)


def assert_exact(got, frames, h, w, F):
    want = es.reference_counts(frames, h, w, F)
    assert got.dtype == (torch.uint8 if F <= 255 else torch.uint16)
    assert tuple(got.shape) == want.shape
    assert np.array_equal(got.cpu().to(torch.int64).numpy(), want)


@pytest.mark.parametrize("compression,codec", CODECS)
@pytest.mark.parametrize("h,w", [(64, 48), (1000, 777)])
def test_random_frames_in_strips_cut_inside_codes(tmp_path, compression, codec, h, w):
    frames = es.random_frames(np.random.default_rng(h + compression), 6, h * w, 0.05)
    got = render_written(tmp_path, frames, h, w, 2, compression, codec, n_strips=5, bigtiff=h > 100)
    assert_exact(got, frames, h, w, 2)


def test_full_size_frames():
    import tempfile
    from pathlib import Path

    h = w = 4096
    frames = es.random_frames(np.random.default_rng(7), 4, h * w, 0.025)
    with tempfile.TemporaryDirectory() as d:
        assert_exact(render_written(Path(d), frames, h, w, 2, n_strips=3), frames, h, w, 2)


@pytest.mark.parametrize("compression,codec", CODECS)
def test_escape_gaps_first_and_last_pixel(tmp_path, compression, codec):
    h, w = 120, 90
    m = (1 << rle_of(compression, codec)) - 1  # the escape value
    n = h * w
    gaps = np.array([m, 2 * m, 3 * m, m - 1, m + 1, 0, 5 * m])
    inner = np.cumsum(gaps + 1)  # electron k sits `gaps[k]` pixels after the previous one
    frames = [np.array([0, *inner[inner < n - 1], n - 1]),  # first and last pixel
              np.array([n - 1 - m]),                       # the final gap is exactly one escape
              np.array([0]),                               # the final gap is n - 1
              np.arange(0, n, m + 1)[: n // (m + 1)],      # every gap exactly m
              np.array([n - 1]),
              np.array([m])]                               # an escape, then an electron at offset 0
    frames = [np.unique(f[f < n]) for f in frames]
    got = render_written(tmp_path, frames, h, w, 1, compression, codec, n_strips=2)
    assert_exact(got, frames, h, w, 1)


@pytest.mark.parametrize("compression,codec", CODECS)
def test_empty_frames_and_dense_rows(tmp_path, compression, codec):
    h, w = 64, 48
    n = h * w
    frames = [np.array([], dtype=np.int64), np.concatenate([np.arange(3 * w, 4 * w), np.arange(7 * w, 9 * w)]),
              np.arange(n), np.array([], dtype=np.int64)]
    got = render_written(tmp_path, frames, h, w, 2, compression, codec, n_strips=3)
    assert_exact(got, frames, h, w, 2)


def test_hand_built_frame(tmp_path):
    # the frame of tests/test_eer_io.py: 16 x 16, electrons at 0, 130 (after an escape) and 255, 65001
    frames = [np.array([0, 130, 255]), np.array([1, 2, 3])]
    assert_exact(render_written(tmp_path, frames, 16, 16, 1), frames, 16, 16, 1)


@pytest.mark.parametrize("F", [1, 7, 255, 256])
def test_fraction_sizes(tmp_path, F):
    """F = 255 / 256 is the uint8 -> uint16 switch: pixel 5 holds an electron in every frame, so a fraction's count
    reaches F there; 520 frames leave a remainder (dropped) for F = 7, 255 and 256."""
    rng = np.random.default_rng(F)
    frames = [np.union1d(f, [5]) for f in es.random_frames(rng, 520, 32 * 32, 0.3)]
    got = render_written(tmp_path, frames, 32, 32, F)
    assert got.shape[0] == 520 // F
    assert int(got[0, 0, 5]) == F
    assert_exact(got, frames, 32, 32, F)


def test_too_few_fractions_is_an_error(tmp_path):
    frames = es.random_frames(np.random.default_rng(0), 5, 64, 0.1)
    path = tmp_path / "few.eer"
    es.write_eer(path, frames, 8, 8)
    with pytest.raises(ValueError, match="need >= 2"):
        tmc.render_eer(movie_io.read_eer(path), 3, device=DEV)


def test_calls_are_bitwise_repeatable(tmp_path):
    frames = es.random_frames(np.random.default_rng(3), 8, 1000 * 777, 0.05)
    path = tmp_path / "r.eer"
    es.write_eer(path, frames, 1000, 777, compression=65000, n_strips=4)
    eer = movie_io.read_eer(path)
    first = tmc.render_eer(eer, 4, device=DEV)
    out = torch.full_like(first, 7)
    again = tmc.render_eer(eer, 4, device=DEV, out=out)
    assert again is out and torch.equal(first, again)


def test_malformed_frames_are_reported_and_the_rest_is_exact(tmp_path):
    h, w = 200, 150
    n = h * w
    rng = np.random.default_rng(11)
    frames = es.random_frames(rng, 6, n, 0.05)
    frames[4] = np.union1d(frames[4][frames[4] < n - 2], [n - 2])
    streams = [es.encode_frame(f, n, 7, 4, rng) for f in frames]
    streams[2] = streams[2][: len(streams[2]) // 2]  # runs out of bytes half way
    # written for 5 more pixels: after the electron at n - 2 the final gap (6) moves past n without landing on it
    streams[4] = es.encode_frame(frames[4], n + 5, 7, 4, rng)
    path = tmp_path / "bad.eer"
    es.write_eer(path, None, h, w, streams=streams)
    eer = movie_io.read_eer(path)
    with pytest.raises(ValueError, match=r"malformed EER frame\(s\) 2, 4:"):
        tmc.render_eer(eer, 1, device=DEV)
    # the same render without the check: every other frame exact, the malformed ones contribute nothing
    counts = prepare.eer_counts_buffer((6, h, w), torch.uint8, DEV)
    status = torch.empty((6,), dtype=torch.int32, device=DEV)
    prepare.render_eer_into(eer.payload.to(DEV), eer.frame_offsets.to(DEV), eer, 1, counts, status)
    assert status.cpu().tolist() == [0, 0, 1, 0, 1, 0]
    want = es.reference_counts(frames, h, w, 1)
    want[[2, 4]] = 0
    assert np.array_equal(counts.cpu().to(torch.int64).numpy(), want)


def test_pipeline_matches_host_rendered_counts(tmp_path):
    h = w = 128
    F = 10
    kwargs = dict(patch_sidelength=64, frequency_range=(80, 5), n_iterations=0, dose_per_frame=1.5)
    gain = 1.0 + 0.1 * torch.rand((h, w), generator=torch.Generator().manual_seed(1))
    paths, host = [], []
    for i in range(3):
        frames = es.random_frames(np.random.default_rng(20 + i), 100 + 3 * i, h * w, 0.1)  # 0, 3 and 6 frames dropped
        paths.append(tmp_path / f"p{i}.eer")
        es.write_eer(paths[-1], frames, h, w, compression=65000 + i, codec=(7, 2, 2) if i == 2 else None)
        host.append(torch.from_numpy(es.reference_counts(frames, h, w, F).astype(np.uint8)).pin_memory())
    got = [(s.clone(), f.cpu()) for s, f in
           tmc.motion_correct_many(tmc.eer_movies(paths), 1.0, device=DEV, eer_frames_per_fraction=F, gain=gain, **kwargs)]
    want = [(s.clone(), f.cpu()) for s, f in tmc.motion_correct_many(host, 1.0, device=DEV, gain=gain, **kwargs)]
    assert len(got) == 3
    for (gs, gf), (ws, wf) in zip(got, want):
        assert torch.equal(gs, ws) and torch.equal(gf, wf)
    with pytest.raises(ValueError, match="eer_frames_per_fraction"):
        list(tmc.motion_correct_many(tmc.eer_movies(paths), 1.0, device=DEV, **kwargs))


def test_pipeline_reports_a_malformed_movie(tmp_path):
    h = w = 128
    frames = es.random_frames(np.random.default_rng(4), 20, h * w, 0.1)
    rng = np.random.default_rng(0)
    streams = [es.encode_frame(f, h * w, 7, 4, rng) for f in frames]
    streams[13] = streams[13][:-30]
    es.write_eer(tmp_path / "ok.eer", frames, h, w)
    es.write_eer(tmp_path / "bad.eer", None, h, w, streams=streams)
    results = tmc.motion_correct_many(tmc.eer_movies([tmp_path / "ok.eer", tmp_path / "bad.eer"]), 1.0, device=DEV,
                                      eer_frames_per_fraction=4, patch_sidelength=64, frequency_range=(80, 5))
    next(results)
    with pytest.raises(ValueError, match=r"frame\(s\) 13:"):
        next(results)


# ---- end to end: drift recovered from rendered fractions --------------------------------------------------------

# 600 EER frames of a 1024^2 specimen at 0.05 e-/px each, rendered in 20-frame fractions (30 fractions of 1 e-/px);
# the specimen drifts linearly by DRIFT px in y and x over the movie.  Measured RMS error: see DESIGN §4.
E2E_DRIFT = (6.0, -4.0)
E2E_BOUND_PX = 0.5


def test_motion_correct_recovers_the_drift_of_an_eer_movie(tmp_path):
    from scipy import ndimage

    n, t, F, rate = 1024, 600, 20, 0.05
    rng = np.random.default_rng(42)
    spec = ndimage.gaussian_filter(rng.normal(size=(n + 64, n + 64)), 3.0)
    spec = np.clip(1.0 + 0.6 * spec / spec.std(), 0.0, 2.5)
    nf = t // F
    truth = np.outer(np.linspace(0, 1, nf), E2E_DRIFT)  # content displacement of each fraction (y, x) in px
    frames = []
    for k in range(nf):
        img = ndimage.shift(spec, truth[k], order=3, mode="wrap")[32:32 + n, 32:32 + n].reshape(-1)
        p = np.clip(rate * img, 0.0, 1.0)
        for _ in range(F):
            frames.append(np.flatnonzero(rng.random(n * n) < p))
    path = tmp_path / "drift.eer"
    es.write_eer(path, frames, n, n, bigtiff=True)
    counts = tmc.render_eer(movie_io.read_eer(path), F, device=DEV)
    assert_exact(counts, frames, n, n, F)
    _, field = tmc.motion_correct(tmc.prepare_movie(counts), 1.0, patch_sidelength=512)
    est = field.mean(dim=(2, 3)).T.cpu().numpy().astype(np.float64)  # (nf, 2) y, x in px (pixel spacing 1)
    err = np.sqrt((((est - est.mean(0)) - (truth - truth.mean(0))) ** 2).sum(-1).mean())
    print(f"EER end to end: RMS drift error {err:.3f} px over {nf} fractions")
    assert err <= E2E_BOUND_PX, err
