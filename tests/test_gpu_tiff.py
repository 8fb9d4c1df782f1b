"""LZW TIFF movies decoded on the device (``tmc_tiff_lzw_decode``) against the frames they were written from: files of
the test writer (``tests/lzw_synth.py``), of Pillow and of OpenCV (both write through libtiff)."""

import numpy as np
import pytest
import torch

import eer_synth as es
import lzw_synth as ls
import torch_motion_correction_b200 as tmc
from torch_motion_correction_b200 import movie_io, prepare

pytestmark = pytest.mark.gpu

DEV = "cuda"


def decoded(path):
    return tmc.decode_tiff(tmc.read_tiff_movie(path), device=DEV).cpu().numpy()


def poisson(rng, shape, rate, dtype=np.uint8):
    return rng.poisson(rate, size=shape).astype(dtype)


def wrapping(rng, shape, dtype):
    """Samples spanning the whole type, so that undoing the differences wraps both ways."""
    info = np.iinfo(dtype)
    return rng.integers(info.min, info.max, size=shape, endpoint=True).astype(dtype)


@pytest.mark.parametrize("dtype", [np.uint8, np.int8, np.uint16, np.int16])
@pytest.mark.parametrize("predictor", [1, 2])
def test_sample_types_and_predictors(tmp_path, dtype, predictor):
    rng = np.random.default_rng(1)
    frames = np.concatenate([poisson(rng, (2, 61, 77), 0.8, dtype), wrapping(rng, (2, 61, 77), dtype)])
    path = tmp_path / "m.tif"
    ls.write_lzw_tiff(path, frames, rows_per_strip=9, predictor=predictor)
    got = decoded(path)
    assert got.dtype == frames.dtype and np.array_equal(got, frames)


def test_pillow_default_strips(tmp_path):
    Image = pytest.importorskip("PIL.Image")
    rng = np.random.default_rng(2)
    frames = poisson(rng, (3, 409, 576), 0.8)
    path = tmp_path / "p.tif"
    ims = [Image.fromarray(f) for f in frames]
    ims[0].save(path, compression="tiff_lzw", save_all=True, append_images=ims[1:])
    movie = tmc.read_tiff_movie(path)
    assert movie.n_strips > 3  # Pillow's ~64 KB strips
    assert np.array_equal(tmc.decode_tiff(movie, device=DEV).cpu().numpy(), frames)


def write_opencv(cv2, path, frames, rows_per_strip):
    params = [cv2.IMWRITE_TIFF_COMPRESSION, 5, cv2.IMWRITE_TIFF_ROWSPERSTRIP, rows_per_strip]
    assert cv2.imwritemulti(str(path), list(frames), params)


@pytest.mark.parametrize("rows_per_strip", [1, 64, 409])
@pytest.mark.parametrize("dtype", [np.uint8, np.uint16])
def test_opencv_strip_layouts(tmp_path, rows_per_strip, dtype):
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(3)
    frames = poisson(rng, (3, 409, 577), 0.8, dtype)
    path = tmp_path / "o.tif"
    write_opencv(cv2, path, frames, rows_per_strip)
    movie = tmc.read_tiff_movie(path)
    assert movie.predictor == 2  # OpenCV's default for LZW
    assert movie.n_strips == 3 * -(-409 // rows_per_strip)
    assert np.array_equal(tmc.decode_tiff(movie, device=DEV).cpu().numpy(), frames)


EDGE_CASES = {
    "no_leading_clear": dict(leading_clear=False),
    "no_eoi": dict(eoi=False),
    "extra_clears": dict(clears_after=(1, 2, 3, 100, 101, 5000)),
    "clear_at_9_to_10": dict(max_codes=254),
    "clear_at_10_to_11": dict(max_codes=766),
    "clear_at_11_to_12": dict(max_codes=1790),
    "clear_before_9_to_10": dict(max_codes=253),
    "full_table": dict(max_codes=3839),
    "no_clear_no_eoi": dict(leading_clear=False, eoi=False),
}


@pytest.mark.parametrize("case", sorted(EDGE_CASES))
def test_writer_edge_cases(tmp_path, case):
    rng = np.random.default_rng(4)
    frames = np.concatenate([poisson(rng, (2, 150, 333), 0.3), wrapping(rng, (1, 150, 333), np.uint8)])
    frames[0, :40] = 0  # long runs: KwKwK codes and long strings
    # every strip opens with a literal >= 2: without a leading Clear a first literal of 0 or 1 makes the strip's first
    # byte 0, which readers (libtiff, read_tiff_movie) take for the pre-TIFF-6 variant
    frames[:, ::70, 0] = 7
    kw = EDGE_CASES[case]
    path = tmp_path / "e.tif"
    strips = ls.write_lzw_tiff(path, frames, rows_per_strip=70, **kw)  # last strip of each frame: 10 rows
    assert all(not s.startswith(b"\x00") for page in strips for s in page)
    assert np.array_equal(decoded(path), frames)


def test_kwkwk_codes_are_exercised():
    _, _, stats = ls.lzw_codes(bytes(5000))
    assert stats["kwkwk"] > 50


@pytest.mark.parametrize("w", [1, 3, 255, 1001])
def test_odd_widths_at_16_bits(tmp_path, w):
    rng = np.random.default_rng(5)
    frames = wrapping(rng, (2, 37, w), np.uint16)
    path = tmp_path / "w.tif"
    ls.write_lzw_tiff(path, frames, rows_per_strip=5, predictor=2)
    assert np.array_equal(decoded(path), frames)


def test_k3_counting_movie_one_row_strips():
    """40 x 4092 x 5760 uint8 in one-row strips: 163 680 strips in one call."""
    import tempfile
    from pathlib import Path

    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(6)
    frames = poisson(rng, (40, 4092, 5760), 0.8)
    with tempfile.TemporaryDirectory() as d:
        path = Path(d) / "k3.tif"
        write_opencv(cv2, path, frames, 1)
        movie = tmc.read_tiff_movie(path)
        assert movie.n_strips == 40 * 4092 > 65535
        got = tmc.decode_tiff(movie, device=DEV)
    assert torch.equal(got.cpu(), torch.from_numpy(frames))


def test_super_resolution_stack_one_strip_per_frame():
    import tempfile
    from pathlib import Path

    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(7)
    frames = poisson(rng, (8, 8184, 11520), 0.2)
    with tempfile.TemporaryDirectory() as d:
        path = Path(d) / "sr.tif"
        write_opencv(cv2, path, frames, 8184)
        got = decoded(path)
    assert np.array_equal(got, frames)


def malformed_streams(frames):
    """Frame 1 strip 2: a code naming an undefined entry; frame 2 strip 0: a table overflowing without a Clear; frame 2
    strip 3: EOI before the rows are full; frame 3 strip 1: the bytes end before the rows are full."""
    raw = ls.strip_bytes(frames, 10)
    bad = {}
    v, w, _ = ls.lzw_codes(raw[1][2])
    v = list(v)
    v[40] = 258 + 45  # code 39 of the segment (after the leading Clear) names entry 303: not defined yet
    bad[(1, 2)] = ls.pack_msb(v, w)
    bad[(2, 0)] = ls.lzw_encode(raw[2][0], max_codes=3840)  # a data code at index 3839 would define entry 4096
    v, w, _ = ls.lzw_codes(raw[2][3])
    bad[(2, 3)] = ls.pack_msb(v[:len(v) // 2] + [ls.EOI], w[:len(v) // 2 + 1])
    bad[(3, 1)] = ls.lzw_encode(raw[3][1])[:-40]
    return bad


def test_malformed_strips_are_reported_and_the_rest_is_exact(tmp_path):
    rng = np.random.default_rng(8)
    frames = wrapping(rng, (5, 40, 700), np.uint8)  # incompressible: a strip overflows its table well before its end
    bad = malformed_streams(frames)
    path = tmp_path / "bad.tif"
    ls.write_lzw_tiff(path, frames, rows_per_strip=10, streams=bad)
    movie = tmc.read_tiff_movie(path)
    with pytest.raises(ValueError, match=r"frame 1 strip 2, frame 2 strip 0, frame 2 strip 3, frame 3 strip 1 "):
        tmc.decode_tiff(movie, device=DEV)
    out = torch.empty(movie.shape, dtype=torch.uint8, device=DEV)
    ws = torch.empty((prepare.tiff_workspace_bytes(movie),), dtype=torch.uint8, device=DEV)
    status = torch.empty((movie.n_strips,), dtype=torch.int32, device=DEV)
    prepare.decode_tiff_into(movie.payload.to(DEV), movie.strip_offsets.to(DEV), movie.out_offsets.to(DEV), movie, out,
                             ws, status)
    want_status = np.zeros((5, 4), np.int32)
    for f, s in bad:
        want_status[f, s] = 1
    assert np.array_equal(status.cpu().numpy().reshape(5, 4), want_status)
    got = out.cpu().numpy().reshape(5, 4, 10, 700)
    ok = want_status == 0
    assert np.array_equal(got[ok], frames.reshape(5, 4, 10, 700)[ok])


def test_calls_are_bitwise_repeatable(tmp_path):
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(9)
    frames = poisson(rng, (6, 1000, 777), 0.5, np.uint16)
    path = tmp_path / "r.tif"
    write_opencv(cv2, path, frames, 1000)
    movie = tmc.read_tiff_movie(path)
    first = tmc.decode_tiff(movie, device=DEV)
    out = torch.full_like(first, 7)
    again = tmc.decode_tiff(movie, device=DEV, out=out)
    assert again is out and torch.equal(first, again)
    assert np.array_equal(first.cpu().numpy(), frames)


def test_pipeline_matches_host_frames_and_mixes_with_eer_and_tensors(tmp_path):
    cv2 = pytest.importorskip("cv2")
    h = w = 128
    kwargs = dict(patch_sidelength=64, frequency_range=(80, 5), n_iterations=0, dose_per_frame=1.5)
    gain = 1.0 + 0.1 * torch.rand((h, w), generator=torch.Generator().manual_seed(1))
    paths, host = [], []
    for i, rps in enumerate([1, 64, 128]):
        frames = poisson(np.random.default_rng(30 + i), (12 + 2 * i, h, w), 1.0)
        paths.append(tmp_path / f"t{i}.tif")
        write_opencv(cv2, paths[-1], frames, rps)
        host.append(torch.from_numpy(frames).pin_memory())
    got = [(s.clone(), f.cpu()) for s, f in tmc.motion_correct_many(tmc.tiff_movies(paths), 1.0, device=DEV, gain=gain,
                                                                       **kwargs)]
    want = [(s.clone(), f.cpu()) for s, f in tmc.motion_correct_many(host, 1.0, device=DEV, gain=gain, **kwargs)]
    assert len(got) == 3
    for (gs, gf), (ws, wf) in zip(got, want):
        assert torch.equal(gs, ws) and torch.equal(gf, wf)

    # TIFF, EER and tensor items in one sequence, each equal to the same frames passed as uint8 host tensors
    F = 10
    ev = es.random_frames(np.random.default_rng(40), 100, h * w, 0.1)
    es.write_eer(tmp_path / "e.eer", ev, h, w)
    eer_counts = torch.from_numpy(es.reference_counts(ev, h, w, F).astype(np.uint8)).pin_memory()
    mixed = [movie_io.read_tiff_movie(paths[0]), movie_io.read_eer(tmp_path / "e.eer"), host[1],
             movie_io.read_tiff_movie(paths[2]), movie_io.read_eer(tmp_path / "e.eer")]
    plain = [host[0], eer_counts, host[1], host[2], eer_counts]
    got = [(s.clone(), f.cpu()) for s, f in tmc.motion_correct_many(mixed, 1.0, device=DEV, gain=gain,
                                                                       eer_frames_per_fraction=F, **kwargs)]
    want = [(s.clone(), f.cpu()) for s, f in tmc.motion_correct_many(plain, 1.0, device=DEV, gain=gain, **kwargs)]
    assert len(got) == 5
    for (gs, gf), (ws, wf) in zip(got, want):
        assert torch.equal(gs, ws) and torch.equal(gf, wf)


def test_pipeline_reports_a_malformed_movie(tmp_path):
    rng = np.random.default_rng(12)
    frames = wrapping(rng, (5, 128, 700), np.uint8)  # 13 strips of 10 rows (the last of 8), large enough for 64-px patches
    ls.write_lzw_tiff(tmp_path / "ok.tif", frames, rows_per_strip=10)
    ls.write_lzw_tiff(tmp_path / "bad.tif", frames, rows_per_strip=10, streams=malformed_streams(frames))
    results = tmc.motion_correct_many(tmc.tiff_movies([tmp_path / "ok.tif", tmp_path / "bad.tif"]), 1.0, device=DEV,
                                      patch_sidelength=64, frequency_range=(80, 5))
    next(results)
    with pytest.raises(ValueError, match=r"malformed LZW strip\(s\): frame 1 strip 2"):
        next(results)
