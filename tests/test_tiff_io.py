"""LZW TIFF container (``movie_io.read_tiff_movie``) without a GPU: parsing, payload and offset layout, frame slices,
the uncompressed pass-through, every rejection, and the test writer (``tests/lzw_synth.py``) pinned to libtiff."""

import numpy as np
import pytest
import torch

import eer_synth as es
import lzw_synth as ls
from torch_motion_correction_b200 import movie_io


def frames_of(dtype=np.uint8, shape=(3, 37, 53), seed=0):
    rng = np.random.default_rng(seed)
    return (rng.poisson(0.8, size=shape) * (1 if np.dtype(dtype).itemsize == 1 else 997)).astype(dtype)


def test_payload_and_offset_layout(tmp_path):
    frames = frames_of(np.uint16)
    path = tmp_path / "m.tif"
    strips = ls.write_lzw_tiff(path, frames, rows_per_strip=10, predictor=2)
    m = movie_io.read_tiff_movie(path, pinned=False)
    assert isinstance(m, movie_io.TiffMovie)
    assert (m.n_frames, m.h, m.w, m.dtype, m.predictor, m.n_strips) == (3, 37, 53, torch.uint16, 2, 12)
    flat = [s for page in strips for s in page]
    offs = m.strip_offsets.numpy()
    assert offs.dtype == np.int64 and offs[0] == 0
    assert np.array_equal(np.diff(offs), [len(s) + 8 for s in flat])
    payload = m.payload.numpy().tobytes()
    for s, o in zip(flat, offs[:-1]):
        assert payload[o:o + len(s)] == s and payload[o + len(s):o + len(s) + 8] == bytes(8)
    row = 53 * 2
    want = [(f * 37 + r) * row for f in range(3) for r in (0, 10, 20, 30)] + [3 * 37 * row]
    assert m.out_offsets.dtype == torch.int64 and m.out_offsets.tolist() == want


def test_frame_slices(tmp_path):
    frames = frames_of(shape=(6, 20, 30))
    path = tmp_path / "m.tif"
    strips = ls.write_lzw_tiff(path, frames, rows_per_strip=7)
    m = movie_io.read_tiff_movie(path, pinned=False, frames=slice(2, 5))
    assert m.n_frames == 3 and m.n_strips == 9
    assert m.out_offsets.tolist()[:4] == [0, 7 * 30, 14 * 30, 20 * 30]
    assert m.payload.numpy().tobytes()[:len(strips[2][0])] == strips[2][0]
    with pytest.raises(ValueError, match="contiguous"):
        movie_io.read_tiff_movie(path, frames=slice(0, 6, 2))


@pytest.mark.parametrize("dtype", [np.uint8, np.uint16, np.int16, np.float32])
def test_uncompressed_pages_pass_through(tmp_path, dtype):
    frames = frames_of(dtype, shape=(4, 9, 11))
    bits, fmt = {np.uint8: (8, 1), np.uint16: (16, 1), np.int16: (16, 2), np.float32: (32, 3)}[dtype]
    pages = [({256: (es.SHORT, [11]), 257: (es.SHORT, [9]), 258: (es.SHORT, [bits]), 259: (es.SHORT, [1]),
               339: (es.SHORT, [fmt])}, [f.tobytes()]) for f in frames]
    path = tmp_path / "u.tif"
    es.write_tiff(path, pages)
    got = movie_io.read_tiff_movie(path, pinned=False)
    assert isinstance(got, torch.Tensor) and got.shape == (4, 9, 11)
    assert np.array_equal(got.view(torch.int16).numpy().view(np.uint16) if dtype == np.uint16 else got.numpy(), frames)
    part = movie_io.read_tiff_movie(path, pinned=False, frames=slice(1, 3))
    assert part.shape == (2, 9, 11) and torch.equal(part, got[1:3])
    assert [type(m) for m in movie_io.tiff_movies([path], pinned=False)] == [torch.Tensor]


REJECTED_TAGS = {
    "deflate": ({259: (es.SHORT, [8])}, "compression 8"),
    "adobe_deflate": ({259: (es.SHORT, [32946])}, "compression 32946"),
    "jpeg": ({259: (es.SHORT, [7])}, "compression 7"),
    "zstd": ({259: (es.SHORT, [50000])}, "compression 50000"),
    "packbits": ({259: (es.SHORT, [32773])}, "compression 32773"),
    "predictor_3": ({317: (es.SHORT, [3])}, "Predictor 3"),
    "tiled": ({322: (es.SHORT, [16])}, "tiled"),
    "fill_order_2": ({266: (es.SHORT, [2])}, "FillOrder 2"),
    "two_samples": ({277: (es.SHORT, [2])}, "2 samples per pixel"),
}


@pytest.mark.parametrize("case", sorted(REJECTED_TAGS))
def test_rejections_name_the_page(tmp_path, case):
    tags, msg = REJECTED_TAGS[case]
    frames = frames_of()
    path = tmp_path / "x.tif"
    ls.write_lzw_tiff(path, frames[:1], tags={})
    ls_pages = []  # page 1 carries the rejected tag
    raw = ls.strip_bytes(frames, 37)
    for f in range(3):
        t = {256: (es.LONG, [53]), 257: (es.LONG, [37]), 258: (es.SHORT, [8]), 259: (es.SHORT, [5]),
             277: (es.SHORT, [1]), 278: (es.LONG, [37])}
        if f == 1:
            t.update(tags)
        ls_pages.append((t, [ls.lzw_encode(raw[f][0])]))
    es.write_tiff(path, ls_pages)
    with pytest.raises(ValueError, match=f"page 1 .*{msg}|{msg}.*page 1|page 1 is {msg}"):
        movie_io.read_tiff_movie(path)


def test_mixed_pages_are_rejected(tmp_path):
    frames = frames_of()
    raw = ls.strip_bytes(frames, 37)
    base = {256: (es.LONG, [53]), 257: (es.LONG, [37]), 258: (es.SHORT, [8]), 277: (es.SHORT, [1])}
    pages = [({**base, 259: (es.SHORT, [5])}, [ls.lzw_encode(raw[0][0])]),
             ({**base, 259: (es.SHORT, [1])}, [raw[1][0]])]
    es.write_tiff(tmp_path / "a.tif", pages)
    with pytest.raises(ValueError, match="mixed pages"):
        movie_io.read_tiff_movie(tmp_path / "a.tif")
    pages = [({**base, 259: (es.SHORT, [5]), 317: (es.SHORT, [p])}, [ls.lzw_encode(raw[0][0])]) for p in (1, 2)]
    es.write_tiff(tmp_path / "b.tif", pages)
    with pytest.raises(ValueError, match="mixed pages"):
        movie_io.read_tiff_movie(tmp_path / "b.tif")
    pages = [({**base, 259: (es.SHORT, [5]), 258: (es.SHORT, [b])}, [ls.lzw_encode(raw[0][0])]) for b in (8, 16)]
    es.write_tiff(tmp_path / "c.tif", pages)
    with pytest.raises(ValueError, match="mixed pages"):
        movie_io.read_tiff_movie(tmp_path / "c.tif")
    pages = [({**base, 259: (es.SHORT, [5]), 257: (es.LONG, [n])}, [ls.lzw_encode(raw[0][0][:n * 53])])
             for n in (37, 36)]
    es.write_tiff(tmp_path / "d.tif", pages)
    with pytest.raises(ValueError, match="different sizes"):
        movie_io.read_tiff_movie(tmp_path / "d.tif")


def test_old_style_lzw_strips_are_rejected(tmp_path):
    frames = frames_of()
    ls.write_lzw_tiff(tmp_path / "o.tif", frames, rows_per_strip=10, streams={(2, 1): b"\x00\x01\x55\xaa"})
    with pytest.raises(ValueError, match="page 2 .*old-style"):
        movie_io.read_tiff_movie(tmp_path / "o.tif")


def test_unsupported_sample_types_are_rejected(tmp_path):
    frames = frames_of()
    ls.write_lzw_tiff(tmp_path / "f.tif", frames, tags={258: (es.SHORT, [32]), 339: (es.SHORT, [3])})
    with pytest.raises(ValueError, match="LZW samples of 32 bits"):
        movie_io.read_tiff_movie(tmp_path / "f.tif")


def pillow_frames(path):
    Image = pytest.importorskip("PIL.Image")
    im = Image.open(path)
    out = []
    for i in range(im.n_frames):
        im.seek(i)
        out.append(np.array(im))
    return np.stack(out)


WRITER_CASES = {
    "default": {},
    "no_eoi": dict(eoi=False),
    "extra_clears": dict(clears_after=(1, 2, 3, 100, 101, 5000)),
    "clear_at_9_to_10": dict(max_codes=254),
    "clear_at_10_to_11": dict(max_codes=766),
    "clear_at_11_to_12": dict(max_codes=1790),
    "clear_before_9_to_10": dict(max_codes=253),
    "full_table": dict(max_codes=3839),
}


@pytest.mark.parametrize("dtype", [np.uint8, np.int8, np.uint16, np.int16])
@pytest.mark.parametrize("predictor", [1, 2])
@pytest.mark.parametrize("case", sorted(WRITER_CASES))
def test_libtiff_decodes_the_writer_s_files(tmp_path, dtype, predictor, case):
    """Pillow's libtiff reads every file the writer makes back as the source frames (signed samples compared by
    their bits: Pillow widens int16 and reads int8 as uint8).  The writer's one switch libtiff does not follow is a
    strip without a leading Clear, which libtiff rejects ("Using code not yet in table") and the decoder accepts."""
    rng = np.random.default_rng(3)
    info = np.iinfo(dtype)
    frames = rng.integers(info.min, info.max, size=(2, 150, 333), endpoint=True).astype(dtype)
    frames[0, :60] = rng.poisson(0.3, size=(60, 333)).astype(dtype)
    path = tmp_path / "w.tif"
    ls.write_lzw_tiff(path, frames, rows_per_strip=70, predictor=predictor, **WRITER_CASES[case])
    got = pillow_frames(path)
    assert np.array_equal(got.astype(dtype) if got.dtype != frames.dtype else got, frames)
    m = movie_io.read_tiff_movie(path, pinned=False)
    assert m.n_strips == 6 and m.predictor == predictor


def test_libtiff_reads_codes_past_a_full_table(tmp_path):
    """Where libtiff is more lenient than the decoder: after a segment's table holds 4096 entries it reads further
    12-bit codes without defining entries.  ``tmc_tiff_lzw_decode`` reports such a strip as malformed instead
    (DESIGN §6); this pins what libtiff does with it."""
    rng = np.random.default_rng(4)
    frames = rng.integers(0, 255, size=(1, 20, 700), endpoint=True).astype(np.uint8)
    ls.write_lzw_tiff(tmp_path / "t.tif", frames, max_codes=3840)
    assert np.array_equal(pillow_frames(tmp_path / "t.tif"), frames)


def test_writer_reaches_every_code_width_and_kwkwk():
    values, widths, stats = ls.lzw_codes(bytes(np.random.default_rng(5).integers(0, 3, 40000, dtype=np.uint8)))
    assert set(widths) == {9, 10, 11, 12} and stats["kwkwk"] > 0 and stats["max_index"] == ls.MAX_CODES - 1
    _, _, stats = ls.lzw_codes(bytes(3000))
    assert stats["kwkwk"] > 50


def test_opencv_files_parse(tmp_path):
    cv2 = pytest.importorskip("cv2")
    frames = frames_of(shape=(2, 100, 120))
    for rps, n in ((1, 200), (64, 4), (100, 2)):
        path = tmp_path / f"o{rps}.tif"
        assert cv2.imwritemulti(str(path), list(frames),
                                [cv2.IMWRITE_TIFF_COMPRESSION, 5, cv2.IMWRITE_TIFF_ROWSPERSTRIP, rps])
        m = movie_io.read_tiff_movie(path, pinned=False)
        assert (m.n_strips, m.predictor, m.dtype) == (n, 2, torch.uint8)
