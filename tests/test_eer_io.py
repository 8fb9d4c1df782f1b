"""EER and TIFF containers (torch_motion_correction_b200.movie_io.read_eer / read_tiff): the bit stream of a hand-built
frame, IFD parsing of classic TIFF and BigTIFF files with every entry type and strip layout, the payload layout, the
errors of damaged files.  CPU only: the events are decoded on the GPU (tests/test_gpu_eer.py)."""

import numpy as np
import pytest
import torch

import eer_synth as es
from torch_motion_correction_b200 import movie_io


def bits_to_bytes(bits: str) -> bytes:
    """'0110...' in stream order (bit i = bit i % 8 of byte i / 8), zero-filled to whole bytes."""
    bits = bits + "0" * (-len(bits) % 8)
    return bytes(int(bits[i:i + 8][::-1], 2) for i in range(0, len(bits), 8))


def field(value: int, width: int) -> str:
    """A field of `width` bits, least significant bit first."""
    return "".join(str((value >> i) & 1) for i in range(width))


def test_hand_built_frame_pins_bit_order_escape_and_termination(tmp_path):
    # 65001: 7-bit run lengths (escape 127), 2 + 2 sub-pixel bits; a 16 x 16 frame, electrons at 0, 130 and 255
    rng = np.random.default_rng(5)
    sub = np.random.default_rng(5).integers(0, 16, size=4)
    bits = (field(0, 7) + field(int(sub[0]), 4)        # electron at 0
            + field(127, 7)                             # escape: cursor 1 -> 128
            + field(2, 7) + field(int(sub[1]), 4)       # electron at 130
            + field(124, 7) + field(int(sub[2]), 4)     # electron at 255; the cursor is now 256 = h * w
            + field(0, 7))                              # terminating code: lands on 256
    want = bits_to_bytes(bits)
    assert es.encode_frame(np.array([0, 130, 255]), 256, 7, 4, rng) == want
    path = tmp_path / "hand.eer"
    es.write_eer(path, None, 16, 16, compression=65001, streams=[want, want])
    eer = movie_io.read_eer(path, pinned=False)
    assert (eer.h, eer.w, eer.rle_bits, eer.sub_bits, eer.n_frames) == (16, 16, 7, 4, 2)
    n = len(want)
    assert eer.frame_offsets.tolist() == [0, n + 8, 2 * n + 16]
    assert bytes(eer.payload.numpy()) == want + bytes(8) + want + bytes(8)


def test_escape_run_landing_on_the_end_needs_no_terminating_code():
    # 65000: escape 255; a 16 x 32 frame (512 px) with one electron at 1: after it the gap 510 = 2 escapes exactly
    rng = np.random.default_rng(0)
    sub = int(np.random.default_rng(0).integers(0, 16, size=2)[0])
    want = bits_to_bytes(field(1, 8) + field(sub, 4) + field(255, 8) + field(255, 8))
    assert es.encode_frame(np.array([1]), 512, 8, 4, rng) == want


@pytest.mark.parametrize("bigtiff", [False, True])
@pytest.mark.parametrize("n_strips", [1, 3])
@pytest.mark.parametrize("compression,codec,bits", [(65000, None, (8, 4)), (65001, None, (7, 4)),
                                                    (65002, (5, 1, 2), (5, 3))])
def test_ifd_parsing_and_payload_layout(tmp_path, bigtiff, n_strips, compression, codec, bits):
    rng = np.random.default_rng(n_strips)
    h, w = 24, 40
    frames = es.random_frames(rng, 5, h * w, 0.1)
    path = tmp_path / "m.eer"
    # one strip: the offset / count tables sit inside the entries; three: out of line (in BigTIFF two LONGs still fit)
    streams = es.write_eer(path, frames, h, w, compression=compression, codec=codec, bigtiff=bigtiff, n_strips=n_strips)
    eer = movie_io.read_eer(path, pinned=False)
    assert (eer.h, eer.w, (eer.rle_bits, eer.sub_bits), eer.n_frames) == (h, w, bits, 5)
    assert eer.payload.dtype == torch.uint8 and eer.frame_offsets.dtype == torch.int64
    want = b"".join(s + bytes(8) for s in streams)
    assert bytes(eer.payload.numpy()) == want
    assert eer.frame_offsets.tolist() == np.concatenate(([0], np.cumsum([len(s) + 8 for s in streams]))).tolist()


@pytest.mark.parametrize("bigtiff,size_type,offsets_type", [(False, es.SHORT, es.LONG), (False, es.LONG, es.SHORT),
                                                            (True, es.LONG8, es.LONG8), (True, es.SHORT, es.LONG)])
def test_short_long_and_long8_entries(tmp_path, bigtiff, size_type, offsets_type):
    frames = es.random_frames(np.random.default_rng(1), 3, 20 * 30, 0.05)
    path = tmp_path / "t.eer"
    streams = es.write_eer(path, frames, 20, 30, bigtiff=bigtiff, size_type=size_type, offsets_type=offsets_type,
                           n_strips=2)
    eer = movie_io.read_eer(path, pinned=False)
    assert (eer.h, eer.w) == (20, 30)
    assert bytes(eer.payload.numpy()) == b"".join(s + bytes(8) for s in streams)


def test_frame_slices(tmp_path):
    frames = es.random_frames(np.random.default_rng(2), 6, 16 * 16, 0.2)
    path = tmp_path / "s.eer"
    streams = es.write_eer(path, frames, 16, 16)
    for sl, want in [(slice(2, 5), streams[2:5]), (slice(None, 2), streams[:2]), (slice(4, None), streams[4:]),
                     (slice(-2, None), streams[-2:]), (slice(5, 3), [])]:
        eer = movie_io.read_eer(path, pinned=False, frames=sl)
        assert eer.n_frames == len(want)
        assert bytes(eer.payload.numpy()) == b"".join(s + bytes(8) for s in want)
    with pytest.raises(ValueError, match="contiguous"):
        movie_io.read_eer(path, pinned=False, frames=slice(0, 6, 2))
    with pytest.raises(ValueError, match="contiguous"):
        movie_io.read_eer(path, pinned=False, frames=[0, 1])


def test_eer_movies_yields_each_file(tmp_path):
    paths = []
    for i in range(2):
        paths.append(tmp_path / f"{i}.eer")
        es.write_eer(paths[-1], es.random_frames(np.random.default_rng(i), 2 + i, 64, 0.1), 8, 8)
    assert [m.n_frames for m in movie_io.eer_movies(paths, pinned=False)] == [2, 3]


def small_movie(tmp_path, **kw):
    path = tmp_path / "e.eer"
    es.write_eer(path, es.random_frames(np.random.default_rng(3), 3, 12 * 12, 0.1), 12, 12, **kw)
    return path


def test_big_endian_is_rejected(tmp_path):
    path = small_movie(tmp_path)
    raw = bytearray(path.read_bytes())
    raw[0:4] = b"MM\x00\x2a"
    path.write_bytes(bytes(raw))
    with pytest.raises(ValueError, match="big-endian"):
        movie_io.read_eer(path)


def test_unknown_compression_is_rejected(tmp_path):
    with pytest.raises(ValueError, match="compression 5"):
        movie_io.read_eer(small_movie(tmp_path, compression=5))


def test_mixed_frame_sizes_are_rejected(tmp_path):
    path = tmp_path / "mixed.eer"
    es.write_eer(path, es.random_frames(np.random.default_rng(0), 3, 144, 0.1), 12, 12,
                 sizes=[(12, 12), (12, 12), (12, 13)])
    with pytest.raises(ValueError, match="different sizes"):
        movie_io.read_eer(path)


def test_strips_beyond_the_end_of_the_file_are_rejected(tmp_path):
    path = small_movie(tmp_path)
    raw = path.read_bytes()
    path.write_bytes(raw[:-3])  # the strips come after the IFDs: this cuts the last frame's strip
    with pytest.raises(ValueError, match="beyond the end of the file"):
        movie_io.read_eer(path)


def test_truncated_files_are_rejected(tmp_path):
    path = small_movie(tmp_path, n_strips=3)
    raw = path.read_bytes()
    for keep in (4, 12, 40):  # inside the header, inside the first IFD, inside a later IFD or its strip tables
        path.write_bytes(raw[:keep])
        with pytest.raises(ValueError, match="truncated|not a TIFF"):
            movie_io.read_eer(path)


def test_a_file_without_eer_tags_is_not_an_eer_movie(tmp_path):
    path = tmp_path / "plain.tif"
    es.write_tiff(path, [({256: (es.SHORT, [4]), 257: (es.SHORT, [2]), 259: (es.SHORT, [1])}, [bytes(8)])])
    with pytest.raises(ValueError, match="compression 1"):
        movie_io.read_eer(path)


def tiff_pages(stack: np.ndarray, bits: int, fmt: int, n_strips: int):
    pages = []
    for plane in stack:
        raw = np.ascontiguousarray(plane.astype(plane.dtype.newbyteorder("<"))).tobytes()
        tags = {256: (es.SHORT, [plane.shape[1]]), 257: (es.SHORT, [plane.shape[0]]), 258: (es.SHORT, [bits]),
                259: (es.SHORT, [1]), 277: (es.SHORT, [1]), 339: (es.SHORT, [fmt])}
        pages.append((tags, es.split_stream(raw, n_strips)))
    return pages


@pytest.mark.parametrize("dtype,bits,fmt", [(np.uint8, 8, 1), (np.uint16, 16, 1), (np.int16, 16, 2),
                                            (np.float32, 32, 3)])
@pytest.mark.parametrize("pages,bigtiff", [(1, False), (3, False), (2, True)])
def test_read_tiff_round_trips(tmp_path, dtype, bits, fmt, pages, bigtiff):
    rng = np.random.default_rng(bits + pages)
    stack = (rng.normal(size=(pages, 7, 9)) * 1000).astype(dtype)
    path = tmp_path / "g.tif"
    es.write_tiff(path, tiff_pages(stack, bits, fmt, n_strips=2), bigtiff=bigtiff)
    got = movie_io.read_tiff(path, pinned=False)
    want = stack[0] if pages == 1 else stack
    assert tuple(got.shape) == want.shape
    arr = got.view(torch.int16).numpy().view(np.uint16) if got.dtype == torch.uint16 else got.numpy()
    assert arr.dtype == np.dtype(dtype) and np.array_equal(arr, want)


def test_read_tiff_rejects_compressed_and_short_pages(tmp_path):
    path = tmp_path / "lzw.tif"
    pages = tiff_pages(np.zeros((1, 4, 4), np.uint8), 8, 1, 1)
    pages[0][0][259] = (es.SHORT, [5])
    es.write_tiff(path, pages)
    with pytest.raises(ValueError, match="compression 5"):
        movie_io.read_tiff(path)
    pages = tiff_pages(np.zeros((1, 4, 4), np.uint8), 8, 1, 1)
    es.write_tiff(path, [(pages[0][0], [bytes(15)])])
    with pytest.raises(ValueError, match="holds 15 bytes"):
        movie_io.read_tiff(path)
