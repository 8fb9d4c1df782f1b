"""TIFF LZW movie WRITER for the tests and the timing tool, built from the format rules (TIFF 6.0 §13), not from the decoder.

Codes are packed MSB-first.  Inside a segment (the codes after a Clear, 256, or from the start of the strip) code k is 9
bits for k < 254, 10 for k < 766, 11 for k < 1790 and 12 after that ("early change"); a Clear is written when a segment
holds ``max_codes`` data codes, before the table could pass 4096 entries.  Switches produce the cases a decoder must
tolerate or reject: no leading Clear, no EOI, extra Clears after chosen data codes, and segments of any length (so that
a Clear falls exactly on a width boundary).  The container is ``eer_synth.write_tiff``'s little-endian TIFF."""

from __future__ import annotations

import numpy as np

from eer_synth import LONG, SHORT, write_tiff

CLEAR, EOI = 256, 257
#: data codes per segment before the writer's Clear: code 3836 defines entry 4094 in the decoder, as libtiff's tables end
MAX_CODES = 3837


def code_width(k: int) -> int:
    return 9 if k < 254 else 10 if k < 766 else 11 if k < 1790 else 12


def pack_msb(values, widths) -> bytes:
    """Codes (value, width <= 12 bits) one after the other, MSB-first, into bytes (the last one zero-filled)."""
    v = np.asarray(values, dtype=np.uint32)
    wd = np.asarray(widths, dtype=np.int64)
    if v.size == 0:
        return b""
    bits = ((v[:, None] >> np.arange(11, -1, -1, dtype=np.uint32)) & 1).astype(np.uint8)
    keep = np.arange(12)[None, :] >= (12 - wd)[:, None]
    return np.packbits(bits[keep]).tobytes()


def lzw_codes(data: bytes, leading_clear: bool = True, eoi: bool = True, clears_after=(), max_codes: int = MAX_CODES):
    """``(values, widths, stats)`` of the LZW stream of ``data``.  ``clears_after``: data-code counts (over the whole
    stream) after which an extra Clear is written.  ``stats``: ``kwkwk`` (codes naming the entry the decoder is about
    to define), ``segments``, ``max_index`` (largest data-code index inside a segment)."""
    values, widths = [], []
    stats = {"kwkwk": 0, "segments": 1, "max_index": 0}
    k = 0
    table, nxt = {}, 258
    extra = set(clears_after)

    def put(c):
        nonlocal k
        values.append(c)
        widths.append(code_width(k))
        k += 1

    def clear():
        nonlocal k, table, nxt
        put(CLEAR)
        k, table, nxt = 0, {}, 258
        stats["segments"] += 1

    if leading_clear:
        put(CLEAR)
        k = 0
    n_data = 0
    if data:
        w = data[0]
        for b in data[1:]:
            hit = table.get((w << 8) | b)
            if hit is not None:
                w = hit
                continue
            if w == nxt - 1 and w >= 258:
                stats["kwkwk"] += 1
            stats["max_index"] = max(stats["max_index"], k)
            put(w)
            n_data += 1
            if nxt < 4096:
                table[(w << 8) | b] = nxt
                nxt += 1
            w = b
            if k >= max_codes or n_data in extra:
                clear()
        if w == nxt - 1 and w >= 258:
            stats["kwkwk"] += 1
        stats["max_index"] = max(stats["max_index"], k)
        put(w)
    if eoi:
        put(EOI)
    return values, widths, stats


def lzw_encode(data: bytes, **kw) -> bytes:
    values, widths, _ = lzw_codes(data, **kw)
    return pack_msb(values, widths)


def difference_rows(frames: np.ndarray) -> np.ndarray:
    """Predictor 2: every sample minus its left neighbour, modulo 2^bits (the first sample of a row kept)."""
    u = frames.view(np.uint8 if frames.dtype.itemsize == 1 else np.uint16)
    d = u.copy()
    d[..., 1:] = u[..., 1:] - u[..., :-1]
    return d


_FORMATS = {np.dtype(np.uint8): (8, 1), np.dtype(np.int8): (8, 2), np.dtype(np.uint16): (16, 1),
            np.dtype(np.int16): (16, 2)}


def strip_bytes(frames: np.ndarray, rows_per_strip: int, predictor: int = 1):
    """Per frame, the raw little-endian bytes of each strip (after differencing for Predictor 2)."""
    src = difference_rows(frames) if predictor == 2 else frames
    src = np.ascontiguousarray(src.astype(src.dtype.newbyteorder("<"), copy=False))
    n, h, _ = src.shape
    return [[src[f, r:r + rows_per_strip].tobytes() for r in range(0, h, rows_per_strip)] for f in range(n)]


def write_lzw_tiff(path, frames: np.ndarray, rows_per_strip: int | None = None, predictor: int = 1,
                   bigtiff: bool = False, streams=None, tags=None, **encode):
    """Write the (n, h, w) ``frames`` (uint8 / int8 / uint16 / int16) as an LZW TIFF, one page per frame.
    ``encode``: ``lzw_codes`` switches for every strip; ``streams``: {(frame, strip): bytes} written instead of the
    encoded strip; ``tags``: extra or replaced tags {tag: (type, values)}.  Returns the encoded strips per frame."""
    frames = np.asarray(frames)
    n, h, w = frames.shape
    rps = rows_per_strip or h
    bits, fmt = _FORMATS[frames.dtype]
    raw = strip_bytes(frames, rps, predictor)
    encoded = [[lzw_encode(s, **encode) for s in page] for page in raw]
    pages = []
    for f, page in enumerate(encoded):
        strips = [streams.get((f, i), s) if streams else s for i, s in enumerate(page)]
        t = {256: (LONG, [w]), 257: (LONG, [h]), 258: (SHORT, [bits]), 259: (SHORT, [5]), 262: (SHORT, [1]),
             277: (SHORT, [1]), 278: (LONG, [rps]), 317: (SHORT, [predictor]), 339: (SHORT, [fmt])}
        t.update(tags or {})
        pages.append((t, strips))
    write_tiff(path, pages, bigtiff=bigtiff)
    return encoded
