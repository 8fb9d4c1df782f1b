"""EER movie WRITER for the tests and the timing tool, built from the format rules (DESIGN §4), not from the decoder.

A frame is a list of electron pixel indices p = row * w + col (at most one per pixel).  Its stream: for each electron in
ascending order, the gap from the cursor as escapes (2^rle_bits - 1, rle_bits bits each) while the gap is at least that,
then the remainder (rle_bits bits) and sub_bits random sub-pixel bits; the cursor moves to p + 1.  After the last electron
the gap to h * w is written the same way, without sub-pixel bits, and ends the frame (no further code when escapes
alone land on h * w).  Codes are packed LSB-first (bit i is bit i % 8 of byte i / 8); the last byte is zero-filled.

The container is a little-endian TIFF or BigTIFF with one IFD per frame; a frame's stream may be cut into several strips
at any byte, including inside a code.  Everything is vectorised with numpy so that full-size movies can be built."""

from __future__ import annotations

import numpy as np

SHORT, LONG, LONG8 = 3, 4, 16
_TYPE_BYTES = {SHORT: 2, LONG: 4, LONG8: 8}
CODECS = {65000: (8, 2, 2), 65001: (7, 2, 2)}  # compression -> (rle_bits, horizontal bits, vertical bits)


def pack_codes(values, widths) -> bytes:
    """Codes (value, width <= 32 bits) one after the other, LSB-first, into bytes (the last one zero-filled)."""
    values = np.asarray(values, dtype=np.uint64)
    widths = np.asarray(widths, dtype=np.int64)
    if values.size == 0:
        return b""
    starts = np.zeros(values.size, dtype=np.int64)
    np.cumsum(widths[:-1], out=starts[1:])
    total = int(starts[-1] + widths[-1])
    words = np.zeros((total + 63) // 64 + 1, dtype=np.uint64)
    idx = starts >> 6
    shift = (starts & 63).astype(np.uint64)
    lo = values << shift  # wraps: the bits above 64 go to the next word
    hi = np.where(shift > 0, values >> (np.uint64(64) - np.where(shift > 0, shift, np.uint64(1))), np.uint64(0))
    first = np.flatnonzero(np.r_[True, idx[1:] != idx[:-1]])
    words[idx[first]] += np.add.reduceat(lo, first)  # codes never share a bit: adding is OR-ing
    words[idx[first] + 1] += np.add.reduceat(hi, first)
    return words.astype("<u8").tobytes()[:(total + 7) // 8]


def frame_codes(positions, npix: int, rle_bits: int, sub_bits: int, rng):
    """(values, widths) of one frame's codes; ``positions`` sorted, unique, in [0, npix)."""
    pos = np.asarray(positions, dtype=np.int64)
    esc = (1 << rle_bits) - 1
    cursor = np.concatenate(([0], pos + 1))  # where each gap starts; the last one runs to npix
    gaps = np.concatenate((pos - cursor[:-1], [npix - cursor[-1]]))
    n_esc = gaps // esc
    rem = gaps % esc
    last = gaps.size - 1
    # the terminating gap needs its remainder code unless the escapes alone land on npix
    has_rem = np.ones(gaps.size, dtype=bool)
    has_rem[last] = rem[last] > 0 or n_esc[last] == 0
    sub = rng.integers(0, 1 << sub_bits, size=gaps.size, dtype=np.int64) if sub_bits else np.zeros(gaps.size, np.int64)
    rem_values = rem | (sub << rle_bits)
    rem_widths = np.full(gaps.size, rle_bits + sub_bits, dtype=np.int64)
    rem_values[last], rem_widths[last] = rem[last], rle_bits
    # per gap: n_esc escapes, then its remainder code
    per_gap = n_esc + has_rem
    order_start = np.zeros(gaps.size, dtype=np.int64)
    np.cumsum(per_gap[:-1], out=order_start[1:])
    n_codes = int(per_gap.sum())
    values = np.full(n_codes, esc, dtype=np.int64)
    widths = np.full(n_codes, rle_bits, dtype=np.int64)
    at = (order_start + n_esc)[has_rem]
    values[at] = rem_values[has_rem]
    widths[at] = rem_widths[has_rem]
    return values, widths


def encode_frame(positions, npix: int, rle_bits: int, sub_bits: int, rng) -> bytes:
    values, widths = frame_codes(positions, npix, rle_bits, sub_bits, rng)
    return pack_codes(values, widths)


def random_frames(rng, n_frames: int, npix: int, rate: float):
    """Electron positions of ``n_frames`` frames, each pixel hit with probability ``rate`` (geometric gaps)."""
    out = []
    for _ in range(n_frames):
        n = int(npix * rate * 1.2 + 64)
        p = np.cumsum(rng.geometric(rate, size=n)) - 1
        while p[-1] < npix:
            p = np.concatenate((p, p[-1] + np.cumsum(rng.geometric(rate, size=n))))
        out.append(p[p < npix])
    return out


def reference_counts(frames, h: int, w: int, frames_per_fraction: int) -> np.ndarray:
    """np.add.at counts (n_frames // F, h, w) of the electron lists; trailing frames dropped."""
    n = len(frames) // frames_per_fraction
    out = np.zeros((n, h * w), dtype=np.int64)
    for f in range(n * frames_per_fraction):
        np.add.at(out[f // frames_per_fraction], np.asarray(frames[f], dtype=np.int64), 1)
    return out.reshape(n, h, w)


def write_tiff(path, pages, bigtiff: bool = False, offsets_type: int | None = None) -> None:
    """Little-endian TIFF / BigTIFF with one IFD per page.  ``pages``: list of (tags, strips): ``tags`` a dict
    tag -> (type, values) (SHORT / LONG / LONG8), ``strips`` a list of bytes.  StripOffsets and StripByteCounts are
    added with ``offsets_type`` (default LONG, LONG8 for BigTIFF); the IFDs come first, the strips after them, so a cut
    file loses strip bytes before IFD bytes."""
    offsets_type = offsets_type or (LONG8 if bigtiff else LONG)
    head_bytes, count_bytes, entry_bytes, inline = (16, 8, 20, 8) if bigtiff else (8, 2, 12, 4)
    # sizes of each IFD (entries + next pointer) and its out-of-line values
    layouts = []
    for tags, strips in pages:
        entries = dict(tags)
        entries[273] = (offsets_type, [0] * len(strips))
        entries[279] = (offsets_type, [len(s) for s in strips])
        entries = sorted(entries.items())
        extra = sum(len(v) * _TYPE_BYTES[t] for _, (t, v) in entries if len(v) * _TYPE_BYTES[t] > inline)
        layouts.append((entries, count_bytes + len(entries) * entry_bytes + (8 if bigtiff else 4), extra))
    data_at = head_bytes + sum(a + b for _, a, b in layouts)
    data_at += data_at % 2
    out = bytearray()
    out += b"II" + ((43).to_bytes(2, "little") + (8).to_bytes(2, "little") + bytes(2) if bigtiff else (42).to_bytes(2, "little"))
    ifd_at = head_bytes
    out += ifd_at.to_bytes(8 if bigtiff else 4, "little")
    data = bytearray()
    for i, ((tags, strips), (entries, ifd_size, extra)) in enumerate(zip(pages, layouts)):
        offs = []
        for s in strips:
            offs.append(data_at + len(data))
            data += s
        entries = [(t, (ty, offs if t == 273 else v)) for t, (ty, v) in entries]
        extra_at = ifd_at + ifd_size
        table = bytearray(len(entries).to_bytes(count_bytes, "little"))
        blob = bytearray()
        for tag, (ty, vals) in entries:
            raw = b"".join(int(v).to_bytes(_TYPE_BYTES[ty], "little") for v in vals)
            table += tag.to_bytes(2, "little") + ty.to_bytes(2, "little") + len(vals).to_bytes(8 if bigtiff else 4, "little")
            if len(raw) <= inline:
                table += raw + bytes(inline - len(raw))
            else:
                table += (extra_at + len(blob)).to_bytes(inline, "little")
                blob += raw
        nxt = ifd_at + ifd_size + extra if i + 1 < len(pages) else 0
        table += nxt.to_bytes(8 if bigtiff else 4, "little")
        out += table + blob
        ifd_at = nxt
    out += bytes(data_at - len(out))
    out += data
    with open(path, "wb") as f:
        f.write(out)


def split_stream(stream: bytes, n_strips: int):
    """A frame's stream in ``n_strips`` nearly equal pieces, cut at arbitrary bytes (inside codes)."""
    cuts = np.linspace(0, len(stream), n_strips + 1).astype(int)
    return [stream[a:b] for a, b in zip(cuts[:-1], cuts[1:])]


def write_eer(path, frames, h: int, w: int, compression: int = 65001, codec=None, bigtiff: bool = False,
              n_strips: int = 1, size_type: int = SHORT, offsets_type: int | None = None, seed: int = 0, streams=None,
              sizes=None):
    """Write an EER movie of the electron lists ``frames`` (or ready ``streams``).  ``codec`` (rle, horz, vert) with
    compression 65002; ``sizes``: per-frame (h, w) written to the IFDs instead of (h, w).  Returns the streams."""
    if compression == 65002:
        rle, horz, vert = codec
    else:
        rle, horz, vert = CODECS.get(compression, (7, 2, 2))
    rng = np.random.default_rng(seed)
    if streams is None:
        streams = [encode_frame(p, h * w, rle, horz + vert, rng) for p in frames]
    pages = []
    for i, s in enumerate(streams):
        fh, fw = sizes[i] if sizes is not None else (h, w)
        rows_type = LONG if size_type == SHORT and max(fh, fw) > 65535 else size_type
        tags = {256: (rows_type, [fw]), 257: (rows_type, [fh]), 259: (SHORT, [compression]),
                278: (rows_type, [fh]), 262: (SHORT, [0]), 258: (SHORT, [1]), 277: (SHORT, [1])}
        if compression == 65002:
            tags.update({65007: (SHORT, [rle]), 65008: (SHORT, [horz]), 65009: (SHORT, [vert])})
        pages.append((tags, split_stream(s, n_strips)))
    write_tiff(path, pages, bigtiff=bigtiff, offsets_type=offsets_type)
    return streams
