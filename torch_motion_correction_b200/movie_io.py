"""Movie files either side of the hot path: MRC2014 stacks and EER electron-event movies in, aligned sums out.

The reference's example script reads movies with third-party readers (``mrcfile``, ``eerfile``, ``tifffile``:
``examples/ttMotion.py:1-4,40-62,357``), none of which ship with the package.  This module covers

* MRC2014 (CCP-EM, Cheng et al. 2015: a 1024-byte header, an optional extended header, raw voxels, x fastest), handed over
  in the FILE data type: int8 / uint8 / int16 / uint16 / float16 movies cross PCIe at 1-2 bytes per pixel and are
  converted on the device (``tmc_convert_stack`` behind ``motion_correct_many`` / ``prepare_movie``);
* EER (Falcon 4 / 4i electron-event lists in a little-endian TIFF or BigTIFF, one IFD per hardware frame, compression
  65000 / 65001 / 65002): ``read_eer`` only reads the compressed strips into one pinned buffer; the events are rendered
  into count fractions on the device (``prepare.render_eer``, ``csrc/eer.cu``), so only the compressed bytes cross PCIe;
* uncompressed TIFF images and stacks (``read_tiff``): Falcon gain references.

Compressed TIFF (LZW, deflate), 8K rendering from the EER sub-pixel bits and the EER XML metadata stay out of scope.

PARITY UNPINNED against ``mrcfile`` and against a real Falcon EER file (neither is available here): the MRC layout is
the published one and is pinned by ``tests/test_movie_io.py`` on hand-built headers; the EER container and bit stream
follow the published EER description and RELION's open-source decoder as restated in DESIGN §4, and are pinned by
``tests/test_eer_io.py`` and ``tests/test_gpu_eer.py`` on files written from those rules (``tests/eer_synth.py``)."""

from __future__ import annotations

import os
from pathlib import Path
from typing import Iterable, Iterator, Union

import numpy as np
import torch

_HEADER_BYTES = 1024
#: MRC mode -> numpy dtype of the voxels (little-endian files; byte-swapped when the machine stamp says big-endian)
_MODE_DTYPES = {0: np.int8, 1: np.int16, 2: np.float32, 6: np.uint16, 12: np.float16}
_DTYPE_MODES = {np.dtype(np.int8): 0, np.dtype(np.int16): 1, np.dtype(np.float32): 2, np.dtype(np.uint16): 6,
                np.dtype(np.float16): 12}


class MrcHeader:
    """The fields of the 1024-byte MRC2014 header this package uses."""

    def __init__(self, nx: int, ny: int, nz: int, mode: int, cella=(0.0, 0.0, 0.0), mx: int = 0, my: int = 0, mz: int = 0,
                 nsymbt: int = 0, big_endian: bool = False, unsigned_bytes: bool = False):
        self.nx, self.ny, self.nz, self.mode = nx, ny, nz, mode
        self.cella = tuple(float(v) for v in cella)
        self.mx, self.my, self.mz = mx or nx, my or ny, mz or nz
        self.nsymbt = nsymbt
        self.big_endian = big_endian
        self.unsigned_bytes = unsigned_bytes

    @property
    def pixel_spacing(self) -> float:
        """Angstrom per pixel along x (cell length / grid sampling), 0 if the file does not say."""
        return self.cella[0] / self.mx if self.mx and self.cella[0] > 0 else 0.0

    @property
    def dtype(self) -> np.dtype:
        if self.mode not in _MODE_DTYPES:
            raise ValueError(f"MRC mode {self.mode} is not a real-valued image type this package reads "
                             f"(supported: {sorted(_MODE_DTYPES)})")
        dt = np.dtype(np.uint8 if (self.mode == 0 and self.unsigned_bytes) else _MODE_DTYPES[self.mode])
        return dt.newbyteorder(">") if self.big_endian and dt.itemsize > 1 else dt

    @property
    def data_offset(self) -> int:
        return _HEADER_BYTES + self.nsymbt


def read_mrc_header(path: Union[str, Path]) -> MrcHeader:
    """Parse the fixed header: words 1-4 nx ny nz mode, 8-10 mx my mz, 11-13 cell lengths, 24 nsymbt, bytes 208-211 'MAP ',
    212-215 machine stamp (0x44 little endian, 0x11 big endian).  Mode 0 is signed unless the IMOD flag (bytes 152-159:
    stamp 1146047817, bit 0 of the flags word) says unsigned."""
    with open(path, "rb") as f:
        raw = f.read(_HEADER_BYTES)
    if len(raw) < _HEADER_BYTES:
        raise ValueError(f"{path}: shorter than an MRC header")
    stamp = raw[212]
    big = stamp == 0x11
    order = ">" if big else "<"
    i4 = np.frombuffer(raw, dtype=np.dtype(order + "i4"), count=56)
    f4 = np.frombuffer(raw, dtype=np.dtype(order + "f4"), count=56)
    nx, ny, nz, mode = (int(v) for v in i4[:4])
    if raw[208:211] != b"MAP" and not (0 < nx < 1 << 20 and 0 < ny < 1 << 20 and 0 < nz < 1 << 20 and 0 <= mode <= 101):
        raise ValueError(f"{path}: not an MRC file")
    imod_unsigned = int(i4[38]) == 1146047817 and not (int(i4[39]) & 1)  # IMOD: bit 0 set = signed bytes
    return MrcHeader(nx, ny, nz, mode, cella=f4[10:13], mx=int(i4[7]), my=int(i4[8]), mz=int(i4[9]), nsymbt=max(int(i4[23]), 0),
                     big_endian=big, unsigned_bytes=imod_unsigned)


def read_mrc(path: Union[str, Path], pinned: bool = True, frames: slice | None = None):
    """``(movie, header)``: the (nz, ny, nx) stack as a HOST tensor in the file's data type (int8 / uint8 / int16 / uint16 /
    float16 / float32), page-locked by default so that ``motion_correct_many`` can copy it asynchronously.

    The voxels are read straight into the (pinned) destination buffer; big-endian files are byte-swapped on the way."""
    hdr = read_mrc_header(path)
    dt = hdr.dtype
    first, last, step = (frames or slice(None)).indices(hdr.nz)
    if step != 1:
        raise ValueError("read_mrc: frames must be a contiguous slice")
    n = max(last - first, 0)
    plane = hdr.ny * hdr.nx
    need = hdr.data_offset + (first + n) * plane * dt.itemsize
    if os.path.getsize(path) < need:
        raise ValueError(f"{path}: truncated ({os.path.getsize(path)} bytes, header promises {need})")
    native = dt.newbyteorder("=")
    torch_dtype = {np.dtype(np.int8): torch.int8, np.dtype(np.uint8): torch.uint8, np.dtype(np.int16): torch.int16,
                   np.dtype(np.uint16): torch.uint16, np.dtype(np.float16): torch.float16,
                   np.dtype(np.float32): torch.float32}[native]
    out = torch.empty((n, hdr.ny, hdr.nx), dtype=torch_dtype, pin_memory=bool(pinned and torch.cuda.is_available()))
    view = out.numpy() if torch_dtype != torch.uint16 else out.view(torch.int16).numpy().view(np.uint16)
    with open(path, "rb") as f:
        f.seek(hdr.data_offset + first * plane * dt.itemsize)
        got = f.readinto(memoryview(view.reshape(-1)).cast("B"))
    if got != n * plane * dt.itemsize:
        raise ValueError(f"{path}: short read")
    if dt.byteorder == ">":
        view.byteswap(inplace=True)
    return out, hdr


def write_mrc(path: Union[str, Path], data, pixel_spacing: float = 0.0, overwrite: bool = True) -> None:
    """Write a (ny, nx) image or (nz, ny, nx) stack (tensor or array; int8 / int16 / uint16 / float16 / float32; anything
    else is stored as float32) as a little-endian MRC2014 file with density statistics and the cell set from
    ``pixel_spacing`` (Angstrom per pixel)."""
    arr = data.detach().cpu() if isinstance(data, torch.Tensor) else data
    if isinstance(arr, torch.Tensor):
        arr = arr.view(torch.int16).numpy().view(np.uint16) if arr.dtype == torch.uint16 else arr.numpy()
    arr = np.asarray(arr)
    if arr.ndim == 2:
        arr = arr[None]
    if arr.ndim != 3:
        raise ValueError(f"write_mrc: expected a (ny, nx) image or (nz, ny, nx) stack, got shape {arr.shape}")
    if arr.dtype not in _DTYPE_MODES:
        arr = arr.astype(np.float32)
    arr = np.ascontiguousarray(arr.astype(arr.dtype.newbyteorder("<"), copy=False))
    nz, ny, nx = arr.shape
    if not overwrite and os.path.exists(path):
        raise FileExistsError(path)
    head = np.zeros(256, dtype="<i4")
    fview = head.view("<f4")
    head[0:3] = (nx, ny, nz)
    head[3] = _DTYPE_MODES[arr.dtype.newbyteorder("=")]
    head[7:10] = (nx, ny, nz)
    fview[10:13] = (nx * pixel_spacing, ny * pixel_spacing, nz * pixel_spacing)
    fview[13:16] = 90.0
    head[16:19] = (1, 2, 3)
    stats = arr.astype(np.float64) if arr.size else np.zeros(1)
    fview[19:22] = (stats.min(), stats.max(), stats.mean())
    fview[54] = stats.std()
    head[22] = 1 if nz == 1 else 0  # space group: 1 = volume-like single image, 0 = image stack
    head[27] = 20140  # NVERSION
    raw = bytearray(head.tobytes())
    raw[208:212] = b"MAP "
    raw[212:216] = bytes([0x44, 0x44, 0x00, 0x00])
    Path(path).parent.mkdir(parents=True, exist_ok=True)
    with open(path, "wb") as f:
        f.write(raw)
        f.write(memoryview(arr.reshape(-1)).cast("B"))


def mrc_movies(paths: Iterable[Union[str, Path]], pinned: bool = True) -> Iterator[torch.Tensor]:
    """The movies of ``paths`` one after the other as pinned host tensors in their file data type: the input
    ``motion_correct_many`` pipelines (disk read of movie i+1 overlaps the device work on movie i through its prefetch)."""
    for p in paths:
        yield read_mrc(p, pinned=pinned)[0]


# ---- TIFF container (EER movies, gain references) ---------------------------------------------------------------

_TIFF_TYPE_SIZES = {1: 1, 3: 2, 4: 4, 16: 8}  # BYTE, SHORT, LONG, LONG8: the integer types of the tags read here
_TAG_WIDTH, _TAG_LENGTH, _TAG_BITS, _TAG_COMPRESSION = 256, 257, 258, 259
_TAG_STRIP_OFFSETS, _TAG_SAMPLES, _TAG_ROWS_PER_STRIP, _TAG_STRIP_COUNTS, _TAG_SAMPLE_FORMAT = 273, 277, 278, 279, 339
_TAG_EER_RLE, _TAG_EER_HORZ, _TAG_EER_VERT = 65007, 65008, 65009
#: EER compression -> (rle_bits, sub_bits) of the fixed codecs; 65002 reads them from tags 65007-65009
_EER_CODECS = {65000: (8, 4), 65001: (7, 4)}
_MAX_IFDS = 1 << 20


def _tiff_ifds(path, wanted) -> list:
    """Walk the IFD chain of a little-endian TIFF / BigTIFF: one ``{tag: tuple of ints}`` per IFD holding the tags of
    ``wanted`` that are present.  Values of up to 4 (classic) / 8 (BigTIFF) bytes sit in the entry, longer ones at the
    offset it holds.  Raises ``ValueError`` for big-endian or damaged files."""
    size = os.path.getsize(path)
    with open(path, "rb") as f:
        head = f.read(16)
        if head[:2] == b"MM":
            raise ValueError(f"{path}: big-endian TIFF is not supported")
        if head[:2] != b"II" or len(head) < 8:
            raise ValueError(f"{path}: not a TIFF file")
        magic = int.from_bytes(head[2:4], "little")
        if magic == 42:
            big, first = False, int.from_bytes(head[4:8], "little")
        elif magic == 43 and len(head) >= 16 and int.from_bytes(head[4:6], "little") == 8:
            big, first = True, int.from_bytes(head[8:16], "little")
        else:
            raise ValueError(f"{path}: not a TIFF or BigTIFF file (magic {magic})")
        count_bytes, entry_bytes, inline = (8, 20, 8) if big else (2, 12, 4)

        def read_at(offset, n):
            if offset < 0 or offset + n > size:
                raise ValueError(f"{path}: truncated (needs bytes {offset}..{offset + n}, file has {size})")
            f.seek(offset)
            return f.read(n)

        ifds, seen, offset = [], set(), first
        while offset:
            if offset in seen or len(ifds) >= _MAX_IFDS:
                raise ValueError(f"{path}: the IFD chain loops")
            seen.add(offset)
            n = int.from_bytes(read_at(offset, count_bytes), "little")
            table = read_at(offset + count_bytes, n * entry_bytes + (8 if big else 4))  # entries + next-IFD offset
            tags = {}
            for i in range(n):
                e = table[i * entry_bytes:(i + 1) * entry_bytes]
                tag, typ = int.from_bytes(e[0:2], "little"), int.from_bytes(e[2:4], "little")
                if tag not in wanted:
                    continue
                if typ not in _TIFF_TYPE_SIZES:
                    raise ValueError(f"{path}: tag {tag} has TIFF type {typ}, expected BYTE, SHORT, LONG or LONG8")
                cnt = int.from_bytes(e[4:12] if big else e[4:8], "little")
                field = e[12:20] if big else e[8:12]
                nbytes = cnt * _TIFF_TYPE_SIZES[typ]
                raw = field[:nbytes] if nbytes <= inline else read_at(int.from_bytes(field, "little"), nbytes)
                dt = np.dtype({1: "<u1", 3: "<u2", 4: "<u4", 16: "<u8"}[typ])
                tags[tag] = tuple(int(v) for v in np.frombuffer(raw, dtype=dt, count=cnt))
            ifds.append(tags)
            nxt = table[n * entry_bytes:n * entry_bytes + (8 if big else 4)]
            offset = int.from_bytes(nxt, "little")
    if not ifds:
        raise ValueError(f"{path}: no image in the TIFF file")
    return ifds


def _tag(path, ifd, index, tag):
    if tag not in ifd or not ifd[tag]:
        raise ValueError(f"{path}: IFD {index} lacks TIFF tag {tag}")
    return ifd[tag]


def _strips(path, ifds, size):
    """[(offset, byte count) per strip] of every IFD, checked to lie inside the file."""
    out = []
    for i, ifd in enumerate(ifds):
        offsets, counts = _tag(path, ifd, i, _TAG_STRIP_OFFSETS), _tag(path, ifd, i, _TAG_STRIP_COUNTS)
        if len(offsets) != len(counts):
            raise ValueError(f"{path}: IFD {i} has {len(offsets)} strip offsets but {len(counts)} strip byte counts")
        for o, c in zip(offsets, counts):
            if o + c > size:
                raise ValueError(f"{path}: strip of IFD {i} at {o} + {c} bytes lies beyond the end of the file ({size})")
        out.append(list(zip(offsets, counts)))
    return out


def _frame_size(path, ifds):
    sizes = {(_tag(path, d, i, _TAG_LENGTH)[0], _tag(path, d, i, _TAG_WIDTH)[0]) for i, d in enumerate(ifds)}
    if len(sizes) != 1:
        raise ValueError(f"{path}: frames of different sizes {sorted(sizes)}")
    h, w = sizes.pop()
    if h < 1 or w < 1:
        raise ValueError(f"{path}: empty frames ({h} x {w})")
    return h, w


def _contiguous(frames, n, who):
    if not isinstance(frames, (slice, type(None))):
        raise ValueError(f"{who}: frames must be a contiguous slice")
    first, last, step = (frames or slice(None)).indices(n)
    if step != 1:
        raise ValueError(f"{who}: frames must be a contiguous slice")
    return first, max(last, first)


class EerMovie:
    """An EER movie read by ``read_eer``: the compressed bit streams of its frames, ready for ``render_eer`` /
    ``motion_correct_many``.

    ``payload`` (uint8 host tensor, pinned by default) holds frame f's stream at bytes
    ``[frame_offsets[f], frame_offsets[f + 1] - 8)``, followed by 8 zero bytes; ``frame_offsets`` (int64, n_frames + 1).
    ``h``, ``w``: frame size in pixels; ``rle_bits``, ``sub_bits``: the codec's run-length and sub-pixel bit widths."""

    def __init__(self, payload: torch.Tensor, frame_offsets: torch.Tensor, h: int, w: int, rle_bits: int, sub_bits: int):
        self.payload, self.frame_offsets = payload, frame_offsets
        self.h, self.w, self.rle_bits, self.sub_bits = int(h), int(w), int(rle_bits), int(sub_bits)

    @property
    def n_frames(self) -> int:
        return int(self.frame_offsets.shape[0]) - 1

    def __repr__(self):
        return (f"EerMovie({self.n_frames} frames of {self.h} x {self.w}, rle_bits={self.rle_bits}, "
                f"sub_bits={self.sub_bits}, {int(self.payload.numel())} payload bytes)")


def read_eer(path: Union[str, Path], pinned: bool = True, frames: slice | None = None) -> EerMovie:
    """The frames of an EER movie (``frames``: a contiguous slice of them, as in ``read_mrc``) as an ``EerMovie``.

    Walks and checks the IFD chain (one IFD per hardware frame: equal frame sizes, one EER compression, strips inside the
    file) and reads the selected frames' strips, concatenated in order, into one page-locked buffer, each frame padded
    with 8 zero bytes.  Nothing is decoded here."""
    wanted = {_TAG_WIDTH, _TAG_LENGTH, _TAG_COMPRESSION, _TAG_STRIP_OFFSETS, _TAG_ROWS_PER_STRIP, _TAG_STRIP_COUNTS,
              _TAG_EER_RLE, _TAG_EER_HORZ, _TAG_EER_VERT}
    ifds = _tiff_ifds(path, wanted)
    h, w = _frame_size(path, ifds)
    codecs = set()
    for i, d in enumerate(ifds):
        comp = _tag(path, d, i, _TAG_COMPRESSION)[0]
        if comp in _EER_CODECS:
            codecs.add(_EER_CODECS[comp])
        elif comp == 65002:
            rle, horz, vert = (_tag(path, d, i, t)[0] for t in (_TAG_EER_RLE, _TAG_EER_HORZ, _TAG_EER_VERT))
            codecs.add((rle, horz + vert))
        else:
            raise ValueError(f"{path}: IFD {i} has compression {comp}, not an EER codec (65000, 65001, 65002)")
    if len(codecs) != 1:
        raise ValueError(f"{path}: frames with different EER codecs {sorted(codecs)}")
    rle_bits, sub_bits = codecs.pop()
    if not (1 <= rle_bits <= 16 and 0 <= sub_bits and rle_bits + sub_bits <= 32):
        raise ValueError(f"{path}: EER codec with {rle_bits} run-length and {sub_bits} sub-pixel bits is not supported")
    first, last = _contiguous(frames, len(ifds), "read_eer")
    strips = _strips(path, ifds[first:last], os.path.getsize(path))
    lengths = np.array([sum(c for _, c in s) for s in strips], dtype=np.int64)
    offsets = np.zeros(len(strips) + 1, dtype=np.int64)
    np.cumsum(lengths + 8, out=offsets[1:])
    pin = bool(pinned and torch.cuda.is_available())
    payload = torch.empty((int(offsets[-1]),), dtype=torch.uint8, pin_memory=pin)
    view = memoryview(payload.numpy())
    with open(path, "rb") as f:
        for frame, (start, frame_strips) in enumerate(zip(offsets[:-1], strips)):
            pos = int(start)
            for o, c in frame_strips:
                f.seek(o)
                if f.readinto(view[pos:pos + c]) != c:
                    raise ValueError(f"{path}: short read in frame {first + frame}")
                pos += c
            view[pos:pos + 8] = bytes(8)
    table = torch.from_numpy(offsets)
    return EerMovie(payload, table.pin_memory() if pin else table, h, w, rle_bits, sub_bits)


def eer_movies(paths: Iterable[Union[str, Path]], pinned: bool = True) -> Iterator[EerMovie]:
    """The EER movies of ``paths`` one after the other (``read_eer``): the EER counterpart of ``mrc_movies`` for
    ``motion_correct_many(..., eer_frames_per_fraction=F)``."""
    for p in paths:
        yield read_eer(p, pinned=pinned)


_TIFF_SAMPLE_TYPES = {(8, 1): torch.uint8, (16, 1): torch.uint16, (16, 2): torch.int16, (32, 3): torch.float32}


def read_tiff(path: Union[str, Path], pinned: bool = True) -> torch.Tensor:
    """An uncompressed (compression 1) little-endian TIFF / BigTIFF image as a (h, w) host tensor, or a stack of
    equal-sized pages as (n, h, w): uint8, uint16, int16 or float32 samples (BitsPerSample / SampleFormat), one sample per
    pixel.  For Falcon gain references, passed on as ``gain=``."""
    wanted = {_TAG_WIDTH, _TAG_LENGTH, _TAG_BITS, _TAG_COMPRESSION, _TAG_STRIP_OFFSETS, _TAG_SAMPLES, _TAG_STRIP_COUNTS,
              _TAG_SAMPLE_FORMAT}
    ifds = _tiff_ifds(path, wanted)
    h, w = _frame_size(path, ifds)
    kinds = set()
    for i, d in enumerate(ifds):
        comp = d.get(_TAG_COMPRESSION, (1,))[0]
        if comp != 1:
            raise ValueError(f"{path}: page {i} has compression {comp}; only uncompressed TIFF is read")
        if d.get(_TAG_SAMPLES, (1,))[0] != 1:
            raise ValueError(f"{path}: page {i} has {d[_TAG_SAMPLES][0]} samples per pixel, expected 1")
        kinds.add((d.get(_TAG_BITS, (1,))[0], d.get(_TAG_SAMPLE_FORMAT, (1,))[0]))
    if len(kinds) != 1 or next(iter(kinds)) not in _TIFF_SAMPLE_TYPES:
        raise ValueError(f"{path}: sample types {sorted(kinds)} (bits, format); supported: uint8, uint16, int16, float32")
    dtype = _TIFF_SAMPLE_TYPES[kinds.pop()]
    strips = _strips(path, ifds, os.path.getsize(path))
    out = torch.empty((len(ifds), h, w), dtype=dtype, pin_memory=bool(pinned and torch.cuda.is_available()))
    raw = memoryview((out.view(torch.int16) if dtype == torch.uint16 else out).numpy().reshape(-1)).cast("B")
    plane = h * w * out.element_size()
    with open(path, "rb") as f:
        for i, page in enumerate(strips):
            pos = i * plane
            for o, c in page:
                if pos + c > (i + 1) * plane:
                    raise ValueError(f"{path}: page {i} holds more than {h} x {w} samples")
                f.seek(o)
                if f.readinto(raw[pos:pos + c]) != c:
                    raise ValueError(f"{path}: short read in page {i}")
                pos += c
            if pos != (i + 1) * plane:
                raise ValueError(f"{path}: page {i} holds {pos - i * plane} bytes, expected {plane}")
    return out[0] if len(ifds) == 1 else out
