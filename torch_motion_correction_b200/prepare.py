"""Movie preparation ahead of the estimators (additive API): detector-native pixel types -> fp32, gain multiply,
hot-pixel replacement, per-frame mean removal -- the NumPy pre-processing of the reference's example workflow
(``examples/ttMotion.py:90-202``: ``gain_correct``, ``remove_hot_pixels``, ``set_frames_mean_zero``, and the cast to
float32 at ``:357``) as CUDA kernels behind the C ABI (``csrc/prepare.cu``)."""

from __future__ import annotations

import torch

from ._common import resolve_device
from ._lib import call, ptr, query, stream_ptr

DTYPE_CODES = {torch.uint8: 0, torch.uint16: 1, torch.int16: 2, torch.float16: 3, torch.float32: 4, torch.int8: 5}


def oriented_gain(gain: torch.Tensor, flip_gain: int = 0, rot_gain: int = 0) -> torch.Tensor:
    """The gain map as ``gain_correct`` orients it (examples/ttMotion.py:115-123): flip (1 = flipY, 2 = flipX), then
    ``np.rot90(k=-rot_gain)``."""
    if flip_gain == 1:
        gain = torch.flip(gain, dims=(0,))
    elif flip_gain == 2:
        gain = torch.flip(gain, dims=(1,))
    if rot_gain != 0:
        gain = torch.rot90(gain, k=-int(rot_gain), dims=(0, 1))
    return gain.contiguous()


def prepare_movie(movie: torch.Tensor, gain: torch.Tensor | None = None, hot_pixel_threshold: float | None = None,
                  zero_frame_means: bool = False, device=None, out: torch.Tensor | None = None,
                  max_hot_pixels: int = 1 << 20, return_hot_pixel_count: bool = False):
    """(t, h, w) movie of dtype uint8 / int8 / uint16 / int16 / float16 / float32 -> fp32 device tensor.

    ``gain`` (h, w): multiplied in (``gain_correct``); ``hot_pixel_threshold``: pixels further than that many standard
    deviations from their frame's mean are replaced by a neighbour (``remove_hot_pixels``; the reference picks the
    neighbour with ``np.random.choice``, here a hash of the pixel position picks it, reproducibly); ``zero_frame_means``:
    every frame minus its own mean (``set_frames_mean_zero``).  Same order as the example's ``main``.  One pass over the
    stack converts, applies the gain and accumulates the per-frame moments the other two steps need."""
    if movie.ndim != 3:
        raise ValueError(f"movie must be (t, h, w), got {tuple(movie.shape)}")
    if movie.dtype not in DTYPE_CODES:
        raise TypeError(f"unsupported movie dtype {movie.dtype}: expected one of {sorted(str(d) for d in DTYPE_CODES)}")
    dev = resolve_device(movie, device)
    src = movie.detach().to(dev).contiguous()
    t, h, w = src.shape
    n = h * w
    if out is None:
        out = torch.empty((t, h, w), dtype=torch.float32, device=dev)
    elif out.shape != src.shape or out.dtype != torch.float32 or not out.is_contiguous():
        raise ValueError("out must be a contiguous float32 tensor of the movie's shape")
    gain_dev = None
    if gain is not None:
        if tuple(gain.shape) != (h, w):
            raise ValueError(f"gain must be ({h}, {w}), got {tuple(gain.shape)}")
        gain_dev = gain.detach().to(device=dev, dtype=torch.float32).contiguous()
    need_moments = hot_pixel_threshold is not None or zero_frame_means
    moments = torch.empty((t, 2), dtype=torch.float64, device=dev) if need_moments else None
    count = None
    with torch.cuda.device(dev):
        stream = stream_ptr(dev)
        call("tmc_convert_stack", ptr(src), DTYPE_CODES[movie.dtype], t, n, ptr(gain_dev), ptr(out), ptr(moments), stream)
        if hot_pixel_threshold is not None:
            ws = torch.empty((query("tmc_hot_pixel_workspace_bytes", int(max_hot_pixels)),), dtype=torch.uint8, device=dev)
            count = torch.zeros((1,), dtype=torch.int32, device=dev)
            call("tmc_remove_hot_pixels", ptr(out), t, h, w, ptr(moments), float(hot_pixel_threshold), int(max_hot_pixels), ptr(ws),
                 ptr(count), stream)
        if zero_frame_means:
            call("tmc_subtract_frame_means", ptr(out), t, n, ptr(moments), stream)
    if return_hot_pixel_count:
        return out, count
    return out


def eer_fractions(eer, frames_per_fraction) -> tuple[int, torch.dtype]:
    """``(n_fractions, counts dtype)`` of rendering ``eer`` in fractions of ``frames_per_fraction`` hardware frames:
    ``n_frames // F`` fractions of uint8 counts for F <= 255, uint16 for F <= 65535 (a frame holds at most one electron
    per pixel, so a fraction's count never exceeds F).  ``ValueError`` for fewer than 2 fractions or a bad F."""
    import numbers

    if isinstance(frames_per_fraction, bool) or not isinstance(frames_per_fraction, numbers.Integral) or not (
            1 <= frames_per_fraction <= 65535):
        raise ValueError(f"frames_per_fraction must be an integer in 1 .. 65535, got {frames_per_fraction!r}")
    n = eer.n_frames // int(frames_per_fraction)
    if n < 2:
        raise ValueError(f"{eer.n_frames} EER frames in fractions of {frames_per_fraction} give {n} fraction(s), need >= 2")
    return n, torch.uint8 if frames_per_fraction <= 255 else torch.uint16


def eer_counts_buffer(shape, dtype, device) -> torch.Tensor:
    """A counts tensor of ``shape`` whose storage is padded to a whole number of 4-byte words, as the render kernel's
    word-wide increments need."""
    n = shape[0] * shape[1] * shape[2]
    words = (n * (1 if dtype == torch.uint8 else 2) + 3) // 4
    return torch.empty((words,), dtype=torch.int32, device=device).view(dtype)[:n].view(shape)


def render_eer_into(payload, frame_offsets, eer, frames_per_fraction, counts, status) -> None:
    """Enqueue the render of the first ``counts.shape[0] * F`` frames (device ``payload`` / ``frame_offsets`` laid out as
    ``eer``'s) into ``counts`` on the current stream; ``status`` (int32, one per rendered frame) gets 0 for a decoded
    frame, 1 for a malformed one.  No synchronisation."""
    n_frames = counts.shape[0] * frames_per_fraction
    call("tmc_eer_render", ptr(payload), int(payload.numel()), ptr(frame_offsets), n_frames, eer.h, eer.w, eer.rle_bits,
         eer.sub_bits, frames_per_fraction, counts.element_size(), ptr(counts), ptr(status), stream_ptr(counts.device))


def check_eer_status(status_host: torch.Tensor, first_frame: int = 0) -> None:
    """Raise ``ValueError`` naming the frames a render reported as malformed."""
    bad = torch.nonzero(status_host).flatten().tolist()
    if bad:
        shown = ", ".join(str(first_frame + i) for i in bad[:20]) + (", ..." if len(bad) > 20 else "")
        raise ValueError(f"malformed EER frame(s) {shown}: the bit stream runs out or moves past the frame's last pixel")


def render_eer(eer, frames_per_fraction: int, device=None, out: torch.Tensor | None = None) -> torch.Tensor:
    """EER movie (``read_eer``) -> electron counts (n_frames // F, h, w) on the device, F = ``frames_per_fraction``:
    fraction k holds the electrons of hardware frames [k F, (k + 1) F).  uint8 for F <= 255, uint16 otherwise.

    The trailing n_frames % F frames are DROPPED, as RELION's EER grouping does (``group_frames`` instead folds leftovers
    into its last group): the fractions are the movie's frames for everything downstream, the exposure filter included,
    so they must all carry the same dose.  Raises ``ValueError`` for fewer than 2 fractions.

    Only the compressed payload crosses PCIe; the events are decoded on the device (``tmc_eer_render``).  A malformed
    frame (its stream runs out, or moves past the last pixel, before it ends) contributes nothing and makes this raise
    ``ValueError`` naming it: that check reads the per-frame status back, one host synchronisation per call.  The counts
    go on through ``prepare_movie`` (gain, hot pixels, frame means -> fp32) like any other integer movie.
    ``out``: a contiguous tensor of that shape and dtype whose size is a multiple of 4 bytes, reused instead of a new one."""
    n, dtype = eer_fractions(eer, frames_per_fraction)
    dev = resolve_device(eer.payload, device if device is not None else "cuda")  # the payload is a host tensor
    shape = (n, eer.h, eer.w)
    if out is None:
        out = eer_counts_buffer(shape, dtype, dev)
    elif tuple(out.shape) != shape or out.dtype != dtype or not out.is_contiguous() or out.device != dev or (
            out.numel() * out.element_size()) % 4:
        raise ValueError(f"out must be a contiguous {dtype} tensor of shape {shape} on {dev} with a size that is a "
                         "multiple of 4 bytes")
    used = n * frames_per_fraction
    with torch.cuda.device(dev):
        payload = eer.payload[:int(eer.frame_offsets[used])].to(dev, non_blocking=True)
        offsets = eer.frame_offsets[:used + 1].to(dev, non_blocking=True)
        status = torch.empty((used,), dtype=torch.int32, device=dev)
        render_eer_into(payload, offsets, eer, frames_per_fraction, out, status)
        check_eer_status(status.cpu())
    return out


def group_frames(movie: torch.Tensor, frame_group: int, device=None) -> torch.Tensor:
    """(t, h, w) movie -> (t // frame_group, h, w) fp32 sums of ``frame_group`` consecutive frames, the last group also
    taking the ``t % frame_group`` leftover frames (``frame_groups.frame_groups`` has the rule).  Each sum adds the frames
    in ascending order, one fp32 rounding per add.  ``frame_group == 1`` returns ``movie`` itself.

    These are the frames ``estimate_motion(..., frame_group=...)`` estimates on: summing a few low-dose frames gives the
    cross-correlation peaks a usable signal."""
    from ._common import as_f32
    from ._ops import group_frames as _group_frames
    from .frame_groups import frame_groups

    if movie.ndim != 3:
        raise ValueError(f"movie must be (t, h, w), got {tuple(movie.shape)}")
    groups = frame_groups(movie.shape[0], frame_group)
    if groups.group_size == 1:
        return movie
    return _group_frames(as_f32(movie, resolve_device(movie, device)), groups.group_size)


def fourier_crop_shape(shape, factor) -> tuple[int, int]:
    """(h, w) -> (h', w') = (h / factor, w / factor), the frame size ``fourier_crop`` returns; the one place its argument
    rules live.  Raised before any CUDA call:

    * ``ValueError`` unless ``factor`` is a real number >= 1; for ``factor == 1`` the result is (h, w) and nothing else is
      checked;
    * ``ValueError`` unless h and w are even and h / factor, w / factor are whole numbers (to 1e-6 relative) that are even
      too: factor 2 takes 11520 x 8184 to 5760 x 4092, factor 1.5 takes 5760 x 4092 to 3840 x 2728;
    * ``NotImplementedError`` unless all four sides are lengths of the full-spectrum transforms
      (``_fourier.unsupported_lengths``)."""
    import math
    import numbers

    from ._fourier import unsupported_lengths

    h, w = (int(n) for n in shape)
    if isinstance(factor, bool) or not isinstance(factor, numbers.Real) or not math.isfinite(factor) or factor < 1:
        raise ValueError(f"factor must be a real number >= 1, got {factor!r}")
    if factor == 1:
        return h, w
    if h % 2 or w % 2:
        raise ValueError(f"Fourier cropping needs even frame sides, got ({h}, {w})")
    out = []
    for n in (h, w):
        exact = n / float(factor)
        m = round(exact)
        if m < 2 or m % 2 or abs(exact - m) > 1e-6 * exact:
            raise ValueError(f"factor {factor} takes side {n} to {exact:g}, which is not an even whole number")
        out.append(m)
    for ny, nx in ((h, w), tuple(out)):
        msg = unsupported_lengths(ny, nx, full=True)
        if msg:
            raise NotImplementedError(msg)
    return out[0], out[1]


def fourier_crop(image: torch.Tensor, factor, device=None) -> torch.Tensor:
    """Fourier crop ("binning", MotionCor2 ``-FtBin``): (h, w) or (t, h, w) -> (h', w') or (t, h', w') fp32 with
    (h', w') = ``fourier_crop_shape((h, w), factor)``.  ``factor == 1`` returns ``image`` itself.

    Per frame: rfft2, keep the box ky in [-h'/2, h'/2), kx in [0, w'/2], irfft2 at (h', w'), times h' w' / (h w) so the
    mean pixel value is kept.  The box's columns kx = 0 and kx = w'/2 enter through their Hermitian part, as in
    numpy's and torch's irfft2.  Output pixel (i, j) is the band-limited image sampled at input position
    (factor i, factor j): the field of view is unchanged and the pixel spacing becomes ``factor`` times the input's.

    Deformation fields are in Angstrom on normalised coordinates, so a field estimated on the cropped movie also
    describes the original one.  Normalised y maps to input row y factor (h' - 1) instead of y (h - 1), which is at most
    factor - 1 input pixels apart at the far edge (the same for x).  To estimate on the binned movie but correct at full
    resolution and crop afterwards, compose: ``fourier_crop(correct_motion_sums(movie, field, px)["sum"], 2)``."""
    from ._common import as_f32
    from ._fourier import CropPlan

    if image.ndim not in (2, 3) or (image.ndim == 3 and image.shape[0] == 0):
        raise ValueError(f"image must be (h, w) or (t, h, w) with t >= 1, got {tuple(image.shape)}")
    h, w = image.shape[-2:]
    out_h, out_w = fourier_crop_shape((h, w), factor)
    if factor == 1:
        return image
    dev = resolve_device(image, device)
    stack = as_f32(image, dev)
    out = CropPlan(h, w, out_h, out_w, dev).crop(stack if image.ndim == 3 else stack[None])
    return out if image.ndim == 3 else out[0]
