"""Host-side plans for the band-limited FFT kernels: cached tables (twiddles, masks, Fourier
weights), band-box geometry, workspace chunking.  No arithmetic on image data happens here."""

from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import _lib
from ._lib import call, ptr, query, stream_ptr

_C64 = 8  # bytes per complex64
#: row -> column intermediates of one launch are capped at this many bytes.  Measured on B200 (C2 step): 48 MB 29.8 ms,
#: 96 MB (L2-sized, the first design) 28.5 ms, 192 MB 28.0 ms, 768 MB 27.4 ms, 4 GB 27.3 ms -- fewer, larger launches
#: (less tail, fewer twiddle-table loads) beat L2 residency of the intermediate
CHUNK_BYTES = 1 << 30

_twiddles: dict = {}
_masks: dict = {}
_mask_margins: dict = {}  # mask.data_ptr() -> number of all-zero columns at either side (masks live as long as the process)
_weights: dict = {}


def _dev_key(device: torch.device):
    return (device.type, device.index)


def twiddles(n: int, device: torch.device) -> torch.Tensor:
    """Per-length transform plan (twiddles; plus Bluestein chirp tables for non-power-of-two n)."""
    key = (_dev_key(device), n)
    tw = _twiddles.get(key)
    if tw is None:
        elems = query("tmc_fft_plan_elems", n)
        tw = torch.empty((elems, 2), dtype=torch.float32, device=device)
        with torch.cuda.device(device):
            call("tmc_fft_plan_init", n, ptr(tw), stream_ptr(device))
        _twiddles[key] = tw
    return tw


def soft_disc_mask(shape, radius: float, smoothing_radius: float, device: torch.device):
    """(mask (h, w) f32, ylo, yhi): ``torch_grid_utils.circle`` and a conservative row support."""
    h, w = shape
    key = (_dev_key(device), h, w, float(radius), float(smoothing_radius))
    hit = _masks.get(key)
    if hit is None:
        mask = torch.empty((h, w), dtype=torch.float32, device=device)
        ws = torch.empty((h,), dtype=torch.int32, device=device)
        with torch.cuda.device(device):
            call("tmc_soft_disc_mask", h, w, float(radius), float(smoothing_radius), ptr(mask), ptr(ws), stream_ptr(device))
        reach = int(radius + smoothing_radius) + 2
        ylo, yhi = max(0, h // 2 - reach), min(h, h // 2 + reach + 1)
        hit = (mask, ylo, yhi)
        _mask_margins[mask.data_ptr()] = max(0, min(w // 2 - reach, w - (w // 2 + reach + 1)))
        _masks[key] = hit
    return hit


def band_edges(frequency_range, pixel_spacing: float):
    """(low, high) in cycles/px exactly as the reference computes them (utils.py:99-102; fp32)."""
    cuton, cutoff_max = torch.as_tensor(frequency_range).float()
    cutoff = torch.lerp(cuton, cutoff_max, 1.0)
    low = torch.as_tensor(1 / cuton, dtype=torch.float32) * pixel_spacing
    high = torch.as_tensor(1 / cutoff, dtype=torch.float32) * pixel_spacing
    return float(low), float(high)


def _max_index_within(n: int, high: float) -> int:
    """Largest k in [0, n//2] with fl32(k * fl32(1/n)) <= high (-1 if none)."""
    k = np.arange(n // 2 + 1, dtype=np.float32) * np.float32(1.0 / n)
    ok = np.nonzero(k <= np.float32(high))[0]
    return int(ok[-1]) if len(ok) else -1


def unsupported_lengths(ny: int, nx: int, full: bool) -> str | None:
    """Why BandPlan(ny, nx, full=full) cannot be built, or None if it can (host query, no CUDA call)."""
    for n in (ny, nx):
        kind = query("tmc_fft_supported_length", n)
        if kind == 0 or (full and kind != 1):
            return (
                f"transform length {n} is not supported: the sm_100a FFT kernels take powers of two in [16, 8192], "
                f"arbitrary lengths up to 4096 and 2..8 times such a length (K3 5760 x 4092, super-resolution "
                f"11520 x 8184); full-spectrum transforms (correct_motion_fast, dose_weight) of the latter stop at "
                f"12158 (plus 12288 and 16384), the band-limited ones of the motion estimators at 32768"
            )
    return None


class BandPlan:
    """Geometry + tables of one band-limited 2-D transform size."""

    def __init__(self, ny: int, nx: int, device: torch.device, pixel_spacing: float | None = None,
                 b_factor: float | None = None, frequency_range=None, full: bool = False):
        msg = unsupported_lengths(ny, nx, full)
        if msg:
            raise NotImplementedError(msg)
        self.ny, self.nx, self.device = ny, nx, device
        self.tw_y, self.tw_x = twiddles(ny, device), twiddles(nx, device)
        if full:
            self.kx, self.ky, self.ky_start, self.weight = nx // 2 + 1, ny, 0, None
            return
        low, high = band_edges(frequency_range, pixel_spacing)
        kxm, kym = max(_max_index_within(nx, high), 0), max(_max_index_within(ny, high), 0)
        self.kx = kxm + 1
        if 2 * kym + 1 > ny:
            self.ky, self.ky_start = ny, -(ny // 2)
        else:
            self.ky, self.ky_start = 2 * kym + 1, -kym
        key = (_dev_key(device), ny, nx, float(pixel_spacing), float(b_factor), low, high)
        self.key = key
        wt = _weights.get(key)
        if wt is None:
            wt = torch.empty((self.ky, self.kx), dtype=torch.float32, device=device)
            with torch.cuda.device(device):
                call("tmc_band_weights", ny, nx, self.ky, self.kx, self.ky_start, low, high, 1, float(b_factor),
                     float(pixel_spacing), 1, ptr(wt), stream_ptr(device))
            _weights[key] = wt
        self.weight = wt

    @property
    def plane_elems(self) -> int:
        return self.ky * self.kx

    # -- forward ------------------------------------------------------------------------------
    def forward(self, image: torch.Tensor, mean_std, mask, ylo: int, yhi: int, jobs: torch.Tensor, out=None, job_mode: int = 0,
                frame_shifts: torch.Tensor | None = None):
        """jobs (njobs, 6) int32 device -> spectra (2*njobs, KY, KX) complex64 (as float pairs).

        ``frame_shifts`` (t, 2) int32 device: whole-pixel (dy, dx) added to the window origin of every frame (wrapping
        around the frame edges), see ``integer_shifts``.

        ``job_mode`` promises a structure shared by all jobs (lets the row kernel drop its generic
        loops): 1 = one frame under mask powers (1, 2); 2 = two frames (or one), power 1; 0 = generic."""
        t, h, w = image.shape
        njobs = jobs.shape[0]
        dev = image.device
        if out is None:
            out = torch.empty((2 * njobs, self.ky, self.kx, 2), dtype=torch.float32, device=dev)
        per_job = 2 * self.ny * self.kx * _C64
        chunk = max(1, min(njobs, CHUNK_BYTES // per_job))
        tmp = torch.empty((chunk * per_job // 4,), dtype=torch.float32, device=dev)
        jobs_base, out_base = jobs.data_ptr(), out.data_ptr()
        x_margin = _mask_margins.get(mask.data_ptr(), 0) if mask is not None else 0
        with torch.cuda.device(dev):
            stream = stream_ptr(dev)
            for j0 in range(0, njobs, chunk):
                n = min(chunk, njobs - j0)
                call("tmc_rfft2_band", ptr(image), t, h, w, ptr(mean_std), ptr(mask), self.ny, self.nx,
                     jobs_base + j0 * 6 * 4, n, int(job_mode), ptr(frame_shifts), x_margin, ylo, yhi, self.kx, self.ky,
                     self.ky_start, ptr(self.weight),
                     ptr(self.tw_x), ptr(self.tw_y), ptr(tmp), out_base + 2 * j0 * self.plane_elems * _C64, stream)
        return out

    def dose_filter(self, spec: torch.Tensor, jobs: torch.Tensor, total_frames: int, pixel_size: float, pre_exposure: float,
                    dose_per_frame: float, voltage: float) -> None:
        """In place: plane 2 job + {0, 1} of ``spec`` *= exposure filter of jobs[job].frame_a / frame_b."""
        njobs = jobs.shape[0]
        dev = spec.device
        tables = torch.empty((2, self.ky, self.kx), dtype=torch.float32, device=dev)
        chunk = 32000
        with torch.cuda.device(dev):
            for j0 in range(0, njobs, chunk):
                n = min(chunk, njobs - j0)
                call("tmc_dose_filter_spectra", spec.data_ptr() + 2 * j0 * self.plane_elems * _C64, jobs.data_ptr() + j0 * 6 * 4, n,
                     self.ny, self.nx, self.ky, self.kx, self.ky_start, int(total_frames), float(pixel_size), float(pre_exposure),
                     float(dose_per_frame), float(voltage), ptr(tables), stream_ptr(dev))

    # -- inverse + peak ---------------------------------------------------------------------------
    def peaks(self, prod: torch.Tensor, sub_pixel: bool, shifts=None, workspace_out: list | None = None):
        """prod (nitems, KY, KX, 2) -> (nitems, 2) px shifts (dy, dx).  ``workspace_out``: a list that receives the
        search's workspace (tmc_xc_peaks_workspace_bytes; None when the band needs none)."""
        nitems = prod.shape[0]
        dev = prod.device
        if shifts is None:
            shifts = torch.empty((nitems, 2), dtype=torch.float32, device=dev)
        per_item = self.ny * self.kx * _C64
        chunk = max(1, min(nitems, CHUNK_BYTES // per_item))
        tmp = torch.empty((chunk * per_item // 4,), dtype=torch.float32, device=dev)
        nparts = query("tmc_xc_peak_partials", self.ny, self.nx)
        partial = torch.empty((chunk * nparts * 2,), dtype=torch.float32, device=dev)
        ws_bytes = query("tmc_xc_peaks_workspace_bytes", chunk, self.ny, self.nx, self.kx)
        workspace = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev) if ws_bytes else None
        prod_base, shifts_base = prod.data_ptr(), shifts.data_ptr()
        with torch.cuda.device(dev):
            stream = stream_ptr(dev)
            for i0 in range(0, nitems, chunk):
                n = min(chunk, nitems - i0)
                call("tmc_xc_peaks", prod_base + i0 * self.plane_elems * _C64, n, self.ny, self.nx, self.kx, self.ky,
                     self.ky_start, int(sub_pixel), ptr(self.tw_x), ptr(self.tw_y), ptr(tmp), ptr(partial),
                     ptr(workspace), shifts_base + i0 * 2 * 4, stream)
        if workspace_out is not None:
            workspace_out.append(workspace)
        return shifts

    def shift_frames(self, image: torch.Tensor, mean_std, field: torch.Tensor) -> torch.Tensor:
        """Fused whole-frame Fourier shift (3 passes); ``field`` (2, t, 1, 1) px, applied as is."""
        t, h, w = image.shape
        dev = image.device
        out = torch.empty_like(image)
        per_job = 2 * self.ny * self.kx * _C64
        chunk_jobs = max(1, min((t + 1) // 2, (8 * CHUNK_BYTES) // per_job))
        tmp = torch.empty((chunk_jobs * per_job // 4,), dtype=torch.float32, device=dev)
        phase = torch.empty((2 * chunk_jobs * self.ny, 2), dtype=torch.float32, device=dev)
        flat = field.reshape(2, t)
        with torch.cuda.device(dev):
            stream = stream_ptr(dev)
            for f0 in range(0, t, 2 * chunk_jobs):
                n = min(2 * chunk_jobs, t - f0)
                jobs = frame_pair_jobs(n, dev, frame_offset=f0)
                sub = flat[:, f0 : f0 + n].contiguous()
                call("tmc_fourier_shift_frames", ptr(image), n, h, w, ptr(mean_std), ptr(jobs), jobs.shape[0], ptr(sub), 1.0,
                     ptr(self.tw_x), ptr(self.tw_y), ptr(tmp), ptr(phase), out.data_ptr() + f0 * h * w * 4, stream)
        return out

    def inverse_full(self, spec: torch.Tensor, out: torch.Tensor):
        """spec (n, ny, nx/2+1, 2) -> out (n, ny, nx) real (irfftn, backward normalisation)."""
        n = spec.shape[0]
        dev = spec.device
        per_item = self.ny * self.kx * _C64
        chunk = max(1, min(n, (4 * CHUNK_BYTES) // per_item))
        tmp = torch.empty((chunk * per_item // 4,), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            stream = stream_ptr(dev)
            for i0 in range(0, n, chunk):
                m = min(chunk, n - i0)
                call("tmc_irfft2_full", spec.data_ptr() + i0 * per_item, m, self.ny, self.nx, ptr(self.tw_x), ptr(self.tw_y),
                     ptr(tmp), out.data_ptr() + i0 * self.ny * self.nx * 4, stream)
        return out


class CropPlan:
    """Tables of one Fourier crop (h, w) -> (out_h, out_w) of whole frames (tmc_fourier_crop); the sizes have passed
    ``prepare.fourier_crop_shape``."""

    def __init__(self, h: int, w: int, out_h: int, out_w: int, device: torch.device):
        self.h, self.w, self.out_h, self.out_w, self.device = h, w, out_h, out_w, device
        self.tw = [twiddles(n, device) for n in (w, h, out_w, out_h)]

    def crop(self, image: torch.Tensor) -> torch.Tensor:
        """(t, h, w) contiguous fp32 on the plan's device -> (t, out_h, out_w).  Frames go through in chunks whose
        row -> column intermediate stays near CHUNK_BYTES."""
        t = image.shape[0]
        dev = self.device
        out = torch.empty((t, self.out_h, self.out_w), dtype=torch.float32, device=dev)
        geometry = (self.h, self.w, self.out_h, self.out_w)
        per_job = query("tmc_fourier_crop_workspace_bytes", 2, *geometry)
        chunk = 2 * max(1, min((t + 1) // 2, CHUNK_BYTES // per_job))  # frames per call
        ws = torch.empty((query("tmc_fourier_crop_workspace_bytes", min(chunk, t), *geometry),), dtype=torch.uint8, device=dev)
        in_frame, out_frame = self.h * self.w * 4, self.out_h * self.out_w * 4
        with torch.cuda.device(dev):
            stream = stream_ptr(dev)
            for f0 in range(0, t, chunk):
                n = min(chunk, t - f0)
                jobs = frame_pair_jobs(n, dev)
                call("tmc_fourier_crop", image.data_ptr() + f0 * in_frame, n, *geometry, ptr(jobs), jobs.shape[0],
                     *(ptr(tw) for tw in self.tw), ptr(ws), out.data_ptr() + f0 * out_frame, stream)
        return out


_tiles: dict = {}
_self_paired: dict = {}


def band_tiles(plan: "BandPlan") -> torch.Tensor:
    """(n_tiles, 2) int32 device tensor (ty, tx): the 8 x 16-bin tiles of the band box that hold at least one
    pass-band bin (layout of tmc_local_tile_spectra).  Cached per plan geometry."""
    key = plan.key
    hit = _tiles.get(key)
    if hit is None:
        w = plan.weight
        ky, kx = w.shape
        pad = torch.zeros((8 * ((ky + 7) // 8), 16 * ((kx + 15) // 16)), dtype=torch.float32, device=w.device)
        pad[:ky, :kx] = w
        live = pad.reshape(pad.shape[0] // 8, 8, pad.shape[1] // 16, 16).abs().amax(dim=(1, 3)) > 0
        hit = live.nonzero().to(torch.int32).contiguous()
        if hit.shape[0] == 0:
            hit = torch.zeros((1, 2), dtype=torch.int32, device=w.device)
        _tiles[key] = hit
    return hit


def self_paired_weight(plan: "BandPlan") -> bool:
    """True if the pass band weights a bin that the real-space losses ("cc", "ncc") see only through its Hermitian
    part: the Nyquist column kx = nx/2 (nx even), or the ky = -ny/2 bin of the DC column (ny even).  irfftn keeps
    only the real part of those columns after its transform along y, so a fractional shift changes what the loss sees
    there (csrc/optimizer.cu, header).  The generic loss kernels handle these bins; the tiled iteration does not.
    Cached per plan geometry."""
    key = plan.key
    hit = _self_paired.get(key)
    if hit is None:
        w = plan.weight
        live = torch.zeros((), dtype=torch.bool, device=w.device)
        if plan.nx % 2 == 0 and plan.kx == plan.nx // 2 + 1:
            live |= (w[:, -1] != 0).any()
        if plan.ny % 2 == 0 and plan.ky == plan.ny and plan.ky_start == -(plan.ny // 2):
            live |= w[0, 0] != 0
        hit = bool(live)
        _self_paired[key] = hit
    return hit


def frame_pair_jobs(t: int, device: torch.device, frame_offset: int = 0) -> torch.Tensor:
    """Whole-frame jobs packing frames (2i, 2i+1): plane index == frame index."""
    from ._common import cached_device_tensor

    def build():
        rows = []
        for i in range(0, t, 2):
            fb = i + 1 if i + 1 < t else -1
            rows.append([frame_offset + i, 1, (frame_offset + fb) if fb >= 0 else -1, 1, 0, 0])
        return torch.tensor(rows, dtype=torch.int32)

    return cached_device_tensor(("frame_pair_jobs", t, frame_offset), build, device)


def integer_shifts(field: torch.Tensor, scale: float = 1.0):
    """(2, t, 1, 1) rigid field -> ((t, 2) int32 whole-pixel window shifts, device int flag "some value is not whole")."""
    dev = field.device
    t = field.shape[1]
    flat = field.detach().to(torch.float32).reshape(2, t).contiguous()
    shifts = torch.empty((t, 2), dtype=torch.int32, device=dev)
    flag = torch.empty((1,), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        call("tmc_integer_shifts", ptr(flat), t, float(scale), ptr(shifts), ptr(flag), stream_ptr(dev))
    return shifts, flag


def pair_products(spec: torch.Tensor, ref_plane: torch.Tensor, cur_plane: torch.Tensor, plane_elems: int) -> torch.Tensor:
    n = ref_plane.shape[0]
    out = torch.empty((n, plane_elems, 2), dtype=torch.float32, device=spec.device)
    with torch.cuda.device(spec.device):
        call("tmc_xc_pair_products", ptr(spec), ptr(ref_plane), ptr(cur_plane), n, plane_elems, ptr(out),
             stream_ptr(spec.device))
    return out


def leave_one_out_products(spec: torch.Tensor, t: int, g: int, plane_elems: int, delta_offsets, deltas,
                           k_begin: int = 0, k_count: int | None = None) -> torch.Tensor:
    """Products for frames [k_begin, k_begin + k_count) given the spectra of ALL t frames."""
    k_count = t - k_begin if k_count is None else k_count
    out = torch.empty((k_count * g, plane_elems, 2), dtype=torch.float32, device=spec.device)
    with torch.cuda.device(spec.device):
        call("tmc_xc_leave_one_out_products", ptr(spec), t, g, plane_elems, ptr(delta_offsets), ptr(deltas), k_begin, k_count,
             ptr(out), stream_ptr(spec.device))
    return out
