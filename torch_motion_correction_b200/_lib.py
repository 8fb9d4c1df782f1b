"""ctypes binding of the C-ABI CUDA library ``libtmc_b200.so`` (declared in ``include/tmc_b200.h``).

There is NO CPU fallback: if the library is missing or no CUDA device is present every
entry point raises.  PyTorch is used for device memory and streams only.
"""

from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_double, c_float, c_int, c_long, c_void_p

import torch

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
# TMC_B200_LIB: an alternative build of the same library (A/B experiments: tools/build_variant.sh)
LIB_PATH = os.environ.get("TMC_B200_LIB") or os.path.join(_PKG_DIR, "libtmc_b200.so")

_lib = None

P = c_void_p
I = c_int
L = c_long
F = c_float
D = c_double

# name -> (restype, argtypes); the trailing stream argument is always a cudaStream_t
_SIGNATURES = {
    "tmc_version": (I, []),
    "tmc_last_error": (c_char_p, []),
    "tmc_sm_count": (I, []),
    "tmc_launch_count": (L, []),
    "tmc_kernel_timing": (I, [I]),
    "tmc_kernel_timing_report": (L, [ctypes.c_char_p, L]),
    "tmc_upload_pinned": (I, [P, P, L, P]),
    "tmc_stack_stats_workspace_doubles": (I, []),
    "tmc_stack_stats": (I, [P, I, I, I, I, I, I, I, P, P, P]),
    "tmc_stack_moments": (I, [P, I, I, I, I, I, I, I, P, P, P]),
    "tmc_moments_to_mean_std": (I, [P, P, P]),
    "tmc_convert_stack": (I, [P, I, I, L, P, P, P, P]),
    "tmc_hot_pixel_workspace_bytes": (L, [I]),
    "tmc_remove_hot_pixels": (I, [P, I, I, I, P, F, I, P, P, P]),
    "tmc_subtract_frame_means": (I, [P, I, L, P, P]),
    "tmc_group_frames": (I, [P, I, I, I, I, P, P]),
    "tmc_eer_render": (I, [P, L, P, I, I, I, I, I, I, I, P, P, P]),
    "tmc_spline_workspace_floats": (L, [I, I, I, I]),
    "tmc_spline_eval": (I, [P, I, I, I, I, I, P, L, P, P, P]),
    "tmc_spline_eval_backward": (I, [I, I, I, I, I, P, L, P, F, P, P, P]),
    "tmc_spline_lattice": (I, [P, I, I, I, I, I, P, I, I, I, I, I, I, I, I, I, P, P, P]),
    "tmc_spline_lattice_times": (I, [P, I, I, I, I, I, P, I, I, I, I, I, P, I, I, P, P, P]),
    "tmc_warp_workspace_floats": (L, [I, I, I]),
    "tmc_warp_lattice": (I, [P, I, I, I, P, I, I, F, P, P, P, I, P, P]),
    "tmc_warp_lattice_sums": (I, [P, I, I, I, P, I, I, F, P, I, P, P, P]),
    "tmc_pixel_shifts": (I, [P, I, I, I, I, F, P, P]),
    "tmc_warp_lattice_backward": (I, [P, I, I, I, P, I, I, F, P, P, P, P]),
    "tmc_lattice_tyx": (I, [I, I, I, I, I, P, P]),
    "tmc_warp_dense_shifts": (I, [P, I, I, I, P, P, P]),
    "tmc_pixel_tyx": (I, [I, I, I, I, I, P, P]),
    "tmc_fft_supported_length": (I, [I]),
    "tmc_fft_plan_elems": (L, [I]),
    "tmc_fft_plan_init": (I, [I, P, P]),
    "tmc_fft_c2c_rows": (I, [P, I, I, P, P, P]),
    "tmc_rfft2_band": (I, [P, I, I, I, P, P, I, I, P, I, I, P, I, I, I, I, I, I, P, P, P, P, P, P]),
    "tmc_integer_shifts": (I, [P, I, F, P, P, P]),
    "tmc_xc_pair_products": (I, [P, P, P, I, L, P, P]),
    "tmc_xc_leave_one_out_products": (I, [P, I, I, L, P, P, I, I, P, P]),
    "tmc_xc_peak_partials": (I, [I, I]),
    "tmc_xc_peaks": (I, [P, I, I, I, I, I, I, I, P, P, P, P, P, P]),
    "tmc_irfft2_full": (I, [P, I, I, I, P, P, P, P, P]),
    "tmc_fourier_crop_workspace_bytes": (L, [I, I, I, I, I]),
    "tmc_fourier_crop": (I, [P, I, I, I, I, I, P, I, P, P, P, P, P, P, P]),
    "tmc_fourier_shift": (I, [P, I, I, I, P, F, P]),
    "tmc_fourier_shift_frames_supported": (I, [I, I]),
    "tmc_fourier_shift_frames": (I, [P, I, I, I, P, P, I, P, F, P, P, P, P, P, P]),
    "tmc_soft_disc_mask": (I, [I, I, F, F, P, P, P]),
    "tmc_band_weights": (I, [I, I, I, I, I, F, F, I, F, F, I, P, P]),
    "tmc_dose_filter_spectra": (I, [P, P, I, I, I, I, I, I, I, F, F, F, F, P, P]),
    "tmc_dose_weighted_sum": (I, [P, I, I, I, F, F, F, F, I, P, P, I, P]),
    "tmc_dose_lowrank_combine": (I, [P, I, I, I, F, F, P, I, F, P, I, P, P]),
    "tmc_xc_postprocess": (I, [P, I, I, F, I, I, F, I, I, I, P, P, P]),
    "tmc_global_shifts_to_field": (I, [P, I, F, I, P, P]),
    "tmc_subtract_mean": (I, [P, L, P]),
    "tmc_local_spectra_norms": (I, [P, I, I, I, I, I, I, I, I, I, P, P]),
    "tmc_local_loss_workspace_bytes": (L, [I, I, I, I]),
    "tmc_local_loss_grad": (I, [P, P, P, P, P, P, I, I, I, I, I, I, I, I, F, I, P, P, P, P]),
    "tmc_advance_counter": (I, [P, P]),
    "tmc_adam_step": (I, [P, P, P, P, I, D, D, D, D, D, P, P]),
    "tmc_local_steps_supported": (I, [I, I, I, I]),
    "tmc_local_tile_spectra": (I, [P, I, I, I, I, I, P, I, I, P, P]),
    "tmc_local_steps_workspace_bytes": (L, [I, I, I]),
    "tmc_local_steps": (I, [P, P, I, I, I, I, I, I, I, I, P, P, P, P, I, I, P, F, I, P, P, P, D, D, D, D, D, I, I, I, P, P,
                            P, P]),
}


def exported_symbols():
    return sorted(_SIGNATURES)


def register(name, restype, argtypes):
    _SIGNATURES[name] = (restype, argtypes)


def load() -> ctypes.CDLL:
    """Load the library (once).  Raises RuntimeError when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `python -m torch_motion_correction_b200._build`). torch_motion_correction_b200 has no CPU fallback."
        )
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in _SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the header and the library drift apart
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib


def require_cuda() -> None:
    if not torch.cuda.is_available():
        raise RuntimeError(
            "torch_motion_correction_b200 needs a CUDA device (sm_100a); there is no CPU fallback. "
            "Use the reference package (or this repo's oracle/) for CPU execution."
        )


def stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    return t.data_ptr()


#: optional per-entry-point device timing (bench.py): name -> list of (start_event, end_event)
TIMING: dict | None = None
#: number of C-ABI compute calls issued (bench.py reports kernels launched through them)
CALLS: dict = {}
#: kernels launched by CUDA-graph replays of captured library calls (not visible to tmc_launch_count)
GRAPH_LAUNCHES = 0


def call(name: str, *args):
    """Call an ``int``-returning entry point; non-zero status raises with ``tmc_last_error()``."""
    lib = load()
    CALLS[name] = CALLS.get(name, 0) + 1
    if TIMING is not None and not torch.cuda.is_current_stream_capturing():
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()  # current stream of the current device == the stream passed to the call
        status = getattr(lib, name)(*args)
        end.record()
        TIMING.setdefault(name, []).append((start, end))
    else:
        status = getattr(lib, name)(*args)
    if status != 0:
        msg = lib.tmc_last_error().decode("utf-8", "replace")
        if status == 1:
            raise ValueError(f"{name}: {msg}")
        if status == 3:
            raise NotImplementedError(f"{name}: {msg}")
        raise RuntimeError(f"{name} failed (status {status}): {msg}")


def kernel_timing(enable: bool) -> None:
    """Switch the library's per-kernel CUDA-event timing on (dropping earlier records) or off (bench.py)."""
    load().tmc_kernel_timing(1 if enable else 0)


def kernel_timing_report() -> dict:
    """{kernel: (launches, total device ms)} of the launches recorded since ``kernel_timing(True)``."""
    lib = load()
    need = lib.tmc_kernel_timing_report(None, 0)
    buf = ctypes.create_string_buffer(int(need) + 16)
    lib.tmc_kernel_timing_report(buf, len(buf))
    out = {}
    for line in buf.value.decode().splitlines():
        name, n, ms = line.rsplit(",", 2)
        out[name] = (int(n), float(ms))
    return out


def query(name: str, *args):
    """Call a value-returning query entry point."""
    return getattr(load(), name)(*args)
