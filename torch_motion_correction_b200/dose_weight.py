"""Dose weighting of an aligned movie (additive API; the reference only does this in its example script,
``examples/ttMotion.py:331-351``, through ``torch_fourier_filter.dose_weight.dose_weight_movie``)."""

from __future__ import annotations

import functools
from dataclasses import dataclass

import numpy as np
import torch

from . import _fourier
from ._common import as_f32, resolve_device
from ._lib import call, ptr, stream_ptr

#: frames transformed per block: bounds the (frames, ny, nx/2+1) complex64 spectra held at once
_BLOCK_BYTES = 4 << 30


def dose_weight(
    movie: torch.Tensor,
    pixel_size: float,
    pre_exposure: float = 0.0,
    dose_per_frame: float = 1.0,
    voltage: float = 300.0,
    device: torch.device = None,
) -> torch.Tensor:
    """``sum_t irfft2(rfft2(frame_t) * q_t / sqrt(sum_t q_t^2))`` with the Grant & Grigorieff exposure filter
    ``q_t = exp(-N_t / (2 N_e(k)))``, ``N_t = pre_exposure + (t + 1) * dose_per_frame``: the dose-weighted sum
    ``(h, w)`` of an already motion-corrected ``(t, h, w)`` stack.  The filter is applied to the Fourier-space SUM
    (linear), so only one inverse transform is needed."""
    dev = resolve_device(movie, device)
    stack = as_f32(movie, dev)
    t, h, w = stack.shape
    plan = _fourier.BandPlan(h, w, dev, full=True)
    kxn = w // 2 + 1
    acc = torch.zeros((h, kxn, 2), dtype=torch.float32, device=dev)
    den2 = torch.zeros((h, kxn), dtype=torch.float32, device=dev)
    block = max(2, min(t, int(_BLOCK_BYTES // (h * kxn * 8)) // 2 * 2))
    for f0 in range(0, t, block):
        n = min(block, t - f0)
        spec = plan.forward(stack[f0 : f0 + n], None, None, 0, h, _fourier.frame_pair_jobs(n, dev), job_mode=2)[:n]
        with torch.cuda.device(dev):
            call("tmc_dose_weighted_sum", ptr(spec), n, h, w, float(pixel_size), float(pre_exposure), float(dose_per_frame),
                 float(voltage), f0, ptr(acc), ptr(den2), int(f0 + n >= t), stream_ptr(dev))
        del spec
    out = torch.empty((1, h, w), dtype=torch.float32, device=dev)
    plan.inverse_full(acc.reshape(1, h, kxn, 2), out)
    return out[0]


# ---- low-rank exposure filter (correct_motion_sums) ------------------------------------------------------------------------
# The normalised weights w_t(k) = q_t(k) / sqrt(sum_t q_t(k)^2), q_t = exp(-N_t / (2 N_e(k))), depend on k only through
# x = 1 / N_e(k), and as a (frames x x) matrix they have very low rank.  With w_t(x) ~= sum_r U_r(t) v_r(x) the dose-weighted
# sum is F^-1[sum_r v_r(x(k)) F[sum_t U_r(t) c_t]]: R frame-weighted real-space sums (formed in the warp's frame loop), R
# full-frame transforms and one inverse, whatever the number of frames.

#: bound on the L2 norm over frames of w(x) - U v(x) at every x of the rfft grid (projection and table interpolation)
LOWRANK_TOLERANCE = 1e-6
#: largest rank accepted; real exposures need at most 8 (frames 10..2000, 0.3..0.83 A/px, 0.02..5 e/A^2/frame, 200/300 kV)
LOWRANK_MAX_RANK = 12
#: uniform nodes of x in [0, x_max] on which v_r is tabulated (linear interpolation error ~5e-8 at 4096)
LOWRANK_TABLE_NODES = 4096
_SVD_NODES = 1024  # the time basis U comes from an SVD on this coarser grid; the residual is checked on the table grid


def inverse_critical_exposure(k, voltage: float = 300.0):
    """x = 1 / N_e(k) (float64) for spatial frequencies k in 1/Angstrom: the Grant & Grigorieff critical exposure of
    ``csrc/tables.cu`` (scaled by 0.8 below 300 kV), k clamped to 1e-10 like the kernels."""
    scale = 1.0 if voltage >= 300.0 else 0.8
    k = np.maximum(np.asarray(k, dtype=np.float64), 1e-10)
    return 1.0 / (scale * (0.24499 * k**-1.6649 + 2.8141))


def rfft_grid_x(ny: int, nx: int, pixel_size: float, voltage: float = 300.0) -> np.ndarray:
    """x = 1 / N_e(|k|) of every bin of the (ny, nx/2+1) rfft grid, float64."""
    fy = np.fft.fftfreq(ny)[:, None]
    fx = np.arange(nx // 2 + 1)[None, :] / nx
    return inverse_critical_exposure(np.sqrt(fy * fy + fx * fx) / pixel_size, voltage)


def exposure_weights(x, exposures, rows=None) -> np.ndarray:
    """w_t(x) (len(rows), len(x)) float64 for the frames of cumulative exposure ``exposures`` (e/A^2), normalised over
    ALL of them; ``rows`` selects the frames returned (half sets share the full set's normalisation)."""
    q = np.exp(np.outer(np.asarray(exposures, np.float64), -0.5 * np.asarray(x, np.float64)))
    w = q / np.sqrt(np.einsum("tn,tn->n", q, q))
    return w if rows is None else w[rows]


@dataclass(frozen=True)
class LowRankGroup:
    frames: np.ndarray  # global indices of the group's frames
    basis: np.ndarray  # U (len(frames), R) float64, orthonormal columns
    table: np.ndarray  # v (R, LOWRANK_TABLE_NODES) float64: v_r = sum_t U_r(t) w_t on the x nodes
    residual: float  # worst L2 residual over the table nodes and the midpoints between them (linear interpolation)


@dataclass(frozen=True)
class LowRankExposureFilter:
    x_max: float  # the table spans x in [0, x_max], x_max = 1 / N_e at the corner of the rfft grid
    groups: dict  # "all", or "even" and "odd" (global frame index parity) -> LowRankGroup


def _factor_group(frames_pos, exposures, x_nodes) -> tuple[np.ndarray, np.ndarray, float]:
    n = len(frames_pos)
    if n == 0:
        return np.zeros((0, 0)), np.zeros((0, len(x_nodes))), 0.0
    x_svd = np.linspace(0.0, x_nodes[-1], _SVD_NODES)
    u = np.linalg.svd(exposure_weights(x_svd, exposures, frames_pos), full_matrices=False)[0]
    u = u[:, : min(LOWRANK_MAX_RANK, n)]
    x_mid = 0.5 * (x_nodes[1:] + x_nodes[:-1])
    m_nodes = exposure_weights(x_nodes, exposures, frames_pos)
    v = u.T @ m_nodes
    v_mid = 0.5 * (v[:, 1:] + v[:, :-1])  # what the device interpolates half way between two nodes
    e_nodes, e_mid = m_nodes, exposure_weights(x_mid, exposures, frames_pos)
    for r in range(u.shape[1]):
        e_nodes = e_nodes - np.outer(u[:, r], v[r])
        e_mid = e_mid - np.outer(u[:, r], v_mid[r])
        worst = max(np.sqrt((e_nodes * e_nodes).sum(0)).max(), np.sqrt((e_mid * e_mid).sum(0)).max())
        if worst <= LOWRANK_TOLERANCE:
            return u[:, : r + 1], v[: r + 1], float(worst)
    raise ValueError(
        f"the exposure filter of these frames needs more than {LOWRANK_MAX_RANK} low-rank components for a residual of "
        f"{LOWRANK_TOLERANCE:g} (worst {worst:.2e} at rank {u.shape[1]}); use dose_weight() on the corrected stack"
    )


def exposure_filter_lowrank(ny: int, nx: int, pixel_size: float, frames: range, dose_per_frame: float,
                            pre_exposure: float = 0.0, voltage: float = 300.0, half_sets: bool = False) -> LowRankExposureFilter:
    """Low-rank factorisation (float64, deterministic for given inputs) of the exposure filter of ``frames`` (a range of
    global frame indices; N_t = pre_exposure + (t + 1) dose_per_frame) on the (ny, nx) rfft grid at ``pixel_size``,
    normalised over ``frames``.  Groups: "all", or with ``half_sets`` "even" and "odd" (same normalisation, so the two
    halves sum to the whole).  Each group uses the smallest rank whose worst residual is <= LOWRANK_TOLERANCE.  Cached:
    the factorisation takes 10 ms (40 frames) to 0.5 s (400 frames) of host time; its arrays must not be modified."""
    if not dose_per_frame > 0:
        raise ValueError(f"dose_per_frame must be > 0, got {dose_per_frame}")
    return _exposure_filter_lowrank(int(ny), int(nx), float(pixel_size), range(frames.start, frames.stop),
                                    float(dose_per_frame), float(pre_exposure), float(voltage), bool(half_sets))


@functools.lru_cache(maxsize=16)
def _exposure_filter_lowrank(ny, nx, pixel_size, frames, dose_per_frame, pre_exposure, voltage, half_sets):
    frames = np.arange(frames.start, frames.stop, dtype=np.int64)
    exposures = pre_exposure + (frames + 1) * float(dose_per_frame)
    x_max = float(inverse_critical_exposure(np.hypot((ny // 2) / ny, (nx // 2) / nx) / pixel_size, voltage))
    x_max *= 1.0 + 1e-6  # the kernels compute x in fp32: keep the corner bins inside the table
    x_nodes = np.linspace(0.0, x_max, LOWRANK_TABLE_NODES)
    select = {"even": frames % 2 == 0, "odd": frames % 2 == 1} if half_sets else {"all": np.ones(len(frames), bool)}
    groups = {}
    for name, mask in select.items():
        pos = np.flatnonzero(mask)
        u, v, worst = _factor_group(pos, exposures, x_nodes)
        groups[name] = LowRankGroup(frames[pos], u, v, worst)
    return LowRankExposureFilter(x_max, groups)
