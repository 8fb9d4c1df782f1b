"""Frame grouping on the GPU: the group sums bit for bit against an fp32 loop, the lattice at a time table against the
linspace lattice, the grouped correction against the oracle evaluated at tau(f), the fused sums, the pipeline, and a
known answer in the low-dose regime grouping exists for."""

import functools

import numpy as np
import pytest
import torch

import torch_motion_correction_b200 as tmc
from oracle import reference_path as rp
from torch_motion_correction_b200 import _ops
from torch_motion_correction_b200.frame_groups import frame_groups

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")


def _rel(a, b):
    return float(torch.linalg.norm((a - b).double()) / torch.linalg.norm(b.double()))


def _loop_sums(movie, g):
    """fp32 in-place adds in ascending frame order, the last group taking the leftovers"""
    n = movie.shape[0] // g
    out = []
    for k in range(n):
        stop = movie.shape[0] if k == n - 1 else (k + 1) * g
        acc = movie[k * g].clone()
        for f in range(k * g + 1, stop):
            acc += movie[f]
        out.append(acc)
    return torch.stack(out)


def _group_sizes(t):
    return sorted({g for g in (1, 2, 3, 10, t // 2) if g >= 1 and t // g >= 2})


@pytest.mark.parametrize("shape,aligned", [((41, 96, 132), True), ((400, 256, 256), True), ((7, 33, 35), True),
                                           ((41, 96, 132), False)])
def test_group_sums_are_an_fp32_loop_bit_for_bit(shape, aligned):
    t, h, w = shape
    g = torch.Generator(device=DEV).manual_seed(t + h)
    base = torch.randn((t * h * w + 1,), generator=g, device=DEV)
    movie = base[: t * h * w].view(t, h, w) if aligned else base[1:].view(t, h, w)
    assert (movie.data_ptr() % 16 == 0) == aligned
    for size in _group_sizes(t):
        got = tmc.group_frames(movie, size)
        if size == 1:
            assert got is movie
            continue
        assert got.shape == (t // size, h, w) and got.dtype == torch.float32
        assert torch.equal(got, _loop_sums(movie, size)), size


def _linspace01(i, n):
    """common.cuh linspace01 in float32"""
    if n <= 1:
        return np.float32(0)
    step = np.float32(1) / np.float32(n - 1)
    if i < n // 2:
        return step * np.float32(i)
    return np.float32(1) - step * np.float32(n - 1 - i)


@pytest.mark.parametrize("kind", [0, 1])
@pytest.mark.parametrize("n_frames,offset,total", [(17, 0, 17), (9, 5, 30), (1, 40, 41)])
def test_lattice_at_linspace_times_is_the_linspace_lattice(kind, n_frames, offset, total):
    g = torch.Generator(device=DEV).manual_seed(n_frames + offset)
    field = 4.0 * torch.randn((2, 3, 4, 5), generator=g, device=DEV)
    times = torch.tensor([_linspace01(offset + f, total) for f in range(n_frames)], dtype=torch.float32, device=DEV)
    want = _ops.spline_lattice(field, kind, n_frames, 40, 50, frame_offset=offset, total_frames=total)
    got = _ops.spline_lattice(field, kind, n_frames, 40, 50, times=times)
    assert torch.equal(got, want)


def _case(t, h, w, nt, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    movie = torch.randn((t, h, w), generator=g, device=DEV)
    field = 3.0 * torch.randn((2, nt, 3, 4), generator=g, device=DEV)
    field[:, 1] += 4.0  # real time structure: the middle node stands apart
    return movie, field


@pytest.mark.parametrize("grid", ["catmull_rom", "bspline"])
@pytest.mark.parametrize("shape,group", [((11, 64, 80), 3), ((9, 64, 90), 2)])  # 90 % 4 != 0: global-memory warp
def test_grouped_correction_matches_the_oracle_at_tau(grid, shape, group):
    movie, field = _case(*shape, nt=3, seed=shape[0] + group)
    px = 0.9
    got = tmc.correct_motion(movie, field, px, grid_type=grid, frame_group=group).cpu()
    tau = frame_groups(shape[0], group).times
    gh, gw = field.shape[-2:]
    f_cpu, m_cpu = field.cpu(), movie.cpu()
    for f in range(shape[0]):
        lattice = rp.evaluate_deformation_field_at_t(f_cpu, float(tau[f]), (10 * gh, 10 * gw), grid)
        want = rp.correct_frame(m_cpu[f], px, lattice)
        assert _rel(got[f], want) <= 1e-4, (f, _rel(got[f], want))
    # grouping changes the result: the frames are not evaluated at linspace(0, 1, t)
    assert _rel(got, tmc.correct_motion(movie, field, px, grid_type=grid).cpu()) > 1e-3


def _exact_dose_weighted(stack, frames, px, dose, kv=300.0):
    """float64 sum_t irfft2(rfft2(stack_t) q_t / sqrt(sum_t q_t^2)) over the frames of ``stack`` (global indices)"""
    from oracle import deps

    h, w = stack.shape[-2:]
    fy = torch.fft.fftfreq(h, dtype=torch.float64, device=stack.device)[:, None]
    fx = torch.fft.rfftfreq(w, dtype=torch.float64, device=stack.device)[None, :]
    ne = deps.critical_exposure(torch.sqrt(fy * fy + fx * fx) / px, kv)
    den2 = sum(torch.exp(-((t + 1) * dose) / ne) for t in frames)
    acc = torch.zeros((h, w // 2 + 1), dtype=torch.complex128, device=stack.device)
    for frame, t in zip(stack, frames):
        acc += torch.fft.rfft2(frame.double()) * torch.exp(-0.5 * ((t + 1) * dose) / ne)
    return torch.fft.irfft2(acc / torch.sqrt(den2), s=(h, w))


@pytest.mark.parametrize("shape,group", [((23, 96, 128), 4), ((13, 64, 90), 3)])
def test_grouped_sums(shape, group):
    t = shape[0]
    movie, field = _case(*shape, nt=3, seed=7 + t)
    px, dose = 0.83, 0.4
    fused = tmc.correct_motion_sum(movie, field, px, frame_group=group)
    sums = tmc.correct_motion_sums(movie, field, px, dose_per_frame=dose, half_sets=True, frame_group=group)
    assert torch.equal(sums["sum"], fused)
    stack = tmc.correct_motion(movie, field, px, frame_group=group)
    assert _rel(fused, stack.sum(0)) <= 1e-6
    assert _rel(sums["sum_even"], stack[0::2].sum(0)) <= 1e-6  # parity of the raw frame index
    assert _rel(sums["dose_weighted"], _exact_dose_weighted(stack, range(t), px, dose)) <= 1e-5
    # blocks of frames add up to the whole movie
    k = t // 2 + 1
    a = tmc.correct_motion_sums(movie, field, px, frame_range=(0, k), frame_group=group)["sum"]
    b = tmc.correct_motion_sums(movie, field, px, frame_range=(k, t), frame_group=group)["sum"]
    assert _rel(a + b, fused) <= 1e-6
    part = tmc.correct_motion_sum(movie[:k], field, px, frame_offset=0, total_frames=t, frame_group=group)
    tmc.correct_motion_sum(movie[k:], field, px, out=part, accumulate=True, frame_offset=k, total_frames=t,
                           frame_group=group)
    assert _rel(part, fused) <= 1e-6


def _pipeline_movie():
    movie, _ = rp.synthetic_movie_large(24, 384, 384, seed=4, noise=2.0, drift=4.0, local=0.5)
    return movie.to(DEV)


PIPE = dict(patch_sidelength=128, frequency_range=(120.0, 6.0))


def test_estimate_motion_runs_on_the_group_sums():
    movie = _pipeline_movie()
    px, group = 1.1, 4
    got, centres = tmc.estimate_motion(movie, px, frame_group=group, dose_per_frame=0.2, **PIPE)
    want, want_centres = tmc.estimate_motion(tmc.group_frames(movie, group), px, dose_per_frame=0.2 * group, **PIPE)
    assert got.shape[1] == 24 // group
    assert torch.equal(got, want) and torch.equal(centres, want_centres)


def test_motion_correct_corrects_every_raw_frame_with_the_grouped_field():
    movie = _pipeline_movie()
    px, group = 1.1, 5
    total, field = tmc.motion_correct(movie, px, frame_group=group, **PIPE)
    assert field.shape[1] == 24 // group
    assert torch.equal(total, tmc.correct_motion_sum(movie, field, px, grid_type="bspline", frame_group=group))
    dw, field_dw = tmc.motion_correct(movie, px, frame_group=group, dose_per_frame=0.1, **PIPE)
    want = tmc.correct_motion_sums(movie, field_dw, px, "bspline", dose_per_frame=0.1, frame_group=group)["dose_weighted"]
    assert torch.equal(dw, want)
    # motion_correct_many forwards the keyword
    host = [movie.cpu().pin_memory(), (movie.flip(1) * 0.5).cpu().pin_memory()]
    for (s, f), m in zip(tmc.motion_correct_many(host, px, frame_group=group, **PIPE), host):
        want_s, want_f = tmc.motion_correct(m.to(DEV), px, frame_group=group, **PIPE)
        assert torch.equal(f, want_f) and torch.equal(s.to(DEV), want_s)


def test_no_grouping_is_todays_result():
    movie = _pipeline_movie()
    px = 1.1
    ref_sum, ref_field = tmc.motion_correct(movie, px, **PIPE)
    for group in (None, 1):
        s, f = tmc.motion_correct(movie, px, frame_group=group, **PIPE)
        assert torch.equal(f, ref_field) and torch.equal(s, ref_sum), group
        assert torch.equal(tmc.correct_motion(movie, ref_field, px, frame_group=group), tmc.correct_motion(movie, ref_field, px))


# ---- known answer: 120 low-dose frames, where single frames do not give a usable field ----------------------------

# Per-pixel noise over a unit-variance specimen.  At this seed single frames lose the track from noise 24 on (RMS error
# 13 px on a B200, against 0.48 px at noise 16) while 10-frame groups stay at 0.43 px.  The drift is kept at 1 px: the
# synthetic walk is a random walk, and at 8 px its frame-to-frame jitter alone leaves any 10-frame grouping (with the
# estimator's 5-sample temporal smoothing) about 1.1 px off at every noise level; beam-induced motion is smooth.
KNOWN_NOISE = 24.0
KNOWN_DRIFT = 1.0


@functools.lru_cache(maxsize=4)
def _known_movie(t, n, patch, seed, drift, local):
    """noise-free synthetic_movie_large, its patch centres (y, x) and the (t, n_patches, 2) px content displacement of
    each frame at each centre: the global walk plus the local B-spline field (the generator's draws replayed)."""
    from oracle import deps
    from torch_motion_correction_b200.patch_grid import patch_grid_centers

    centres = patch_grid_centers((t, n, n), (1, patch, patch), (1, patch // 2, patch // 2), distribute_patches=True)
    centres_yx = centres[0, :, :, 1:].reshape(-1, 2).float()
    clean, walk = rp.synthetic_movie_large(t, n, n, seed=seed, noise=0.0, drift=drift, local=local)
    g = torch.Generator().manual_seed(seed)
    torch.randn((n + 128, n + 128), generator=g)  # specimen
    torch.randn((t, 2), generator=g)  # walk steps
    coef = torch.randn((2, 3, 4, 4), generator=g) * local
    cy, cx = centres_yx[:, 0] / (n - 1), centres_yx[:, 1] / (n - 1)
    truth = torch.empty((t, len(cy), 2))
    for k in range(t):
        tyx = torch.stack([torch.full_like(cy, k / (t - 1)), cy, cx], dim=-1)
        truth[k] = walk[k] + deps.evaluate_cubic_grid_3d(coef, tyx, deps.BSPLINE_MATRIX)
    return clean, centres_yx, truth - truth.mean(dim=(0, 1))


def known_answer_errors(noise=KNOWN_NOISE, group=10, t=120, n=1024, px=1.0, patch=256, seed=5, drift=KNOWN_DRIFT,
                        local=1.0):
    """RMS over frames and patch centres of |estimated field at tau(f) - true shift| in px (means removed per axis),
    estimated on the group sums and on the raw frames"""
    clean, centres_yx, truth = _known_movie(t, n, patch, seed, drift, local)
    g = torch.Generator(device=DEV).manual_seed(seed)
    movie = clean.to(DEV) + noise * torch.randn(clean.shape, generator=g, device=DEV)
    errors = {}
    for label, fg in (("grouped", group), ("ungrouped", None)):
        field, got_centres = tmc.estimate_motion(movie, px, patch_sidelength=patch, frame_group=fg)
        assert torch.equal(got_centres[0, :, :, 1:].reshape(-1, 2).cpu().float(), centres_yx)
        gh, gw = field.shape[-2:]
        tau = frame_groups(t, fg).times if fg else np.linspace(0, 1, t, dtype=np.float32)
        iy, ix = torch.meshgrid(torch.linspace(0, 1, gh), torch.linspace(0, 1, gw), indexing="ij")
        est = torch.empty((t, gh * gw, 2))
        for k in range(t):  # Catmull-Rom interpolates: at the spatial nodes this is each patch's own track
            tyx = torch.stack([torch.full_like(iy, float(tau[k])), iy, ix], dim=-1).reshape(-1, 3)
            est[k] = rp.evaluate_deformation_field(field.cpu(), tyx, "catmull_rom") / px
        est = est - est.mean(dim=(0, 1))
        errors[label] = float(torch.sqrt(((est - truth) ** 2).sum(-1).mean()))
    return errors


def test_grouping_recovers_the_motion_of_a_low_dose_movie():
    errors = known_answer_errors()
    assert errors["grouped"] <= 0.5, errors
    assert errors["ungrouped"] >= 2 * errors["grouped"], errors
