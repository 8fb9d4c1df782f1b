"""correct_motion_sums: the plain, half-set and low-rank dose-weighted frame sums against correct_motion_sum and an
exact float64 exposure filter applied to the correct_motion stack, on the TMA and the global-memory warp."""

import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")


def _case(t, h, w, seed):
    """white-noise movie and a smooth field of a few Angstrom (both on the GPU)"""
    g = torch.Generator(device=DEV).manual_seed(seed)
    movie = torch.randn((t, h, w), generator=g, device=DEV)
    field = 3.0 * torch.randn((2, min(t, 3), 3, 4), generator=g, device=DEV)
    return movie, field


def _rel(a, b):
    return float(torch.linalg.norm((a - b).double()) / torch.linalg.norm(b.double()))


def _exact_dose_weighted(stack, frames, px, dose, pre, kv, total_rows):
    """float64 sum_t irfft2(rfft2(stack_t) q_t / sqrt(sum_{t in total_rows} q_t^2)) over the frames of ``stack``
    (global indices ``frames``); q_t = exp(-N_t / (2 N_e)), N_e from oracle.deps.critical_exposure"""
    from oracle import deps

    h, w = stack.shape[-2:]
    fy = torch.fft.fftfreq(h, dtype=torch.float64, device=stack.device)[:, None]
    fx = torch.fft.rfftfreq(w, dtype=torch.float64, device=stack.device)[None, :]
    ne = deps.critical_exposure(torch.sqrt(fy * fy + fx * fx) / px, kv)
    den2 = sum(torch.exp(-(pre + (t + 1) * dose) / ne) for t in total_rows)
    acc = torch.zeros((h, w // 2 + 1), dtype=torch.complex128, device=stack.device)
    for frame, t in zip(stack, frames):
        acc += torch.fft.rfft2(frame.double()) * torch.exp(-0.5 * (pre + (t + 1) * dose) / ne)
    return torch.fft.irfft2(acc / torch.sqrt(den2), s=(h, w))


@pytest.mark.parametrize("tma", ["1", "0"])
@pytest.mark.parametrize("shape", [(6, 96, 128), (7, 64, 90), (3, 600, 5000), (25, 256, 384)])
def test_sum_is_correct_motion_sum(shape, tma, monkeypatch):
    import torch_motion_correction_b200 as tmc

    monkeypatch.setenv("TMC_WARP_TMA", tma)
    movie, field = _case(*shape, seed=1)
    got = tmc.correct_motion_sums(movie, field, 0.83, half_sets=True)
    want = tmc.correct_motion_sum(movie, field, 0.83)
    assert float((got["sum"] - want).abs().max()) <= 1e-6 * float(want.abs().max())
    assert torch.equal(got["sum"], want)  # fmaf(1, v, acc) == acc + v: same operations as the plain sum
    assert _rel(got["sum_even"] + got["sum_odd"], want) <= 1e-6
    stack = tmc.correct_motion(movie, field, 0.83)
    assert _rel(got["sum_even"], stack[0::2].sum(0)) <= 1e-6
    assert _rel(got["sum_odd"], stack[1::2].sum(0)) <= 1e-6


@pytest.mark.parametrize(
    "shape,px,dose,pre,kv",
    [((6, 96, 128), 1.0, 1.0, 0.0, 300.0), ((7, 64, 90), 0.83, 2.0, 1.5, 200.0), ((3, 600, 5000), 0.83, 1.0, 0.0, 300.0),
     ((40, 4096, 4096), 0.83, 1.0, 0.0, 300.0), ((400, 512, 512), 0.83, 0.1, 0.0, 300.0)],
)
def test_dose_weighted_sums_match_the_exact_filter(shape, px, dose, pre, kv):
    import torch_motion_correction_b200 as tmc

    movie, field = _case(*shape, seed=2)
    t = shape[0]
    got = tmc.correct_motion_sums(movie, field, px, dose_per_frame=dose, pre_exposure=pre, voltage=kv, half_sets=True)
    assert set(got) == {"sum", "sum_even", "sum_odd", "dose_weighted", "dose_weighted_even", "dose_weighted_odd"}
    assert all(v.shape == shape[1:] and v.dtype == torch.float32 for v in got.values())
    assert _rel(got["sum_even"] + got["sum_odd"], got["sum"]) <= 1e-6
    assert _rel(got["dose_weighted_even"] + got["dose_weighted_odd"], got["dose_weighted"]) <= 1e-6
    stack = tmc.correct_motion(movie, field, px)
    del movie
    rows = range(t)
    for name, sel in (("dose_weighted", slice(None)), ("dose_weighted_even", slice(0, None, 2)),
                      ("dose_weighted_odd", slice(1, None, 2))):
        want = _exact_dose_weighted(stack[sel], list(rows)[sel], px, dose, pre, kv, rows)
        assert _rel(got[name], want) <= 1e-5, (name, _rel(got[name], want))


def test_dose_weighted_matches_the_oracle_dose_weight():
    import torch_motion_correction_b200 as tmc
    from oracle import reference_path as rp

    movie, field = _case(8, 128, 160, seed=3)
    got = tmc.correct_motion_sums(movie, field, 1.1, dose_per_frame=1.5, pre_exposure=2.0)
    assert set(got) == {"sum", "dose_weighted"}
    want = rp.dose_weight(tmc.correct_motion(movie, field, 1.1).cpu(), 1.1, 2.0, 1.5)
    assert _rel(got["dose_weighted"].cpu(), want) <= 1e-4


@pytest.mark.parametrize("tma", ["1", "0"])
def test_frame_range(tma, monkeypatch):
    import torch_motion_correction_b200 as tmc

    monkeypatch.setenv("TMC_WARP_TMA", tma)
    movie, field = _case(12, 128, 128, seed=4)
    a, b = 3, 10
    got = tmc.correct_motion_sums(movie, field, 0.9, dose_per_frame=1.2, pre_exposure=0.7, half_sets=True, frame_range=(a, b))
    want = tmc.correct_motion_sum(movie[a:b], field, 0.9, frame_offset=a, total_frames=12)
    assert torch.equal(got["sum"], want)
    stack = tmc.correct_motion(movie, field, 0.9)[a:b]
    assert _rel(got["sum_even"], stack[1::2].sum(0)) <= 1e-6  # frames 4, 6, 8: parity of the global index
    rows = range(a, b)
    assert _rel(got["dose_weighted"], _exact_dose_weighted(stack, rows, 0.9, 1.2, 0.7, 300.0, rows)) <= 1e-5
    want_odd = _exact_dose_weighted(stack[0::2], rows[0::2], 0.9, 1.2, 0.7, 300.0, rows)
    assert _rel(got["dose_weighted_odd"], want_odd) <= 1e-5


def test_peak_memory_stays_below_one_stack():
    import torch_motion_correction_b200 as tmc

    movie, field = _case(160, 512, 512, seed=5)
    stack_bytes = movie.numel() * 4
    tmc.correct_motion_sums(movie, field, 0.83, dose_per_frame=1.0, half_sets=True)  # warm-up (plans, tables)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    out = tmc.correct_motion_sums(movie, field, 0.83, dose_per_frame=1.0, half_sets=True)
    torch.cuda.synchronize()
    fused = torch.cuda.max_memory_allocated() - base
    del out
    torch.cuda.reset_peak_memory_stats()
    tmc.dose_weight(tmc.correct_motion(movie, field, 0.83), 0.83, dose_per_frame=1.0)
    torch.cuda.synchronize()
    materialising = torch.cuda.max_memory_allocated() - base
    assert fused < stack_bytes < materialising, (fused, stack_bytes, materialising)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import torch_motion_correction_b200 as tmc
        from torch_motion_correction_b200.distributed import correct_motion_sums_frame_split, frame_range

        movie, field = _case(9, 128, 192, seed=6)
        t = movie.shape[0]
        f0, f1 = frame_range(t, rank, world)
        kw = dict(dose_per_frame=0.8, pre_exposure=1.0, half_sets=True)
        got = correct_motion_sums_frame_split(movie[f0:f1].clone(), field, 1.05, f0, t, **kw)
        want = tmc.correct_motion_sums(movie, field, 1.05, **kw)
        assert set(got) == set(want)
        for name in want:
            assert _rel(got[name], want[name]) <= 1e-6, (name, _rel(got[name], want[name]))
        with open(os.path.join(out_dir, f"ok{rank}"), "w") as f:
            f.write("ok")
    finally:
        dist.destroy_process_group()


def test_frame_split_matches_single_process_world2(tmp_path):
    mp.spawn(_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    assert all((tmp_path / f"ok{r}").exists() for r in range(2))
