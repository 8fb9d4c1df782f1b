"""Generate the committed golden vectors from the UNMODIFIED reference source.

Run in the build container only (needs ``/root/reference``):

    python tests/golden/make_golden.py

It imports ``/root/reference/src/torch_motion_correction`` verbatim on top of the restated
third-party layer (``oracle.deps``; the real packages are not installable here), runs the
reference's own public functions on small seeded movies on the CPU and stores inputs and
outputs in ``tests/golden/*.npz``.  The ``-m "not gpu"`` tests check ``oracle.reference_path``
against these files; the ``-m gpu`` tests check the CUDA path against them as well.
"""

from __future__ import annotations

import os
import random
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import deps, verbatim  # noqa: E402
from oracle.reference_path import synthetic_movie, synthetic_movie_large  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))


def np32(x):
    return x.detach().cpu().numpy()


def smooth_field(seed, shape, scale):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn((2, *shape), generator=g) * scale).float()


def case_small(ref):
    """6x96x96 movie: every public entry point once."""
    out = {}
    px = 1.3
    movie, walk = synthetic_movie(6, 96, 96, seed=11, noise=0.5, drift=3.0, local=0.8, sigma_f=0.07)
    out["movie"] = np32(movie)
    out["pixel_spacing"] = np.float64(px)
    fr = (120.0, 6.0)  # wide enough to keep a useful band on 32/48 px patches
    out["frequency_range"] = np.asarray(fr)
    with verbatim.quiet():
        out["global_field"] = np32(ref.estimate_global_motion(movie.clone(), px, frequency_range=fr))
        out["global_field_ref0_b1000"] = np32(
            ref.estimate_global_motion(movie.clone(), px, reference_frame=0, b_factor=1000, frequency_range=fr)
        )
        for strat in ("mean_except_current", "middle_frame"):
            f, pos = ref.estimate_motion_cross_correlation_patches(
                movie.clone(), px, reference_strategy=strat, patch_sidelength=32, frequency_range=fr,
                temporal_smoothing=False, outlier_rejection=False,
            )
            out[f"xc_raw_{strat}"] = np32(f)
            f, pos = ref.estimate_motion_cross_correlation_patches(
                movie.clone(), px, reference_strategy=strat, patch_sidelength=32, frequency_range=fr,
                smoothing_window_size=3, outlier_threshold=1.5,
            )
            out[f"xc_full_{strat}"] = np32(f)
            out["xc_positions"] = np32(pos)
        f, _ = ref.estimate_motion_cross_correlation_patches(
            movie.clone(), px, patch_sidelength=32, frequency_range=fr, sub_pixel_refinement=False,
            temporal_smoothing=False, outlier_rejection=False,
        )
        out["xc_integer"] = np32(f)
        # cumulative paths: (2,t,1,1) field -> correct_motion_fast (Q2), full field -> correct_motion(bspline)
        g0 = torch.as_tensor(out["global_field"]).clone()
        f, _ = ref.estimate_motion_cross_correlation_patches(
            movie.clone(), px, patch_sidelength=32, frequency_range=fr, deformation_field=g0
        )
        out["xc_cumulative_global"] = np32(f)
        out["xc_cumulative_global_field_after"] = np32(g0)  # Q2: negated in place
        f0 = smooth_field(5, (6, 3, 3), 1.5)
        f, _ = ref.estimate_motion_cross_correlation_patches(
            movie.clone(), px, patch_sidelength=32, frequency_range=fr, deformation_field=f0.clone()
        )
        out["xc_cumulative_full_in"] = np32(f0)
        out["xc_cumulative_full"] = np32(f)

        # correction: every other row of the corrected stacks (keeps the file under 1 MB)
        field = smooth_field(3, (3, 4, 4), 2.0)
        out["field_344"] = np32(field)
        out["correct_catmull"] = np32(ref.correct_motion(movie, field.clone(), px)[:, ::2])
        out["correct_bspline"] = np32(ref.correct_motion(movie, field.clone(), px, grid_type="bspline")[:, ::2])
        field1 = smooth_field(4, (6, 1, 1), 2.5)
        out["field_611"] = np32(field1)
        out["correct_611_catmull"] = np32(ref.correct_motion(movie, field1.clone(), px)[:, ::2])
        fast_in = field1.clone()
        out["correct_fast"] = np32(ref.correct_motion_fast(movie, fast_in)[:, ::2])
        out["correct_fast_field_after"] = np32(fast_in)
        out["correct_slow"] = np32(ref.correct_motion_slow(movie, field.clone())[:, ::2])
        new = ref.correct_motion.__globals__["CubicCatmullRomGrid3d"].from_grid_data(smooth_field(6, (3, 4, 4), 0.7))
        base = ref.correct_motion.__globals__["CubicCatmullRomGrid3d"].from_grid_data(field.clone())
        out["two_grids_new"] = np32(new.data)
        out["correct_two_grids"] = np32(
            ref.correct_motion_two_grids(movie, new, base, px, grad=False)[:, ::2]
        )
        # pixel shifts of one frame
        lattice = ref.deformation_field_utils.evaluate_deformation_field_at_t(field, 0.4, (40, 40), "bspline")
        out["lattice_t04_bspline"] = np32(lattice)
        grid = deps.coordinate_grid((96, 96))
        out["pixel_shifts"] = np32(ref.get_pixel_shifts(movie[0], px, lattice, grid))
        # spline evaluation
        g = torch.Generator().manual_seed(9)
        tyx = torch.rand((257, 3), generator=g)
        tyx[0] = 0.0
        tyx[1] = 1.0
        out["tyx"] = np32(tyx)
        out["eval_catmull"] = np32(ref.evaluate_deformation_field(field, tyx))
        out["eval_bspline"] = np32(ref.evaluate_deformation_field(field, tyx, grid_type="bspline"))
        out["eval_611_catmull"] = np32(ref.evaluate_deformation_field(field1, tyx))
        out["resample_to_534"] = np32(ref.deformation_field_utils.resample_deformation_field(field, (5, 3, 4)))

        # spline optimiser
        init = torch.as_tensor(out["xc_full_mean_except_current"]).clone()
        for name, kw in {
            "adam_catmull_mse": dict(optimizer_type="adam", grid_type="catmull_rom", loss_type="mse"),
            "adam_bspline_mse": dict(optimizer_type="adam", grid_type="bspline", loss_type="mse"),
            "sgd_bspline_ncc": dict(optimizer_type="sgd", grid_type="bspline", loss_type="ncc"),
            "rmsprop_catmull_cc": dict(optimizer_type="rmsprop", grid_type="catmull_rom", loss_type="cc",
                                       optimizer_kwargs={"lr": 0.001}),
            "lbfgs_bspline_mse": dict(optimizer_type="lbfgs", grid_type="bspline", loss_type="mse"),
        }.items():
            random.seed(1234)
            res, traj = ref.estimate_local_motion(
                movie.clone(), px, (32, 32), (3, 3, 3), init.clone(), n_iterations=6, frequency_range=fr,
                return_trajectory=True, **kw,
            )
            out[f"local_{name}"] = np32(res)
            out[f"local_{name}_losses"] = np.asarray([c.loss for c in traj.checkpoints])
        random.seed(77)
        res = ref.estimate_local_motion(
            movie.clone(), px, (48, 48), (2, 2, 2), None, n_iterations=4, frequency_range=fr
        )
        out["local_noinit_p48"] = np32(res)
    np.savez_compressed(os.path.join(OUT, "small.npz"), **out)
    print("small.npz", {k: v.shape for k, v in out.items() if hasattr(v, "shape")})


def case_eviction(ref):
    """T=60 > 50 cache entries: the irregular Q1 regime (cache eviction)."""
    out = {}
    px = 1.0
    movie, _ = synthetic_movie(60, 64, 64, seed=21, noise=0.7, drift=2.5, local=0.0, sigma_f=0.09)
    out["movie"] = np32(movie.half().float())  # values exactly representable in fp16 -> smaller file
    movie = torch.as_tensor(out["movie"])
    fr = (100.0, 5.0)
    out["frequency_range"] = np.asarray(fr)
    with verbatim.quiet():
        for strat in ("mean_except_current", "middle_frame"):
            f, _ = ref.estimate_motion_cross_correlation_patches(
                movie.clone(), px, reference_strategy=strat, patch_sidelength=32, frequency_range=fr,
                temporal_smoothing=False, outlier_rejection=False,
            )
            out[f"xc_raw_{strat}"] = np32(f)
    out["movie"] = out["movie"].astype(np.float16)
    np.savez_compressed(os.path.join(OUT, "eviction.npz"), **out)
    print("eviction.npz done")


def case_c1(ref):
    """BASELINE config 1: 10x512x512, known integer global shifts, patch 128 (6x6)."""
    out = {}
    px = 1.0
    movie, walk = synthetic_movie(10, 512, 512, seed=0, noise=1.0, drift=6.0, integer_shifts=True, sigma_f=0.08)
    out["seed"] = np.int64(0)
    out["true_shifts"] = np32(walk)
    with verbatim.quiet():
        g = ref.estimate_global_motion(movie.clone(), px)
        out["global_field"] = np32(g)
        f, pos = ref.estimate_motion_cross_correlation_patches(movie.clone(), px, patch_sidelength=128)
        out["xc_field"] = np32(f)
        out["xc_positions"] = np32(pos)
        corr = ref.correct_motion(movie, f, px, grid_type="bspline")
        s = corr.sum(dim=0)
        out["corrected_sum_crop"] = np32(s[192:320, 192:320])
        out["corrected_sum_norm"] = np.float64(torch.linalg.norm(s.double()))
        out["corrected_sum_rows"] = np32(s[::64, :])
        random.seed(5)
        res, traj = ref.estimate_local_motion(
            movie.clone(), px, (128, 128), (3, 5, 5), f.clone(), n_iterations=3, grid_type="bspline",
            return_trajectory=True,
        )
        out["local_field"] = np32(res)
        out["local_losses"] = np.asarray([c.loss for c in traj.checkpoints])
    np.savez_compressed(os.path.join(OUT, "c1.npz"), **out)
    print("c1.npz done")


# ---- benchmark-sized cases (BASELINE configs 2-4 code paths: p = 1024 patches, T = 40 / 60, 4096-point whole-frame
# transforms).  Only fields, crops and norms are stored (KBs); the tests regenerate the movies from their seeds with
# oracle.reference_path.synthetic_movie_large / synthetic_movie.

LARGE = dict(c2half=dict(t=40, size=2048, seed=40, px=0.83, resolution=(3, 5, 5), iters=4),
             c3half=dict(t=60, size=2048, seed=60, px=0.83, resolution=(5, 6, 6), iters=3),
             # BASELINE configs 2 and 3 at their full size (about 5 and 8 CPU-minutes, ~25 GB of host memory)
             c2full=dict(t=40, size=4096, seed=41, px=0.83, resolution=(3, 5, 5), iters=3),
             c3full=dict(t=60, size=4096, seed=61, px=0.83, resolution=(5, 6, 6), iters=2),
             # BASELINE config 4's code paths (8192-point whole-frame transforms, 15 x 15 / 14 x 14 patch grids) on 10 frames
             c4short=dict(t=10, size=8192, seed=81, px=0.83, resolution=(3, 5, 5), iters=2))


def sum_samples(s):
    """What is kept of an (h, w) frame sum: centre crop, corner crop (border taps / zero-outside), strided rows, norm."""
    h, w = s.shape
    return {
        "sum_centre": np32(s[h // 2 - 96 : h // 2 + 96, w // 2 - 96 : w // 2 + 96]),
        "sum_corner": np32(s[:96, :96]),
        "sum_rows": np32(s[:: h // (16 if h <= 4096 else 8), :]),  # 8 rows of 8192^2: keeps the file under 1 MB
        "sum_norm": np.float64(torch.linalg.norm(s.double())),
    }


def case_large(ref, name):
    import time

    cfg = LARGE[name]
    t, n, px = cfg["t"], cfg["size"], cfg["px"]
    movie, walk = synthetic_movie_large(t, n, n, seed=cfg["seed"], noise=1.0, drift=6.0, local=1.5)
    out = {"seed": np.int64(cfg["seed"]), "t": np.int64(t), "size": np.int64(n), "pixel_spacing": np.float64(px),
           "true_global": np32(walk), "movie_checksum": np.float64(movie.double().sum()),
           "movie_probe": np32(movie[:: max(t // 4, 1), ::257, ::263])}
    tic = time.time()
    with verbatim.quiet():
        g = ref.estimate_global_motion(movie.clone(), px)
        out["global_field"] = np32(g)
        f, pos = ref.estimate_motion_cross_correlation_patches(movie.clone(), px, patch_sidelength=1024)
        out["xc_field"] = np32(f)
        out["xc_positions"] = np32(pos)
        fraw, _ = ref.estimate_motion_cross_correlation_patches(
            movie.clone(), px, patch_sidelength=1024, temporal_smoothing=False, outlier_rejection=False)
        out["xc_raw"] = np32(fraw)
        if name.startswith("c2"):
            # the rigid pre-field route the pipeline drives: (2,t,1,1) field in PIXELS handed over (quirk Q2: used as px,
            # negated in place, shifts accumulated on the negated field)
            pre = (g / px).clone()
            fp, _ = ref.estimate_motion_cross_correlation_patches(
                movie.clone(), px, patch_sidelength=1024, deformation_field=pre, temporal_smoothing=False)
            out["xc_pre_nosmooth"] = np32(fp)
            out["xc_pre_field_after"] = np32(pre)
            pre = (g / px).clone()
            fp, _ = ref.estimate_motion_cross_correlation_patches(
                movie.clone(), px, patch_sidelength=1024, deformation_field=pre)
            out["xc_pre"] = np32(fp)
        print(name, "xc done", time.time() - tic, file=sys.__stdout__, flush=True)
        random.seed(2024)
        res, traj = ref.estimate_local_motion(
            movie.clone(), px, (1024, 1024), cfg["resolution"], f.clone(), n_iterations=cfg["iters"], grid_type="bspline",
            return_trajectory=True,
        )
        out["local_field"] = np32(res)
        out["local_losses"] = np.asarray([c.loss for c in traj.checkpoints])
        print(name, "local done", time.time() - tic, file=sys.__stdout__, flush=True)
        if name.startswith("c2") or name.startswith("c4"):
            corr = ref.correct_motion(movie, res, px, grid_type="bspline")
            out.update(sum_samples(corr.sum(dim=0)))
            del corr
            corr = ref.correct_motion(movie[:6], f[:, :6].contiguous(), px)  # (2, t, gh, gw) field, Catmull-Rom default
            out.update({"xcfield_" + k: v for k, v in sum_samples(corr.sum(dim=0)).items()})
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
    print(name, "done", time.time() - tic, file=sys.__stdout__, flush=True)


def case_whole4096(ref, n=4096, seed=7):
    """4 frames of n^2: the n-point whole-frame transforms (global estimate, rigid Fourier-shift correction)."""
    out = {}
    px = 0.83
    movie, walk = synthetic_movie(4, n, n, seed=seed, noise=1.0, drift=9.0, integer_shifts=True, sigma_f=0.08)
    out["seed"] = np.int64(seed)
    out["true_shifts"] = np32(walk)
    with verbatim.quiet():
        g = ref.estimate_global_motion(movie.clone(), px)
        out["global_field"] = np32(g)
        field = torch.tensor([[1.5, -2.25, 0.0, 3.7], [-0.5, 4.125, 2.0, -6.3]]).reshape(2, 4, 1, 1)
        out["fast_field"] = np32(field)
        corr = ref.correct_motion_fast(movie, field.clone())
        out["fast_centre"] = np32(corr[:, n // 2 - 64 : n // 2 + 64, n // 2 - 64 : n // 2 + 64])
        out["fast_corner"] = np32(corr[:, :64, :64])
        out["fast_rows"] = np32(corr[:, :: n // (8 if n <= 4096 else 4), :])  # 4 rows of 8192^2: keeps the file under 1 MB
        out["fast_norm"] = np.float64(torch.linalg.norm(corr.double()))
    np.savez_compressed(os.path.join(OUT, f"whole{n}.npz"), **out)
    print(f"whole{n}.npz done", file=sys.__stdout__, flush=True)


def main():
    torch.set_num_threads(os.cpu_count() or 1)
    ref = verbatim.load()
    import torch_motion_correction.deformation_field_utils  # noqa: F401  (attribute access below)

    which = sys.argv[1:] or ["small", "eviction", "c1"]  # the benchmark-sized cases take ~10 CPU-minutes each: by name
    for name in which:
        if name in LARGE:
            case_large(ref, name)
        else:
            {"small": case_small, "eviction": case_eviction, "c1": case_c1, "whole4096": case_whole4096,
             "whole8192": lambda r: case_whole4096(r, 8192, 8)}[name](ref)


if __name__ == "__main__":
    main()
