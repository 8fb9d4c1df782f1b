"""Frame grouping (MotionCor2 ``-Group``, RELION "group frames"): the one rule that says which raw frames form each
group and where each raw frame sits on the time axis of a field estimated on the group sums.  Pure host code.

For ``n_frames`` frames and group size G:

* ``n_groups = n_frames // G`` (at least 2); frame f belongs to group ``min(f // G, n_groups - 1)``, so the last group
  also takes the ``n_frames % G`` leftover frames;
* ``c_g``, the mean frame index of group g, is where group g's sum sits in time; on the grouped movie the estimators put
  group g at the normalised time ``g / (n_groups - 1)``;
* raw frame f gets the time tau(f): the piecewise-linear interpolation of the points ``(c_g, g / (n_groups - 1))``, the
  first and last segments extended linearly before ``c_0`` and after the last centre.  Computed in float64 and rounded
  to float32 once.

tau lies slightly below 0 and above 1 for the outer half groups.  It is not clamped: the spline kernels (like the
reference's grids) clamp the interval a time falls in, not the time, so the field's first and last intervals' cubics are
extended there.  With G = 1 tau is ``linspace(0, 1, n_frames)`` (to within float32 rounding)."""

from __future__ import annotations

from dataclasses import dataclass

import numpy as np


@dataclass(frozen=True)
class FrameGroups:
    n_frames: int
    group_size: int
    starts: np.ndarray  # (n_groups,) int64: first raw frame of each group
    counts: np.ndarray  # (n_groups,) int64: raw frames in each group
    centres: np.ndarray  # (n_groups,) float64: mean raw frame index of each group

    @property
    def n_groups(self) -> int:
        return len(self.starts)

    def group_of(self, frames) -> np.ndarray:
        """Group index of each raw frame index."""
        return np.minimum(np.asarray(frames) // self.group_size, self.n_groups - 1)

    def time_at(self, frames) -> np.ndarray:
        """tau at (possibly fractional) raw frame positions, float64."""
        f = np.asarray(frames, dtype=np.float64)
        c = self.centres
        k = np.clip(np.searchsorted(c, f, side="right") - 1, 0, self.n_groups - 2)
        return (k + (f - c[k]) / (c[k + 1] - c[k])) / (self.n_groups - 1)

    @property
    def times(self) -> np.ndarray:
        """(n_frames,) float32: tau of every raw frame."""
        return self.time_at(np.arange(self.n_frames)).astype(np.float32)


def frame_groups(n_frames: int, frame_group) -> FrameGroups:
    """The group layout of an ``n_frames`` movie for group size ``frame_group``; ``ValueError`` unless ``frame_group`` is
    an int >= 1 that leaves at least two groups."""
    if isinstance(frame_group, bool) or not isinstance(frame_group, (int, np.integer)):
        raise ValueError(f"frame_group must be an int >= 1, got {frame_group!r}")
    g = int(frame_group)
    if g < 1:
        raise ValueError(f"frame_group must be an int >= 1, got {g}")
    n_groups = int(n_frames) // g
    if n_groups < 2:
        raise ValueError(f"frame_group={g} leaves {n_groups} group(s) of a {n_frames}-frame movie; at least 2 are needed "
                         f"(frame_group <= {int(n_frames) // 2})")
    starts = np.arange(n_groups, dtype=np.int64) * g
    counts = np.full(n_groups, g, dtype=np.int64)
    counts[-1] = n_frames - starts[-1]
    centres = starts + (counts - 1) / 2.0
    return FrameGroups(int(n_frames), g, starts, counts, centres)

