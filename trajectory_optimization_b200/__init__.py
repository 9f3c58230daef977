"""trajectory_optimization_b200 — B200-native differentiable visibility/coverage objective.

Drop-in for the hot path of ctu-vras/trajectory_optimization (`src/model.py`, `src/tools.py`):
the Python surface below mirrors the reference's; the compute lives in `libcovb200.so`
(hand-written sm_100a CUDA behind the C ABI declared in `include/coverage_b200.h`).
There is no CPU fallback: without the library or without a CUDA device the ops raise.
"""
from . import _lib  # noqa: F401
from .ops import (coverage_pose, coverage_traj, frustum_cull, spherical_flip, hpr_hull_mask,  # noqa: F401
                  sweep_rewards, coverage_sweep, coverage_pose_batch, traj_logodds)

__all__ = ["coverage_pose", "coverage_traj", "frustum_cull", "spherical_flip", "hpr_hull_mask", "sweep_rewards",
           "coverage_sweep", "coverage_pose_batch", "traj_logodds"]
