"""The trajectory objective with per-point weights, restated on top of the prior oracle — TEST INFRASTRUCTURE.

`traj_objective_weighted` is the weighted mean mean_w = sum_j w_j r_j / sum_j w_j (r_j as in tests/_prior_oracle.py, with
or without a prior) and the gradients of vis = 1/(mean_w + eps): pass B's partials with G_j = w_j r_j (1 - r_j) and the
epilogue with sum_j w_j in place of N.  `WeightOracleBackend` is the CPU stand-in of ops.CudaBackend with the weight
arguments.  Nothing under trajectory_optimization_b200/ imports this file."""
import numpy as np
import torch

from oracle import coverage_oracle as orc
from tests._prior_oracle import PriorOracleBackend, traj_partials_prior


def traj_objective_weighted(points, poses, quats, K, img_width, img_height, weight, prior=None, min_dist=1.0,
                            max_dist=5.0, dtype=np.float64):
    """dict(rewards, mean, vis, g_poses, g_quats) of the weighted objective (gradients of vis)."""
    w = np.asarray(weight, dtype=np.float64)
    part = traj_partials_prior(points, poses, quats, K, img_width, img_height, min_dist, max_dist, dtype=dtype,
                               upstream=w, prior=prior)
    part["sum_r"] = (w * part["rewards"].astype(np.float64)).sum()
    out = orc.traj_grads_from_partials(part, poses, quats, w.sum())
    out["rewards"] = part["rewards"]
    return out


class WeightOracleBackend(PriorOracleBackend):
    """ops.CudaBackend's weight arguments on the oracle: G_j times w_j, the reward sum weighted, the epilogues' denominator
    read from the (1,) tensor."""

    def weight_sums(self, weight, prior=None):
        w = weight.double().numpy()
        r0 = 0.5 if prior is None else 1.0 / (1.0 + np.exp(-prior.double().numpy()))
        return torch.tensor([(w * r0).sum(), w.sum()], dtype=torch.float64)

    def traj_fused(self, pts, P, Q, Kd, cam, minmax, upstream, rewards, reward_index=None, boxes=None, ws=None,
                   dense=None, prefilled=False, prior=None, prior_sum=None, weight=None, wsums=None):
        if weight is None:
            return super().traj_fused(pts, P, Q, Kd, cam, minmax, upstream, rewards, prior=prior, prior_sum=prior_sum)
        assert upstream is None
        acc = super().traj_fused(pts, P, Q, Kd, cam, minmax, weight, rewards, prior=prior, prior_sum=prior_sum)
        acc[-1] = float((weight.double() * rewards.double()).sum())
        return acc

    def sweep_sums(self, pts, P, Q, T, Pn, Kd, cam, boxes, minmax, prior=None, prior_sum=None, weight=None, wsums=None):
        if weight is None:
            return super().sweep_sums(pts, P, Q, T, Pn, Kd, cam, boxes, minmax, prior, prior_sum)
        W, w = len(P), weight.double().numpy()
        x0 = 0.0 if prior is None else prior.double().numpy()
        sums = np.zeros(T)
        for t in range(T):
            mm = torch.cat([minmax[t * Pn:(t + 1) * Pn], minmax[W + t * Pn:W + (t + 1) * Pn]])
            L, _ = self._logodds(pts, P[t * Pn:(t + 1) * Pn], Q[t * Pn:(t + 1) * Pn], Kd, cam, mm)
            sums[t] = (w / (1 + np.exp(-(x0 + L)))).sum()
        return torch.from_numpy(sums)

    def sweep_fused(self, pts, P, Q, T, Pn, Kd, cam, boxes, minmax, ws=None, prior=None, prior_sum=None, weight=None,
                    wsums=None):
        if weight is None:
            return super().sweep_fused(pts, P, Q, T, Pn, Kd, cam, boxes, minmax, ws, prior, prior_sum)
        scratch = torch.empty(pts.shape[0], dtype=torch.float32)
        return torch.cat([self.traj_fused(pts, P[t * Pn:(t + 1) * Pn], Q[t * Pn:(t + 1) * Pn], Kd, cam,
                                          self._mm(minmax, t, T, Pn), None, scratch, prior=prior, weight=weight,
                                          wsums=wsums)
                          for t in range(T)])

    def traj_epilogue(self, acc, minmax, Q, n_total, upstream_mode, den=None):
        if den is None:
            return super().traj_epilogue(acc, minmax, Q, n_total, upstream_mode)
        return super().traj_epilogue(acc, minmax, Q, float(den[0]), 0)

    def sweep_epilogue(self, acc, minmax, Q, T, Pn, n_total, den=None):
        return super().sweep_epilogue(acc, minmax, Q, T, Pn, n_total if den is None else float(den[0]))


class ReversingWeightOracleBackend(WeightOracleBackend):
    """The stand-in with a cloud ordering that reverses the points, so that the ops' permutation of the weight (and of
    the prior) with the cloud is exercised."""

    def order_cloud(self, pts, spatial_sort_cloud=True):
        perm = torch.arange(pts.shape[0] - 1, -1, -1, dtype=torch.int32)
        return pts[perm.long()].contiguous(), perm, None
