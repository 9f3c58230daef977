"""The trajectory objective with prior log-odds (map memory), restated on top of the numpy oracle — TEST INFRASTRUCTURE.

`traj_partials_prior` is `oracle.coverage_oracle.traj_partials` with the prior entering after the fusion: L_j = sum_w lo_jw
in pose order, then x_j = prior_j + L_j, r_j = 1/(1 + exp(-x_j)), G_j = r_j (1 - r_j); everything per pose is unchanged.
`PriorOracleBackend` is the CPU stand-in of ops.CudaBackend with the prior arguments, for the autograd plumbing and the
collectives over gloo.  Nothing under trajectory_optimization_b200/ imports this file."""
import numpy as np
import torch

from oracle import coverage_oracle as orc
from tests._standins import ACC
from tests.test_sweep_grad_cpu import SweepOracleBackend


def traj_partials_prior(points, poses, quats, K, img_width, img_height, min_dist=1.0, max_dist=5.0, eps=1e-6,
                        dtype=np.float64, minmax=None, want_grad=True, upstream=None, prior=None):
    """orc.traj_partials with a per-point prior (None: none at all, the oracle's own arithmetic)."""
    dt = np.dtype(dtype).type
    W = len(poses)
    pts = np.asarray(points, dtype=dtype)
    N = len(pts)
    if minmax is None:
        mins, maxs = orc.traj_minmax(pts, poses, quats, K, img_width, img_height, min_dist, max_dist, eps, dtype)
    else:
        mins, maxs = (np.asarray(v, dtype=dtype) for v in minmax)
    hi = dt(np.float32(1.0 - eps)) if dtype == np.float32 else dt(1.0 - eps)
    L = np.zeros(N, dtype=dtype)
    keep = []
    for w in range(W):
        m, y, g_c, R, q, qn = orc.visibility(pts, poses[w], quats[w], K, img_width, img_height, min_dist, max_dist, eps,
                                             dtype, want_grad=True)
        a = mins[w]
        pm = m - a
        b = dt(maxs[w] - a)
        with np.errstate(divide="ignore", invalid="ignore"):
            p = pm / b
        qc = np.clip(p, dt(0.5), hi)
        L = L + np.log(qc / (dt(1) - qc))
        keep.append((m, y, g_c, p, qc, pm, a, b))
    x = L if prior is None else np.asarray(prior, dtype=dtype) + L
    r = dt(1) / (dt(1) + np.exp(-x))
    out = dict(rewards=r, logodds=x, sum_r=r.sum(dtype=np.float64), mins=mins, maxs=maxs, n=N)
    if not want_grad:
        return out
    G = (r * (dt(1) - r)).astype(np.float64)
    if upstream is not None:
        G = G * np.asarray(upstream, dtype=np.float64)
    acc = dict(main_g=np.zeros((W, 3)), main_yg=np.zeros((W, 3, 3)), se=np.zeros(W), sep=np.zeros(W),
               amax_g=np.zeros((W, 3)), amax_yg=np.zeros((W, 3, 3)), amax_n=np.zeros(W),
               amin_g=np.zeros((W, 3)), amin_yg=np.zeros((W, 3, 3)), amin_n=np.zeros(W))
    for w, (m, y, g_c, p, qc, pm, a, b) in enumerate(keep):
        y64, g64 = y.astype(np.float64), g_c.astype(np.float64)
        gate = (p >= dt(0.5)) & (p <= hi)
        qc64 = qc.astype(np.float64)
        e = np.where(gate, G / (qc64 * (1.0 - qc64)), 0.0)
        om = e / float(b)
        acc["main_g"][w] = (om[:, None] * g64).sum(axis=0)
        acc["main_yg"][w] = np.einsum("j,ja,jb->ab", om, y64, g64)
        acc["se"][w] = e.sum()
        acc["sep"][w] = (e * p.astype(np.float64)).sum()
        tmax, tmin = pm == b, m == a
        acc["amax_g"][w] = g64[tmax].sum(axis=0)
        acc["amax_yg"][w] = np.einsum("ja,jb->ab", y64[tmax], g64[tmax])
        acc["amax_n"][w] = tmax.sum()
        acc["amin_g"][w] = g64[tmin].sum(axis=0)
        acc["amin_yg"][w] = np.einsum("ja,jb->ab", y64[tmin], g64[tmin])
        acc["amin_n"][w] = tmin.sum()
    out.update(acc)
    return out


def traj_objective_prior(points, poses, quats, K, img_width, img_height, prior=None, dtype=np.float64, n_total=None,
                         minmax=None, want_grad=True):
    """orc.traj_objective with a prior: dict(rewards, logodds, mean, vis, g_poses, g_quats) (gradients of vis)."""
    part = traj_partials_prior(points, poses, quats, K, img_width, img_height, dtype=dtype, minmax=minmax,
                               want_grad=want_grad, prior=prior)
    out = orc.traj_grads_from_partials(part, poses, quats, len(points) if n_total is None else n_total,
                                       want_grad=want_grad)
    out["rewards"], out["logodds"] = part["rewards"], part["logodds"]
    return out


class PriorOracleBackend(SweepOracleBackend):
    """ops.CudaBackend's prior arguments on the oracle: the prior is added to L before the sigmoid, the reward-sum base
    is sum_j sigmoid(prior_j)."""

    def prior_sum(self, prior):
        return torch.tensor([float((1.0 / (1.0 + np.exp(-prior.double().numpy()))).sum())], dtype=torch.float64)

    def _logodds(self, pts, P, Q, Kd, cam, minmax):
        W, hi = len(P), float(np.float32(1.0 - cam.eps))
        L, keep = np.zeros(len(pts)), []
        for w in range(W):
            m, y, gy = self._vis(pts, P[w], Q[w], Kd, cam)
            a, b = float(minmax[w]), float(minmax[W + w]) - float(minmax[w])
            p = (m - a) / b
            qc = np.clip(p, 0.5, hi)
            L += np.log(qc / (1 - qc))
            keep.append((m, y, gy, p, qc, a, b))
        return L, keep

    def traj_minmax(self, pts, P, Q, Kd, cam, boxes=None, ws=None, dense=None, prefill=None, prior=None):
        return super().traj_minmax(pts, P, Q, Kd, cam)

    def traj_fused(self, pts, P, Q, Kd, cam, minmax, upstream, rewards, reward_index=None, boxes=None, ws=None,
                   dense=None, prefilled=False, prior=None, prior_sum=None):
        if prior is None:
            return super().traj_fused(pts, P, Q, Kd, cam, minmax, upstream, rewards)
        W, hi = len(P), float(np.float32(1.0 - cam.eps))
        L, keep = self._logodds(pts, P, Q, Kd, cam, minmax)
        r = 1 / (1 + np.exp(-(prior.double().numpy() + L)))
        rewards.copy_(torch.from_numpy(r.astype(np.float32)))
        G = r * (1 - r) * (1.0 if upstream is None else upstream.double().numpy())
        acc = np.zeros(W * ACC + 1)
        for w, (m, y, gy, p, qc, a, b) in enumerate(keep):
            gate = (p >= 0.5) & (p <= hi)
            e = np.where(gate, G / (qc * (1 - qc)), 0.0)
            row = acc[w * ACC:(w + 1) * ACC]
            row[0:3], row[3:6] = ((e / b)[:, None] * gy).sum(0), ((e / b)[:, None] * np.cross(gy, y)).sum(0)
            row[6], row[7] = e.sum(), (e * p).sum()
            for off, sel in ((8, (m - a) == b), (15, (m == a) & (a > 0))):
                row[off:off + 3], row[off + 3:off + 6], row[off + 6] = gy[sel].sum(0), np.cross(gy[sel], y[sel]).sum(0), sel.sum()
        acc[W * ACC] = r.sum()
        return torch.from_numpy(acc)

    def traj_logodds(self, pts, P, Q, Kd, cam, minmax, out, reward_index=None, boxes=None, ws=None, dense=None):
        L, _ = self._logodds(pts, P, Q, Kd, cam, minmax)
        out += torch.from_numpy(L.astype(np.float32))
        return out

    def sweep_sums(self, pts, P, Q, T, Pn, Kd, cam, boxes, minmax, prior=None, prior_sum=None):
        if prior is None:
            return super().sweep_sums(pts, P, Q, T, Pn, Kd, cam, boxes, minmax)
        W = len(P)
        sums = np.zeros(T)
        for t in range(T):
            mm = torch.cat([minmax[t * Pn:(t + 1) * Pn], minmax[W + t * Pn:W + (t + 1) * Pn]])
            L, _ = self._logodds(pts, P[t * Pn:(t + 1) * Pn], Q[t * Pn:(t + 1) * Pn], Kd, cam, mm)
            sums[t] = (1 / (1 + np.exp(-(prior.double().numpy() + L)))).sum()
        return torch.from_numpy(sums)

    def sweep_fused(self, pts, P, Q, T, Pn, Kd, cam, boxes, minmax, ws=None, prior=None, prior_sum=None):
        if prior is None:
            return super().sweep_fused(pts, P, Q, T, Pn, Kd, cam, boxes, minmax, ws)
        scratch = torch.empty(pts.shape[0], dtype=torch.float32)
        return torch.cat([self.traj_fused(pts, P[t * Pn:(t + 1) * Pn], Q[t * Pn:(t + 1) * Pn], Kd, cam,
                                          self._mm(minmax, t, T, Pn), None, scratch, prior=prior, prior_sum=prior_sum)
                          for t in range(T)])
