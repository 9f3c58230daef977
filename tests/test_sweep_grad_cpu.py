"""The differentiable candidate sweep (ops.coverage_sweep) around the C ABI, on CPU: the two new C-ABI calls are replaced
by an oracle-backed stand-in built from the per-trajectory ones (tests only), so that the autograd plumbing, the block
layout of the accumulators and both shardings over two gloo ranks are exercised without a GPU."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tests._standins import ACC, OracleBackend  # noqa: E402


class SweepOracleBackend(OracleBackend):
    """cov_sweep_fused / cov_sweep_epilogue as their definition states them: cov_traj_fused (W = P) and cov_traj_epilogue
    once per trajectory, blocks of 22 P + 1 accumulators, minmax (2, T P)."""

    def sweep_fused_workspace_bytes(self, pts, T, Pn, dense=None):
        return 0

    @staticmethod
    def _mm(minmax, t, T, Pn):
        TP = T * Pn
        return torch.cat([minmax[t * Pn:(t + 1) * Pn], minmax[TP + t * Pn:TP + (t + 1) * Pn]])

    def sweep_fused(self, pts, P, Q, T, Pn, Kd, cam, boxes, minmax, ws=None):
        scratch = torch.empty(pts.shape[0], dtype=torch.float32)
        blocks = [self.traj_fused(pts, P[t * Pn:(t + 1) * Pn], Q[t * Pn:(t + 1) * Pn], Kd, cam, self._mm(minmax, t, T, Pn),
                                  None, scratch) for t in range(T)]
        return torch.cat(blocks)

    def sweep_epilogue(self, acc, minmax, Q, T, Pn, n_total):
        blk = Pn * ACC + 1
        outs = [self.traj_epilogue(acc[t * blk:(t + 1) * blk], self._mm(minmax, t, T, Pn), Q[t * Pn:(t + 1) * Pn], n_total, 0)
                for t in range(T)]
        return torch.cat([torch.stack([o[0] for o in outs]), torch.cat([o[1:1 + 3 * Pn] for o in outs]),
                          torch.cat([o[1 + 3 * Pn:] for o in outs])])


def _case():
    gen = np.random.default_rng(31)
    pts = (gen.random((900, 3)) * np.array([16, 16, 4]) + np.array([-4, -4, -1])).astype(np.float32)
    T, Pn = 5, 3   # 5 trajectories over 2 ranks: an uneven split
    base = np.stack([np.linspace(0, 6, Pn), np.linspace(0, 3, Pn), np.zeros(Pn)], 1)
    poses = (base[None] + gen.normal(0, 0.8, (T, 1, 3)) * np.array([1, 1, 0])).astype(np.float32)
    quats = (gen.normal(0, 0.3, (T, Pn, 4)) + np.array([1.0, 0, 0, 0])).astype(np.float32)
    weights = np.linspace(1.0, 2.0, T).astype(np.float32)
    return pts, poses, quats, weights


def _sweep(pts, poses, quats, weights, **kw):
    from oracle import coverage_oracle as orc
    from trajectory_optimization_b200 import ops
    P = torch.from_numpy(poses.copy()).requires_grad_(True)
    Q = torch.from_numpy(quats.copy()).requires_grad_(True)
    means = ops.coverage_sweep(torch.from_numpy(pts), P, Q, torch.from_numpy(orc.K_DEFAULT.copy()), orc.IMG_WIDTH,
                               orc.IMG_HEIGHT, presorted=True, **kw)
    (torch.from_numpy(weights) * means).sum().backward()
    return means.detach().numpy(), P.grad.numpy(), Q.grad.numpy()


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from trajectory_optimization_b200 import ops
        ops._BACKEND = SweepOracleBackend()
        pts, poses, quats, weights = _case()
        n = len(pts)
        by_traj = _sweep(pts, poses, quats, weights, group=dist.group.WORLD, shard="trajectories")
        lo, hi = rank * n // world, (rank + 1) * n // world
        by_pts = _sweep(pts[lo:hi].copy(), poses, quats, weights, n_total=n, group=dist.group.WORLD, shard="points")
        q.put((rank, by_traj, by_pts))
    except Exception as e:  # surface the failure instead of letting the parent time out
        q.put((rank, repr(e)))
        raise
    finally:
        dist.destroy_process_group()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


@pytest.fixture
def oracle_backend(monkeypatch):
    from trajectory_optimization_b200 import ops
    monkeypatch.setattr(ops, "_BACKEND", SweepOracleBackend())


def test_unsharded_sweep_equals_per_trajectory_objective(oracle_backend):
    """means[t] and the gradient of sum_t g_t means_t are trajectory t's coverage_traj mean and g_t times its gradient."""
    from oracle import coverage_oracle as orc
    from tests.conftest import rel_err
    from trajectory_optimization_b200 import ops
    pts, poses, quats, weights = _case()
    means, gp, gq = _sweep(pts, poses, quats, weights)
    K = torch.from_numpy(orc.K_DEFAULT.copy())
    for t in range(len(poses)):
        P = torch.from_numpy(poses[t].copy()).requires_grad_(True)
        Q = torch.from_numpy(quats[t].copy()).requires_grad_(True)
        _, mean = ops.coverage_traj(torch.from_numpy(pts), P, Q, K, orc.IMG_WIDTH, orc.IMG_HEIGHT)
        mean.backward()
        assert rel_err(means[t], mean.item()) < 1e-6
        assert rel_err(gp[t], weights[t] * P.grad.numpy()) < 1e-6 and rel_err(gq[t], weights[t] * Q.grad.numpy()) < 1e-6
        ref = orc.traj_objective(pts, poses[t], quats[t], *orc.load_intrinsics(), dtype=np.float64, want_grad=False)
        assert rel_err(means[t], ref["mean"]) < 1e-6


def test_two_rank_sweep_gradients_match_unsharded_run(oracle_backend):
    """Both shardings over two gloo ranks (trajectories: uneven 3 + 2 split, all-gather; points: MIN/MAX + SUM of the
    accumulator blocks) reproduce one unsharded run's means and gradients on every rank."""
    from tests.conftest import rel_err
    pts, poses, quats, weights = _case()
    ref = _sweep(pts, poses, quats, weights)
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = sorted([q.get(timeout=240) for _ in range(world)], key=lambda t: t[0])
    assert all(len(r) == 3 for r in results), results
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for _, by_traj, by_pts in results:
        for got in (by_traj, by_pts):
            for a, b in zip(got, ref):
                assert a.shape == b.shape
                assert rel_err(a, b) < 1e-6


def test_sweep_rejects_bad_shapes(oracle_backend):
    from oracle import coverage_oracle as orc
    from trajectory_optimization_b200 import ops
    pts, poses, quats, _ = _case()
    K = torch.from_numpy(orc.K_DEFAULT.copy())
    P, Q = torch.from_numpy(poses), torch.from_numpy(quats)
    for bad_p, bad_q in ((P, Q[:, :2]), (P[:2], Q), (P.reshape(-1, 3), Q.reshape(-1, 4)), (P, Q[..., :3]),
                         (P[:, :0], Q[:, :0])):
        with pytest.raises(ValueError, match="coverage_sweep"):
            ops.coverage_sweep(torch.from_numpy(pts), bad_p, bad_q, K, orc.IMG_WIDTH, orc.IMG_HEIGHT)
    with pytest.raises(ValueError, match="shard"):
        ops.coverage_sweep(torch.from_numpy(pts), P, Q, K, orc.IMG_WIDTH, orc.IMG_HEIGHT, shard="poses")


def test_sweep_on_cpu_tensors_fails_loudly():
    """The product backend: no CPU fallback, the call raises before anything runs."""
    from oracle import coverage_oracle as orc
    from trajectory_optimization_b200 import ops
    pts, poses, quats, _ = _case()
    with pytest.raises(RuntimeError, match="CUDA-only"):
        ops.coverage_sweep(torch.from_numpy(pts), torch.from_numpy(poses), torch.from_numpy(quats),
                           torch.from_numpy(orc.K_DEFAULT.copy()), orc.IMG_WIDTH, orc.IMG_HEIGHT)


def test_model_traj_batch_rejects_differing_strides_and_bad_shapes(oracle_backend):
    from oracle import coverage_oracle as orc
    from trajectory_optimization_b200 import model
    pts, poses, quats, _ = _case()
    K = torch.from_numpy(orc.K_DEFAULT.copy())
    with pytest.raises(ValueError, match="W >= 3"):
        model.ModelTrajBatch(pts, poses[:, :2], quats[:, :2], K, orc.IMG_WIDTH, orc.IMG_HEIGHT, device=torch.device("cpu"))
    with pytest.raises(ValueError, match="same T and W"):
        model.ModelTrajBatch(pts, poses, quats[:2], K, orc.IMG_WIDTH, orc.IMG_HEIGHT, device=torch.device("cpu"))
    stretched = poses.copy()
    stretched[1] *= 4.0   # a 4x longer trajectory: waypoints 4x further apart
    m = model.ModelTrajBatch(pts, stretched, quats, K, orc.IMG_WIDTH, orc.IMG_HEIGHT, device=torch.device("cpu"))
    with pytest.raises(ValueError, match="strides differ"):
        m(vis_wps_dist=6.0)


def test_model_traj_batch_stride_equals_model_traj_on_evenly_spaced_waypoints():
    """The visibility stride is ModelTraj's, rounding included: waypoints 0.1 m apart at vis_wps_dist = 0.5 give an fp32
    quotient of exactly 5 (stride 6) where an fp64 division gives 4.999... (stride 5)."""
    from oracle import coverage_oracle as orc
    from trajectory_optimization_b200 import model
    K = torch.from_numpy(orc.K_DEFAULT.copy())
    pts = torch.zeros(10, 3)
    cpu = torch.device("cpu")
    cases = [(W, torch.arange(W, dtype=torch.float32) * 0.1) for W in range(4, 40)] + [(7, torch.linspace(0, 1, 7))]
    for W, xs in cases:
        p = torch.zeros(W, 3)
        p[:, 0] = xs
        q = torch.tensor([1.0, 0, 0, 0]).repeat(W, 1)
        ref = model.ModelTraj(pts, p, q, K, orc.IMG_WIDTH, orc.IMG_HEIGHT, device=cpu)
        batch = model.ModelTrajBatch(pts, torch.stack([p, p + torch.tensor([0.0, 2.0, 0.0])]), q.repeat(2, 1, 1), K,
                                     orc.IMG_WIDTH, orc.IMG_HEIGHT, device=cpu)
        for dist_ in (0.5, 0.3, 1.0):
            assert batch._wps_step(dist_) == ref._wps_step(dist_), (W, dist_)
