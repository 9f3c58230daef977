"""The prefix sweep (ops.sweep_prefix_rewards, ModelTrajBatch.prefix_means) around the C ABI, on CPU: the new C-ABI call is
replaced by an oracle-backed stand-in built from truncated sweeps (tests only), so that the shared sweep plumbing (cloud
ordering, prior and weight sums, both shardings over two gloo ranks) and the argument checks run without a GPU."""
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

from tests._prior_oracle import traj_objective_prior  # noqa: E402
from tests._weight_oracle import ReversingWeightOracleBackend, WeightOracleBackend, traj_objective_weighted  # noqa: E402


def _truncated_sums(B, pts, P, Q, T, Pn, Kd, cam, boxes, minmax, prior, base, weight):
    """cov_sweep_prefix_rewards as its definition states it: entry t Pn + i = the sweep sum of trajectory t cut after
    pose i, from the stand-in's sweep_sums on the truncated trajectories (normalisers are per pose: sliced)."""
    W = T * Pn
    mins, maxs = minmax[:W].reshape(T, Pn), minmax[W:].reshape(T, Pn)
    out = torch.zeros(T, Pn, dtype=torch.float64)
    for i in range(Pn):
        Pt = P.reshape(T, Pn, 3)[:, :i + 1].reshape(-1, 3)
        Qt = Q.reshape(T, Pn, 4)[:, :i + 1].reshape(-1, 4)
        mm = torch.cat([mins[:, :i + 1].reshape(-1), maxs[:, :i + 1].reshape(-1)])
        if weight is not None:
            s = B.sweep_sums(pts, Pt, Qt, T, i + 1, Kd, cam, boxes, mm, prior=prior, weight=weight, wsums=base)
        elif prior is not None:
            s = B.sweep_sums(pts, Pt, Qt, T, i + 1, Kd, cam, boxes, mm, prior, base)
        else:
            assert base is None
            s = B.sweep_sums(pts, Pt, Qt, T, i + 1, Kd, cam, boxes, mm)
        out[:, i] = s
    return out.reshape(-1)


class PrefixOracleBackend(WeightOracleBackend):
    def sweep_prefix_sums(self, pts, P, Q, T, Pn, Kd, cam, boxes, minmax, prior=None, base=None, weight=None):
        return _truncated_sums(self, pts, P, Q, T, Pn, Kd, cam, boxes, minmax, prior, base, weight)


class ReversingPrefixOracleBackend(ReversingWeightOracleBackend):
    def sweep_prefix_sums(self, pts, P, Q, T, Pn, Kd, cam, boxes, minmax, prior=None, base=None, weight=None):
        return _truncated_sums(self, pts, P, Q, T, Pn, Kd, cam, boxes, minmax, prior, base, weight)


def _case(seed=5):
    gen = np.random.default_rng(seed)
    pts = (gen.random((600, 3)) * np.array([16, 16, 4]) + np.array([-4, -4, -1])).astype(np.float32)
    T, Pn = 5, 4   # 5 trajectories over 2 ranks: an uneven split
    base = np.stack([np.linspace(0, 6, Pn), np.linspace(0, 3, Pn), np.zeros(Pn)], 1)
    poses = (base[None] + gen.normal(0, 0.8, (T, 1, 3)) * np.array([1, 1, 0])).astype(np.float32)
    quats = (gen.normal(0, 0.3, (T, Pn, 4)) + np.array([1.0, 0, 0, 0])).astype(np.float32)
    prior = gen.normal(0, 2, len(pts)).astype(np.float32)
    weight = (gen.random(len(pts)) * 3).astype(np.float32)
    return pts, poses, quats, prior, weight


def _k():
    from oracle import coverage_oracle as orc
    return orc.K_DEFAULT.copy(), orc.IMG_WIDTH, orc.IMG_HEIGHT


def _kw(prior, weight, variant):
    return {"plain": {}, "prior": dict(prior_logodds=torch.from_numpy(prior)),
            "weight": dict(weight=torch.from_numpy(weight)),
            "both": dict(prior_logodds=torch.from_numpy(prior), weight=torch.from_numpy(weight))}[variant]


@pytest.fixture
def prefix_backend(monkeypatch):
    from trajectory_optimization_b200 import ops
    monkeypatch.setattr(ops, "_BACKEND", PrefixOracleBackend())


@pytest.mark.parametrize("variant", ["plain", "prior", "weight", "both"])
def test_prefix_columns_are_truncated_sweeps_and_the_oracle(prefix_backend, variant):
    """[:, i] is sweep_rewards of the trajectories cut after pose i ([:, -1]: of the whole trajectories), and each entry
    is the oracle's mean (weighted mean) of that prefix."""
    from tests.conftest import rel_err
    from trajectory_optimization_b200 import ops
    pts, poses, quats, prior, weight = _case()
    K, Wd, Hd = _k()
    args = (torch.from_numpy(pts), torch.from_numpy(poses), torch.from_numpy(quats), torch.from_numpy(K), Wd, Hd)
    kw = _kw(prior, weight, variant)
    got = ops.sweep_prefix_rewards(*args, presorted=True, **kw)
    T, Pn = poses.shape[:2]
    assert got.shape == (T, Pn) and got.dtype == torch.float64
    assert rel_err(got[:, -1].numpy(), ops.sweep_rewards(*args, presorted=True, **kw).numpy()) < 1e-12
    p64 = prior.astype(np.float64) if "prior_logodds" in kw else None
    for i in range(Pn):
        cut = ops.sweep_rewards(args[0], args[1][:, :i + 1], args[2][:, :i + 1], *args[3:], presorted=True, **kw)
        assert rel_err(got[:, i].numpy(), cut.numpy()) < 1e-12
        for t in range(T):
            if "weight" in kw:
                ref = traj_objective_weighted(pts, poses[t, :i + 1], quats[t, :i + 1], K, Wd, Hd, weight, prior=p64)
            else:
                ref = traj_objective_prior(pts, poses[t, :i + 1], quats[t, :i + 1], K, Wd, Hd, prior=p64)
            assert rel_err(got[t, i].item(), ref["mean"]) < 1e-6
    # coverage only grows along a trajectory
    assert bool((got[:, 1:] >= got[:, :-1] - 1e-9).all())


def test_prefix_sweep_permutes_prior_and_weight_with_the_cloud(monkeypatch):
    from tests.conftest import rel_err
    from trajectory_optimization_b200 import ops
    pts, poses, quats, prior, weight = _case()
    K, Wd, Hd = _k()
    args = (torch.from_numpy(pts), torch.from_numpy(poses), torch.from_numpy(quats), torch.from_numpy(K), Wd, Hd)
    kw = _kw(prior, weight, "both")
    monkeypatch.setattr(ops, "_BACKEND", PrefixOracleBackend())
    ref = ops.sweep_prefix_rewards(*args, presorted=True, **kw)
    monkeypatch.setattr(ops, "_BACKEND", ReversingPrefixOracleBackend())
    got = ops.sweep_prefix_rewards(*args, **kw)
    assert rel_err(got.numpy(), ref.numpy()) < 1e-12


def test_prefix_sweep_argument_errors(prefix_backend):
    from trajectory_optimization_b200 import ops
    pts, poses, quats, prior, weight = _case()
    K, Wd, Hd = _k()
    X, P, Q, Kt = torch.from_numpy(pts), torch.from_numpy(poses), torch.from_numpy(quats), torch.from_numpy(K)
    for bad_p, bad_q in ((P, Q[:, :2]), (P[:2], Q), (P.reshape(-1, 3), Q.reshape(-1, 4)), (P, Q[..., :3]),
                         (P[:, :0], Q[:, :0]), (P[:0], Q[:0]), (poses, Q)):
        with pytest.raises(ValueError, match="sweep_prefix_rewards"):
            ops.sweep_prefix_rewards(X, bad_p, bad_q, Kt, Wd, Hd, presorted=True)
    with pytest.raises(ValueError, match="shard"):
        ops.sweep_prefix_rewards(X, P, Q, Kt, Wd, Hd, shard="poses")
    with pytest.raises(ValueError, match="prior_logodds"):
        ops.sweep_prefix_rewards(X, P, Q, Kt, Wd, Hd, prior_logodds=torch.from_numpy(prior[:-1]))
    with pytest.raises(ValueError, match="weight"):
        ops.sweep_prefix_rewards(X, P, Q, Kt, Wd, Hd, weight=torch.from_numpy(weight).double())


def test_prefix_sweep_on_cpu_tensors_fails_loudly():
    """The product backend: no CPU fallback, the call raises before anything runs."""
    from trajectory_optimization_b200 import ops
    pts, poses, quats, _, _ = _case()
    K, Wd, Hd = _k()
    with pytest.raises(RuntimeError, match="CUDA-only"):
        ops.sweep_prefix_rewards(torch.from_numpy(pts), torch.from_numpy(poses), torch.from_numpy(quats),
                                 torch.from_numpy(K), Wd, Hd)


@pytest.mark.parametrize("variant", ["plain", "both"])
def test_model_traj_batch_prefix_means(prefix_backend, variant):
    """prefix_means is the op on the strided waypoints with the model's prior and weight; its last column is `means`."""
    from tests.conftest import rel_err
    from trajectory_optimization_b200 import model, ops
    pts, poses, quats, prior, weight = _case()
    K, Wd, Hd = _k()
    T = poses.shape[0]
    # 7 evenly spaced waypoints (0.5 m apart) per trajectory: stride 2 at vis_wps_dist = 0.9 evaluates waypoints 0, 2, 4, 6
    xs = np.arange(7, dtype=np.float32) * 0.5
    wp = np.stack([np.stack([xs, np.full(7, 0.3 * t, np.float32), np.zeros(7, np.float32)], 1) for t in range(T)])
    wq = np.broadcast_to(quats[:, :1], (T, 7, 4)).copy()
    m = model.ModelTrajBatch(pts, torch.from_numpy(wp), torch.from_numpy(wq), torch.from_numpy(K), Wd, Hd,
                             device=torch.device("cpu"))
    kw = {}
    if variant == "both":
        m.set_prior_logodds(torch.from_numpy(prior))
        m.set_point_weight(torch.from_numpy(weight))
        kw = _kw(prior, weight, "both")
    m(vis_wps_dist=0.9)
    got = m.prefix_means(vis_wps_dist=0.9)
    step = m._wps_step(0.9)
    assert step == 2 and got.shape == (T, 4)
    ref = ops.sweep_prefix_rewards(torch.from_numpy(pts), torch.from_numpy(wp[:, ::step]), torch.from_numpy(wq[:, ::step]),
                                   torch.from_numpy(K), Wd, Hd, presorted=True, **kw)
    assert rel_err(got.numpy(), ref.numpy()) < 1e-12
    assert rel_err(got[:, -1].numpy(), m.means.detach().numpy()) < 1e-6
    assert not got.requires_grad


def _run(pts, poses, quats, prior, weight, **kw):
    from trajectory_optimization_b200 import ops
    K, Wd, Hd = _k()
    out = []
    for variant in ("plain", "both"):
        out.append(ops.sweep_prefix_rewards(torch.from_numpy(pts), torch.from_numpy(poses), torch.from_numpy(quats),
                                            torch.from_numpy(K), Wd, Hd, presorted=True, **_kw(prior, weight, variant),
                                            **kw).numpy())
    return out


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from trajectory_optimization_b200 import ops
        ops._BACKEND = PrefixOracleBackend()
        pts, poses, quats, prior, weight = _case()
        n = len(pts)
        g = dist.group.WORLD
        by_traj = _run(pts, poses, quats, prior, weight, group=g, shard="trajectories")
        sl = slice(rank * n // world, (rank + 1) * n // world)
        by_pts = _run(pts[sl].copy(), poses, quats, prior[sl].copy(), weight[sl].copy(), n_total=n, group=g,
                      shard="points")
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


def test_two_rank_prefix_sweeps_match_unsharded(prefix_backend):
    """Both shardings over two gloo ranks (trajectories: uneven 3 + 2 split, all-gather of the rank blocks; points: MAX
    of the normalisers, SUM of the T P sums and of the weighted denominator) reproduce one unsharded run."""
    from tests.conftest import rel_err
    pts, poses, quats, prior, weight = _case()
    ref = _run(pts, poses, quats, prior, weight)
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
                assert a.shape == b.shape and rel_err(a, b) < 1e-12
