"""Per-point weights around the C ABI, on CPU: the weighted oracle (weight of ones = the unweighted oracle, closed-form
gradients against fp64 autograd), the ops' plumbing on an oracle-backed stand-in (tests/_weight_oracle.py): the weight
permuted with the cloud, argument errors, the models' checks, and the point and trajectory shardings over two gloo
ranks (the global sum_j w_j)."""
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
from tests._weight_oracle import (ReversingWeightOracleBackend, WeightOracleBackend,  # noqa: E402
                                  traj_objective_weighted)


def _case(seed=11):
    gen = np.random.default_rng(seed)
    pts = (gen.random((700, 3)) * np.array([16, 16, 4]) + np.array([-4, -4, -1])).astype(np.float32)
    T, Pn = 3, 4
    base = np.stack([np.linspace(0, 6, Pn), np.linspace(0, 3, Pn), np.zeros(Pn)], 1)
    poses = (base[None] + gen.normal(0, 0.8, (T, 1, 3)) * np.array([1, 1, 0])).astype(np.float32)
    quats = (gen.normal(0, 0.3, (T, Pn, 4)) + np.array([1.0, 0, 0, 0])).astype(np.float32)
    prior = gen.normal(0, 2, len(pts)).astype(np.float32)
    weight = gen.random(len(pts)).astype(np.float32) * 3
    weight[gen.choice(len(pts), 100, replace=False)] = 0.0
    return pts, poses, quats, prior, weight


def _k():
    from oracle import coverage_oracle as orc
    return orc.K_DEFAULT.copy(), orc.IMG_WIDTH, orc.IMG_HEIGHT


@pytest.fixture
def weight_backend(monkeypatch):
    from trajectory_optimization_b200 import ops
    monkeypatch.setattr(ops, "_BACKEND", WeightOracleBackend())


@pytest.mark.parametrize("with_prior", [False, True])
def test_oracle_weight_of_ones_equals_unweighted_exactly(with_prior):
    pts, poses, quats, prior, _ = _case()
    K, Wd, Hd = _k()
    pr = prior.astype(np.float64) if with_prior else None
    ref = traj_objective_prior(pts, poses[0], quats[0], K, Wd, Hd, prior=pr)
    got = traj_objective_weighted(pts, poses[0], quats[0], K, Wd, Hd, np.ones(len(pts)), prior=pr)
    for key in ("rewards", "mean", "vis", "g_poses", "g_quats"):
        assert np.array_equal(np.asarray(got[key]), np.asarray(ref[key])), key


@pytest.mark.parametrize("with_prior", [False, True])
def test_oracle_weighted_gradients_match_fp64_autograd(with_prior):
    """Closed-form fp64 gradients of vis = 1/(sum_j w_j r_j / sum_j w_j + eps) against torch autograd."""
    from oracle import torch_port
    from tests.conftest import rel_err
    pts, poses, quats, prior, weight = _case()
    K, Wd, Hd = _k()
    pr = prior.astype(np.float64) if with_prior else None
    ref = traj_objective_weighted(pts, poses[0], quats[0], K, Wd, Hd, weight, prior=pr)
    P = torch.from_numpy(poses[0].astype(np.float64)).requires_grad_(True)
    Q = torch.from_numpy(quats[0].astype(np.float64)).requires_grad_(True)
    X = torch.from_numpy(pts.astype(np.float64))
    Kt = torch.from_numpy(K.astype(np.float64))
    lo = torch.zeros(len(pts), dtype=torch.float64) if pr is None else torch.from_numpy(pr)
    for i in range(len(P)):
        m = torch_port.visibility(X, Q[i].unsqueeze(0), P[i].unsqueeze(0), Kt, Wd, Hd, 1.0, 5.0, 1e-6)
        p = (m - m.min()) / (m - m.min()).max()
        p = torch.clip(p, 0.5, 1.0 - 1e-6)
        lo = lo + torch.log(p / (1.0 - p))
    w = torch.from_numpy(weight.astype(np.float64))
    vis = 1.0 / ((w / (1.0 + torch.exp(-lo))).sum() / w.sum() + 1e-6)
    vis.backward()
    assert rel_err(ref["vis"], vis.item()) < 1e-12
    assert rel_err(ref["g_poses"], P.grad.numpy()) < 1e-12
    assert rel_err(ref["g_quats"], Q.grad.numpy()) < 1e-12


def test_ops_with_weight_agree_with_oracle(weight_backend):
    from tests.conftest import rel_err
    from trajectory_optimization_b200 import ops
    pts, poses, quats, prior, weight = _case()
    K, Wd, Hd = _k()
    Kt, X, pr, w = torch.from_numpy(K), torch.from_numpy(pts), torch.from_numpy(prior), torch.from_numpy(weight)
    for with_prior in (False, True):
        kw = dict(prior_logodds=pr) if with_prior else {}
        p64 = prior.astype(np.float64) if with_prior else None
        refs = [traj_objective_weighted(pts, poses[t], quats[t], K, Wd, Hd, weight, prior=p64) for t in range(len(poses))]
        for t, ref in enumerate(refs):
            P = torch.from_numpy(poses[t].copy()).requires_grad_(True)
            Q = torch.from_numpy(quats[t].copy()).requires_grad_(True)
            rewards, mean = ops.coverage_traj(X, P, Q, Kt, Wd, Hd, weight=w, **kw)
            (1.0 / (mean + 1e-6)).backward()
            assert rel_err(rewards.detach().numpy(), ref["rewards"]) < 1e-5 and rel_err(mean.item(), ref["mean"]) < 1e-5
            assert rel_err(P.grad.numpy(), ref["g_poses"]) < 1e-4 and rel_err(Q.grad.numpy(), ref["g_quats"]) < 1e-4
            # the rewards do not depend on the weight
            r0, _ = ops.coverage_traj(X, P.detach(), Q.detach(), Kt, Wd, Hd, **kw)
            assert torch.equal(rewards.detach(), r0)
        means = ops.sweep_rewards(X, torch.from_numpy(poses), torch.from_numpy(quats), Kt, Wd, Hd, presorted=True,
                                  weight=w, **kw)
        assert rel_err(means.numpy(), [r["mean"] for r in refs]) < 1e-5
        P = torch.from_numpy(poses.copy()).requires_grad_(True)
        Q = torch.from_numpy(quats.copy()).requires_grad_(True)
        means = ops.coverage_sweep(X, P, Q, Kt, Wd, Hd, presorted=True, weight=w, **kw)
        (1.0 / (means + 1e-6)).sum().backward()
        assert rel_err(means.detach().numpy(), [r["mean"] for r in refs]) < 1e-5
        for t, ref in enumerate(refs):
            assert rel_err(P.grad[t].numpy(), ref["g_poses"]) < 1e-4 and rel_err(Q.grad[t].numpy(), ref["g_quats"]) < 1e-4


def test_sweeps_permute_the_weight_with_the_cloud(monkeypatch):
    """A sweep that orders the cloud itself permutes the weight (and the prior) with it: the result equals the call on
    the cloud as given."""
    from tests.conftest import rel_err
    from trajectory_optimization_b200 import ops
    pts, poses, quats, prior, weight = _case()
    K, Wd, Hd = _k()
    args = (torch.from_numpy(pts), torch.from_numpy(poses), torch.from_numpy(quats), torch.from_numpy(K), Wd, Hd)
    kw = dict(weight=torch.from_numpy(weight), prior_logodds=torch.from_numpy(prior))
    monkeypatch.setattr(ops, "_BACKEND", WeightOracleBackend())
    ref_s = ops.sweep_rewards(*args, presorted=True, **kw)
    ref_m = ops.coverage_sweep(*args, presorted=True, **kw)
    monkeypatch.setattr(ops, "_BACKEND", ReversingWeightOracleBackend())
    got_s = ops.sweep_rewards(*args, **kw)
    got_m = ops.coverage_sweep(*args, **kw)
    assert rel_err(got_s.numpy(), ref_s.numpy()) < 1e-12
    assert rel_err(got_m.detach().numpy(), ref_m.detach().numpy()) < 1e-6
    # and the permutation matters: the reversed cloud with the weight as given is another objective
    bad = ops.sweep_rewards(torch.from_numpy(pts[::-1].copy()), *args[1:], presorted=True, **kw)
    assert rel_err(bad.numpy(), ref_s.numpy()) > 1e-3


def test_weight_argument_errors_name_the_argument(weight_backend):
    from trajectory_optimization_b200 import ops
    pts, poses, quats, _, weight = _case()
    K, Wd, Hd = _k()
    Kt, X, P, Q = torch.from_numpy(K), torch.from_numpy(pts), torch.from_numpy(poses), torch.from_numpy(quats)
    bad = [torch.from_numpy(weight).double(), torch.from_numpy(weight[:-1]), torch.from_numpy(weight).reshape(-1, 1),
           weight]
    bad.append(torch.from_numpy(weight).cuda() if torch.cuda.is_available() else torch.from_numpy(weight).to("meta"))
    for b in bad:
        with pytest.raises(ValueError, match="weight"):
            ops.coverage_traj(X, P[0], Q[0], Kt, Wd, Hd, weight=b)
        with pytest.raises(ValueError, match="weight"):
            ops.sweep_rewards(X, P, Q, Kt, Wd, Hd, presorted=True, weight=b)
        with pytest.raises(ValueError, match="weight"):
            ops.coverage_sweep(X, P, Q, Kt, Wd, Hd, presorted=True, weight=b)


@pytest.mark.parametrize("batch", [False, True])
def test_models_check_the_weight_once_per_state(weight_backend, batch):
    from trajectory_optimization_b200 import model
    pts, poses, quats, prior, weight = _case()
    K, Wd, Hd = _k()
    cpu = torch.device("cpu")

    def make(w):
        if batch:
            return model.ModelTrajBatch(pts, torch.from_numpy(poses), torch.from_numpy(quats), torch.from_numpy(K), Wd,
                                        Hd, device=cpu, point_weight=torch.from_numpy(w))
        return model.ModelTraj(pts, torch.from_numpy(poses[0]), torch.from_numpy(quats[0]), torch.from_numpy(K), Wd, Hd,
                               device=cpu, point_weight=torch.from_numpy(w))

    for v, msg in ((np.inf, "finite"), (np.nan, "finite"), (-1.0, ">= 0")):
        w = weight.copy()
        w[5] = v
        with pytest.raises(ValueError, match=msg):
            make(w)(vis_wps_dist=0.0)
    with pytest.raises(ValueError, match="positive sum"):
        make(np.zeros_like(weight))(vis_wps_dist=0.0)
    with pytest.raises(ValueError, match="point_weight"):
        make(weight[:-1])(vis_wps_dist=0.0)
    # a valid weight: the model's loss is the weighted objective; an in-place edit to something invalid is seen
    m = make(weight)
    m(vis_wps_dist=0.0)
    m.point_weight[3] = -2.0
    with pytest.raises(ValueError, match=">= 0"):
        m(vis_wps_dist=0.0)
    with pytest.raises(ValueError, match="finite"):
        m.set_point_weight(torch.full((len(pts),), float("nan")))


def test_model_traj_weighted_loss_and_criterion(weight_backend):
    from tests.conftest import rel_err
    from trajectory_optimization_b200 import model
    pts, poses, quats, prior, weight = _case()
    K, Wd, Hd = _k()
    m = model.ModelTraj(pts, torch.from_numpy(poses[0]), torch.from_numpy(quats[0]), torch.from_numpy(K), Wd, Hd,
                        device=torch.device("cpu"), point_weight=torch.from_numpy(weight),
                        prior_logodds=torch.from_numpy(prior))
    m(vis_wps_dist=0.0)
    ref = traj_objective_weighted(pts, poses[0], quats[0], K, Wd, Hd, weight, prior=prior.astype(np.float64))
    assert rel_err(m.loss["vis"].item(), ref["vis"]) < 1e-5
    # criterion of rewards from elsewhere: the weighted mean too
    m.criterion(m.rewards.detach().clone())
    assert rel_err(m.loss["vis"].item(), ref["vis"]) < 1e-5
    # set_point_weight(ones) gives the unweighted objective
    m.set_point_weight(torch.ones(len(pts)))
    m(vis_wps_dist=0.0)
    ref1 = traj_objective_prior(pts, poses[0], quats[0], K, Wd, Hd, prior=prior.astype(np.float64))
    assert rel_err(m.loss["vis"].item(), ref1["vis"]) < 1e-5


def _run_all(pts, poses, quats, prior, weight, **kw):
    from trajectory_optimization_b200 import ops
    K, Wd, Hd = _k()
    Kt = torch.from_numpy(K)
    c = torch.linspace(1.0, 2.0, len(poses))
    P = torch.from_numpy(poses.copy()).requires_grad_(True)
    Q = torch.from_numpy(quats.copy()).requires_grad_(True)
    wk = dict(prior_logodds=torch.from_numpy(prior), weight=torch.from_numpy(weight))
    means = ops.coverage_sweep(torch.from_numpy(pts), P, Q, Kt, Wd, Hd, presorted=True, **wk, **kw)
    (c * means).sum().backward()
    sums = ops.sweep_rewards(torch.from_numpy(pts), torch.from_numpy(poses), torch.from_numpy(quats), Kt, Wd, Hd,
                             presorted=True, **wk, **kw)
    return means.detach().numpy(), P.grad.numpy(), Q.grad.numpy(), sums.numpy()


def _run_traj(pts, poses, quats, prior, weight, **kw):
    from trajectory_optimization_b200 import ops
    K, Wd, Hd = _k()
    P = torch.from_numpy(poses[0].copy()).requires_grad_(True)
    Q = torch.from_numpy(quats[0].copy()).requires_grad_(True)
    _, mean = ops.coverage_traj(torch.from_numpy(pts), P, Q, torch.from_numpy(K), Wd, Hd,
                                prior_logodds=torch.from_numpy(prior), weight=torch.from_numpy(weight), **kw)
    mean.backward()
    return mean.detach().numpy(), P.grad.numpy(), Q.grad.numpy()


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from trajectory_optimization_b200 import ops
        ops._BACKEND = WeightOracleBackend()
        pts, poses, quats, prior, weight = _case()
        n = len(pts)
        lo, hi = rank * n // world, (rank + 1) * n // world
        g = dist.group.WORLD
        by_traj = _run_all(pts, poses, quats, prior, weight, group=g, shard="trajectories")
        sl = slice(lo, hi)
        by_pts = _run_all(pts[sl].copy(), poses, quats, prior[sl].copy(), weight[sl].copy(), group=g, shard="points")
        traj = _run_traj(pts[sl].copy(), poses, quats, prior[sl].copy(), weight[sl].copy(), group=g)
        q.put((rank, by_traj, by_pts, traj))
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


def test_two_rank_weighted_runs_match_unsharded(weight_backend):
    """Both sweep shardings and the point-sharded coverage_traj with a weight and a prior, over two gloo ranks, reproduce
    one unsharded run: each rank's base adds up through the accumulators, the denominator is all-reduced."""
    from tests.conftest import rel_err
    pts, poses, quats, prior, weight = _case()
    ref_all = _run_all(pts, poses, quats, prior, weight)
    ref_traj = _run_traj(pts, poses, quats, prior, weight)
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = sorted([q.get(timeout=240) for _ in range(world)], key=lambda t: t[0])
    assert all(len(r) == 4 for r in results), results
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for _, by_traj, by_pts, traj in results:
        for got in (by_traj, by_pts):
            for a, b in zip(got, ref_all):
                assert a.shape == b.shape and rel_err(a, b) < 1e-6
        for a, b in zip(traj, ref_traj):
            assert rel_err(a, b) < 1e-6
