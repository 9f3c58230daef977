"""Prior log-odds (map memory) around the C ABI, on CPU: the oracle's semantics (prior added after the fusion), its
closed-form gradients against fp64 autograd, the ops' plumbing on an oracle-backed stand-in (tests/_prior_oracle.py),
argument checks, and the point and trajectory shardings over two gloo ranks."""
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

from tests._prior_oracle import PriorOracleBackend, traj_objective_prior, traj_partials_prior  # noqa: E402


def _case(seed=5):
    gen = np.random.default_rng(seed)
    pts = (gen.random((700, 3)) * np.array([16, 16, 4]) + np.array([-4, -4, -1])).astype(np.float32)
    T, Pn = 3, 4
    base = np.stack([np.linspace(0, 6, Pn), np.linspace(0, 3, Pn), np.zeros(Pn)], 1)
    poses = (base[None] + gen.normal(0, 0.8, (T, 1, 3)) * np.array([1, 1, 0])).astype(np.float32)
    quats = (gen.normal(0, 0.3, (T, Pn, 4)) + np.array([1.0, 0, 0, 0])).astype(np.float32)
    prior = gen.normal(0, 2, len(pts)).astype(np.float32)
    prior[gen.choice(len(pts), 12, replace=False)] = np.where(gen.random(12) < 0.5, -30, 30)
    return pts, poses, quats, prior


def _k():
    from oracle import coverage_oracle as orc
    return orc.K_DEFAULT.copy(), orc.IMG_WIDTH, orc.IMG_HEIGHT


@pytest.fixture
def prior_backend(monkeypatch):
    from trajectory_optimization_b200 import ops
    monkeypatch.setattr(ops, "_BACKEND", PriorOracleBackend())


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_oracle_zero_prior_equals_no_prior_exactly(dtype):
    from oracle import coverage_oracle as orc
    pts, poses, quats, _ = _case()
    K, Wd, Hd = _k()
    ref = orc.traj_partials(pts, poses[0], quats[0], K, Wd, Hd, dtype=dtype)
    got = traj_partials_prior(pts, poses[0], quats[0], K, Wd, Hd, dtype=dtype, prior=np.zeros(len(pts), dtype))
    for key, v in ref.items():
        assert np.array_equal(np.asarray(got[key]), np.asarray(v)), key


def test_oracle_prior_gradients_match_fp64_autograd():
    """Closed-form fp64 gradients of vis = 1/(mean_j sigmoid(prior_j + sum_w lo_jw) + eps) against torch autograd."""
    from oracle import torch_port
    pts, poses, quats, prior = _case()
    prior[np.abs(prior) > 20] = 0.0   # autograd of a saturated sigmoid is exactly 0 both ways; keep the test sharp
    K, Wd, Hd = _k()
    ref = traj_objective_prior(pts, poses[0], quats[0], K, Wd, Hd, prior=prior.astype(np.float64))
    P = torch.from_numpy(poses[0].astype(np.float64)).requires_grad_(True)
    Q = torch.from_numpy(quats[0].astype(np.float64)).requires_grad_(True)
    X = torch.from_numpy(pts.astype(np.float64))
    Kt = torch.from_numpy(K.astype(np.float64))
    lo = torch.from_numpy(prior.astype(np.float64))
    for i in range(len(P)):
        m = torch_port.visibility(X, Q[i].unsqueeze(0), P[i].unsqueeze(0), Kt, Wd, Hd, 1.0, 5.0, 1e-6)
        p = (m - m.min()) / (m - m.min()).max()
        p = torch.clip(p, 0.5, 1.0 - 1e-6)
        lo = lo + torch.log(p / (1.0 - p))
    vis = 1.0 / ((1.0 / (1.0 + torch.exp(-lo))).mean() + 1e-6)
    vis.backward()
    from tests.conftest import rel_err
    assert rel_err(ref["vis"], vis.item()) < 1e-12
    assert rel_err(ref["g_poses"], P.grad.numpy()) < 1e-12
    assert rel_err(ref["g_quats"], Q.grad.numpy()) < 1e-12


def test_ops_with_prior_agree_with_oracle(prior_backend):
    from tests.conftest import rel_err
    from trajectory_optimization_b200 import ops
    pts, poses, quats, prior = _case()
    K, Wd, Hd = _k()
    Kt, X, pr = torch.from_numpy(K), torch.from_numpy(pts), torch.from_numpy(prior)
    refs = [traj_objective_prior(pts, poses[t], quats[t], K, Wd, Hd, prior=prior.astype(np.float64))
            for t in range(len(poses))]
    for t, ref in enumerate(refs):
        P = torch.from_numpy(poses[t].copy()).requires_grad_(True)
        Q = torch.from_numpy(quats[t].copy()).requires_grad_(True)
        rewards, mean = ops.coverage_traj(X, P, Q, Kt, Wd, Hd, prior_logodds=pr)
        (1.0 / (mean + 1e-6)).backward()
        # the stand-in clips at fp32(1 - 1e-6) (as the kernels do), the fp64 oracle at 1 - 1e-6: ~1e-6 apart
        assert rel_err(rewards.detach().numpy(), ref["rewards"]) < 1e-5 and rel_err(mean.item(), ref["mean"]) < 1e-5
        assert rel_err(P.grad.numpy(), ref["g_poses"]) < 1e-4 and rel_err(Q.grad.numpy(), ref["g_quats"]) < 1e-4
        lo = ops.traj_logodds(X, torch.from_numpy(poses[t]), torch.from_numpy(quats[t]), Kt, Wd, Hd, prior_logodds=pr)
        assert rel_err(torch.sigmoid(lo.double()).numpy(), ref["rewards"]) < 1e-5
        lo0 = ops.traj_logodds(X, torch.from_numpy(poses[t]), torch.from_numpy(quats[t]), Kt, Wd, Hd)
        assert torch.equal(lo, pr + lo0)
    means = ops.sweep_rewards(X, torch.from_numpy(poses), torch.from_numpy(quats), Kt, Wd, Hd, presorted=True,
                              prior_logodds=pr)
    assert rel_err(means.numpy(), [r["mean"] for r in refs]) < 1e-5
    means = ops.coverage_sweep(X, torch.from_numpy(poses), torch.from_numpy(quats), Kt, Wd, Hd, presorted=True,
                               prior_logodds=pr)
    assert rel_err(means.detach().numpy(), [r["mean"] for r in refs]) < 1e-5


def test_prior_argument_errors_name_the_argument(prior_backend):
    from trajectory_optimization_b200 import ops
    pts, poses, quats, prior = _case()
    K, Wd, Hd = _k()
    Kt, X, P, Q = torch.from_numpy(K), torch.from_numpy(pts), torch.from_numpy(poses), torch.from_numpy(quats)
    bad = [torch.from_numpy(prior).double(), torch.from_numpy(prior[:-1]), torch.from_numpy(prior).reshape(-1, 1),
           prior]
    if torch.cuda.is_available():
        bad.append(torch.from_numpy(prior).cuda())
    else:
        bad.append(torch.from_numpy(prior).to("meta"))
    for b in bad:
        with pytest.raises(ValueError, match="prior_logodds"):
            ops.coverage_traj(X, P[0], Q[0], Kt, Wd, Hd, prior_logodds=b)
        with pytest.raises(ValueError, match="prior_logodds"):
            ops.traj_logodds(X, P[0], Q[0], Kt, Wd, Hd, prior_logodds=b)
        with pytest.raises(ValueError, match="prior_logodds"):
            ops.sweep_rewards(X, P, Q, Kt, Wd, Hd, presorted=True, prior_logodds=b)
        with pytest.raises(ValueError, match="prior_logodds"):
            ops.coverage_sweep(X, P, Q, Kt, Wd, Hd, presorted=True, prior_logodds=b)


def test_model_rejects_non_finite_prior(prior_backend):
    from trajectory_optimization_b200 import model
    pts, poses, quats, prior = _case()
    K, Wd, Hd = _k()
    prior[3] = np.inf
    m = model.ModelTraj(pts, torch.from_numpy(poses[0]), torch.from_numpy(quats[0]), torch.from_numpy(K), Wd, Hd, device=torch.device("cpu"),
                        prior_logodds=torch.from_numpy(prior))
    with pytest.raises(ValueError, match="finite"):
        m(vis_wps_dist=0.0)


def _run_all(pts, poses, quats, prior, **kw):
    from trajectory_optimization_b200 import ops
    K, Wd, Hd = _k()
    Kt = torch.from_numpy(K)
    weights = torch.linspace(1.0, 2.0, len(poses))
    P = torch.from_numpy(poses.copy()).requires_grad_(True)
    Q = torch.from_numpy(quats.copy()).requires_grad_(True)
    means = ops.coverage_sweep(torch.from_numpy(pts), P, Q, Kt, Wd, Hd, presorted=True, prior_logodds=torch.from_numpy(prior),
                               **kw)
    (weights * means).sum().backward()
    sums = ops.sweep_rewards(torch.from_numpy(pts), torch.from_numpy(poses), torch.from_numpy(quats), Kt, Wd, Hd,
                             presorted=True, prior_logodds=torch.from_numpy(prior), **kw)
    return means.detach().numpy(), P.grad.numpy(), Q.grad.numpy(), sums.numpy()


def _run_traj(pts, poses, quats, prior, **kw):
    from trajectory_optimization_b200 import ops
    K, Wd, Hd = _k()
    P = torch.from_numpy(poses[0].copy()).requires_grad_(True)
    Q = torch.from_numpy(quats[0].copy()).requires_grad_(True)
    _, mean = ops.coverage_traj(torch.from_numpy(pts), P, Q, torch.from_numpy(K), Wd, Hd,
                                prior_logodds=torch.from_numpy(prior), **kw)
    mean.backward()
    return mean.detach().numpy(), P.grad.numpy(), Q.grad.numpy()


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from trajectory_optimization_b200 import ops
        ops._BACKEND = PriorOracleBackend()
        pts, poses, quats, prior = _case()
        n = len(pts)
        lo, hi = rank * n // world, (rank + 1) * n // world
        g = dist.group.WORLD
        by_traj = _run_all(pts, poses, quats, prior, group=g, shard="trajectories")
        by_pts = _run_all(pts[lo:hi].copy(), poses, quats, prior[lo:hi].copy(), n_total=n, group=g, shard="points")
        traj = _run_traj(pts[lo:hi].copy(), poses, quats, prior[lo:hi].copy(), n_total=n, group=g)
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


def test_two_rank_prior_runs_match_unsharded(prior_backend):
    """Both sweep shardings and the point-sharded coverage_traj with a prior, over two gloo ranks, reproduce one unsharded
    run: each rank's slice of the prior adds its own sum_j sigmoid(prior_j), the SUM all-reduce makes it global."""
    from tests.conftest import rel_err
    pts, poses, quats, prior = _case()
    ref_all = _run_all(pts, poses, quats, prior)
    ref_traj = _run_traj(pts, poses, quats, prior)
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
