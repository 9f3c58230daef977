"""Prior log-odds (map memory) on the GPU: a zero prior reproduces the calls without one, a random prior matches the oracle
on the dense and the pruned path (pruned == dense bit for bit), the compact cloud's arg-min path, shard additivity of the
accumulators, the sweeps against per-trajectory calls, the fused log-odds output (fold), and the models (eager, CUDA
graphs, in-place edits, refresh_points_)."""
import numpy as np
import pytest
import torch

from oracle import coverage_oracle as orc
from tests._prior_oracle import traj_objective_prior
from tests.conftest import load_golden, rel_err, row_rel_err

pytestmark = pytest.mark.gpu
TOL, TOL_ROW = 1e-4, 2e-4


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def mod():
    from trajectory_optimization_b200 import _lib, model, ops, tools
    _lib.lib()
    return model, tools, ops


def _sig(x):
    return 1.0 / (1.0 + torch.exp(-x))   # the kernels' expression, on the device


def _prior(gen, n, dev=None):
    p = gen.normal(0, 2, n).astype(np.float32)
    p[gen.choice(n, max(4, n // 5000), replace=False)] = np.where(gen.random(max(4, n // 5000)) < 0.5, -30, 30)
    t = torch.from_numpy(p)
    return t if dev is None else t.to(dev)


def _path(gen, W=10, length=9.0):
    xs = np.linspace(0, length, W)
    poses = np.stack([xs, 0.5 * xs + 0.3 * np.sin(xs), np.zeros(W)], 1).astype(np.float32)
    quats = (gen.standard_normal((W, 4)) * 0.4 + np.array([1.0, 0, 0, 0])).astype(np.float32)
    return poses, quats


def _big_cloud(gen, n):
    lo, hi = np.array([-10, -10, -1], np.float32), np.array([30, 30, 4], np.float32)
    return (gen.random((n, 3), dtype=np.float32) * (hi - lo) + lo).astype(np.float32)


def _passes(ops, pts, P, Q, K, Wd, Hd, dense, prior=None, reward_index=None):
    """Pass A + pass B through the backend (the C ABI): rewards, minmax and the raw fp64 accumulators."""
    B = ops._BACKEND
    cam = ops._lib.camera(Wd, Hd, 1.0, 5.0, 1e-6)
    Kd = K.reshape(9).contiguous()
    rewards = torch.empty(pts.shape[0], dtype=torch.float32, device=pts.device)
    prefill = rewards if B.prefill_applies(pts, dense) else None
    mm = B.traj_minmax(pts, P, Q, Kd, cam, None, None, dense, prefill, prior)
    if prior is None:
        acc = B.traj_fused(pts, P, Q, Kd, cam, mm, None, rewards, reward_index, None, None, dense, prefill is not None)
    else:
        acc = B.traj_fused(pts, P, Q, Kd, cam, mm, None, rewards, reward_index, None, None, dense, prefill is not None,
                           prior, B.prior_sum(prior))
    return rewards, mm, acc


@pytest.mark.parametrize("dense", [False, True])
def test_zero_prior_reproduces_no_prior(dense, dev, mod, sample_inputs):
    model, tools, ops = mod
    gen = np.random.default_rng(1)
    K, Wd, Hd = tools.load_intrinsics(dev)
    for pts_np in (sample_inputs["pts"], _big_cloud(gen, 300_000)):
        pts, perm = ops.spatial_sort(torch.from_numpy(pts_np).to(dev))
        poses, quats = _path(gen)
        P, Q = torch.from_numpy(poses).to(dev), torch.from_numpy(quats).to(dev)
        zero = torch.zeros(pts.shape[0], device=dev)
        r0, mm0, a0 = _passes(ops, pts, P, Q, K, Wd, Hd, dense, None, perm)
        r1, mm1, a1 = _passes(ops, pts, P, Q, K, Wd, Hd, dense, zero, perm)
        assert torch.equal(r0, r1) and torch.equal(mm0, mm1)
        assert rel_err(a1.cpu().numpy(), a0.cpu().numpy()) < 1e-12
        T = 3
        Ps = P[None].repeat(T, 1, 1) + torch.randn(T, 1, 3, device=dev) * torch.tensor([0.5, 0.5, 0.0], device=dev)
        Qs = Q[None].repeat(T, 1, 1)
        with ops.evaluation(dense=dense):
            s0 = ops.sweep_rewards(pts, Ps, Qs, K, Wd, Hd, presorted=True)
            s1 = ops.sweep_rewards(pts, Ps, Qs, K, Wd, Hd, presorted=True, prior_logodds=zero)
            assert rel_err(s1.cpu().numpy(), s0.cpu().numpy()) < 1e-12
            cam = ops._lib.camera(Wd, Hd, 1.0, 5.0, 1e-6)
            B = ops._BACKEND
            mm = B.sweep_minmax(pts, Ps.reshape(-1, 3), Qs.reshape(-1, 4), K.reshape(9).contiguous(), cam)
            args = (pts, Ps.reshape(-1, 3), Qs.reshape(-1, 4), T, Ps.shape[1], K.reshape(9).contiguous(), cam, None, mm)
            f0 = B.sweep_fused(*args)
            f1 = B.sweep_fused(*args, None, zero, B.prior_sum(zero))
            assert rel_err(f1.cpu().numpy(), f0.cpu().numpy()) < 1e-12


@pytest.mark.parametrize("which", ["sample_dense", "million_pruned"])
def test_random_prior_matches_oracle_and_pruned_equals_dense(which, dev, mod, sample_inputs):
    model, tools, ops = mod
    gen = np.random.default_rng(2)
    K, Wd, Hd = tools.load_intrinsics(dev)
    Kn, Wn, Hn = orc.load_intrinsics()
    if which == "sample_dense":
        g = load_golden("traj_sample")
        pts_np = sample_inputs["pts"]
        poses, quats = g["in_poses"][::int(g["out_wps_step"])].astype(np.float32), g["in_quats"][::int(g["out_wps_step"])].astype(np.float32)
    else:
        pts_np = _big_cloud(gen, 1_000_000)
        poses, quats = _path(gen)
    prior = _prior(gen, len(pts_np))
    pts, perm = ops.spatial_sort(torch.from_numpy(pts_np).to(dev))
    pr = prior.to(dev)
    outs = {}
    for dense in (False, True):
        P = torch.from_numpy(poses).to(dev).requires_grad_(True)
        Q = torch.from_numpy(quats).to(dev).requires_grad_(True)
        rewards, mean = ops.coverage_traj(pts, P, Q, K, Wd, Hd, reward_index=perm, dense=dense, prior_logodds=pr)
        (1.0 / (mean + 1e-6)).backward()
        outs[dense] = (rewards.detach(), mean.item(), P.grad.cpu().numpy(), Q.grad.cpu().numpy())
        mm = _passes(ops, pts, P.detach(), Q.detach(), K, Wd, Hd, dense, pr, perm)[1]
        outs[dense] += (mm,)
    assert torch.equal(outs[False][0], outs[True][0])   # rewards
    assert torch.equal(outs[False][4], outs[True][4])   # normalisers
    ref = traj_objective_prior(pts_np, poses, quats, Kn, Wn, Hn, prior=prior.numpy().astype(np.float64))
    for dense in (False, True):
        r, mean, gp, gq, _ = outs[dense]
        assert rel_err(r.cpu().numpy(), ref["rewards"]) < TOL
        assert rel_err(1.0 / (mean + 1e-6), ref["vis"]) < TOL
        assert row_rel_err(gp, ref["g_poses"]) < TOL_ROW and row_rel_err(gq, ref["g_quats"]) < TOL_ROW


def test_compact_cloud_argmin_path_with_prior(dev, mod):
    model, tools, ops = mod
    g = load_golden("traj_compact")
    K, Wd, Hd = tools.load_intrinsics(dev)
    Kn, Wn, Hn = orc.load_intrinsics()
    pts_np = g["in_points"].astype(np.float32)
    prior = _prior(np.random.default_rng(3), len(pts_np))
    P = torch.from_numpy(g["in_poses"].astype(np.float32)).to(dev).requires_grad_(True)
    Q = torch.from_numpy(g["in_quats"].astype(np.float32)).to(dev).requires_grad_(True)
    md, xd = float(g["in_min_d"]), float(g["in_max_d"])
    _, mean = ops.coverage_traj(torch.from_numpy(pts_np).to(dev), P, Q, K, Wd, Hd, md, xd, prior_logodds=prior.to(dev))
    (1.0 / (mean + 1e-6)).backward()
    from tests._prior_oracle import traj_partials_prior
    part = traj_partials_prior(pts_np, g["in_poses"], g["in_quats"], Kn, Wn, Hn, md, xd, prior=prior.numpy().astype(np.float64))
    assert part["amin_n"].sum() > 0   # the arg-min tie path carries gradient here
    ref = orc.traj_grads_from_partials(part, g["in_poses"], g["in_quats"], len(pts_np))
    assert rel_err(1.0 / (mean.item() + 1e-6), ref["vis"]) < TOL
    assert row_rel_err(P.grad.cpu().numpy(), ref["g_poses"]) < TOL_ROW
    assert row_rel_err(Q.grad.cpu().numpy(), ref["g_quats"]) < TOL_ROW


def test_accumulators_are_shard_additive_with_prior(dev, mod):
    """Two halves, each with its half of the prior and its own sum_j sigmoid(prior_j), add up to the whole cloud."""
    model, tools, ops = mod
    gen = np.random.default_rng(4)
    K, Wd, Hd = tools.load_intrinsics(dev)
    pts, _ = ops.spatial_sort(torch.from_numpy(_big_cloud(gen, 400_000)).to(dev))
    pr = _prior(gen, pts.shape[0], dev)
    poses, quats = _path(gen)
    P, Q = torch.from_numpy(poses).to(dev), torch.from_numpy(quats).to(dev)
    B = ops._BACKEND
    cam = ops._lib.camera(Wd, Hd, 1.0, 5.0, 1e-6)
    Kd = K.reshape(9).contiguous()
    mm = B.traj_minmax(pts, P, Q, Kd, cam)
    whole = B.traj_fused(pts, P, Q, Kd, cam, mm, None, torch.empty(pts.shape[0], device=dev), prior=pr,
                         prior_sum=B.prior_sum(pr))
    h = pts.shape[0] // 2 + 77
    parts = []
    for sl in (slice(0, h), slice(h, None)):
        x, p = pts[sl].clone(), pr[sl].clone()   # fresh, aligned allocations, as two ranks would hold them
        parts.append(B.traj_fused(x, P, Q, Kd, cam, mm, None, torch.empty(x.shape[0], device=dev), prior=p,
                                  prior_sum=B.prior_sum(p)))
    assert rel_err((parts[0] + parts[1]).cpu().numpy(), whole.cpu().numpy()) < 1e-12


def test_sweeps_with_prior_equal_per_trajectory_calls(dev, mod):
    model, tools, ops = mod
    gen = np.random.default_rng(5)
    K, Wd, Hd = tools.load_intrinsics(dev)
    pts_np = _big_cloud(gen, 200_000)
    X = torch.from_numpy(pts_np).to(dev)
    pr = _prior(gen, len(pts_np), dev)
    T = 4
    base, quats = _path(gen, W=8)
    poses = np.repeat(base[None], T, 0) + gen.normal(0, 0.6, (T, 1, 3)).astype(np.float32) * np.array([1, 1, 0], np.float32)
    P = torch.from_numpy(poses.astype(np.float32)).to(dev).requires_grad_(True)
    Q = torch.from_numpy(np.repeat(quats[None], T, 0)).to(dev).requires_grad_(True)
    sums = ops.sweep_rewards(X, P.detach(), Q.detach(), K, Wd, Hd, prior_logodds=pr)
    means = ops.coverage_sweep(X, P, Q, K, Wd, Hd, prior_logodds=pr)
    (1.0 / (means + 1e-6)).sum().backward()
    for t in range(T):
        Pt = P.detach()[t].clone().requires_grad_(True)
        Qt = Q.detach()[t].clone().requires_grad_(True)
        _, mean = ops.coverage_traj(X, Pt, Qt, K, Wd, Hd, prior_logodds=pr)
        (1.0 / (mean + 1e-6)).backward()
        assert rel_err(sums[t].item(), mean.item()) < 1e-6 and rel_err(means[t].item(), mean.item()) < 1e-6
        assert row_rel_err(P.grad[t].cpu().numpy(), Pt.grad.cpu().numpy()) < TOL_ROW
        assert row_rel_err(Q.grad[t].cpu().numpy(), Qt.grad.cpu().numpy()) < TOL_ROW
    # ModelTrajBatch(prior) against separate ModelTraj(prior) models
    mb = model.ModelTrajBatch(X, P.detach(), Q.detach(), K, Wd, Hd, device=dev, prior_logodds=pr)
    loss = mb(vis_wps_dist=0.5)
    loss.backward()
    for t in range(T):
        m = model.ModelTraj(X, P.detach()[t], Q.detach()[t], K, Wd, Hd, device=dev, prior_logodds=pr)
        m(vis_wps_dist=0.5).backward()
        assert rel_err(mb.losses["vis"][t].item(), float(m.loss["vis"])) < 1e-6
        assert row_rel_err(mb.poses.grad[t].cpu().numpy(), m.poses.grad.cpu().numpy()) < TOL_ROW
        assert row_rel_err(mb.quats.grad[t].cpu().numpy(), m.quats.grad.cpu().numpy()) < TOL_ROW


@pytest.mark.parametrize("dense", [False, True])
def test_fold_executed_path_into_the_map(dense, dev, mod):
    model, tools, ops = mod
    gen = np.random.default_rng(6)
    K, Wd, Hd = tools.load_intrinsics(dev)
    pts, perm = ops.spatial_sort(torch.from_numpy(_big_cloud(gen, 250_000)).to(dev))
    pr = _prior(gen, pts.shape[0], dev)
    poses, quats = _path(gen, W=12)
    P, Q = torch.from_numpy(poses).to(dev), torch.from_numpy(quats).to(dev)
    kw = dict(reward_index=perm, dense=dense)
    lo = ops.traj_logodds(pts, P, Q, K, Wd, Hd, prior_logodds=pr, **kw)
    rewards, _ = ops.coverage_traj(pts, P, Q, K, Wd, Hd, prior_logodds=pr, **kw)
    assert torch.equal(_sig(lo), rewards)
    lo0 = ops.traj_logodds(pts, P, Q, K, Wd, Hd, **kw)
    assert torch.equal(lo, pr + lo0)
    # path A, then path B on the map A left, against A and B evaluated at once (fp32 summation order apart)
    A, Bp = slice(0, 6), slice(6, 12)
    mapA = ops.traj_logodds(pts, P[A], Q[A], K, Wd, Hd, **kw)
    rB, _ = ops.coverage_traj(pts, P[Bp], Q[Bp], K, Wd, Hd, prior_logodds=mapA, **kw)
    rAB, _ = ops.coverage_traj(pts, P, Q, K, Wd, Hd, **kw)
    assert rel_err(rB.cpu().numpy(), rAB.cpu().numpy()) < 1e-5


def test_model_traj_prior_graphs_edits_and_refresh(dev, mod):
    from trajectory_optimization_b200.graphs import GraphedStep
    model, tools, ops = mod
    gen = np.random.default_rng(7)
    K, Wd, Hd = tools.load_intrinsics(dev)
    pts = torch.from_numpy(_big_cloud(gen, 150_000))
    poses, quats = _path(gen)
    pr = _prior(gen, len(pts), dev)
    finals = []
    for graphed in (False, True):
        m = model.ModelTraj(pts, torch.from_numpy(poses), torch.from_numpy(quats), K, Wd, Hd, device=dev,
                            prior_logodds=pr.clone())
        opt = torch.optim.Adam([{"params": [m.poses], "lr": 0.02}, {"params": [m.quats], "lr": 0.01}], capturable=True)
        if graphed:
            g = GraphedStep(m, opt, forward_kwargs=dict(vis_wps_dist=0.0), warmup=1)
            for _ in range(3):
                loss = g.step()
        else:
            for _ in range(4):
                opt.zero_grad()
                loss = m(vis_wps_dist=0.0)
                loss.backward()
                opt.step()
        torch.cuda.synchronize()
        finals.append((loss.item(), m.poses.detach().clone(), m))
    assert rel_err(finals[1][0], finals[0][0]) < 1e-5
    assert rel_err(finals[1][1].cpu().numpy(), finals[0][1].cpu().numpy()) < 1e-5
    # in-place edit of the prior: the next eager forward sees it
    m = finals[0][2]
    m(vis_wps_dist=0.0)
    before = m.rewards.detach().clone()
    m.prior_logodds.add_(1.0)
    m(vis_wps_dist=0.0)
    ref, _ = ops.coverage_traj(m._cloud(), m.poses.detach(), m.quats.detach(), K, Wd, Hd, reward_index=m._perm,
                               prior_logodds=m.prior_logodds)
    assert not torch.equal(before, m.rewards) and torch.equal(m.rewards.detach(), ref)
    assert torch.equal(_sig(m.observed_logodds(vis_wps_dist=0.0)), m.rewards.detach())
    # refresh_points_ with a captured graph: the replay evaluates the new cloud on the same prior
    m2 = model.ModelTraj(pts, torch.from_numpy(poses), torch.from_numpy(quats), K, Wd, Hd, device=dev,
                         prior_logodds=pr.clone())
    opt2 = torch.optim.Adam([m2.poses, m2.quats], lr=0.0, capturable=True)
    g2 = GraphedStep(m2, opt2, forward_kwargs=dict(vis_wps_dist=0.0), warmup=1)
    new_pts = pts.flip(0) + 0.25
    m2.refresh_points_(new_pts.to(dev))
    g2.step()
    torch.cuda.synchronize()
    _, mean = ops.coverage_traj(new_pts.to(dev), m2.poses.detach(), m2.quats.detach(), K, Wd, Hd, prior_logodds=pr)
    assert rel_err(m2._mean.item(), mean.item()) < 1e-6
