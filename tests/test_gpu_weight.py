"""Per-point weights on the GPU: the rewards do not change (bit for bit), the weighted mean and its gradients equal what
torch computes from the unweighted call's rewards (and autograd through its rewards), pruned == dense, a weight of ones
reproduces the unweighted calls, weight + prior against the oracle, a region of interest, the compact cloud's arg-min
path, shard additivity, the sweeps against per-trajectory calls, and the models (eager, CUDA graphs, set_point_weight,
in-place edits, refresh_points_)."""
import numpy as np
import pytest
import torch

from oracle import coverage_oracle as orc
from tests._weight_oracle import traj_objective_weighted
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


def _prior(gen, n, dev):
    return torch.from_numpy(gen.normal(0, 2, n).astype(np.float32)).to(dev)


def _weight(gen, n, dev):
    w = (gen.random(n) * 2).astype(np.float32)
    w[gen.random(n) < 0.3] = 0.0
    return torch.from_numpy(w).to(dev)


def _path(gen, W=10, length=9.0):
    xs = np.linspace(0, length, W)
    poses = np.stack([xs, 0.5 * xs + 0.3 * np.sin(xs), np.zeros(W)], 1).astype(np.float32)
    quats = (gen.standard_normal((W, 4)) * 0.4 + np.array([1.0, 0, 0, 0])).astype(np.float32)
    return poses, quats


def _big_cloud(gen, n):
    lo, hi = np.array([-10, -10, -1], np.float32), np.array([30, 30, 4], np.float32)
    return (gen.random((n, 3), dtype=np.float32) * (hi - lo) + lo).astype(np.float32)


def _traj(ops, pts, poses, quats, K, Wd, Hd, **kw):
    """(rewards, mean, d vis/d poses, d vis/d quats) of one coverage_traj call with vis = 1/(mean + eps)."""
    P = torch.from_numpy(poses).to(pts.device).requires_grad_(True)
    Q = torch.from_numpy(quats).to(pts.device).requires_grad_(True)
    rewards, mean = ops.coverage_traj(pts, P, Q, K, Wd, Hd, **kw)
    (1.0 / (mean + 1e-6)).backward()
    return rewards.detach(), mean.item(), P.grad.cpu().numpy(), Q.grad.cpu().numpy()


def _torch_weighted(ops, pts, poses, quats, K, Wd, Hd, w, **kw):
    """The weighted objective composed in torch from the unweighted call: its gradient runs through g_rewards."""
    P = torch.from_numpy(poses).to(pts.device).requires_grad_(True)
    Q = torch.from_numpy(quats).to(pts.device).requires_grad_(True)
    rewards, _ = ops.coverage_traj(pts, P, Q, K, Wd, Hd, **kw)
    w64 = w.double()
    mean = (w64 * rewards.double()).sum() / w64.sum()
    (1.0 / (mean + 1e-6)).backward()
    return mean.item(), P.grad.cpu().numpy(), Q.grad.cpu().numpy()


@pytest.mark.parametrize("with_prior", [False, True])
def test_weighted_traj_rewards_mean_gradients_pruned_and_dense(with_prior, dev, mod):
    model, tools, ops = mod
    gen = np.random.default_rng(21)
    K, Wd, Hd = tools.load_intrinsics(dev)
    pts, perm = ops.spatial_sort(torch.from_numpy(_big_cloud(gen, 600_000)).to(dev))
    poses, quats = _path(gen)
    w = _weight(gen, pts.shape[0], dev)
    kw = dict(reward_index=perm, prior_logodds=_prior(gen, pts.shape[0], dev) if with_prior else None)
    means = {}
    for dense in (False, True):
        r0, _, _, _ = _traj(ops, pts, poses, quats, K, Wd, Hd, dense=dense, **kw)
        r1, m1, gp1, gq1 = _traj(ops, pts, poses, quats, K, Wd, Hd, dense=dense, weight=w, **kw)
        assert torch.equal(r0, r1)   # the weight changes no reward
        ref_mean = ((w.double() * r1.double()).sum() / w.double().sum()).item()
        assert rel_err(m1, ref_mean) < 1e-6
        mt, gpt, gqt = _torch_weighted(ops, pts, poses, quats, K, Wd, Hd, w, dense=dense, **kw)
        assert row_rel_err(gp1, gpt) < TOL_ROW and row_rel_err(gq1, gqt) < TOL_ROW
        assert rel_err(gp1, gpt) < TOL and rel_err(gq1, gqt) < TOL
        means[dense] = m1
    assert rel_err(means[False], means[True]) < 1e-6   # same rewards, fp64 sums in another order


@pytest.mark.parametrize("dense", [False, True])
def test_weight_of_ones_reproduces_unweighted(dense, dev, mod, sample_inputs):
    model, tools, ops = mod
    gen = np.random.default_rng(22)
    K, Wd, Hd = tools.load_intrinsics(dev)
    for pts_np in (sample_inputs["pts"], _big_cloud(gen, 300_000)):
        pts, perm = ops.spatial_sort(torch.from_numpy(pts_np).to(dev))
        poses, quats = _path(gen)
        ones = torch.ones(pts.shape[0], device=dev)
        for pr in (None, _prior(gen, pts.shape[0], dev)):
            kw = dict(reward_index=perm, dense=dense, prior_logodds=pr)
            r0, m0, gp0, gq0 = _traj(ops, pts, poses, quats, K, Wd, Hd, **kw)
            r1, m1, gp1, gq1 = _traj(ops, pts, poses, quats, K, Wd, Hd, weight=ones, **kw)
            assert torch.equal(r0, r1)
            assert rel_err(m1, m0) < 1e-6
            assert rel_err(gp1, gp0) < 1e-5 and rel_err(gq1, gq0) < 1e-5
            T = 3
            Ps = torch.from_numpy(poses).to(dev)[None].repeat(T, 1, 1) + torch.randn(T, 1, 3, device=dev) * torch.tensor(
                [0.5, 0.5, 0.0], device=dev)
            Qs = torch.from_numpy(quats).to(dev)[None].repeat(T, 1, 1)
            with ops.evaluation(dense=dense):
                s0 = ops.sweep_rewards(pts, Ps, Qs, K, Wd, Hd, presorted=True, prior_logodds=pr)
                s1 = ops.sweep_rewards(pts, Ps, Qs, K, Wd, Hd, presorted=True, prior_logodds=pr, weight=ones)
                assert rel_err(s1.cpu().numpy(), s0.cpu().numpy()) < 1e-12
                c0 = ops.coverage_sweep(pts, Ps, Qs, K, Wd, Hd, presorted=True, prior_logodds=pr)
                c1 = ops.coverage_sweep(pts, Ps, Qs, K, Wd, Hd, presorted=True, prior_logodds=pr, weight=ones)
                assert rel_err(c1.cpu().numpy(), c0.cpu().numpy()) < 1e-6


@pytest.mark.parametrize("dense", [False, True])
def test_weight_and_prior_match_oracle(dense, dev, mod):
    model, tools, ops = mod
    gen = np.random.default_rng(23)
    K, Wd, Hd = tools.load_intrinsics(dev)
    Kn, Wn, Hn = orc.load_intrinsics()
    pts_np = _big_cloud(gen, 200_000)
    poses, quats = _path(gen)
    pr, w = _prior(gen, len(pts_np), dev), _weight(gen, len(pts_np), dev)
    pts, perm = ops.spatial_sort(torch.from_numpy(pts_np).to(dev))
    r, mean, gp, gq = _traj(ops, pts, poses, quats, K, Wd, Hd, reward_index=perm, dense=dense, prior_logodds=pr, weight=w)
    ref = traj_objective_weighted(pts_np, poses, quats, Kn, Wn, Hn, w.cpu().numpy(), prior=pr.cpu().numpy().astype(np.float64))
    assert rel_err(r.cpu().numpy(), ref["rewards"]) < TOL
    assert rel_err(1.0 / (mean + 1e-6), ref["vis"]) < TOL
    assert row_rel_err(gp, ref["g_poses"]) < TOL_ROW and row_rel_err(gq, ref["g_quats"]) < TOL_ROW


def test_region_of_interest(dev, mod):
    """Weights 1 inside a box and 0 outside: the mean over the points inside, with the normalisers of the whole cloud."""
    model, tools, ops = mod
    gen = np.random.default_rng(24)
    K, Wd, Hd = tools.load_intrinsics(dev)
    pts, perm = ops.spatial_sort(torch.from_numpy(_big_cloud(gen, 400_000)).to(dev))
    poses, quats = _path(gen)
    X = pts[perm.argsort().long()] if perm is not None else pts   # the caller's order, as the rewards come back
    inside = ((X[:, 0] > 2) & (X[:, 0] < 10) & (X[:, 1] > 0) & (X[:, 1] < 8)).float()
    for dense in (False, True):
        r, mean, _, _ = _traj(ops, pts, poses, quats, K, Wd, Hd, reward_index=perm, dense=dense, weight=inside)
        ref = r.double()[inside.bool()].mean().item()
        assert rel_err(mean, ref) < 1e-6
        r_sub, _ = ops.coverage_traj(X[inside.bool()], torch.from_numpy(poses).to(dev), torch.from_numpy(quats).to(dev),
                                     K, Wd, Hd, dense=dense)
        assert not torch.equal(r_sub, r[inside.bool()])   # the normalisers are the whole cloud's, not the box's


def test_compact_cloud_argmin_path_with_weight(dev, mod):
    model, tools, ops = mod
    g = load_golden("traj_compact")
    K, Wd, Hd = tools.load_intrinsics(dev)
    Kn, Wn, Hn = orc.load_intrinsics()
    pts_np = g["in_points"].astype(np.float32)
    gen = np.random.default_rng(25)
    w = _weight(gen, len(pts_np), dev)
    md, xd = float(g["in_min_d"]), float(g["in_max_d"])
    _, mean, gp, gq = _traj(ops, torch.from_numpy(pts_np).to(dev), g["in_poses"].astype(np.float32),
                            g["in_quats"].astype(np.float32), K, Wd, Hd, min_dist=md, max_dist=xd, weight=w)
    ref = traj_objective_weighted(pts_np, g["in_poses"], g["in_quats"], Kn, Wn, Hn, w.cpu().numpy(), min_dist=md,
                                  max_dist=xd)
    assert rel_err(1.0 / (mean + 1e-6), ref["vis"]) < TOL
    assert row_rel_err(gp, ref["g_poses"]) < TOL_ROW and row_rel_err(gq, ref["g_quats"]) < TOL_ROW


def test_weighted_accumulators_are_shard_additive(dev, mod):
    model, tools, ops = mod
    gen = np.random.default_rng(26)
    K, Wd, Hd = tools.load_intrinsics(dev)
    pts, _ = ops.spatial_sort(torch.from_numpy(_big_cloud(gen, 400_000)).to(dev))
    pr, w = _prior(gen, pts.shape[0], dev), _weight(gen, pts.shape[0], dev)
    poses, quats = _path(gen)
    P, Q = torch.from_numpy(poses).to(dev), torch.from_numpy(quats).to(dev)
    B = ops._BACKEND
    cam = ops._lib.camera(Wd, Hd, 1.0, 5.0, 1e-6)
    Kd = K.reshape(9).contiguous()
    mm = B.traj_minmax(pts, P, Q, Kd, cam)
    for prior in (None, pr):
        whole_s = B.weight_sums(w, prior)
        whole = B.traj_fused(pts, P, Q, Kd, cam, mm, None, torch.empty(pts.shape[0], device=dev), prior=prior, weight=w,
                             wsums=whole_s)
        h = pts.shape[0] // 2 + 77
        parts, sums = [], []
        for sl in (slice(0, h), slice(h, None)):
            x, ww = pts[sl].clone(), w[sl].clone()   # fresh, aligned allocations, as two ranks would hold them
            p = None if prior is None else prior[sl].clone()
            s = B.weight_sums(ww, p)
            sums.append(s)
            parts.append(B.traj_fused(x, P, Q, Kd, cam, mm, None, torch.empty(x.shape[0], device=dev), prior=p, weight=ww,
                                      wsums=s))
        # sums are fp32 within a (128-point item, pose) and fp64 above: the split moves the item boundaries of the second
        # half, so the fp32 partials of the weighted rows differ in their last bits
        assert rel_err((parts[0] + parts[1]).cpu().numpy(), whole.cpu().numpy()) < 1e-8
        assert rel_err((sums[0] + sums[1]).cpu().numpy(), whole_s.cpu().numpy()) < 1e-12


@pytest.mark.parametrize("dense", [False, True])
def test_weighted_sweeps_equal_per_trajectory_calls(dense, dev, mod):
    model, tools, ops = mod
    gen = np.random.default_rng(27)
    K, Wd, Hd = tools.load_intrinsics(dev)
    X = torch.from_numpy(_big_cloud(gen, 200_000)).to(dev)
    pr, w = _prior(gen, X.shape[0], dev), _weight(gen, X.shape[0], dev)
    T = 4
    base, quats = _path(gen, W=8)
    poses = np.repeat(base[None], T, 0) + gen.normal(0, 0.6, (T, 1, 3)).astype(np.float32) * np.array([1, 1, 0], np.float32)
    for prior in (None, pr):
        P = torch.from_numpy(poses.astype(np.float32)).to(dev).requires_grad_(True)
        Q = torch.from_numpy(np.repeat(quats[None], T, 0)).to(dev).requires_grad_(True)
        with ops.evaluation(dense=dense):
            sums = ops.sweep_rewards(X, P.detach(), Q.detach(), K, Wd, Hd, prior_logodds=prior, weight=w)
            means = ops.coverage_sweep(X, P, Q, K, Wd, Hd, prior_logodds=prior, weight=w)
        (1.0 / (means + 1e-6)).sum().backward()
        for t in range(T):
            _, mean, gp, gq = _traj(ops, X, poses[t].astype(np.float32), quats, K, Wd, Hd, dense=dense, prior_logodds=prior,
                                    weight=w)
            assert rel_err(sums[t].item(), mean) < 1e-6 and rel_err(means[t].item(), mean) < 1e-6
            assert row_rel_err(P.grad[t].cpu().numpy(), gp) < TOL_ROW
            assert row_rel_err(Q.grad[t].cpu().numpy(), gq) < TOL_ROW
    # ModelTrajBatch(point_weight) against separate ModelTraj(point_weight) models
    mb = model.ModelTrajBatch(X, P.detach(), Q.detach(), K, Wd, Hd, device=dev, prior_logodds=pr, point_weight=w,
                              spatial_sort=not dense)
    mb(vis_wps_dist=0.5).backward()
    for t in range(T):
        m = model.ModelTraj(X, P.detach()[t], Q.detach()[t], K, Wd, Hd, device=dev, prior_logodds=pr, point_weight=w,
                            spatial_sort=not dense)
        m(vis_wps_dist=0.5).backward()
        assert rel_err(mb.losses["vis"][t].item(), m.loss["vis"].item()) < 1e-6
        assert row_rel_err(mb.poses.grad[t].cpu().numpy(), m.poses.grad.cpu().numpy()) < TOL_ROW
        assert row_rel_err(mb.quats.grad[t].cpu().numpy(), m.quats.grad.cpu().numpy()) < TOL_ROW


@pytest.mark.parametrize("batch", [False, True])
def test_models_weight_graphs_edits_and_refresh(batch, dev, mod):
    from trajectory_optimization_b200.graphs import GraphedStep
    model, tools, ops = mod
    gen = np.random.default_rng(28)
    K, Wd, Hd = tools.load_intrinsics(dev)
    pts = torch.from_numpy(_big_cloud(gen, 150_000))
    poses, quats = _path(gen)
    if batch:
        poses = np.stack([poses, poses + np.array([0.0, 1.0, 0.0], np.float32)])
        quats = np.stack([quats, quats])
    w = _weight(gen, len(pts), dev)
    pr = _prior(gen, len(pts), dev)

    def make(ptsx):
        cls = model.ModelTrajBatch if batch else model.ModelTraj
        return cls(ptsx, torch.from_numpy(poses), torch.from_numpy(quats), K, Wd, Hd, device=dev, prior_logodds=pr.clone(),
                   point_weight=w.clone())

    def mean_of(m):
        return (m.means if batch else m._mean).detach().clone()

    finals = []
    for graphed in (False, True):
        m = make(pts)
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
        finals.append((loss.item(), m.poses.detach().clone(), m, g if graphed else None))
    assert rel_err(finals[1][0], finals[0][0]) < 1e-5
    assert rel_err(finals[1][1].cpu().numpy(), finals[0][1].cpu().numpy()) < 1e-5
    # set_point_weight between replays: the captured graph evaluates the new weight
    m, g = finals[1][2], finals[1][3]
    w2 = _weight(gen, len(pts), dev)
    m.set_point_weight(w2)
    p_before, q_before = m.poses.detach().clone(), m.quats.detach().clone()   # the replay's forward sees these
    g.step()
    torch.cuda.synchronize()
    got = mean_of(m)
    ref = make(pts)
    ref.poses.data.copy_(p_before)
    ref.quats.data.copy_(q_before)
    ref.set_point_weight(w2)
    ref(vis_wps_dist=0.0)
    assert rel_err(got.cpu().numpy(), mean_of(ref).cpu().numpy()) < 1e-6
    # in-place edit of the weight: the next eager forward sees it
    e = finals[0][2]
    e(vis_wps_dist=0.0)
    before = mean_of(e)
    e.point_weight.mul_(torch.linspace(0.0, 2.0, len(pts), device=dev))
    e(vis_wps_dist=0.0)
    ref2 = make(pts)
    ref2.poses.data.copy_(e.poses.detach())
    ref2.quats.data.copy_(e.quats.detach())
    ref2.set_point_weight(e.point_weight.clone())
    ref2(vis_wps_dist=0.0)
    assert not torch.equal(before, mean_of(e))
    assert rel_err(mean_of(e).cpu().numpy(), mean_of(ref2).cpu().numpy()) < 1e-6
    # refresh_points_ with a captured graph: the replay evaluates the new cloud with the same weight
    m2 = make(pts)
    opt2 = torch.optim.Adam([m2.poses, m2.quats], lr=0.0, capturable=True)
    g2 = GraphedStep(m2, opt2, forward_kwargs=dict(vis_wps_dist=0.0), warmup=1)
    new_pts = pts.flip(0) + 0.25
    m2.refresh_points_(new_pts.to(dev))
    g2.step()
    torch.cuda.synchronize()
    ref3 = make(new_pts)
    ref3.poses.data.copy_(m2.poses.detach())
    ref3.quats.data.copy_(m2.quats.detach())
    ref3(vis_wps_dist=0.0)
    assert rel_err(mean_of(m2).cpu().numpy(), mean_of(ref3).cpu().numpy()) < 1e-6
