"""Trajectories longer than one pruned call takes (cov_traj_fused_long, cov_traj_logodds_long) on the GPU: the carry
reproduces the single call wherever both run (rewards bit for bit, accumulators up to the fp64 addition order, the same
work counters), results do not depend on the pose chunk above the cap, the numpy oracle, the fold, ModelTraj (eager,
CUDA graphs, prior and weight edits, observed_logodds) and the documented errors."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import coverage_oracle as orc
from tests.conftest import load_golden, rel_err, row_rel_err

pytestmark = pytest.mark.gpu
VARIANTS = ["plain", "prior", "weight", "prior_weight", "upstream"]


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


def _cloud_np(gen, n):
    lo, hi = np.array([-10, -10, -1], np.float32), np.array([30, 30, 4], np.float32)
    return (gen.random((n, 3), dtype=np.float32) * (hi - lo) + lo).astype(np.float32)


def _long_path(W, seed=1):
    """W poses on a spiral through the cloud (every pose sees part of it)."""
    gen = np.random.default_rng(seed)
    t = np.linspace(0.0, 1.0, W)
    r = 4.0 + 10.0 * t
    poses = np.stack([10 + r * np.cos(6 * np.pi * t), 10 + r * np.sin(6 * np.pi * t), 0.3 * np.sin(40 * t)], 1)
    quats = gen.standard_normal((W, 4)) * 0.4 + np.array([1.0, 0, 0, 0])
    return poses.astype(np.float32), quats.astype(np.float32)


class Case:
    def __init__(self, ops, dev, pts_np, ordered, min_d=1.0, max_d=5.0):
        from trajectory_optimization_b200 import tools
        self.ops, self.dev = ops, dev
        pts = torch.from_numpy(pts_np).to(dev)
        self.perm = None
        if ordered:
            pts, self.perm = ops.spatial_sort(pts)
        self.pts, self.boxes = pts, ops.tile_boxes(pts)
        K, self.Wd, self.Hd = tools.load_intrinsics(dev)
        self.K, self.Kd = K, K.reshape(9).contiguous()
        self.cam = ops._lib.camera(self.Wd, self.Hd, min_d, max_d, 1e-6)

    def tensors(self, poses, quats):
        return torch.from_numpy(poses).to(self.dev), torch.from_numpy(quats).to(self.dev)


@pytest.fixture(scope="module")
def big(dev, mod):
    return Case(mod[2], dev, _cloud_np(np.random.default_rng(11), 1_000_000), True)


@pytest.fixture(scope="module")
def small(dev, mod):
    return Case(mod[2], dev, _cloud_np(np.random.default_rng(12), 40_000), False)


@pytest.fixture(scope="module")
def compact(dev, mod):
    g = load_golden("traj_compact")
    c = Case(mod[2], dev, g["in_points"].astype(np.float32), False, float(g["in_min_d"]), float(g["in_max_d"]))
    c.poses, c.quats = g["in_poses"].astype(np.float32), g["in_quats"].astype(np.float32)
    return c


def _terms(c, variant, ridx, seed=3):
    """prior, weight, upstream and the matching base of a variant (indexed like the rewards)."""
    B, n, gen = c.ops._BACKEND, c.pts.shape[0], np.random.default_rng(seed)
    prior = weight = up = base = None
    if "prior" in variant:
        p = gen.normal(0, 2, n).astype(np.float32)
        p[gen.choice(n, 8, replace=False)] = 30.0
        prior = torch.from_numpy(p).to(c.dev)
    if "weight" in variant:
        weight = torch.from_numpy(gen.random(n).astype(np.float32) * 2).to(c.dev)
    if variant == "upstream":
        up = torch.from_numpy(gen.standard_normal(n).astype(np.float32)).to(c.dev)
    if weight is not None:
        base = B.weight_sums(weight, prior)
    elif prior is not None:
        base = B.prior_sum(prior)
    return prior, weight, up, base


def _single(c, P, Q, mm, variant, ridx):
    """cov_traj_fused (one call): rewards, acc, epilogue output, work counters."""
    B, ops = c.ops._BACKEND, c.ops
    prior, weight, up, base = _terms(c, variant, ridx)
    r = torch.empty(c.pts.shape[0], dtype=torch.float32, device=c.dev)
    stats = torch.zeros(8, dtype=torch.int64, device=c.dev)
    with ops.evaluation(stats=stats):
        if weight is not None:
            acc = B.traj_fused(c.pts, P, Q, c.Kd, c.cam, mm, None, r, ridx, c.boxes, None, False, False, prior=prior,
                               weight=weight, wsums=base)
        elif prior is not None:
            acc = B.traj_fused(c.pts, P, Q, c.Kd, c.cam, mm, up, r, ridx, c.boxes, None, False, False, prior, base)
        else:
            acc = B.traj_fused(c.pts, P, Q, c.Kd, c.cam, mm, up, r, ridx, c.boxes, None, False, False)
    return r, acc, _epilogue(c, acc, mm, Q, up, weight, base), stats


def _long(c, P, Q, mm, variant, ridx, chunk):
    B, ops = c.ops._BACKEND, c.ops
    prior, weight, up, base = _terms(c, variant, ridx)
    r = torch.empty(c.pts.shape[0], dtype=torch.float32, device=c.dev)
    stats = torch.zeros(8, dtype=torch.int64, device=c.dev)
    with ops.evaluation(stats=stats):
        acc = B.traj_fused_long(c.pts, P, Q, c.Kd, c.cam, mm, up, r, ridx, c.boxes, None, False, prior, base, weight,
                                chunk)
    return r, acc, _epilogue(c, acc, mm, Q, up, weight, base), stats


def _epilogue(c, acc, mm, Q, up, weight, base):
    B = c.ops._BACKEND
    if weight is not None:
        return B.traj_epilogue(acc, mm, Q, c.pts.shape[0], 0, base[1:])
    return B.traj_epilogue(acc, mm, Q, c.pts.shape[0], 0 if up is None else 1)


def _compare(a, b, W, tol_grad, counters=True, tol_mean=1e-12):
    ra, acca, oa, sa = a
    rb, accb, ob, sb = b
    assert torch.equal(ra, rb)
    assert rel_err(accb[W * 22].item(), acca[W * 22].item()) < tol_mean
    oa, ob = oa.cpu().numpy(), ob.cpu().numpy()
    assert row_rel_err(ob[1:1 + 3 * W].reshape(W, 3), oa[1:1 + 3 * W].reshape(W, 3)) < tol_grad
    assert row_rel_err(ob[1 + 3 * W:].reshape(W, 4), oa[1 + 3 * W:].reshape(W, 4)) < tol_grad
    if counters:
        assert sa[1].item() == sb[1].item() and sa[4].item() == sb[4].item() and sa[1].item() > 0


@pytest.mark.parametrize("ridx", [False, True])
@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("chunk", [1, 37, 1024])
@pytest.mark.parametrize("W", [320, 1100, 2048])
def test_carry_reproduces_the_single_call_pruned(W, chunk, variant, ridx, big):
    c = big
    P, Q = c.tensors(*_long_path(W))
    mm = c.ops._BACKEND.sweep_minmax(c.pts, P, Q, c.Kd, c.cam, c.boxes)
    idx = c.perm if ridx else None
    _compare(_single(c, P, Q, mm, variant, idx), _long(c, P, Q, mm, variant, idx, chunk), W, 1e-5)


def _dense_mean_tol(variant):
    # the pruned kernels add r_j - sigmoid(prior_j), formed in fp32, to sum_j sigmoid(prior_j) where the dense kernel adds
    # r_j: with a prior the means of the two paths differ by those roundings (~1e-11), as the single pruned call's do
    return 1e-9 if "prior" in variant else 1e-12


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("chunk", [1, 37, 1024])
@pytest.mark.parametrize("W", [320, 1100])
def test_carry_reproduces_the_dense_single_call_on_small_clouds(W, chunk, variant, small):
    c = small
    P, Q = c.tensors(*_long_path(W))
    mm = c.ops._BACKEND.sweep_minmax(c.pts, P, Q, c.Kd, c.cam, c.boxes)
    _compare(_single(c, P, Q, mm, variant, None), _long(c, P, Q, mm, variant, None, chunk), W, 5e-6, counters=False,
             tol_mean=_dense_mean_tol(variant))


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("chunk", [1, 2, 1024])
def test_carry_on_the_compact_cloud_with_argmin_ties(chunk, variant, compact):
    c = compact
    P, Q = c.tensors(c.poses, c.quats)
    mm = c.ops._BACKEND.sweep_minmax(c.pts, P, Q, c.Kd, c.cam, c.boxes)
    assert int((mm[:5] > 0).sum()) >= 4   # minima above 0: the arg-min tie accumulators run
    _compare(_single(c, P, Q, mm, variant, None), _long(c, P, Q, mm, variant, None, chunk), 5, 5e-6, counters=False,
             tol_mean=_dense_mean_tol(variant))


@pytest.mark.parametrize("W", [2049, 4096, 4097, 6000])
def test_chunk_invariance_above_the_cap(W, big):
    c = big
    P, Q = c.tensors(*_long_path(W, seed=W))
    mm = c.ops._BACKEND.sweep_minmax(c.pts, P, Q, c.Kd, c.cam, c.boxes)
    variant = "prior" if W % 2 else "plain"
    ref = _long(c, P, Q, mm, variant, c.perm, 2048)
    for chunk in (1000, 333):
        _compare(ref, _long(c, P, Q, mm, variant, c.perm, chunk), W, 1e-5)


def test_chunk_invariance_on_a_compact_cloud(compact):
    c = compact
    gen = np.random.default_rng(4)
    W = 2100
    poses = np.tile(c.poses, (W // 5, 1)) + gen.normal(0, 2e-3, (W, 3)).astype(np.float32)
    quats = np.tile(c.quats, (W // 5, 1)) + gen.normal(0, 2e-3, (W, 4)).astype(np.float32)
    P, Q = c.tensors(poses.astype(np.float32), quats.astype(np.float32))
    mm = c.ops._BACKEND.sweep_minmax(c.pts, P, Q, c.Kd, c.cam, c.boxes)
    pos = (mm[:W] > 0).cpu()
    assert int(pos.sum()) >= W * 3 // 4   # minima above 0: the arg-min accumulators run in every chunk
    ref = _long(c, P, Q, mm, "plain", None, 2048)
    assert bool((ref[1][21:W * 22:22].cpu()[pos] > 0).all())   # every such pose has its arg-min ties
    for chunk in (1000, 333):
        _compare(ref, _long(c, P, Q, mm, "plain", None, chunk), W, 1e-5)


def _circle_path(W, seed):
    """W poses on two turns of a 3 m circle inside the dense oracle cloud (each pose sees many points, so that no pose's
    gradient hangs on the fp32 gate of a handful of points)."""
    gen = np.random.default_rng(seed)
    t = np.linspace(0.0, 4 * np.pi, W)
    poses = np.stack([10 + 3 * np.cos(t), 10 + 3 * np.sin(t), 0.2 * np.sin(5 * t)], 1)
    quats = gen.standard_normal((W, 4)) * 0.2 + np.array([1.0, 0, 0, 0])
    return poses.astype(np.float32), quats.astype(np.float32)


def test_long_trajectory_matches_the_oracle(dev, mod):
    _, tools, ops = mod
    gen = np.random.default_rng(22)
    pts = (gen.random((20_000, 3)) * np.array([12, 12, 3]) + np.array([4, 4, -1])).astype(np.float32)
    poses, quats = _circle_path(2500, seed=5)
    K, Wd, Hd = tools.load_intrinsics(dev)
    P = torch.from_numpy(poses).to(dev).requires_grad_(True)
    Q = torch.from_numpy(quats).to(dev).requires_grad_(True)
    rewards, mean = ops.coverage_traj(torch.from_numpy(pts).to(dev), P, Q, K, Wd, Hd)
    vis = 1.0 / (mean + 1e-6)
    gp, gq = torch.autograd.grad(vis, [P, Q])
    Kn, Wn, Hn = orc.load_intrinsics()
    ref = orc.traj_objective(pts, poses, quats, Kn, Wn, Hn, dtype=np.float64)
    assert rel_err(rewards.detach().cpu().numpy(), ref["rewards"]) < 1e-4
    assert rel_err(vis.item(), ref["vis"]) < 1e-4
    assert row_rel_err(gp.cpu().numpy(), ref["g_poses"]) < 2e-4
    assert row_rel_err(gq.cpu().numpy(), ref["g_quats"]) < 2e-4


@pytest.mark.parametrize("with_prior", [False, True])
def test_fold_equals_the_rewards_bit_for_bit(with_prior, big):
    c, ops = big, big.ops
    P, Q = c.tensors(*_long_path(4097, seed=9))
    prior = _terms(c, "prior", c.perm)[0] if with_prior else None
    kw = dict(reward_index=c.perm, boxes=c.boxes, prior_logodds=prior)
    lo = ops.traj_logodds(c.pts, P, Q, c.K, c.Wd, c.Hd, **kw)
    rewards, _ = ops.coverage_traj(c.pts, P, Q, c.K, c.Wd, c.Hd, **kw)
    assert torch.equal(_sig(lo), rewards)
    assert int((lo != (0 if prior is None else prior)).sum()) > 0


def test_model_traj_with_a_long_path(dev, mod):
    from trajectory_optimization_b200.graphs import GraphedStep
    model, tools, ops = mod
    gen = np.random.default_rng(31)
    K, Wd, Hd = tools.load_intrinsics(dev)
    pts = torch.from_numpy(_cloud_np(gen, 200_000))
    poses, quats = _long_path(2600, seed=7)
    n = pts.shape[0]
    # a few Adam steps reduce the loss (on the camera orientations: the path's smoothness and length terms stay put)
    m = model.ModelTraj(pts, torch.from_numpy(poses), torch.from_numpy(quats), K, Wd, Hd, device=dev)
    opt = torch.optim.Adam([m.quats], lr=0.005)
    losses = []
    for _ in range(4):
        opt.zero_grad()
        loss = m(vis_wps_dist=0.0)
        loss.backward()
        opt.step()
        losses.append(loss.item())
    assert losses[-1] < losses[0]
    m(vis_wps_dist=0.0)   # the rewards at the current poses
    assert torch.equal(_sig(m.observed_logodds(vis_wps_dist=0.0)), m.rewards.detach())
    # a replay computes what the eager step computes; prior and weight edits are seen by the replay
    pr = torch.from_numpy(gen.normal(0, 1, n).astype(np.float32)).to(dev)
    wt = torch.from_numpy(gen.random(n).astype(np.float32)).to(dev)
    m2 = model.ModelTraj(pts, torch.from_numpy(poses), torch.from_numpy(quats), K, Wd, Hd, device=dev,
                         prior_logodds=pr.clone(), point_weight=wt.clone())
    opt2 = torch.optim.Adam([m2.poses, m2.quats], lr=0.0, capturable=True)
    g = GraphedStep(m2, opt2, forward_kwargs=dict(vis_wps_dist=0.0), warmup=1)
    g.step()
    torch.cuda.synchronize()
    replay = m2.rewards.detach().clone()
    mean_replay = m2._mean.item()
    ref, mean = ops.coverage_traj(m2._cloud(), m2.poses.detach(), m2.quats.detach(), K, Wd, Hd, reward_index=m2._perm,
                                  boxes=m2._boxes, prior_logodds=pr, weight=wt)
    assert torch.equal(replay, ref) and rel_err(mean_replay, mean.item()) < 1e-6
    m2.set_prior_logodds(pr + 1.5)
    m2.set_point_weight(wt * wt)
    g.step()
    torch.cuda.synchronize()
    ref2, mean2 = ops.coverage_traj(m2._cloud(), m2.poses.detach(), m2.quats.detach(), K, Wd, Hd, reward_index=m2._perm,
                                    boxes=m2._boxes, prior_logodds=pr + 1.5, weight=wt * wt)
    assert not torch.equal(ref2, replay)
    assert torch.equal(m2.rewards.detach(), ref2) and rel_err(m2._mean.item(), mean2.item()) < 1e-6


def test_errors(big):
    c, ops = big, big.ops
    P, Q = c.tensors(*_long_path(2049))
    with pytest.raises(RuntimeError, match="exceed"):
        ops.coverage_traj(c.pts, P, Q, c.K, c.Wd, c.Hd, dense=True)
    L = ops._lib.lib()
    n, W = c.pts.shape[0], P.shape[0]
    mm = ops._BACKEND.sweep_minmax(c.pts, P, Q, c.Kd, c.cam, c.boxes)
    rewards = torch.empty(n, dtype=torch.float32, device=c.dev)
    acc = torch.empty(W * 22 + 1, dtype=torch.float64, device=c.dev)
    need = L.cov_traj_long_workspace_bytes(n, W, 0)
    ws = torch.empty(need + 256, dtype=torch.uint8, device=c.dev)
    p = ops._ptr
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def call(chunk, ws_ptr, ws_bytes):
        return L.cov_traj_fused_long(p(c.pts), n, p(P), p(Q), W, p(c.Kd), ctypes.byref(c.cam), p(c.boxes), p(mm), None,
                                     None, p(rewards), p(acc), None, None, None, chunk, None, ws_ptr, ws_bytes, stream)

    assert call(-1, p(ws), need) == -1 and call(2049, p(ws), need) == -1        # COV_ERR_ARG
    assert call(0, p(ws), need - 1) == -3                                         # COV_ERR_WORKSPACE
    assert call(0, ctypes.c_void_p(ws.data_ptr() + 16), need) == -5               # COV_ERR_ALIGN
    lo = torch.zeros(n, dtype=torch.float32, device=c.dev)
    assert L.cov_traj_logodds_long(p(c.pts), n, p(P), p(Q), W, p(c.Kd), ctypes.byref(c.cam), p(c.boxes), p(mm), None,
                                   p(lo), 5000, None, p(ws), need, stream) == -1
    assert call(0, p(ws), need) == 0
    torch.cuda.synchronize()
