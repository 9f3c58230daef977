"""The prefix sweep on the GPU: every column of ops.sweep_prefix_rewards is the sweep of the trajectories cut after that
pose (to 1e-12: only the order of fp64 additions differs), with and without prior and weight, on the pruned and the dense
path, across pose chunks, for P = 1 and P = 2048, against coverage_traj, for padded ragged candidates, through a pose
that sees nothing, in ModelTrajBatch.prefix_means, and the errors of the op and of the raw C ABI."""
import ctypes

import numpy as np
import pytest
import torch

from tests.conftest import rel_err

pytestmark = pytest.mark.gpu
TIGHT = 1e-12


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def mod():
    from trajectory_optimization_b200 import _lib, model, ops, tools
    _lib.lib()
    return model, tools, ops


def _cloud(gen, n):
    lo, hi = np.array([-10, -10, -1], np.float32), np.array([30, 30, 4], np.float32)
    return (gen.random((n, 3), dtype=np.float32) * (hi - lo) + lo).astype(np.float32)


def _candidates(gen, T, P, step=1.2):
    """T trajectories of P poses `step` apart on circles inside the cloud (every pose sees points), random orientations."""
    centre = gen.uniform([2, 2, 0], [18, 18, 1], (T, 1, 3))
    radius = gen.uniform(2, 7, (T, 1))
    ang = gen.uniform(0, 2 * np.pi, (T, 1)) + step / radius * np.arange(P)[None, :]
    poses = centre + np.stack([radius * np.cos(ang), radius * np.sin(ang), np.zeros((T, P))], 2)
    quats = gen.standard_normal((T, P, 4)) * 0.4 + np.array([1.0, 0, 0, 0])
    return poses.astype(np.float32), quats.astype(np.float32)


@pytest.fixture(scope="module")
def cloud(dev, mod):
    """A Morton-ordered 300 k-point cloud, its boxes, a prior and a weight in the cloud's order."""
    _, _, ops = mod
    gen = np.random.default_rng(41)
    pts, _ = ops.spatial_sort(torch.from_numpy(_cloud(gen, 300_000)).to(dev))
    n = pts.shape[0]
    prior = torch.from_numpy(gen.normal(0, 2, n).astype(np.float32)).to(dev)
    w = (gen.random(n) * 2).astype(np.float32)
    w[gen.random(n) < 0.3] = 0.0
    return pts, ops.tile_boxes(pts), prior, torch.from_numpy(w).to(dev)


def _variants(prior, weight):
    return {"plain": {}, "prior": dict(prior_logodds=prior), "weight": dict(weight=weight),
            "both": dict(prior_logodds=prior, weight=weight)}


def _check_columns(ops, pts, boxes, P, Q, K, Wd, Hd, got, cols, **kw):
    """got[:, i] == sweep_rewards of the trajectories cut after pose i, for every i in cols."""
    for i in cols:
        cut = ops.sweep_rewards(pts, P[:, :i + 1], Q[:, :i + 1], K, Wd, Hd, boxes=boxes, presorted=True, **kw)
        assert rel_err(got[:, i].cpu().numpy(), cut.cpu().numpy()) < TIGHT, i


@pytest.mark.parametrize("T,Pn", [(20, 9), (20, 1), (70, 33)])
def test_prefix_columns_equal_truncated_sweeps(T, Pn, dev, mod, cloud):
    """(70, 33): 2310 poses, two chunks of 62 trajectories and an uneven last one of 8."""
    _, tools, ops = mod
    pts, boxes, _, _ = cloud
    K, Wd, Hd = tools.load_intrinsics(dev)
    poses, quats = _candidates(np.random.default_rng(T * 100 + Pn), T, Pn)
    P, Q = torch.from_numpy(poses).to(dev), torch.from_numpy(quats).to(dev)
    got = ops.sweep_prefix_rewards(pts, P, Q, K, Wd, Hd, boxes=boxes, presorted=True)
    assert got.shape == (T, Pn) and got.dtype == torch.float64 and bool(torch.isfinite(got).all())
    _check_columns(ops, pts, boxes, P, Q, K, Wd, Hd, got, range(Pn))


def test_prefix_of_2048_poses(dev, mod, cloud):
    _, tools, ops = mod
    pts, boxes, _, _ = cloud
    K, Wd, Hd = tools.load_intrinsics(dev)
    poses, quats = _candidates(np.random.default_rng(2048), 2, 2048, step=0.02)
    P, Q = torch.from_numpy(poses).to(dev), torch.from_numpy(quats).to(dev)
    got = ops.sweep_prefix_rewards(pts, P, Q, K, Wd, Hd, boxes=boxes, presorted=True)
    assert got.shape == (2, 2048)
    _check_columns(ops, pts, boxes, P, Q, K, Wd, Hd, got, (0, 1, 1023, 2047))


def test_prefix_with_prior_and_weight(dev, mod, cloud):
    """Prior, weight and both against the truncated sweeps with the same prior and weight; a zero prior and unit weights
    reproduce the plain prefixes; every row is non-decreasing."""
    _, tools, ops = mod
    pts, boxes, prior, weight = cloud
    K, Wd, Hd = tools.load_intrinsics(dev)
    T, Pn = 20, 9
    poses, quats = _candidates(np.random.default_rng(9), T, Pn)
    P, Q = torch.from_numpy(poses).to(dev), torch.from_numpy(quats).to(dev)
    run = lambda **kw: ops.sweep_prefix_rewards(pts, P, Q, K, Wd, Hd, boxes=boxes, presorted=True, **kw)  # noqa: E731
    for name, kw in _variants(prior, weight).items():
        got = run(**kw)
        assert bool(torch.isfinite(got).all()), name
        _check_columns(ops, pts, boxes, P, Q, K, Wd, Hd, got, range(Pn), **kw)
        assert bool((got[:, 1:] >= got[:, :-1] - 1e-9).all()), name
    plain = run()
    zero, ones = torch.zeros_like(prior), torch.ones_like(weight)
    for kw in (dict(prior_logodds=zero), dict(weight=ones), dict(prior_logodds=zero, weight=ones)):
        assert rel_err(run(**kw).cpu().numpy(), plain.cpu().numpy()) < TIGHT


def test_prefix_equals_coverage_traj_means(dev, mod, cloud):
    _, tools, ops = mod
    pts, boxes, prior, weight = cloud
    K, Wd, Hd = tools.load_intrinsics(dev)
    T, Pn = 20, 9
    poses, quats = _candidates(np.random.default_rng(9), T, Pn)
    P, Q = torch.from_numpy(poses).to(dev), torch.from_numpy(quats).to(dev)
    for kw in ({}, dict(prior_logodds=prior, weight=weight)):
        got = ops.sweep_prefix_rewards(pts, P, Q, K, Wd, Hd, boxes=boxes, presorted=True, **kw)
        for t in (0, 7, 19):
            for i in range(Pn):
                _, mean = ops.coverage_traj(pts, P[t, :i + 1], Q[t, :i + 1], K, Wd, Hd, boxes=boxes, **kw)
                assert rel_err(got[t, i].item(), mean.item()) < 1e-6, (t, i)


@pytest.mark.parametrize("n", [50_000, 300_000])
def test_dense_prefix(n, dev, mod, cloud):
    """evaluation(dense=True): the dense kernel's prefixes match the pruned ones to 1e-6 and the dense sweeps of the
    truncated trajectories to 1e-12."""
    _, tools, ops = mod
    pts, boxes, prior, weight = cloud
    pts, boxes, prior, weight = (pts, boxes, prior, weight) if n == pts.shape[0] else \
        (pts[:n].contiguous(), ops.tile_boxes(pts[:n].contiguous()), prior[:n].contiguous(), weight[:n].contiguous())
    K, Wd, Hd = tools.load_intrinsics(dev)
    T, Pn = 12, 7
    poses, quats = _candidates(np.random.default_rng(n), T, Pn)
    P, Q = torch.from_numpy(poses).to(dev), torch.from_numpy(quats).to(dev)
    for kw in ({}, dict(prior_logodds=prior, weight=weight)):
        pruned = ops.sweep_prefix_rewards(pts, P, Q, K, Wd, Hd, boxes=boxes, presorted=True, **kw)
        with ops.evaluation(dense=True):
            dense = ops.sweep_prefix_rewards(pts, P, Q, K, Wd, Hd, boxes=boxes, presorted=True, **kw)
            _check_columns(ops, pts, boxes, P, Q, K, Wd, Hd, dense, range(Pn), **kw)
        assert rel_err(dense.cpu().numpy(), pruned.cpu().numpy()) < 1e-6


def test_ragged_candidates_by_padding(dev, mod, cloud):
    """Trajectories of lengths 3 .. P padded to P by repeating their last pose: column len_t - 1 is the sweep of each
    unpadded trajectory alone."""
    _, tools, ops = mod
    pts, boxes, _, _ = cloud
    K, Wd, Hd = tools.load_intrinsics(dev)
    Pn = 10
    lengths = list(range(3, Pn + 1))
    poses, quats = _candidates(np.random.default_rng(77), len(lengths), Pn)
    for t, ln in enumerate(lengths):
        poses[t, ln:], quats[t, ln:] = poses[t, ln - 1], quats[t, ln - 1]
    P, Q = torch.from_numpy(poses).to(dev), torch.from_numpy(quats).to(dev)
    got = ops.sweep_prefix_rewards(pts, P, Q, K, Wd, Hd, boxes=boxes, presorted=True)
    for t, ln in enumerate(lengths):
        alone = ops.sweep_rewards(pts, P[t:t + 1, :ln], Q[t:t + 1, :ln], K, Wd, Hd, boxes=boxes, presorted=True)
        assert rel_err(got[t, ln - 1].item(), alone.item()) < TIGHT, t


def test_pose_that_sees_nothing(dev, mod, cloud):
    """A pose far from the cloud in the middle of trajectory 3: its earlier prefixes are finite and match the truncated
    sweeps, from it on they are NaN as the truncated sweeps are; the other trajectories are unaffected."""
    _, tools, ops = mod
    pts, boxes, _, _ = cloud
    K, Wd, Hd = tools.load_intrinsics(dev)
    T, Pn, t_far, k_far = 6, 8, 3, 4
    poses, quats = _candidates(np.random.default_rng(5), T, Pn)
    poses[t_far, k_far] = (1.0e4, 1.0e4, 0.0)
    P, Q = torch.from_numpy(poses).to(dev), torch.from_numpy(quats).to(dev)
    got = ops.sweep_prefix_rewards(pts, P, Q, K, Wd, Hd, boxes=boxes, presorted=True)
    g = got.cpu().numpy()
    assert np.isfinite(g[t_far, :k_far]).all() and np.isnan(g[t_far, k_far:]).all()
    for i in range(Pn):
        cut = ops.sweep_rewards(pts, P[:, :i + 1], Q[:, :i + 1], K, Wd, Hd, boxes=boxes, presorted=True).cpu().numpy()
        assert np.array_equal(np.isnan(g[:, i]), np.isnan(cut)), i
        ok = np.isfinite(cut)
        assert rel_err(g[ok, i], cut[ok]) < TIGHT, i
    others = [t for t in range(T) if t != t_far]
    alone = ops.sweep_prefix_rewards(pts, P[others], Q[others], K, Wd, Hd, boxes=boxes, presorted=True).cpu().numpy()
    assert np.isfinite(g[others]).all() and rel_err(g[others], alone) < TIGHT


@pytest.mark.parametrize("dense", [False, True])
def test_model_traj_batch_prefix_means(dense, dev, mod, cloud):
    """prefix_means equals the op on the strided waypoints with the model's prior and weight (set through the setters);
    its last column is `means` of a forward."""
    model, tools, ops = mod
    pts, _, prior, weight = cloud
    K, Wd, Hd = tools.load_intrinsics(dev)
    T, W = 6, 13
    xs = np.arange(W, dtype=np.float32) * 0.4   # waypoints 0.4 m apart: stride 2 at vis_wps_dist = 0.5
    gen = np.random.default_rng(13)
    wp = np.stack([np.stack([xs + o[0], np.full(W, o[1], np.float32), np.zeros(W, np.float32)], 1)
                   for o in gen.uniform(-3, 15, (T, 2)).astype(np.float32)])
    wq = (gen.standard_normal((T, W, 4)) * 0.3 + np.array([1.0, 0, 0, 0])).astype(np.float32)
    m = model.ModelTrajBatch(pts, torch.from_numpy(wp), torch.from_numpy(wq), K, Wd, Hd, device=dev, spatial_sort=not dense)
    for kw in ({}, dict(prior_logodds=prior, weight=weight)):
        if kw:
            # the model takes them in the order of its points (the cloud as given)
            m.set_prior_logodds(prior)
            m.set_point_weight(weight)
        m(vis_wps_dist=0.5)
        got = m.prefix_means(vis_wps_dist=0.5)
        step = m._wps_step(0.5)
        assert got.shape == (T, len(range(0, W, step))) and not got.requires_grad
        with ops.evaluation(dense=dense):
            ref = ops.sweep_prefix_rewards(pts, m.poses.detach()[:, ::step], m.quats.detach()[:, ::step], K, Wd, Hd,
                                           presorted=dense, **kw)
        assert rel_err(got.cpu().numpy(), ref.cpu().numpy()) < 1e-9
        assert rel_err(got[:, -1].cpu().numpy(), m.means.detach().cpu().numpy()) < 1e-6


def test_errors(dev, mod, cloud):
    from trajectory_optimization_b200 import _lib
    _, tools, ops = mod
    pts, boxes, prior, weight = cloud
    K, Wd, Hd = tools.load_intrinsics(dev)
    poses, quats = _candidates(np.random.default_rng(1), 1, 2049, step=0.02)
    with pytest.raises(RuntimeError, match="exceed the pose mask"):
        ops.sweep_prefix_rewards(pts, torch.from_numpy(poses).to(dev), torch.from_numpy(quats).to(dev), K, Wd, Hd,
                                 boxes=boxes, presorted=True)
    # raw C ABI: base_dev must match the prior / weight pointers
    L = _lib.lib()
    T, Pn = 2, 3
    poses, quats = _candidates(np.random.default_rng(2), T, Pn)
    P = torch.from_numpy(poses).to(dev).reshape(-1, 3)
    Q = torch.from_numpy(quats).to(dev).reshape(-1, 4)
    Kd = K.reshape(9).contiguous()
    cam = _lib.camera(Wd, Hd, 1.0, 5.0, 1e-6)
    minmax = ops._BACKEND.sweep_minmax(pts, P, Q, Kd, cam, boxes)
    n = pts.shape[0]
    ws_bytes = L.cov_sweep_workspace_bytes(n, T, Pn)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    out = torch.empty(T * Pn, dtype=torch.float64, device=dev)
    base = torch.zeros(2, dtype=torch.float64, device=dev)
    p = lambda t: ctypes.c_void_p(0 if t is None else t.data_ptr())  # noqa: E731
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)

    def call(pr, w, b):
        return L.cov_sweep_prefix_rewards(p(pts), n, p(P), p(Q), T, Pn, p(Kd), ctypes.byref(cam), p(boxes), p(minmax),
                                          p(pr), p(w), p(b), p(out), None, p(ws), ws_bytes, stream)

    for pr, w, b in ((None, None, base), (prior, None, None), (None, weight, None), (prior, weight, None)):
        assert call(pr, w, b) == -1   # COV_ERR_ARG
        assert b"base" in L.cov_last_error() or b"null" in L.cov_last_error()
    assert call(None, None, None) == 0
    torch.cuda.synchronize(dev)
    ref = ops.sweep_prefix_rewards(pts, P.reshape(T, Pn, 3), Q.reshape(T, Pn, 4), K, Wd, Hd, boxes=boxes, presorted=True)
    assert rel_err((out / n).reshape(T, Pn).cpu().numpy(), ref.cpu().numpy()) < TIGHT
