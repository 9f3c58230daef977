"""The differentiable candidate sweep on the GPU: cov_sweep_fused / cov_sweep_epilogue against the single-trajectory
pass B and epilogue, ops.coverage_sweep against coverage_traj, sweep_rewards, the dense path and the reference fixtures,
the rig front end, and ModelTrajBatch against T separate ModelTraj models (eager and CUDA-graphed)."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import coverage_oracle as orc
from tests.conftest import load_golden, rel_err, row_rel_err

pytestmark = pytest.mark.gpu
TOL_ROW = 2e-4   # per-pose gradient rows, each against its own magnitude (as test_gpu_coverage.py)
ACC = 22


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def mod():
    from trajectory_optimization_b200 import model, tools, ops, _lib
    _lib.lib()  # fail loudly if the extension is not built
    return model, tools, ops


def _box(gen, n, lo=(-10, -10, -1), hi=(30, 30, 4)):
    lo, hi = np.array(lo, np.float32), np.array(hi, np.float32)
    return (gen.random((n, 3), dtype=np.float32) * (hi - lo) + lo).astype(np.float32)


def _candidates(gen, T, Pn, length=10.0, spread=1.0):
    xs = np.linspace(0, length, Pn)
    base = np.stack([xs, 0.5 * xs + 0.3 * np.sin(xs), np.zeros(Pn)], 1).astype(np.float32)
    yaw = np.arctan2(0.5 + 0.3 * np.cos(xs), 1.0)
    poses = base[None] + gen.normal(0, spread, (T, 1, 3)).astype(np.float32) * np.array([1, 1, 0], np.float32)
    ang = yaw[None, :] + gen.normal(0, 0.3, (T, Pn))
    quats = np.stack([np.cos(ang / 2), 0 * ang, 0 * ang, np.sin(ang / 2)], -1).astype(np.float32)
    return poses.astype(np.float32), quats


def _compact(gen, n, T, Pn):
    """A cloud in front of every camera and within a few metres: min_j m > 0 for every pose (arg-min ties carry
    gradient, ctrl[1] is set)."""
    pts = _box(gen, n, (1.0, 1.0, 1.5), (4.0, 4.0, 4.5))
    poses = (gen.random((T, Pn, 3), dtype=np.float32) * 0.6 - 0.3).astype(np.float32)
    quats = (np.array([1.0, 0, 0, 0]) + gen.normal(0, 0.15, (T, Pn, 4))).astype(np.float32)
    return pts, poses, quats


def _row_rel(a, b):
    """max over rows of |a - b|_inf / |b|_inf (rows that are zero in b must be zero in a)."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    nb = np.abs(b).max(axis=1)
    d = np.abs(a - b).max(axis=1)
    return float(np.where(nb > 0, d / np.where(nb > 0, nb, 1.0), d).max())


@pytest.mark.parametrize("case", ["P7", "P32", "P33_two_chunks_ragged", "compact"])
def test_sweep_accumulators_match_single_trajectory_pass_b(case, dev, mod):
    """Raw C ABI: every block of cov_sweep_fused is cov_traj_fused(W = P) of that trajectory on the same cloud, boxes and
    normalisers: tie counts equal, gradient and tie rows to 1e-12 per row (only the fp64 addition order differs), the
    reward sum to 1e-6."""
    model, tools, ops = mod
    from trajectory_optimization_b200 import _lib
    gen = np.random.default_rng({"P7": 1, "P32": 2, "P33_two_chunks_ragged": 3, "compact": 4}[case])
    if case == "compact":
        T, Pn = 9, 6
        pts_np, poses, quats = _compact(gen, 300_001, T, Pn)
    else:
        T, Pn, n = {"P7": (12, 7, 300_000), "P32": (8, 32, 400_000), "P33_two_chunks_ragged": (70, 33, 300_017)}[case]
        pts_np = _box(gen, n)
        poses, quats = _candidates(gen, T, Pn)
    pts, _ = ops.spatial_sort(torch.from_numpy(pts_np).to(dev))
    boxes = ops.tile_boxes(pts)
    K, Wd, Hd = tools.load_intrinsics(dev)
    Kd = K.reshape(9).contiguous()
    cam = _lib.camera(Wd, Hd, 1.0, 5.0, 1e-6)
    P = torch.from_numpy(poses).to(dev).reshape(-1, 3)
    Q = torch.from_numpy(quats).to(dev).reshape(-1, 4)
    B = ops._BACKEND
    stats = torch.zeros(8, dtype=torch.int64, device=dev)
    minmax = B.sweep_minmax(pts, P, Q, Kd, cam, boxes)
    with ops.evaluation(stats=stats):
        acc = B.sweep_fused(pts, P, Q, T, Pn, Kd, cam, boxes, minmax).cpu().numpy()
    TP = T * Pn
    rewards = torch.empty(pts.shape[0], dtype=torch.float32, device=dev)
    blk = Pn * ACC + 1
    if case == "compact":
        assert int((minmax[:TP] > 0).sum()) >= TP // 2
    for t in range(T):
        mm = torch.cat([minmax[t * Pn:(t + 1) * Pn], minmax[TP + t * Pn:TP + (t + 1) * Pn]])
        ref = B.traj_fused(pts, P[t * Pn:(t + 1) * Pn], Q[t * Pn:(t + 1) * Pn], Kd, cam, mm, None, rewards,
                           boxes=boxes).cpu().numpy()
        got = acc[t * blk:(t + 1) * blk]
        rows, rrows = got[:-1].reshape(Pn, ACC), ref[:-1].reshape(Pn, ACC)
        assert np.array_equal(rows[:, 14], rrows[:, 14]) and np.array_equal(rows[:, 21], rrows[:, 21]), (case, t)
        for lo, hi in ((0, 8), (8, 14), (15, 21)):
            assert _row_rel(rows[:, lo:hi], rrows[:, lo:hi]) < 1e-12, (case, t, lo)
        assert rel_err(got[-1], ref[-1]) < 1e-6
    s = stats.cpu().numpy()
    assert s[1] > 0 and s[4] > 0 and s[6] >= s[1] >= s[4] and s[0] >= s[6]


def test_sweep_epilogue_is_bit_identical_to_traj_epilogue(dev, mod):
    model, tools, ops = mod
    gen = np.random.default_rng(8)
    T, Pn = 13, 11
    acc = gen.normal(0, 1.0, (T, Pn * ACC + 1))
    rows = acc[:, :-1].reshape(T, Pn, ACC)
    rows[..., 14] = gen.integers(0, 3, (T, Pn))
    rows[..., 21] = gen.integers(0, 2, (T, Pn))
    acc[:, -1] = gen.random(T) * 1000
    mn = gen.random(T * Pn).astype(np.float32) * 0.1
    mx = mn + 0.5 + gen.random(T * Pn).astype(np.float32)
    minmax = torch.from_numpy(np.concatenate([mn, mx]).astype(np.float32)).to(dev)
    Q = torch.from_numpy(gen.normal(0, 1, (T * Pn, 4)).astype(np.float32)).to(dev)
    acc_d = torch.from_numpy(acc.reshape(-1)).to(dev)
    out = ops._BACKEND.sweep_epilogue(acc_d, minmax, Q, T, Pn, 12345).cpu()
    TP = T * Pn
    for t in range(T):
        mm = torch.cat([minmax[t * Pn:(t + 1) * Pn], minmax[TP + t * Pn:TP + (t + 1) * Pn]])
        ref = ops._BACKEND.traj_epilogue(acc_d[t * (Pn * ACC + 1):(t + 1) * (Pn * ACC + 1)], mm, Q[t * Pn:(t + 1) * Pn],
                                         12345, 0).cpu()
        assert torch.equal(out[t], ref[0])
        assert torch.equal(out[T + 3 * t * Pn:T + 3 * (t + 1) * Pn], ref[1:1 + 3 * Pn])
        assert torch.equal(out[T + 3 * TP + 4 * t * Pn:T + 3 * TP + 4 * (t + 1) * Pn], ref[1 + 3 * Pn:])


def _sweep_grads(ops, pts, poses, quats, K, Wd, Hd, weights=None, **kw):
    P = poses.clone().requires_grad_(True)
    Q = quats.clone().requires_grad_(True)
    means = ops.coverage_sweep(pts, P, Q, K, Wd, Hd, **kw)
    (means.sum() if weights is None else (weights * means).sum()).backward()
    return means.detach(), P.grad, Q.grad


def test_coverage_sweep_matches_coverage_traj_sweep_rewards_and_dense(dev, mod):
    model, tools, ops = mod
    gen = np.random.default_rng(12)
    T, Pn = 20, 9
    pts = torch.from_numpy(_box(gen, 300_000)).to(dev)
    poses_np, quats_np = _candidates(gen, T, Pn)
    poses, quats = torch.from_numpy(poses_np).to(dev), torch.from_numpy(quats_np).to(dev)
    K, Wd, Hd = tools.load_intrinsics(dev)
    means, gp, gq = _sweep_grads(ops, pts, poses, quats, K, Wd, Hd)
    assert means.shape == (T,) and means.dtype == torch.float32 and gp.shape == (T, Pn, 3) and gq.shape == (T, Pn, 4)
    for t in range(T):
        P = poses[t].clone().requires_grad_(True)
        Q = quats[t].clone().requires_grad_(True)
        _, mean = ops.coverage_traj(pts, P, Q, K, Wd, Hd)
        mean.backward()
        assert rel_err(means[t].item(), mean.item()) < 1e-6
        assert row_rel_err(gp[t].cpu().numpy(), P.grad.cpu().numpy()) < TOL_ROW
        assert row_rel_err(gq[t].cpu().numpy(), Q.grad.cpu().numpy()) < TOL_ROW
    fwd = ops.sweep_rewards(pts, poses, quats, K, Wd, Hd)
    assert rel_err(means.double().cpu().numpy(), fwd.cpu().numpy()) < 1e-6
    with ops.evaluation(dense=True):
        md, gpd, gqd = _sweep_grads(ops, pts, poses, quats, K, Wd, Hd)
    assert rel_err(md.cpu().numpy(), means.cpu().numpy()) < 1e-5
    assert row_rel_err(gp.cpu().numpy(), gpd.cpu().numpy()) < 1e-5
    assert row_rel_err(gq.cpu().numpy(), gqd.cpu().numpy()) < 1e-5
    # arbitrary upstream weights: trajectory t's gradient scaled by g_t
    g = torch.from_numpy(gen.normal(0, 1, T).astype(np.float32)).to(dev)
    _, gpw, gqw = _sweep_grads(ops, pts, poses, quats, K, Wd, Hd, weights=g)
    assert rel_err(gpw.cpu().numpy(), (g[:, None, None] * gp).cpu().numpy()) < 1e-6
    assert rel_err(gqw.cpu().numpy(), (g[:, None, None] * gq).cpu().numpy()) < 1e-6


def test_small_cloud_takes_the_dense_path(dev, mod):
    model, tools, ops = mod
    gen = np.random.default_rng(13)
    T, Pn = 6, 5
    pts = torch.from_numpy(_box(gen, 50_000, (-2, -2, -1), (14, 10, 3))).to(dev)
    poses_np, quats_np = _candidates(gen, T, Pn)
    poses, quats = torch.from_numpy(poses_np).to(dev), torch.from_numpy(quats_np).to(dev)
    K, Wd, Hd = tools.load_intrinsics(dev)
    means, gp, gq = _sweep_grads(ops, pts, poses, quats, K, Wd, Hd)
    for t in range(T):
        P = poses[t].clone().requires_grad_(True)
        Q = quats[t].clone().requires_grad_(True)
        _, mean = ops.coverage_traj(pts, P, Q, K, Wd, Hd)
        mean.backward()
        assert rel_err(means[t].item(), mean.item()) < 1e-6
        assert row_rel_err(gp[t].cpu().numpy(), P.grad.cpu().numpy()) < 1e-5
        assert row_rel_err(gq[t].cpu().numpy(), Q.grad.cpu().numpy()) < 1e-5


@pytest.mark.parametrize("name", ["traj_compact", "traj_sample"])
def test_sweep_reproduces_reference_fixtures(name, dev, mod, sample_inputs):
    """The fixture's trajectory among perturbed copies: its mean and visibility gradients as the reference computed."""
    model, tools, ops = mod
    g = load_golden(name)
    pts = torch.from_numpy(g["in_points"] if "in_points" in g else sample_inputs["pts"]).to(dev)
    K, Wd, Hd = tools.load_intrinsics(dev)
    step = int(g["out_wps_step"])
    gen = np.random.default_rng(14)
    p0, q0 = g["in_poses"].astype(np.float32), g["in_quats"].astype(np.float32)
    T, k = 4, 2
    poses = np.repeat(p0[None], T, 0) + gen.normal(0, 0.3, (T, 1, 3)).astype(np.float32)
    quats = np.repeat(q0[None], T, 0) + gen.normal(0, 0.05, (T,) + q0.shape).astype(np.float32)
    poses[k], quats[k] = p0, q0
    P = torch.from_numpy(poses).to(dev).requires_grad_(True)
    Q = torch.from_numpy(quats).to(dev).requires_grad_(True)
    means = ops.coverage_sweep(pts, P[:, ::step], Q[:, ::step], K, Wd, Hd, float(g["in_min_d"]), float(g["in_max_d"]))
    vis = 1.0 / (means[k] + 1e-6)
    vis.backward()
    assert rel_err(vis.item(), g["out_vis64"]) < 1e-4
    for got, ref in ((P.grad[k], g["out_gv_poses64"]), (Q.grad[k], g["out_gv_quats64"])):
        got = got.cpu().numpy()
        assert rel_err(got, ref) < 1e-4 and row_rel_err(got, ref) < TOL_ROW
    others = [t for t in range(T) if t != k]
    assert float(P.grad[others].abs().max()) == 0.0   # d vis_k / d poses_t = 0 for t != k


def test_rig_chain_through_the_sweep(dev, mod):
    """T rigs: camera_poses_fused on (T n_body, 4) bodies -> (T, n_body C, .) -> coverage_sweep gives every body the
    gradient of its own trajectory's coverage_traj chain."""
    from trajectory_optimization_b200 import multicam
    model, tools, ops = mod
    gen = np.random.default_rng(17)
    pts = torch.from_numpy(_box(gen, 200_000)).to(dev)
    K, Wd, Hd = tools.load_intrinsics(dev)
    rig7 = multicam.rig_tensor(multicam.ring_rig(3, lever=(0.3, -0.1, 0.2)), dev)
    T, nb, C = 5, 6, 3
    xs = np.linspace(0, 8, nb)
    base = np.stack([xs, 0.5 * xs, np.zeros(nb), np.full(nb, 0.4)], 1)
    body0 = torch.from_numpy((base[None] + gen.normal(0, 0.5, (T, 1, 4)) * np.array([1, 1, 0, 0.3]))
                             .astype(np.float32)).to(dev)
    body = body0.clone().requires_grad_(True)
    t, q = multicam.camera_poses_fused(body.reshape(T * nb, 4), rig7)
    means = ops.coverage_sweep(pts, t.reshape(T, nb * C, 3), q.reshape(T, nb * C, 4), K, Wd, Hd)
    (1.0 / (means + 1e-6)).sum().backward()
    for i in range(T):
        b = body0[i].clone().requires_grad_(True)
        ti, qi = multicam.camera_poses_fused(b, rig7)
        _, mean = ops.coverage_traj(pts, ti, qi, K, Wd, Hd)
        (1.0 / (mean + 1e-6)).backward()
        assert rel_err(means[i].item(), mean.item()) < 1e-6
        assert row_rel_err(body.grad[i].cpu().numpy(), b.grad.cpu().numpy()) < TOL_ROW


def _batch_case(gen, T=4, W=10):
    pts = torch.from_numpy(_box(gen, 150_000))
    poses, quats = _candidates(gen, T, W, length=9.0, spread=0.4)
    return pts, torch.from_numpy(poses), torch.from_numpy(quats)


@pytest.mark.parametrize("spacing", ["curved", "even"])
def test_model_traj_batch_equals_separate_models(spacing, dev, mod):
    """Per-trajectory losses and gradients of T separate ModelTraj models.  "even": straight rows of waypoints 0.1 m
    apart, where ModelTraj's fp32 stride arithmetic picks stride 6 at vis_wps_dist = 0.5 (an fp64 division would give 5)."""
    model, tools, ops = mod
    gen = np.random.default_rng(19)
    pts, poses, quats = _batch_case(gen)
    if spacing == "even":
        T, W = 4, 12
        xs = torch.arange(W, dtype=torch.float32) * 0.1
        poses = torch.zeros(T, W, 3)
        poses[:, :, 0] = xs + 2.0
        poses[:, :, 1] = torch.arange(T, dtype=torch.float32)[:, None] * 0.5
        poses[:, :, 2] = 0.5
        yaw = torch.from_numpy(gen.normal(0, 0.3, (T, W)).astype(np.float32))
        quats = torch.stack([torch.cos(yaw / 2), 0 * yaw, 0 * yaw, torch.sin(yaw / 2)], -1)
    K, Wd, Hd = tools.load_intrinsics(dev)
    mb = model.ModelTrajBatch(pts, poses, quats, K, Wd, Hd, device=dev)
    mb.poses.data.add_(torch.from_numpy(gen.normal(0, 0.05, tuple(poses.shape)).astype(np.float32)).to(dev))
    loss = mb(vis_wps_dist=0.5)
    loss.backward()
    if spacing == "even":
        assert mb._wps_step(0.5) == 6
    assert mb.means.shape == (len(poses),) and all(v.shape == (len(poses),) for v in mb.losses.values())
    total = 0.0
    for t in range(len(poses)):
        m = model.ModelTraj(pts, poses[t], quats[t], K, Wd, Hd, device=dev)
        m.poses.data.copy_(mb.poses.data[t])
        lt = m(vis_wps_dist=0.5)
        lt.backward()
        total += lt.item()
        for key in ("vis", "l2", "smooth", "length"):
            assert rel_err(mb.losses[key][t].item(), float(m.loss[key])) < 1e-6, key
        assert row_rel_err(mb.poses.grad[t].cpu().numpy(), m.poses.grad.cpu().numpy()) < TOL_ROW
        assert row_rel_err(mb.quats.grad[t].cpu().numpy(), m.quats.grad.cpu().numpy()) < TOL_ROW
    assert rel_err(loss.item(), total) < 1e-6


def test_model_traj_batch_graphed_steps_equal_eager(dev, mod):
    from trajectory_optimization_b200.graphs import GraphedStep
    model, tools, ops = mod
    gen = np.random.default_rng(20)
    pts, poses, quats = _batch_case(gen)
    K, Wd, Hd = tools.load_intrinsics(dev)
    finals = []
    for graphed in (False, True):
        m = model.ModelTrajBatch(pts, poses, quats, K, Wd, Hd, device=dev)
        opt = torch.optim.Adam([{"params": [m.poses], "lr": 0.02}, {"params": [m.quats], "lr": 0.01}], capturable=True)
        if graphed:
            g = GraphedStep(m, opt, warmup=1)   # one eager warm-up step, then 3 replays
            for _ in range(3):
                loss = g.step()
        else:
            for _ in range(4):
                opt.zero_grad()
                loss = m()
                loss.backward()
                opt.step()
        torch.cuda.synchronize()
        finals.append((loss.item(), m.poses.detach().clone(), m.quats.detach().clone()))
    assert rel_err(finals[1][0], finals[0][0]) < 1e-5
    assert rel_err(finals[1][1].cpu().numpy(), finals[0][1].cpu().numpy()) < 1e-5
    assert rel_err(finals[1][2].cpu().numpy(), finals[0][2].cpu().numpy()) < 1e-5


def test_model_traj_batch_rejects_differing_strides(dev, mod):
    model, tools, ops = mod
    gen = np.random.default_rng(21)
    pts, poses, quats = _batch_case(gen)
    poses[1] *= 3.0
    K, Wd, Hd = tools.load_intrinsics(dev)
    m = model.ModelTrajBatch(pts, poses, quats, K, Wd, Hd, device=dev)
    with pytest.raises(ValueError, match="strides differ"):
        m(vis_wps_dist=2.0)


def test_sweep_errors_are_loud(dev, mod):
    model, tools, ops = mod
    from trajectory_optimization_b200 import _lib
    L = _lib.lib()
    gen = np.random.default_rng(22)
    K, Wd, Hd = tools.load_intrinsics(dev)
    big = torch.from_numpy(_box(gen, 70_000)).to(dev)
    too_many = L.cov_traj_max_poses_pruned() + 1
    P = torch.zeros(1, too_many, 3, device=dev)
    Q = torch.tensor([1.0, 0, 0, 0], device=dev).repeat(1, too_many, 1)
    with pytest.raises(RuntimeError, match="cov_sweep_fused.*exceed"):
        ops.coverage_sweep(big, P, Q, K, Wd, Hd)
    dense_max = L.cov_traj_max_poses() + 1
    with ops.evaluation(dense=True), pytest.raises(RuntimeError, match="cov_sweep_fused.*exceed"):
        ops.coverage_sweep(big, P[:, :dense_max], Q[:, :dense_max], K, Wd, Hd)
    with pytest.raises(ValueError, match="coverage_sweep"):
        ops.coverage_sweep(big, torch.zeros(2, 3, 3, device=dev), torch.zeros(2, 4, 4, device=dev), K, Wd, Hd)
    # the raw C ABI: a misaligned workspace and a null accumulator are refused with the library's codes
    cam = _lib.camera(Wd, Hd, 1.0, 5.0, 1e-6)
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    n = big.shape[0]
    ws_bytes = L.cov_sweep_fused_workspace_bytes(n, 2, 3, None)
    ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device=dev)
    P2, Q2 = torch.zeros(6, 3, device=dev), torch.tensor([1.0, 0, 0, 0], device=dev).repeat(6, 1)
    mm = torch.ones(12, device=dev)
    acc = torch.empty(2 * (3 * ACC + 1), dtype=torch.float64, device=dev)
    Kd = K.reshape(9).contiguous()
    args = [big.data_ptr(), n, P2.data_ptr(), Q2.data_ptr(), 2, 3, Kd.data_ptr(), ctypes.byref(cam), None, mm.data_ptr()]
    assert L.cov_sweep_fused(*args, acc.data_ptr(), None, ws.data_ptr() + 16, ws_bytes, stream) == -5
    assert L.cov_sweep_fused(*args, None, None, ws.data_ptr(), ws_bytes, stream) == -1
    assert L.cov_sweep_fused(*args, acc.data_ptr(), None, ws.data_ptr(), ws_bytes - 1, stream) == -3
