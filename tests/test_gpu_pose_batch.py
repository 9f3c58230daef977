"""The batched ModelPose objective on the GPU: ops.coverage_pose_batch against coverage_pose per pose and against the
reference fixtures, cov_pose_batch_epilogue against cov_pose_epilogue, the pruned path against the dense one, shard
additivity of the accumulators, and ModelPoseBatch against K separate ModelPose models (eager and CUDA-graphed)."""
import ctypes

import numpy as np
import pytest
import torch

from tests.conftest import load_golden, rel_err, row_rel_err

pytestmark = pytest.mark.gpu
TOL_ROW = 2e-4   # per-pose gradient rows, each against its own magnitude (as test_gpu_coverage.py)
POSE_CASES = ["pose_sample", "pose_synth0", "pose_synth1", "pose_synth2", "pose_synth_clip"]


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


def _poses(gen, K, lo=(-5, -5, -0.5), hi=(25, 25, 1.5)):
    lo, hi = np.array(lo, np.float32), np.array(hi, np.float32)
    trans = (gen.random((K, 3), dtype=np.float32) * (hi - lo) + lo).astype(np.float32)
    yaw = gen.uniform(-np.pi, np.pi, K)
    quats = np.stack([np.cos(yaw / 2), 0 * yaw, 0 * yaw, np.sin(yaw / 2)], 1) + gen.normal(0, 0.1, (K, 4))
    return trans, quats.astype(np.float32)


def _batch_grads(ops, pts, trans, quats, K, Wd, Hd, weight=None, gk=None, **kw):
    T = trans.clone().requires_grad_(True)
    Q = quats.clone().requires_grad_(True)
    totals = ops.coverage_pose_batch(pts, T, Q, K, Wd, Hd, weight=weight, **kw)
    (totals.sum() if gk is None else (gk * totals).sum()).backward()
    return totals.detach(), T.grad, Q.grad


@pytest.mark.parametrize("n,K,weighted", [(100_003, 1, False), (100_003, 37, True), (77, 37, False), (77, 5, True),
                                          (20_001, 1500, False), (20_001, 1500, True)])
def test_batch_matches_coverage_pose_per_pose(n, K, weighted, dev, mod):
    """Every candidate's total and gradient as coverage_pose computes it for that pose alone (n not a multiple of 4 or
    128, a cloud smaller than one box, one pose, and more poses than one shared-memory chunk holds)."""
    model, tools, ops = mod
    gen = np.random.default_rng(n + K + weighted)
    pts = torch.from_numpy(_box(gen, n)).to(dev)
    trans_np, quats_np = _poses(gen, K)
    trans, quats = torch.from_numpy(trans_np).to(dev), torch.from_numpy(quats_np).to(dev)
    weight = torch.from_numpy(gen.random(n, dtype=np.float32) * 2).to(dev) if weighted else None
    Kc, Wd, Hd = tools.load_intrinsics(dev)
    gk = torch.from_numpy(gen.normal(0, 1, K).astype(np.float32)).to(dev)
    totals, gt, gq = _batch_grads(ops, pts, trans, quats, Kc, Wd, Hd, weight, gk)
    assert totals.shape == (K,) and totals.dtype == torch.float32 and gt.shape == (K, 3) and gq.shape == (K, 4)
    ref_tot, ref_t, ref_q = [], [], []
    for k in range(K):
        t = trans[k:k + 1].clone().requires_grad_(True)
        q = quats[k:k + 1].clone().requires_grad_(True)
        _, total = ops.coverage_pose(pts, t, q, Kc, Wd, Hd, weight=weight)
        (gk[k] * total).backward()
        ref_tot.append(total.item())
        ref_t.append(t.grad[0].cpu().numpy())
        ref_q.append(q.grad[0].cpu().numpy())
    ref_tot = np.array(ref_tot)
    assert np.abs(ref_tot).max() > 0
    assert row_rel_err(totals.cpu().numpy()[:, None], ref_tot[:, None]) < 1e-5
    assert row_rel_err(gt.cpu().numpy(), np.array(ref_t)) < TOL_ROW
    assert row_rel_err(gq.cpu().numpy(), np.array(ref_q)) < TOL_ROW


@pytest.mark.parametrize("name", POSE_CASES)
def test_batch_reproduces_reference_fixtures(name, dev, mod, sample_inputs):
    """The fixture's pose among perturbed candidates: its loss and gradients as the reference computed them, at the bars
    test_gpu_coverage.py sets for ModelPose; the other candidates get no gradient from its loss."""
    model, tools, ops = mod
    g = load_golden(name)
    pts = torch.from_numpy(g["in_points"] if "in_points" in g else sample_inputs["pts"]).to(dev)
    Kc, Wd, Hd = tools.load_intrinsics(dev)
    gen = np.random.default_rng(23)
    t0, q0 = g["in_trans"].astype(np.float32).reshape(1, 3), g["in_quat"].astype(np.float32).reshape(1, 4)
    Kn, k = 8, 3
    trans = np.repeat(t0, Kn, 0) + gen.normal(0, 0.3, (Kn, 3)).astype(np.float32)
    quats = np.repeat(q0, Kn, 0) + gen.normal(0, 0.05, (Kn, 4)).astype(np.float32)
    trans[k], quats[k] = t0[0], q0[0]
    T = torch.from_numpy(trans).to(dev).requires_grad_(True)
    Q = torch.from_numpy(quats).to(dev).requires_grad_(True)
    weight = torch.from_numpy(g["in_weight"]).to(dev) if "in_weight" in g else None
    totals = ops.coverage_pose_batch(pts, T, Q, Kc, Wd, Hd, float(g["in_min_d"]), float(g["in_max_d"]), weight=weight)
    loss = 1.0 / (totals[k] + 1e-6)
    loss.backward()
    for sfx in ("", "64"):
        assert rel_err(loss.item(), g["out_loss" + sfx]) < 1e-4
        assert rel_err(T.grad[k].cpu().numpy(), g["out_g_trans" + sfx].reshape(3)) < 1e-4
        assert rel_err(Q.grad[k].cpu().numpy(), g["out_g_quat" + sfx].reshape(4)) < 1e-4
    others = [i for i in range(Kn) if i != k]
    assert float(T.grad[others].abs().max()) == 0.0 and float(Q.grad[others].abs().max()) == 0.0


def test_batch_epilogue_is_bit_identical_to_pose_epilogue(dev, mod):
    model, tools, ops = mod
    gen = np.random.default_rng(8)
    K = 300
    acc = gen.normal(0, 1.0, (K, 8)) * np.array([1e3, 1, 1, 1, 10, 10, 10, 0])
    quats = gen.normal(0, 1, (K, 4)).astype(np.float32)
    quats[0] = 0.0   # |q~| below the 1e-12 floor
    acc_d = torch.from_numpy(acc.reshape(-1)).to(dev)
    Q = torch.from_numpy(quats).to(dev)
    out = ops._BACKEND.pose_batch_epilogue(acc_d, Q).cpu()
    assert out.shape == (K, 8)
    for k in range(K):
        ref = ops._BACKEND.pose_epilogue(acc_d[8 * k:8 * k + 8], None, Q[k]).cpu()
        assert torch.equal(out[k], ref), k


def test_pruned_equals_dense_on_a_large_map(dev, mod):
    """A 400 x 400 m map: the warps skip most (box, pose) pairs, and the sums equal the dense evaluation up to the order
    of the fp64 additions; a pose whose whole support lies outside the cloud has total exactly 0 on both paths."""
    model, tools, ops = mod
    gen = np.random.default_rng(31)
    pts, _ = ops.spatial_sort(torch.from_numpy(_box(gen, 2_000_003, (0, 0, 0), (400, 400, 5))).to(dev))
    boxes = ops.tile_boxes(pts)
    trans_np, quats_np = _poses(gen, 24, (10, 10, 0.5), (390, 390, 2))
    trans_np[-1] = (2000.0, 2000.0, 1.0)   # hundreds of metres from every point
    trans, quats = torch.from_numpy(trans_np).to(dev), torch.from_numpy(quats_np).to(dev)
    Kc, Wd, Hd = tools.load_intrinsics(dev)
    from trajectory_optimization_b200 import _lib
    cam = _lib.camera(Wd, Hd, 1.0, 5.0, 1e-6)
    Kd = Kc.reshape(9).contiguous()
    B = ops._BACKEND
    stats = torch.zeros(8, dtype=torch.int64, device=dev)
    with ops.evaluation(stats=stats):
        acc_p = B.pose_batch_fused(pts, trans, quats, Kd, cam, None, boxes).cpu().numpy().reshape(-1, 8)
    s = stats.cpu().numpy()
    assert s[0] == 24 * ((pts.shape[0] + 127) // 128) and 0 < s[1] < s[0] // 10   # more than 90 % skipped
    with ops.evaluation(dense=True):
        acc_d = B.pose_batch_fused(pts, trans, quats, Kd, cam, None, boxes).cpu().numpy().reshape(-1, 8)
    assert row_rel_err(acc_p[:-1, :7], acc_d[:-1, :7]) < 1e-9
    assert np.all(acc_p[:, 7] == 0) and np.all(acc_d[:, 7] == 0)
    assert np.all(acc_p[-1] == 0) and np.all(acc_d[-1] == 0)
    tp, gtp, gqp = _batch_grads(ops, pts, trans, quats, Kc, Wd, Hd, boxes=boxes, presorted=True)
    with ops.evaluation(dense=True):
        td, gtd, gqd = _batch_grads(ops, pts, trans, quats, Kc, Wd, Hd, boxes=boxes, presorted=True)
    assert rel_err(tp.cpu().numpy(), td.cpu().numpy()) < 1e-6
    assert row_rel_err(gtp.cpu().numpy(), gtd.cpu().numpy()) < 1e-6
    assert row_rel_err(gqp.cpu().numpy(), gqd.cpu().numpy()) < 1e-6
    assert tp[-1].item() == 0.0 and td[-1].item() == 0.0


def test_shard_blocks_add_up_to_the_whole_cloud(dev, mod):
    """Raw C ABI: the sums of two halves of a cloud (split on a box boundary) add up to the whole cloud's."""
    model, tools, ops = mod
    gen = np.random.default_rng(33)
    pts, _ = ops.spatial_sort(torch.from_numpy(_box(gen, 300_001)).to(dev))
    weight = torch.from_numpy(gen.random(pts.shape[0], dtype=np.float32)).to(dev)
    trans_np, quats_np = _poses(gen, 70)
    trans, quats = torch.from_numpy(trans_np).to(dev), torch.from_numpy(quats_np).to(dev)
    Kc, Wd, Hd = tools.load_intrinsics(dev)
    from trajectory_optimization_b200 import _lib
    cam = _lib.camera(Wd, Hd, 1.0, 5.0, 1e-6)
    Kd = Kc.reshape(9).contiguous()
    B = ops._BACKEND
    h = 128 * 1000
    parts = [(pts[:h], weight[:h]), (pts[h:], weight[h:])]
    acc = [B.pose_batch_fused(p, trans, quats, Kd, cam, w, ops.tile_boxes(p)) for p, w in parts]
    whole = B.pose_batch_fused(pts, trans, quats, Kd, cam, weight, ops.tile_boxes(pts))
    summed = (acc[0] + acc[1]).cpu().numpy().reshape(-1, 8)
    assert row_rel_err(summed, whole.cpu().numpy().reshape(-1, 8)) < 1e-12


def _model_case(gen, K=6, n=60_000):
    pts = torch.from_numpy(_box(gen, n, (-5, -5, -1), (15, 15, 3)))
    trans, quats = _poses(gen, K, (-2, -2, 0), (12, 12, 1))
    return pts, torch.from_numpy(trans), torch.from_numpy(quats)


@pytest.mark.parametrize("hpr", [False, True])
def test_model_pose_batch_equals_separate_models(hpr, dev, mod):
    model, tools, ops = mod
    gen = np.random.default_rng(37)
    pts, trans, quats = _model_case(gen, n=20_000 if hpr else 60_000)
    Kc, Wd, Hd = tools.load_intrinsics(dev)
    mb = model.ModelPoseBatch(pts, trans, quats, Kc, Wd, Hd, device=dev)
    loss = mb(hpr=hpr)
    loss.backward()
    assert mb.totals.shape == (len(trans),) and mb.losses.shape == (len(trans),)
    total = 0.0
    for k in range(len(trans)):
        m = model.ModelPose(pts, trans[k:k + 1], quats[k:k + 1], Kc, Wd, Hd, device=dev)
        lk = m(hpr=hpr)
        lk.backward()
        total += lk.item()
        assert rel_err(mb.losses[k].item(), lk.item()) < 1e-5
        assert row_rel_err(mb.trans.grad[k:k + 1].cpu().numpy(), m.trans.grad.cpu().numpy()) < TOL_ROW
        assert row_rel_err(mb.quat.grad[k:k + 1].cpu().numpy(), m.quat.grad.cpu().numpy()) < TOL_ROW
    assert rel_err(loss.item(), total) < 1e-5


def test_model_pose_batch_graphed_steps_equal_eager(dev, mod):
    from trajectory_optimization_b200.graphs import GraphedStep
    model, tools, ops = mod
    gen = np.random.default_rng(39)
    pts, trans, quats = _model_case(gen, K=256)
    Kc, Wd, Hd = tools.load_intrinsics(dev)
    finals = []
    for graphed in (False, True):
        m = model.ModelPoseBatch(pts, trans, quats, Kc, Wd, Hd, device=dev)
        opt = torch.optim.Adam([{"params": [m.trans], "lr": 0.02}, {"params": [m.quat], "lr": 0.01}], capturable=True)
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
        finals.append((loss.item(), m.trans.detach().clone(), m.quat.detach().clone()))
    assert rel_err(finals[1][0], finals[0][0]) < 1e-5
    assert rel_err(finals[1][1].cpu().numpy(), finals[0][1].cpu().numpy()) < 1e-5
    assert rel_err(finals[1][2].cpu().numpy(), finals[0][2].cpu().numpy()) < 1e-5


def test_batch_errors_are_loud(dev, mod):
    model, tools, ops = mod
    from trajectory_optimization_b200 import _lib
    L = _lib.lib()
    gen = np.random.default_rng(41)
    Kc, Wd, Hd = tools.load_intrinsics(dev)
    pts = torch.from_numpy(_box(gen, 10_000)).to(dev)
    trans_np, quats_np = _poses(gen, 3)
    trans, quats = torch.from_numpy(trans_np).to(dev), torch.from_numpy(quats_np).to(dev)
    with pytest.raises(RuntimeError, match="CUDA-only"):
        ops.coverage_pose_batch(pts.cpu(), trans, quats, Kc, Wd, Hd)
    with pytest.raises(ValueError, match="coverage_pose_batch"):
        ops.coverage_pose_batch(pts, trans[:0], quats[:0], Kc, Wd, Hd)
    with pytest.raises(ValueError, match="ModelPoseBatch"):
        model.ModelPoseBatch(pts, trans[:0], quats[:0], Kc, Wd, Hd, device=dev)
    # the raw C ABI: its codes for no poses, null pointers, misaligned pointers and a short workspace
    cam = _lib.camera(Wd, Hd, 1.0, 5.0, 1e-6)
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    n = pts.shape[0]
    ws_bytes = L.cov_pose_batch_workspace_bytes(n, 3, None)
    ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device=dev)
    acc = torch.empty(3 * 8, dtype=torch.float64, device=dev)
    w = torch.ones(n + 4, device=dev)
    Kd = Kc.reshape(9).contiguous()
    tq = [trans.data_ptr(), quats.data_ptr()]

    def call(xyz=pts.data_ptr(), wp=None, K=3, acc_p=acc.data_ptr(), ws_p=ws.data_ptr(), nbytes=ws_bytes):
        return L.cov_pose_batch_fused(xyz, n, wp, *tq, K, Kd.data_ptr(), ctypes.byref(cam), None, acc_p, None, ws_p, nbytes,
                                      stream)

    assert call() == 0
    assert call(K=0) == -1 and call(acc_p=None) == -1 and call(ws_p=None) == -1
    assert call(xyz=pts.data_ptr() + 4) == -5 and call(wp=w.data_ptr() + 4) == -5 and call(ws_p=ws.data_ptr() + 8) == -5
    assert call(nbytes=ws_bytes - 1) == -3
    out = torch.empty(3, 8, device=dev)
    assert L.cov_pose_batch_epilogue(acc.data_ptr(), quats.data_ptr(), 0, out.data_ptr(), stream) == -1
    assert L.cov_pose_batch_epilogue(None, quats.data_ptr(), 3, out.data_ptr(), stream) == -1
    torch.cuda.synchronize()
