"""The batched ModelPose objective (ops.coverage_pose_batch, model.ModelPoseBatch) around the C ABI, on CPU: the two new
C-ABI calls are replaced by an oracle-backed stand-in built from the single-pose ones (tests only), so that the autograd
plumbing, the (K, 8) layout, the weight's permutation and point sharding over two gloo ranks are exercised without a
GPU."""
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

from tests._standins import OracleBackend  # noqa: E402


class PoseBatchOracleBackend(OracleBackend):
    """cov_pose_batch_fused / cov_pose_batch_epilogue as their definition states them: cov_pose_fused and
    cov_pose_epilogue once per pose, K blocks of 8 sums, (K, 8) rows."""

    def pose_batch_workspace_bytes(self, pts, K):
        return 0

    def pose_batch_fused(self, pts, T, Q, Kd, cam, w, boxes=None, ws=None):
        return torch.cat([self.pose_fused(pts, T[k], Q[k], Kd, cam, w, None) for k in range(T.shape[0])])

    def pose_batch_epilogue(self, acc, Q):
        return torch.stack([self.pose_epilogue(acc[8 * k:8 * k + 8], None, Q[k]) for k in range(Q.shape[0])])


class PermutingBackend(PoseBatchOracleBackend):
    """Orders the cloud by a fixed non-trivial permutation, as the Morton sort would: sorted[j] = points[perm[j]]."""

    def order_cloud(self, pts, spatial_sort_cloud=True):
        perm = torch.from_numpy(np.random.default_rng(5).permutation(pts.shape[0]).astype(np.int32))
        return pts[perm.long()].contiguous(), perm, None


def _case(K=5):
    gen = np.random.default_rng(41)
    pts = (gen.random((700, 3)) * np.array([12, 12, 4]) + np.array([-2, -2, -1])).astype(np.float32)
    trans = (gen.random((K, 3)) * np.array([6, 6, 1])).astype(np.float32)
    quats = (gen.normal(0, 0.3, (K, 4)) + np.array([1.0, 0, 0, 0])).astype(np.float32)
    weight = gen.random(len(pts)).astype(np.float32)
    gk = np.linspace(0.5, 2.0, K).astype(np.float32)
    return pts, trans, quats, weight, gk


def _batch(pts, trans, quats, gk, weight=None, **kw):
    from oracle import coverage_oracle as orc
    from trajectory_optimization_b200 import ops
    T = torch.from_numpy(trans.copy()).requires_grad_(True)
    Q = torch.from_numpy(quats.copy()).requires_grad_(True)
    w = None if weight is None else torch.from_numpy(weight)
    totals = ops.coverage_pose_batch(torch.from_numpy(pts), T, Q, torch.from_numpy(orc.K_DEFAULT.copy()), orc.IMG_WIDTH,
                                     orc.IMG_HEIGHT, weight=w, **kw)
    (torch.from_numpy(gk) * totals).sum().backward()
    return totals.detach().numpy(), T.grad.numpy(), Q.grad.numpy()


def _per_pose(pts, trans, quats, weight=None):
    from oracle import coverage_oracle as orc
    from trajectory_optimization_b200 import ops
    out = []
    for k in range(len(trans)):
        t = torch.from_numpy(trans[k:k + 1].copy()).requires_grad_(True)
        q = torch.from_numpy(quats[k:k + 1].copy()).requires_grad_(True)
        _, total = ops.coverage_pose(torch.from_numpy(pts), t, q, torch.from_numpy(orc.K_DEFAULT.copy()), orc.IMG_WIDTH,
                                     orc.IMG_HEIGHT, weight=None if weight is None else torch.from_numpy(weight))
        total.backward()
        out.append((total.item(), t.grad.numpy()[0], q.grad.numpy()[0]))
    return out


@pytest.fixture
def oracle_backend(monkeypatch):
    from trajectory_optimization_b200 import ops
    monkeypatch.setattr(ops, "_BACKEND", PoseBatchOracleBackend())


@pytest.mark.parametrize("weighted", [False, True])
def test_batch_equals_per_pose_objective(weighted, oracle_backend):
    """totals[k] and the gradient of sum_k g_k totals_k are pose k's coverage_pose total and g_k times its gradient."""
    from tests.conftest import rel_err
    pts, trans, quats, weight, gk = _case()
    w = weight if weighted else None
    totals, gt, gq = _batch(pts, trans, quats, gk, w)
    assert totals.shape == (len(trans),) and gt.shape == trans.shape and gq.shape == quats.shape
    for k, (total, t_grad, q_grad) in enumerate(_per_pose(pts, trans, quats, w)):
        assert rel_err(totals[k], total) < 1e-6
        assert rel_err(gt[k], gk[k] * t_grad) < 1e-6 and rel_err(gq[k], gk[k] * q_grad) < 1e-6


def test_weight_is_gathered_with_the_cloud_permutation(monkeypatch):
    """The op orders the cloud itself (presorted=False): the weight, given in the caller's order, must follow its points."""
    from tests.conftest import rel_err
    from trajectory_optimization_b200 import ops
    pts, trans, quats, weight, gk = _case()
    monkeypatch.setattr(ops, "_BACKEND", PoseBatchOracleBackend())
    ref = _batch(pts, trans, quats, gk, weight, presorted=True)
    # the permutation is not a symmetry of this weight: a weight left in the caller's order would change the totals
    shuffled = _batch(pts, trans, quats, gk, weight[np.random.default_rng(5).permutation(len(pts))], presorted=True)
    assert rel_err(shuffled[0], ref[0]) > 1e-3
    monkeypatch.setattr(ops, "_BACKEND", PermutingBackend())
    got = _batch(pts, trans, quats, gk, weight)
    for a, b in zip(got, ref):
        assert rel_err(a, b) < 1e-6


def test_model_pose_batch_equals_separate_models(oracle_backend):
    """Per-candidate totals and losses, the summed loss and the gradients of K separate ModelPose models."""
    from oracle import coverage_oracle as orc
    from tests.conftest import rel_err
    from trajectory_optimization_b200 import model
    pts, trans, quats, _, _ = _case()
    K = torch.from_numpy(orc.K_DEFAULT.copy())
    cpu = torch.device("cpu")
    mb = model.ModelPoseBatch(torch.from_numpy(pts), torch.from_numpy(trans), torch.from_numpy(quats), K, orc.IMG_WIDTH,
                              orc.IMG_HEIGHT, device=cpu)
    loss = mb()
    loss.backward()
    assert mb.totals.shape == (len(trans),) and mb.losses.shape == (len(trans),)
    total = 0.0
    for k in range(len(trans)):
        m = model.ModelPose(torch.from_numpy(pts), torch.from_numpy(trans[k:k + 1]), torch.from_numpy(quats[k:k + 1]), K,
                            orc.IMG_WIDTH, orc.IMG_HEIGHT, device=cpu)
        lk = m()
        lk.backward()
        total += lk.item()
        assert rel_err(mb.losses[k].item(), lk.item()) < 1e-6
        assert rel_err(mb.trans.grad[k].numpy(), m.trans.grad[0].numpy()) < 1e-6
        assert rel_err(mb.quat.grad[k].numpy(), m.quat.grad[0].numpy()) < 1e-6
    assert rel_err(loss.item(), total) < 1e-6
    mb.detach_state()
    assert mb.totals.grad_fn is None and mb.losses.grad_fn is None


def test_batch_rejects_bad_shapes(oracle_backend):
    from oracle import coverage_oracle as orc
    from trajectory_optimization_b200 import model, ops
    pts, trans, quats, weight, _ = _case()
    K = torch.from_numpy(orc.K_DEFAULT.copy())
    T, Q = torch.from_numpy(trans), torch.from_numpy(quats)
    for bad_t, bad_q in ((T, Q[:, :3]), (T[:2], Q), (T[:0], Q[:0]), (T.reshape(-1), Q.reshape(-1)), (T[None], Q[None])):
        with pytest.raises(ValueError, match="coverage_pose_batch"):
            ops.coverage_pose_batch(torch.from_numpy(pts), bad_t, bad_q, K, orc.IMG_WIDTH, orc.IMG_HEIGHT)
    with pytest.raises(ValueError, match="weight"):
        ops.coverage_pose_batch(torch.from_numpy(pts), T, Q, K, orc.IMG_WIDTH, orc.IMG_HEIGHT,
                                weight=torch.from_numpy(weight[:-1]))
    with pytest.raises(ValueError, match="ModelPoseBatch"):
        model.ModelPoseBatch(torch.from_numpy(pts), T[:0], Q[:0], K, orc.IMG_WIDTH, orc.IMG_HEIGHT, device=torch.device("cpu"))


def test_batch_on_cpu_tensors_fails_loudly():
    """The product backend: no CPU fallback, the call raises before anything runs."""
    from oracle import coverage_oracle as orc
    from trajectory_optimization_b200 import ops
    pts, trans, quats, _, _ = _case()
    with pytest.raises(RuntimeError, match="CUDA-only"):
        ops.coverage_pose_batch(torch.from_numpy(pts), torch.from_numpy(trans), torch.from_numpy(quats),
                                torch.from_numpy(orc.K_DEFAULT.copy()), orc.IMG_WIDTH, orc.IMG_HEIGHT)


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from trajectory_optimization_b200 import ops
        ops._BACKEND = PoseBatchOracleBackend()
        pts, trans, quats, weight, gk = _case()
        n = len(pts)
        lo, hi = rank * n // world, (rank + 1) * n // world
        q.put((rank, _batch(pts[lo:hi].copy(), trans, quats, gk, weight[lo:hi].copy(), group=dist.group.WORLD)))
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


def test_two_rank_point_sharding_matches_unsharded_run(oracle_backend):
    """Each rank holds half of the cloud and of the weight; the K x 8 sums are all-reduced (SUM): every rank gets one
    unsharded call's totals and gradients."""
    from tests.conftest import rel_err
    pts, trans, quats, weight, gk = _case()
    ref = _batch(pts, trans, quats, gk, weight)
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = sorted([q.get(timeout=240) for _ in range(world)], key=lambda t: t[0])
    assert all(isinstance(r[1], tuple) for r in results), results
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for _, got in results:
        for a, b in zip(got, ref):
            assert a.shape == b.shape
            assert rel_err(a, b) < 1e-6
