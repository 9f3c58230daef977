"""Trajectories longer than one pruned call takes, without a GPU: which calls take the long path, the long-path workspace
size, the argument errors of cov_traj_fused_long / cov_traj_logodds_long, and a two-rank gloo run of the long path with
the oracle stand-in (extended here with the long path's backend calls) against the unsharded oracle."""
import ctypes
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


class LongOracleBackend(OracleBackend):
    """The oracle stand-in with the long path's two backend calls: the oracle takes any number of poses, so the long
    path's results are those of its single call over all of them."""

    def sweep_minmax(self, pts, P, Q, Kd, cam, boxes=None, ws=None, dense=None, prefill=None, prior=None):
        return self.traj_minmax(pts, P, Q, Kd, cam)

    def traj_fused_long(self, pts, P, Q, Kd, cam, minmax, upstream, rewards, reward_index=None, boxes=None, ws=None,
                        prefilled=False, prior=None, base=None, weight=None, pose_chunk=0):
        return self.traj_fused(pts, P, Q, Kd, cam, minmax, upstream, rewards, reward_index, boxes, ws)


class RecordingBackend(LongOracleBackend):
    def __init__(self):
        self.calls = []
        self._in_long = False

    def traj_fused(self, *a, **k):
        if not self._in_long:   # the stand-in's long path is its single call
            self.calls.append("traj_fused")
        return super().traj_fused(*a, **k)

    def traj_fused_long(self, *a, **k):
        self.calls.append("traj_fused_long")
        self._in_long = True
        try:
            return super().traj_fused_long(*a, **k)
        finally:
            self._in_long = False

    def traj_logodds(self, pts, P, Q, Kd, cam, minmax, out, *a, **k):
        self.calls.append("traj_logodds")
        return out

    def traj_logodds_long(self, pts, P, Q, Kd, cam, minmax, out, *a, **k):
        self.calls.append("traj_logodds_long")
        return out


def _path(W, seed=0):
    gen = np.random.default_rng(seed)
    xs = np.linspace(0, 6, W)
    poses = np.stack([xs, 0.5 * xs, np.zeros(W)], 1).astype(np.float32)
    quats = (gen.standard_normal((W, 4)) * 0.3 + np.array([1.0, 0, 0, 0])).astype(np.float32)
    return torch.from_numpy(poses), torch.from_numpy(quats)


@pytest.mark.parametrize("W,long", [(3, False), (2048, False), (2049, True), (2300, True)])
def test_routing(W, long, monkeypatch):
    from oracle import coverage_oracle as orc
    from trajectory_optimization_b200 import ops
    B = RecordingBackend()
    monkeypatch.setattr(ops, "_BACKEND", B)
    gen = np.random.default_rng(1)
    pts = torch.from_numpy((gen.random((40, 3)) * np.array([8, 8, 2])).astype(np.float32))
    P, Q = _path(W)
    P.requires_grad_(True)
    K = torch.from_numpy(orc.K_DEFAULT.copy())
    rewards, mean = ops.coverage_traj(pts, P, Q, K, orc.IMG_WIDTH, orc.IMG_HEIGHT)
    (mean + rewards.sum()).backward()   # the g_rewards backward takes the same path
    ops.traj_logodds(pts, P.detach(), Q, K, orc.IMG_WIDTH, orc.IMG_HEIGHT)
    want = ["traj_fused_long", "traj_fused_long", "traj_logodds_long"] if long else ["traj_fused", "traj_fused",
                                                                                       "traj_logodds"]
    assert B.calls == want
    if long:   # dense mode never takes the long path (and raises above the cap on the GPU)
        B.calls.clear()
        ops.coverage_traj(pts, P.detach(), Q, K, orc.IMG_WIDTH, orc.IMG_HEIGHT, dense=True)
        assert B.calls == ["traj_fused"]


def test_workspace_size_is_pure_and_monotone():
    from trajectory_optimization_b200 import _lib
    L = _lib.lib()
    f = L.cov_traj_long_workspace_bytes
    assert f(10**6, 4096, 0) == f(10**6, 4096, 0) == f(10**6, 4096, 2048)
    for n in (1, 1500, 70_000, 10**6):
        for W in (1, 320, 2048, 2049, 6000):
            prev = None
            for c in (1, 2, 37, 333, 1000, 1024, 1025, 2048):
                b = f(n, W, c)
                assert b >= L.cov_traj_workspace_bytes(n, min(W, 2048))
                assert prev is None or b <= prev   # never grows with the chunk
                prev = b
    for c in (1, 333, 2048):
        assert all(f(n, 4097, c) <= f(n * 3 + 7, 4097, c) for n in (1, 999, 10**5, 10**6))
        assert all(f(10**5, W, c) <= f(10**5, W + d, c) for W in (1, 300, 2048, 4096) for d in (1, 77, 2048))
    # one mask row of the chunk's width per listed box per chunk, next to n floats of carried log-odds
    n = 10**6
    assert f(n, 8192, 2048) >= 4 * (n * 2 + 4 * n // 128 * 4) + 4 * n


def test_argument_errors():
    from trajectory_optimization_b200 import _lib
    L = _lib.lib()
    cam = _lib.camera(640, 480, 1.0, 5.0, 1e-6)
    fake = ctypes.c_void_p(1 << 20)   # aligned, never dereferenced: every check below fails before any device work
    n, W = 100_000, 3000
    need = L.cov_traj_long_workspace_bytes(n, W, 0)

    def fused(chunk=0, upstream=None, prior=None, base=None, weight=None, ws=fake, ws_bytes=need, opts=None, acc=fake):
        return L.cov_traj_fused_long(fake, n, fake, fake, W, fake, ctypes.byref(cam), None, fake, upstream, None, fake,
                                     acc, prior, base, weight, chunk, opts, ws, ws_bytes, None)

    assert fused(chunk=-1) == -1 and fused(chunk=2049) == -1
    assert fused(acc=None) == -1
    assert fused(base=fake) == -1                              # base without prior and weight
    assert fused(prior=fake) == -1                             # a prior needs its sum
    assert fused(weight=fake) == -1                            # a weight needs its sums
    assert fused(weight=fake, base=fake, upstream=fake) == -1  # weight and upstream are never given together
    dense = _lib.TrajOpts(1, 0, None, None)
    assert fused(opts=ctypes.byref(dense)) == -2               # no dense long path above the cap
    assert fused(ws=None) == -1
    assert fused(ws_bytes=need - 1) == -3
    assert fused(ws=ctypes.c_void_p((1 << 20) + 16)) == -5
    assert L.cov_traj_logodds_long(fake, n, fake, fake, W, fake, ctypes.byref(cam), None, fake, None, fake, 4096, None,
                                   fake, need, None) == -1
    assert b"pose_chunk" in L.cov_last_error()


def _case():
    from tests.conftest import load_golden
    g = load_golden("traj_compact")   # min > 0: the arg-min tie accumulators cross the all-reduce too
    gen = np.random.default_rng(2)
    W = 2050
    poses = np.tile(g["in_poses"], (W // 5, 1)) + gen.normal(0, 1e-2, (W, 3))
    quats = np.tile(g["in_quats"], (W // 5, 1)) + gen.normal(0, 1e-2, (W, 4))
    return g["in_points"][::3].copy(), poses.astype(np.float32), quats.astype(np.float32)


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from oracle import coverage_oracle as orc
        from trajectory_optimization_b200 import ops
        B = RecordingBackend()
        ops._BACKEND = B
        pts, poses, quats = _case()
        n = len(pts)
        lo, hi = rank * n // world, (rank + 1) * n // world
        K = torch.from_numpy(orc.K_DEFAULT.copy())
        P = torch.from_numpy(poses.copy()).requires_grad_(True)
        Q = torch.from_numpy(quats.copy()).requires_grad_(True)
        rewards, mean = ops.coverage_traj(torch.from_numpy(pts[lo:hi].copy()), P, Q, K, orc.IMG_WIDTH, orc.IMG_HEIGHT,
                                          n_total=n, group=dist.group.WORLD)
        vis = 1.0 / (mean + 1e-6)
        vis.backward()
        q.put((rank, vis.item(), P.grad.numpy(), Q.grad.numpy(), rewards.detach().numpy(), list(B.calls)))
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


def test_two_rank_long_path_matches_unsharded_oracle():
    from oracle import coverage_oracle as orc
    from tests.conftest import rel_err, row_rel_err
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = sorted([q.get(timeout=600) for _ in range(world)], key=lambda t: t[0])
    assert all(len(r) == 6 for r in results), results
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    pts, poses, quats = _case()
    K, Wi, Hi = orc.load_intrinsics()
    ref = orc.traj_objective(pts, poses, quats, K, Wi, Hi, dtype=np.float64)
    n = len(pts)
    for rank, vis, gp, gq, rew, calls in results:
        assert calls == ["traj_fused_long"]
        assert rel_err(vis, ref["vis"]) < 1e-6
        assert row_rel_err(gp, ref["g_poses"]) < 1e-5 and row_rel_err(gq, ref["g_quats"]) < 1e-5
        assert rel_err(rew, ref["rewards"][rank * n // world:(rank + 1) * n // world]) < 1e-6
    assert np.allclose(results[0][2], results[1][2]) and np.allclose(results[0][3], results[1][3])
