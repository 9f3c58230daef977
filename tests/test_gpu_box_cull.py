"""The pruned passes' box-level cull: the work list holds 128-point boxes, each with its own pose mask.

The set of (box, pose) pairs the tiles kernels evaluate must be exactly the set of the two-level rule — a pose listed
for a 1024-point tile (the tile's box passes `!(box_q2lb > cap)`, after the 8-tile group's box did) and the box's own box
passing the same test — so the work counters are checked against that rule restated in torch on the pose table and the
boxes, and every output against the dense evaluation (bit-identical rewards and normalisers)."""
import ctypes

import numpy as np
import pytest
import torch

from tests.conftest import rel_err

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def env():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from trajectory_optimization_b200 import _lib, ops, tools
    dev = torch.device("cuda:0")
    L = _lib.lib()
    K, Wd, Hd = tools.load_intrinsics(dev)
    return dict(dev=dev, L=L, lib=_lib, ops=ops, K=K, cam=_lib.camera(Wd, Hd, 1.0, 5.0, 1e-6))


def _align256(v):
    return (v + 255) & ~255


def _table_v3(ws, n, W):
    """Row 3 of pass B's pose table in the workspace: (camera position, qthr)."""
    nchunks = ((n + 1023) // 1024 + 63) // 64
    ctrl_bytes = ((16 * 4 + 2 * W * 4 + 7) & ~7) + nchunks * 8
    off = _align256(ctrl_bytes)
    return ws[off:off + W * 6 * 16].view(torch.float32).view(W, 6, 4)[:, 3]


def _q2lb(lo, hi, v3):
    """box_q2lb (cov_common.cuh) for every (box, pose): fp32 differences and maxima, the fused multiply-adds in fp64."""
    lo, hi, c = lo[:, None, :3], hi[:, None, :3], v3[None, :, :3]
    d = torch.clamp_min(torch.maximum(lo - c, c - hi), 0.0)
    dx, dy, dz = d[..., 0], d[..., 1], d[..., 2]
    t = (dy.double() * dy.double() + (dx * dx).double()).float()
    return (dz.double() * dz.double() + t.double()).float()


def _rule(boxes, n, v3):
    """What the two-level rule lists: per box the poses to evaluate, per box its tile's poses (torch, on the device)."""
    ntiles = (n + 1023) // 1024
    nb = ntiles * 8
    lo, hi = boxes[:nb, :4], boxes[:nb, 4:]  # (nb, 8): lo | hi
    ng = (ntiles + 7) // 8
    pad = ng * 8 - ntiles
    inf = torch.full((pad * 8, 4), float("inf"), device=boxes.device)
    tlo = torch.cat([lo, inf]).view(ng * 8, 8, 4).amin(1)
    thi = torch.cat([hi, -inf]).view(ng * 8, 8, 4).amax(1)
    glo, ghi = tlo.view(ng, 8, 4).amin(1), thi.view(ng, 8, 4).amax(1)
    cap = v3[None, :, 3]
    g_hit = ~(_q2lb(glo, ghi, v3) > cap)
    t_hit = ~(_q2lb(tlo[:ntiles], thi[:ntiles], v3) > cap) & g_hit.repeat_interleave(8, 0)[:ntiles]
    tile_of_box = t_hit.repeat_interleave(8, 0)
    b_hit = ~(_q2lb(lo, hi, v3) > cap) & tile_of_box
    return b_hit, tile_of_box


def _passes(e, pts, boxes, P, Q, minmax=None, dense=False):
    """Pass A (unless `minmax` is given) and pass B through the C ABI; returns the normalisers, rewards, accumulators,
    work counters and the workspace after pass B."""
    L, lib, dev = e["L"], e["lib"], e["dev"]
    n, W = pts.shape[0], P.shape[0]
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    stats = torch.zeros(8, dtype=torch.int64, device=dev)
    wsb = L.cov_traj_workspace_bytes(n, W)
    ws = torch.zeros(wsb, dtype=torch.uint8, device=dev)
    mm = torch.empty(2 * W, device=dev)
    if minmax is None:
        lib.check(L.cov_traj_minmax(pts.data_ptr(), n, P.data_ptr(), Q.data_ptr(), W, e["K"].data_ptr(),
                                    ctypes.byref(e["cam"]), boxes.data_ptr(), mm.data_ptr(),
                                    ctypes.byref(lib.traj_opts(dense=dense, stats=stats)), ws.data_ptr(), wsb, stream),
                  "cov_traj_minmax")
    else:
        mm.copy_(minmax)
    rewards = torch.empty(n, device=dev)
    acc = torch.empty(W * lib.ACC_STRIDE + 1, dtype=torch.float64, device=dev)
    lib.check(L.cov_traj_fused(pts.data_ptr(), n, P.data_ptr(), Q.data_ptr(), W, e["K"].data_ptr(), ctypes.byref(e["cam"]),
                               boxes.data_ptr(), mm.data_ptr(), None, None, rewards.data_ptr(), acc.data_ptr(),
                               ctypes.byref(lib.traj_opts(dense=dense, stats=stats)), ws.data_ptr(), wsb, stream),
              "cov_traj_fused")
    torch.cuda.synchronize()
    return mm, rewards, acc, [int(x) for x in stats.tolist()], ws


def _check(e, pts, P, Q, minmax=None):
    """Pruned against dense (every output bit of the normalisers and rewards), the counters against the rule.
    Returns (work-list length, empty boxes of listed tiles, evaluated pairs)."""
    ops = e["ops"]
    boxes = ops.tile_boxes(pts)
    n, W = pts.shape[0], P.shape[0]
    mm1, r1, a1, st, ws = _passes(e, pts, boxes, P, Q, minmax)
    mm0, r0, a0, _, _ = _passes(e, pts, boxes, P, Q, minmax, dense=True)
    assert torch.equal(mm1, mm0) and torch.equal(r1, r0)
    assert rel_err(a1[-1].item(), a0[-1].item()) < 1e-12
    assert rel_err(a1[:-1].cpu().numpy(), a0[:-1].cpu().numpy()) < 2e-6
    b_hit, tile_of_box = _rule(boxes, n, _table_v3(ws, n, W))
    head = ws[:40].cpu()
    items = int(head[:4].view(torch.int32)[0])
    pairs_all, pairs_in, empty = [int(x) for x in head[16:40].view(torch.int64)]
    box_any, tile_any = b_hit.any(1), tile_of_box.any(1)
    assert items == int(box_any.sum())
    assert st[1] == int(b_hit.sum())                       # every pair of the box masks, nothing else
    assert st[6] == pairs_all == int(tile_of_box.sum())    # (box, pose) pairs of the poses listed per tile
    inside = (torch.arange(b_hit.shape[0], device=b_hit.device) * 128 < n)[:, None]
    assert pairs_in == int((tile_of_box & inside).sum())
    assert empty == int((tile_any & ~box_any).sum())
    assert st[4] <= st[1] and st[0] == ((n + 1023) // 1024) * 8 * W
    return items, empty, st[1]


def _box_cloud(gen, n, lo=(-10, -10, -1), hi=(30, 30, 4)):
    return (gen.random((n, 3), dtype=np.float32) * (np.array(hi, np.float32) - np.array(lo, np.float32))
            + np.array(lo, np.float32)).astype(np.float32)


def _s_curve(W, L=14.0):
    xs = np.linspace(0, L, W)
    yaw = np.arctan2(0.5 + 0.3 * np.cos(xs), 1.0)
    poses = np.stack([xs - 5, 0.5 * xs + 0.3 * np.sin(xs) - 8, np.zeros(W)], 1).astype(np.float32)
    quats = np.stack([np.cos(yaw / 2), 0 * yaw, 0 * yaw, np.sin(yaw / 2)], 1).astype(np.float32)
    return poses, quats


def _sorted(e, pts_np):
    pts, _ = e["ops"].spatial_sort(torch.from_numpy(pts_np).to(e["dev"]))
    return pts


@pytest.mark.parametrize("kind,n,W", [("uniform", 1_000_000, 40), ("clustered", 700_001, 45), ("ragged", 300_037, 33),
                                      ("uniform", 262_144, 70)])
def test_box_lists_follow_the_two_level_rule(kind, n, W, env):
    """Seeded clouds (a uniform box, Gaussian clusters, a size that is not a multiple of 128) and pose counts that are
    not multiples of 32: the counters equal the rule's, and the outputs the dense evaluation's."""
    gen = np.random.default_rng(n + W)
    if kind == "clustered":
        centres = _box_cloud(gen, 40)
        pts_np = (centres[gen.integers(0, 40, n)] + gen.normal(0, 0.6, (n, 3))).astype(np.float32)
    else:
        pts_np = _box_cloud(gen, n)
    poses, quats = _s_curve(W)
    quats = quats + gen.normal(0, 0.1, quats.shape).astype(np.float32)
    P, Q = torch.from_numpy(poses).to(env["dev"]), torch.from_numpy(quats).to(env["dev"])
    items, empty, evaluated = _check(env, _sorted(env, pts_np), P, Q)
    assert 0 < items < ((n + 1023) // 1024) * 8 and evaluated > 0


def test_ball_touching_one_box_lists_that_box_alone(env):
    """One pose whose cap ball reaches exactly one 128-point box of a tile: the tile is listed, that box alone is a
    work item, the tile's 7 other boxes are counted as empty."""
    dev, gen = env["dev"], np.random.default_rng(7)
    n = 65_536
    P = torch.tensor([[0.0, 0.0, 0.0]], device=dev)
    Q = torch.tensor([[1.0, 0.0, 0.0, 0.0]], device=dev)
    # normalisers fixed by the caller (min 0, max 0.8): the cap ball depends on them and the pose only
    mm = torch.tensor([0.0, 0.8], device=dev)
    probe = torch.from_numpy(_box_cloud(gen, n, (50, 50, 50), (60, 60, 60))).to(dev)
    _, _, _, _, ws = _passes(env, probe, env["ops"].tile_boxes(probe), P, Q, minmax=mm)
    v3 = _table_v3(ws, n, 1)[0].cpu().numpy()  # the ball: centre v3.xyz, squared radius qthr = v3.w
    R = float(np.sqrt(v3[3]))
    assert np.isfinite(R) and R > 0
    # tile 0: box 0 just inside the ball (nearest point at 0.98 R), boxes 1..7 just outside (1.02 R and beyond) in
    # other directions, so the tile's box contains the centre; every other tile far away
    pts = np.empty((n, 3), np.float32)
    dirs = np.array([[1, 0, 0], [-1, 0, 0], [0, 1, 0], [0, -1, 0], [0, 0, 1], [0, 0, -1], [1, 1, 0], [-1, -1, 0]], np.float32)
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    for b in range(8):
        r = (0.98 if b == 0 else 1.02) * R + gen.random(128).astype(np.float32) * 0.3 * R
        pts[b * 128:(b + 1) * 128] = dirs[b] * r[:, None]
    pts[1024:] = _box_cloud(gen, n - 1024, (5 * R, 5 * R, 5 * R), (9 * R, 9 * R, 9 * R))
    pts += v3[:3]
    items, empty, evaluated = _check(env, torch.from_numpy(pts).to(dev), P, Q, minmax=mm)
    assert (items, empty, evaluated) == (1, 7, 1)


def test_cloud_with_no_listed_box(env):
    """Caller normalisers whose cap ball reaches no box: an empty work list, every reward 1/2, as the dense pass."""
    dev, gen = env["dev"], np.random.default_rng(11)
    n = 100_003
    P, Q = torch.from_numpy(_s_curve(5)[0]).to(dev), torch.from_numpy(_s_curve(5)[1]).to(dev)
    mm = torch.tensor([0.0] * 5 + [0.8] * 5, device=dev)
    pts = torch.from_numpy(_box_cloud(gen, n, (400, 400, 400), (500, 500, 500))).to(dev)
    _, _, _, _, ws = _passes(env, pts, env["ops"].tile_boxes(pts), P, Q, minmax=mm)
    assert float(_table_v3(ws, n, 5)[:, 3].max()) < 300.0 ** 2  # the balls are far smaller than the distance
    items, empty, evaluated = _check(env, pts, P, Q, minmax=mm)
    assert (items, empty, evaluated) == (0, 0, 0)


def test_pass_a_extrema_match_dense_on_a_sorted_cloud(env):
    """Pass A's minima and maxima, pruned on box lists, against the dense pass: every bit, also for W = 100."""
    dev, gen = env["dev"], np.random.default_rng(3)
    pts = _sorted(env, _box_cloud(gen, 2_000_003))
    poses, quats = _s_curve(100, 18.0)
    P, Q = torch.from_numpy(poses).to(dev), torch.from_numpy(quats).to(dev)
    boxes = env["ops"].tile_boxes(pts)
    mm1 = _passes(env, pts, boxes, P, Q)[0]
    mm0 = _passes(env, pts, boxes, P, Q, dense=True)[0]
    assert torch.equal(mm1, mm0)
    assert float((mm1[100:] > 0).float().mean()) > 0.5
