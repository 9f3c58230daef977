"""Cost of a prior log-odds map (map memory) on the benchmark workloads (bench.py): each timed path with and without a
prior, alternated within one process.

    python scripts/prior_bench.py [--points-c4 100000000] [--points-c5 50000000] [--repeats 5]

  c4        one step of the c4 objective: 64 waypoints x 5 cameras (320 poses) through the rig, coverage_traj on the
            Morton-ordered cloud (reward_index, boxes and workspace kept), forward + backward
  c5_fwd    ops.sweep_rewards, 1024 trajectories x 32 poses, Morton-ordered cloud, boxes given
  c5_grad   ops.coverage_sweep forward + means.sum().backward()

The prior looks like a map after one executed path: the folded log-odds (ops.traj_logodds) of the c4 trajectory shifted
by 3 m, so most entries are exactly 0 and a few percent carry large values.  Its sum_j sigmoid(prior_j) is computed once
(as the models keep it) for c4; the sweeps compute it per call, as the public ops do.  Prints one JSON line: per
repetition and median, in ms (CUDA events, after a warm-up of every timed path), the share of non-zero prior entries,
and the card's name and power limit read in the same run.  Both clouds are far larger than L2."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or "unknown"


def timed(fn):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def alternate(paths, repeats):
    for fn in paths.values():   # warm-up: modules, occupancy queries, allocator
        fn()
    res = {k: [] for k in paths}
    for _ in range(repeats):
        for k, fn in paths.items():
            res[k].append(timed(fn))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--points-c4", type=int, default=bench.N_POINTS_C4)
    ap.add_argument("--points-c5", type=int, default=bench.N_POINTS_C5)
    ap.add_argument("--repeats", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("prior_bench.py needs a CUDA device")
    from trajectory_optimization_b200 import multicam, ops, tools
    dev = torch.device("cuda:0")
    K, img_w, img_h = tools.load_intrinsics(dev)
    rig7 = multicam.rig_tensor(multicam.ring_rig(bench.N_CAMS), dev)
    out = {"card": card()}

    # ---- c4 ----
    pts = bench.make_cloud_shard(args.points_c4, 0, 1, dev)
    spts, perm = ops.spatial_sort(pts)
    boxes = ops.tile_boxes(spts)
    n = pts.shape[0]
    ws = ops._BACKEND.traj_workspace(spts, bench.N_WAYPOINTS * bench.N_CAMS)
    body0 = bench.body_waypoints().to(dev)
    with torch.no_grad():
        t, q = multicam.camera_poses_fused(body0 + torch.tensor([0.0, 3.0, 0.0, 0.0], device=dev), rig7)
        prior = ops.traj_logodds(spts, t, q, K, img_w, img_h, reward_index=perm, boxes=boxes, workspace=ws)
    del pts
    prior_sum = ops._BACKEND.prior_sum(prior)
    out["c4_prior_nonzero_share"] = float((prior != 0).float().mean())
    cam = ops._lib.camera(img_w, img_h, 1.0, 5.0, 1e-6)
    body = body0.clone().requires_grad_(True)

    def c4(with_prior):
        def step():
            body.grad = None
            t, q = multicam.camera_poses_fused(body, rig7)
            _, mean = ops.CoverageTrajFn.apply(spts, t, q, K, cam, n, None, perm, boxes, None, ws,
                                               prior if with_prior else None, prior_sum if with_prior else None)
            (1.0 / (mean + 1e-6)).backward()
        return step

    res = alternate({"c4_no_prior": c4(False), "c4_prior": c4(True)}, args.repeats)
    del spts, perm, boxes, ws, prior
    torch.cuda.empty_cache()

    # ---- c5 ----
    pts = bench.make_cloud_shard(args.points_c5, 0, 1, dev)
    spts, perm = ops.spatial_sort(pts)
    del pts
    boxes = ops.tile_boxes(spts)
    P, Q = (x.to(dev) for x in bench.c5_trajectories())
    T, Pn = P.shape[0], P.shape[1]
    with torch.no_grad():
        t, q = multicam.camera_poses_fused(body0 + torch.tensor([0.0, 3.0, 0.0, 0.0], device=dev), rig7)
        prior5 = ops.traj_logodds(spts, t, q, K, img_w, img_h, boxes=boxes)   # in the cloud's (Morton) order
    out["c5_prior_nonzero_share"] = float((prior5 != 0).float().mean())
    sws = torch.empty(ops._BACKEND.sweep_fused_workspace_bytes(spts, T, Pn), dtype=torch.uint8, device=dev)

    def fwd(with_prior):
        return lambda: ops.sweep_rewards(spts, P, Q, K, img_w, img_h, boxes=boxes, presorted=True,
                                         prior_logodds=prior5 if with_prior else None)

    def grad(with_prior):
        def run():
            Pg, Qg = P.detach().requires_grad_(True), Q.detach().requires_grad_(True)
            means = ops.coverage_sweep(spts, Pg, Qg, K, img_w, img_h, boxes=boxes, presorted=True, workspace=sws,
                                       prior_logodds=prior5 if with_prior else None)
            means.sum().backward()
        return run

    res.update(alternate({"c5_fwd_no_prior": fwd(False), "c5_fwd_prior": fwd(True), "c5_grad_no_prior": grad(False),
                          "c5_grad_prior": grad(True)}, args.repeats))
    med = {k: statistics.median(v) for k, v in res.items()}
    out.update(config=f"c4: {args.points_c4} points, {bench.N_WAYPOINTS} x {bench.N_CAMS} poses; c5: {args.points_c5} points, "
                      f"{T} x {Pn} poses", ms=res, median_ms=med,
               prior_over_no_prior={w: med[w + "_prior"] / med[w + "_no_prior"] for w in ("c4", "c5_fwd", "c5_grad")})
    print(json.dumps(out))


if __name__ == "__main__":
    main()
