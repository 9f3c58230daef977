"""Cost of per-point weights on the benchmark workloads (bench.py): each timed path unweighted and weighted, with and
without a prior, alternated within one process.

    python scripts/weight_bench.py [--points-c4 100000000] [--points-c5 50000000] [--repeats 5]

  c4        one step of the c4 objective: 64 waypoints x 5 cameras (320 poses) through the rig, coverage_traj on the
            Morton-ordered cloud (reward_index, boxes and workspace kept), forward + backward, three ways:
              plain     the unweighted mean
              weighted  the weighted mean of coverage_traj(weight=) (sums kept, as the models keep them)
              torch     (w * rewards).sum() / w.sum() composed in torch: its backward runs a second pass B
  c5_fwd    ops.sweep_rewards, 1024 trajectories x 32 poses, Morton-ordered cloud, boxes given
  c5_grad   ops.coverage_sweep forward + means.sum().backward()

The weight is a region of interest with a soft edge: 1 inside a 40 m x 20 m box about the c4 path, 0.2 outside.  The
prior is the one of scripts/prior_bench.py (the folded log-odds of the c4 trajectory shifted by 3 m).  The sweeps compute
their weight sums per call, as the public ops do.  Prints one JSON line: per repetition and median, in ms (CUDA events,
after a warm-up of every timed path), and the card's name and power limit read in the same run.  Both clouds are far
larger than L2."""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402
from scripts.prior_bench import alternate, card  # noqa: E402


def roi_weight(pts):
    x, y = pts[:, 0], pts[:, 1]
    inside = (x > -5) & (x < 35) & (y > -10) & (y < 10)
    return torch.where(inside, 1.0, 0.2).float().contiguous()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--points-c4", type=int, default=bench.N_POINTS_C4)
    ap.add_argument("--points-c5", type=int, default=bench.N_POINTS_C5)
    ap.add_argument("--repeats", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("weight_bench.py needs a CUDA device")
    from trajectory_optimization_b200 import multicam, ops, tools
    dev = torch.device("cuda:0")
    K, img_w, img_h = tools.load_intrinsics(dev)
    rig7 = multicam.rig_tensor(multicam.ring_rig(bench.N_CAMS), dev)
    out = {"card": card()}

    # ---- c4 ----
    pts = bench.make_cloud_shard(args.points_c4, 0, 1, dev)
    w = roi_weight(pts)                                   # in the caller's order, like the rewards
    spts, perm = ops.spatial_sort(pts)
    boxes = ops.tile_boxes(spts)
    n = pts.shape[0]
    ws = ops._BACKEND.traj_workspace(spts, bench.N_WAYPOINTS * bench.N_CAMS)
    body0 = bench.body_waypoints().to(dev)
    with torch.no_grad():
        t, q = multicam.camera_poses_fused(body0 + torch.tensor([0.0, 3.0, 0.0, 0.0], device=dev), rig7)
        prior = ops.traj_logodds(spts, t, q, K, img_w, img_h, reward_index=perm, boxes=boxes, workspace=ws)
    del pts
    B = ops._BACKEND
    prior_sum = B.prior_sum(prior)
    sums = {False: B.weight_sums(w), True: B.weight_sums(w, prior)}
    w64 = w.double()
    wtot = w64.sum()
    cam = ops._lib.camera(img_w, img_h, 1.0, 5.0, 1e-6)
    body = body0.clone().requires_grad_(True)

    def c4(mode, with_prior):
        pr, ps = (prior, prior_sum) if with_prior else (None, None)

        def step():
            body.grad = None
            t, q = multicam.camera_poses_fused(body, rig7)
            if mode == "weighted":
                s = sums[with_prior]
                _, mean = ops.CoverageTrajFn.apply(spts, t, q, K, cam, n, None, perm, boxes, None, ws, pr, ps, w, s, s[1:])
            else:
                rewards, mean = ops.CoverageTrajFn.apply(spts, t, q, K, cam, n, None, perm, boxes, None, ws, pr, ps)
                if mode == "torch":
                    mean = (w64 * rewards.double()).sum() / wtot
            (1.0 / (mean + 1e-6)).backward()
        return step

    paths = {}
    for with_prior in (False, True):
        sfx = "_prior" if with_prior else ""
        for mode in ("plain", "weighted", "torch"):
            paths[f"c4_{mode}{sfx}"] = c4(mode, with_prior)
    res = alternate(paths, args.repeats)
    del spts, perm, boxes, ws, prior, w, w64
    torch.cuda.empty_cache()

    # ---- c5 ----
    pts = bench.make_cloud_shard(args.points_c5, 0, 1, dev)
    spts, perm = ops.spatial_sort(pts)
    del pts
    boxes = ops.tile_boxes(spts)
    w5 = roi_weight(spts)                                 # in the cloud's (Morton) order
    P, Q = (x.to(dev) for x in bench.c5_trajectories())
    T, Pn = P.shape[0], P.shape[1]
    with torch.no_grad():
        t, q = multicam.camera_poses_fused(body0 + torch.tensor([0.0, 3.0, 0.0, 0.0], device=dev), rig7)
        prior5 = ops.traj_logodds(spts, t, q, K, img_w, img_h, boxes=boxes)
    sws = torch.empty(B.sweep_fused_workspace_bytes(spts, T, Pn), dtype=torch.uint8, device=dev)

    def fwd(weighted, with_prior):
        return lambda: ops.sweep_rewards(spts, P, Q, K, img_w, img_h, boxes=boxes, presorted=True,
                                         prior_logodds=prior5 if with_prior else None, weight=w5 if weighted else None)

    def grad(weighted, with_prior):
        def run():
            Pg, Qg = P.detach().requires_grad_(True), Q.detach().requires_grad_(True)
            means = ops.coverage_sweep(spts, Pg, Qg, K, img_w, img_h, boxes=boxes, presorted=True, workspace=sws,
                                       prior_logodds=prior5 if with_prior else None, weight=w5 if weighted else None)
            means.sum().backward()
        return run

    paths = {}
    for with_prior in (False, True):
        sfx = "_prior" if with_prior else ""
        for weighted in (False, True):
            tag = "weighted" if weighted else "plain"
            paths[f"c5_fwd_{tag}{sfx}"] = fwd(weighted, with_prior)
            paths[f"c5_grad_{tag}{sfx}"] = grad(weighted, with_prior)
    res.update(alternate(paths, args.repeats))
    med = {k: statistics.median(v) for k, v in res.items()}
    ratios = {}
    for sfx in ("", "_prior"):
        ratios[f"c4_weighted_over_plain{sfx}"] = med[f"c4_weighted{sfx}"] / med[f"c4_plain{sfx}"]
        ratios[f"c4_torch_over_weighted{sfx}"] = med[f"c4_torch{sfx}"] / med[f"c4_weighted{sfx}"]
        for w in ("c5_fwd", "c5_grad"):
            ratios[f"{w}_weighted_over_plain{sfx}"] = med[f"{w}_weighted{sfx}"] / med[f"{w}_plain{sfx}"]
    out.update(config=f"c4: {args.points_c4} points, {bench.N_WAYPOINTS} x {bench.N_CAMS} poses; c5: {args.points_c5} points, "
                      f"{T} x {Pn} poses", ms=res, median_ms=med, ratios=ratios)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
