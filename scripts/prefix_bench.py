"""Cost of the prefix sweep on the c5 workload (bench.py): 1024 trajectories x 32 poses on the Morton-ordered cloud,
boxes given, the paths alternated within one process.

    python scripts/prefix_bench.py [--points 50000000] [--repeats 5]

  sweep          ops.sweep_rewards: one mean per trajectory
  prefix         ops.sweep_prefix_rewards: the mean of every prefix of every trajectory (1024 x 32)
  prefix_prior   ... with a prior log-odds
  prefix_weight  ... with a point weight
  prefix_both    ... with both
  loop32         the same numbers without the prefix sweep: sweep_rewards of poses[:, :k] for k = 1 .. 32

The prior is the one of scripts/prior_bench.py (the folded log-odds of the c4 trajectory shifted by 3 m), the weight the
region of interest of scripts/weight_bench.py.  Every call computes its normalisers (pass A) and its prior and weight sums,
as the public ops do.  Prints one JSON line: per repetition and median, in ms (CUDA events, after a warm-up of every timed
path), the prefix/sweep ratios, the largest relative difference between the last prefix column and sweep_rewards, and
the card's name, power limit and max SM clock read in the same run.  The cloud (600 MB) is far larger than L2."""
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
from scripts.weight_bench import roi_weight  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--points", type=int, default=bench.N_POINTS_C5)
    ap.add_argument("--repeats", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("prefix_bench.py needs a CUDA device")
    from trajectory_optimization_b200 import multicam, ops, tools
    dev = torch.device("cuda:0")
    K, img_w, img_h = tools.load_intrinsics(dev)
    out = {"card": card()}
    pts = bench.make_cloud_shard(args.points, 0, 1, dev)
    spts, _ = ops.spatial_sort(pts)
    del pts
    boxes = ops.tile_boxes(spts)
    weight = roi_weight(spts)                             # in the cloud's (Morton) order
    P, Q = (x.to(dev) for x in bench.c5_trajectories())
    T, Pn = P.shape[0], P.shape[1]
    rig7 = multicam.rig_tensor(multicam.ring_rig(bench.N_CAMS), dev)
    with torch.no_grad():
        t, q = multicam.camera_poses_fused(bench.body_waypoints().to(dev) + torch.tensor([0.0, 3.0, 0.0, 0.0], device=dev),
                                           rig7)
        prior = ops.traj_logodds(spts, t, q, K, img_w, img_h, boxes=boxes)
    common = dict(boxes=boxes, presorted=True)

    def sweep():
        return ops.sweep_rewards(spts, P, Q, K, img_w, img_h, **common)

    def prefix(**kw):
        return lambda: ops.sweep_prefix_rewards(spts, P, Q, K, img_w, img_h, **common, **kw)

    def loop32():
        return [ops.sweep_rewards(spts, P[:, :k], Q[:, :k], K, img_w, img_h, **common) for k in range(1, Pn + 1)]

    paths = {"sweep": sweep, "prefix": prefix(), "prefix_prior": prefix(prior_logodds=prior),
             "prefix_weight": prefix(weight=weight), "prefix_both": prefix(prior_logodds=prior, weight=weight),
             "loop32": loop32}
    res = alternate(paths, args.repeats)
    med = {k: statistics.median(v) for k, v in res.items()}
    ratios = {f"{k}_over_sweep": med[k] / med["sweep"] for k in med if k != "sweep"}
    ratios["loop32_over_prefix"] = med["loop32"] / med["prefix"]
    s, p = sweep(), paths["prefix"]()
    last_col = float(((p[:, -1] - s).abs().max() / s.abs().max()).item())
    out.update(config=f"c5: {args.points} points, {T} x {Pn} poses", ms=res, median_ms=med, ratios=ratios,
               last_column_vs_sweep_rel=last_col)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
