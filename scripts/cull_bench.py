#!/usr/bin/env python
"""A/B measurement of the pruned pipeline's cull and tiles kernels between builds of the library, in one process.

Runs pass A (cov_traj_minmax, pre-filling the rewards) and pass B (cov_traj_fused) of the bench.py c4 workload
(Morton-ordered cloud, 64 waypoints x 5 cameras) with each library in turn, alternating the libraries within every
repetition, and writes JSON lines to <out>/cull_bench.jsonl:
  {"kind": "device"}     name, power limit and max SM clock of the card (nvidia-smi), read in the same run
  {"kind": "counters"}   per library: the 8 work counters of one pass A + one pass B, the work-list length of each
                         pass and the number of boxes of listed tiles that no pose reaches (control words of the
                         workspace; 0 for a build whose cull does not count them)
  {"kind": "parity"}     rewards and normalisers of each library against the first one (bit equality), the reward
                         sum and the pose accumulators as relative differences (fp64 addition order)
  {"kind": "rep"}        per repetition and library: CUDA-event times of pass A and pass B (mean over `--calls`
                         calls), and per-kernel device times from torch.profiler (mean per launch)
  {"kind": "summary"}    per library: median, min and max over the repetitions

usage: cull_bench.py [--lib NAME=PATH ...] [--points N] [--reps R] [--calls C] [--out DIR]
(default library: the in-tree build, or COV_B200_LIB)."""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from trajectory_optimization_b200 import _lib, multicam, ops, tools  # noqa: E402

KERNELS = ("cov_cull_kernel", "cov_traj_minmax_tiles_kernel", "cov_traj_fused_tiles_kernel", "cov_traj_prepare_kernel",
           "cov_traj_table_kernel")


def load(path):
    handle = ctypes.CDLL(path)
    for name in ("cov_traj_workspace_bytes", "cov_traj_minmax", "cov_traj_fused", "cov_last_error"):
        res, args = _lib.PROTOTYPES[name]
        fn = getattr(handle, name)
        fn.restype, fn.argtypes = res, args
    return handle


def device_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
    except Exception as e:  # noqa: BLE001 - reported, not fatal
        name, power, clock = torch.cuda.get_device_name(0), "unknown (%s)" % e, "unknown"
    return {"kind": "device", "name": name, "power_limit": power, "max_sm_clock": clock}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", default=[], help="NAME=PATH of a build of libcovb200.so")
    ap.add_argument("--points", type=int, default=bench.N_POINTS_C4)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--out", default="cull_bench_out")
    args = ap.parse_args()
    libs = [tuple(s.split("=", 1)) for s in args.lib] or [("tree", _lib.LIB_PATH)]
    os.makedirs(args.out, exist_ok=True)
    sink = open(os.path.join(args.out, "cull_bench.jsonl"), "w")

    def emit(rec):
        line = json.dumps(rec)
        print(line, flush=True)
        sink.write(line + "\n")
        sink.flush()

    dev = torch.device("cuda:0")
    emit(device_info())
    n = args.points
    pts, perm = ops.spatial_sort(bench.make_cloud_shard(n, 0, 1, dev))
    boxes = ops.tile_boxes(pts)
    K, iw, ih = tools.load_intrinsics(dev)
    t, q = multicam.camera_poses_fused(bench.body_waypoints().to(dev), multicam.rig_tensor(multicam.ring_rig(bench.N_CAMS), dev))
    P, Q = t.reshape(-1, 3).contiguous(), q.reshape(-1, 4).contiguous()
    W = P.shape[0]
    cam = _lib.camera(iw, ih, 1.0, 5.0, 1e-6)
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    stats = torch.zeros(8, dtype=torch.int64, device=dev)

    handles = {name: load(path) for name, path in libs}
    state = {}
    for name, L in handles.items():
        wsb = L.cov_traj_workspace_bytes(n, W)
        state[name] = dict(ws=torch.empty(wsb, dtype=torch.uint8, device=dev), wsb=wsb,
                           minmax=torch.empty(2 * W, device=dev), rewards=torch.empty(n, device=dev),
                           acc=torch.empty(W * _lib.ACC_STRIDE + 1, dtype=torch.float64, device=dev))

    def check(L, rc, what):
        if rc != 0:
            raise RuntimeError("%s failed (%d): %s" % (what, rc, L.cov_last_error().decode()))

    def pass_a(name, with_stats=False):
        L, s = handles[name], state[name]
        o = _lib.traj_opts(prefill=s["rewards"], stats=stats if with_stats else None)
        check(L, L.cov_traj_minmax(pts.data_ptr(), n, P.data_ptr(), Q.data_ptr(), W, K.data_ptr(), ctypes.byref(cam),
                                   boxes.data_ptr(), s["minmax"].data_ptr(), ctypes.byref(o), s["ws"].data_ptr(), s["wsb"],
                                   stream), "cov_traj_minmax")

    def pass_b(name, with_stats=False):
        L, s = handles[name], state[name]
        o = _lib.traj_opts(rewards_prefilled=True, stats=stats if with_stats else None)
        check(L, L.cov_traj_fused(pts.data_ptr(), n, P.data_ptr(), Q.data_ptr(), W, K.data_ptr(), ctypes.byref(cam),
                                  boxes.data_ptr(), s["minmax"].data_ptr(), None, perm.data_ptr(), s["rewards"].data_ptr(),
                                  s["acc"].data_ptr(), ctypes.byref(o), s["ws"].data_ptr(), s["wsb"], stream),
              "cov_traj_fused")

    def ctrl_words(name):  # ctrl[0] list length, ctrl[8..9] boxes of listed tiles that no pose reaches
        head = state[name]["ws"][:40].clone().cpu()
        return int(head[:4].view(torch.int32)[0]), int(head[32:40].view(torch.int64)[0])

    # counters and outputs of one pass A + one pass B per library
    outs = {}
    for name in handles:
        pass_a(name)
        pass_b(name)  # warm-up
        stats.zero_()
        pass_a(name, True)
        torch.cuda.synchronize()
        items_a, empty_a = ctrl_words(name)
        pass_b(name, True)
        torch.cuda.synchronize()
        items_b, empty_b = ctrl_words(name)
        s = state[name]
        outs[name] = (s["minmax"].clone(), s["rewards"].clone(), s["acc"].clone())
        emit({"kind": "counters", "lib": name, "stats": [int(x) for x in stats.tolist()], "items_a": items_a,
              "items_b": items_b, "empty_items_a": empty_a, "empty_items_b": empty_b})
    ref = next(iter(handles))
    for name in handles:
        mm0, r0, a0 = outs[ref]
        mm1, r1, a1 = outs[name]
        rows0, rows1 = a0[:-1], a1[:-1]
        emit({"kind": "parity", "lib": name, "against": ref, "minmax_equal": bool(torch.equal(mm0, mm1)),
              "rewards_equal": bool(torch.equal(r0, r1)), "reward_sum_rel_diff": abs(a1[-1].item() - a0[-1].item()) / abs(a0[-1].item()),
              "acc_rows_max_rel_diff": float(((rows1 - rows0).abs().max() / rows0.abs().max().clamp_min(1e-300)).item())})

    def events(fn, calls):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(calls):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e3 / calls  # us per call

    def kernel_times(name, calls):
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(calls):
                pass_a(name)
                pass_b(name)
            torch.cuda.synchronize()
        per = {}
        for ev in prof.events():
            if ev.device_type != torch.autograd.DeviceType.CUDA:
                continue
            key = next((k for k in KERNELS if k in ev.name), None)
            if key is not None:
                per.setdefault(key, []).append(ev.time_range.elapsed_us())
        out = {}
        for k, v in per.items():
            if k == "cov_cull_kernel":  # in launch order: pass A's, then pass B's
                out["cull_a_us"] = sum(v[0::2]) / len(v[0::2])
                out["cull_b_us"] = sum(v[1::2]) / len(v[1::2])
            else:
                out[k + "_us"] = sum(v) / len(v)
        return out

    reps = {name: [] for name in handles}
    for r in range(args.reps):
        order = list(handles) if r % 2 == 0 else list(reversed(list(handles)))
        for name in order:
            pass_a(name)
            pass_b(name)
            rec = {"pass_a_us": events(lambda: pass_a(name), args.calls), "pass_b_us": events(lambda: pass_b(name), args.calls)}
            rec.update(kernel_times(name, max(5, args.calls // 4)))
            reps[name].append(rec)
            emit(dict({"kind": "rep", "rep": r, "lib": name}, **rec))
    for name, rows in reps.items():
        summ = {}
        for key in rows[0]:
            vals = [row[key] for row in rows if key in row]
            summ[key] = {"median": statistics.median(vals), "min": min(vals), "max": max(vals)}
        emit({"kind": "summary", "lib": name, "reps": len(rows), "times": summ})
    sink.close()


if __name__ == "__main__":
    main()
