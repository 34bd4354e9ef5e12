#!/usr/bin/env python
"""Multi-scale ball query: the grid kernel (spsk_ball_query_msg_grid, build + query launches) against the brute-force scan
(spsk_ball_query_msg), at op level and inside IASSD_Backbone(waymo_iassd_cfg()).

    python scripts/bench_ball_query.py [--out FILE.json] [--rounds 3] [--calls 20] [--steps 5]

Op level: B = 8 Waymo-shaped scenes (scenes.py) of N points, M = N/4 and N/16 centres picked by D-FPS, and the radius /
nsample pairs of IA-SSD's layers 0/1/2.  CUDA events around `--calls` back-to-back calls; the two arms alternate within each
of `--rounds` rounds after a warm-up, and the median round is reported.  Every call reads the same inputs, which stay
resident in the 126 MB L2 (at most 8 x 262144 x 12 B = 25 MB of points), as they are when the SA layer runs the query
right after sampling.  The lists of both arms are compared bit for bit first.  The grid's two launches are timed apart in
a separate torch.profiler pass.

Backbone level: eager forward of IASSD_Backbone(waymo_iassd_cfg()) on 4 scenes of 131072 and of 262144 points, with the
automatic choice (grid) and with the brute-force kernel forced, alternating; the profiler pass reports the share of the
forward's kernel time spent in D-FPS and in the ball query.  The GPU name and power limit are read in the same run."""
import argparse
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from spsnet_b200 import backbone as bb  # noqa: E402
from spsnet_b200 import pointnet2_utils as pu  # noqa: E402
from spsnet_b200 import scenes  # noqa: E402

LAYERS = [([0.2, 0.8], [16, 32]), ([0.8, 1.6], [16, 32]), ([1.6, 4.8], [16, 32])]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[0] if q.returncode == 0 else None}


def time_calls(fn, calls):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(calls):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / calls


def kernel_us(fn, calls, names):
    """Mean device time per call of the kernels whose name contains one of `names`, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    out = {k: 0.0 for k in names}
    total = 0.0
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        total += t
        for k in names:
            if k in e.key:
                out[k] += t
    return {k: v / calls for k, v in out.items()}, total / calls


def op_level(a, rows):
    for n in (16384, 65536, 131072, 262144):
        B = 8
        xyz = torch.from_numpy(np.ascontiguousarray(scenes.make_batch(100, B, n, "waymo")[:, :, :3])).cuda()
        for m in (n // 4, n // 16):
            new_xyz = pu.gather_rows(xyz, pu.furthest_point_sample(xyz, m)).contiguous()
            for li, (radii, ns) in enumerate(LAYERS):
                grid = lambda: pu.ball_query_msg(radii, ns, xyz, new_xyz, grid=True)  # noqa: E731
                brute = lambda: pu.ball_query_msg(radii, ns, xyz, new_xyz, grid=False)  # noqa: E731
                for g, f in zip(grid(), brute()):
                    assert torch.equal(g, f), f"grid != brute force at N={n} M={m} layer {li}"
                for fn in (grid, brute):
                    time_calls(fn, 2)
                tg, tb = [], []
                for _ in range(a.rounds):
                    tg.append(time_calls(grid, a.calls))
                    tb.append(time_calls(brute, a.calls))
                split, _ = kernel_us(grid, a.calls, ["bq_grid_build_kernel", "bq_grid_query_kernel"])
                row = {"B": B, "N": n, "M": m, "layer": li, "radii": radii, "nsample": ns,
                       "us_grid": float(np.median(tg)), "us_brute": float(np.median(tb)),
                       "us_grid_spread": [float(min(tg)), float(max(tg))], "us_brute_spread": [float(min(tb)), float(max(tb))],
                       "us_grid_build": split["bq_grid_build_kernel"], "us_grid_query": split["bq_grid_query_kernel"],
                       "lists_identical": True}
                row["speedup"] = row["us_brute"] / row["us_grid"]
                rows.append(row)
                print(f"N={n:6d} M={m:6d} layer {li} r={radii}  grid {row['us_grid']:9.1f} us (build {row['us_grid_build']:7.1f}, "
                      f"query {row['us_grid_query']:8.1f})  brute {row['us_brute']:10.1f} us  x{row['speedup']:.1f}", flush=True)
        del xyz
        torch.cuda.empty_cache()


def backbone_level(a, rows):
    real = pu.ball_query_msg
    forced = lambda *x, **k: real(*x, **{**k, "grid": False})  # noqa: E731
    for n in (131072, 262144):
        B = 4
        torch.manual_seed(0)
        net = bb.IASSD_Backbone(bb.waymo_iassd_cfg(), num_class=3, input_channels=5)
        bb.randomize_bn_stats(net, seed=0)
        net = net.cuda().eval()
        pts = torch.from_numpy(scenes.to_points(scenes.make_batch(200, B, n, "waymo"))).cuda()

        def fwd():
            with torch.no_grad():
                return net({"batch_size": B, "points": pts})

        arms = {"auto": real, "brute": forced}
        outs = {}
        for name, f in arms.items():
            pu.ball_query_msg = f
            o = fwd()
            outs[name] = [o["centers"].clone(), o["centers_features"].clone()]
            time_calls(fwd, 1)
        same = all(torch.equal(x, y) for x, y in zip(outs["auto"], outs["brute"]))
        t = {k: [] for k in arms}
        for _ in range(a.rounds):
            for name, f in arms.items():
                pu.ball_query_msg = f
                t[name].append(time_calls(fwd, a.steps))
        row = {"B": B, "N": n, "outputs_identical": same}
        for name, f in arms.items():
            pu.ball_query_msg = f
            us = float(np.median(t[name]))
            ks, total = kernel_us(fwd, 2, ["fps", "bq_grid", "ball_query"])
            row[name] = {"ms_per_forward": us / 1e3, "scenes_per_s": B / (us / 1e6),
                         "ms_spread": [min(t[name]) / 1e3, max(t[name]) / 1e3],
                         "kernel_ms": total / 1e3, "fps_share": ks["fps"] / total,
                         "ball_query_share": (ks["bq_grid"] + ks["ball_query"]) / total}
        pu.ball_query_msg = real
        rows.append(row)
        print(f"backbone 4 x {n}: auto {row['auto']['scenes_per_s']:.1f} scenes/s (FPS {100 * row['auto']['fps_share']:.0f} %, "
              f"ball query {100 * row['auto']['ball_query_share']:.0f} % of kernel time)  brute {row['brute']['scenes_per_s']:.1f} "
              f"scenes/s (ball query {100 * row['brute']['ball_query_share']:.0f} %)  identical={same}", flush=True)
        del net, pts
        torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--steps", type=int, default=5)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "bench_ball_query.py measures on a CUDA device"
    info = gpu_info()
    print(info)
    ops, net = [], []
    op_level(a, ops)
    backbone_level(a, net)
    res = dict(info, inputs="op level: the same inputs every call, L2-resident (<= 25 MB of points), as in the SA layer",
               timing=f"CUDA events, {a.calls} calls (op) / {a.steps} forwards (backbone) per round, {a.rounds} rounds "
                      "alternating the arms, median round; build / query split and kernel shares from torch.profiler",
               op_level=ops, backbone=net)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
