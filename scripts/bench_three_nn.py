#!/usr/bin/env python
"""three_nn: spsk_three_nn as shipped (the grid kernel above the thresholds of include/spsk.h) against the all-pairs kernel.

    python scripts/bench_three_nn.py [--out FILE.json] [--rounds 5] [--calls 10]

The all-pairs arm calls spsk_three_nn once on the unknown points cut into chunks of THREE_NN_GRID_MIN_N - 1 and stacked along
the batch (each chunk with a copy of its scene's known points): that always takes the all-pairs kernel, with as many CTAs as
an uncut call, and gives the same result (unknown points are independent).  Shapes: the three feature-propagation layers of a KITTI
batch (B 16), three Waymo-shaped ones (B 8), and one shape on each side of each threshold.  Inputs are scenes.py's
LiDAR-shaped scenes; known points are a D-FPS subset of them.  CUDA events around `--calls` back-to-back calls; the two arms
alternate within each of `--rounds` rounds after a warm-up, and the median round and the spread are reported.  Every call
reads the same inputs, which stay resident in the 126 MB L2 (at most 8 x 262144 x 12 B = 25 MB of unknown points), as they
are when an FP layer runs right after the layer before it.  Both arms' dist2 and idx are compared bit for bit first.  The GPU
name and power limit are read in the same run."""
import argparse
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from spsnet_b200 import pointnet2_utils as pu  # noqa: E402
from spsnet_b200 import scenes  # noqa: E402
from spsnet_b200._lib import check, lib  # noqa: E402

MIN_N, MIN_M, MAX_M = pu.THREE_NN_GRID_MIN_N, pu.THREE_NN_GRID_MIN_M, pu.THREE_NN_GRID_MAX_M
SHAPES = [  # (label, B, kind, n unknown, m known)
    ("kitti fp0", 16, "kitti", 16384, 4096), ("kitti fp1", 16, "kitti", 4096, 1024), ("kitti fp2", 16, "kitti", 1024, 256),
    ("waymo", 8, "waymo", 65536, 16384), ("waymo", 8, "waymo", 262144, 65536), ("waymo", 8, "waymo", 262144, 16384),
    ("n below MIN_N", 16, "kitti", MIN_N - 1, 1024), ("n at MIN_N", 16, "kitti", MIN_N, 1024),
    ("m below MIN_M", 16, "kitti", 16384, MIN_M - 1), ("m at MIN_M", 16, "kitti", 16384, MIN_M),
    ("m at MAX_M", 2, "waymo", 262144, MAX_M), ("m above MAX_M", 2, "waymo", 262144, MAX_M + 1),
]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[0] if q.returncode == 0 else None}


def raw(unknown, known, out):
    B, N, _ = unknown.shape
    check(lib.spsk_three_nn(B, N, known.shape[1], unknown.data_ptr(), known.data_ptr(), out[0].data_ptr(), out[1].data_ptr(),
                            torch.cuda.current_stream().cuda_stream), "three_nn")


def arms(unknown, known):
    """The shipped call, and the all-pairs kernel in ONE launch: the unknown points cut into chunks of MIN_N - 1 (the last one
    padded with repeated rows), stacked along the batch, each chunk with its own copy of its scene's known points."""
    B, N, _ = unknown.shape
    auto_out = (torch.empty(B, N, 3, device="cuda"), torch.empty(B, N, 3, dtype=torch.int32, device="cuda"))
    step = MIN_N - 1
    nch = (N + step - 1) // step
    pad = nch * step - N
    u = torch.cat([unknown, unknown[:, :pad]], 1) if pad else unknown
    us = u.reshape(B * nch, step, 3).contiguous()
    ks = known.repeat_interleave(nch, 0).contiguous()
    chunk_out = (torch.empty(B * nch, step, 3, device="cuda"), torch.empty(B * nch, step, 3, dtype=torch.int32, device="cuda"))

    def auto():
        raw(unknown, known, auto_out)

    def brute():
        raw(us, ks, chunk_out)

    def brute_result():
        return tuple(o.reshape(B, nch * step, 3)[:, :N] for o in chunk_out)

    return auto, brute, auto_out, brute_result


def time_calls(fn, calls):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(calls):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / calls


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--calls", type=int, default=10)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "bench_three_nn.py measures on a CUDA device"
    info = gpu_info()
    print(info, flush=True)
    rows = []
    for label, B, kind, n, m in SHAPES:
        xyz = torch.from_numpy(np.ascontiguousarray(scenes.make_batch(300, B, n, kind)[:, :, :3])).cuda()
        known = pu.gather_rows(xyz, pu.furthest_point_sample(xyz, m)).contiguous()
        auto, brute, auto_out, brute_result = arms(xyz, known)
        auto()
        brute()
        torch.cuda.synchronize()
        bd, bi = brute_result()
        identical = torch.equal(auto_out[1], bi) and torch.equal(auto_out[0].view(torch.int32), bd.view(torch.int32))
        assert identical, f"{label}: B={B} n={n} m={m}: grid and all-pairs results differ"
        grid = n >= MIN_N and MIN_M <= m <= MAX_M   # the kernel choice of spsk_three_nn (asserted by the GPU tests)
        ta, tb = [], []
        for _ in range(a.rounds):
            ta.append(time_calls(auto, a.calls))
            tb.append(time_calls(brute, a.calls))
        row = {"shape": label, "B": B, "n": n, "m": m, "auto_kernel": "three_nn_cluster_kernel" if grid else "three_nn_kernel",
               "us_auto": float(np.median(ta)), "us_allpairs": float(np.median(tb)),
               "us_auto_spread": [float(min(ta)), float(max(ta))], "us_allpairs_spread": [float(min(tb)), float(max(tb))],
               "pair_tests_allpairs": B * n * m, "outputs_identical": identical}
        row["speedup"] = row["us_allpairs"] / row["us_auto"]
        rows.append(row)
        print(f"{label:14s} B={B:2d} n={n:6d} m={m:6d} {row['auto_kernel']:24s} auto {row['us_auto']:10.1f} us "
              f"[{min(ta):.1f}, {max(ta):.1f}]  all-pairs {row['us_allpairs']:10.1f} us [{min(tb):.1f}, {max(tb):.1f}]  "
              f"x{row['speedup']:.2f}", flush=True)
        del xyz, known
        torch.cuda.empty_cache()
    res = dict(info, thresholds={"MIN_N": MIN_N, "MIN_M": MIN_M, "MAX_M": MAX_M},
               inputs="scenes.py batches, known = D-FPS subset; the same inputs every call, L2-resident (<= 25 MB)",
               timing=f"CUDA events, {a.calls} calls per round, {a.rounds} rounds alternating the arms, median round and "
                      "[min, max] over rounds; the all-pairs arm is one launch over chunks of MIN_N - 1 unknown points stacked along the batch",
               rows=rows)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
