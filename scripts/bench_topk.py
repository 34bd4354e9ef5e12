#!/usr/bin/env python
"""Score-based down-sampling: pu.score_topk (one launch; one CTA per scene up to 16384 points, a 2/4/8/16-CTA cluster above)
against the reference's own torch chain, torch.topk(torch.sigmoid(cls.max(dim=-1)[0]), k, dim=-1)[1].int(), and its
stability-weighted ('sss') variant.

    python scripts/bench_topk.py [--out FILE.json] [--rounds 5] [--calls 20]

CUDA events around `--calls` back-to-back calls; the two arms alternate within each of `--rounds` rounds after a warm-up of
every shape, and the median round is reported.  Inputs are read from HBM, not L2: each call takes the next input set of a
pool larger than twice the 126 MB L2.  Before timing, each shape checks that pu.score_topk equals torch's stable
descending sort of the same scores.  The GPU name and power limit are read in the same run."""
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

POOL_BYTES = 256 << 20   # > 2 x the 126 MB L2 of a B200
CTA_KEYS = 16384


def torch_chain(cls, k, stds=None):
    s = torch.sigmoid(cls.max(dim=-1)[0])
    if stds is not None:
        s = s * (1 - torch.sigmoid(stds / 8 - 3))
    return torch.topk(s, k, dim=-1)[1].int()


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[0] if q.returncode == 0 else None}


_cursor = [0]   # the next input set of the pool, shared by both arms: a set is read again only after the whole pool


def time_calls(fn, pool, calls):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(calls):
        fn(*pool[_cursor[0] % len(pool)])
        _cursor[0] += 1
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / calls


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--calls", type=int, default=20)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "bench_topk.py measures on a CUDA device"
    info = gpu_info()
    print(info)
    rows = []
    gen = torch.Generator(device="cuda").manual_seed(0)
    for B in (1, 8):
        for n in (16384, 32768, 65536, 131072, 262144):
            set_bytes = B * n * 4 * 4   # cls (3 classes) + stds
            pool = []
            for _ in range(max(2, -(-POOL_BYTES // set_bytes))):
                cls = torch.randn(B, n, 3, device="cuda", generator=gen) * 2
                stds = 8 * torch.exp(0.5 * torch.randn(B, n, device="cuda", generator=gen))
                pool.append((cls, stds))
            csize = max(1, (1 << (n - 1).bit_length()) // CTA_KEYS)
            for k in (n // 4, n // 2):
                for with_stds in (False, True):
                    ours = (lambda c, s: pu.score_topk(c, k, stds=s)) if with_stds else (lambda c, s: pu.score_topk(c, k))
                    ref = (lambda c, s: torch_chain(c, k, s)) if with_stds else (lambda c, s: torch_chain(c, k))
                    c0, s0 = pool[0]
                    t = torch.sigmoid(c0.max(dim=-1)[0]) * ((1 - torch.sigmoid(s0 / 8 - 3)) if with_stds else 1)
                    want = torch.sort(t, dim=-1, descending=True, stable=True)[1][:, :k].int()
                    assert torch.equal(ours(c0, s0), want), f"score_topk differs from torch's stable sort at B={B} n={n} k={k}"
                    for fn in (ours, ref):   # warm-up
                        time_calls(fn, pool, 3)
                    t_ours, t_ref = [], []
                    for _ in range(a.rounds):
                        t_ours.append(time_calls(ours, pool, a.calls))
                        t_ref.append(time_calls(ref, pool, a.calls))
                    row = {"B": B, "n": n, "k": k, "stds": with_stds, "csize": csize, "sms_held": B * csize,
                           "us_ours": float(np.median(t_ours)), "us_torch": float(np.median(t_ref)),
                           "us_ours_spread": [float(min(t_ours)), float(max(t_ours))],
                           "us_torch_spread": [float(min(t_ref)), float(max(t_ref))]}
                    row["speedup"] = row["us_torch"] / row["us_ours"]
                    rows.append(row)
                    print(f"B={B} n={n:6d} k={k:6d} stds={int(with_stds)} csize={csize:2d} SMs={B * csize:3d}  "
                          f"ours {row['us_ours']:8.1f} us  torch {row['us_torch']:8.1f} us  x{row['speedup']:.2f}", flush=True)
            del pool
            torch.cuda.empty_cache()
    res = dict(info, inputs=f"each call reads the next input set of a pool of >= {POOL_BYTES >> 20} MB (> 2 x L2): from HBM",
               timing=f"CUDA events, {a.calls} calls per round, {a.rounds} rounds alternating the arms, median round", rows=rows)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
