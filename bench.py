#!/usr/bin/env python
"""bench.py -- IA-SSD set-abstraction backbone throughput (BASELINE.json metric) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference|reference-cpu] [--workload kitti|spsnet|waymo|...]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W [--scaling strong]

A step = one forward of the full KITTI IA-SSD SA stack (BASELINE.json configs[1]: D-FPS 16384->4096->1024,
ctr-aware top-k ->512->256, vote layer, MSG ball query + shared MLP) over one batch of 16 synthetic
16384-point scenes, eval mode.  Scenes are independent: with N > 1 every rank runs its own batches
(weak scaling, no data-path collective); NCCL carries only the timing reduction.  `--scaling strong` instead cuts ONE
host batch of 128 scenes per step into contiguous per-rank shards (spsnet_b200.sharding.shard_range).

Prints ONE JSON line (rank 0).  `value` = whole-job scenes/s with inputs resident in HBM (a pool of
distinct batches larger than L2 is cycled); `e2e` = the same metric through `BackbonePipeline.submit_host`
(pinned host input -> H2D -> forward -> D2H of the centre features, every step); `depth1` = the same with ONE batch in
flight (latency view); `roofline` describes the dominant kernel of the step (CUDA-event timed in an instrumented eager pass
of the same run); `cpu_baseline` = the CPU oracle port (oracle/) timed on a bounded sample on the host cores;
`verified` = verdict of the parity gate: before anything is timed, a helper process (`bench.py --verify-only`) runs one
full-size batch through this arm (eager and graph replay) and through the unmodified reference (oracle/_ref, TF32 off) with
the bars of tests/test_gpu_timed_path.py -- D-FPS layers bit-exact, every layer teacher-forced, features / logits <= 1e-3.

--impl reference runs the UNMODIFIED reference (its pointnet2_batch CUDA ops rebuilt for sm_100a + its own
pointnet2_modules.py + IASSD_backbone.py, installed by oracle/build_ref.sh into oracle/_ref) on the same GPU, the same
seeded weights, the same inputs; that process imports spsnet_b200.configs / scenes only and maps none of this repo's
kernels (`native_so_loaded` lists what it did map).  When oracle/_ref is unavailable it falls back to the CPU oracle
port (--impl reference-cpu forces the CPU port).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "IA-SSD SA-backbone scenes/s (16k pts)"
# what the path computes in (a label, not a precision claim): shared-MLP chains of layers 1/2/5 multiply fp32 values rounded to
# fp16 (11-bit significand, like the TF32 the reference's cuDNN convolutions use) and accumulate in fp32; narrow chains (K <= 64)
# and every Conv1d GEMM carry hi + lo fp16 halves (fp32-grade); sampling / ball query / top-k are exact fp32 + int32
DTYPE = "fp16 operands / fp32 accumulate (split-fp16 hi+lo for K <= 64 chains and all Conv1d GEMMs); fp32 + int32 sampling"
DTYPE_REF = "fp32 storage, cuDNN TF32 convolutions (stock cudnn.allow_tf32=True), fp32 + int32 sampling"
UNIT = "scenes/s"
BATCH = 16
NPTS = 16384
NCOLS = 5  # [batch_idx, x, y, z, intensity]
L2_BYTES = 126 * 1024 * 1024
WORKLOAD = ("IA-SSD KITTI cfg full SA stack (D-FPS 16384->4096->1024, ctr-aware top-k ->512->256, vote, "
            "MSG ball query + shared MLP), batch 16 x 16384 pts per GPU, eval")
KIND = "kitti"

# BASELINE.json configs: [1] = kitti (the headline, default), [2] = spsnet (stability-aware top-k), [3] = waymo
WORKLOADS = {
    "kitti": dict(batch=16, npts=16384, ncols=5, kind="kitti", cfg="kitti_iassd_cfg", bb="IASSD_Backbone", text=WORKLOAD),
    "spsnet": dict(batch=16, npts=16384, ncols=5, kind="kitti", cfg="kitti_spsnet_cfg", bb="PAGNet_Backbone",
                   text="SPSNet-IA KITTI cfg: stability-score (sss_aware) top-k sampling in SA layers 2,3 with per-point stds, "
                        "otherwise the IA-SSD SA stack, batch 16 x 16384 pts per GPU, eval"),
    "spsnet_sf": dict(batch=16, npts=16384, ncols=5, kind="kitti", cfg="kitti_spsnet_surface_cfg", bb="PAGNet_Backbone",
                      text="SPSNet-IA backbone exactly as shipped (SPSNet.yaml): stability-score top-k with per-point stds, USE_SURFACE "
                           "(4 DenseEdgeConv units on all 16384 points -> 60 surface channels into the vote layer), 124-wide layer-1 "
                           "MLPs, batch 16 x 16384 pts per GPU, eval"),
    "spsnet_full": dict(batch=16, npts=16384, ncols=5, kind="kitti", cfg="kitti_spsnet_surface_cfg", bb="SPSNET_DET",
                        text="SPSNet-IA detector as shipped (SPSNet.yaml), inference: stability generator (-> stds) -> PAGNet_Backbone with "
                             "stability-score top-k + USE_SURFACE -> MLT_SSD_Head -> decode + rotated-IoU NMS, batch 16 x 16384 pts per GPU"),
    "spsnet_e2e": dict(batch=16, npts=16384, ncols=5, kind="kitti", cfg="kitti_spsnet_cfg", bb="SPSNetIA",
                       text="SPSNet-IA end to end on the path: stability generator (SA layer with M = N = 16384 centres + logvar "
                            "head -> stds) feeding the PAGNet backbone with stability-score top-k, batch 16 x 16384 pts per GPU, eval"),
    "kitti_det": dict(batch=16, npts=16384, ncols=5, kind="kitti", cfg="kitti_iassd_cfg", bb="IASSD_DET",
                      text="IA-SSD KITTI detector, inference: the full SA stack + IASSD_Head (2 x 3-layer FC on 256 centres x 512 ch) + box "
                           "decode + score filter + rotated-IoU NMS -> final boxes (SURVEY.md 8f rank 3), batch 16 x 16384 pts per GPU"),
    "waymo_det": dict(batch=8, npts=65536, ncols=6, kind="waymo", cfg="waymo_iassd_cfg", bb="IASSD_DET",
                      text="IA-SSD Waymo detector, inference: the Waymo SA stack (65536 -> 16384 -> 4096 -> 2048 -> 1024 centres) + IASSD_Head + "
                           "box decode + score filter + rotated-IoU NMS over 1024 boxes per scene, batch 8 x 65536 pts per GPU"),
    "waymo": dict(batch=8, npts=65536, ncols=6, kind="waymo", cfg="waymo_iassd_cfg", bb="IASSD_Backbone",
                  text="IA-SSD Waymo cfg full SA stack (D-FPS 65536->16384->4096, ctr-aware top-k ->2048->1024, vote, MSG ball "
                       "query + shared MLP), batch 8 x 65536 pts per GPU, eval"),
}
_WL = WORKLOADS["kitti"]


def set_workload(name: str):
    global BATCH, NPTS, NCOLS, WORKLOAD, KIND, _WL, METRIC
    _WL = WORKLOADS[name]
    if _WL["bb"] == "IASSD_DET":
        METRIC = "IA-SSD detector (SA backbone + head + NMS) scenes/s (%s pts)" % ("64k" if _WL["kind"] == "waymo" else "16k")
    if _WL["bb"] == "SPSNET_DET":
        METRIC = "SPSNet-IA detector (stability generator + SA backbone + head + NMS) scenes/s (16k pts)"
    BATCH, NPTS, NCOLS, WORKLOAD, KIND = _WL["batch"], _WL["npts"], _WL["ncols"], _WL["text"], _WL["kind"]


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int, enabled: bool = True):
        self.gpu = gpu_index
        self.enabled = enabled
        self.proc = None
        self.path = Path(f"/tmp/spsk_clocks_{os.getpid()}.csv")

    def start(self):
        if not self.enabled:
            return
        try:
            self.fh = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "100"], stdout=self.fh, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.fh.close()
        sm, mx, reasons = [], [], set()
        for line in self.path.read_text().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        try:
            self.path.unlink()
        except OSError:
            pass
        return out


def build_net(seed=0):
    from spsnet_b200 import backbone as bb

    torch.manual_seed(seed)
    if _WL["bb"] == "IASSD_DET":
        from spsnet_b200 import detector

        if KIND == "waymo":
            from spsnet_b200 import dense_head as dh

            net = detector.IASSD({"BACKBONE_3D": bb.waymo_iassd_cfg(), "POINT_HEAD": dh.waymo_iassd_head_cfg(),
                                  "POST_PROCESSING": dh.waymo_post_processing()}, num_class=3, input_channels=NCOLS - 1)
        else:
            net = detector.IASSD(num_class=3, input_channels=NCOLS - 1)
    elif _WL["bb"] == "SPSNET_DET":
        from spsnet_b200 import detector
        from spsnet_b200 import stability as st

        net = detector.SPSNetIA(num_class=3, input_channels=NCOLS - 1, generator=st.Generate_center(st.sf_unc_cfg()))
    elif _WL["bb"] == "SPSNetIA":
        from spsnet_b200 import stability as st

        net = st.SPSNetIAFrontEnd(st.Generate_center(st.sf_unc_cfg()),
                                  bb.PAGNet_Backbone(getattr(bb, _WL["cfg"])(), num_class=3, input_channels=NCOLS - 1))
    else:
        net = getattr(bb, _WL["bb"])(getattr(bb, _WL["cfg"])(), num_class=3, input_channels=NCOLS - 1)
    bb.randomize_bn_stats(net, seed=seed)
    return net.eval()


def extra_inputs(device):
    """Per-point stability `stds` for the SPSNet workload (generator output stand-in, SURVEY.md section 8d)."""
    if _WL["bb"] != "PAGNet_Backbone":
        return None
    from spsnet_b200 import scenes

    return {"stds": torch.from_numpy(scenes.make_stds(77, BATCH, NPTS)).to(device)}


def make_pool(rank: int, n_batches: int):
    """n_batches distinct batches in OpenPCDet `points` layout, pinned host tensors."""
    from spsnet_b200 import scenes

    pool = []
    for i in range(n_batches):
        arr = scenes.to_points(scenes.make_batch(100000 * rank + i * BATCH, BATCH, NPTS, KIND))
        pool.append(torch.from_numpy(arr).pin_memory())
    return pool


def cpu_baseline(net_cpu, sample_scenes: int):
    """The oracle port (oracle/oracle.py + oracle.c, all host threads) on a bounded sample of the workload."""
    from oracle import oracle as O
    from spsnet_b200 import scenes

    pts = scenes.make_batch(0, sample_scenes, NPTS, KIND)
    det = hasattr(net_cpu, "point_head")
    backbone = net_cpu.backbone_3d if det else net_cpu

    def run(p):
        out = O.backbone_forward(backbone, p, dtype=torch.float32)
        if det:  # head + decode + post-processing restatement (oracle.py: head_forward, post_processing)
            import types

            from spsnet_b200 import dense_head as dh

            h = net_cpu.point_head
            ns = types.SimpleNamespace(cls_center_layers=h.cls_center_layers, box_center_layers=h.box_center_layers,
                                       mean_size=h.box_coder._mean_np, bin_size=h.box_coder.bin_size)
            centers = np.concatenate([np.repeat(np.arange(p.shape[0]), out["centers"].shape[1])[:, None].astype(np.float32),
                                      out["centers"].reshape(-1, 3)], axis=1)
            cls, _, boxes = O.head_forward(ns, out["centers_features"], centers, dtype=torch.float32)
            pp = dh.waymo_post_processing() if KIND == "waymo" else dh.KITTI_POST_PROCESSING
            nc = pp["NMS_CONFIG"]
            O.post_processing(cls, boxes, p.shape[0], pp["SCORE_THRESH"], nc["NMS_THRESH"], nc["NMS_PRE_MAXSIZE"], nc["NMS_POST_MAXSIZE"])

    run(pts[:1])  # warm (page in, build)
    t0 = time.perf_counter()
    for s0 in range(0, sample_scenes, 8):   # 8 scenes at a time: the torch-CPU conv outputs of a whole sample would take GBs
        run(pts[s0:s0 + 8])
    dt = time.perf_counter() - t0
    cores = max(O.num_threads(), torch.get_num_threads())
    return {"value": sample_scenes / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{sample_scenes} scenes of the same workload (full SA stack, fp32), oracle/oracle.c ops (OpenMP) + torch-CPU "
                      f"conv/BN, {dt:.1f} s; host has {os.cpu_count()} logical cpus"}


# --------------------------------------------------------------------------------------------------
# kernel table: algorithmic work per launch (SURVEY.md section 8d) for the roofline object
# --------------------------------------------------------------------------------------------------

def profile_kernels(net, dev_points, steps: int):
    """Instrumented eager pass: CUDA events around every libspsk call on the launching stream."""
    from spsnet_b200 import _lib

    records = []
    originals = {}
    names = [n for n in _lib.SIGNATURES if n not in ("spsk_last_error", "spsk_abi_version", "spsk_built_for_sm", "spsk_launch_count")]

    def wrap(name, fn):
        def inner(*a):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            rc = fn(*a)
            e1.record()
            if name == "spsk_grouped_linear":  # a[0] is byref(GroupDesc): read the row count while it is alive
                g = a[0]._obj
                a = (int(g.b) * int(g.m) * int(g.nsample),) + tuple(a[1:])
            elif name == "spsk_sa_mma_forward":
                g = a[0]._obj
                nl = int(g.nlayers)
                a = (int(g.b) * int(g.m) * int(g.nsample), [int(g.kpad[i]) for i in range(nl)], [int(g.cpad[i]) for i in range(nl)],
                     int(g.cout_last), int(g.split), int(g.c_feat) + (3 if g.use_xyz else 0))
            elif name == "spsk_pw_mma_forward":
                g = a[0]._obj
                a = (int(g.rows), int(g.k), int(g.n))
            elif name.startswith("spsk_ball_query_msg"):
                a = tuple(a[:5]) + ([int(a[5][i]) for i in range(int(a[3]))],)
            elif name == "spsk_detect_postprocess":
                g = a[0]._obj
                a = (int(g.batch), int(g.m), int(g.post_max))
            records.append((name, a, e0, e1))
            return rc
        return inner

    for n in names:
        originals[n] = getattr(_lib.lib, n)
        setattr(_lib.lib, n, wrap(n, originals[n]))
    # per-kernel durations must not include a concurrent kernel: keep the layer-1 FPS prefetch (side stream) off in this pass
    prev_prefetch = os.environ.get("SPSK_FPS_PREFETCH")
    os.environ["SPSK_FPS_PREFETCH"] = "0"
    try:
        with torch.no_grad():
            for i in range(steps):
                d = {"batch_size": BATCH, "points": dev_points[i % len(dev_points)]}
                d.update(extra_inputs("cuda") or {})
                net.forward_padded(d) if hasattr(net, "forward_padded") else net(d)
        torch.cuda.synchronize()
    finally:
        for n in names:
            setattr(_lib.lib, n, originals[n])
        if prev_prefetch is None:
            os.environ.pop("SPSK_FPS_PREFETCH", None)
        else:
            os.environ["SPSK_FPS_PREFETCH"] = prev_prefetch
    table = {}
    order = []
    for name, a, e0, e1 in records:
        key = name
        if name in ("spsk_farthest_point_sampling",):
            key = f"{name}[n={a[1]},m={a[2]}]"
        elif name in ("spsk_ball_query_msg", "spsk_ball_query_msg_grid"):
            key = f"{name}[n={a[1]},m={a[2]}]"
        elif name == "spsk_grouped_linear":
            key = f"{name}[cin={a[3]},cout={a[6]}]"
        elif name == "spsk_sa_mma_forward":
            key = f"{name}[rows={a[0]},cout={a[3]}{',split' if a[4] else ''}]"
        elif name == "spsk_pw_mma_forward":
            key = f"{name}[rows={a[0]},k={a[1]},n={a[2]}]"
        ms = e0.elapsed_time(e1)
        t = table.setdefault(key, {"ms": 0.0, "launches": 0, "args": a})
        t["ms"] += ms
        t["launches"] += 1
        order.append(key)
    dump = os.environ.get("SPSK_DUMP_CALLS")
    if dump:   # the library calls of ONE step, in launch order (scripts/ncu_traffic.py aligns an ncu launch list with it)
        per = len(order) // steps
        Path(dump).write_text(json.dumps(order[-per:]))
    return table, steps


N_SMS = 148


def _fps_sms(b, n):
    return b * (1 if n <= 16384 else (2 if n <= 32768 else (4 if n <= 65536 else 8)))


def _roof_entry(key, t, peaks, traffic):
    """Roofline of one kernel class: ALGORITHMIC work per launch (SURVEY.md section 8d) / mean CUDA-event duration."""
    avg_s = t["ms"] / t["launches"] / 1e3
    a = t["args"]
    hbm = peaks.get("hbm_gbs", 6650.0)          # measured copy bandwidth, GB/s
    tens = peaks.get("bf16_tflops", 1500.0)     # measured dense bf16 (burst: these kernels are timed alone), TFLOP/s
    sms = N_SMS
    e = {"kernel": key, "avg_us": avg_s * 1e6}
    if key.startswith("spsk_farthest_point_sampling"):
        b, n, m = a[0], a[1], a[2]
        sms = _fps_sms(b, n)
        alg_bytes = b * (n * 12 + m * 4)  # read xyz once + write idx
        pairs = b * n * (m - 1)
        lane_peak = N_SMS * 128 * 1.965e9  # fp32 lane-ops/s at max clock
        e.update(bound="hbm", achieved=alg_bytes / avg_s / 1e9, peak=hbm, unit="GB/s",
                 note="FPS is latency-bound (m-1 strictly sequential arg-max steps, one CTA or CTA-cluster per scene): neither "
                      "the HBM nor the tensor roofline applies; see us_per_iter / cycles_per_iter / lane_frac",
                 us_per_iter=avg_s * 1e6 / max(m - 1, 1), cycles_per_iter=avg_s * 1.965e9 / max(m - 1, 1),
                 pair_evals_per_s=pairs / avg_s, lane_frac=pairs * 10 / avg_s / lane_peak)
    elif key.startswith("spsk_sa_mma_forward"):
        rows_n, kpad, cpad, cout_last, split, k0 = a
        widths = [k0] + list(cpad[:-1]) + [cout_last]
        flops = 2.0 * rows_n * sum(x * y for x, y in zip(widths[:-1], widths[1:]))
        e.update(bound="tensor", achieved=flops / avg_s / 1e12, peak=tens, unit="TFLOP/s",
                 note="fused gather + shared MLP + max-pool; algorithmic flops from the true layer widths (split-fp16 chains "
                      "issue 3x these on the tensor cores); peak = measured dense bf16 cuBLAS throughput")
    elif key.startswith("spsk_pw_mma_forward"):
        rows_n, k, n = a
        e.update(bound="tensor", achieved=2.0 * rows_n * k * n / avg_s / 1e12, peak=tens, unit="TFLOP/s",
                 note="point-wise Conv1d GEMM (hi+lo fp16 operands: 3x these flops issued)")
    elif key.startswith("spsk_grouped_linear") or key.startswith("spsk_pointwise_linear"):
        if key.startswith("spsk_grouped_linear"):
            rows_n, cin, cout = a[0], a[3], a[6]
        else:
            rows_n, cin, cout = a[0] * a[1], a[3], a[6]
        e.update(bound="tensor", achieved=2.0 * rows_n * cin * cout / avg_s / 1e12, peak=74.4, unit="TFLOP/s",
                 note="exact-fp32 FFMA path: peak is the fp32 CUDA-core peak (148 SM x 128 lanes x 2 x 1.965 GHz)")
    elif key.startswith("spsk_ball_query_msg"):
        b, n, m = a[0], a[1], a[2]
        nsum = sum(int(x) for x in a[5][:a[3]]) if len(a) > 5 else 48
        alg_bytes = b * (n * 12 + m * 12 + m * nsum * 4)
        e.update(bound="hbm", achieved=alg_bytes / avg_s / 1e9, peak=hbm, unit="GB/s",
                 note="algorithmic bytes = xyz + centres + index lists; the kernel is fp32-issue / latency bound, not HBM bound")
    elif key.startswith("spsk_edge_conv_point"):
        rows_n, cin = int(a[1]), int(a[3])
        e.update(bound="tensor", achieved=2.0 * rows_n * (cin * 24 + 24 * 48) / avg_s / 1e12, peak=74.4, unit="TFLOP/s",
                 note="per-point transform FC + [P|Q|R2|R3] projections of a DenseEdgeConv unit, fp32 FFMA with constant-bank "
                      "weights; peak = fp32 CUDA-core peak")
    elif key.startswith("spsk_edge_conv_aggregate"):
        b, n, k = int(a[1]), int(a[2]), int(a[3])
        e.update(bound="tensor", achieved=2.0 * b * n * k * 432 / avg_s / 1e12, peak=74.4, unit="TFLOP/s",
                 note="per-(point, neighbour) dense edge MLP + max over neighbours, fp32 FFMA (432 MACs per row; repeated padding "
                      "indices are skipped, so this is an upper bound of the work done); peak = fp32 CUDA-core peak")
    elif key.startswith("spsk_detect_postprocess"):
        b, m, post = a
        alg_bytes = b * m * (33 + 3 + 7 + 2) * 4 + b * post * (7 + 1 + 2 + 2) * 4   # logits + encodings + centres in, boxes/scores/labels out
        e.update(bound="hbm", achieved=alg_bytes / avg_s / 1e9, peak=hbm, unit="GB/s",
                 note="3 launches (decode + score sort, IoU bit mask, greedy pass); latency-bound: 256 boxes per scene, the greedy "
                      "pass is sequential over 64-box blocks -- neither roofline applies")
    else:
        e.update(bound="hbm", achieved=None, peak=hbm, unit="GB/s")
    e["frac"] = (e["achieved"] / e["peak"]) if e.get("achieved") else None
    e["sms_used"] = sms
    e["sm_time_ms_per_step"] = None
    # DRAM bytes of THIS kernel instance (one launch) from the committed ncu --set full capture; null when that instance
    # was not captured (never the number of a sibling instance of the same kernel class)
    e["traffic"] = traffic.get(key) if traffic else None
    e["peak_source"] = "MEASURED_PEAKS.json" if peaks else "fallback (B200_PROFILING.md)"
    return e


def roofline_from_table(table, steps, peaks):
    """Rooflines of the step's kernels.  Returned: (dominant, per-kernel rows, list of rooflines).  "Dominant" = largest
    SM-time (duration x SMs held / 148): with several batches in flight the step is bound by SM-time, and the
    latency-bound FPS (16 of 148 SMs) would otherwise hide the kernels that actually fill the GPU."""
    total = sum(t["ms"] for t in table.values())
    traffic = {}
    tp = ROOT / "profiles" / "traffic_r02.json"   # {kernel key incl. its shape: dram bytes per launch}, scripts/ncu_traffic.py
    if tp.exists():
        try:
            traffic = json.loads(tp.read_text())
        except Exception:
            traffic = {}
    rows, roofs = [], []
    for key, t in sorted(table.items(), key=lambda kv: -kv[1]["ms"]):
        rows.append({"kernel": key, "ms_per_step": t["ms"] / steps, "launches_per_step": t["launches"] / steps,
                     "share": t["ms"] / total})
        if t["ms"] / total >= 0.01:
            e = _roof_entry(key, t, peaks, traffic)
            e["sm_time_ms_per_step"] = t["ms"] / steps * e["sms_used"] / N_SMS
            roofs.append(e)
    roofs.sort(key=lambda e: -e["sm_time_ms_per_step"])
    return roofs[0], rows, roofs


def load_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return json.loads(p.read_text())
        except Exception:
            return {}
    return {}


# --------------------------------------------------------------------------------------------------
# arms
# --------------------------------------------------------------------------------------------------

def timed_region(pipe, inputs, steps, warmup, host: bool, world: int, per_step: int = 1):
    """W warm-up steps, then EXACTLY K steps bracketed by barrier + synchronize; device-side events.  A step submits `per_step`
    batches (1 in weak scaling; this rank's share of the host batch in strong scaling).  Returns (ms, wall seconds, the
    pipeline slot of the last batch)."""
    import torch.distributed as dist

    submit = pipe.submit_host if host else pipe.submit_device
    k = 0
    for _ in range(warmup * per_step):
        submit(inputs[k % len(inputs)])
        k += 1
    pipe.sync()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    main = torch.cuda.current_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(main)
    pipe.fork(main)
    t0 = time.perf_counter()
    for _ in range(steps * per_step):
        last = submit(inputs[k % len(inputs)])
        k += 1
    pipe.join(main)
    e1.record(main)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    if world > 1:
        dist.barrier()
    from spsnet_b200 import sharding

    # the only communication of the path: SUM of scenes, MAX of the device-timed milliseconds (spsnet_b200/sharding.py)
    _, ms = sharding.reduce_report(BATCH * steps * per_step, e0.elapsed_time(e1), device="cuda")
    return ms, wall, last


def dump_outputs(outs, out_dir, budget=64 << 20):
    """The arrays a caller of the timed path receives, as <name>.npy: floats in float32, integers in float64 (exact).  An
    array above its share of `budget` keeps a fixed, seeded sample of its rows, so two builds compare output for output."""
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    share = budget // max(len(outs), 1)
    for k, v in outs.items():
        a = v.float().numpy() if v.is_floating_point() else v.numpy().astype(np.float64)
        if a.nbytes > share:
            keep = max(1, share * a.shape[0] // a.nbytes)
            a = a[np.sort(np.random.RandomState(0).choice(a.shape[0], keep, replace=False))]
        np.save(out_dir / f"{k}.npy", np.ascontiguousarray(a))


class EagerRef:
    """Adapter giving the reference backbone the same submit/sync surface (no graphs: its forward host-syncs)."""

    def __init__(self, net, outputs=("centers_features", "centers"), extra=None):
        self.net, self.outputs = net, outputs
        self.extra = extra or {}
        self.stream = torch.cuda.current_stream()
        self.host_outs = None
        self.dev_in = torch.zeros((BATCH * NPTS, NCOLS), dtype=torch.float32, device="cuda")
        self.last = None

    def _fwd(self, pts):
        with torch.no_grad():
            out = self.net({"batch_size": BATCH, "points": pts, **self.extra})
        self.last = {k: out[k] for k in self.outputs}

    def submit_device(self, dev_points):
        self._fwd(dev_points)

    def submit_host(self, host_points):
        self.dev_in.copy_(host_points, non_blocking=True)
        self._fwd(self.dev_in)
        if self.host_outs is None or any(self.host_outs[k].shape != v.shape for k, v in self.last.items()):
            # (the reference detector returns variable-length results: fresh pinned mirrors when the shapes change)
            self.host_outs = {k: torch.empty(v.shape, dtype=v.dtype, pin_memory=True) for k, v in self.last.items()}
        for k, v in self.last.items():
            self.host_outs[k].copy_(v, non_blocking=True)

    def sync(self):
        torch.cuda.synchronize()

    def fork(self, stream):
        pass

    def join(self, stream):
        pass

    def h2d_bytes(self):
        return BATCH * NPTS * NCOLS * 4

    def d2h_bytes(self):
        return sum(v.numel() * v.element_size() for v in self.last.values())


class RefDetector(torch.nn.Module):
    """The reference's own detector pieces, unmodified, wired the way Detector3DTemplate does: IASSD_Backbone ->
    IASSD_Head (pcdet/models/dense_heads/IASSD_head.py) -> post_processing (detector3d_template.py:207-290, the
    class-agnostic branch, restated here around the reference's class_agnostic_nms / nms_gpu because the template class
    itself imports the whole of pcdet)."""

    def __init__(self, backbone, head, post_cfg, nms_utils):
        super().__init__()
        self.backbone_3d, self.point_head = backbone, head
        self.post_cfg, self.nms_utils = post_cfg, nms_utils

    def forward(self, batch_dict):
        batch_dict = self.point_head(self.backbone_3d(batch_dict))
        cfg = self.post_cfg
        boxes_out, scores_out, labels_out = [], [], []
        for index in range(batch_dict["batch_size"]):
            batch_mask = batch_dict["batch_index"] == index
            box_preds = batch_dict["batch_box_preds"][batch_mask]
            cls_preds = torch.sigmoid(batch_dict["batch_cls_preds"][batch_mask])
            cls_preds, label_preds = torch.max(cls_preds, dim=-1)
            label_preds = label_preds + 1
            selected, selected_scores = self.nms_utils.class_agnostic_nms(
                box_scores=cls_preds, box_preds=box_preds, nms_config=cfg.NMS_CONFIG, score_thresh=cfg.SCORE_THRESH)
            boxes_out.append(box_preds[selected])
            scores_out.append(selected_scores)
            labels_out.append(label_preds[selected])
        counts = torch.tensor([b.shape[0] for b in boxes_out], dtype=torch.int32)
        return {"det_boxes": torch.cat(boxes_out), "det_scores": torch.cat(scores_out), "det_labels": torch.cat(labels_out),
                "det_count": counts}


# --------------------------------------------------------------------------------------------------
# the reference arm's model: built from the SEED alone, through spsnet_b200.configs (which does not load libspsk.so)
# and oracle/_ref only -- no product module is imported, so the arm's process maps none of this repo's kernels.
# Same torch seed + same constructor order + configs.randomize_bn_stats == the very weights of our arm
# (tests/test_gpu_timed_path.py::test_same_seed_gives_reference_identical_weights; `bench.py --verify-only` re-checks it).
# --------------------------------------------------------------------------------------------------

def _ref_import(name):
    import importlib
    import types
    import warnings

    ref_root = ROOT / "oracle" / "_ref"
    so = ref_root / "pcdet" / "ops" / "pointnet2" / "pointnet2_batch" / "pointnet2_batch_cuda.so"
    if not so.exists():
        raise RuntimeError("oracle/_ref not built (run oracle/build_ref.sh where /root/reference exists)")
    if str(ref_root) not in sys.path:
        sys.path.insert(0, str(ref_root))
    sys.modules.setdefault("SharedArray", types.ModuleType("SharedArray"))  # absent dependency of pcdet.utils.common_utils, unused here
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return importlib.import_module(name)


def build_reference_from_seed(seed=0):
    import copy

    from spsnet_b200 import configs as cf

    if _WL["bb"] not in ("IASSD_Backbone", "IASSD_DET", "PAGNet_Backbone"):
        raise RuntimeError("the reference arm runs the IASSD_Backbone / PAGNet_Backbone workloads (kitti, waymo, kitti_det, waymo_det, spsnet, spsnet_sf)")
    cls_name = "PAGNet_Backbone" if _WL["bb"] == "PAGNet_Backbone" else "IASSD_Backbone"
    mod = _ref_import("pcdet.models.backbones_3d." + cls_name.replace("_Backbone", "_backbone"))
    torch.manual_seed(seed)
    backbone = getattr(mod, cls_name)(getattr(cf, _WL["cfg"])(), num_class=3, input_channels=NCOLS - 1)
    if _WL["bb"] != "IASSD_DET":
        cf.randomize_bn_stats(backbone, seed=seed)
        return backbone.eval()
    hm = _ref_import("pcdet.models.dense_heads.IASSD_head")
    nu = _ref_import("pcdet.models.model_utils.model_nms_utils")
    hcfg = copy.deepcopy(dict(cf.waymo_iassd_head_cfg()) if KIND == "waymo" else cf.KITTI_IASSD_HEAD)
    hcfg["LOSS_CONFIG"] = {"LOSS_CLS": "WeightedCrossEntropy", "LOSS_REG": "WeightedSmoothL1Loss", "LOSS_INS": "WeightedCrossEntropy",
                           "CORNER_LOSS_REGULARIZATION": False, "CENTERNESS_REGULARIZATION": False, "IOU3D_REGULARIZATION": False,
                           "LOSS_WEIGHTS": {"code_weights": [1.0] * 6}}
    head = hm.IASSD_Head(3, 512, cf.Cfg(hcfg))
    det = RefDetector(backbone, head, cf.Cfg(cf.waymo_post_processing() if KIND == "waymo" else cf.KITTI_POST_PROCESSING), nu)
    cf.randomize_bn_stats(det, seed=seed)
    return det.eval()


def loaded_repo_libraries():
    """Which of this repo's shared objects are mapped into this process (the arm's own evidence for `native_so_loaded`)."""
    out = set()
    try:
        for ln in open("/proc/self/maps"):
            path = ln.rstrip().split(" ")[-1]
            if path.endswith(".so") and str(ROOT) in path:
                out.add(os.path.relpath(path, ROOT))
    except OSError:
        pass
    return sorted(out)


def pin_rank_to_cores(local: int, world: int):
    """One block of host cores per rank (8 submit loops + 8 clock samplers otherwise migrate over the same NUMA node)."""
    try:
        cores = sorted(os.sched_getaffinity(0))
        per = max(1, len(cores) // max(world, 1))
        mine = cores[local * per:(local + 1) * per] or cores
        os.sched_setaffinity(0, mine)
        return f"{mine[0]}-{mine[-1]}"
    except (AttributeError, OSError):
        return None


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=64)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-cpu"])
    ap.add_argument("--depth", type=int, default=8, help="pipeline slots (streams) of BackbonePipeline: batches in flight; hides the\n                    latency-bound FPS (16 of 148 SMs per batch) behind the GEMM-heavy kernels of other batches")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--pool", type=int, default=0, help="distinct input batches (0 = enough to exceed L2)")
    ap.add_argument("--cpu-sample", type=int, default=64, help="scenes in the cpu_baseline sample (0 = skip): 64 scenes = 10-15 s of host work")
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--no-depth1", action="store_true", help="skip the extra single-batch-in-flight (latency) measurement")
    ap.add_argument("--no-verify", action="store_true", help="skip the parity gate (a helper process: this arm vs oracle/_ref on one full-size batch)")
    ap.add_argument("--verify-only", action="store_true", help="run the parity gate alone and print its JSON verdict")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: every rank runs its own batches of 16 scenes (default, the driver's scaling run); strong: ONE host batch of "
                         "--total-scenes scenes per step is cut into contiguous shards by spsnet_b200.sharding.shard_range")
    ap.add_argument("--total-scenes", type=int, default=128, help="strong scaling: scenes in the host batch of one step")
    ap.add_argument("--pin", action="store_true", help="pin each rank to its own block of host cores (opt-in: on the 16-core / 8-GPU boxes of "
                    "this pool two cores per rank starve the CUDA helper threads: e2e 70.6k vs 78.2k scenes/s at N = 8, profiles/r02_*)")
    ap.add_argument("--out16", action="store_true", help="e2e: return centre features as fp16 (halves the D2H bytes; opt-in, default fp32 like the reference)")
    ap.add_argument("--timeline", action="store_true", help="e2e: CUDA-event timeline of H2D / forward / D2H per step (rank 0), printed in `e2e.timeline`")
    ap.add_argument("--dump-outputs", metavar="DIR", help="--impl ours: after the timed steps, write what the last timed step "
                    "returned as DIR/<name>.npy (float32 / float64; a fixed, seeded sample of rows where the outputs exceed 64 MB); "
                    "with several ranks, rank 0's batch")
    ap.add_argument("--workload", default="kitti", choices=sorted(WORKLOADS), help="kitti = BASELINE.json configs[1] (headline)")
    return ap.parse_args()


def strong_plan(args, rank, world):
    """(first scene of this rank inside the host batch, batches this rank runs per step)."""
    from spsnet_b200 import sharding

    lo, hi = sharding.shard_range(args.total_scenes, rank, world)
    if (hi - lo) % BATCH != 0 or hi == lo:
        raise SystemExit(f"strong scaling: the shard of rank {rank} ({hi - lo} scenes) must be a positive multiple of {BATCH}")
    return lo, (hi - lo) // BATCH


def make_pool_for(args, rank, world):
    """Pinned host batches this rank cycles through; together larger than L2."""
    from spsnet_b200 import scenes

    if args.scaling == "weak":
        n_pool = args.pool or (L2_BYTES // (BATCH * NPTS * NCOLS * 4) + 2)
        return make_pool(rank, n_pool), 1, n_pool
    lo, per_step = strong_plan(args, rank, world)
    n_host = args.pool or max(2, (L2_BYTES // (args.total_scenes // world * NPTS * NCOLS * 4)) + 2)
    pool = []
    for i in range(n_host):           # host batch i = scenes [i * total, (i + 1) * total); this rank owns [lo, hi) of each
        for b in range(per_step):
            arr = scenes.to_points(scenes.make_batch(i * args.total_scenes + lo + b * BATCH, BATCH, NPTS, KIND))
            pool.append(torch.from_numpy(arr).pin_memory())
    return pool, per_step, n_host * per_step


def run_verify_only(args):
    """The parity gate: one full-size batch through this arm (eager AND the graph-replay pipeline) and through the unmodified
    reference (oracle/_ref, TF32 off), with the bars of tests/test_gpu_timed_path.py.  Prints {"verified": true|false, ...}."""
    verdict = {"verified": False, "workload": args.workload}
    try:
        from oracle import parity
        from spsnet_b200.runtime import BackbonePipeline

        torch.cuda.set_device(0)
        net = build_net().cuda()
        ref = build_reference_from_seed().cuda()
        mine_bb = net.backbone_3d if hasattr(net, "backbone_3d") else net
        ref_bb = ref.backbone_3d if hasattr(ref, "backbone_3d") else ref
        a, b = net.state_dict(), ref.state_dict()
        same = set(a) == set(b) and all(torch.equal(a[k], b[k]) for k in a)
        verdict["weights_identical_from_seed"] = bool(same)
        assert same, "the reference arm's seed-built weights differ from this arm's"
        from spsnet_b200 import scenes

        pts = torch.from_numpy(scenes.to_points(scenes.make_batch(4242, BATCH, NPTS, KIND))).cuda()
        extra = extra_inputs("cuda") or {}
        rep = parity.teacher_forced_check(mine_bb, ref_bb, BATCH, pts, extra=extra)
        verdict["fps_layers_bit_exact"] = rep["fps_layers_bit_exact"]
        verdict["sampled_set_overlap"] = rep["sampled_set_overlap"]
        worst_f = worst_l = 0.0
        for rec in rep["layers"].values():
            for k, v in rec.items():
                if isinstance(v, dict):
                    if k.endswith("logits"):
                        worst_l = max(worst_l, v["range_rel"])
                    else:
                        worst_f = max(worst_f, v["range_rel"])
        verdict["max_feature_err_range_rel"] = worst_f
        verdict["max_logit_err_range_rel"] = worst_l
        verdict["tolerance"] = parity.REL_TOL
        if not hasattr(net, "forward_padded"):
            # the timed API: graph replay on a slot stream == eager forward of the same batch
            pipe = BackbonePipeline(net, BATCH, NPTS, NCOLS, depth=2, use_graph=True, extra_inputs=extra or None)
            pipe.prepare(pts)
            pts2 = torch.from_numpy(scenes.to_points(scenes.make_batch(777, BATCH, NPTS, KIND)))
            for host in (pts.cpu().pin_memory(), pts2.pin_memory(), pts.cpu().pin_memory()):
                slot = pipe.submit_host(host)
                out = {k: v.clone() for k, v in pipe.host_out(slot).items()}
                with torch.no_grad():
                    want = net({"batch_size": BATCH, "points": host.cuda(), **extra})
                for k in out:
                    assert torch.equal(out[k], want[k].cpu()), f"pipeline output `{k}` differs from the eager forward"
            verdict["pipeline_equals_eager"] = True
        verdict["verified"] = True
        verdict["against"] = "oracle/_ref: unmodified reference backbone + its CUDA ops (sm_100a), TF32 off, teacher-forced per layer"
    except Exception as e:  # the verdict must always be printed
        verdict["error"] = f"{type(e).__name__}: {e}"[:500]
    print("VERIFY " + json.dumps(verdict), flush=True)


def verify_in_helper_process(args, local):
    """Run `bench.py --verify-only` in its own process BEFORE this one touches the GPU's timed state: the reference extension is
    never mapped into the timed process."""
    if _WL["bb"] not in ("IASSD_Backbone", "PAGNet_Backbone", "IASSD_DET"):
        return {"verified": None, "reason": "no reference arm for this workload"}
    env = dict(os.environ)
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT", "TORCHELASTIC_RUN_ID", "GROUP_RANK", "LOCAL_WORLD_SIZE"):
        env.pop(k, None)
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    env["CUDA_VISIBLE_DEVICES"] = vis.split(",")[local] if vis else str(local)
    try:
        r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--verify-only", "--workload", args.workload], env=env,
                           capture_output=True, text=True, timeout=900)
        for ln in r.stdout.splitlines():
            if ln.startswith("VERIFY "):
                return json.loads(ln[len("VERIFY "):])
        return {"verified": False, "error": (r.stderr or r.stdout)[-400:]}
    except Exception as e:
        return {"verified": False, "error": f"{type(e).__name__}: {e}"[:400]}


def main():
    args = parse_args()
    set_workload(args.workload)
    rank, world, local = dist_env()
    args.warmup = max(args.warmup, 3)

    if args.dump_outputs and args.impl != "ours":
        raise SystemExit("bench.py: --dump-outputs writes the outputs of --impl ours only")
    if args.verify_only:
        return run_verify_only(args)
    if args.impl == "reference-cpu" or (args.impl == "reference" and not torch.cuda.is_available()):
        return run_reference_cpu(args, rank, world)

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local)
    pinned = pin_rank_to_cores(local, world) if (args.pin and world > 1) else None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    peaks = load_peaks()

    line = {"metric": METRIC, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": DTYPE, "data": "synthetic"}
    cfg = {"workload": WORKLOAD, "batch_per_gpu": BATCH, "points_per_scene": NPTS,
           "parallelism": f"scene-sharded x{world}, no data-path collective"}
    if args.scaling == "strong":
        cfg["strong_scaling"] = (f"one host batch of {args.total_scenes} scenes per step, cut into contiguous shards by "
                                 f"spsnet_b200.sharding.shard_range ({args.total_scenes // world} scenes = {args.total_scenes // world // BATCH} "
                                 f"sub-batches of {BATCH} per rank)")

    if args.impl == "reference":
        return run_reference_gpu(args, rank, world, local, line, cfg)

    # ---- our arm
    verdict = None
    if rank == 0 and not args.no_verify:
        verdict = verify_in_helper_process(args, local)
    if world > 1:
        import torch.distributed as dist

        dist.barrier()
    from spsnet_b200 import _lib
    from spsnet_b200.runtime import BackbonePipeline

    net = build_net().cuda()
    host_pool, per_step, n_pool = make_pool_for(args, rank, world)
    dev_pool = [t.cuda() for t in host_pool]
    cfg["l2_policy"] = f"input pool of {n_pool} distinct batches ({n_pool * BATCH * NPTS * NCOLS * 4 / 2**20:.0f} MiB > 126 MiB L2) cycled"
    outputs = ("det_boxes", "det_scores", "det_labels", "det_count") if _WL["bb"] in ("IASSD_DET", "SPSNET_DET") else ("centers_features", "centers")
    pipe = BackbonePipeline(net, BATCH, NPTS, NCOLS, depth=args.depth, use_graph=not args.no_graph, extra_inputs=extra_inputs("cuda"),
                            outputs=outputs, out16=args.out16, timeline=args.timeline and rank == 0)
    pipe.prepare(dev_pool[0])
    sampler = ClockSampler(local, enabled=rank == 0)   # one nvidia-smi poller per job, not one per rank (8 pollers contend for the driver)
    sampler.start()
    ms, wall, last = timed_region(pipe, dev_pool, args.steps, args.warmup, host=False, world=world, per_step=per_step)
    # the slot's static outputs are overwritten by the next region: keep the last timed step's on the host
    dumped = {k: v.cpu() for k, v in pipe.slots[last].outs.items()} if args.dump_outputs else None
    pipe.reset_timeline()
    ms_e2e, _, _ = timed_region(pipe, host_pool, args.steps, args.warmup, host=True, world=world, per_step=per_step)
    clocks = sampler.stop()
    scenes_total = world * BATCH * args.steps * per_step
    value = scenes_total / (ms / 1e3)
    e2e = scenes_total / (ms_e2e / 1e3)
    line.update(impl="ours", value=value, ms_per_step=ms / args.steps, clocks=clocks,
                gpu_launches=int(pipe.launches_per_step * args.steps * per_step),
                e2e={"value": e2e, "unit": UNIT, "h2d_bytes_per_step": pipe.h2d_bytes() * per_step, "d2h_bytes_per_step": pipe.d2h_bytes() * per_step,
                     "ms_per_step": ms_e2e / args.steps, "outputs_dtype": "fp16" if args.out16 else "fp32"})
    if args.timeline and rank == 0:
        line["e2e"]["timeline"] = pipe.timeline_summary()
    cfg.update(pipeline_depth=args.depth, cuda_graph=not args.no_graph, launches_per_step=int(pipe.launches_per_step) * per_step)
    if pinned:
        cfg["host_cores_of_rank0"] = pinned
    if verdict is not None:
        line["verified"] = bool(verdict.get("verified"))
        line["verify"] = verdict
    line["native_so_loaded"] = loaded_repo_libraries()

    if not args.no_depth1 and args.depth != 1 and args.scaling == "weak":
        # latency view: ONE batch in flight (the pipeline cannot hide the FPS chain behind other batches)
        pipe1 = BackbonePipeline(net, BATCH, NPTS, NCOLS, depth=1, use_graph=not args.no_graph, extra_inputs=extra_inputs("cuda"), outputs=outputs)
        pipe1.prepare(dev_pool[0])
        s1 = max(8, min(args.steps, 32))
        ms1, _, _ = timed_region(pipe1, dev_pool, s1, 3, host=False, world=world)
        ms1h, _, _ = timed_region(pipe1, host_pool, s1, 3, host=True, world=world)
        line["depth1"] = {"value": world * BATCH * s1 / (ms1 / 1e3), "ms_per_step": ms1 / s1, "steps": s1, "unit": UNIT,
                          "e2e": world * BATCH * s1 / (ms1h / 1e3),
                          "note": "same workload with ONE batch in flight (pipeline_depth 1): ms_per_step here is the latency of a batch"}
        del pipe1

    if rank == 0 and not args.no_profile:
        table, psteps = profile_kernels(net, dev_pool, steps=min(args.steps, 5))
        roof, rows, roofs = roofline_from_table(table, psteps, peaks)
        line["roofline"] = roof
        line["rooflines"] = roofs[:8]
        line["kernels"] = rows[:12]
        line["eager_ms_per_step_sum_of_kernels"] = sum(r["ms_per_step"] for r in rows)
    if rank == 0 and world == 1 and args.cpu_sample > 0:
        try:
            line["cpu_baseline"] = cpu_baseline(build_net(), args.cpu_sample)
        except Exception as e:  # pragma: no cover
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": f"failed: {e}"}
    line["config"] = cfg
    if dumped is not None and rank == 0:
        dump_outputs(dumped, args.dump_outputs)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        import torch.distributed as dist

        dist.barrier()
        dist.destroy_process_group()


def run_reference_gpu(args, rank, world, local, line, cfg):
    """The UNMODIFIED reference (oracle/_ref: its CUDA ops rebuilt for sm_100a + its own python modules) on the same GPU, same
    seeded weights, same inputs.  Nothing of this repo's product is imported: the process maps oracle/_ref's libraries only."""
    try:
        ref = build_reference_from_seed().cuda()
    except Exception as e:  # fall back to the CPU port of the oracle
        if rank == 0:
            sys.stderr.write(f"[bench] reference CUDA module unavailable ({e}); using the CPU oracle port\n")
        return run_reference_cpu(args, rank, world)
    host_pool, per_step, n_pool = make_pool_for(args, rank, world)
    dev_pool = [t.cuda() for t in host_pool]
    cfg["l2_policy"] = f"input pool of {n_pool} distinct batches ({n_pool * BATCH * NPTS * NCOLS * 4 / 2**20:.0f} MiB > 126 MiB L2) cycled"
    torch.backends.cudnn.allow_tf32 = True  # the reference's stock setting (SURVEY.md A.5)
    pipe = EagerRef(ref, outputs=("det_boxes", "det_scores", "det_labels", "det_count") if _WL["bb"] == "IASSD_DET"
                    else ("centers_features", "centers"), extra=extra_inputs("cuda"))
    pipe.submit_device(dev_pool[0])
    pipe.sync()
    sampler = ClockSampler(local, enabled=rank == 0)
    sampler.start()
    ms, _, _ = timed_region(pipe, dev_pool, args.steps, args.warmup, host=False, world=world, per_step=per_step)
    ms_e2e, _, _ = timed_region(pipe, host_pool, args.steps, args.warmup, host=True, world=world, per_step=per_step)
    clocks = sampler.stop()
    scenes_total = world * BATCH * args.steps * per_step
    value = scenes_total / (ms / 1e3)
    e2e = scenes_total / (ms_e2e / 1e3)
    line.update(impl="reference", dtype=DTYPE_REF, value=value, ms_per_step=ms / args.steps, clocks=clocks, gpu_launches=None,
                e2e={"value": e2e, "unit": UNIT, "h2d_bytes_per_step": pipe.h2d_bytes() * per_step, "d2h_bytes_per_step": pipe.d2h_bytes() * per_step,
                     "ms_per_step": ms_e2e / args.steps, "outputs_dtype": "fp32"},
                depth1={"value": value, "ms_per_step": ms / args.steps / per_step, "steps": args.steps, "unit": UNIT, "e2e": e2e,
                        "note": "the reference has no pipelining: one batch in flight is its only mode"},
                cpu_baseline={"value": value, "unit": UNIT, "cores": 0, "kind": "reference",
                              "sample": "not a CPU run: the reference's own CUDA ops (pointnet2_batch rebuilt for sm_100a) + its "
                                        "pointnet2_modules.py / IASSD_backbone.py on the same B200, cudnn.allow_tf32=True (stock); "
                                        "use --impl reference-cpu for the CPU oracle port"},
                native_so_loaded=loaded_repo_libraries())
    cfg["reference"] = "unmodified reference from oracle/_ref on GPU (eager, as shipped), weights built from the same seed"
    line["config"] = cfg
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        import torch.distributed as dist

        dist.destroy_process_group()


def run_reference_cpu(args, rank, world):
    """CPU oracle port as the reference arm (only when the rebuilt reference cannot run): rank 0 only."""
    if rank != 0:
        return
    torch.set_num_threads(os.cpu_count() or 1)
    net = build_net()
    from oracle import oracle as O
    from spsnet_b200 import scenes

    sample = 2
    pts = [scenes.make_batch(i * sample, sample, NPTS, KIND) for i in range(2)]
    for _ in range(min(args.warmup, 1)):
        O.backbone_forward(net, pts[0][:1], dtype=torch.float32)
    steps = min(args.steps, 5)
    t0 = time.perf_counter()
    for i in range(steps):
        O.backbone_forward(net, pts[i % 2], dtype=torch.float32)
    dt = time.perf_counter() - t0
    v = sample * steps / dt
    cores = max(O.num_threads(), torch.get_num_threads())
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": world, "steps": steps,
            "warmup": min(args.warmup, 1), "ms_per_step": dt / steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "fp32 (CPU oracle port)", "data": "synthetic",
            "config": {"workload": WORKLOAD, "sample": f"each step = {sample} scenes of the workload on the host CPU"},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": f"{sample} scenes per step x {steps} steps, oracle/oracle.c (OpenMP) + torch-CPU conv/BN"},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
