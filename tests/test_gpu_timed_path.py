"""-m gpu parity of the TIMED path itself (VERDICT round 1, "what's weak" #1):

  (a) the headline configurations at full size -- KITTI 16 x 16384, SPSNet-IA 16 x 16384 with stds, Waymo 8 x 65536 --
      against a recorded forward of the same batch (tests/helpers.py::check_backbone_vs_recorded: every layer's samples
      bit-exact, features / logits within 1e-3) and, where oracle/_ref is installed, against the unmodified reference backbone,
      D-FPS layers bit-exact end to end, every layer teacher-forced;
  (b) `BackbonePipeline(depth=8, use_graph=True)` -- per-slot streams, graph replay, static buffers, pinned mirrors, FPS
      prefetch side stream: >= 24 DISTINCT batches, every slot's outputs torch.equal to the eager forward of the same batch;
  (c) the persistent-tile loops of `sa_mma` (ring / phase parities across tiles) against the ORACLE (C grouping + fp32 torch-CPU
      chain, not the FFMA sibling) at >= 8 tiles per CTA for every chain class: resident narrow (split), resident plain, ring,
      ring + overlay, two epilogue warpgroups.
"""
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parents[1]
from helpers import REL_TOL, check_backbone_vs_recorded, rel_err  # noqa: E402
from spsnet_b200 import scenes  # noqa: E402


def _net(workload):
    from spsnet_b200 import backbone as bb

    cfg_fn, cls_name, B, N, cols, kind = {
        "kitti": (bb.kitti_iassd_cfg, "IASSD_Backbone", 16, 16384, 4, "kitti"),
        "spsnet": (bb.kitti_spsnet_cfg, "PAGNet_Backbone", 16, 16384, 4, "kitti"),
        "waymo": (bb.waymo_iassd_cfg, "IASSD_Backbone", 8, 65536, 5, "waymo"),
    }[workload]
    torch.manual_seed(0)
    net = getattr(bb, cls_name)(cfg_fn(), num_class=3, input_channels=cols)
    bb.randomize_bn_stats(net, seed=0)
    return net.cuda().eval(), B, N, kind, (cls_name, cfg_fn, cols)


@pytest.mark.parametrize("workload", ["kitti", "spsnet", "waymo"])
def test_headline_config_vs_reference(ref_ops, recorded, workload):
    """BASELINE.json configs[1], [2], [3] at their full sizes (TF32 off) against a recorded forward of the same batch
    (tests/helpers.py::check_backbone_vs_recorded) and, where oracle/_ref is installed, against the reference's own backbone +
    CUDA ops, teacher-forced layer by layer (oracle/parity.py)."""
    from oracle import parity

    net, B, N, kind, (cls_name, cfg_fn, cols) = _net(workload)
    pts = torch.from_numpy(scenes.to_points(scenes.make_batch(4242, B, N, kind))).cuda()
    extra = {"stds": torch.from_numpy(scenes.make_stds(77, B, N)).cuda()} if workload == "spsnet" else {}
    with parity._Fp32Reference(), torch.no_grad():
        out = net({"batch_size": B, "points": pts.clone(), **extra})
    check_backbone_vs_recorded(recorded, out)
    if ref_ops is not None:
        ref = parity.reference_backbone(cls_name, cfg_fn(), cols).cuda().eval()
        assert list(ref.state_dict().keys()) == list(net.state_dict().keys())
        ref.load_state_dict(net.state_dict())
        rep = parity.teacher_forced_check(net, ref, B, pts, extra=extra, feat_tol=REL_TOL, logit_tol=REL_TOL)
        print(f"[timed-path parity] {workload}: {rep}")
        assert rep["fps_layers_bit_exact"] == [1, 2]


def test_same_seed_gives_reference_identical_weights(ref_ops, recorded):
    """bench.py's reference arm builds the reference's modules from the seed alone (it must not import this package's
    kernels): same torch seed + same randomize_bn_stats => the very weights our arm uses.  Checked against the reference's
    classes where oracle/_ref is installed, and always against the recorded weights (every key and value, bit for bit)."""
    from spsnet_b200 import backbone as bb
    from spsnet_b200 import configs

    for cls_name, cfg_fn, cols in [("IASSD_Backbone", bb.kitti_iassd_cfg, 4), ("PAGNet_Backbone", bb.kitti_spsnet_cfg, 4),
                                   ("IASSD_Backbone", bb.waymo_iassd_cfg, 5)]:
        torch.manual_seed(0)
        mine = getattr(bb, cls_name)(cfg_fn(), num_class=3, input_channels=cols)
        configs.randomize_bn_stats(mine, seed=0)
        a = mine.state_dict()
        blob = b"".join(k.encode() + np.ascontiguousarray(v.numpy()).tobytes() for k, v in a.items())
        recorded.exact(f"{cls_name}_{cols}", np.frombuffer(blob, np.uint8))
        if ref_ops is not None:
            from oracle import parity

            torch.manual_seed(0)
            ref = parity.reference_backbone(cls_name, cfg_fn(), cols)
            configs.randomize_bn_stats(ref, seed=0)
            b = ref.state_dict()
            assert list(a) == list(b)
            for k in a:
                assert torch.equal(a[k], b[k]), k


@pytest.mark.parametrize("workload,depth", [("kitti", 8), ("spsnet", 3)])
def test_pipeline_graph_replay_equals_eager(workload, depth):
    """24 distinct batches through BackbonePipeline.submit_host (H2D -> graph replay on the slot's stream -> D2H), 8 in
    flight: every slot's pinned outputs are bit-identical to the eager forward of that batch on the default stream."""
    from spsnet_b200 import backbone as bb
    from spsnet_b200.runtime import BackbonePipeline

    B, N, cols = 16, 16384, 5
    cfg_fn, cls = (bb.kitti_iassd_cfg, bb.IASSD_Backbone) if workload == "kitti" else (bb.kitti_spsnet_cfg, bb.PAGNet_Backbone)
    torch.manual_seed(0)
    net = cls(cfg_fn(), num_class=3, input_channels=cols - 1)
    bb.randomize_bn_stats(net, seed=0)
    net = net.cuda().eval()
    extra = {"stds": torch.from_numpy(scenes.make_stds(77, B, N)).cuda()} if workload == "spsnet" else None
    n_batches = 24
    host = [torch.from_numpy(scenes.to_points(scenes.make_batch(9000 + i * B, B, N))).pin_memory() for i in range(n_batches)]
    pipe = BackbonePipeline(net, B, N, cols, depth=depth, use_graph=True, extra_inputs=extra)
    pipe.prepare(host[0].cuda())
    got = [None] * n_batches
    for g0 in range(0, n_batches, depth):
        slots = [pipe.submit_host(host[i]) for i in range(g0, min(g0 + depth, n_batches))]
        for i, s in zip(range(g0, g0 + depth), slots):
            out = pipe.host_out(s)
            got[i] = {k: v.clone() for k, v in out.items()}
    pipe.sync()
    with torch.no_grad():
        for i in range(n_batches):
            d = {"batch_size": B, "points": host[i].cuda()}
            d.update(extra or {})
            want = net(d)
            for k in ("centers_features", "centers"):
                assert torch.equal(got[i][k], want[k].cpu()), f"batch {i} (slot {i % depth}): `{k}` differs between graph replay and eager"
    # the device-input entry point replays the same graphs
    dev = [h.cuda() for h in host[:depth]]
    slots = [pipe.submit_device(t) for t in dev]
    pipe.sync()
    for i, s in enumerate(slots):
        assert torch.equal(pipe.slots[s].outs["centers_features"].cpu(), got[i]["centers_features"])


MANY_TILE_CASES = {  # name: (c_feat, nsample, radius, widths)  -- one per chain class of sa_mma.cu
    "l0s2_resident_split": (1, 32, 0.8, [32, 32, 64]),
    "l1s2_resident_plain": (64, 32, 1.6, [64, 96, 128]),
    "l2s2_ring": (128, 32, 4.8, [128, 256, 256]),
    "l5s1_ring_two_groups": (256, 16, 4.8, [256, 256, 512]),
    "l5s2_ring_overlay_two_groups": (256, 32, 6.4, [256, 512, 1024]),
}


@pytest.mark.parametrize("name", list(MANY_TILE_CASES))
def test_sa_mma_many_tiles_per_cta_vs_oracle(oracle, name):
    from spsnet_b200 import pointnet2_utils as pu
    from test_gpu_mma import _chain

    c_feat, ns, radius, widths = MANY_TILE_CASES[name]
    chain = _chain(c_feat, widths, seed=11)
    packed = pu.MmaChain(chain, c_feat, True)
    assert packed.ok
    tiles = 8 * 148 * packed.ctas_per_sm + 37   # >= 8 tiles for every persistent CTA, plus a ragged tail
    B, N = 2, 8192
    M = (tiles * 128 // ns + B - 1) // B
    rng = np.random.default_rng(5)
    xyz_np = np.ascontiguousarray(scenes.make_batch(11, B, N)[:, :, :3])
    feats_np = rng.standard_normal((B, c_feat, N)).astype(np.float32)
    ctr_np = np.ascontiguousarray(xyz_np[:, rng.integers(0, N, M)] + rng.normal(0, 0.05, (B, M, 3)).astype(np.float32))
    xyz, feats, new_xyz = (torch.from_numpy(a).cuda() for a in (xyz_np, feats_np, ctr_np))
    idx = pu.ball_query(radius, ns, xyz, new_xyz)
    idx_np = idx.cpu().numpy()
    np.testing.assert_array_equal(idx_np[:, :64], oracle.ball_query(radius, ns, xyz_np, ctr_np[:, :64]))
    twin = pu.make_twin(feats, packed.cpad8) if not packed.split else None
    cout = widths[-1]
    got = torch.full((B, cout, M), -7.0, device="cuda")
    pu.sa_mma_forward(xyz=xyz, new_xyz=new_xyz, idx=idx, chain=packed, twin=twin, features=feats if packed.split else None, out_pooled=got)
    torch.cuda.synchronize()
    got = got.cpu().numpy()
    # oracle: C grouping (reference pointnet2_utils.py:307-315) + the fp32 chain on the host, a slab of centres at a time
    cpu_chain = [(wt.cpu(), b.cpu()) for wt, b, _ in chain]
    want = np.empty((B, cout, M), np.float32)
    step = max(1, (1 << 21) // ns)
    for m0 in range(0, M, step):
        m1 = min(M, m0 + step)
        grouped, _ = oracle.query_and_group(radius, ns, xyz_np, ctr_np[:, m0:m1], feats_np, True, idx=np.ascontiguousarray(idx_np[:, m0:m1]))
        x = torch.from_numpy(grouped).permute(0, 2, 3, 1).reshape(-1, c_feat + 3)
        for wt, b in cpu_chain:
            x = torch.relu(x @ wt + b)
        want[:, :, m0:m1] = x.reshape(B, m1 - m0, ns, cout).amax(dim=2).permute(0, 2, 1).numpy()
    e = rel_err(got, want)
    tol = 2e-5 if packed.split else REL_TOL
    print(f"[many tiles] {name}: {tiles} tiles, ctas/SM={packed.ctas_per_sm} resident={packed.resident} stages={packed.nstages} "
          f"split={packed.split}: rel err vs oracle {e:.2e}")
    assert e <= tol, f"{name}: {e:.3e} > {tol}"


def test_pw_mma_many_rows_vs_oracle():
    """Point-wise GEMM (aggregation shape 1536 -> 512) with far more row tiles than CTAs, against torch-CPU fp64."""
    from spsnet_b200 import pointnet2_utils as pu

    rows, c_in, c_out = 148 * 32 * 9 + 13, 1536, 512
    g = torch.Generator().manual_seed(2)
    x = torch.randn(rows, c_in, generator=g)
    xh = x.half()
    x16 = torch.cat([xh, (x - xh.float()).half()], dim=1).cuda().contiguous()
    wt = torch.randn(c_in, c_out, generator=g) * (1.3 / np.sqrt(c_in))
    b = torch.randn(c_out, generator=g) * 0.1
    layer = pu.PwLayer(wt.cuda(), b.cuda(), True, split=True)
    out_pm = torch.full((1, rows, c_out), -7.0, device="cuda")
    pu.pw_mma_forward(x16, layer, xlo=c_in, out_pm=out_pm)
    torch.cuda.synchronize()
    want = (x.double() @ wt.double() + b.double()).clamp_min(0)
    e = rel_err(out_pm.cpu().double().reshape(rows, c_out).numpy(), want.numpy())
    print(f"[pw many rows] {rows} x {c_in} -> {c_out}: {e:.2e}")
    assert e <= 2e-5


def test_fp16_range_guard_falls_back_to_exact_kernels(ref_ops, recorded):
    """VERDICT round 1, task 9.  BN gains that push the hidden activations of SA layers 1, 2 and 5 far beyond 65504 (the
    largest fp16 value) while the reference's fp32 / TF32 result stays finite: the tensor-core kernels flag the overflow, the
    backbone's eager forward polls the flag, moves the affected modules to the exact-fp32 kernels and re-runs -- same sampled
    points, features within 1e-3 of the recorded exact-kernel forward (TF32 off) and, where oracle/_ref is installed, of the
    UNMODIFIED reference, teacher-forced.  Without the guard the fp16 path returns non-finite / wrong features, which the test
    demonstrates too."""
    import os
    import warnings

    from oracle import parity
    from spsnet_b200 import backbone as bb
    from spsnet_b200 import pointnet2_utils as pu

    cfg = bb.Cfg({"SA_CONFIG": {**bb.KITTI_IASSD_SA_CONFIG, "NPOINT_LIST": [[1024], [256], [128], [64], [-1], [64]]}})
    torch.manual_seed(6)
    net = bb.IASSD_Backbone(cfg, num_class=3, input_channels=4)
    bb.randomize_bn_stats(net, seed=6)
    gain = 3.0e5
    with torch.no_grad():
        for li in (1, 2, 5):
            for mlp in net.SA_modules[li].mlps:
                mlp[1].weight.mul_(gain)      # BN after the first conv: hidden activations ~1e5..1e6
                mlp[1].bias.mul_(gain)
                mlp[3].weight.div_(gain)      # the next conv undoes the scale: everything downstream stays O(1)
    net = net.cuda().eval()
    B, N = 2, 4096
    pts = torch.from_numpy(scenes.to_points(scenes.make_batch(31, B, N))).cuda()
    pu.fp16_overflow(clear=True)
    # (1) guard off: the overflow is real
    os.environ["SPSK_FP16_GUARD"] = "0"
    try:
        with torch.no_grad():
            bad = net({"batch_size": B, "points": pts.clone()})
        assert pu.fp16_overflow(clear=True) != 0, "the kernels did not flag the fp16 overflow"
        f = bad["encoder_features"][2]
    finally:
        del os.environ["SPSK_FP16_GUARD"]
    # (2) guard on (default): detected, exact fallback, reference-grade results
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        with parity._Fp32Reference(), torch.no_grad():
            good = net({"batch_size": B, "points": pts.clone()})
    assert any("fp16 range" in str(x.message) for x in w), "the guard did not report the fallback"
    assert [bool(getattr(m, "_spsk_exact", False)) for m in net.SA_modules] == [False, True, True, False, False, True]
    check_backbone_vs_recorded(recorded, good)
    assert not torch.isfinite(f).all() or recorded.err("encoder_features2", f) > 1e-2
    if ref_ops is not None:
        ref = parity.reference_backbone("IASSD_Backbone", cfg, 4).cuda().eval()
        ref.load_state_dict(net.state_dict())
        with torch.no_grad():
            f_ref = ref({"batch_size": B, "points": pts.clone()})["encoder_features"][2]
        assert not torch.isfinite(f).all() or parity.rel_err(f.cpu().numpy(), f_ref.cpu().numpy()) > 1e-2
        rep = parity.teacher_forced_check(net, ref, B, pts, fps_layers=(1, 2))
        print(f"[fp16 guard] teacher-forced after fallback: {rep['layers']}")
    with torch.no_grad():
        out = net({"batch_size": B, "points": pts.clone()})
    assert torch.isfinite(out["centers_features"]).all()
    # the pipeline checks while it warms up, BEFORE it captures: a fresh copy of the same weights ends up on the exact kernels too
    from spsnet_b200.runtime import BackbonePipeline

    net2 = bb.IASSD_Backbone(cfg, num_class=3, input_channels=4).cuda().eval()
    net2.load_state_dict(net.state_dict())
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        pipe = BackbonePipeline(net2, B, N, 5, depth=2, use_graph=True)
        pipe.prepare(pts)
    slot = pipe.submit_device(pts)
    pipe.sync()
    pipe.check_overflow()
    assert torch.equal(pipe.slots[slot].outs["centers_features"], out["centers_features"])
