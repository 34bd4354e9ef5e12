"""-m gpu: the op-level drop-in (VERDICT round 1, task 10).  spsnet_b200/shims/{pointnet2_batch_cuda,iou3d_nms_cuda}.py carry
the exact pybind11 names of the reference's extensions (pointnet2_api.cpp:10-26, iou3d_nms_api.cpp:9-15) over libspsk.so.
A helper process injects them under the reference's module paths and runs the reference's UNMODIFIED `pointnet2_utils.py`,
`pointnet2_modules.py`, `IASSD_backbone.py` and `iou3d_nms_utils.py` on them; this process runs the same code on the rebuilt
reference extension.  Indices / copies / boxes: bit-exact; conv outputs: same cuDNN path on both sides."""
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parents[1]
from spsnet_b200 import configs, scenes  # noqa: E402


def test_reference_python_layer_runs_unmodified_over_the_shim(ref_ops, ref_det, tmp_path):
    if ref_ops is None or ref_det is None:
        pytest.skip("runs the reference's own Python layer from oracle/_ref (oracle/build_ref.sh), which the repository does not hold")
    out = tmp_path / "shim.npz"
    r = subprocess.run([sys.executable, str(ROOT / "tests" / "run_reference_over_shim.py"), str(out)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    got = np.load(out)
    import importlib

    ref_bb = importlib.import_module("pcdet.models.backbones_3d.IASSD_backbone")
    pu = ref_ops.utils
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        B, N = 2, 4096
        cfg = configs.Cfg({"SA_CONFIG": {**configs.KITTI_IASSD_SA_CONFIG, "NPOINT_LIST": [[1024], [256], [128], [64], [-1], [64]]}})
        torch.manual_seed(4)
        net = ref_bb.IASSD_Backbone(cfg, num_class=3, input_channels=4)
        configs.randomize_bn_stats(net, seed=4)
        net = net.cuda().eval()
        pts = torch.from_numpy(scenes.to_points(scenes.make_batch(90, B, N))).cuda()
        with torch.no_grad():
            res = net({"batch_size": B, "points": pts})
        for i, t in enumerate(res["encoder_xyz"]):
            np.testing.assert_array_equal(got[f"encoder_xyz_{i}"], t.cpu().numpy(), err_msg=f"encoder_xyz[{i}]")
        np.testing.assert_allclose(got["centers_features"], res["centers_features"].cpu().numpy(), rtol=0, atol=1e-5)
        np.testing.assert_array_equal(got["centers"], res["centers"].cpu().numpy())
        xyz = pts[:, 1:4].reshape(B, N, 3).contiguous()
        idx = pu.furthest_point_sample(xyz, 300)
        np.testing.assert_array_equal(got["fps"], idx.cpu().numpy())
        new_xyz = pu.gather_operation(xyz.transpose(1, 2).contiguous(), idx).transpose(1, 2).contiguous()
        ball = pu.ball_query(0.8, 16, xyz, new_xyz)
        np.testing.assert_array_equal(got["ball"], ball.cpu().numpy())
        np.testing.assert_array_equal(got["ball_dilated"], pu.ball_query_dilated(1.6, 0.8, 16, xyz, new_xyz).cpu().numpy())
        f = torch.randn(B, 6, N, generator=torch.Generator().manual_seed(1)).cuda().requires_grad_(True)
        g = pu.grouping_operation(f, ball)
        g.sum().backward()
        np.testing.assert_array_equal(got["group"], g.detach().cpu().numpy())
        np.testing.assert_allclose(got["group_grad"], f.grad.cpu().numpy(), rtol=0, atol=1e-4)   # atomics: order differs
        d, i3 = pu.three_nn(xyz, new_xyz)
        np.testing.assert_array_equal(got["three_nn_i"], i3.cpu().numpy())
        np.testing.assert_array_equal(got["three_nn_d"], d.cpu().numpy())
        w = torch.softmax(-d, dim=-1).contiguous()
        np.testing.assert_array_equal(got["three_interp"], pu.three_interpolate(f.detach()[:, :, :300].contiguous(), i3, w).cpu().numpy())
        dist = torch.cdist(xyz[:, :512], xyz[:, :512]).pow(2).contiguous()
        np.testing.assert_array_equal(got["ffps"], pu.furthest_point_sample_with_dist(dist, 64).cpu().numpy())
        boxes = torch.from_numpy(scenes.make_boxes(3, 300)).cuda()
        scores = torch.linspace(1, 0, 300).cuda()
        keep, _ = ref_det.utils.nms_gpu(boxes, scores, 0.1)
        np.testing.assert_array_equal(got["nms_keep"], keep.cpu().numpy())
        np.testing.assert_array_equal(got["iou_bev"], ref_det.utils.boxes_iou_bev(boxes[:50], boxes[50:120]).cpu().numpy())
        np.testing.assert_array_equal(got["iou3d"], ref_det.utils.boxes_iou3d_gpu(boxes[:50], boxes[50:120]).cpu().numpy())
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def test_torch_library_ops_opcheck_and_match_python_api():
    """torch.ops.spsk.* (spsnet_b200/torch_ops.py): torch.library.opcheck (schema, fake tensor, autograd registration) on real
    inputs, results identical to the autograd.Function aliases, gradients through register_autograd equal to theirs."""
    import spsnet_b200.torch_ops  # noqa: F401
    from spsnet_b200 import pointnet2_utils as pu

    B, N, M = 2, 777, 64
    xyz = torch.from_numpy(np.ascontiguousarray(scenes.make_batch(3, B, N)[:, :, :3])).cuda()
    f = torch.randn(B, 6, N, device="cuda")
    ops = torch.ops.spsk
    idx = ops.furthest_point_sample(xyz, M)
    assert torch.equal(idx, pu.furthest_point_sample(xyz, M))
    ctr = ops.gather_rows(xyz, idx)
    ball = ops.ball_query(0.8, 16, xyz, ctr)
    assert torch.equal(ball, pu.ball_query(0.8, 16, xyz, ctr))
    assert torch.equal(ops.ball_query_dilated(1.6, 0.8, 8, xyz, ctr), pu.ball_query_dilated(1.6, 0.8, 8, xyz, ctr))
    assert torch.equal(ops.gather_points(f, idx), pu.gather_operation(f, idx))
    assert torch.equal(ops.group_points(f, ball), pu.grouping_operation(f, ball))
    d, i3 = ops.three_nn(ctr, xyz)
    d2, i32 = pu.three_nn(ctr, xyz)
    assert torch.equal(d, d2) and torch.equal(i3, i32)
    w = torch.softmax(-d, dim=-1).contiguous()
    assert torch.equal(ops.three_interpolate(f, i3, w), pu.three_interpolate(f, i3, w))
    cls = torch.from_numpy(scenes.make_cls_logits(1, B, N)).cuda()
    assert torch.equal(ops.score_topk(cls, 100), pu.score_topk(cls, 100))
    # gradients
    for op, fn, args in [(ops.gather_points, pu.gather_operation, (idx,)), (ops.group_points, pu.grouping_operation, (ball,)),
                         (ops.three_interpolate, pu.three_interpolate, (i3, w))]:
        a = f.clone().requires_grad_(True)
        b = f.clone().requires_grad_(True)
        ya, yb = op(a, *args), fn(b, *args)
        g = torch.randn_like(ya)
        ya.backward(g)
        yb.backward(g)
        assert torch.allclose(a.grad, b.grad, atol=1e-4)
    tests = ("test_schema", "test_faketensor", "test_autograd_registration")
    torch.library.opcheck(ops.furthest_point_sample.default, (xyz, M), test_utils=tests)
    torch.library.opcheck(ops.ball_query.default, (0.8, 16, xyz, ctr), test_utils=tests)
    torch.library.opcheck(ops.gather_points.default, (f.clone().requires_grad_(True), idx), test_utils=tests)
    torch.library.opcheck(ops.group_points.default, (f.clone().requires_grad_(True), ball), test_utils=tests)
    torch.library.opcheck(ops.three_interpolate.default, (f.clone().requires_grad_(True), i3, w), test_utils=tests)
    torch.library.opcheck(ops.score_topk.default, (cls, 100), test_utils=tests)
