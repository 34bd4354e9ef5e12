"""-m gpu: score-based down-sampling of scenes with 16384 < n <= 262144 points (one thread-block cluster of 2/4/8/16 CTAs
per scene, spsk_score_topk).  Indices and scores are compared bit for bit with torch's own op chain followed by a stable
descending sort (descending score, ties by ascending index, NaN first), through every layer above the C-ABI: pu.score_topk,
torch.ops.spsk.score_topk, CUDA-graph replay and PointnetSAModuleMSG_WithSampling."""
import copy

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from helpers import assert_close  # noqa: E402
from spsnet_b200 import scenes  # noqa: E402

CTA_KEYS = 16384   # keys per CTA of the cluster kernel


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def torch_scores(cls, stds=None):
    """The reference's op chain (pointnet2_modules.py:287-303) on the device."""
    t = torch.sigmoid(cls.max(dim=-1)[0])
    if stds is not None:
        t = t * (1 - torch.sigmoid(stds / 8 - 3))
    return t


def stable_topk(t, k):
    v, i = torch.sort(t, dim=-1, descending=True, stable=True)
    return i[:, :k].int(), v[:, :k]


def scene_inputs(b, n, k, num_class, seed):
    """Logits and stds with exact ties across CTA slices and at the k-th position: rounded values on every fifth point and on
    a block around the first slice boundary, and a block of logits of 30.0 (sigmoid == 1.0f) centred on the middle slice
    boundary, longer than k where it fits, so that the cut at k falls inside a group of equal scores."""
    cls = scenes.make_cls_logits(seed, b, n, num_class)
    stds = scenes.make_stds(seed + 1, b, n)
    rounded = np.zeros(n, bool)
    rounded[::5] = True
    rounded[max(0, CTA_KEYS - n // 16): CTA_KEYS + n // 16] = True
    cls[:, rounded] = np.round(cls[:, rounded])
    stds[:, rounded] = np.round(stds[:, rounded])
    csize = 1 << max(0, (n - 1).bit_length() - 14)
    centre = CTA_KEYS * max(1, csize // 2)
    length = max(2, min(n // 2, k + max(1, k // 4)))
    lo = max(0, min(centre - length // 2, n - length))
    cls[:, lo: lo + length, :] = 30.0
    return cls, stds


def check_against_torch(idx, sc, cls_d, stds_d, k):
    want_idx, want_sc = stable_topk(torch_scores(cls_d, stds_d), k)
    assert torch.equal(idx, want_idx), "indices differ from torch's stable descending sort"
    np.testing.assert_array_equal(sc.cpu().numpy(), want_sc.cpu().numpy())   # NaN-aware, otherwise exact
    finite = torch.isfinite(want_sc)
    assert torch.equal(sc[finite].view(torch.int32), want_sc[finite].view(torch.int32)), "score bits differ from torch's"


LARGE_CASES = [  # (b, n, k): every cluster size (2, 4, 8, 16 CTAs) and the edges of each
    (2, 16385, 1), (2, 16385, 16385), (2, 20000, 5000), (1, 32768, 16385), (4, 65536, 16384), (1, 65536, 65536),
    (1, 100000, 4096), (2, 131072, 32768), (1, 131073, 1000), (1, 262144, 65536), (1, 262144, 262144),
]


@pytest.mark.parametrize("num_class", [1, 3])
@pytest.mark.parametrize("with_stds", [False, True])
@pytest.mark.parametrize("b,n,k", LARGE_CASES)
def test_large_score_topk_matches_torch(oracle, b, n, k, with_stds, num_class):
    from spsnet_b200 import pointnet2_utils as pu

    cls, stds = scene_inputs(b, n, k, num_class, seed=n + k)
    st = stds if with_stds else None
    cls_d, st_d = dev(cls), (dev(st) if with_stds else None)
    idx, sc = pu.score_topk(cls_d, k, stds=st_d, return_scores=True)
    check_against_torch(idx, sc, cls_d, st_d, k)
    want_idx, _ = oracle.score_topk(cls, k, st)
    assert oracle.same_topk(idx.cpu().numpy(), want_idx, oracle.topk_scores(cls, st))


@pytest.mark.parametrize("b,n,k", [(2, 40000, 40000), (1, 262144, 65536)])
def test_large_score_topk_all_equal_scores(b, n, k):
    from spsnet_b200 import pointnet2_utils as pu

    idx = pu.score_topk(torch.zeros(b, n, 3, device="cuda"), k)
    assert torch.equal(idx, torch.arange(k, dtype=torch.int32, device="cuda").expand(b, k))


def test_large_score_topk_nan_ranks_first():
    """torch.max propagates NaN and a descending sort puts NaN first; NaNs in several CTA slices come first, by index."""
    from spsnet_b200 import pointnet2_utils as pu

    n, k = 100000, 3000
    cls = scenes.make_cls_logits(31, 2, n)
    nans = [[5, 17000, 49151, 49152, 99999], [16383, 16384, 65536, 70000]]
    for bb, pos in enumerate(nans):
        for j, p in enumerate(pos):
            cls[bb, p, j % 3] = np.nan
    for with_stds in (False, True):
        st_d = dev(scenes.make_stds(32, 2, n)) if with_stds else None
        cls_d = dev(cls)
        idx, sc = pu.score_topk(cls_d, k, stds=st_d, return_scores=True)
        for bb, pos in enumerate(nans):
            assert idx[bb, :len(pos)].tolist() == sorted(pos)
            assert torch.isnan(sc[bb, :len(pos)]).all() and not torch.isnan(sc[bb, len(pos):]).any()
        check_against_torch(idx, sc, cls_d, st_d, k)


def test_single_cta_and_cluster_kernels_agree():
    """A scene of 16384 points (single-CTA kernel) and the same scene with one more point of the lowest score (2-CTA
    cluster kernel) give the same picks."""
    from spsnet_b200 import pointnet2_utils as pu

    cls, stds = scene_inputs(2, CTA_KEYS, 4096, 3, seed=77)
    cls1 = np.concatenate([cls, np.full((2, 1, 3), -1000.0, np.float32)], axis=1)   # sigmoid(-1000) == 0.0f
    stds1 = np.concatenate([stds, np.ones((2, 1), np.float32)], axis=1)
    for k in (4096, CTA_KEYS):
        for st, st1 in ((None, None), (stds, stds1)):
            a = pu.score_topk(dev(cls), k, stds=dev(st) if st is not None else None)
            b = pu.score_topk(dev(cls1), k, stds=dev(st1) if st1 is not None else None)
            assert torch.equal(a, b)


def test_large_score_topk_is_one_launch_and_deterministic():
    from spsnet_b200 import _lib
    from spsnet_b200 import pointnet2_utils as pu

    cls = dev(scenes.make_cls_logits(41, 2, 200000))
    stds = dev(scenes.make_stds(42, 2, 200000))
    pu.score_topk(cls, 50000, stds=stds)
    torch.cuda.synchronize()
    n0 = _lib.lib.spsk_launch_count()
    a = pu.score_topk(cls, 50000, stds=stds)
    assert _lib.lib.spsk_launch_count() - n0 == 1
    b = pu.score_topk(cls, 50000, stds=stds)
    assert torch.equal(a, b)


@pytest.mark.parametrize("n,k", [(65536, 16384), (262144, 65536)])
def test_large_score_topk_cuda_graph(n, k):
    from spsnet_b200 import pointnet2_utils as pu

    b = 2
    static_cls = dev(scenes.make_cls_logits(50, b, n))
    static_stds = dev(scenes.make_stds(51, b, n))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):   # warm-up outside the capture (function attributes, cluster check)
        pu.score_topk(static_cls, k, stds=static_stds)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = pu.score_topk(static_cls, k, stds=static_stds)
    for seed in (52, 54):
        cls, stds = dev(scenes.make_cls_logits(seed, b, n)), dev(scenes.make_stds(seed + 1, b, n))
        static_cls.copy_(cls)
        static_stds.copy_(stds)
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, pu.score_topk(cls, k, stds=stds))


def test_large_score_topk_opcheck():
    import spsnet_b200.torch_ops  # noqa: F401  (registers torch.ops.spsk)

    cls = dev(scenes.make_cls_logits(60, 2, 65536))
    assert torch.equal(torch.ops.spsk.score_topk(cls, 16384), stable_topk(torch_scores(cls), 16384)[0])
    torch.library.opcheck(torch.ops.spsk.score_topk.default, (cls, 16384),
                          test_utils=("test_schema", "test_faketensor", "test_autograd_registration"))


# ---- PointnetSAModuleMSG_WithSampling on large score-sampled inputs ---------------------------------------------------------
MODULES = {
    "ctr": dict(npoint_list=[4096], sample_type_list=["ctr_aware"], radii=[0.8, 1.6], nsamples=[16, 32],
                mlps=[[8, 16, 32], [8, 16, 32]], aggregation_mlp=[32], confidence_mlp=[16]),
    "sss": dict(npoint_list=[4096], sample_type_list=["sss_aware"], radii=[0.8, 1.6], nsamples=[16, 32],
                mlps=[[8, 16, 32], [8, 16, 32]], aggregation_mlp=[32], confidence_mlp=[16]),
    "gather": dict(npoint_list=[16384], sample_type_list=["ctr_aware"], radii=[], nsamples=[], mlps=[],
                   aggregation_mlp=[32], confidence_mlp=None),
}


def _module(kind, impl=None):
    from spsnet_b200 import backbone as bb
    from spsnet_b200 import pointnet2_modules as pm

    torch.manual_seed(8)
    m = (impl or pm).PointnetSAModuleMSG_WithSampling(sample_range_list=[-1], num_class=3, **copy.deepcopy(MODULES[kind]))
    bb.randomize_bn_stats(m, seed=8)
    return m.eval()


@pytest.mark.parametrize("kind,n", [("ctr", 32768), ("sss", 32768), ("gather", 65536)])
def test_sa_module_samples_large_scenes(oracle, ref_ops, kind, n):
    B, cin = 2, 8
    m = _module(kind)
    rng = np.random.default_rng(9)
    xyz = np.ascontiguousarray(scenes.make_batch(44, B, n)[:, :, :3])
    feats = rng.standard_normal((B, cin, n)).astype(np.float32)
    cls = scenes.make_cls_logits(45, B, n)
    stds = scenes.make_stds(46, B, n) if kind == "sss" else None
    kw = {"stds": dev(stds).view(B, 1, n)} if stds is not None else {}
    mg = copy.deepcopy(m).cuda()
    with torch.no_grad():
        got = mg(dev(xyz), dev(feats), dev(cls), **kw)
    npoint = MODULES[kind]["npoint_list"][0]
    want_idx, _ = stable_topk(torch_scores(dev(cls), dev(stds) if stds is not None else None), npoint)
    assert torch.equal(got[3], want_idx), "sampled indices differ from torch's stable descending sort"
    want = oracle.sa_forward(m, xyz, feats, cls, stds=stds, forced_idx=want_idx.cpu().numpy())
    np.testing.assert_array_equal(got[0].cpu().numpy(), want[0])
    assert_close(got[1].cpu().numpy(), want[1], what=f"{kind} new_features")
    if want[2] is not None:
        assert_close(got[2].cpu().numpy(), want[2], what=f"{kind} cls_features")
    if stds is not None:
        np.testing.assert_array_equal(got[4].cpu().numpy().reshape(B, -1), np.take_along_axis(stds, want[3].astype(np.int64), 1))
    if ref_ops is None or stds is not None:
        return
    ref = _module(kind, impl=ref_ops.modules).cuda()
    ref.load_state_dict(mg.state_dict())
    with torch.no_grad():
        r = ref(dev(xyz), dev(feats), dev(cls))
    # torch.topk leaves the order of equal scores unspecified: the picks agree up to exact ties
    scores = torch_scores(dev(cls)).cpu().numpy()
    assert oracle.same_topk(got[3].cpu().numpy(), r[3].cpu().numpy(), scores, ulps=0, atol=0.0)
    if torch.equal(got[3], r[3].int()):
        np.testing.assert_array_equal(got[0].cpu().numpy(), r[0].cpu().numpy())
        assert_close(got[1].cpu().numpy(), r[1].cpu().numpy(), what=f"{kind} new_features vs reference")
