"""-m gpu parity tests of the native ops: candidate (libspsk.so through the C-ABI) vs the C oracle, vs the recorded outputs
of the reference's own CUDA ops, and vs those ops themselves (oracle/_ref) when that module is present.  Indices / copies:
bit-exact."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from spsnet_b200 import scenes  # noqa: E402


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _xyz(b, n, seed=0, kind="kitti"):
    return np.ascontiguousarray(scenes.make_batch(seed, b, n, kind)[:, :, :3])


FPS_CASES = [  # (b, n, m)
    (2, 1, 1), (1, 7, 5), (2, 33, 20), (3, 100, 64), (2, 1000, 300), (2, 1024, 512), (2, 1500, 700),
    (4, 4096, 1024), (2, 5000, 1200), (2, 8192, 2048), (2, 12000, 3000), (4, 16384, 4096),
]


@pytest.mark.parametrize("b,n,m", FPS_CASES)
def test_fps_vs_oracle(oracle, ref_ops, b, n, m):
    from spsnet_b200 import pointnet2_utils as pu

    xyz = _xyz(b, n, seed=n)
    got = pu.furthest_point_sample(dev(xyz), m).cpu().numpy()
    want = oracle.fps(xyz, m)
    assert got.dtype == np.int32 and got.shape == (b, m)
    np.testing.assert_array_equal(got, want)
    if ref_ops is not None:
        ref = ref_ops.utils.furthest_point_sample(dev(xyz), m).cpu().numpy()
        np.testing.assert_array_equal(ref, want, err_msg="ORACLE disagrees with the reference CUDA op")


def test_ops_vs_recorded_reference_ops():
    """The reference's own CUDA ops as recorded on a B200 (tests/golden/reference_ops_b200.npz, made by
    tests/golden/make_golden.py; tests/test_oracle_cpu.py holds the oracle to the same file): FPS, F-FPS, ball query
    (plain and dilated), three_nn and three_interpolate on the same seeded inputs, bit-exact."""
    import importlib.util
    from pathlib import Path

    from spsnet_b200 import pointnet2_utils as pu

    spec = importlib.util.spec_from_file_location("make_golden", Path(__file__).parent / "golden" / "make_golden.py")
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)
    g = np.load(Path(__file__).parent / "golden" / "reference_ops_b200.npz")
    for b, n, m, seed in mg.FPS_CASES:
        np.testing.assert_array_equal(pu.furthest_point_sample(dev(mg.case_xyz(b, n, seed)), m).cpu().numpy(), g[f"fps_{b}_{n}_{m}"])
        np.testing.assert_array_equal(pu.furthest_point_sample(dev(mg.lattice_xyz(b, n, seed)), m).cpu().numpy(), g[f"fpslat_{b}_{n}_{m}"])
    f = np.random.default_rng(99).standard_normal((2, 600, 6)).astype(np.float32)
    d = ((f[:, :, None, :] - f[:, None, :, :]) ** 2).sum(-1).astype(np.float32)
    np.testing.assert_array_equal(pu.furthest_point_sample_with_dist(dev(d), 200).cpu().numpy(), g["fpsdist_2_600_200"])
    for b, n, m, r, ns, seed in mg.BQ_CASES:
        xyz = mg.case_xyz(b, n, seed)
        c = mg.centres_for(xyz, m, seed)
        key = f"{b}_{n}_{m}_{r}_{ns}"
        np.testing.assert_array_equal(pu.ball_query(r, ns, dev(xyz), dev(c)).cpu().numpy(), g[f"bq_{key}"])
        np.testing.assert_array_equal(pu.ball_query_dilated(r, 0.0, ns, dev(xyz), dev(c)).cpu().numpy(), g[f"bqd_{key}"])
        np.testing.assert_array_equal(pu.ball_query_dilated(r, r * 0.5, ns, dev(xyz), dev(c)).cpu().numpy(), g[f"bqd2_{key}"])
    for b, n, m, c, seed in mg.NN_CASES:
        unknown = mg.case_xyz(b, n, seed)
        known = mg.case_xyz(b, m, seed + 100)
        known[:, 3] = known[:, 1]
        dist, idx = pu.three_nn(dev(unknown), dev(known))
        np.testing.assert_array_equal(idx.cpu().numpy(), g[f"nn_idx_{b}_{n}_{m}"])
        np.testing.assert_array_equal(dist.cpu().numpy(), g[f"nn_dist_{b}_{n}_{m}"])
        feats = np.random.default_rng(seed).standard_normal((b, c, m)).astype(np.float32)
        w = np.random.default_rng(seed + 1).uniform(0, 1, (b, n, 3)).astype(np.float32)
        np.testing.assert_array_equal(pu.three_interpolate(dev(feats), idx, dev(w)).cpu().numpy(), g[f"interp_{b}_{n}_{m}"])


def test_fps_ties_grid(oracle, ref_ops):
    """Integer lattice + many duplicates: every step is a massive tie -> checks the block-tree tie-break."""
    from spsnet_b200 import pointnet2_utils as pu

    rng = np.random.default_rng(5)
    for n, m in [(3000, 200), (16384, 600), (700, 300)]:
        xyz = rng.integers(0, 6, (2, n, 3)).astype(np.float32)
        got = pu.furthest_point_sample(dev(xyz), m).cpu().numpy()
        np.testing.assert_array_equal(got, oracle.fps(xyz, m))
        if ref_ops is not None:
            np.testing.assert_array_equal(ref_ops.utils.furthest_point_sample(dev(xyz), m).cpu().numpy(), got)


@pytest.mark.parametrize("b,n,m,kind", [(2, 16385, 300, "kitti"), (2, 20000, 500, "waymo"), (2, 65536, 1500, "waymo"),
                                        (1, 131072, 200, "waymo"), (3, 40001, 257, "waymo")])
def test_fps_cluster_vs_oracle(oracle, ref_ops, b, n, m, kind):
    """n > 16384: one 8-CTA cluster per scene with a DSMEM arg-max (Waymo-shaped scenes) -- same samples, bit-exact."""
    from spsnet_b200 import pointnet2_utils as pu

    xyz = _xyz(b, n, seed=n, kind=kind)
    got = pu.furthest_point_sample(dev(xyz), m).cpu().numpy()
    want = oracle.fps(xyz, m)
    np.testing.assert_array_equal(got, want)
    if ref_ops is not None and n <= 65536:
        np.testing.assert_array_equal(ref_ops.utils.furthest_point_sample(dev(xyz), m).cpu().numpy(), want)


def test_fps_cluster_ties(oracle):
    """Lattice points spread over the 8 CTAs of a cluster: the tie-break key must hold across CTAs."""
    from spsnet_b200 import pointnet2_utils as pu

    rng = np.random.default_rng(9)
    xyz = rng.integers(0, 7, (2, 40000, 3)).astype(np.float32)
    got = pu.furthest_point_sample(dev(xyz), 400).cpu().numpy()
    np.testing.assert_array_equal(got, oracle.fps(xyz, 400))


@pytest.mark.parametrize("b,n,m", [(1, 140000, 120), (2, 200000, 300), (1, 262144, 150)])
def test_fps_16cta_cluster(oracle, b, n, m):
    """131072 < n <= 262144: one 16-CTA cluster per scene (non-portable cluster size; the streaming kernel takes over where
    the device cannot co-schedule it) -- same samples, also with lattice ties across all 16 CTAs."""
    from spsnet_b200 import pointnet2_utils as pu

    xyz = _xyz(b, n, seed=3, kind="waymo")
    got = pu.furthest_point_sample(dev(xyz), m).cpu().numpy()
    np.testing.assert_array_equal(got, oracle.fps(xyz, m))
    lat = np.random.default_rng(n).integers(0, 9, (1, n, 3)).astype(np.float32)
    np.testing.assert_array_equal(pu.furthest_point_sample(dev(lat), 200).cpu().numpy(), oracle.fps(lat, 200))


def test_fps_large_n_generic(oracle):
    """n > 262144: running minima in the caller-provided `temp` scratch (L2), same samples."""
    from spsnet_b200 import pointnet2_utils as pu

    xyz = _xyz(1, 270000, seed=3, kind="waymo")
    got = pu.furthest_point_sample(dev(xyz), 60).cpu().numpy()
    np.testing.assert_array_equal(got, oracle.fps(xyz, 60))


@pytest.mark.parametrize("b,n,m", [(2, 64, 20), (2, 1000, 128), (1, 2048, 512)])
def test_fps_with_dist(oracle, ref_ops, b, n, m):
    from spsnet_b200 import pointnet2_utils as pu

    rng = np.random.default_rng(n)
    f = rng.standard_normal((b, n, 6)).astype(np.float32)
    d = ((f[:, :, None, :] - f[:, None, :, :]) ** 2).sum(-1).astype(np.float32)
    got = pu.furthest_point_sample_with_dist(dev(d), m).cpu().numpy()
    np.testing.assert_array_equal(got, oracle.fps_with_dist(d, m))
    if ref_ops is not None:
        np.testing.assert_array_equal(ref_ops.utils.furthest_point_sample_with_dist(dev(d), m).cpu().numpy(), got)


BQ_CASES = [  # (b, n, m, radius, nsample)
    (2, 100, 10, 5.0, 8), (2, 1000, 77, 2.0, 16), (2, 4096, 1024, 0.8, 16), (2, 4096, 1024, 1.6, 32),
    (2, 16384, 512, 0.2, 16), (1, 16384, 300, 0.8, 32), (2, 1024, 512, 4.8, 32), (2, 3000, 100, 0.01, 16),
    (1, 2000, 50, 1000.0, 64), (1, 50, 20, 3.0, 40),
]


@pytest.mark.parametrize("b,n,m,radius,nsample", BQ_CASES)
def test_ball_query(oracle, ref_ops, b, n, m, radius, nsample):
    from spsnet_b200 import pointnet2_utils as pu

    xyz = _xyz(b, n, seed=7 + n)
    sel = oracle.fps(xyz, m)
    new_xyz = np.ascontiguousarray(np.take_along_axis(xyz, sel[..., None].astype(np.int64), axis=1))
    new_xyz[:, -1] += 500.0  # a centre with an empty ball -> untouched (zero) row
    got = pu.ball_query(radius, nsample, dev(xyz), dev(new_xyz)).cpu().numpy()
    want = oracle.ball_query(radius, nsample, xyz, new_xyz)
    np.testing.assert_array_equal(got, want)
    if ref_ops is not None:
        np.testing.assert_array_equal(ref_ops.utils.ball_query(radius, nsample, dev(xyz), dev(new_xyz)).cpu().numpy(), want)


def test_ball_query_msg_equals_separate(oracle):
    from spsnet_b200 import pointnet2_utils as pu

    xyz = _xyz(2, 4096, seed=11)
    sel = oracle.fps(xyz, 512)
    new_xyz = np.ascontiguousarray(np.take_along_axis(xyz, sel[..., None].astype(np.int64), axis=1))
    new_xyz[:, 5] -= 300.0
    radii, ns = [0.2, 0.8, 3.0], [16, 32, 48]
    outs = pu.ball_query_msg(radii, ns, dev(xyz), dev(new_xyz))
    for r, s, o in zip(radii, ns, outs):
        np.testing.assert_array_equal(o.cpu().numpy(), oracle.ball_query(r, s, xyz, new_xyz))


@pytest.mark.parametrize("rmax,rmin", [(0.8, 0.0), (1.6, 0.8), (4.8, 1.6)])
def test_ball_query_dilated(oracle, ref_ops, rmax, rmin):
    from spsnet_b200 import pointnet2_utils as pu

    xyz = _xyz(2, 3000, seed=13)
    sel = oracle.fps(xyz, 200)
    new_xyz = np.ascontiguousarray(np.take_along_axis(xyz, sel[..., None].astype(np.int64), axis=1))
    got = pu.ball_query_dilated(rmax, rmin, 16, dev(xyz), dev(new_xyz)).cpu().numpy()
    want = oracle.ball_query_dilated(rmax, rmin, 16, xyz, new_xyz)
    np.testing.assert_array_equal(got, want)
    if ref_ops is not None:
        np.testing.assert_array_equal(ref_ops.utils.ball_query_dilated(rmax, rmin, 16, dev(xyz), dev(new_xyz)).cpu().numpy(), want)


def test_gather_group(oracle, ref_ops):
    from spsnet_b200 import pointnet2_utils as pu

    rng = np.random.default_rng(0)
    for b, c, n, m, s in [(2, 3, 100, 17, 5), (2, 64, 4096, 1024, 32), (1, 1, 16384, 4096, 16), (3, 13, 777, 300, 7)]:
        f = rng.standard_normal((b, c, n)).astype(np.float32)
        i1 = rng.integers(0, n, (b, m)).astype(np.int32)
        i2 = rng.integers(0, n, (b, m, s)).astype(np.int32)
        np.testing.assert_array_equal(pu.gather_operation(dev(f), dev(i1)).cpu().numpy(), oracle.gather(f, i1))
        np.testing.assert_array_equal(pu.grouping_operation(dev(f), dev(i2)).cpu().numpy(), oracle.group(f, i2))
        pts = np.ascontiguousarray(np.transpose(f, (0, 2, 1)))
        np.testing.assert_array_equal(pu.gather_rows(dev(pts), dev(i1)).cpu().numpy(),
                                      np.take_along_axis(pts, i1[..., None].astype(np.int64), axis=1))
        if ref_ops is not None:
            np.testing.assert_array_equal(ref_ops.utils.gather_operation(dev(f), dev(i1)).cpu().numpy(), oracle.gather(f, i1))
            np.testing.assert_array_equal(ref_ops.utils.grouping_operation(dev(f), dev(i2)).cpu().numpy(), oracle.group(f, i2))


def test_gather_group_backward(oracle):
    from spsnet_b200 import pointnet2_utils as pu

    rng = np.random.default_rng(1)
    b, c, n, m, s = 2, 8, 300, 64, 9
    f = torch.from_numpy(rng.standard_normal((b, c, n)).astype(np.float32)).cuda().requires_grad_(True)
    i1 = rng.integers(0, n, (b, m)).astype(np.int32)
    i2 = rng.integers(0, n, (b, m, s)).astype(np.int32)
    g1 = rng.standard_normal((b, c, m)).astype(np.float32)
    g2 = rng.standard_normal((b, c, m, s)).astype(np.float32)
    pu.gather_operation(f, dev(i1)).backward(dev(g1))
    np.testing.assert_allclose(f.grad.cpu().numpy(), oracle.gather_grad(g1, i1, n), rtol=1e-5, atol=1e-5)
    f.grad = None
    pu.grouping_operation(f, dev(i2)).backward(dev(g2))
    np.testing.assert_allclose(f.grad.cpu().numpy(), oracle.group_grad(g2, i2, n), rtol=1e-5, atol=1e-5)


def test_three_nn_interpolate(oracle, ref_ops):
    from spsnet_b200 import pointnet2_utils as pu

    rng = np.random.default_rng(2)
    for b, n, m, c in [(2, 1000, 256, 16), (1, 4096, 1024, 5), (2, 50, 2, 3), (1, 300, 2500, 4)]:
        unknown = _xyz(b, n, seed=21)
        known = np.ascontiguousarray(_xyz(b, max(m, 4), seed=22)[:, :m])
        if m >= 8:
            known[:, 3] = known[:, 1]  # exact duplicate -> tie on distance, first index must win
        d2, idx = oracle.three_nn(unknown, known)
        gd, gi = pu.three_nn(dev(unknown), dev(known))
        np.testing.assert_array_equal(gi.cpu().numpy(), idx)
        np.testing.assert_array_equal(gd.cpu().numpy(), np.sqrt(d2))
        feats = rng.standard_normal((b, c, m)).astype(np.float32)
        w = rng.uniform(0, 1, (b, n, 3)).astype(np.float32)
        got = pu.three_interpolate(dev(feats), dev(idx), dev(w)).cpu().numpy()
        np.testing.assert_array_equal(got, oracle.three_interpolate(feats, idx, w))
        if ref_ops is not None:
            rd, ri = ref_ops.utils.three_nn(dev(unknown), dev(known))
            np.testing.assert_array_equal(ri.cpu().numpy(), idx)
            np.testing.assert_array_equal(rd.cpu().numpy(), np.sqrt(d2))
            np.testing.assert_array_equal(ref_ops.utils.three_interpolate(dev(feats), dev(idx), dev(w)).cpu().numpy(), got)
        # backward
        ft = dev(feats).requires_grad_(True)
        g = rng.standard_normal((b, c, n)).astype(np.float32)
        pu.three_interpolate(ft, dev(idx), dev(w)).backward(dev(g))
        np.testing.assert_allclose(ft.grad.cpu().numpy(), oracle.three_interpolate_grad(g, idx, w, m), rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize("b,n,k", [(2, 1024, 512), (4, 512, 256), (2, 4096, 2048), (1, 1000, 333), (2, 16384, 4096)])
def test_score_topk(oracle, b, n, k):
    from spsnet_b200 import pointnet2_utils as pu

    cls = scenes.make_cls_logits(n, b, n)
    cls[:, : n // 8] = np.round(cls[:, : n // 8])          # exact ties
    cls[:, n // 8: n // 6, :] = 30.0                       # saturated sigmoid == 1.0f
    stds = scenes.make_stds(n + 1, b, n)
    for st in (None, stds):
        idx, sc = pu.score_topk(dev(cls), k, stds=dev(st) if st is not None else None, return_scores=True)
        idx, sc = idx.cpu().numpy(), sc.cpu().numpy()
        want_idx, _ = oracle.score_topk(cls, k, st)
        full = oracle.topk_scores(cls, st)
        assert oracle.same_topk(idx, want_idx, full), "top-k differs from the oracle beyond near-ties"
        # internal consistency: scores descending, ties by ascending index, scores match torch's formula on device
        assert np.all(np.diff(sc, axis=1) <= 0)
        tie = np.diff(sc, axis=1) == 0
        assert np.all(np.diff(idx, axis=1)[tie] > 0)
        t = torch.sigmoid(dev(cls).max(dim=-1)[0])
        if st is not None:
            t = t * (1 - torch.sigmoid(dev(st) / 8 - 3))
        tv, ti = torch.topk(t, k, dim=-1)
        np.testing.assert_array_equal(sc, tv.cpu().numpy())  # same score bits as torch's op chain
        mism = ti.int().cpu().numpy() != idx
        if mism.any():  # only inside groups of exactly equal scores
            tt = t.cpu().numpy()
            for bb, jj in zip(*np.nonzero(mism)):
                assert tt[bb, ti[bb, jj]] == tt[bb, idx[bb, jj]]


def test_fps_pruned_equals_dense(oracle, monkeypatch):
    """The Morton-pruned kernel and the dense kernel return identical indices (and both equal the oracle)."""
    from spsnet_b200 import pointnet2_utils as pu

    rng = np.random.default_rng(17)
    cases = [(_xyz(2, 16384, seed=31), 4096), (_xyz(3, 4096, seed=32), 1024), (_xyz(2, 3000, seed=33), 2999),
             (rng.integers(0, 4, (2, 9000, 3)).astype(np.float32), 500),          # massive ties
             (np.ascontiguousarray(_xyz(1, 8192, seed=34, kind="waymo")), 2048),
             (np.zeros((1, 2048, 3), np.float32), 64)]                              # all points identical
    for xyz, m in cases:
        monkeypatch.setenv("SPSK_FPS", "dense")
        a = pu.furthest_point_sample(dev(xyz), m).cpu().numpy()
        monkeypatch.delenv("SPSK_FPS")
        b = pu.furthest_point_sample(dev(xyz), m).cpu().numpy()
        np.testing.assert_array_equal(a, b)
        np.testing.assert_array_equal(b, oracle.fps(xyz, m))


@pytest.mark.parametrize("b,n,m,radii,ns", [
    (2, 16384, 1024, [0.2, 0.8], [16, 32]), (2, 4096, 700, [0.8, 1.6], [16, 32]), (1, 2048, 300, [1.6, 4.8], [16, 32]),
    (2, 5000, 333, [0.05], [8]), (1, 3000, 64, [1000.0, 2.0, 0.5], [64, 32, 4]), (1, 65536, 512, [0.4, 1.0], [16, 32]),
])
def test_ball_query_grid_equals_bruteforce(oracle, b, n, m, radii, ns):
    """Grid kernel == brute-force kernel == oracle, incl. centres far outside the scene (empty rows), duplicates,
    a radius larger than the scene, and lattice data where many points sit exactly on cell borders."""
    from spsnet_b200 import pointnet2_utils as pu

    kind = "waymo" if n > 16384 else "kitti"
    xyz = _xyz(b, n, seed=50 + n, kind=kind)
    rng = np.random.default_rng(n)
    sel = np.stack([rng.choice(n, m, replace=False) for _ in range(b)])
    new_xyz = np.ascontiguousarray(np.take_along_axis(xyz, sel[..., None], axis=1))
    new_xyz[:, 0] += 500.0
    new_xyz[:, 1] -= 0.3           # off-point centres
    new_xyz[:, 2, 1] += 2000.0
    g = pu.ball_query_msg(radii, ns, dev(xyz), dev(new_xyz), grid=True)
    bf = pu.ball_query_msg(radii, ns, dev(xyz), dev(new_xyz), grid=False)
    for r, s, a, c in zip(radii, ns, g, bf):
        np.testing.assert_array_equal(a.cpu().numpy(), c.cpu().numpy())
        if n <= 16384:
            np.testing.assert_array_equal(a.cpu().numpy(), oracle.ball_query(r, s, xyz, new_xyz))
    # lattice: coordinates are exact multiples of the cell edge candidates
    lat = rng.integers(0, 40, (1, 4096, 3)).astype(np.float32) * np.float32(0.25)
    ctr = np.ascontiguousarray(lat[:, :256])
    a = pu.ball_query_msg([0.5, 1.0], [16, 32], dev(lat), dev(ctr), grid=True)
    for r, s, o in zip([0.5, 1.0], [16, 32], a):
        np.testing.assert_array_equal(o.cpu().numpy(), oracle.ball_query(r, s, lat, ctr))


@pytest.mark.parametrize("n,m,sigma", [(4096, 4096, 0.3), (16384, 2048, 0.5), (3000, 700, 0.05), (8192, 1024, 2.0)])
def test_ball_query_grid_dense_scenes(oracle, n, m, sigma):
    """Dense scenes (thousands of candidates per 3 x 3 neighbourhood, e.g. the feature-space queries of SPSNet's
    DenseEdgeConv) take the index-order prefix scan inside the grid kernel: same lists as the brute-force kernel and the
    oracle, also for centres that stay sparse (prefix finds too few, the grid finishes) and for mixed scenes in one batch."""
    from spsnet_b200 import pointnet2_utils as pu

    rng = np.random.default_rng(n + m)
    dense = rng.normal(0.0, sigma, (1, n, 3)).astype(np.float32)
    dense[0, n // 2:, :] = np.maximum(dense[0, n // 2:, :], 0.0)       # ReLU-like: many exact zeros / duplicates
    mixed = dense.copy()
    mixed[0, : n // 8] = rng.uniform(-60, 60, (n // 8, 3)).astype(np.float32)   # sparse outliers, also inside the prefix
    sparse = _xyz(1, n, seed=9, kind="kitti")
    xyz = np.concatenate([dense, mixed, sparse], axis=0)
    sel = rng.choice(n, m, replace=False)
    new_xyz = np.ascontiguousarray(xyz[:, sel])
    radii, ns = [0.8, 0.2], [16, 32]
    g = pu.ball_query_msg(radii, ns, dev(xyz), dev(new_xyz), grid=True)
    bf = pu.ball_query_msg(radii, ns, dev(xyz), dev(new_xyz), grid=False)
    for r, s, a, c in zip(radii, ns, g, bf):
        np.testing.assert_array_equal(a.cpu().numpy(), c.cpu().numpy())
        np.testing.assert_array_equal(a.cpu().numpy(), oracle.ball_query(r, s, xyz, new_xyz))


@pytest.mark.parametrize("b,c,n,npoint,nsample", [(2, 7, 300, 64, 5), (3, 64, 4096, 1024, 32), (1, 5, 50, 200, 16), (2, 16, 1000, 1, 1)])
def test_deterministic_backward_matches_atomics_and_repeats(oracle, monkeypatch, b, c, n, npoint, nsample):
    """SPSK_DETERMINISTIC_GRAD=1: gather / group / three_interpolate backward through the sorted segment reduction
    (spsk_scatter_grad): equal to the oracle's scatter (reference :46-63, :14-31, :127-149) up to summation order, equal to
    the atomic path, and BIT-identical from run to run (heavily repeated indices included)."""
    from spsnet_b200 import pointnet2_utils as pu

    rng = np.random.default_rng(b * 1000 + n)
    f_np = rng.standard_normal((b, c, n)).astype(np.float32)
    gi = rng.integers(0, n, (b, npoint)).astype(np.int32)
    gi[:, : max(1, npoint // 4)] = 3 % n                    # a hot target: long runs in the segment reduction
    qi = rng.integers(0, n, (b, npoint, nsample)).astype(np.int32)
    qi[:, :, 0] = qi[:, :1, 0]                              # every centre shares one neighbour
    g1 = rng.standard_normal((b, c, npoint)).astype(np.float32)
    g2 = rng.standard_normal((b, c, npoint, nsample)).astype(np.float32)
    ti = rng.integers(0, n, (b, npoint, 3)).astype(np.int32)
    tw = rng.random((b, npoint, 3)).astype(np.float32)

    def grads():
        out = []
        f = dev(f_np).requires_grad_(True)
        pu.gather_operation(f, dev(gi)).backward(dev(g1))
        out.append(f.grad.clone()); f.grad = None
        pu.grouping_operation(f, dev(qi)).backward(dev(g2))
        out.append(f.grad.clone()); f.grad = None
        pu.three_interpolate(f, dev(ti), dev(tw)).backward(dev(g1))
        out.append(f.grad.clone())
        return out

    monkeypatch.delenv("SPSK_DETERMINISTIC_GRAD", raising=False)
    atomic = grads()
    monkeypatch.setenv("SPSK_DETERMINISTIC_GRAD", "1")
    assert pu.deterministic_grads()
    det_a, det_b = grads(), grads()
    want = [oracle.gather_grad(g1, gi, n), oracle.group_grad(g2, qi, n), oracle.three_interpolate_grad(g1, ti, tw, n)]
    for a, d1, d2, w in zip(atomic, det_a, det_b, want):
        assert torch.equal(d1, d2), "the sorted segment reduction must be bit-reproducible"
        scale = max(1.0, float(np.abs(w).max()))
        assert float((d1.cpu() - torch.from_numpy(w)).abs().max()) <= 2e-5 * scale
        assert float((d1 - a).abs().max()) <= 2e-5 * scale


# ---- round-2 regressions (ADVICE.md round 1) -------------------------------------------------------------------------

@pytest.mark.parametrize("n,chunks", [(16384, 1), (65536, 4), (32768, 2)])
def test_fps_top_corner_point_is_not_padding(oracle, ref_ops, n, chunks):
    """A CTA that owns exactly 16384 points has no padding slot; the LAST point of every 16384-point chunk sits in the top
    Morton cell of that chunk (max x, y and z), which used to produce the padding sort key 0xFFFFFFFF and was silently
    dropped.  Such an extreme corner is one of the first picks."""
    from spsnet_b200 import pointnet2_utils as pu

    xyz = _xyz(2, n, seed=77, kind="waymo" if n > 16384 else "kitti")
    per = n // chunks
    top = xyz.max(axis=1)
    for c in range(chunks):
        # strict maximum of its chunk (and of the scene) in all three axes, and a far outlier: FPS must pick every one of them early
        xyz[:, (c + 1) * per - 1] = top + np.float32(100.0 * (c + 1))
    m = 64
    got = pu.furthest_point_sample(dev(xyz), m).cpu().numpy()
    want = oracle.fps(xyz, m)
    np.testing.assert_array_equal(got, want)
    assert (n - 1) in want[0] and (n - 1) in got[0], "the global corner point must be sampled early"
    for c in range(chunks):
        assert ((c + 1) * per - 1) in got[0], f"corner point of chunk {c} was dropped"
    if ref_ops is not None:
        np.testing.assert_array_equal(ref_ops.utils.furthest_point_sample(dev(xyz), m).cpu().numpy(), want)


def test_fps_with_dist_above_16384(oracle, monkeypatch):
    """F-FPS on a distance matrix with 16384 < N <= 131072 (no cluster variant in that mode): the wrapper must hand the
    streaming kernel its `temp` scratch instead of raising; same for D-FPS with the dense kernels forced."""
    from spsnet_b200 import pointnet2_utils as pu

    n, m = 16500, 24
    f = torch.randn(1, n, 4, generator=torch.Generator().manual_seed(3)).cuda()
    d = torch.cdist(f, f).pow(2).contiguous()
    got = pu.furthest_point_sample_with_dist(d, m).cpu().numpy()
    np.testing.assert_array_equal(got, oracle.fps_with_dist(d.cpu().numpy(), m))
    del d
    xyz = _xyz(1, 20000, seed=5, kind="waymo")
    monkeypatch.setenv("SPSK_FPS", "dense")
    a = pu.furthest_point_sample(dev(xyz), 100).cpu().numpy()
    monkeypatch.delenv("SPSK_FPS")
    np.testing.assert_array_equal(a, oracle.fps(xyz, 100))


def test_ball_query_msg_four_scales_large_n_falls_back(oracle):
    """4 scales x 60000 points: the grid kernel's per-warp bitmaps exceed its shared-memory budget -> the automatic choice
    must be the brute-force scan (same lists), not SPSK_ERR_UNSUPPORTED."""
    from spsnet_b200 import pointnet2_utils as pu

    xyz = _xyz(1, 60000, seed=8, kind="waymo")
    new_xyz = np.ascontiguousarray(xyz[:, ::600])
    radii, ns = [0.4, 0.8, 1.6, 3.2], [8, 16, 16, 32]
    outs = pu.ball_query_msg(radii, ns, dev(xyz), dev(new_xyz))
    for r, s, o in zip(radii, ns, outs):
        np.testing.assert_array_equal(o.cpu().numpy(), pu.ball_query(r, s, dev(xyz), dev(new_xyz)).cpu().numpy())


def test_score_topk_nan_ranks_first_like_torch():
    """torch.max propagates NaN and torch.topk ranks NaN first; so does the fused kernel."""
    from spsnet_b200 import pointnet2_utils as pu

    cls = scenes.make_cls_logits(3, 2, 1024)
    cls[0, 17, 1] = np.nan
    cls[1, 900, 0] = np.nan
    cls[1, 5, 2] = np.nan
    idx = pu.score_topk(dev(cls), 256).cpu().numpy()
    t = torch.sigmoid(dev(cls).max(dim=-1)[0])
    ti = torch.topk(t, 256, dim=-1)[1].cpu().numpy()
    assert idx[0, 0] == 17 and set(idx[1, :2]) == {5, 900}
    assert set(ti[0, :1]) == {17} and set(ti[1, :2]) == {5, 900}
    np.testing.assert_array_equal(idx[0, 1:], ti[0, 1:])
    np.testing.assert_array_equal(idx[1, 2:], ti[1, 2:])
