"""-m gpu: the grid ball query on scenes of 65536 < n <= 262144 points (and four scales above 32768 points), which walks
the point ids in windows of 65536 (32768 with four scales).  Every list is compared bit for bit with the brute-force
kernel (spsk_ball_query_msg), and where stated with the C oracle: first `nsample` hits in index order, first-hit
padding, zero rows."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from spsnet_b200 import scenes  # noqa: E402


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _xyz(b, n, seed=0, kind="waymo"):
    return np.ascontiguousarray(scenes.make_batch(seed, b, n, kind)[:, :, :3])


def grid_equals_bruteforce(radii, ns, xyz, new_xyz):
    """Lists of the grid kernel, after checking them against the brute-force kernel."""
    from spsnet_b200 import pointnet2_utils as pu

    g = pu.ball_query_msg(radii, ns, dev(xyz), dev(new_xyz), grid=True)
    bf = pu.ball_query_msg(radii, ns, dev(xyz), dev(new_xyz), grid=False)
    out = []
    for r, s, a, c in zip(radii, ns, g, bf):
        a, c = a.cpu().numpy(), c.cpu().numpy()
        np.testing.assert_array_equal(a, c, err_msg=f"grid != brute force at r={r}, nsample={s}, n={xyz.shape[1]}")
        out.append(a)
    return out


def _centres(xyz, m, seed):
    """m centres per scene drawn from the points, with a few far outside the scene (empty rows) and a few off-point."""
    b, n, _ = xyz.shape
    rng = np.random.default_rng(seed)
    sel = np.stack([rng.choice(n, m, replace=False) for _ in range(b)])
    c = np.ascontiguousarray(np.take_along_axis(xyz, sel[..., None], axis=1))
    c[:, 0] += 500.0
    c[:, 1, 1] -= 2000.0
    c[:, 2:10] += np.float32(0.07)
    return c


@pytest.mark.parametrize("b,n,m,radii,ns", [
    (1, 65537, 1024, [0.2], [16]),
    (2, 100000, 2048, [0.2, 0.8], [16, 32]),
    (1, 131072, 4096, [0.8, 1.6, 4.8], [16, 32, 64]),
    (2, 131072, 2048, [1.6, 4.8], [16, 32]),
    (2, 200003, 2048, [0.4, 0.8, 1.6, 3.2], [8, 16, 16, 32]),
    (1, 262144, 4096, [6.4, 1.6], [64, 16]),
    (2, 262144, 8192, [0.2, 0.8], [16, 32]),
    (1, 262144, 512, [1000.0, 0.2, 3.2], [64, 8, 32]),   # a radius larger than the scene
])
def test_large_grid_equals_bruteforce(b, n, m, radii, ns):
    """Waymo-shaped scenes (3 % duplicate points), centres far outside the scene and off-point centres."""
    xyz = _xyz(b, n, seed=n + b)
    new_xyz = _centres(xyz, m, seed=n)
    out = grid_equals_bruteforce(radii, ns, xyz, new_xyz)
    for r, o in zip(radii, out):
        if r < 100.0:
            assert (o[:, 0] == 0).all(), "a centre 500 m outside the scene must give a zero row"


@pytest.mark.parametrize("n,scales", [(100000, 2), (262144, 4)])
def test_large_grid_lattice_on_cell_borders(oracle, n, scales):
    """Coordinates on a 0.25 lattice, so that many points sit exactly on cell borders and at equal distances."""
    rng = np.random.default_rng(n)
    lat = np.concatenate([rng.integers(0, 480, (1, n, 2)), rng.integers(0, 16, (1, n, 1))], axis=2).astype(np.float32) * np.float32(0.25)
    ctr = np.ascontiguousarray(lat[:, rng.choice(n, 512, replace=False)])
    radii, ns = [0.5, 1.0, 0.25, 2.0][:scales], [16, 32, 8, 64][:scales]
    out = grid_equals_bruteforce(radii, ns, lat, ctr)
    for r, s, o in zip(radii[:2], ns[:2], out):
        np.testing.assert_array_equal(o, oracle.ball_query(r, s, lat, ctr))


# ---- window boundaries, built on purpose -----------------------------------------------------------------------------
# Background points fill x in [40, 170] m; each planted centre sits at (3 j, 0, 0) with its hits at the listed ids, 0.01 m
# apart along y, so every centre sees exactly its own planted points inside radius 0.5.
PLANTED = [   # ids are distinct across spots
    [65529, 65532, 65534, 65537, 65540, 131068, 131070, 131073, 131075],   # both sides of 65535/65536 and 131071/131072
    [140000, 150000, 200000],                        # first hit in window 2: padding with an id >= 131072
    [200001, 230000, 262143],                        # first hit in window 3
    [5, 70000, 140001, 250000],                      # fewer than nsample hits, spread over all four windows
    [100, 200, 300, 400, 500, 600, 700, 65536],      # exactly 8 hits, the last one the first id of window 1
    [10, 20, 30, 40, 50, 60, 70, 131072],            # ... of window 2
    [11, 21, 31, 41, 51, 61, 71, 32768],             # ... of the second 32768-id window (four scales)
    list(range(1000, 1020)) + list(range(66000, 66020)),   # more hits than nsample, across a boundary
    [65535, 196608, 196609],                         # the last id of window 0, the first ids of window 3
]


def planted_scene(n, seed, spots):
    rng = np.random.default_rng(seed)
    xyz = np.stack([rng.uniform(40, 170, n), rng.uniform(-75, 75, n), rng.uniform(-2, 4, n)], axis=1).astype(np.float32)
    ctr = []
    for j, ids in enumerate(spots):
        c = np.array([3.0 * j, 0.0, 0.0], np.float32)
        ids = [i for i in ids if i < n]
        for k, i in enumerate(ids):
            xyz[i] = c + np.array([0.0, 0.01 * (k % 20), 0.0], np.float32)
        ctr.append(c)
    return xyz[None], np.stack(ctr)[None].astype(np.float32)


@pytest.mark.parametrize("n", [262144, 200003, 131073])
def test_window_boundaries(oracle, n):
    xyz, ctr = planted_scene(n, seed=n, spots=PLANTED)
    for radii, ns in (([0.5], [8]), ([0.5, 1.0], [16, 32]), ([0.5, 0.3, 1.0, 2.0], [8, 4, 16, 64])):
        out = grid_equals_bruteforce(radii, ns, xyz, ctr)
        for r, s, o in zip(radii, ns, out):
            np.testing.assert_array_equal(o, oracle.ball_query(r, s, xyz, ctr))
    # spot by spot, what the lists must hold (nsample 16, radius 0.5)
    o = grid_equals_bruteforce([0.5], [16], xyz, ctr)[0][0]
    for j, ids in enumerate(PLANTED):
        hits = sorted(i for i in ids if i < n)[:16]
        want = hits + [hits[0]] * (16 - len(hits)) if hits else [0] * 16
        assert o[j].tolist() == want, f"spot {j}"


def test_last_window_holds_one_point(oracle):
    """n = 65537: window 1 holds the single id 65536."""
    n = 65537
    xyz, ctr = planted_scene(n, seed=5, spots=[[65536], [3, 65535], [7, 65534]])
    for radii, ns in (([0.5], [4]), ([0.5, 0.3, 1.0, 2.0], [8, 4, 16, 2])):
        out = grid_equals_bruteforce(radii, ns, xyz, ctr)
        for r, s, o in zip(radii, ns, out):
            np.testing.assert_array_equal(o, oracle.ball_query(r, s, xyz, ctr))
    o = grid_equals_bruteforce([0.5], [4], xyz, ctr)[0][0]
    assert o[0].tolist() == [65536] * 4


@pytest.mark.parametrize("n", [51201, 60000, 65536])
def test_four_scales_take_the_grid_below_65536(n):
    """Four scales above 51200 points: eight warps' bitmaps of 65536 ids do not fit shared memory, so the grid walks two
    windows of 32768 ids; the automatic choice is the grid (two launches), with the brute-force kernel's lists."""
    from spsnet_b200 import _lib
    from spsnet_b200 import pointnet2_utils as pu

    xyz = _xyz(2, n, seed=n)
    new_xyz = _centres(xyz, 2048, seed=n + 1)
    radii, ns = [0.4, 0.8, 1.6, 3.2], [8, 16, 16, 32]
    want = grid_equals_bruteforce(radii, ns, xyz, new_xyz)
    torch.cuda.synchronize()
    n0 = _lib.lib.spsk_launch_count()
    got = pu.ball_query_msg(radii, ns, dev(xyz), dev(new_xyz))
    assert _lib.lib.spsk_launch_count() - n0 == 2
    for a, w in zip(got, want):
        np.testing.assert_array_equal(a.cpu().numpy(), w)


@pytest.mark.parametrize("n,dense", [(131072, 90000), (262144, 150000)])
def test_dense_neighbourhoods_prefix_scan_across_windows(oracle, n, dense):
    """A dense blob of `dense` points spread over all ids: the centres near it have more than BG_PREFIX_MIN candidates, so
    the kernel scans an index-order prefix of about that many points first, ending past a window boundary; the tiny
    radius leaves most of them short of nsample, so the grid phase finishes them above tn.  Sparse centres of the same
    scene and a LiDAR-shaped scene share the batch."""
    rng = np.random.default_rng(n)
    a = np.stack([rng.uniform(-75, 75, n), rng.uniform(-75, 75, n), rng.uniform(-2, 4, n)], axis=1).astype(np.float32)
    pos = rng.choice(n, dense, replace=False)
    a[pos] = rng.normal(0.0, 0.4, (dense, 3)).astype(np.float32)
    a[pos[: dense // 4]] = np.maximum(a[pos[: dense // 4]], 0.0)     # exact zeros and duplicates
    xyz = np.stack([a, _xyz(1, n, seed=3)[0]])
    sel = np.concatenate([pos[:384], rng.choice(n, 128, replace=False)])
    new_xyz = np.ascontiguousarray(xyz[:, sel])
    radii, ns = [0.8, 0.02], [16, 32]
    out = grid_equals_bruteforce(radii, ns, xyz, new_xyz)
    for r, s, o in zip(radii, ns, out):
        np.testing.assert_array_equal(o, oracle.ball_query(r, s, xyz, new_xyz))
    short = (out[1][0, :384] == out[1][0, :384, :1]).sum(-1) > 1
    assert short.any() and (~short).any(), "want centres that fill nsample in the prefix and centres that do not"


def test_large_grid_against_oracle(oracle):
    """The C oracle (independent of both kernels) on a few hundred centres of a 262144-point scene."""
    xyz = _xyz(1, 262144, seed=11)
    new_xyz = _centres(xyz, 300, seed=12)
    from spsnet_b200 import pointnet2_utils as pu

    for radii, ns in (([0.2, 0.8], [16, 32]), ([1.6, 4.8], [16, 32])):
        got = pu.ball_query_msg(radii, ns, dev(xyz), dev(new_xyz))
        for r, s, g in zip(radii, ns, got):
            np.testing.assert_array_equal(g.cpu().numpy(), oracle.ball_query(r, s, xyz, new_xyz))


def test_ball_query_single_radius_takes_the_grid_above_65536():
    """pu.ball_query (QueryAndGroup's query) runs the grid kernel above 65536 points: two launches, the same zero-filled
    lists as the brute-force kernel."""
    from spsnet_b200 import _lib
    from spsnet_b200 import pointnet2_utils as pu

    xyz = _xyz(2, 131072, seed=21)
    new_xyz = _centres(xyz, 4096, seed=22)
    pu.ball_query(0.8, 32, dev(xyz), dev(new_xyz))
    torch.cuda.synchronize()
    n0 = _lib.lib.spsk_launch_count()
    got = pu.ball_query(0.8, 32, dev(xyz), dev(new_xyz))
    assert _lib.lib.spsk_launch_count() - n0 == 2
    want = pu.ball_query_msg([0.8], [32], dev(xyz), dev(new_xyz), grid=False)[0]
    assert torch.equal(got, want)


def test_large_grid_two_launches_and_cuda_graph():
    from spsnet_b200 import _lib
    from spsnet_b200 import pointnet2_utils as pu

    b, n, m = 2, 262144, 8192
    radii, ns = [0.2, 0.8], [16, 32]
    static_xyz = dev(_xyz(b, n, seed=30))
    static_ctr = dev(_centres(static_xyz.cpu().numpy(), m, seed=31))
    pu.ball_query_msg(radii, ns, static_xyz, static_ctr)
    torch.cuda.synchronize()
    n0 = _lib.lib.spsk_launch_count()
    pu.ball_query_msg(radii, ns, static_xyz, static_ctr)
    assert _lib.lib.spsk_launch_count() - n0 == 2
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        pu.ball_query_msg(radii, ns, static_xyz, static_ctr)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        outs = pu.ball_query_msg(radii, ns, static_xyz, static_ctr)
    for seed in (32, 34):
        xyz = _xyz(b, n, seed=seed)
        ctr = _centres(xyz, m, seed=seed + 1)
        static_xyz.copy_(dev(xyz))
        static_ctr.copy_(dev(ctr))
        g.replay()
        torch.cuda.synchronize()
        want = grid_equals_bruteforce(radii, ns, xyz, ctr)
        for o, w in zip(outs, want):
            np.testing.assert_array_equal(o.cpu().numpy(), w)


# ---- the backbone, end to end ---------------------------------------------------------------------------------------------

def _tensors(x, path="out"):
    if isinstance(x, torch.Tensor):
        yield path, x
    elif isinstance(x, dict):
        for k in sorted(x):
            yield from _tensors(x[k], f"{path}.{k}")
    elif isinstance(x, (list, tuple)):
        for i in range(len(x)):
            yield from _tensors(x[i], f"{path}[{i}]")


@pytest.mark.parametrize("b,n", [(2, 131072), (1, 262144)])
def test_waymo_backbone_same_with_grid_and_bruteforce(monkeypatch, b, n):
    """IASSD_Backbone(waymo_iassd_cfg()) in eval mode on Waymo-shaped scenes: the automatic ball query (grid) and the
    brute-force kernel give torch.equal outputs -- sampled points, features, class logits, centres.  Only the ball-query
    kernel differs between the two runs."""
    from helpers import make_backbone
    from spsnet_b200 import backbone as bb
    from spsnet_b200 import pointnet2_utils as pu

    net = make_backbone(bb.waymo_iassd_cfg(), input_channels=5, seed=3).cuda()
    pts = dev(scenes.to_points(scenes.make_batch(40, b, n, "waymo")))

    def run():
        with torch.no_grad():
            out = net({"batch_size": b, "points": pts.clone()})
        return dict(_tensors({k: v for k, v in out.items() if k != "points"}))

    auto = run()
    real = pu.ball_query_msg
    monkeypatch.setattr(pu, "ball_query_msg", lambda *a, **k: real(*a, **{**k, "grid": False}))
    forced = run()
    assert auto.keys() == forced.keys() and len(auto) > 20
    for k in auto:
        assert torch.equal(auto[k], forced[k]), k
