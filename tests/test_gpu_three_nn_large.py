"""-m gpu: three_nn through the grid kernel (n >= THREE_NN_GRID_MIN_N, THREE_NN_GRID_MIN_M <= m <= THREE_NN_GRID_MAX_M).
The reference for every call is the all-pairs kernel itself, reached by calling spsk_three_nn on chunks of fewer than
THREE_NN_GRID_MIN_N unknown points (unknown points are independent, so the chunked result is exact); idx and the bits of
dist2 must match in full.  Sampled rows are checked against the C oracle as well."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from spsnet_b200 import scenes  # noqa: E402


def _pu():
    from spsnet_b200 import pointnet2_utils as pu

    return pu


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).cuda()


def raw_three_nn(unknown, known):
    """(dist2, idx) of spsk_three_nn: squared distances, unlike pu.three_nn, which returns their square roots."""
    from spsnet_b200._lib import check, lib

    B, N, _ = unknown.shape
    dist2 = torch.empty((B, N, 3), dtype=torch.float32, device=unknown.device)
    idx = torch.empty((B, N, 3), dtype=torch.int32, device=unknown.device)
    check(lib.spsk_three_nn(B, N, known.shape[1], unknown.data_ptr(), known.data_ptr(), dist2.data_ptr(), idx.data_ptr(),
                            torch.cuda.current_stream().cuda_stream), "three_nn")
    return dist2, idx


def bruteforce_three_nn(unknown, known):
    """The all-pairs kernel's (dist2, idx), computed on chunks of unknown points below THREE_NN_GRID_MIN_N."""
    step = _pu().THREE_NN_GRID_MIN_N - 1
    parts = [raw_three_nn(unknown[:, i:i + step].contiguous(), known) for i in range(0, unknown.shape[1], step)]
    return torch.cat([p[0] for p in parts], 1), torch.cat([p[1] for p in parts], 1)


def assert_same(got, want, what=""):
    (gd, gi), (wd, wi) = got, want
    gi, wi = gi.cpu().numpy(), wi.cpu().numpy()
    gb, wb = gd.cpu().numpy().view(np.uint32), wd.cpu().numpy().view(np.uint32)
    bad = np.argwhere((gi != wi).any(-1) | (gb != wb).any(-1))
    assert bad.size == 0, f"{what}: {len(bad)} rows differ, first {bad[:3].tolist()}: " \
                          f"{gi[tuple(bad[0])].tolist()} {gd.cpu().numpy()[tuple(bad[0])].tolist()} vs " \
                          f"{wi[tuple(bad[0])].tolist()} {wd.cpu().numpy()[tuple(bad[0])].tolist()}"


def grid_equals_bruteforce(unknown, known, what=""):
    u, k = dev(unknown), dev(known)
    got = raw_three_nn(u, k)
    assert_same(got, bruteforce_three_nn(u, k), what)
    return got


def check_oracle_rows(oracle, unknown, known, got, rows=2048, seed=0):
    """Rows sampled from every scene against the C oracle."""
    rng = np.random.default_rng(seed)
    B, N, _ = unknown.shape
    sel = np.sort(rng.choice(N, min(rows, N), replace=False))
    od, oi = oracle.three_nn(np.ascontiguousarray(unknown[:, sel]), known)
    gd, gi = got[0].cpu().numpy()[:, sel], got[1].cpu().numpy()[:, sel]
    np.testing.assert_array_equal(gi, oi)
    np.testing.assert_array_equal(gd.view(np.uint32), od.view(np.uint32))


def waymo_case(b, n, m, seed, fps=True):
    """Unknown points: every point of Waymo-shaped scenes (3 % duplicates).  Known points: a D-FPS or random subset."""
    xyz = np.ascontiguousarray(scenes.make_batch(seed, b, n, "waymo")[:, :, :3])
    if fps:
        sel = _pu().furthest_point_sample(dev(xyz), m).long().cpu().numpy()
    else:
        rng = np.random.default_rng(seed)
        sel = np.stack([rng.choice(n, m, replace=False) for _ in range(b)])
    known = np.ascontiguousarray(np.take_along_axis(xyz, sel[..., None], axis=1))
    return xyz, known


# cluster sizes 1 / 2 / 4 / 8 / 16 (8192 known points per CTA), with m just above each boundary
@pytest.mark.parametrize("b,n,m,fps", [
    (2, 16384, 4096, True),      # 1 CTA
    (2, 32768, 8192, False),     # 1 CTA, full
    (2, 65536, 8193, True),      # 2 CTAs
    (1, 131072, 16385, False),   # 4 CTAs
    (2, 131072, 32769, True),    # 8 CTAs
    (1, 262144, 65537, False),   # 16 CTAs
    (2, 262144, 131072, False),  # 16 CTAs, full
    (3, 5000, 1500, False),      # a few unknown points per cluster
])
def test_grid_equals_bruteforce(oracle, b, n, m, fps):
    unknown, known = waymo_case(b, n, m, seed=n + m, fps=fps)
    got = grid_equals_bruteforce(unknown, known, f"b={b} n={n} m={m}")
    check_oracle_rows(oracle, unknown, known, got, seed=m)


def test_unknown_subset_of_known_and_far_outside(oracle):
    """Known points that are also unknown points (d = 0, duplicates tie at 0), and unknown points 500 m outside the box."""
    xyz = np.ascontiguousarray(scenes.make_batch(5, 2, 65536, "waymo")[:, :, :3])
    known = np.ascontiguousarray(xyz[:, :20000])
    unknown = xyz.copy()
    unknown[:, :3000, 0] += 500.0
    unknown[:, 3000:4000, 1] -= 500.0
    unknown[:, 4000:4500, :2] += 700.0
    got = grid_equals_bruteforce(unknown, known, "far outside")
    check_oracle_rows(oracle, unknown, known, got, seed=1)
    np.testing.assert_array_equal(oracle.three_nn(unknown[:, :64], known)[1], got[1].cpu().numpy()[:, :64])


# ---- adversarial inputs, all on the grid path ------------------------------------------------------------------------------

def test_lattice_ties_on_cell_borders(oracle):
    """Coordinates on a 0.25 lattice: points on cell borders, exact distance ties broken by the lower id."""
    rng = np.random.default_rng(3)
    n, m = 32768, 16000
    lat = lambda k: np.concatenate([rng.integers(0, 200, (2, k, 2)), rng.integers(0, 8, (2, k, 1))], 2).astype(np.float32) * np.float32(0.25)
    unknown, known = lat(n), lat(m)
    got = grid_equals_bruteforce(unknown, known, "lattice")
    check_oracle_rows(oracle, unknown, known, got, seed=3)


def test_all_known_points_identical():
    pu = _pu()
    m = pu.THREE_NN_GRID_MIN_M + 7
    known = np.full((1, m, 3), 1.5, np.float32)
    rng = np.random.default_rng(4)
    unknown = rng.uniform(-10, 10, (1, pu.THREE_NN_GRID_MIN_N, 3)).astype(np.float32)
    unknown[0, 0] = 1.5
    d, i = grid_equals_bruteforce(unknown, known, "identical")
    assert (i.cpu().numpy() == np.array([0, 1, 2], np.int32)).all()
    assert (d[0, 0] == 0).all()


@pytest.mark.parametrize("axis", ["x", "y", "xy"])
def test_collinear_known_points(oracle, axis):
    """Known points on a line: zero y extent, zero x extent, or a diagonal."""
    rng = np.random.default_rng(5)
    m, n = 20000, 16384
    t = rng.uniform(-40, 40, (2, m)).astype(np.float32)
    known = np.zeros((2, m, 3), np.float32)
    if axis in ("x", "xy"):
        known[..., 0] = t
    if axis in ("y", "xy"):
        known[..., 1] = t
    known[..., 2] = 0.5
    unknown = rng.uniform(-60, 60, (2, n, 3)).astype(np.float32)
    got = grid_equals_bruteforce(unknown, known, f"collinear {axis}")
    check_oracle_rows(oracle, unknown, known, got, seed=5)


@pytest.mark.parametrize("where", ["known", "unknown", "both"])
def test_non_finite_coordinates(where):
    """NaN and +-inf coordinates: in the known points they make the box infinite (one cell, the full scan); in the unknown
    points they make every distance inf or NaN (empty rows).  The known points of scene 1 stay finite."""
    rng = np.random.default_rng(6)
    unknown = rng.uniform(-50, 50, (2, 8192, 3)).astype(np.float32)
    known = rng.uniform(-50, 50, (2, 12000, 3)).astype(np.float32)
    if where in ("known", "both"):
        known[0, 10, 0] = np.nan
        known[0, 11, 1] = np.inf
        known[0, 12, 2] = -np.inf
        known[0, 13] = np.nan
    if where in ("unknown", "both"):
        unknown[:, 5, 0] = np.nan
        unknown[:, 6, 1] = -np.inf
        unknown[:, 7, 2] = np.inf
        unknown[:, 8, 2] = np.nan
    grid_equals_bruteforce(unknown, known, f"non-finite {where}")


def test_nan_only_coordinate_axis_and_huge_box():
    """Every known x NaN except a few; known points 1e30 apart; a known point at +inf in x only in one scene."""
    rng = np.random.default_rng(7)
    unknown = rng.uniform(-50, 50, (3, 4096, 3)).astype(np.float32)
    known = rng.uniform(-50, 50, (3, 2000, 3)).astype(np.float32)
    known[0, 5:, 0] = np.nan
    known[1, :2, :2] = np.float32(1e30)
    known[1, 2, :2] = np.float32(-1e30)
    known[2, 0, 0] = np.inf
    grid_equals_bruteforce(unknown, known, "nan axis / huge box")


# ---- path, launches, graphs, opcheck -----------------------------------------------------------------------------------------

def _kernels_run(fn):
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events() if e.device_type.name == "CUDA"}


def test_path_taken_above_and_below_the_thresholds():
    pu = _pu()
    N, M = pu.THREE_NN_GRID_MIN_N, pu.THREE_NN_GRID_MIN_M
    xyz = dev(scenes.make_batch(8, 1, 2 * N, "waymo")[:, :, :3])
    for n, m, grid in [(N, M, True), (N - 1, M, False), (N, M - 1, False), (2 * N, pu.THREE_NN_GRID_MAX_M + 1, False),
                       (2 * N, pu.THREE_NN_GRID_MAX_M, True)]:
        u = xyz[:, :n].contiguous()
        k = dev(np.random.default_rng(m).uniform(-70, 70, (1, m, 3)))
        names = _kernels_run(lambda: raw_three_nn(u, k))
        assert any("three_nn_cluster_kernel" in s for s in names) == grid, (n, m, names)
        assert any("three_nn_kernel" in s and "cluster" not in s for s in names) == (not grid), (n, m, names)


def test_one_launch_and_cuda_graph():
    from spsnet_b200 import _lib

    b, n, m = 2, 131072, 32768
    unknown, known = waymo_case(b, n, m, seed=40, fps=False)
    su, sk = dev(unknown), dev(known)
    raw_three_nn(su, sk)
    torch.cuda.synchronize()
    n0 = _lib.lib.spsk_launch_count()
    raw_three_nn(su, sk)
    assert _lib.lib.spsk_launch_count() - n0 == 1
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        raw_three_nn(su, sk)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = raw_three_nn(su, sk)
    for seed in (41, 42):
        unknown, known = waymo_case(b, n, m, seed=seed, fps=False)
        su.copy_(dev(unknown))
        sk.copy_(dev(known))
        g.replay()
        torch.cuda.synchronize()
        assert_same(out, raw_three_nn(dev(unknown), dev(known)), f"graph replay {seed}")
        assert_same(out, bruteforce_three_nn(dev(unknown), dev(known)), f"graph replay {seed} vs brute force")


def test_opcheck_above_the_thresholds():
    import spsnet_b200.torch_ops  # noqa: F401

    unknown, known = waymo_case(2, 16384, 4096, seed=50, fps=False)
    u, k = dev(unknown), dev(known)
    d, i = torch.ops.spsk.three_nn(u, k)
    d2, i2 = _pu().three_nn(u, k)
    assert torch.equal(d, d2) and torch.equal(i, i2)
    torch.library.opcheck(torch.ops.spsk.three_nn.default, (u, k),
                          test_utils=("test_schema", "test_faketensor", "test_autograd_registration"))


def test_fp_module_end_to_end(monkeypatch):
    """PointnetFPModule on (2, 262144) <- (2, 65536): torch.equal to the same module built on chunked all-pairs three_nn."""
    from spsnet_b200 import pointnet2_modules as pm

    pu = _pu()
    torch.manual_seed(0)
    fp = pm.PointnetFPModule(mlp=[64 + 32, 64, 64]).cuda().eval()
    unknown, known = waymo_case(2, 262144, 65536, seed=60, fps=False)
    u, k = dev(unknown), dev(known)
    uf = torch.randn(2, 32, 262144, device="cuda")
    kf = torch.randn(2, 64, 65536, device="cuda")
    with torch.no_grad():
        auto = fp(u, k, uf, kf)
    real = pu.three_nn

    def chunked(unknown, known):
        step = pu.THREE_NN_GRID_MIN_N - 1
        parts = [real(unknown[:, i:i + step].contiguous(), known) for i in range(0, unknown.shape[1], step)]
        return torch.cat([p[0] for p in parts], 1), torch.cat([p[1] for p in parts], 1)

    monkeypatch.setattr(pu, "three_nn", chunked)
    with torch.no_grad():
        forced = fp(u, k, uf, kf)
    assert torch.equal(auto, forced)
