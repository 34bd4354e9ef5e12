"""CPU checks of spsk_ball_query_msg_grid's argument validation for scenes of up to 262144 points: every argument and the
workspace size are checked before any CUDA call, so these run without a GPU."""
import ctypes as C

import pytest

FAKE = 0x1000   # a non-null device address that is never dereferenced: every call below returns before any CUDA call


def _args(nscales=2, idx_null=False):
    r = (C.c_float * nscales)(*([0.8] * nscales))
    ns = (C.c_int * nscales)(*([16] * nscales))
    idx = (C.c_void_p * nscales)(*([None if idx_null else FAKE] * nscales))
    return r, ns, idx


def parent_workspace_bytes(b, n):
    """The formula of spsk_ball_query_grid_workspace_bytes when the grid query took at most 65536 points:
    GridParams (32 B) per scene, one cell_start array of 11265 ints per scene, one float4 per point, 256 B of slack."""
    return 32 * b + 4 * b * 11265 + 16 * b * n + 256


def test_ball_query_grid_rejects_more_than_262144_points():
    from spsnet_b200 import _lib

    lib = _lib.lib
    r, ns, idx = _args()
    assert lib.spsk_ball_query_msg_grid(1, 262145, 64, 2, r, ns, None, None, idx, None, 0, None) == -2
    assert b"262144" in lib.spsk_last_error()


def test_ball_query_grid_checks_pointers_and_workspace_before_any_cuda_call():
    from spsnet_b200 import _lib

    lib = _lib.lib
    n, b, m = 262144, 2, 4096
    need = int(lib.spsk_ball_query_grid_workspace_bytes(b, n))
    r, ns, idx = _args()
    assert lib.spsk_ball_query_msg_grid(b, n, m, 2, r, ns, None, FAKE, idx, FAKE, need, None) == -1
    assert b"null" in lib.spsk_last_error()
    assert lib.spsk_ball_query_msg_grid(b, n, m, 2, None, ns, FAKE, FAKE, idx, FAKE, need, None) == -1
    r, ns, idx0 = _args(idx_null=True)
    assert lib.spsk_ball_query_msg_grid(b, n, m, 2, r, ns, FAKE, FAKE, idx0, FAKE, need, None) == -1
    assert b"null idx" in lib.spsk_last_error()
    assert lib.spsk_ball_query_msg_grid(b, n, m, 5, r, ns, FAKE, FAKE, idx, FAKE, need, None) == -1   # > 4 scales
    assert lib.spsk_ball_query_msg_grid(b, n, m, 2, r, ns, FAKE, FAKE, idx, FAKE, need - 1, None) == -4
    assert str(need).encode() in lib.spsk_last_error()
    assert lib.spsk_ball_query_msg_grid(b, n, m, 2, r, ns, FAKE, FAKE, idx, None, need, None) == -4


@pytest.mark.parametrize("b,n", [(1, 1), (1, 2048), (3, 16384), (8, 65535), (2, 65536)])
def test_ball_query_grid_workspace_unchanged_up_to_65536_points(b, n):
    from spsnet_b200 import _lib

    assert int(_lib.lib.spsk_ball_query_grid_workspace_bytes(b, n)) == parent_workspace_bytes(b, n)


def test_ball_query_grid_workspace_grows_with_windows():
    """One cell_start array per 65536-point window of each scene."""
    from spsnet_b200 import _lib

    for b, n in [(1, 65537), (2, 131072), (2, 131073), (4, 262144)]:
        windows = -(-n // 65536)
        want = parent_workspace_bytes(b, n) + 4 * b * 11265 * (windows - 1)
        assert int(_lib.lib.spsk_ball_query_grid_workspace_bytes(b, n)) == want
