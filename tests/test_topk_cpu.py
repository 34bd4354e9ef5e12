"""CPU checks of spsk_score_topk's argument validation for the large-scene (thread-block cluster) path: every argument is
checked before any CUDA call, so these run without a GPU."""


def test_score_topk_rejects_more_than_262144_points():
    from spsnet_b200 import _lib

    lib = _lib.lib
    assert lib.spsk_score_topk(1, 262145, 3, 10, None, None, None, None, None) == -2
    assert b"262144" in lib.spsk_last_error()


def test_score_topk_checks_pointers_before_any_cuda_call():
    from spsnet_b200 import _lib

    lib = _lib.lib
    assert lib.spsk_score_topk(1, 262144, 3, 10, None, None, None, None, None) == -1
    assert b"null" in lib.spsk_last_error()
    assert lib.spsk_score_topk(2, 65536, 3, 70000, None, None, None, None, None) == -1  # npoint > n
    assert b"70000" in lib.spsk_last_error()
