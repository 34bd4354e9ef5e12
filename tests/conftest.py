import os
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def _has_gpu():
    try:
        import torch

        return torch.cuda.is_available()
    except Exception:
        return False


def pytest_collection_modifyitems(config, items):
    if _has_gpu():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


def _require_ref() -> bool:
    """oracle/_ref (the upstream reference rebuilt by oracle/build_ref.sh) is not part of the repository: without it the
    `if ref_ops is not None` side-by-side comparisons are left out, and the tests compare against the oracle and the
    recorded outputs under tests/golden/.  SPSK_REQUIRE_REF=1 makes a missing or broken oracle/_ref a failure."""
    return os.environ.get("SPSK_REQUIRE_REF") == "1"


@pytest.fixture(scope="session")
def oracle():
    from oracle import oracle as O

    O.build()
    return O


@pytest.fixture(scope="session")
def ref_ops():
    """The reference's own pointnet2_batch (rebuilt unmodified for sm_100a by oracle/build_ref.sh), or None."""
    ref_root = ROOT / "oracle" / "_ref"
    so = ref_root / "pcdet" / "ops" / "pointnet2" / "pointnet2_batch" / "pointnet2_batch_cuda.so"
    if not so.exists():
        if _require_ref():
            pytest.fail(f"{so} is missing (SPSK_REQUIRE_REF=1; build it with "
                        "oracle/build_ref.sh)")
        return None
    import importlib
    import warnings

    if str(ref_root) not in sys.path:
        sys.path.insert(0, str(ref_root))
    try:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            utils = importlib.import_module("pcdet.ops.pointnet2.pointnet2_batch.pointnet2_utils")
            modules = importlib.import_module("pcdet.ops.pointnet2.pointnet2_batch.pointnet2_modules")
    except Exception as e:  # pragma: no cover
        if _require_ref():
            pytest.fail(f"reference extension in oracle/_ref is not importable: {e}")
        print("reference ext not importable:", e)
        return None

    class R:
        pass

    R.utils, R.modules = utils, modules
    return R


@pytest.fixture(scope="session")
def ref_det():
    """The reference's own iou3d_nms extension, IASSD_Head, box coder and class_agnostic_nms (oracle/_ref, unmodified,
    rebuilt by oracle/build_ref.sh), or None.  `SharedArray` -- an absent dependency of pcdet.utils.common_utils that
    nothing on this path uses -- is satisfied with an empty module."""
    ref_root = ROOT / "oracle" / "_ref"
    if not (ref_root / "pcdet" / "ops" / "iou3d_nms" / "iou3d_nms_cuda.so").exists():
        if _require_ref():
            pytest.fail("oracle/_ref/pcdet/ops/iou3d_nms/iou3d_nms_cuda.so is missing (SPSK_REQUIRE_REF=1; oracle/build_ref.sh)")
        return None
    import importlib
    import types
    import warnings

    if str(ref_root) not in sys.path:
        sys.path.insert(0, str(ref_root))
    sys.modules.setdefault("SharedArray", types.ModuleType("SharedArray"))
    try:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            R = types.SimpleNamespace(
                cuda=importlib.import_module("pcdet.ops.iou3d_nms.iou3d_nms_cuda"),
                utils=importlib.import_module("pcdet.ops.iou3d_nms.iou3d_nms_utils"),
                nms_utils=importlib.import_module("pcdet.models.model_utils.model_nms_utils"),
                head=importlib.import_module("pcdet.models.dense_heads.IASSD_head"),
                coder=importlib.import_module("pcdet.utils.box_coder_utils"),
            )
    except Exception as e:  # pragma: no cover
        if _require_ref():
            pytest.fail(f"reference detection modules in oracle/_ref are not importable: {e}")
        print("reference detection modules not importable:", e)
        return None
    return R


@pytest.fixture
def recorded(request):
    """tests/helpers.py::Recorded for this test (keyed by its name and parameters)."""
    from helpers import Recorded

    rec = Recorded(request.node.name)
    yield rec
    rec.save()
