"""The Python mirror of the three_nn kernel-choice macros of include/spsk.h."""
import re
from pathlib import Path

from spsnet_b200 import pointnet2_utils as pu

ROOT = Path(__file__).resolve().parents[1]


def test_three_nn_grid_constants_match_the_header():
    hdr = (ROOT / "include" / "spsk.h").read_text()
    macros = dict(re.findall(r"#define\s+SPSK_(THREE_NN_GRID_\w+)\s+(\d+)", hdr))
    assert sorted(macros) == ["THREE_NN_GRID_MAX_M", "THREE_NN_GRID_MIN_M", "THREE_NN_GRID_MIN_N"]
    for name, value in macros.items():
        assert getattr(pu, name) == int(value), name
    assert pu.THREE_NN_GRID_MIN_M <= pu.THREE_NN_GRID_MAX_M
