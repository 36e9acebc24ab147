"""The torch-CPU baseline port prints exactly what the unmodified reference prints
(tests/golden/final_text.json, written by tests/golden/gen_golden_final_text.py)."""
import json
import os

import numpy as np
import pytest
import torch as T

import golden_io
from oracle import lev_ref_port as port

FINAL_TEXT = os.path.join(golden_io.GOLDEN_DIR, "final_text.json")


@pytest.mark.parametrize("name", [c["name"] for c in golden_io.LEV_CASES])
def test_port_prints_reference_text(name):
    case = golden_io.lev_case(name)
    oc = golden_io.draw_outcomes(case)
    want = json.load(open(FINAL_TEXT))[name]
    v0, top, grid = T.tensor(case["v0"]), case["top"], case["grid"]
    if case["kind"] == "coin":
        t = T.tensor(oc.astype(np.float32))
        rows, levs = port.fixed_final("coin", t, top, v0, (case["up_r"], case["down_r"]), grid)
    elif case["kind"] == "dice":
        t = T.tensor(oc.astype(np.int64))
        rows, levs = port.fixed_final("dice", t, top, v0, (case["up_r"], case["down_r"], case["mid_r"]), grid)
    elif case["kind"] == "dice_sh":
        t = T.tensor(oc.astype(np.int64))
        rows, levs = port.fixed_final("dice_sh", t, top, v0, (case["up_r"], case["down_r"], case["mid_r"]), grid,
                                      sh=case["sh"])
    else:
        t = T.tensor(oc)
        rows, levs = port.fixed_final("gbm", t, top, v0, None, grid)
    assert want == port.format_rows(rows, levs)
