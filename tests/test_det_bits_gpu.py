"""Every deterministic backward (ptk_*_bwd_det), and the plain-store grad_p1 of the default 1-NN and K-NN backward, gives
the committed bits on the seeded cases of tools/det_bits.py, with the kernel launch count include/ptk.h documents."""
import importlib.util
import json
import os

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_spec = importlib.util.spec_from_file_location("det_bits", os.path.join(ROOT, "tools", "det_bits.py"))
det_bits = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(det_bits)

pytestmark = pytest.mark.gpu
CASES = det_bits.cases()

with open(det_bits.OUT) as f:
    WANT = json.load(f)["cases"]


def test_every_case_has_committed_digests():
    assert sorted(CASES) == sorted(WANT)


@pytest.mark.parametrize("name", sorted(CASES))
def test_det_bits(name):
    run, launches = CASES[name]
    outs, n = run()
    torch.cuda.synchronize()
    assert n == launches
    assert det_bits.coverage(outs) >= det_bits.MIN_COVERAGE
    assert det_bits.digest(outs) == WANT[name]
