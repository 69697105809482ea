"""The filter scan picks its chunk width from the layout of the clouds (64 targets when every cloud is 16-byte aligned,
16 otherwise).  Every layout must give the exact scan's results bit for bit."""
import pytest
import torch

import ptk_b200

pytestmark = pytest.mark.gpu


def _clouds(B, P, offset, g):
    buf = torch.rand(B * P * 3 + offset, device="cuda", generator=g) - 0.5
    return buf[offset:].view(B, P, 3)


@pytest.mark.parametrize("B,P1,P2,off", [
    (3, 1001, 998, 0),    # P % 4 != 0: odd clouds are not 16-byte aligned
    (2, 1000, 1000, 1),   # a view starting 4 bytes into its storage
    (2, 1000, 1000, 0),   # aligned, last 64-target chunk partial (1000 % 64 = 40)
    (1, 6000, 4999, 0),   # one pair: the target range is split across CTAs, split ends on 64-target boundaries
])
def test_filter_equals_exact_for_every_layout(B, P1, P2, off):
    g = torch.Generator(device="cuda").manual_seed(B * 7 + P1 + off)
    x, y = _clouds(B, P1, off, g), _clouds(B, P2, off, g)
    try:
        ptk_b200.ops.set_chamfer_algo("exact")
        c0, ix0, iy0 = ptk_b200.ops.chamfer(x, y)
        ptk_b200.ops.set_chamfer_algo("filter")
        c1, ix1, iy1 = ptk_b200.ops.chamfer(x, y)
    finally:
        ptk_b200.ops.set_chamfer_algo("auto")
    assert torch.equal(ix0, ix1) and torch.equal(iy0, iy1) and torch.equal(c0, c1)
