"""3x3 conv weight gradients in row mode (one filter row per CTA, a TMA box per tap) vs the oracle.

The weight-gradient kernel takes column mode (one halo box per filter column) for every 3x3 layer whose padded width
is at least 8 pixels; row mode remains the path of 1x1 layers and of 3x3 layers with W <= 4.  These shapes are the
tensor-core (Cin, Cout multiples of 64) 3x3 layers that reach row mode."""
import math
import os

import pytest
import torch

from gpu_util import TOL_BF16, TOL_F32, call, dev, rel_inf

pytestmark = pytest.mark.gpu


def rnd(*shape, seed=0, scale=1.0):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed)) * scale


@pytest.mark.parametrize("B,Cin,Cout,H,W", [
    (4, 64, 64, 4, 4),
    (3, 128, 64, 3, 3),
    (3, 128, 64, 4, 2),
    (4, 64, 128, 3, 3),
])
def test_conv2d_k3_backward_row_mode(ub, oracle, B, Cin, Cout, H, W):
    torch.set_num_threads(os.cpu_count() or 1)
    x = rnd(B, Cin, H, W, seed=1).requires_grad_(True)
    w = (rnd(Cout, Cin, 3, 3, seed=2) / math.sqrt(9 * Cin)).requires_grad_(True)
    b = rnd(Cout, seed=3).requires_grad_(True)
    dout = rnd(B, Cout, H, W, seed=4)
    oracle.conv3x3(x, w, b).backward(dout)
    dx_, dw_, db_ = dev(x.detach()), dev(w.detach()), dev(b.detach())
    gdx, gdw, gdb = torch.empty_like(dx_), torch.empty_like(dw_), torch.empty_like(db_)
    call(ub, "conv2d_k3_backward2", dev(dout), dx_, dw_, None, None, gdx, gdw, gdb, B, Cin, Cout, H, W)
    assert rel_inf(gdx, x.grad) <= TOL_BF16
    assert rel_inf(gdw, w.grad) <= TOL_BF16
    assert rel_inf(gdb, b.grad) <= TOL_F32
