"""Head size 64 (guided-diffusion's num_head_channels = 64) without a GPU: the parameter planner accepts it and counts
what the oracle counts (qkv is (3C, C) and proj (C, C) whatever the head size), other head sizes are refused, and the
oracle's multi-head attention agrees with torch's scaled_dot_product_attention at hs = 64 (and hs = 32), forward and
gradients.  The golden vectors cover hs = 32 only; this pins the oracle where the GPU tests of head size 64 use it."""
import pytest
import torch
import torch.nn.functional as F


def test_head_size_64_param_count(ub, oracle):
    n = ub.num_params(ub.default_config(head_size=64))
    assert n == 20494211
    assert n == oracle.num_params(oracle.UNetConfig(head_size=64))
    kw = dict(H=128, W=128, channel_mult=(1, 1, 2, 3, 4), att_start_level=3, head_size=64)
    assert ub.num_params(ub.default_config(**kw)) == 21082755


@pytest.mark.parametrize("hs", [16, 48, 128])
def test_other_head_sizes_rejected(ub, hs):
    assert ub.num_params(ub.default_config(head_size=hs)) == 0


def _sdpa_mha(qkv, n_heads):
    """Same contract as oracle.mha, (B, 3C, T) -> (B, C, T), through torch's scaled_dot_product_attention."""
    B, width, T = qkv.shape
    C = width // 3
    hs = C // n_heads
    q, k, v = (a.reshape(B, n_heads, hs, T).transpose(2, 3) for a in qkv.chunk(3, dim=1))  # (B, NH, T, hs)
    y = F.scaled_dot_product_attention(q, k, v)                                               # scale 1/sqrt(hs)
    return y.transpose(2, 3).reshape(B, C, T)


@pytest.mark.parametrize("B,T,C,NH", [(2, 64, 192, 3), (3, 16, 128, 2), (1, 256, 64, 1), (2, 64, 192, 6)])
def test_oracle_mha_matches_sdpa(oracle, B, T, C, NH):
    g = torch.Generator().manual_seed(11)
    qkv = (torch.randn(B, 3 * C, T, generator=g, dtype=torch.float64) * 1.5)
    dy = torch.randn(B, C, T, generator=g, dtype=torch.float64)
    a = qkv.clone().requires_grad_(True)
    b = qkv.clone().requires_grad_(True)
    ya, yb = oracle.mha(a, NH), _sdpa_mha(b, NH)
    ya.backward(dy)
    yb.backward(dy)
    torch.testing.assert_close(ya, yb, rtol=1e-10, atol=1e-12)
    torch.testing.assert_close(a.grad, b.grad, rtol=1e-10, atol=1e-12)
