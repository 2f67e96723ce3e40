"""Super-resolution models (UbConfig.super_res, guided-diffusion's SuperResModel) without a GPU: parameter counts
against the oracle built with in_channels = 6, the configs the library refuses, and the interpolation arithmetic the
conditioning kernel restates."""
import numpy as np
import pytest
import torch

import superres_oracle as SR

CONFIG5 = dict(H=128, W=128, channel_mult=(1, 1, 2, 3, 4))


@pytest.mark.parametrize("kw,okw,expect", [
    ({}, {}, 20495939),
    (dict(CONFIG5, att_start_level=3), dict(CONFIG5, attn_start_level=3), 21084483),
])
def test_num_params_match_oracle(ub, oracle, kw, okw, expect):
    """The input conv grows to (C_model * mult[0], 2 * C_in, 3, 3): 1 728 more weights at C_model = 64."""
    n = ub.num_params(ub.default_config(super_res=4, **kw))
    assert n == oracle.num_params(oracle.UNetConfig(in_channels=6, **okw)) == expect
    assert n - ub.num_params(ub.default_config(**kw)) == 64 * 3 * 9


@pytest.mark.parametrize("kw", [
    dict(super_res=1), dict(super_res=-2), dict(super_res=-4),
    dict(super_res=3),                                   # divides neither 64 nor 64
    dict(super_res=16, H=72), dict(super_res=16, W=72),  # divides W but not H, H but not W
    dict(super_res=4, C_in=1, C_out=1), dict(super_res=4, C_in=4, C_out=4),
    dict(super_res=4, C_out=1),
    dict(super_res=4, W=260, channel_mult=(1, 2)), dict(super_res=4, W=512),
])
def test_refused_configs(ub, kw):
    cfg = ub.default_config(**kw)
    assert ub.num_params(cfg) == 0
    cfg.super_res = 0
    assert ub.num_params(cfg) > 0  # the same config without super_res is accepted


def test_default_config_is_not_super_res(ub):
    assert ub.default_config().super_res == 0
    assert ub.UbConfig.super_res.offset == ub.UbConfig.dropout.offset + 4  # the last field


def _bilinear_ref(lo: np.ndarray, H: int, W: int) -> np.ndarray:
    """The conditioning kernel's index arithmetic in float32: src = (dst + 0.5) * in / out - 0.5 clamped at 0,
    i1 = min(i0 + 1, in - 1)."""
    h, w = lo.shape[-2:]

    def axis(n_in, n_out):
        scale = np.float32(n_in) / np.float32(n_out)
        src = np.maximum(scale * (np.arange(n_out, dtype=np.float32) + np.float32(0.5)) - np.float32(0.5), 0)
        i0 = src.astype(np.int64)
        return i0, np.minimum(i0 + 1, n_in - 1), (src - i0).astype(np.float32)

    y0, y1, ly = axis(h, H)
    x0, x1, lx = axis(w, W)
    ly, lx = ly[:, None], lx[None, :]
    g = lambda yi, xi: lo[..., yi[:, None], xi[None, :]]
    return (1 - ly) * ((1 - lx) * g(y0, x0) + lx * g(y0, x1)) + ly * ((1 - lx) * g(y1, x0) + lx * g(y1, x1))


@pytest.mark.parametrize("f,H,W", [(2, 64, 64), (4, 64, 64), (4, 64, 32), (8, 32, 256), (3, 48, 48)])
def test_condition_helper_matches_interpolate(f, H, W):
    """superres_oracle.condition is guided-diffusion's two F.interpolate calls, and the area mean + index arithmetic
    of the conditioning kernel reproduce them to float32 rounding; mirroring commutes with both at integer factors."""
    x0 = torch.rand(3, 3, H, W, generator=torch.Generator().manual_seed(f)) * 2 - 1
    ref = torch.nn.functional.interpolate(
        torch.nn.functional.interpolate(x0, (H // f, W // f), mode="area"), (H, W), mode="bilinear",
        align_corners=False)
    assert torch.equal(SR.condition(x0, f), ref)
    lo = x0.numpy().reshape(3, 3, H // f, f, W // f, f).mean(axis=(3, 5), dtype=np.float32)
    assert np.abs(_bilinear_ref(lo, H, W) - ref.numpy()).max() <= 1e-6
    assert (SR.condition(torch.flip(x0, dims=[-1]), f) - torch.flip(ref, dims=[-1])).abs().max() <= 1e-6
