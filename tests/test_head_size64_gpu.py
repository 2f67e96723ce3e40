"""Head size 64 on the GPU.

Layer: the native-layout attention core, tcgen05 kernels (impl 0) and SIMT fallback (impl 1), against oracle.mha on the
same bf16-rounded inputs: an odd head count (the default model's 16x16 level at head size 64 has C = 192, NH = 3), a
ragged last tile, NH = 1, T = 16 (eight images per 128-row tile), the full-size B = 32 case and T = 1024 (SIMT only).

Trainer: one forward + backward against the oracle with the bounds of test_trainer_gpu.py, then captured-graph steps,
for the default 64x64 model, the 128x128 five-level model and a 32x32 model whose attention runs at 32x32 (T = 1024,
SIMT fallback) and 16x16 (T = 256, tcgen05).  Where the attention backward is to be checked inside the trainer, the
zero-initialised layers (proj among them) are perturbed so that the attention core sits on the forward and backward
path.  Sampler: ub_trainer_sample against oracle.ddpm_sample."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from gpu_util import TOL_BF16, rel_inf
from test_trainer_gpu import check_grads

pytestmark = pytest.mark.gpu

SHAPES = [(4, 256, 192, 3), (4, 64, 256, 4), (3, 64, 128, 2), (2, 128, 64, 1), (5, 16, 64, 1), (32, 256, 192, 3),
          (2, 1024, 128, 2)]


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


@pytest.mark.parametrize("impl", [0, 1])
@pytest.mark.parametrize("B,T,Cc,NH", SHAPES)
def test_attention_nhwc_hs64(ub, oracle, B, T, Cc, NH, impl):
    assert Cc == 64 * NH
    if impl == 1 and B == 32:
        pytest.skip("full-size case is for the tensor-core path")
    if impl == 0 and T > 256:
        pytest.skip("T > 256 is the SIMT fallback's")
    g = torch.Generator().manual_seed(7)
    qkv = (torch.randn(B, T, 3 * Cc, generator=g) * 1.5).bfloat16()
    dout = torch.randn(B, T, Cc, generator=g).bfloat16()
    x = qkv.float().permute(0, 2, 1).contiguous().requires_grad_(True)
    y = oracle.mha(x, NH)                      # (B, C, T)
    y.backward(dout.float().permute(0, 2, 1).contiguous())
    y_ref = y.detach().permute(0, 2, 1)        # (B, T, C)
    dqkv_ref = x.grad.permute(0, 2, 1)         # (B, T, 3C)

    L = ub.lib()
    d_qkv, d_dout = qkv.cuda(), dout.cuda()
    d_out = torch.zeros(B, T, Cc, dtype=torch.bfloat16, device="cuda")
    d_lse = torch.zeros(B, NH, T, dtype=torch.float32, device="cuda")
    rc = L.ub_attention_nhwc_forward(_p(d_qkv), _p(d_out), _p(d_lse), B, T, Cc, NH, impl)
    torch.cuda.synchronize()
    assert rc == 0, L.ub_last_error()
    assert rel_inf(d_out, y_ref) <= TOL_BF16
    d_dqkv = torch.zeros(B, T, 3 * Cc, dtype=torch.bfloat16, device="cuda")
    d_dsum = torch.zeros(B, NH, T, dtype=torch.float32, device="cuda")
    rc = L.ub_attention_nhwc_backward(_p(d_qkv), _p(d_out), _p(d_dout), _p(d_lse), _p(d_dqkv), _p(d_dsum), B, T, Cc, NH,
                                      impl)
    torch.cuda.synchronize()
    assert rc == 0, L.ub_last_error()
    for name, sl in (("dq", slice(0, Cc)), ("dk", slice(Cc, 2 * Cc)), ("dv", slice(2 * Cc, 3 * Cc))):
        assert rel_inf(d_dqkv[..., sl], dqkv_ref[..., sl]) <= TOL_BF16, name


def test_attention_hs64_rejections(ub):
    L = ub.lib()
    t = torch.zeros(8, device="cuda")
    f = lambda B, T, Cc, NH, impl: L.ub_attention_nhwc_forward(_p(t), _p(t), _p(t), B, T, Cc, NH, impl)
    b = lambda B, T, Cc, NH, impl: L.ub_attention_nhwc_backward(_p(t), _p(t), _p(t), _p(t), _p(t), _p(t), B, T, Cc, NH,
                                                                impl)
    for fn in (f, b):
        assert fn(1, 1024, 128, 2, 0) != 0            # tcgen05 kernels: T <= 256
        assert b"T in {16,32,64,128,256}" in L.ub_last_error()
        for impl in (0, 1):
            assert fn(1, 64, 256, 2, impl) != 0       # head size 128
            assert b"head size must be 32 or 64" in L.ub_last_error()
            assert fn(1, 64, 144, 3, impl) != 0       # head size 48
        assert fn(1, 64, 96, 3, 0) != 0               # head size 32 still needs an even NH on impl 0


def _run_and_compare(ub, O, kw, okw, B, what, perturb=True):
    torch.set_num_threads(os.cpu_count() or 1)
    cfg = O.UNetConfig(head_size=64, **okw)
    flat = O.flatten_params(cfg, O.init_params(cfg, seed=0))
    if perturb:
        flat = O.perturb_zero_params(cfg, flat)
    x0, t, noise = O.synthetic_batch(cfg, B)
    tr = ub.Trainer(B=B, head_size=64, **kw)
    assert tr.nparams == flat.numel()
    tr.set_params(flat.numpy())
    loss = tr.forward_backward(x0.numpy(), t.numpy(), noise.numpy())
    out, g = tr.get_output(), tr.get_grads()
    loss_ref, out_ref, g_ref = O.train_step_grads(cfg, flat, x0, t, noise)
    assert abs(loss - float(loss_ref)) <= 2e-3 * float(loss_ref)
    assert np.abs(out - out_ref.numpy()).max() <= 3e-2 * np.abs(out_ref.numpy()).max()
    check_grads(O, cfg, g, g_ref.numpy(), what)
    losses = [tr.train_step(x0.numpy(), t.numpy(), noise.numpy(), lr=1e-4) for _ in range(3)]  # captured graph
    assert np.isfinite(losses).all(), losses
    tr.close()
    return flat, (x0, t, noise), g_ref.numpy()


def test_trainer_hs64_default_model(ub, oracle):
    O = oracle
    flat, batch, g_ref = _run_and_compare(ub, O, {}, {}, 4, "hs64 default B=4")
    # not vacuous: with the same weights at head size 32 the oracle's qkv-weight gradients lie beyond the per-tensor
    # bound (TOL_TENSOR_L2 = 6e-2) that check_grads applied above
    cfg = O.UNetConfig()
    _, _, g32 = O.train_step_grads(cfg, flat, *batch)
    g32, off, rel = g32.numpy(), 0, []
    for name, shape in O.param_spec(cfg):
        n = int(np.prod(shape))
        if name.endswith(".qkv.weight"):
            a, b = g_ref[off:off + n], g32[off:off + n]
            rel.append(float(np.linalg.norm(a - b) / np.linalg.norm(a)))
        off += n
    assert np.median(rel) > 6e-2, rel


def test_trainer_hs64_config5_128px(ub, oracle):
    """128x128, channel_mult (1,1,2,3,4), attention at 16x16 (C = 192, NH = 3) and 8x8 (C = 256, NH = 4).  Initial
    weights as in test_config5_128px_five_levels_matches_oracle: with the zero-initialised layers perturbed, the
    GroupNorm gradients of this deep model's 8x8 blocks (norms ~1e-4) reach the per-tensor bound from run to run
    (4.7e-2 .. 6.0e-2 seen), whatever the head size.  The attention output still enters every proj-weight gradient;
    the attention backward at these (T, C, NH) runs in test_trainer_hs64_default_model (same attention shapes) and in
    the layer tests."""
    _run_and_compare(ub, oracle, dict(H=128, W=128, channel_mult=(1, 1, 2, 3, 4), att_start_level=3),
                     dict(H=128, W=128, channel_mult=(1, 1, 2, 3, 4), attn_start_level=3), 2, "hs64 config5 B=2",
                     perturb=False)


def test_trainer_hs64_attention_at_32x32(ub, oracle):
    """Attention at 32x32 (T = 1024, C = 64, NH = 1: SIMT fallback) and 16x16 (T = 256, C = 128, NH = 2: tcgen05)."""
    _run_and_compare(ub, oracle, dict(H=32, W=32, channel_mult=(1, 2), att_start_level=0),
                     dict(H=32, W=32, channel_mult=(1, 2), attn_start_level=0), 2, "hs64 32x32 T=1024")


def test_sampler_hs64_matches_oracle(ub, oracle):
    """Three injected-noise iterations at small t, B = 2, as test_sampler_matches_oracle."""
    O = oracle
    torch.set_num_threads(os.cpu_count() or 1)
    cfg = O.UNetConfig(head_size=64)
    flat = O.perturb_zero_params(cfg, O.flatten_params(cfg, O.init_params(cfg, seed=0)))
    P = O.unflatten_params(cfg, flat)
    g = torch.Generator().manual_seed(21)
    x = torch.randn(2, 3, 64, 64, generator=g)
    noises = [torch.randn(2, 3, 64, 64, generator=g) for _ in range(3)]
    ref = O.ddpm_sample(cfg, P, x, 40, 38, noises).numpy()
    tr = ub.Trainer(B=2, head_size=64)
    tr.set_params(flat.numpy())
    out = tr.sample(x.numpy(), 40, 38, torch.stack(noises).numpy())
    assert np.abs(out - ref).max() <= 3e-2 * np.abs(ref).max()
    tr.close()
