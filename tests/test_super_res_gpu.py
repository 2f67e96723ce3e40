"""Super-resolution models (UbConfig.super_res = f, guided-diffusion's SuperResModel) on the GPU.

Condition: the channels a training step computes on the device equal guided-diffusion's
F.interpolate(F.interpolate(x0, (H/f, W/f), "area"), (H, W), "bilinear") within 1e-6 (f = 2 and 4, a non-square model,
random_flip against the flipped batch, a captured train_step).  Training: one forward + backward against the oracle run
on cat([x_t, cond]) with in_channels = 6, with the bounds of test_trainer_gpu.py; the input conv's weight gradient
columns 3-5 (the conditioning channels) are checked on their own.  Inference: predict / sample / sample_spaced after
set_low_res against the conditioned oracle.  Rejections and checkpoints."""
import os

import numpy as np
import pytest
import torch

import spaced_oracle as SO
import superres_oracle as SR
from test_trainer_gpu import TOL_TENSOR_L2, check_grads

pytestmark = pytest.mark.gpu

NONSQUARE = (dict(H=64, W=32, channel_mult=(1, 2, 4), att_start_level=1, n_res_blocks=1),
             dict(H=64, W=32, channel_mult=(1, 2, 4), attn_start_level=1, num_res_blocks=1))


def _ocfg(O, okw):
    return O.UNetConfig(in_channels=6, out_channels=3, **okw)


def _batch(O, cfg, B, seed=1234):
    x0, t, noise = O.synthetic_batch(cfg, B, seed)
    return x0[:, :3].contiguous(), t, noise[:, :3].contiguous()


@pytest.mark.parametrize("f,kw,okw", [(2, {}, {}), (4, {}, {}), (4,) + NONSQUARE])
def test_condition_matches_interpolate(ub, oracle, f, kw, okw):
    O = oracle
    cfg = _ocfg(O, okw)
    x0, t, noise = _batch(O, cfg, 3)
    tr = ub.Trainer(B=3, super_res=f, **kw)
    tr.set_params(O.flatten_params(cfg, O.init_params(cfg, seed=0)).numpy())
    tr.forward_backward(x0.numpy(), t.numpy(), noise.numpy())
    cond = tr.get_cond()
    assert np.abs(cond - SR.condition(x0, f).numpy()).max() <= 1e-6
    tr.close()


def test_condition_with_random_flip_and_captured_step(ub, oracle):
    O = oracle
    cfg = _ocfg(O, {})
    B = 8
    tr = ub.Trainer(B=B, super_res=4, random_flip=1)
    tr.set_params(O.flatten_params(cfg, O.init_params(cfg, seed=0)).numpy())
    seen = set()
    for step in range(3):
        x0 = torch.rand(B, 3, 64, 64, generator=torch.Generator().manual_seed(step)) * 2 - 1
        if step == 0:
            tr.forward_backward(x0.numpy())
        else:
            tr.train_step(x0.numpy(), lr=1e-5)  # one captured graph, replayed
        flips = tr.get_flips()
        seen.update(int(v) for v in flips)
        ref = SR.condition(O.random_flip(x0, flips), 4).numpy()
        assert np.abs(tr.get_cond() - ref).max() <= 1e-6, step
    assert seen == {0, 1}  # both branches of the flip were taken
    tr.close()


def _input_conv_weight(O, cfg, g):
    off = 0
    for name, shape in O.param_spec(cfg):
        n = int(np.prod(shape))
        if name == "input_blocks.0.0.weight":
            return g[off:off + n].reshape(shape)
        off += n
    raise KeyError("input_blocks.0.0.weight")


CASES = [
    ("default B=4", {}, {}, 4, 4),
    ("128px five levels", dict(H=128, W=128, channel_mult=(1, 1, 2, 3, 4), att_start_level=3),
     dict(H=128, W=128, channel_mult=(1, 1, 2, 3, 4), attn_start_level=3), 4, 2),
    ("class-conditional", dict(num_classes=10), dict(num_classes=10), 2, 2),
    ("W=256", dict(H=32, W=256, channel_mult=(1, 2), att_start_level=2, n_res_blocks=1),
     dict(H=32, W=256, channel_mult=(1, 2), attn_start_level=2, num_res_blocks=1), 4, 1),
]


@pytest.mark.parametrize("what,kw,okw,f,B", CASES, ids=[c[0] for c in CASES])
def test_forward_backward_matches_oracle(ub, oracle, what, kw, okw, f, B):
    O = oracle
    torch.set_num_threads(os.cpu_count() or 1)
    cfg = _ocfg(O, okw)
    flat = O.perturb_zero_params(cfg, O.flatten_params(cfg, O.init_params(cfg, seed=0)))
    x0, t, noise = _batch(O, cfg, B)
    y = torch.arange(B) % 10 if cfg.num_classes else None
    tr = ub.Trainer(B=B, super_res=f, **kw)
    assert tr.nparams == flat.numel()
    tr.set_params(flat.numpy())
    if y is not None:
        tr.set_labels(y.numpy())
    loss = tr.forward_backward(x0.numpy(), t.numpy(), noise.numpy())
    out, g = tr.get_output(), tr.get_grads()
    loss_ref, out_ref, g_ref, _ = SR.train_step_grads(O, cfg, flat, x0, t, noise, f, y)
    g_ref = g_ref.numpy()
    assert abs(loss - float(loss_ref)) <= 2e-3 * float(loss_ref)
    assert np.abs(out - out_ref.numpy()).max() <= 3e-2 * np.abs(out_ref.numpy()).max()
    check_grads(O, cfg, g, g_ref, "super_res " + what)
    # the conditioning channels' weight gradient on its own, within the per-tensor bound; the reference is non-zero, so
    # a zero block (conditioning channels not read) would sit at relative distance 1, far beyond the bound
    gc, rc = _input_conv_weight(O, cfg, g)[:, 3:], _input_conv_weight(O, cfg, g_ref)[:, 3:]
    nref = float(np.linalg.norm(rc))
    rel = float(np.linalg.norm(gc - rc)) / nref
    print(f"[super_res {what}] input-conv columns 3-5: rel-L2 {rel:.3e}, |ref| {nref:.3e}")
    assert nref > 0 and rel <= TOL_TENSOR_L2
    losses = [tr.train_step(x0.numpy(), lr=1e-4) for _ in range(2)]  # captured graph
    assert np.isfinite(losses).all()
    tr.close()


def test_dinput_is_the_x_t_gradient(ub, oracle):
    O = oracle
    cfg = _ocfg(O, {})
    flat = O.perturb_zero_params(cfg, O.flatten_params(cfg, O.init_params(cfg, seed=0)))
    x0, t, noise = _batch(O, cfg, 2)
    _, _, _, dxt_ref = SR.train_step_grads(O, cfg, flat, x0, t, noise, 4)
    tr = ub.Trainer(B=2, super_res=4, compute_dinput=1)
    tr.set_params(flat.numpy())
    tr.forward_backward(x0.numpy(), t.numpy(), noise.numpy())
    d, ref = tr.get_dinput(), dxt_ref.numpy()
    assert d.shape == (2, 3, 64, 64)
    assert np.abs(d - ref).max() <= 3e-2 * np.abs(ref).max()
    tr.close()


@pytest.fixture(scope="module")
def sampling(oracle):
    O = oracle
    torch.set_num_threads(os.cpu_count() or 1)
    cfg = _ocfg(O, {})
    flat = O.perturb_zero_params(cfg, O.flatten_params(cfg, O.init_params(cfg, seed=0)))
    g = torch.Generator().manual_seed(21)
    low = torch.rand(2, 3, 16, 16, generator=g) * 2 - 1
    x = torch.randn(2, 3, 64, 64, generator=g)
    noises = torch.stack([torch.randn(2, 3, 64, 64, generator=g) for _ in range(3)])
    return O, cfg, flat, O.unflatten_params(cfg, flat), low, x, noises


def test_predict_and_samplers_match_oracle(ub, sampling):
    O, cfg, flat, P, low, x, noises = sampling
    fn = SR.model_fn(O, cfg, P, low)
    tr = ub.Trainer(B=2, super_res=4)
    tr.set_params(flat.numpy())
    tr.set_low_res(low.numpy())
    t = torch.tensor([[37.0], [512.0]])
    out = tr.predict(x.numpy(), t.numpy())
    with torch.no_grad():
        ref = fn(x, t).numpy()
    assert np.abs(out - ref).max() <= 3e-2 * np.abs(ref).max()
    assert np.abs(tr.get_cond() - SR.upsample(low, 64, 64).numpy()).max() <= 1e-6
    # the last three iterations of each schedule with x_init scaled so that the clip binds, as
    # test_sampler_spaced_gpu.py runs them (at large t, x0 = sqrt(1/acp) x - sqrt(1/acp - 1) eps magnifies the bf16
    # differences of eps and the clip turns them into different values at isolated pixels)
    xs = 3.0 * x
    for sampler, spec in (("ddim", "ddim10"), ("ancestral", "250")):
        ts = ub.space_timesteps(1000, spec)[:3]
        out = tr.sample_spaced(xs.numpy(), ts, sampler=sampler, eta=0.0, noises=noises.numpy())
        ref = SO.spaced_sample(fn, xs, ts, sampler, 0.0, True, list(noises)).numpy()
        assert np.abs(out - ref).max() <= 3e-2 * np.abs(ref).max(), sampler
    out = tr.sample(x.numpy(), 40, 38, noises.numpy())
    ref = SR.ddpm_sample(O, cfg, P, low, x, 40, 38, list(noises)).numpy()
    assert np.abs(out - ref).max() <= 3e-2 * np.abs(ref).max()
    # a training step in between overwrites the conditioning channels; the next inference call upsamples again
    tr.forward_backward(np.zeros((2, 3, 64, 64), np.float32))
    out2 = tr.sample_spaced(xs.numpy(), ts, sampler="ancestral", noises=noises.numpy())
    ref = SO.spaced_sample(fn, xs, ts, "ancestral", 0.0, True, list(noises)).numpy()
    assert np.abs(out2 - ref).max() <= 3e-2 * np.abs(ref).max()
    tr.close()


def test_rejections(ub, sampling, tmp_path):
    O, cfg, flat, P, low, x, noises = sampling
    L = ub.lib()
    tr = ub.Trainer(B=2, super_res=4)
    tr.set_params(flat.numpy())
    t = np.full((2, 1), 10.0, np.float32)
    img = np.zeros((2, 3, 64, 64), np.float32)
    assert L.ub_trainer_predict(tr._h, ub._ptr(img), ub._ptr(t), ub._ptr(img)) == -4  # UB_ERR_STATE: no low-res yet
    assert b"set_low_res" in L.ub_last_error()
    assert L.ub_trainer_sample(tr._h, ub._ptr(img), 40, 38, None, 0, ub._ptr(img)) == -4
    ts = np.array([0, 500], np.int32)
    assert L.ub_trainer_sample_spaced(tr._h, ts.ctypes.data_as(ub.C.c_void_p), 2, 0, 0.0, 1, ub._ptr(img), None, 0,
                                      ub._ptr(img)) == -4
    bad = np.zeros(2 * 3 * 16 * 15, np.float32)
    assert L.ub_trainer_set_low_res(tr._h, ub._ptr(bad), bad.size) == -1  # UB_ERR_SHAPE
    path = str(tmp_path / "sr.bin")
    tr.save(path)
    tr.close()
    plain = ub.Trainer(B=2)
    lo = low.numpy()
    assert L.ub_trainer_set_low_res(plain._h, ub._ptr(lo), lo.size) == -4
    with pytest.raises(ub.UbError):
        plain.get_cond()
    assert L.ub_trainer_load(plain._h, path.encode()) == -1
    plain.close()


def test_checkpoint(ub, sampling, tmp_path):
    O, cfg, flat, P, low, x, noises = sampling
    tr = ub.Trainer(B=2, super_res=4)
    tr.set_params(flat.numpy())
    tr.train_step(np.zeros((2, 3, 64, 64), np.float32), lr=1e-4)
    path = str(tmp_path / "sr.bin")
    tr.save(path, with_adamw=True)
    header, _ = O.read_model_bin(path)
    assert header[2] == 6 and header[3] == 64 and header[4] == 3
    assert os.path.getsize(path) == 4 * 256 + 3 * 4 * tr.nparams
    tr2 = ub.Trainer(B=2, super_res=4)
    tr2.load(path)
    np.testing.assert_array_equal(tr2.get_params(), tr.get_params())
    tr.close(), tr2.close()
