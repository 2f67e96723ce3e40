"""Learned-variance models (UbConfig.learn_sigma, guided-diffusion's `--learn_sigma True` with the hybrid loss) on the
GPU, against learn_sigma_oracle.py and the oracle U-Net built with out_channels = 6.

Head in isolation: the loss terms and the six output-bias gradients the fused head kernel computes, against the
restatement evaluated in float64 on the trainer's own (B, 6, H, W) output -- t = 0, 1, 500 and T - 1 in one batch and
x0 with exact -1 / +1 pixels (every branch of the KL / decoder likelihood), eager, captured and with random_flip.
Whole model: one forward + backward with the bounds of test_trainer_gpu.py, the output conv's v rows on their own.
Training: a 10-step captured loss trace.  Sampling: DDIM and learned-range ancestral parity with injected draws, a
full-list ancestral run, and the training state after sampling.  ABI edges: ub_trainer_sample and checkpoints."""
import os

import numpy as np
import pytest
import torch

import learn_sigma_oracle as LS
import spaced_oracle as SO
from test_trainer_gpu import TOL_TENSOR_L2, check_grads

pytestmark = pytest.mark.gpu

TOL_PARITY = 3e-2   # the bound of test_sampler_spaced_gpu.py (max-abs over max|ref|)
TOL_FULL_L2 = 3e-2  # its bound for a full run (relative L2)


def _model(O, okw=None, v_scale=0.0, seed=0):
    """Oracle config with the six-output head, perturb_zero_params weights; v_scale > 0 adds N(0, v_scale^2) to the
    head's v rows (weights 3-5), so that v -- and frac -- varies between pixels."""
    torch.set_num_threads(os.cpu_count() or 1)
    cfg = O.UNetConfig(out_channels=6, **(okw or {}))
    flat = O.perturb_zero_params(cfg, O.flatten_params(cfg, O.init_params(cfg, seed=seed)))
    if v_scale:
        off, n, shape = _head_weight(O, cfg)
        w = flat[off:off + n].reshape(shape).clone()
        w[3:] += v_scale * torch.randn(w[3:].shape, generator=torch.Generator().manual_seed(7))
        flat = flat.clone()
        flat[off:off + n] = w.reshape(-1)
    return cfg, flat


def _head_weight(O, cfg):
    off = 0
    for name, shape in O.param_spec(cfg):
        n = int(np.prod(shape))
        if name == "out.2.weight":
            return off, n, shape
        off += n
    raise KeyError("out.2.weight")


def _batch(B=4, seed=1234, H=64, W=64):
    """x0 with exact -1 / +1 pixels, t = 0, 1, 500, 999 (repeated), N(0, 1) noise."""
    g = torch.Generator().manual_seed(seed)
    x0 = torch.rand(B, 3, H, W, generator=g) * 2 - 1
    x0[:, :, ::7, ::5] = 1.0
    x0[:, :, 3::7, 2::5] = -1.0
    t = torch.tensor([0.0, 1.0, 500.0, 999.0]).repeat(B // 4 + 1)[:B].reshape(B, 1)
    noise = torch.randn(B, 3, H, W, generator=g)
    return x0, t, noise


def _head_reference(O, out, x0, t, noise):
    """The restatement in float64 on the trainer's output: mse, vb (batch means) and the per-channel sums of dL/dout,
    i.e. the output bias gradient."""
    x_t = O.q_sample(x0, t, noise).double()   # the trainer's float32 q-sample
    o = torch.from_numpy(out).double().requires_grad_(True)
    loss, mse, vb = LS.hybrid_loss(LS.tables(), o, x0.double(), x_t, t.reshape(-1).long(), noise.double())
    loss.backward()
    return float(mse.mean().detach()), float(vb.mean().detach()), o.grad.sum(dim=(0, 2, 3)).numpy()


# A head whose 6-output kernel needs more than the default 48 KiB of shared memory: (6 x 128 x 9 + 8 x 6 x 128) x 4 B
# = 51 KiB at C = 128, W = 128 (the default head takes 25.5 KiB)
WIDE = (dict(C_model=128, H=128, W=128, channel_mult=(1, 2), n_res_blocks=1, att_start_level=2),
        dict(model_channels=128, H=128, W=128, channel_mult=(1, 2), num_res_blocks=1, attn_start_level=2))


@pytest.mark.parametrize("mode", ["eager", "captured", "random_flip", "wide"])
def test_head_in_isolation(ub, oracle, mode):
    O = oracle
    kw, okw = WIDE if mode == "wide" else ({}, {})
    H = kw.get("H", 64)
    cfg, flat = _model(O, okw, v_scale=0.05)
    x0, t, noise = _batch(8, H=H, W=H)
    tr = ub.Trainer(B=8, learn_sigma=1, random_flip=int(mode == "random_flip"), **kw)
    tr.set_params(flat.numpy())
    if mode == "captured":
        tr.train_step(x0.numpy(), t.numpy(), noise.numpy(), lr=1e-4, want_loss=False)
        tr.sync()
    else:
        tr.forward_backward(x0.numpy(), t.numpy(), noise.numpy())
    x0_seen = x0
    if mode == "random_flip":
        flips = tr.get_flips()
        assert 0 < flips.sum() < len(flips)
        x0_seen = O.random_flip(x0, flips)
    out = tr.get_output()
    assert out.shape == (8, 6, H, H)
    assert np.abs(out[:, 3:]).max() > 0.05  # v is not constant
    mse_ref, vb_ref, db_ref = _head_reference(O, out, x0_seen, t, noise)
    mse, vb = tr.last_loss_terms()
    print(f"[head {mode}] mse {mse:.7g} (ref {mse_ref:.7g}), vb {vb:.7g} (ref {vb_ref:.7g})")
    assert abs(mse - mse_ref) <= 1e-5 * abs(mse_ref)
    assert abs(vb - vb_ref) <= 1e-4 * abs(vb_ref)
    assert abs(tr.last_loss() - (mse + vb)) <= 1e-6 * (mse + vb)
    if mode != "captured":  # (the captured step's AdamW update consumes the gradients)
        db = tr.get_grads()[-6:]
        print(f"[head {mode}] bias gradient {db} (ref {db_ref})")
        assert np.abs(db - db_ref).max() <= 1e-4 * np.abs(db_ref).max()
        assert np.abs(db[3:]).min() > 0
    tr.close()


CASES = [
    ("default", {}, {}, 4),
    ("class-conditional scale-shift updown hs64",
     dict(num_classes=10, use_scale_shift_norm=1, resblock_updown=1, head_size=64),
     dict(num_classes=10, use_scale_shift_norm=True, resblock_updown=True, head_size=64), 2),
    ("super_res 4", dict(super_res=4), dict(in_channels=6), 4),
    # the 6-output head at 63 KiB of shared memory, and the super-resolution input conv at its widest row
    ("super_res 4 W=256", dict(super_res=4, H=32, W=256, channel_mult=(1, 2), att_start_level=2, n_res_blocks=1),
     dict(in_channels=6, H=32, W=256, channel_mult=(1, 2), attn_start_level=2, num_res_blocks=1), 2),
]


@pytest.mark.parametrize("what,kw,okw,B", CASES, ids=[c[0] for c in CASES])
def test_forward_backward_matches_oracle(ub, oracle, what, kw, okw, B):
    O = oracle
    cfg, flat = _model(O, okw, v_scale=0.05)
    x0, t, noise = _batch(B, H=cfg.H, W=cfg.W)
    y = torch.arange(B) % 10 if cfg.num_classes else None
    tr = ub.Trainer(B=B, learn_sigma=1, **kw)
    assert tr.nparams == flat.numel()
    tr.set_params(flat.numpy())
    if y is not None:
        tr.set_labels(y.numpy().astype(np.int32))
    loss = tr.forward_backward(x0.numpy(), t.numpy(), noise.numpy())
    out, g = tr.get_output(), tr.get_grads()
    loss_ref, mse_ref, vb_ref, out_ref, g_ref = LS.train_step_grads(O, cfg, flat, x0, t, noise, y,
                                                                    kw.get("super_res", 0))
    g_ref = g_ref.numpy()
    print(f"[learn_sigma {what}] loss {loss:.6g} (ref {float(loss_ref):.6g}), terms {tr.last_loss_terms()} "
          f"(ref {float(mse_ref):.6g}, {float(vb_ref):.6g})")
    assert abs(loss - float(loss_ref)) <= 2e-3 * float(loss_ref)
    assert np.abs(out - out_ref.numpy()).max() <= 3e-2 * np.abs(out_ref.numpy()).max()
    check_grads(O, cfg, g, g_ref, "learn_sigma " + what)
    # the output conv's v rows on their own: they learn from vb alone, so a wrong dL/dv shows here
    off, n, shape = _head_weight(O, cfg)
    gv, rv = g[off:off + n].reshape(shape)[3:], g_ref[off:off + n].reshape(shape)[3:]
    nref = float(np.linalg.norm(rv))
    rel = float(np.linalg.norm(gv - rv)) / nref
    print(f"[learn_sigma {what}] output-conv v rows: rel-L2 {rel:.3e}, |ref| {nref:.3e}")
    assert nref > 0 and rel <= TOL_TENSOR_L2
    tr.close()


def test_ten_step_loss_trace(ub, oracle):
    O = oracle
    cfg, flat = _model(O, v_scale=0.05)
    B = 4
    batches = [_batch(B, seed=1234 + i) for i in range(10)]
    losses_ref, flat_ref = LS.train_steps(O, cfg, flat, batches, lr=1e-4)
    tr = ub.Trainer(B=B, learn_sigma=1)
    tr.set_params(flat.numpy())
    losses = [tr.train_step(b[0].numpy(), b[1].numpy(), b[2].numpy(), lr=1e-4) for b in batches]
    print("loss trace", np.array(losses), "oracle", np.array(losses_ref))
    assert np.abs(np.array(losses) - np.array(losses_ref)).max() <= 1e-2
    assert np.abs(tr.get_params() - flat_ref.numpy()).max() <= 2.5e-3
    tr.close()


@pytest.fixture(scope="module")
def sampling(ub, oracle):
    O = oracle
    cfg, flat = _model(O, v_scale=0.1)
    P = O.unflatten_params(cfg, flat)
    tr = ub.Trainer(B=2, learn_sigma=1)
    tr.set_params(flat.numpy())
    fn = lambda x, t: O.unet_forward(cfg, P, x, torch.full((x.shape[0], 1), float(t)))
    yield O, cfg, flat, fn, tr
    tr.close()


def _draws(n, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(2, 3, 64, 64, generator=g) * scale, [torch.randn(2, 3, 64, 64, generator=g) for _ in range(n)]


@pytest.mark.parametrize("clip", [True, False])
@pytest.mark.parametrize("sampler,eta,spec", [("ddim", 0.0, "ddim10"), ("ddim", 1.0, "ddim10"),
                                              ("ancestral", 0.0, "250")])
def test_three_iterations_match_oracle(ub, sampling, sampler, eta, spec, clip):
    O, cfg, flat, fn, tr = sampling
    ts = ub.space_timesteps(1000, spec)[:3]
    x, noises = _draws(3, 21, scale=3.0)
    with torch.no_grad():
        v = fn(x, ts[-1])[:, 3:]
    assert float(v.std()) > 0.05  # frac varies between pixels
    if sampler == "ddim":  # DDIM reads eps and ignores v
        ref = SO.spaced_sample(lambda x_, t_: fn(x_, t_)[:, :3], x, ts, sampler, eta, clip, noises).numpy()
    else:
        ref = LS.p_sample_loop(fn, x, ts, clip, noises).numpy()
    out = tr.sample_spaced(x.numpy(), ts, sampler, eta, clip, torch.stack(noises).numpy())
    err = np.abs(out - ref).max() / np.abs(ref).max()
    assert err <= TOL_PARITY, (sampler, eta, clip, err)


def test_learned_variance_scales_the_draw(ub, sampling):
    """With large injected draws the noise term dominates one ancestral iteration: the result follows the learned
    variance, and the fixed-large variance of a model without learn_sigma is far from it."""
    O, cfg, flat, fn, tr = sampling
    ts = ub.space_timesteps(1000, "250")[:2]
    x, noises = _draws(2, 27)
    noises = [50 * z for z in noises]
    ref = LS.p_sample_loop(fn, x, ts, True, noises).numpy()
    fixed = SO.spaced_sample(lambda x_, t_: fn(x_, t_)[:, :3], x, ts, "ancestral", 0.0, True, noises).numpy()
    out = tr.sample_spaced(x.numpy(), ts, "ancestral", 0.0, True, torch.stack(noises).numpy())
    err = float(np.linalg.norm(out - ref) / np.linalg.norm(ref))
    far = float(np.linalg.norm(fixed - ref) / np.linalg.norm(ref))
    print(f"learned-range draw: relative L2 {err:.3e}, fixed-large variance at {far:.3e}")
    assert err <= TOL_FULL_L2 and far > 10 * TOL_FULL_L2


def test_full_list_ancestral_matches_p_sample_loop(ub, oracle):
    """Every timestep of a 50-step schedule kept: ub_trainer_sample's replacement for a learned-variance model.  (The
    linear schedule scales its betas by 1000 / T, so at T = 20 the last beta is 1 and acp reaches 0.)"""
    O = oracle
    cfg, flat = _model(O, v_scale=0.1)
    P = O.unflatten_params(cfg, flat)
    fn = lambda x, t: O.unet_forward(cfg, P, x, torch.full((x.shape[0], 1), float(t)))
    T = 50
    tr = ub.Trainer(B=2, learn_sigma=1, n_timesteps=T)
    tr.set_params(flat.numpy())
    x, noises = _draws(T, 24)
    ts = list(range(T))
    ref = LS.p_sample_loop(fn, x, ts, True, noises, T=T).numpy()
    out = tr.sample_spaced(x.numpy(), ts, "ancestral", 0.0, True, torch.stack(noises).numpy())
    rel = float(np.linalg.norm(out - ref) / np.linalg.norm(ref))
    print(f"full-list learned-range ancestral run: relative L2 {rel:.3e}")
    assert rel <= TOL_FULL_L2
    tr.close()


def test_sampling_leaves_training_state_untouched(ub, oracle, tmp_path):
    O = oracle
    cfg, flat = _model(O, v_scale=0.1)
    x0, t, noise = (a.numpy() for a in _batch(2))
    tr = ub.Trainer(B=2, learn_sigma=1)
    tr.set_params(flat.numpy())
    tr.train_step(x0, t, noise, lr=1e-4)
    tr.save(str(tmp_path / "before.bin"), with_adamw=True)
    x, noises = _draws(3, 26)
    tr.sample_spaced(x.numpy(), ub.space_timesteps(1000, "ddim10"), "ddim", 1.0, True, None, seed=4)
    tr.sample_spaced(x.numpy(), ub.space_timesteps(1000, "250")[:3], "ancestral", 0.0, False,
                     torch.stack(noises).numpy())
    tr.save(str(tmp_path / "after.bin"), with_adamw=True)
    assert (tmp_path / "before.bin").read_bytes() == (tmp_path / "after.bin").read_bytes()
    tr.close()


def test_abi_edges(ub, oracle, tmp_path):
    O = oracle
    cfg, flat = _model(O)
    L = ub.lib()
    tr = ub.Trainer(B=2, learn_sigma=1)
    tr.set_params(flat.numpy())
    img = np.zeros((2, 3, 64, 64), np.float32)
    assert L.ub_trainer_sample(tr._h, ub._ptr(img), 40, 38, None, 0, ub._ptr(img)) == -4  # UB_ERR_STATE
    assert b"sample_spaced" in L.ub_last_error()
    out = tr.predict(img, np.full((2, 1), 10.0, np.float32))
    assert out.shape == (2, 6, 64, 64)
    tr.train_step(img, lr=1e-4)
    path = str(tmp_path / "ls.bin")
    tr.save(path, with_adamw=True)
    header, _ = O.read_model_bin(path)
    assert header[2] == 3 and header[4] == 6
    hcfg = ub.UbConfig()
    assert L.ub_read_checkpoint_header(path.encode(), ub.C.byref(hcfg)) == 0 and hcfg.C_out == 6
    tr2 = ub.Trainer(B=2, learn_sigma=1)
    tr2.load(path)
    np.testing.assert_array_equal(tr2.get_params(), tr.get_params())
    plain = ub.Trainer(B=2)
    assert L.ub_trainer_load(plain._h, path.encode()) == -1  # UB_ERR_SHAPE
    tr.close(), tr2.close(), plain.close()
