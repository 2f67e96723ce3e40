"""The cosine noise schedule (UbConfig.noise_schedule = UB_SCHEDULE_COSINE, guided-diffusion's `--noise_schedule cosine`)
on the GPU, against noise_schedule_oracle.py and the oracle U-Net.

Whole model: one forward + backward of the default model with t = 0, 998 and 999 among the timesteps, with the bounds of
test_trainer_gpu.py.  Head in isolation: the hybrid loss's terms and the six output-bias gradients at t = 0, 1, 500, 998
and 999 -- where cosine reaches acp = 2.4e-9, sqrt(1/acp) = 2.03e4 and log beta ~ lpost ~ -0.001 -- on the trainer's
own output, eager and captured.  The ImageNet 64x64 configuration: forward + backward with the device's dropout masks
and a 10-step captured loss trace.  Sampling: three-iteration parity of DDIM, fixed-large and learned-range ancestral
sampling, and ub_trainer_sample's refusal."""
import numpy as np
import pytest
import torch

import noise_schedule_oracle as NS
from test_learn_sigma_gpu import _model as _ls_model
from test_trainer_gpu import _resblock_shapes, check_grads

pytestmark = pytest.mark.gpu

COSINE = 1          # UB_SCHEDULE_COSINE
TOL_PARITY = 3e-2   # the bound of test_sampler_spaced_gpu.py (max-abs over max|ref|)
TOL_FULL_L2 = 3e-2  # test_learn_sigma_gpu.py's bound on learned-range draws (relative L2)


def _ts_batch(B, seed, H=64, W=64, special=(0.0, 998.0, 999.0)):
    """x0 ~ U[-1, 1], N(0, 1) noise; the first timesteps are `special`, the rest random."""
    g = torch.Generator().manual_seed(seed)
    x0 = torch.rand(B, 3, H, W, generator=g) * 2 - 1
    t = torch.randint(0, 1000, (B, 1), generator=g).float()
    t[:len(special), 0] = torch.tensor(special[:B])
    noise = torch.randn(B, 3, H, W, generator=g)
    return x0, t, noise


def test_forward_backward_default_model(ub, oracle):
    O = oracle
    cfg = O.UNetConfig()
    flat = O.perturb_zero_params(cfg, O.flatten_params(cfg, O.init_params(cfg, seed=0)))
    x0, t, noise = _ts_batch(4, 1234)
    tr = ub.Trainer(B=4, noise_schedule=COSINE)
    tr.set_params(flat.numpy())
    loss = tr.forward_backward(x0.numpy(), t.numpy(), noise.numpy())
    out, g = tr.get_output(), tr.get_grads()
    loss_ref, out_ref, g_ref = NS.train_step_grads(cfg, flat, x0, t, noise, schedule="cosine")
    print(f"[cosine default] loss {loss:.6g} (ref {float(loss_ref):.6g})")
    assert abs(loss - float(loss_ref)) <= 2e-3 * float(loss_ref)
    assert np.abs(out - out_ref.numpy()).max() <= 3e-2 * np.abs(out_ref.numpy()).max()
    check_grads(O, cfg, g, g_ref.numpy(), "cosine default")
    # the same batch under the linear schedule is far outside both bounds (oracle: 0.44 of max|out|, 0.13 rel-L2)
    _, out_lin, g_lin = NS.train_step_grads(cfg, flat, x0, t, noise, schedule="linear")
    out_ref, g_ref = out_ref.numpy(), g_ref.numpy()
    assert np.abs(out_lin.numpy() - out_ref).max() > 3 * 3e-2 * np.abs(out_ref).max()
    assert float(np.linalg.norm(g_lin.numpy() - g_ref) / np.linalg.norm(g_ref)) > 3 * 2e-2
    tr.close()


def _head_batch(B=10, seed=1234):
    """x0 with exact -1 / +1 pixels, t = 0, 1, 500, 998, 999 (repeated), N(0, 1) noise."""
    g = torch.Generator().manual_seed(seed)
    x0 = torch.rand(B, 3, 64, 64, generator=g) * 2 - 1
    x0[:, :, ::7, ::5] = 1.0
    x0[:, :, 3::7, 2::5] = -1.0
    t = torch.tensor([0.0, 1.0, 500.0, 998.0, 999.0]).repeat(B // 5 + 1)[:B].reshape(B, 1)
    return x0, t, torch.randn(B, 3, 64, 64, generator=g)


@pytest.mark.parametrize("mode", ["eager", "captured"])
def test_head_in_isolation(ub, oracle, mode):
    """The loss terms and bias gradients of the fused head against the float64 restatement on the trainer's output.
    At t = 999 the eps error reaches the model mean as c1 sqrt(1/acp - 1) ~ 31.6 and the KL runs through expm1."""
    import learn_sigma_oracle as LS
    O = oracle
    cfg, flat = _ls_model(O, v_scale=0.05)
    x0, t, noise = _head_batch()
    tr = ub.Trainer(B=10, learn_sigma=1, noise_schedule=COSINE)
    tr.set_params(flat.numpy())
    if mode == "captured":
        tr.train_step(x0.numpy(), t.numpy(), noise.numpy(), lr=1e-4, want_loss=False)
        tr.sync()
    else:
        tr.forward_backward(x0.numpy(), t.numpy(), noise.numpy())
    out = tr.get_output()
    x_t = NS.q_sample(x0, t, noise, "cosine").double()  # the trainer's float32 q-sample
    o = torch.from_numpy(out).double().requires_grad_(True)
    loss, mse, vb = LS.hybrid_loss(NS.tables(1000, "cosine"), o, x0.double(), x_t, t.reshape(-1).long(),
                                   noise.double())
    loss.backward()
    mse_ref, vb_ref, db_ref = float(mse.detach().mean()), float(vb.detach().mean()), o.grad.sum(dim=(0, 2, 3)).numpy()
    mse_d, vb_d = tr.last_loss_terms()
    print(f"[cosine head {mode}] mse {mse_d:.7g} (ref {mse_ref:.7g}), vb {vb_d:.7g} (ref {vb_ref:.7g}); per image vb "
          f"{vb.detach().numpy()[:5]} at t = {t.reshape(-1).numpy()[:5]}")
    assert abs(mse_d - mse_ref) <= 1e-5 * abs(mse_ref)
    assert abs(vb_d - vb_ref) <= 1e-4 * abs(vb_ref)
    if mode == "eager":  # (the captured step's AdamW update consumes the gradients)
        db = tr.get_grads()[-6:]
        print(f"[cosine head] bias gradient {db} (ref {db_ref})")
        assert np.abs(db - db_ref).max() <= 1e-4 * np.abs(db_ref).max()
        assert np.abs(db[3:]).min() > 0
    tr.close()


IMAGENET64 = (dict(att_start_level=1, num_classes=1000, learn_sigma=1, C_model=192, head_size=64, n_res_blocks=3,
                   resblock_updown=1, use_scale_shift_norm=1, dropout=0.1, noise_schedule=COSINE),
              dict(attn_start_level=1, num_classes=1000, out_channels=6, model_channels=192, head_size=64,
                   num_res_blocks=3, resblock_updown=True, use_scale_shift_norm=True, dropout=0.1))


def test_imagenet64_configuration(ub, oracle):
    """guided-diffusion's ImageNet 64x64 model (296 M parameters; attention at 32x32 runs T = 1024 on the SIMT
    fallback) at B = 2: one forward + backward against the oracle with the masks the device drew, then a 10-step
    captured loss trace that stays finite."""
    O = oracle
    kw, okw = IMAGENET64
    cfg = O.UNetConfig(**okw)
    flat = O.perturb_zero_params(cfg, O.flatten_params(cfg, O.init_params(cfg, seed=0)))
    B = 2
    x0, t, noise = _ts_batch(B, 99, special=(999.0, 3.0))
    y = np.array([7, 912], dtype=np.int32)
    tr = ub.Trainer(B=B, **kw)
    assert tr.nparams == flat.numel() == 295904454
    tr.set_params(flat.numpy())
    tr.set_labels(y)
    loss = tr.forward_backward(x0.numpy(), t.numpy(), noise.numpy())
    out, g = tr.get_output(), tr.get_grads()
    masks = [torch.from_numpy(tr.get_dropout_mask(i, *s)) for i, s in enumerate(_resblock_shapes(O, cfg))]
    loss_ref, out_ref, g_ref = NS.train_step_grads(cfg, flat, x0, t, noise, torch.from_numpy(y).long(), masks,
                                                   schedule="cosine")
    print(f"[imagenet64] loss {loss:.6g} (ref {float(loss_ref):.6g}), terms {tr.last_loss_terms()}")
    assert abs(loss - float(loss_ref)) <= 2e-3 * float(loss_ref)
    assert np.abs(out - out_ref.numpy()).max() <= 3e-2 * np.abs(out_ref.numpy()).max()
    check_grads(O, cfg, g, g_ref.numpy(), "imagenet64 cosine")
    losses = []
    for i in range(10):
        x0, t, noise = _ts_batch(B, 100 + i, special=())
        losses.append(tr.train_step(x0.numpy(), t.numpy(), noise.numpy(), lr=1e-4))
    print("[imagenet64] loss trace", np.array(losses))
    assert np.isfinite(losses).all()
    assert np.isfinite(tr.get_params()).all()
    tr.close()


# Chains and their inputs.  Clip on, from t = 999: x0 = clamp(2.03e4 (x - eps)) is a sign function of x - eps, so x_T
# is kept at least 0.5 away from the model's eps and every pixel clamps the same way on both sides; the two smallest
# steps of "250" follow, where sqrt(1/acp) ~ 1.  Clip off: the first step is from 980 (two smallest and the largest
# step of "ddim50"); its update multiplies eps differences by sqrt(acp_20 / acp_980) ~ 32, as it multiplies x.
CHAINS = {True: [0, 4, 999], False: [0, 20, 980]}


def _draws(n, seed):
    g = torch.Generator().manual_seed(seed)
    z = torch.randn(2, 3, 64, 64, generator=g)
    return torch.sign(z) * (2 + z.abs()), [torch.randn(2, 3, 64, 64, generator=g) for _ in range(n)]


@pytest.fixture(scope="module")
def models(ub, oracle):
    O = oracle
    res = {}
    for ls in (False, True):
        cfg, flat = _ls_model(O, v_scale=0.1) if ls else (O.UNetConfig(), None)
        if not ls:
            flat = O.perturb_zero_params(cfg, O.flatten_params(cfg, O.init_params(cfg, seed=0)))
        P = O.unflatten_params(cfg, flat)
        tr = ub.Trainer(B=2, learn_sigma=int(ls), noise_schedule=COSINE)
        tr.set_params(flat.numpy())
        res[ls] = (lambda x, t, cfg=cfg, P=P: O.unet_forward(cfg, P, x, torch.full((x.shape[0], 1), float(t))), tr)
    yield res
    for _, tr in res.values():
        tr.close()


@pytest.mark.parametrize("clip", [True, False])
@pytest.mark.parametrize("sampler,eta,learned", [("ddim", 0.0, False), ("ddim", 1.0, False),
                                                 ("ancestral", 0.0, False), ("ancestral", 0.0, True)])
def test_three_iterations_match_oracle(ub, models, sampler, eta, learned, clip):
    fn, tr = models[learned]
    ts = CHAINS[clip]
    x, noises = _draws(3, 21)
    with torch.no_grad():
        gap = float((x - fn(x, ts[-1])[:, :3]).abs().min())
    assert gap > 0.5
    if learned:
        run = lambda c: NS.p_sample_loop(fn, x, ts, c, noises, schedule="cosine")
    else:
        eps_fn = lambda x_, t_: fn(x_, t_)[:, :3]
        run = lambda c: NS.spaced_sample(eps_fn, x, ts, sampler, eta, c, noises, schedule="cosine")
    ref = run(clip).numpy()
    out = tr.sample_spaced(x.numpy(), ts, sampler, eta, clip, torch.stack(noises).numpy())
    err = float(np.abs(out - ref).max() / np.abs(ref).max())
    rel = float(np.linalg.norm(out - ref) / np.linalg.norm(ref))
    print(f"[cosine {sampler} eta={eta} learned={learned} clip={clip} ts={ts}] max-abs/max|ref| {err:.3e}, "
          f"relative L2 {rel:.3e}")
    assert np.isfinite(out).all()
    if learned:
        # A jump from 999 (980) to 4 (20) spans log beta' ~ 0 to lpost' = log(1 - acp_prev) = -8.4 (-6.4): sigma =
        # exp(0.5 (frac log beta' + (1 - frac) lpost')) has d sigma / dv = 2.1 sigma (1.6 sigma), so an element's bf16
        # error in v reaches x unattenuated, times z.  Two device runs of the same forward differ by up to 1.6e-2 in
        # their output, so the all-oracle chain is met at isolated pixels only to max-abs 8e-2 .. 2.2e-1 (clip on) and
        # 2.6e-2 .. 3.6e-2 (clip off) of max|ref| (B200, 1000 W; relative L2 4.6e-3 and 3.1e-3).  The bound is the
        # relative L2 test_learn_sigma_gpu.py puts on learned-range draws.
        assert rel <= TOL_FULL_L2, rel
    else:
        assert err <= TOL_PARITY, err
    if clip:  # the clip binds: without it the chain is elsewhere
        other = run(False).numpy()
        assert np.abs(other - ref).max() > 0.1 * np.abs(ref).max()


def test_generate_sampler_refuses_cosine(ub, models):
    _, tr = models[False]
    img = np.zeros((2, 3, 64, 64), np.float32)
    L = ub.lib()
    assert L.ub_trainer_sample(tr._h, ub._ptr(img), 40, 38, None, 0, ub._ptr(img)) == -4  # UB_ERR_STATE
    assert b"sample_spaced" in L.ub_last_error() and b"linear" in L.ub_last_error()
