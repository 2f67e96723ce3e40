"""ub_trainer_sample_spaced (guided-diffusion's respaced DDIM / ancestral sampling on the device) against
spaced_oracle.spaced_sample with unet_forward as the model: B = 2, the default model with perturb_zero_params weights (the
zero-initialised output layers perturbed, so eps depends on x and t)."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

import spaced_oracle as S

pytestmark = pytest.mark.gpu

B, SHAPE = 2, (2, 3, 64, 64)
TOL_PARITY = 3e-2   # max-abs over max|ref|, the bound of test_sampler_matches_oracle
TOL_RUNS = 2e-2     # two device runs: GroupNorm-statistics atomics change the summation order
# relative L2 of a full ten-iteration ddim10 run (measured on a B200: 9.6e-3 to 1.0e-2 against the oracle, 8.1e-3 to
# 8.8e-3 between two device runs; its max-abs is not bounded, see test_device_draws)
TOL_DDIM10_L2 = 3e-2


def _model(O, okw=None, head_size=32):
    torch.set_num_threads(os.cpu_count() or 1)
    cfg = O.UNetConfig(head_size=head_size, **(okw or {}))
    flat = O.perturb_zero_params(cfg, O.flatten_params(cfg, O.init_params(cfg, seed=0)))
    return cfg, flat, O.unflatten_params(cfg, flat)


@pytest.fixture(scope="module")
def default_model(oracle):
    return _model(oracle)


@pytest.fixture(scope="module")
def trainer(ub, default_model):
    tr = ub.Trainer(B=B)
    tr.set_params(default_model[1].numpy())
    yield tr
    tr.close()


def _model_fn(O, cfg, P, y=None):
    return lambda x, t: O.unet_forward(cfg, P, x, torch.full((x.shape[0], 1), float(t)), y)


def _draws(n, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(*SHAPE, generator=g) * scale
    return x, [torch.randn(*SHAPE, generator=g) for _ in range(n)]


def _check_parity(O, tr, cfg, P, ts, sampler, eta, clip, x, noises, y=None):
    ref = S.spaced_sample(_model_fn(O, cfg, P, y), x, ts, sampler, eta, clip, noises).numpy()
    out = tr.sample_spaced(x.numpy(), ts, sampler, eta, clip, torch.stack(noises).numpy())
    err = np.abs(out - ref).max() / np.abs(ref).max()
    assert err <= TOL_PARITY, (sampler, eta, clip, err)
    return ref


@pytest.mark.parametrize("clip", [True, False])
@pytest.mark.parametrize("sampler,eta,spec", [("ddim", 0.0, "ddim10"), ("ddim", 1.0, "ddim10"),
                                              ("ancestral", 0.0, "250")])
def test_three_iterations_match_oracle(ub, oracle, default_model, trainer, sampler, eta, spec, clip):
    """The last three iterations of the schedule (its three smallest timesteps, t = 0 among them: the tables of a
    prefix of the kept list are the prefix of its tables), with the oracle's draws injected.  x_init is scaled so that
    the clip binds."""
    O = oracle
    cfg, _, P = default_model
    ts = ub.space_timesteps(1000, spec)[:3]
    assert ts[0] == 0
    x, noises = _draws(3, 21, scale=3.0)
    ref = _check_parity(O, trainer, cfg, P, ts, sampler, eta, clip, x, noises)
    other = S.spaced_sample(_model_fn(O, cfg, P), x, ts, sampler, eta, not clip, noises).numpy()
    assert np.abs(other - ref).max() > 0.1 * np.abs(ref).max()   # the clip changes the result: it binds


def test_full_ddim10_matches_oracle(ub, oracle, default_model, trainer):
    O = oracle
    cfg, _, P = default_model
    ts = ub.space_timesteps(1000, "ddim10")
    x, noises = _draws(10, 22)
    ref = S.spaced_sample(_model_fn(O, cfg, P), x, ts, "ddim", 0.0, True, noises).numpy()
    out = trainer.sample_spaced(x.numpy(), ts, "ddim", 0.0, True, torch.stack(noises).numpy())
    rel = float(np.linalg.norm(out - ref) / np.linalg.norm(ref))
    print(f"ddim10 eta=0 full run against the oracle: relative L2 {rel:.3e}, max-abs/max|ref| "
          f"{np.abs(out - ref).max() / np.abs(ref).max():.3e}")
    assert rel <= TOL_DDIM10_L2, rel


def test_class_conditional_matches_oracle(ub, oracle):
    O = oracle
    cfg, flat, P = _model(O, dict(num_classes=10))
    tr = ub.Trainer(B=B, num_classes=10)
    tr.set_params(flat.numpy())
    y = np.array([3, 7], dtype=np.int32)
    tr.set_labels(y)
    x, noises = _draws(3, 23, scale=3.0)
    ts = ub.space_timesteps(1000, "250")[:3]
    _check_parity(O, tr, cfg, P, ts, "ancestral", 0.0, True, x, noises, torch.from_numpy(y).long())
    tr.close()


def test_head_size64_matches_oracle(ub, oracle):
    O = oracle
    cfg, flat, P = _model(O, head_size=64)
    tr = ub.Trainer(B=B, head_size=64)
    tr.set_params(flat.numpy())
    x, noises = _draws(3, 24, scale=3.0)
    _check_parity(O, tr, cfg, P, ub.space_timesteps(1000, "ddim10")[:3], "ddim", 1.0, True, x, noises)
    tr.close()


def test_device_draws(ub, trainer):
    ts = ub.space_timesteps(1000, "ddim10")
    x, noises = _draws(10, 25)
    # eta = 0 draws nothing: device noise, injected noise and a second run agree up to the atomics -- element by element
    # over the last three iterations; over all ten, x0 = sqrt(1/acp) x - sqrt(1/acp - 1) eps multiplies run-to-run
    # differences of eps by ~60 at t = 900 and the clip turns them into different values at isolated pixels, so the full
    # runs are compared in relative L2
    a = trainer.sample_spaced(x.numpy(), ts[:3], "ddim", 0.0, True, None, seed=1)
    b = trainer.sample_spaced(x.numpy(), ts[:3], "ddim", 0.0, True, torch.stack(noises[:3]).numpy())
    c = trainer.sample_spaced(x.numpy(), ts[:3], "ddim", 0.0, True, None, seed=2)
    assert np.isfinite(a).all()
    assert np.abs(a - b).max() < TOL_RUNS and np.abs(a - c).max() < TOL_RUNS
    a, c = (trainer.sample_spaced(x.numpy(), ts, "ddim", 0.0, True, None, seed=s) for s in (1, 2))
    rel = float(np.linalg.norm(a - c) / np.linalg.norm(c))
    print(f"two full ddim10 eta=0 runs: relative L2 {rel:.3e}, max-abs {np.abs(a - c).max():.3e}")
    assert rel <= TOL_DDIM10_L2
    # eta = 1: the seed reaches the in-graph draws (same x_init, so only z differs); ancestral likewise
    d = trainer.sample_spaced(x.numpy(), ts, "ddim", 1.0, True, None, seed=1)
    e = trainer.sample_spaced(x.numpy(), ts, "ddim", 1.0, True, None, seed=2)
    assert np.isfinite(d).all() and np.abs(d - e).max() > 0.5
    f = trainer.sample_spaced(x.numpy(), ts, "ancestral", 0.0, True, None, seed=1)
    g = trainer.sample_spaced(x.numpy(), ts, "ancestral", 0.0, True, None, seed=2)
    assert np.abs(f - g).max() > 0.5
    # x_init = None draws x_T from the seed; the samples stay inside the clip range's scale
    h = trainer.sample_spaced(None, ts, "ddim", 0.0, True, None, seed=3)
    assert np.isfinite(h).all() and np.abs(h).max() <= 1.0 + 1e-5


def test_sampling_leaves_training_state_untouched(ub, oracle, default_model, tmp_path):
    O = oracle
    cfg, flat, _ = default_model
    x0, t, noise = O.synthetic_batch(cfg, B)
    x0, t, noise = x0.numpy(), t.numpy(), noise.numpy()
    trs = [ub.Trainer(B=B, ema_rate=0.999) for _ in range(2)]
    for tr in trs:
        tr.set_params(flat.numpy())
        tr.train_step(x0, t, noise, lr=1e-4)
    tr, ref = trs
    tr.save(str(tmp_path / "before.bin"), with_adamw=True)   # params, m, v and the step count
    ema = tr.get_ema()
    x, noises = _draws(3, 26)
    ts = ub.space_timesteps(1000, "ddim10")
    tr.sample_spaced(x.numpy(), ts, "ddim", 1.0, True, None, seed=4)
    tr.sample_spaced(x.numpy(), ts[:3], "ancestral", 0.0, False, torch.stack(noises).numpy())
    tr.save(str(tmp_path / "after.bin"), with_adamw=True)
    assert (tmp_path / "before.bin").read_bytes() == (tmp_path / "after.bin").read_bytes()
    assert np.array_equal(tr.get_ema(), ema)
    # the next training step (packed weights, buffers the sampler reused) sees what it would have seen without sampling
    la = tr.train_step(x0, t, noise, lr=1e-4)
    lb = ref.train_step(x0, t, noise, lr=1e-4)
    assert abs(la - lb) <= 1e-3 * abs(lb), (la, lb)
    for tr in trs:
        tr.close()


def test_generate_sampler_unchanged_after_spaced(ub, default_model):
    """ub_trainer_sample keeps its own graph and state: its result does not depend on a spaced run before it."""
    _, flat, _ = default_model
    tr = ub.Trainer(B=B)
    tr.set_params(flat.numpy())
    x, noises = _draws(3, 27)
    a = tr.sample(x.numpy(), 40, 38, torch.stack(noises).numpy())
    tr.sample_spaced(x.numpy(), ub.space_timesteps(1000, "ddim10"), "ddim", 1.0, True, None, seed=9)
    b = tr.sample(x.numpy(), 40, 38, torch.stack(noises).numpy())
    assert np.abs(a - b).max() < TOL_RUNS
    tr.close()


def test_rejections(ub, trainer):
    L = ub.lib()
    c = trainer.cfg
    img = c.B * c.C_in * c.H * c.W
    x = np.zeros(img, dtype=np.float32)
    out = np.zeros(img, dtype=np.float32)

    def call(tr, ts, sampler=0, eta=0.0, clip=1):
        a = np.ascontiguousarray(ts, dtype=np.int32)
        return L.ub_trainer_sample_spaced(tr._h, a.ctypes.data_as(C.c_void_p) if len(ts) else None, len(ts), sampler,
                                          eta, clip, x.ctypes.data_as(C.c_void_p), None, 0,
                                          out.ctypes.data_as(C.c_void_p))

    shape = -1   # UB_ERR_SHAPE
    for ts in ([], [5, 5], [10, 5], [-1, 5], [0, 1000], [0, 999, 998]):
        assert call(trainer, ts) == shape, ts
        assert b"timesteps" in L.ub_last_error()
    for sampler in (-1, 2):
        assert call(trainer, [0, 10], sampler) == shape
    for eta in (-0.1, 1.5, float("nan")):
        assert call(trainer, [0, 10], 0, eta) == shape, eta
    assert call(trainer, [0, 10], 1, 0.5) == shape            # ancestral takes no eta
    assert call(trainer, [10], 1) == shape                    # ancestral needs n >= 2
    assert call(trainer, [10], 0) == 0                        # DDIM with one step is fine
    tr = ub.Trainer(B=B, C_out=4)
    assert call(tr, [0, 10]) == shape
    assert b"C_in == C_out" in L.ub_last_error()
    tr.close()
