"""Respaced sampling without a GPU: ub_space_timesteps (the C library) against the restatement of guided-diffusion's
space_timesteps in spaced_oracle.py, and identities of its respaced tables and sampler steps."""
import numpy as np
import pytest
import torch

import spaced_oracle as S

SPECS = ["ddim10", "ddim50", "ddim250", "250", "1000", "1", "10,10,10", "3,7",
         # strides with exact .5 ties (999/6, 999/12, 999/24; 49/2 at T = 100): Python rounds them to even
         "7", "13", "25"]


@pytest.mark.parametrize("T", [1000, 100])
@pytest.mark.parametrize("spec", SPECS)
def test_space_timesteps_matches_oracle(ub, T, spec):
    try:
        ref = S.space_timesteps(T, spec)
    except ValueError:
        with pytest.raises(ub.UbError):
            ub.space_timesteps(T, spec)
        return
    assert ub.space_timesteps(T, spec) == ref


def test_space_timesteps_ties_round_to_even(ub):
    # 166.5, 499.5, 832.5 -> 166, 500, 832 (round half away from zero would give 167, 500, 833)
    assert ub.space_timesteps(1000, "7") == [0, 166, 333, 500, 666, 832, 999]
    assert ub.space_timesteps(100, "3,7") == S.space_timesteps(100, "3,7") == [0, 24, 49, 50, 58, 66, 74, 83, 91, 99]
    assert ub.space_timesteps(1000, "ddim10") == list(range(0, 1000, 100))
    assert ub.space_timesteps(1000, "1000") == list(range(1000))


def test_space_timesteps_accumulates_the_stride(ub):
    """guided-diffusion adds the fractional stride up (cur_idx += frac_stride); for 21 sections of 999/20 the float64
    sum and j * 999/20 fall on different sides of a tie at j = 10 and j = 14."""
    acc = S.space_timesteps(1000, "21")
    mul = sorted({round(j * 999 / 20) for j in range(21)})
    assert acc != mul
    assert ub.space_timesteps(1000, "21") == acc


@pytest.mark.parametrize("spec", ["ddim999", "ddim0", "ddim1", "1001", "600,600", "", "abc", "ddim", "ddimx", "10,,10",
                                  "10,x", "-5", "0"])
def test_space_timesteps_rejections(ub, spec):
    with pytest.raises(ValueError):
        S.space_timesteps(1000, spec)
    with pytest.raises(ub.UbError):
        ub.space_timesteps(1000, spec)


def test_spaced_acp_equals_base_acp_at_kept_timesteps():
    base = np.cumprod(1.0 - np.linspace(1e-4, 0.02, 1000, dtype=np.float64))
    for spec in ("ddim50", "250", "10,10,10", "3,7"):
        ts = S.space_timesteps(1000, spec)
        tab = S.spaced_tables(1000, ts)
        np.testing.assert_allclose(tab["alphas_cumprod"], base[ts], rtol=0, atol=1e-12)


def test_full_list_gives_the_unspaced_tables(oracle):
    betas = np.linspace(1e-4, 0.02, 1000, dtype=np.float64)
    tab = S.spaced_tables(1000, list(range(1000)))
    np.testing.assert_allclose(tab["betas"], betas, rtol=0, atol=1e-12)
    np.testing.assert_allclose(tab["alphas_cumprod"], np.cumprod(1 - betas), rtol=0, atol=1e-12)
    # the training step's float32 tables, whose betas are rounded to float32 before the product (train_unet.py)
    sa, sb = oracle.diffusion_tables(1000)
    np.testing.assert_allclose(np.sqrt(tab["alphas_cumprod"]), sa, rtol=0, atol=2e-6)
    np.testing.assert_allclose(np.sqrt(1 - tab["alphas_cumprod"]), sb, rtol=0, atol=2e-6)


def test_ddim_eta1_on_the_full_schedule_is_the_posterior():
    """ddim_sample with eta = 1 over every timestep: sigma^2 = posterior variance (fixed small), mean = posterior mean."""
    tab = S.spaced_tables(1000, list(range(1000)))
    g = torch.Generator().manual_seed(3)
    for i in (1, 2, 10, 500, 999):
        x, eps, z = (torch.randn(2, 3, 8, 8, generator=g, dtype=torch.float64) for _ in range(3))
        x0 = (np.sqrt(1 / tab["alphas_cumprod"][i]) * x - np.sqrt(1 / tab["alphas_cumprod"][i] - 1) * eps).clamp(-1, 1)
        mean = tab["posterior_mean_coef1"][i] * x0 + tab["posterior_mean_coef2"][i] * x
        want = mean + np.sqrt(tab["posterior_variance"][i]) * z
        got = S.spaced_step(tab, i, x.float(), eps.float(), "ddim", 1.0, True, z.float()).double()
        # guided-diffusion extracts acp'_{i-1} as float32: 1 - acp'_{i-1} (1e-4 at i = 1) loses ~6e-8 / (1 - acp'_{i-1})
        tol = 1e-5 + 1e-7 / (1 - tab["alphas_cumprod_prev"][i])
        assert float((got - want).abs().max()) <= tol * float(want.abs().max()), i


def _analytic_model(x0):
    """eps(x, t) = (x - sqrt(acp[t]) x0) / sqrt(1 - acp[t]): the exact noise predictor for data that is all x0."""
    acp = np.cumprod(1.0 - np.linspace(1e-4, 0.02, 1000, dtype=np.float64))

    def fn(x, t):
        return (x - float(np.sqrt(acp[t])) * x0) / float(np.sqrt(1 - acp[t]))
    return fn


@pytest.mark.parametrize("spec", ["ddim10", "ddim50", "250", "10,10,10"])
def test_ddim_eta0_recovers_x0_under_the_analytic_model(spec):
    """Pins the acp[t] (not acp[t-1]) convention: the deterministic sampler lands on x0 from any x_T."""
    g = torch.Generator().manual_seed(11)
    x0 = torch.rand(2, 3, 8, 8, generator=g) * 1.8 - 0.9
    xT = torch.randn(2, 3, 8, 8, generator=g) * 1.5
    ts = S.space_timesteps(1000, spec)
    for clip in (True, False):
        out = S.spaced_sample(_analytic_model(x0), xT, ts, "ddim", 0.0, clip)
        assert float((out - x0).abs().max()) <= 1e-5, (spec, clip)
    # with the model one timestep off (acp[t+1] at model input t) the sampler misses x0 by ~2e-2
    model = _analytic_model(x0)
    out = S.spaced_sample(lambda x, t: model(x, min(t + 1, 999)), xT, ts, "ddim", 0.0, False)
    assert float((out - x0).abs().max()) > 1e-3


@pytest.mark.parametrize("spec", ["250", "ddim50", "1000"])
def test_ancestral_without_noise_recovers_x0_under_the_analytic_model(spec):
    g = torch.Generator().manual_seed(12)
    x0 = torch.rand(2, 3, 8, 8, generator=g) * 1.8 - 0.9
    xT = torch.randn(2, 3, 8, 8, generator=g)
    out = S.spaced_sample(_analytic_model(x0), xT, S.space_timesteps(1000, spec), "ancestral", 0.0, True)
    assert float((out - x0).abs().max()) <= 1e-5, spec
