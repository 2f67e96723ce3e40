"""Learned-variance models (UbConfig.learn_sigma, guided-diffusion's `--learn_sigma True`) without a GPU: parameter
counts against the oracle built with out_channels = 6, the configs the library refuses, and identities of the
restatement in learn_sigma_oracle.py that the GPU tests rely on."""
import numpy as np
import pytest
import torch

import learn_sigma_oracle as LS


@pytest.mark.parametrize("kw,okw,expect", [
    ({}, {}, 20495942),
    (dict(super_res=4), dict(in_channels=6), 20497670),
])
def test_num_params_match_oracle(ub, oracle, kw, okw, expect):
    """The output conv grows to (6, C, 3, 3) + 6: 3 * 64 * 9 + 3 = 1 731 more parameters at C_model = 64."""
    n = ub.num_params(ub.default_config(learn_sigma=1, **kw))
    assert n == oracle.num_params(oracle.UNetConfig(out_channels=6, **okw)) == expect
    assert n - ub.num_params(ub.default_config(**kw)) == 3 * 64 * 9 + 3


@pytest.mark.parametrize("kw", [
    dict(learn_sigma=2), dict(learn_sigma=-1),
    dict(learn_sigma=1, C_in=1, C_out=1), dict(learn_sigma=1, C_out=4),
    dict(learn_sigma=1, compute_dinput=1),
    dict(learn_sigma=1, n_timesteps=1),                                 # lpost[0] would be log 0
    dict(learn_sigma=1, W=68, n_levels=2, channel_mult=(1, 2)),        # W % 8
    dict(learn_sigma=1, H=8, W=1024, n_levels=2, channel_mult=(1, 2)),  # the row kernels' shared memory
    dict(learn_sigma=1, C_model=1024),
])
def test_refused_configs(ub, kw):
    cfg = ub.default_config(**kw)
    assert ub.num_params(cfg) == 0
    cfg.learn_sigma = 0
    assert ub.num_params(cfg) > 0  # the same config without learn_sigma is accepted


def test_default_config_is_not_learn_sigma(ub):
    assert ub.default_config().learn_sigma == 0
    assert ub.UbConfig.learn_sigma.offset == ub.UbConfig.super_res.offset + 4  # the last field


def test_tables():
    tab = LS.tables(1000)
    assert tab["alphas_cumprod_prev"][0] == 1.0
    assert tab["posterior_log_variance_clipped"][0] == tab["posterior_log_variance_clipped"][1]
    np.testing.assert_allclose(np.exp(tab["posterior_log_variance_clipped"][1:]), tab["posterior_variance"][1:])
    assert tab["posterior_variance"][0] == 0.0


def _inputs(B=4, seed=0):
    g = torch.Generator().manual_seed(seed)
    x0 = (torch.rand(B, 3, 8, 8, generator=g, dtype=torch.float64) * 2 - 1)
    noise = torch.randn(B, 3, 8, 8, generator=g, dtype=torch.float64)
    out = torch.randn(B, 6, 8, 8, generator=g, dtype=torch.float64)
    t = torch.tensor([0, 1, 500, 999])[:B]
    acp = torch.from_numpy(LS.tables()["alphas_cumprod"])[t].reshape(-1, 1, 1, 1)
    x_t = acp.sqrt() * x0 + (1 - acp).sqrt() * noise
    return x0, noise, out, t, x_t


def test_learned_range_ends():
    """v = +1 gives log beta_t, v = -1 the clipped log posterior variance."""
    tab = LS.tables()
    x0, noise, out, t, x_t = _inputs()
    for v, name in ((1.0, "log_betas"), (-1.0, "posterior_log_variance_clipped")):
        o = out.clone()
        o[:, 3:] = v
        _, logvar, _ = LS.p_mean_variance(tab, o, x_t, t)
        ref = torch.from_numpy(tab[name])[t].reshape(-1, 1, 1, 1).expand_as(logvar)
        torch.testing.assert_close(logvar, ref, rtol=1e-12, atol=1e-12)


def test_kl_vanishes_at_the_posterior():
    """eps = noise and v = -1 give the model the posterior's mean and variance: vb = 0 for t >= 1."""
    tab = LS.tables()
    x0, noise, out, t, x_t = _inputs()
    o = torch.cat([noise, -torch.ones_like(noise)], 1)
    vb = LS.vb_terms_bpd(tab, o, x0, x_t, t)
    assert vb[1:].abs().max() < 1e-9
    assert vb[0] > 0  # t = 0: the decoder's negative log-likelihood


def test_normal_kl_matches_torch_distributions():
    g = torch.Generator().manual_seed(3)
    m1, m2 = torch.randn(100, generator=g, dtype=torch.float64), torch.randn(100, generator=g, dtype=torch.float64)
    l1, l2 = torch.randn(100, generator=g, dtype=torch.float64), torch.randn(100, generator=g, dtype=torch.float64)
    ref = torch.distributions.kl_divergence(torch.distributions.Normal(m1, (0.5 * l1).exp()),
                                            torch.distributions.Normal(m2, (0.5 * l2).exp()))
    torch.testing.assert_close(LS.normal_kl(m1, l1, m2, l2), ref, rtol=1e-10, atol=1e-12)


def test_gradients_split_between_eps_and_v():
    """frozen_out: eps learns from the MSE alone and v from vb alone."""
    tab = LS.tables()
    x0, noise, out, t, x_t = _inputs()
    o = out.clone().requires_grad_(True)
    vb = LS.vb_terms_bpd(tab, torch.cat([o[:, :3].detach(), o[:, 3:]], 1), x0, x_t, t)
    vb.sum().backward()
    assert not o.grad[:, :3].any() and o.grad[:, 3:].abs().sum() > 0
    o.grad = None
    loss, mse, _ = LS.hybrid_loss(tab, o, x0, x_t, t, noise)
    loss.backward()
    torch.testing.assert_close(o.grad[:, :3], 2 * (o[:, :3] - noise).detach() / (4 * 3 * 64))


def test_decoder_edge_branches():
    """x = -1 and +1 take the one-sided CDF tails of discretized_gaussian_log_likelihood; a tail below 1e-12 is
    clamped."""
    x = torch.tensor([-1.0, 1.0, 0.0, -1.0], dtype=torch.float64)
    mean = torch.tensor([-0.9, 0.9, 0.01, 0.0], dtype=torch.float64)
    ls = torch.full((4,), -2.0, dtype=torch.float64)
    lp = LS.discretized_gaussian_log_likelihood(x, mean, ls)
    s = np.exp(2.0)
    cdf = lambda z: float(LS.approx_standard_normal_cdf(torch.tensor(z, dtype=torch.float64)))
    ref = [np.log(cdf(s * (-0.1 + 1 / 255))), np.log(1 - cdf(s * (0.1 - 1 / 255))),
           np.log(cdf(s * (-0.01 + 1 / 255)) - cdf(s * (-0.01 - 1 / 255))), np.log(1e-12)]
    np.testing.assert_allclose(lp.numpy(), ref, rtol=1e-12)
