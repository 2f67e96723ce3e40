"""Restatement of guided-diffusion's learned-variance model (`--learn_sigma True`) for the tests of the trainer's
`learn_sigma` option -- TEST INFRASTRUCTURE ONLY (CPU, plain numpy / torch).  gaussian_diffusion.py with
model_var_type LEARNED_RANGE and loss_type RESCALED_MSE (improved-diffusion's hybrid loss: `use_kl False`,
`rescale_learned_sigmas True`), restated: the float64 tables, normal_kl, approx_standard_normal_cdf,
discretized_gaussian_log_likelihood, _vb_terms_bpd, training_losses with `frozen_out`, and p_mean_variance / p_sample on
a respaced chain.  The U-Net is oracle/unet_oracle.py's, built with out_channels = 6 ([eps | v])."""
from __future__ import annotations

import math
from typing import Dict

import numpy as np
import torch

import spaced_oracle as SO


def tables(T: int = 1000) -> Dict[str, np.ndarray]:
    """GaussianDiffusion.__init__ on the trainer's linear schedule, float64."""
    scale = 1000 / T
    betas = np.linspace(scale * 0.0001, scale * 0.02, T, dtype=np.float64)
    acp = np.cumprod(1.0 - betas)
    acp_prev = np.append(1.0, acp[:-1])
    post_var = betas * (1.0 - acp_prev) / (1.0 - acp)
    return dict(betas=betas, log_betas=np.log(betas), alphas_cumprod=acp, alphas_cumprod_prev=acp_prev,
                sqrt_recip_alphas_cumprod=np.sqrt(1.0 / acp), sqrt_recipm1_alphas_cumprod=np.sqrt(1.0 / acp - 1),
                posterior_variance=post_var,
                posterior_log_variance_clipped=np.log(np.append(post_var[1], post_var[1:])),
                posterior_mean_coef1=betas * np.sqrt(acp_prev) / (1.0 - acp),
                posterior_mean_coef2=(1.0 - acp_prev) * np.sqrt(1.0 - betas) / (1.0 - acp))


def _ex(tab, name, t, like: torch.Tensor) -> torch.Tensor:
    """_extract_into_tensor: per-image entries of a table, broadcast over (C, H, W), in the dtype of `like`."""
    idx = torch.as_tensor(t).reshape(-1).long()
    return torch.from_numpy(tab[name])[idx].to(like.dtype).reshape(-1, *([1] * (like.dim() - 1)))


def normal_kl(mean1, logvar1, mean2, logvar2):
    """losses.normal_kl: KL(N(mean1, exp(logvar1)) || N(mean2, exp(logvar2))) per element, in nats."""
    return 0.5 * (-1.0 + logvar2 - logvar1 + torch.exp(logvar1 - logvar2)
                  + ((mean1 - mean2) ** 2) * torch.exp(-logvar2))


def approx_standard_normal_cdf(x):
    return 0.5 * (1.0 + torch.tanh(math.sqrt(2.0 / math.pi) * (x + 0.044715 * torch.pow(x, 3))))


def discretized_gaussian_log_likelihood(x, means, log_scales):
    """losses.discretized_gaussian_log_likelihood: log-likelihood of x in [-1, 1] discretised to 256 bins."""
    centered_x = x - means
    inv_stdv = torch.exp(-log_scales)
    plus_in = inv_stdv * (centered_x + 1.0 / 255.0)
    cdf_plus = approx_standard_normal_cdf(plus_in)
    min_in = inv_stdv * (centered_x - 1.0 / 255.0)
    cdf_min = approx_standard_normal_cdf(min_in)
    log_cdf_plus = torch.log(cdf_plus.clamp(min=1e-12))
    log_one_minus_cdf_min = torch.log((1.0 - cdf_min).clamp(min=1e-12))
    cdf_delta = cdf_plus - cdf_min
    return torch.where(x < -0.999, log_cdf_plus,
                       torch.where(x > 0.999, log_one_minus_cdf_min, torch.log(cdf_delta.clamp(min=1e-12))))


def p_mean_variance(tab, out, x_t, t, clip: bool = False):
    """p_mean_variance with LEARNED_RANGE: out = [eps | v] (B, 6, H, W); returns model mean, log-variance, x0."""
    eps, v = out[:, :3], out[:, 3:]
    frac = (v + 1) / 2
    logvar = frac * _ex(tab, "log_betas", t, v) + (1 - frac) * _ex(tab, "posterior_log_variance_clipped", t, v)
    x0 = _ex(tab, "sqrt_recip_alphas_cumprod", t, x_t) * x_t - _ex(tab, "sqrt_recipm1_alphas_cumprod", t, x_t) * eps
    if clip:
        x0 = x0.clamp(-1, 1)
    mean = _ex(tab, "posterior_mean_coef1", t, x_t) * x0 + _ex(tab, "posterior_mean_coef2", t, x_t) * x_t
    return mean, logvar, x0


def vb_terms_bpd(tab, out, x0, x_t, t):
    """_vb_terms_bpd with clip_denoised = False: per image, the KL of the posterior against the model (t > 0) or the
    decoder's negative log-likelihood (t = 0), mean over (C, H, W), in bits."""
    true_mean = _ex(tab, "posterior_mean_coef1", t, x_t) * x0 + _ex(tab, "posterior_mean_coef2", t, x_t) * x_t
    true_logvar = _ex(tab, "posterior_log_variance_clipped", t, x_t)
    mean, logvar, _ = p_mean_variance(tab, out, x_t, t)
    kl = normal_kl(true_mean, true_logvar, mean, logvar).mean(dim=(1, 2, 3)) / math.log(2.0)
    nll = -discretized_gaussian_log_likelihood(x0, mean, 0.5 * logvar).mean(dim=(1, 2, 3)) / math.log(2.0)
    return torch.where(torch.as_tensor(t).reshape(-1) == 0, nll, kl)


def hybrid_loss(tab, out, x0, x_t, t, noise, T: int = 1000):
    """training_losses (RESCALED_MSE, LEARNED_RANGE): mse(eps, noise) + T/1000 * vb(frozen_out), frozen_out =
    cat([eps.detach(), v]).  Returns (loss, mse per image, vb per image)."""
    frozen_out = torch.cat([out[:, :3].detach(), out[:, 3:]], dim=1)
    vb = vb_terms_bpd(tab, frozen_out, x0, x_t, t) * (T / 1000.0)
    mse = ((noise - out[:, :3]) ** 2).mean(dim=(1, 2, 3))
    return (mse + vb).mean(), mse, vb


def train_step_grads(O, cfg, flat: torch.Tensor, x0, t, noise, y=None, super_res: int = 0, T: int = 1000):
    """One forward + backward of a learned-variance training step: loss, mse, vb, the (B, 6, H, W) output and the flat
    parameter gradient.  x_t is the trainer's float32 q-sample (oracle.q_sample); super_res = f runs the
    super-resolution model on cat([x_t, condition(x0)]) (superres_oracle)."""
    flat = flat.detach().clone().requires_grad_(True)
    P = O.unflatten_params(cfg, flat)
    x_t = O.q_sample(x0, t, noise)
    x_in = x_t
    if super_res:
        import superres_oracle as SR
        x_in = torch.cat([x_t, SR.condition(x0, super_res)], 1)
    out = O.unet_forward(cfg, P, x_in, t, y)
    loss, mse, vb = hybrid_loss(tables(T), out, x0, x_t, t, noise, T)
    loss.backward()
    return loss.detach(), mse.mean().detach(), vb.mean().detach(), out.detach(), flat.grad.detach()


def train_steps(O, cfg, flat: torch.Tensor, batches, lr=1e-4):
    """n AdamW steps of the hybrid loss; `batches` = list of (x0, t, noise).  Returns the losses and the final flat."""
    m, v = torch.zeros_like(flat), torch.zeros_like(flat)
    losses = []
    for i, (x0, t, noise) in enumerate(batches, 1):
        loss, _, _, _, g = train_step_grads(O, cfg, flat, x0, t, noise)
        flat, m, v = O.adamw_step(flat, g, m, v, i, lr=lr)
        losses.append(float(loss))
    return losses, flat


def spaced_tables(T: int, timesteps) -> Dict[str, np.ndarray]:
    """The respaced chain's tables (SpacedDiffusion on beta'), with the ones LEARNED_RANGE reads."""
    tab = SO.spaced_tables(T, timesteps)
    pv = tab["posterior_variance"]
    tab["log_betas"] = np.log(tab["betas"])
    tab["posterior_log_variance_clipped"] = np.log(np.append(pv[1], pv[1:])) if len(pv) > 1 else np.log(pv)
    return tab


def p_sample_loop(model_fn, x, timesteps, clip: bool = True, noises=None, T: int = 1000):
    """p_sample_loop over the kept `timesteps` with the learned range: model_fn(x, t) returns the (B, 6, H, W) output at
    the ORIGINAL timestep t; noises[k] is the draw of iteration k (largest timestep first)."""
    tab = spaced_tables(T, timesteps)
    n = len(timesteps)
    with torch.no_grad():
        for k, i in enumerate(range(n - 1, -1, -1)):
            out = model_fn(x, int(timesteps[i]))
            # (_extract_into_tensor hands float32 coefficients to the float32 model output)
            mean, logvar, _ = p_mean_variance(_f32(tab), out, x, torch.full((x.shape[0],), i), clip)
            z = torch.zeros_like(x) if noises is None else noises[k]
            x = mean + float(i > 0) * torch.exp(0.5 * logvar) * z
    return x


def _f32(tab):
    return {k: (v.astype(np.float32) if isinstance(v, np.ndarray) and v.dtype == np.float64 else v)
            for k, v in tab.items()}
