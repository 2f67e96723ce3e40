"""Restatement of guided-diffusion's super-resolution model for the tests of the trainer's `super_res` option -- TEST
INFRASTRUCTURE ONLY (CPU, plain torch).  guided-diffusion's SuperResModel is UNetModel(in_channels * 2, ...) whose
forward(x, t, low_res) runs the U-Net on cat([x, F.interpolate(low_res, (H, W), mode="bilinear")], dim=1);
super_res_train.py derives low_res from the training batch with F.interpolate(batch, small_size, mode="area"), and
super_res_sample.py passes the user's low-res images.  The U-Net itself is oracle/unet_oracle.py's, built with
in_channels = 2 * C_in."""
from __future__ import annotations

import torch
import torch.nn.functional as F


def low_res_of(x0: torch.Tensor, f: int) -> torch.Tensor:
    """load_superres_data: the (B, C, H/f, W/f) condition of a training batch."""
    return F.interpolate(x0, (x0.shape[-2] // f, x0.shape[-1] // f), mode="area")


def upsample(low_res: torch.Tensor, H: int, W: int) -> torch.Tensor:
    """SuperResModel.forward: bilinear, align_corners = False, no antialias."""
    return F.interpolate(low_res, (H, W), mode="bilinear")


def condition(x0: torch.Tensor, f: int) -> torch.Tensor:
    """The conditioning channels of a training step on batch x0."""
    return upsample(low_res_of(x0, f), x0.shape[-2], x0.shape[-1])


def model_fn(O, cfg, P, low_res: torch.Tensor, y=None):
    """eps(x_t, t) of the super-resolution model with a fixed low-res batch, for ddpm_sample-style loops."""
    def fn(x, t):
        tt = torch.full((x.shape[0], 1), float(t)) if not torch.is_tensor(t) else t
        return O.unet_forward(cfg, P, torch.cat([x, upsample(low_res, x.shape[-2], x.shape[-1])], 1), tt, y)
    return fn


def train_step_grads(O, cfg, flat: torch.Tensor, x0, t, noise, f: int, y=None):
    """One forward + backward of a super-resolution training step: loss, eps prediction, flat parameter gradient and
    dL/d(x_t) (the gradient with respect to the first C_in input channels)."""
    flat = flat.detach().clone().requires_grad_(True)
    P = O.unflatten_params(cfg, flat)
    x_t = O.q_sample(x0, t, noise).detach().requires_grad_(True)
    out = O.unet_forward(cfg, P, torch.cat([x_t, condition(x0, f)], 1), t, y)
    loss = O.mse_loss(out, noise)
    loss.backward()
    return loss.detach(), out.detach(), flat.grad.detach(), x_t.grad.detach()


def ddpm_sample(O, cfg, P, low_res, x, t_start: int, t_end: int, noises, y=None, T: int = 1000):
    """oracle.ddpm_sample (generate.py's loop) with the conditioned model."""
    import numpy as np
    betas = torch.tensor(O.linear_betas(T), dtype=torch.float32)
    acp = torch.tensor(np.cumprod(1.0 - O.linear_betas(T)), dtype=torch.float32)
    eps_fn = model_fn(O, cfg, P, low_res, y)
    with torch.no_grad():
        for i, t in enumerate(range(t_start, t_end - 1, -1)):
            beta_t, alpha_t, alpha_t_1 = betas[t - 1], acp[t - 1], acp[t - 2]
            eps = eps_fn(x, t)
            mu = (x - (beta_t / torch.sqrt(1 - alpha_t)) * eps) / torch.sqrt(1 - beta_t)
            x = mu + torch.sqrt((1 - alpha_t_1) / (1 - alpha_t) * beta_t) * noises[i]
    return x
