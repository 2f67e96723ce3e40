"""Restatement of guided-diffusion's respaced sampling for the tests of ub_space_timesteps / ub_trainer_sample_spaced
-- TEST INFRASTRUCTURE ONLY (CPU, plain numpy / torch).  The U-Net itself comes from oracle/unet_oracle.py: the GPU
tests pass its unet_forward as `model_fn`."""
from __future__ import annotations

from typing import Dict, List

import numpy as np
import torch


# ------------------------------------------------------------------------------ respaced sampling (guided-diffusion)
# guided-diffusion's respace.py (space_timesteps, SpacedDiffusion) and gaussian_diffusion.py (GaussianDiffusion tables,
# p_sample, ddim_sample) as image_sample.py runs them for a model without learned sigma: model_var_type FIXED_LARGE,
# rescale_timesteps False.  The reference tree has no sampler of this kind, so nothing here is pinned to reference
# output; the restatement follows guided-diffusion's code, with one addition: negative section counts and specs that
# keep no timestep are refused (guided-diffusion accepts them and fails later).
def space_timesteps(T: int, spec: str) -> List[int]:
    """respace.space_timesteps, sorted.  Raises ValueError for a malformed or unsatisfiable spec."""
    if spec.startswith("ddim"):
        want = int(spec[len("ddim"):])
        for i in range(1, T):
            if len(range(0, T, i)) == want:
                return list(range(0, T, i))
        raise ValueError(f"cannot create exactly {want} steps with an integer stride")
    counts = [int(x) for x in spec.split(",")]
    size_per, extra = T // len(counts), T % len(counts)
    start, steps = 0, []
    for i, count in enumerate(counts):
        size = size_per + (1 if i < extra else 0)
        if count < 0 or size < count:
            raise ValueError(f"cannot divide section of {size} steps into {count}")
        frac = 1 if count <= 1 else (size - 1) / (count - 1)
        cur = 0.0
        for _ in range(count):
            steps.append(start + round(cur))
            cur += frac
        start += size
    if not steps:
        raise ValueError(f"spec {spec!r} keeps no timestep")
    return sorted(set(steps))


def spaced_tables(T: int, timesteps) -> Dict[str, np.ndarray]:
    """float64 tables of the respaced chain: SpacedDiffusion.__init__ (beta'_i = 1 - acp[t_i] / acp[t_{i-1}]) then
    GaussianDiffusion.__init__ on beta'.  The base betas are the trainer's linear schedule in float64."""
    scale = 1000 / T
    base = np.cumprod(1.0 - np.linspace(scale * 0.0001, scale * 0.02, T, dtype=np.float64))
    last, betas = 1.0, []
    for t in timesteps:
        betas.append(1 - base[t] / last)
        last = base[t]
    betas = np.array(betas, dtype=np.float64)
    acp = np.cumprod(1.0 - betas)
    acp_prev = np.append(1.0, acp[:-1])
    post_var = betas * (1.0 - acp_prev) / (1.0 - acp)
    return dict(timesteps=np.array(timesteps), betas=betas, alphas_cumprod=acp, alphas_cumprod_prev=acp_prev,
                sqrt_recip_alphas_cumprod=np.sqrt(1.0 / acp), sqrt_recipm1_alphas_cumprod=np.sqrt(1.0 / acp - 1),
                posterior_variance=post_var,
                posterior_mean_coef1=betas * np.sqrt(acp_prev) / (1.0 - acp),
                posterior_mean_coef2=(1.0 - acp_prev) * np.sqrt(1.0 - betas) / (1.0 - acp),
                fixed_large_log_variance=np.log(np.append(post_var[1], betas[1:])) if len(betas) > 1 else None)


def spaced_step(tab: Dict[str, np.ndarray], i: int, x: torch.Tensor, eps: torch.Tensor, sampler: str = "ddim",
                eta: float = 0.0, clip: bool = True, z: torch.Tensor | None = None) -> torch.Tensor:
    """One p_sample / ddim_sample update at spaced index i, coefficients extracted as float32 (_extract_into_tensor)."""
    f = lambda name: torch.tensor(float(tab[name][i]), dtype=torch.float32)
    x0 = f("sqrt_recip_alphas_cumprod") * x - f("sqrt_recipm1_alphas_cumprod") * eps   # _predict_xstart_from_eps
    if clip:
        x0 = x0.clamp(-1, 1)
    z = torch.zeros_like(x) if z is None else z
    nonzero = float(i > 0)
    if sampler == "ancestral":
        mean = f("posterior_mean_coef1") * x0 + f("posterior_mean_coef2") * x
        return mean + nonzero * torch.exp(0.5 * f("fixed_large_log_variance")) * z
    assert sampler == "ddim"
    eps = (f("sqrt_recip_alphas_cumprod") * x - x0) / f("sqrt_recipm1_alphas_cumprod")   # _predict_eps_from_xstart
    ab, ab_prev = f("alphas_cumprod"), f("alphas_cumprod_prev")
    sigma = eta * torch.sqrt((1 - ab_prev) / (1 - ab)) * torch.sqrt(1 - ab / ab_prev)
    mean = x0 * torch.sqrt(ab_prev) + torch.sqrt(1 - ab_prev - sigma ** 2) * eps
    return mean + nonzero * sigma * z


def spaced_sample(model_fn, x: torch.Tensor, timesteps, sampler: str = "ddim", eta: float = 0.0, clip: bool = True,
                  noises=None, T: int = 1000) -> torch.Tensor:
    """p_sample_loop / ddim_sample_loop over the kept `timesteps` (ascending), from spaced index n-1 down to 0.
    model_fn(x, t) returns eps at the ORIGINAL timestep t (an int); noises[k] is the draw of iteration k (largest
    timestep first; None: z = 0)."""
    tab = spaced_tables(T, timesteps)
    n = len(timesteps)
    with torch.no_grad():
        for k, i in enumerate(range(n - 1, -1, -1)):
            eps = model_fn(x, int(timesteps[i]))
            x = spaced_step(tab, i, x, eps, sampler, eta, clip, None if noises is None else noises[k])
    return x
