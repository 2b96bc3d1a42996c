"""fp64 oracle of the DDIM sampler (Song, Meng & Ermon 2021, eq. 12).  TEST INFRASTRUCTURE ONLY.

The reference has no DDIM, so this restatement is written from the equation (DESIGN §9) and pinned by identities instead of golden
files (tests/test_ddim_host.py): at eta = 1 with consecutive steps it is the reference's posterior step
(``oracle.ddpm_oracle.posterior_update``), and at eta = 0 it maps an exactly-noised field to the same field noised at t'.
"""
from __future__ import annotations

import torch


def ddim_step(x, eps, z, t, t_prev, eta, alpha_hat):
    """One DDIM step t -> t_prev (t_prev = -1: the final step, alpha_hat' = 1, returns x0_hat).  z already carries any
    noise_scale; it is ignored where sigma = 0."""
    ah = alpha_hat.double()
    a = ah[t]
    an = ah[t_prev] if t_prev >= 0 else torch.tensor(1.0, dtype=torch.float64)
    x, eps = x.double(), eps.double()
    x0 = (x - torch.sqrt(1 - a) * eps) / torch.sqrt(a)
    sigma = eta * torch.sqrt((1 - an) / (1 - a)) * torch.sqrt(1 - a / an)
    out = torch.sqrt(an) * x0 + torch.sqrt(torch.clamp(1 - an - sigma ** 2, min=0.0)) * eps
    if z is not None:
        out = out + sigma * z.double()
    return out


def ddim_coefficients(t, t_prev, eta, alpha_hat):
    """(cx, ce, sigma) with ddim_step(x, eps, z) = cx x + ce eps + sigma z, read off ddim_step itself on unit inputs."""
    one, zero = torch.ones(1, dtype=torch.float64), torch.zeros(1, dtype=torch.float64)
    return (float(ddim_step(one, zero, zero, t, t_prev, eta, alpha_hat)),
            float(ddim_step(zero, one, zero, t, t_prev, eta, alpha_hat)),
            float(ddim_step(zero, zero, one, t, t_prev, eta, alpha_hat)))


@torch.no_grad()
def ddim_sample(model_fn, x, timesteps, eta, alpha_hat, noise=None, generator=None, noise_scale=1.0):
    """DDIM over ``timesteps`` (tau_0 > ... > tau_{S-1}): S evaluations ``model_fn(x, t_long[B])`` on the fp64 state (an fp32
    model casts it).  ``noise`` [S,B,C,H,W] is indexed by step k; otherwise ``torch.randn`` with ``generator``.  z is drawn only
    where sigma != 0 (eta > 0, not the last step).  Returns x0 in fp64."""
    x = x.double()
    S = len(timesteps)
    for k, t in enumerate(timesteps):
        t_prev = timesteps[k + 1] if k + 1 < S else -1
        eps = model_fn(x, torch.full((x.shape[0],), int(t), dtype=torch.long))
        z = None
        if eta > 0 and t_prev >= 0:
            z = (noise[k] if noise is not None else torch.randn(x.shape, generator=generator)).double() * noise_scale
        x = ddim_step(x, eps, z, int(t), int(t_prev), eta, alpha_hat)
    return x
