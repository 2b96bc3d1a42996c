"""Drop-in ``DiffusionUtils`` for the reference's sampling path.

``DiffusionUtils`` mirrors DDPM_DANRA_conditional/diffusion_DANRA_conditional.py:13-159 (v1: ``sample(x, model, y,
cond_img, lsm_cond, topo_cond)``); ``DiffusionUtilsV2`` mirrors DDPM_clean_application/src/diffusion_modules.py:6-186
(``sample(n, model, channels_hr, y, cond_img, lsm_cond, topo_cond, cfg_scale)``, proper cosine schedule, ``data_scaled``);
``Diffusion`` is the north_star alias (``Diffusion(noise_steps, beta_start, beta_end, img_size).sample(model, n, cond)``).

The schedule tables are built with the same torch expressions as the reference (they are part of the public attribute
surface: ``.betas/.alphas/.alpha_hat``).  The reverse loop itself runs natively: one captured CUDA graph per step, replayed
T-1 times, with the posterior update and (optionally) the Philox normal draws in ``posterior_update_kernel``.
``DiffusionUtils.sample_ddim`` (not in the reference) runs the DDIM sampler over S << T timesteps of the same schedule through the
same graphs, with ``ddim_update_kernel`` in place of the posterior update.
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np
import torch
import torch.nn as nn

from . import _native as N
from .modules import NativeModel


def ddim_coefficients(alpha_hat, t: int, t_prev: int, eta: float):
    """(cx, ce, sigma) of one DDIM step, x' = cx x + ce eps_hat + sigma z: a Python mirror, in double from the fp32 table, of
    ``ddim_coefficients()`` in csrc/elementwise.cuh (the function the native per-step table and ``b2d_op_ddim_update`` use).
    ``t_prev = -1`` is the final step (alpha_hat' = 1)."""
    a = float(np.float32(alpha_hat[t]))
    an = 1.0 if t_prev < 0 else float(np.float32(alpha_hat[t_prev]))
    sigma = float(np.float32(eta)) * math.sqrt((1.0 - an) / (1.0 - a)) * math.sqrt(max(0.0, 1.0 - a / an))
    cx = math.sqrt(an / a)
    ce = math.sqrt(max(0.0, 1.0 - an - sigma * sigma)) - cx * math.sqrt(1.0 - a)
    return float(np.float32(cx)), float(np.float32(ce)), float(np.float32(sigma))


class DiffusionUtils:
    def __init__(self, n_timesteps: int, beta_min: float, beta_max: float, device: str = 'cpu',
                 scheduler: str = 'linear'):
        assert scheduler in ['linear', 'cosine'], 'scheduler must be linear or cosine'
        self.n_timesteps = n_timesteps
        self.beta_min = beta_min
        self.beta_max = beta_max
        self.device = device
        self.scheduler = scheduler
        self.betas = self.betaSamples().to(self.device)
        self.alphas = 1 - self.betas
        self.alpha_hat = torch.cumprod(self.alphas, dim=0)
        self.data_scaled = False

    def betaSamples(self):
        """diffusion_DANRA_conditional.py:53-77 (the v1 'cosine' is a raised-cosine ramp of beta)."""
        if self.scheduler == 'linear':
            return torch.linspace(start=self.beta_min, end=self.beta_max, steps=self.n_timesteps).to(self.device)
        betas = []
        for i in reversed(range(self.n_timesteps)):
            T = self.n_timesteps - 1
            betas.append(self.beta_min + 0.5 * (self.beta_max - self.beta_min) * (1 + np.cos((i / T) * np.pi)))
        return torch.Tensor(betas).to(self.device)

    def sampleTimesteps(self, size: int):
        return torch.randint(low=1, high=self.n_timesteps, size=(size,)).to(self.device)

    def noiseImage(self, x: torch.Tensor, t: torch.LongTensor, *, noise: torch.Tensor = None, seed: int = None):
        """Forward process q(x_t | x_0) (diffusion_DANRA_conditional.py:85-103): returns (x_t, noise).

        CUDA tensors go through ONE fused kernel (``b2d_op_noise_image``): the gather of alpha_hat[t], both square roots, the
        normal draw (Philox, keyed by ``seed`` — taken from torch's global generator when omitted — or the injected ``noise``),
        the data_scaled factor and the blend, writing x_t and the noise in the same pass.  CPU tensors follow the reference's
        torch expressions (training-side convenience, not on the sampling path)."""
        assert len(x.shape) == 4, 'x must be a 4D tensor'
        scale = 0.005 if self.data_scaled else 1.0
        if x.is_cuda:
            xx = x.detach().to(torch.float32).contiguous()
            tt = t.detach().to(x.device, torch.int64).contiguous()
            ah = self.alpha_hat.detach().to(x.device, torch.float32).contiguous()
            nz = None if noise is None else noise.detach().to(x.device, torch.float32).contiguous()
            if seed is None:
                seed = int(torch.randint(0, 2 ** 62, (1,)).item())
            x_t, eps = torch.empty_like(xx), torch.empty_like(xx)
            with torch.cuda.device(x.device):
                N.check(N.lib().b2d_op_noise_image(xx.data_ptr(), tt.data_ptr(), ah.data_ptr(), N.ptr(nz), x_t.data_ptr(),
                                                   eps.data_ptr(), xx.shape[0], xx[0].numel(), int(seed), 0, float(scale),
                                                   torch.cuda.current_stream().cuda_stream))
            return x_t, eps
        alpha_hat_sqrts = torch.sqrt(self.alpha_hat[t])[:, None, None, None]
        one_minus_alpha_hat_sqrt = torch.sqrt(1 - self.alpha_hat[t])[:, None, None, None]
        noise = torch.randn_like(x).to(self.device) if noise is None else noise.clone()
        if self.data_scaled:
            noise *= 0.005
        return (alpha_hat_sqrts * x) + (one_minus_alpha_hat_sqrt * noise), noise

    # ------------------------------------------------------------------ reverse process
    def _run(self, x, model, y, cond_img, lsm_cond, topo_cond, noise, seed, sample_offset, ddim=None):
        assert len(x.shape) == 4, 'x must be a 4D tensor'
        if not x.is_cuda:
            raise N.NativeError("sampling runs only on CUDA (sm_100a); there is no CPU path")
        scale = 0.005 if self.data_scaled else 1.0
        x = x.detach().to(torch.float32).contiguous().clone()
        if seed is None:
            seed = int(torch.randint(0, 2 ** 62, (1,)).item())   # follows torch's global RNG state like randn_like would
        was_training = getattr(model, "training", False)
        model.eval()
        if isinstance(model, NativeModel):
            out = model.native_sample(x, y, cond_img, lsm_cond, topo_cond, self.betas, self.alphas, self.alpha_hat,
                                      noise=noise, seed=seed, sample_offset=sample_offset, noise_scale=scale, ddim=ddim)
        elif ddim is not None:
            out = self._foreign_ddim_loop(x, model, y, cond_img, lsm_cond, topo_cond, noise, seed, sample_offset, scale, ddim)
        else:
            out = self._foreign_model_loop(x, model, y, cond_img, lsm_cond, topo_cond, noise, seed, sample_offset, scale)
        return out, was_training

    def _foreign_model_loop(self, x, model, y, cond_img, lsm_cond, topo_cond, noise, seed, sample_offset, scale):
        """Any other callable eps-model: python loop over the model, native posterior-update kernel."""
        L = N.lib()
        dev = x.device
        betas, alphas, ahat = (v.detach().to(dev, torch.float32).contiguous() for v in (self.betas, self.alphas, self.alpha_hat))
        B = x.shape[0]
        per = x[0].numel()
        with torch.no_grad(), torch.cuda.device(dev):
            for i in reversed(range(1, self.n_timesteps)):
                t = torch.full((B,), i, dtype=torch.long, device=dev)
                eps = model(x, t, y, cond_img, lsm_cond, topo_cond).to(torch.float32).contiguous()
                z = None if noise is None else noise[i].to(dev, torch.float32).contiguous()
                N.check(L.b2d_op_posterior_update(x.data_ptr(), eps.data_ptr(), N.ptr(z), betas.data_ptr(),
                                                  alphas.data_ptr(), ahat.data_ptr(), i, B, per, int(seed),
                                                  int(sample_offset), float(scale),
                                                  torch.cuda.current_stream().cuda_stream))
        return x

    def _foreign_ddim_loop(self, x, model, y, cond_img, lsm_cond, topo_cond, noise, seed, sample_offset, scale, ddim):
        """Any other callable eps-model under DDIM: python loop over the model, native DDIM-update kernel."""
        L = N.lib()
        dev = x.device
        ts, eta = ddim
        ahat = self.alpha_hat.detach().to(dev, torch.float32).contiguous()
        B = x.shape[0]
        per = x[0].numel()
        with torch.no_grad(), torch.cuda.device(dev):
            for k, t in enumerate(ts):
                t_prev = ts[k + 1] if k + 1 < len(ts) else -1
                tt = torch.full((B,), t, dtype=torch.long, device=dev)
                eps = model(x, tt, y, cond_img, lsm_cond, topo_cond).to(torch.float32).contiguous()
                z = None if noise is None else noise[k].to(dev, torch.float32).contiguous()
                N.check(L.b2d_op_ddim_update(x.data_ptr(), eps.data_ptr(), N.ptr(z), ahat.data_ptr(), self.n_timesteps, t,
                                             t_prev, float(eta), B, per, int(seed), int(sample_offset), float(scale),
                                             torch.cuda.current_stream().cuda_stream))
        return x

    def ddim_timesteps(self, steps: int):
        """Default DDIM sequence for ``steps`` = S evaluations: tau_k = (T-1) - floor(k (T-2) / (S-1)), k = 0 ... S-1, so
        tau_0 = T-1 and tau_{S-1} = 1 ([T-1] for S = 1).  Integer arithmetic: strictly decreasing for every 2 <= S <= T-1."""
        T = self.n_timesteps
        steps = int(steps)
        if not 1 <= steps <= T - 1:
            raise ValueError(f"steps must lie in [1, {T - 1}] (T = {T}), got {steps}")
        if steps == 1:
            return [T - 1]
        return [(T - 1) - (k * (T - 2)) // (steps - 1) for k in range(steps)]

    def _ddim_plan(self, steps, eta, timesteps):
        """(sequence, eta) of a DDIM run: ``timesteps`` if given (validated), else the default sequence for ``steps``."""
        eta = float(eta)
        if not 0.0 <= eta <= 1.0:
            raise ValueError(f"eta must lie in [0, 1], got {eta}")
        if timesteps is None:
            return self.ddim_timesteps(steps), eta
        ts = [int(t) for t in (timesteps.tolist() if isinstance(timesteps, torch.Tensor) else timesteps)]
        T = self.n_timesteps
        if not ts:
            raise ValueError("timesteps is empty")
        if any(not 1 <= t <= T - 1 for t in ts):
            raise ValueError(f"timesteps must lie in [1, {T - 1}] (T = {T})")
        if any(b >= a for a, b in zip(ts, ts[1:])):
            raise ValueError("timesteps must be strictly decreasing")
        return ts, eta

    def sample_ddim(self, x: torch.Tensor, model: nn.Module, y: torch.Tensor = None, cond_img: torch.Tensor = None,
                    lsm_cond: torch.Tensor = None, topo_cond: torch.Tensor = None, *, steps: int = 50, eta: float = 0.0,
                    timesteps=None, noise: torch.Tensor = None, seed: int = None, sample_offset: int = 0):
        """DDIM (Song, Meng & Ermon 2021, eq. 12) with this object's trained-DDPM schedule: x is x_T, returns x_0 after S model
        evaluations instead of T-1.  Not in the reference.

        ``timesteps`` is a strictly decreasing sequence in [1, T-1]; without it the default ``ddim_timesteps(steps)`` is used.
        ``eta`` = 0 is the deterministic sampler, 1 has the DDPM posterior variance for consecutive steps.  ``noise``
        [S,B,C,H,W] injects z indexed by step k; otherwise z is drawn in-kernel from the same Philox stream as ``sample``,
        with the step slot set to the timestep.  The data_scaled factor multiplies z as in ``sample``; no x_0 clipping."""
        out, _ = self._run(x, model, y, cond_img, lsm_cond, topo_cond, noise, seed, sample_offset,
                           ddim=self._ddim_plan(steps, eta, timesteps))
        return out

    def sample(self, x: torch.Tensor, model: nn.Module, y: torch.Tensor = None, cond_img: torch.Tensor = None,
               lsm_cond: torch.Tensor = None, topo_cond: torch.Tensor = None, *, noise: torch.Tensor = None,
               seed: int = None, sample_offset: int = 0):
        """v1 contract (diffusion_DANRA_conditional.py:105-159): x is x_T, returns x_0; i = T-1 … 1.

        Keyword-only extras (not in the reference): ``noise`` [T,B,C,H,W] injects host-generated z_i (parity runs);
        ``seed``/``sample_offset`` key the in-kernel Philox stream by global sample index (multi-GPU sharding)."""
        out, _ = self._run(x, model, y, cond_img, lsm_cond, topo_cond, noise, seed, sample_offset)
        return out


    def sample_host(self, x: torch.Tensor, model: nn.Module, y=None, cond_img=None, lsm_cond=None, topo_cond=None, *,
                    noise=None, seed: int = None, sample_offset: int = 0, device="cuda"):
        """Same contract as ``sample`` with HOST tensors in and out — what the reference's generation scripts do around
        the call (``x.to(device)`` … ``generated.detach().cpu()``, generation_DANRA_conditional.py:389-426) — as ONE native
        call: pinned/pageable host buffers -> H2D -> graph-replayed loop -> D2H."""
        if not isinstance(model, NativeModel):
            raise TypeError("sample_host needs a native model (DiffusionNet / UNet_downscale of this package)")
        if seed is None:
            seed = int(torch.randint(0, 2 ** 62, (1,)).item())
        model.eval()
        return model.native_sample_host(x, y, cond_img, lsm_cond, topo_cond, self.betas, self.alphas, self.alpha_hat,
                                        device, noise=noise, seed=seed, sample_offset=sample_offset,
                                        noise_scale=0.005 if self.data_scaled else 1.0)


class DiffusionUtilsV2(DiffusionUtils):
    def __init__(self, n_timesteps: int = 1000, beta_min: float = 1e-4, beta_max: float = 0.02, device: str = 'cpu',
                 scheduler: str = 'linear', img_size: int = 64, data_scaled: bool = False):
        self.img_size = img_size
        super().__init__(n_timesteps, beta_min, beta_max, device, scheduler)
        self.data_scaled = data_scaled

    def betaSamples(self):
        """src/diffusion_modules.py:50-69 (Nichol–Dhariwal cosine, clipped to [1e-4, 0.9999])."""
        if self.scheduler == 'linear':
            return torch.linspace(start=self.beta_min, end=self.beta_max, steps=self.n_timesteps).to(self.device)
        t = torch.linspace(0, self.n_timesteps, self.n_timesteps + 1)
        ft = torch.cos(((t / self.n_timesteps + 0.008) / 1.008) * np.pi / 2) ** 2
        alphat = ft / ft[0]
        betat = 1 - alphat[1:] / alphat[:-1]
        return torch.clip(betat, 0.0001, 0.9999).to(self.device)

    def sample(self, n: int, model: nn.Module, channels_hr: int, y=None, cond_img=None, lsm_cond=None, topo_cond=None,
               cfg_scale: float = 0.0, *, x_T: torch.Tensor = None, noise: torch.Tensor = None, seed: int = None,
               sample_offset: int = 0):
        """v2 contract (src/diffusion_modules.py:101-186): draws x_T itself, optional x0.005 scaling, model.train() at exit.
        cfg_scale > 0 is rejected: in the reference it feeds fewer channels than conv1 expects and cannot run
        (SURVEY.md §2 row 6)."""
        if cfg_scale > 0:
            raise NotImplementedError("classifier-free guidance is not runnable in the reference either (conv1 channel mismatch)")
        dev = self.device
        if x_T is None:
            x_T = torch.randn((n, channels_hr, self.img_size, self.img_size)).to(dev)
            if self.data_scaled:
                x_T = x_T * 0.005
        mv = lambda v: None if v is None else v.to(dev)
        out, _ = self._run(x_T.to(dev), model, mv(y), mv(cond_img), mv(lsm_cond), mv(topo_cond), noise, seed, sample_offset)
        model.train()
        return out


class Diffusion(DiffusionUtilsV2):
    """north_star spelling: Diffusion(noise_steps, beta_start, beta_end, img_size).sample(model, n, cond)."""

    def __init__(self, noise_steps: int = 1000, beta_start: float = 1e-4, beta_end: float = 0.02, img_size: int = 64,
                 device: str = "cuda"):
        super().__init__(noise_steps, beta_start, beta_end, device, 'linear', img_size)

    def sample(self, model, n, cond=None, **kw):
        """cond: dict with any of y / cond_img / lsm_cond / topo_cond (or a bare tensor = cond_img)."""
        c = cond if isinstance(cond, dict) else {"cond_img": cond}
        ch = model.encoder.hr_channels if hasattr(model, "encoder") else 1
        return DiffusionUtilsV2.sample(self, n, model, ch, c.get("y"), c.get("cond_img"), c.get("lsm_cond"),
                                       c.get("topo_cond"), **kw)
