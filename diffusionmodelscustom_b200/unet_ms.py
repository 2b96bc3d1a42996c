"""Drop-in ``UNet_downscale`` (Family D) — DDPM_clean_application/src/unet_ms.py:103-179 — backed by the native library.

Same constructor (``c_in, c_out, time_dim, interp_mode, img_size, device``), same ``state_dict`` keys
(``inc.double_conv.0.weight`` … ``outc.bias``) and the reference's ``forward(x, t, y)`` contract where ``y`` is the
low-resolution field that is bicubic-interpolated to ``x``'s size and concatenated (:156-160).  Parameter holders only;
the arithmetic runs in ``libb200ddpm.so`` (B2D_FAMILY_D program, csrc/family_d.cuh)."""
from __future__ import annotations

import torch
import torch.nn as nn

from . import _native as N
from .modules import NativeModel


class SelfAttention(nn.Module):
    def __init__(self, channels, size):
        super().__init__()
        self.channels = channels
        self.size = size
        self.mha = nn.MultiheadAttention(channels, 4, batch_first=True)
        self.ln = nn.LayerNorm([channels])
        self.ff_self = nn.Sequential(nn.LayerNorm([channels]), nn.Linear(channels, channels), nn.GELU(),
                                     nn.Linear(channels, channels))


class DoubleConv(nn.Module):
    def __init__(self, in_channels, out_channels, mid_channels=None, residual=False):
        super().__init__()
        self.residual = residual
        if not mid_channels:
            mid_channels = out_channels
        self.double_conv = nn.Sequential(
            nn.Conv2d(in_channels, mid_channels, kernel_size=3, padding=1, bias=False), nn.GroupNorm(1, mid_channels),
            nn.GELU(), nn.Conv2d(mid_channels, out_channels, kernel_size=3, padding=1, bias=False),
            nn.GroupNorm(1, out_channels))


class Down(nn.Module):
    def __init__(self, in_channels, out_channels, emb_dim=256):
        super().__init__()
        self.maxpool_conv = nn.Sequential(nn.MaxPool2d(2), DoubleConv(in_channels, in_channels, residual=True),
                                          DoubleConv(in_channels, out_channels))
        self.emb_layer = nn.Sequential(nn.SiLU(), nn.Linear(emb_dim, out_channels))


class Up(nn.Module):
    def __init__(self, in_channels, out_channels, emb_dim=256):
        super().__init__()
        self.up = nn.Upsample(scale_factor=2, mode="bilinear", align_corners=True)
        self.conv = nn.Sequential(DoubleConv(in_channels, in_channels, residual=True),
                                  DoubleConv(in_channels, out_channels, in_channels // 2))
        self.emb_layer = nn.Sequential(nn.SiLU(), nn.Linear(emb_dim, out_channels))


class UNet_downscale(NativeModel):
    _family = N.FAMILY_D

    def __init__(self, c_in=6, c_out=3, time_dim=256, interp_mode='bicubic', img_size=64, device="cuda"):
        super().__init__()
        if time_dim != 256:
            raise NotImplementedError("time_dim must be 256")
        if interp_mode not in N.INTERP_MODES:
            raise NotImplementedError(f"interp_mode must be one of {sorted(N.INTERP_MODES)} (F.interpolate modes built natively)")
        self.device = device
        self.time_dim = time_dim
        self.interp_mode = interp_mode
        self.c_in, self.c_out, self.img_size = c_in, c_out, img_size
        self.inc = DoubleConv(c_in, 64)
        self.down1 = Down(64, 128)
        self.sa1 = SelfAttention(128, img_size // 2)
        self.down2 = Down(128, 256)
        self.sa2 = SelfAttention(256, img_size // 4)
        self.down3 = Down(256, 256)
        self.sa3 = SelfAttention(256, img_size // 8)
        self.bot1 = DoubleConv(256, 256)
        self.bot3 = DoubleConv(256, 256)
        self.up1 = Up(512, 128)
        self.sa4 = SelfAttention(128, img_size // 4)
        self.up2 = Up(256, 64)
        self.sa5 = SelfAttention(64, img_size // 2)
        self.up3 = Up(128, 64)
        self.sa6 = SelfAttention(64, img_size)
        self.outc = nn.Conv2d(64, c_out, kernel_size=1)
        self._c_hr = None

    def _config(self, img_size, max_batch):
        if img_size != self.img_size:
            raise ValueError("UNet_downscale is resolution-specific: SelfAttention sizes are baked from img_size "
                             "(unet_ms.py:121-135)")
        return N.Config(family=N.FAMILY_D, img_size=img_size, max_batch=max_batch, c_hr=self._c_hr, c_out=self.c_out,
                        has_lsm=0, has_topo=0, cond_channels=self.c_in - self._c_hr, num_classes=0, n_heads=4, attn_ff=1,
                        debug_simt_conv=int(self.debug_simt_conv), interp_mode=N.INTERP_MODES[self.interp_mode])

    def _set_conditioning(self, h, B, y, cond_img, lsm_cond, topo_cond, stream):
        low = cond_img if cond_img is not None else y     # the low-res field is forward()'s third positional argument
        lowc = self._f32c(low, "y")
        key = (B, self._tkey(low))
        if key != self._cond_key:
            if lowc is not None and lowc.shape[1] != self.c_in - self._c_hr:
                raise ValueError("low-resolution field must have c_in - x.shape[1] channels")
            ch, cw = (0, 0) if lowc is None else (lowc.shape[-2], lowc.shape[-1])
            N.check(N.lib().b2d_set_conditioning(h, None, None, N.ptr(lowc), ch, cw, None, B, stream))
            self._cond_key = key
            self._cond_refs = (lowc, low)   # the original too: its address keys the cache and must not be recycled

    def _bind(self, x):
        c_hr = x.shape[1]
        if self._c_hr is not None and self._c_hr != c_hr:
            self._release()
        self._c_hr = c_hr

    @torch.no_grad()
    def forward(self, x, t, y=None, cond_img=None, lsm_cond=None, topo_cond=None):
        """Reference contract ``forward(x, t, y)`` (unet_ms.py:148); the extra positional slots exist only so that
        ``DiffusionUtils.sample``'s six-argument call (diffusion_DANRA_conditional.py:146) can drive this model too."""
        if x.dim() != 4 or x.shape[-1] != x.shape[-2]:
            raise ValueError("x must be [B, C, H, H]")
        self._bind(x)
        B, _, H, _ = x.shape
        h = self._ensure(B, H, x.device)
        xx = self._f32c(x, "x")
        with torch.cuda.device(x.device):
            stream = torch.cuda.current_stream().cuda_stream
            self._set_conditioning(h, B, y, cond_img, None, None, stream)
            out = torch.full((B, self.c_out, H, H), float("nan"), device=x.device, dtype=torch.float32)
            th = t.detach().to("cpu", torch.int64).contiguous()
            N.check(N.lib().b2d_forward(h, xx.data_ptr(), th.data_ptr(), out.data_ptr(), B, stream))
        return out

    @torch.no_grad()
    def native_sample(self, x, y, cond_img, lsm_cond, topo_cond, betas, alphas, alpha_hat, noise=None, seed=0,
                      sample_offset=0, noise_scale=1.0, ddim=None):
        self._bind(x)
        B, _, H, _ = x.shape
        h = self._ensure(B, H, x.device)
        if not (x.is_cuda and x.dtype == torch.float32 and x.is_contiguous()):
            raise N.NativeError("x must be a contiguous fp32 CUDA tensor")
        with torch.cuda.device(x.device):
            stream = torch.cuda.current_stream().cuda_stream
            self._set_schedule(h, betas, alphas, alpha_hat)
            self._set_sampler(h, ddim)
            self._set_conditioning(h, B, y, cond_img, None, None, stream)
            nz = self._f32c(noise, "noise")
            N.check(N.lib().b2d_sample(h, x.data_ptr(), N.ptr(nz), int(seed), int(sample_offset), float(noise_scale), B,
                                       stream))
            if nz is not None:
                torch.cuda.current_stream().synchronize()
        return x

    @torch.no_grad()
    def native_sample_host(self, x_host, y, cond_img, lsm_cond, topo_cond, betas, alphas, alpha_hat, device, noise=None,
                           seed=0, sample_offset=0, noise_scale=1.0, ddim=None):
        self._bind(x_host)
        B, _, H, _ = x_host.shape
        device = torch.device(device)
        h = self._ensure(B, H, device)
        low = cond_img if cond_img is not None else y
        hostc = lambda t: None if t is None else t.detach().to(torch.float32).contiguous()
        out, lowc, nz = hostc(x_host).clone(), hostc(low), hostc(noise)
        ch, cw = (0, 0) if lowc is None else (lowc.shape[-2], lowc.shape[-1])
        with torch.cuda.device(device):
            self._set_schedule(h, betas, alphas, alpha_hat)
            self._set_sampler(h, ddim)
            self._cond_key = None
            N.check(N.lib().b2d_sample_host(h, out.data_ptr(), None, None, N.ptr(lowc), ch, cw, None, N.ptr(nz), int(seed),
                                            int(sample_offset), float(noise_scale), B))
        return out

    @torch.no_grad()
    def profile_step(self, x, t, y=None, cond_img=None, lsm_cond=None, topo_cond=None, reps=5):
        import ctypes as C
        self._bind(x)
        B, _, H, _ = x.shape
        h = self._ensure(B, H, x.device)
        xx = self._f32c(x, "x")
        with torch.cuda.device(x.device):
            stream = torch.cuda.current_stream().cuda_stream
            self._set_conditioning(h, B, y, cond_img, None, None, stream)
            torch.cuda.synchronize()
            th = t.detach().to("cpu", torch.int64).contiguous()
            buf = (N.OpProfile * 512)()
            n = C.c_int32()
            N.check(N.lib().b2d_profile_step(h, xx.data_ptr(), th.data_ptr(), B, reps, buf, 512, C.byref(n)))
        return [dict(name=buf[i].name.decode(), klass=buf[i].klass.decode(), flops=buf[i].flops, bytes=buf[i].bytes,
                     ms=buf[i].ms) for i in range(n.value)]
