"""Drop-in model classes for the reference's sampling path (Family R), backed by the native B200 library.

Mirrors the constructor signatures, attribute names and ``state_dict`` keys of
``DDPM_DANRA_conditional/modules_DANRA_conditional.py`` (``Encoder`` :117-199, ``DecoderBlock`` :349-422,
``Decoder`` :465-569, ``DiffusionNet`` :571-616) — and therefore of the byte-near duplicate
``modules_DANRA_flexible.py`` (SURVEY.md §0.3).  The ``nn.Module`` tree below only *holds parameters* (so that
``load_state_dict`` / ``state_dict`` / ``.to()`` behave as in the reference); all arithmetic of
``DiffusionNet.forward`` runs in ``libb200ddpm.so`` through the C ABI of ``include/b200ddpm.h``.
There is no PyTorch/CPU execution path: calling ``forward`` without the CUDA library or a CUDA tensor raises.
"""
from __future__ import annotations

import ctypes as C
from typing import Iterable, Optional

import torch
import torch.nn as nn

from . import _native as N

FMAP_CHANNELS = [64, 64, 128, 256, 512]   # modules_DANRA_conditional.py:170


class SinusoidalEmbedding(nn.Module):
    """Parameter-free placeholder (modules_DANRA_conditional.py:17-63); evaluated inside temb_project_kernel."""

    def __init__(self, dim_size, n: int = 10000):
        assert dim_size % 2 == 0, 'dim_size must be even'
        super().__init__()
        self.dim_size = dim_size
        self.n = n


class ImageSelfAttention(nn.Module):
    """Parameter holder for modules_DANRA_conditional.py:67-110 (keys ``layernorm.*``, ``attention.*``)."""

    def __init__(self, input_channels: int, n_heads: int):
        super().__init__()
        self.input_channels = input_channels
        self.n_heads = n_heads
        self.layernorm = nn.LayerNorm(self.input_channels)
        self.attention = nn.MultiheadAttention(self.input_channels, self.n_heads, batch_first=True)


class _BasicBlock(nn.Module):
    """Parameter holder with torchvision ``BasicBlock`` keys (conv1, bn1, conv2, bn2, downsample.{0,1})."""

    def __init__(self, cin, cout, stride):
        super().__init__()
        self.conv1 = nn.Conv2d(cin, cout, 3, stride, 1, bias=False)
        self.bn1 = nn.BatchNorm2d(cout)
        self.conv2 = nn.Conv2d(cout, cout, 3, 1, 1, bias=False)
        self.bn2 = nn.BatchNorm2d(cout)
        self.downsample = None
        if stride != 1 or cin != cout:
            self.downsample = nn.Sequential(nn.Conv2d(cin, cout, 1, stride, bias=False), nn.BatchNorm2d(cout))
        for m in (self.conv1, self.conv2):
            nn.init.kaiming_normal_(m.weight, mode="fan_out", nonlinearity="relu")


def _time_projection(time_embedding, ch):
    return nn.Sequential(nn.SiLU(), nn.Linear(time_embedding, ch))


class Encoder(nn.Module):
    """ResNet-18-shaped encoder of the reference (modules_DANRA_conditional.py:117-312); parameter holder."""

    def __init__(self, input_channels: int, time_embedding: int, block=None, block_layers: list = [2, 2, 2, 2],
                 n_heads: int = 4, num_classes: int = None, lsm_tensor=None, topo_tensor=None, cond_on_img=False,
                 cond_img_dim=None):
        super().__init__()
        if list(block_layers) != [2, 2, 2, 2]:
            raise NotImplementedError("only block_layers=[2,2,2,2] (BasicBlock) is built; the reference's Decoder "
                                      "asserts against those widths too (modules_DANRA_conditional.py:442)")
        if time_embedding != 256:
            raise NotImplementedError("time_embedding must be 256 (every reference driver uses 256)")
        self.block_layers = block_layers
        self.time_embedding = time_embedding
        self.hr_channels = input_channels
        self.input_channels = input_channels
        self.n_heads = n_heads
        self.num_classes = num_classes
        self.cond_channels = 0
        if lsm_tensor is not None:
            self.register_buffer('lsm', lsm_tensor)
            self.input_channels += 1
        if topo_tensor is not None:
            self.register_buffer('elevation', topo_tensor)
            self.input_channels += 1
        if cond_on_img:
            self.input_channels += cond_img_dim[0]
            self.cond_channels = cond_img_dim[0]
        self.sinusiodal_embedding = SinusoidalEmbedding(self.time_embedding)
        self.bn1 = nn.BatchNorm2d(64)
        cin = 64
        for li, cout in enumerate(FMAP_CHANNELS[1:], start=1):
            setattr(self, f"layer{li}", nn.Sequential(_BasicBlock(cin, cout, 1 if li == 1 else 2),
                                                      _BasicBlock(cout, cout, 1)))
            cin = cout
        self.time_projection_layers = nn.ModuleList([_time_projection(time_embedding, ch) for ch in FMAP_CHANNELS])
        self.attention_layers = nn.ModuleList([ImageSelfAttention(ch, n_heads) for ch in FMAP_CHANNELS])
        self.conv1 = nn.Conv2d(self.input_channels, 64, kernel_size=(8, 8), stride=(2, 2), padding=(3, 3), bias=False)
        self.conv2 = nn.Conv2d(64, 64, kernel_size=(8, 8), stride=(2, 2), padding=(3, 3), bias=False)
        if num_classes is not None:
            self.label_emb = nn.Embedding(num_classes, time_embedding)

    @torch.no_grad()
    def forward(self, x: torch.Tensor, t: torch.Tensor, y: Optional[torch.Tensor] = None, cond_img: Optional[torch.Tensor] = None,
                lsm_cond: Optional[torch.Tensor] = None, topo_cond: Optional[torch.Tensor] = None):
        """``Encoder.forward`` on its own (modules_DANRA_conditional.py:213-312): returns ``(fmap1, ..., fmap5)`` as fp32 NCHW
        CUDA tensors.  Runs the encoder half of the native program (b2d_encoder_forward); inside ``DiffusionNet`` the feature maps
        never leave their fp16 NHWC buffers."""
        if getattr(self, "_runner", None) is None:
            object.__setattr__(self, "_runner", _HalfRunner(encoder=self))
        return self._runner.encode(x, t, y, cond_img, lsm_cond, topo_cond)


class DecoderBlock(nn.Module):
    """Parameter holder for modules_DANRA_conditional.py:349-460."""

    def __init__(self, input_channels: int, output_channels: int, time_embedding: int, upsample_scale: int = 2,
                 activation: nn.Module = nn.ReLU, compute_attn: bool = True, n_heads: int = 4):
        super().__init__()
        if upsample_scale != 2:
            raise NotImplementedError("upsample_scale must be 2")
        self.input_channels = input_channels
        self.output_channels = output_channels
        self.upsample_scale = upsample_scale
        self.time_embedding = time_embedding
        self.compute_attn = compute_attn
        self.n_heads = n_heads
        self.attention = ImageSelfAttention(output_channels, n_heads) if compute_attn else nn.Identity()
        self.sinusiodal_embedding = SinusoidalEmbedding(self.time_embedding)
        self.time_projection_layer = _time_projection(time_embedding, output_channels)
        self.transpose = nn.ConvTranspose2d(input_channels, input_channels, kernel_size=2, stride=2)
        self.instance_norm1 = nn.InstanceNorm2d(input_channels)
        self.conv = nn.Conv2d(input_channels, output_channels, kernel_size=3, stride=1, padding=1)
        self.instance_norm2 = nn.InstanceNorm2d(output_channels)
        self.activation = activation()


class Decoder(nn.Module):
    """Parameter holder for modules_DANRA_conditional.py:465-569."""

    def __init__(self, last_fmap_channels: int, output_channels: int, time_embedding: int, first_fmap_channels: int = 64,
                 n_heads: int = 4):
        super().__init__()
        if last_fmap_channels != 512 or first_fmap_channels != 64:
            raise NotImplementedError("Decoder widths are fixed to 512 -> 64 by the encoder (SURVEY.md §0.3)")
        self.last_fmap_channels = last_fmap_channels
        self.output_channels = output_channels
        self.time_embedding = time_embedding
        self.first_fmap_channels = first_fmap_channels
        self.n_heads = n_heads
        self.residual_layers = self.make_layers()
        self.final_layer = DecoderBlock(self.residual_layers[-1].input_channels, self.output_channels,
                                        time_embedding=self.time_embedding, activation=nn.Identity, compute_attn=False,
                                        n_heads=self.n_heads)
        self.final_layer.instance_norm2 = nn.Identity()

    def make_layers(self, n: int = 4):
        layers = []
        for i in range(n):
            in_ch = self.last_fmap_channels if i == 0 else layers[i - 1].output_channels
            out_ch = in_ch // 2 if i != (n - 1) else self.first_fmap_channels
            layers.append(DecoderBlock(in_ch, out_ch, time_embedding=self.time_embedding, compute_attn=True,
                                       n_heads=self.n_heads))
        return nn.ModuleList(layers)

    @torch.no_grad()
    def forward(self, *fmaps, t: Optional[torch.Tensor] = None):
        """``Decoder.forward(*fmaps, t=t)`` on its own (modules_DANRA_conditional.py:512-536): five fp32 NCHW CUDA feature maps
        (fmap1 ... fmap5 in the encoder's order) and the time steps -> the predicted noise (b2d_decoder_forward)."""
        if len(fmaps) != 5:
            raise ValueError("Decoder.forward expects the five encoder feature maps")
        if t is None:
            raise ValueError("Decoder.forward needs t (the decoder blocks embed it, modules_DANRA_conditional.py:449)")
        if getattr(self, "_runner", None) is None:
            object.__setattr__(self, "_runner", _HalfRunner(decoder=self))
        return self._runner.decode(fmaps, t)


class NativeModel(nn.Module):
    """Owns the opaque ``b2d_handle`` of a model and keeps it in sync with the module's parameters."""

    _family = N.FAMILY_R

    def __init__(self):
        super().__init__()
        self._h = None
        self._h_key = None
        self._w_version = None
        self._cond_key = None
        self._sched_key = None
        self._max_batch = 0
        self._refresh_epoch = 0
        self.debug_simt_conv = False

    # -- to be provided by subclasses
    def _config(self, img_size: int, max_batch: int) -> N.Config:
        raise NotImplementedError

    def _weights_version(self):
        """Identity of the parameter set the native handle was packed from.  ``tensor._version`` misses in-place writes through
        ``.data`` (``m.bias.data.fill_()``, EMA updates — the reference's own scripts do both), so the key also carries a CONTENT
        fingerprint: the L2 norm of every floating-point parameter/buffer (a handful of fused ``_foreach_norm`` kernels and one
        small D2H copy per call).  ``refresh_weights()`` forces a re-pack explicitly."""
        ts = [t for t in list(self.parameters()) + list(self.buffers()) if t.dtype.is_floating_point and t.numel() > 0]
        ident = tuple(int(t._version) for t in ts) + tuple(t.data_ptr() for t in ts) + (self._refresh_epoch,)
        if not ts:
            return ident
        fp = torch.stack(torch._foreach_norm([t.detach() for t in ts])).to("cpu", torch.float64)
        return ident + (fp.numpy().tobytes(),)

    def refresh_weights(self):
        """Drop the native handle so that the next call re-packs the current parameter values (use after any weight update the
        automatic detection could miss)."""
        self._refresh_epoch += 1
        self._release()

    def load_state_dict(self, *a, **k):
        r = super().load_state_dict(*a, **k)
        self.refresh_weights()
        return r

    @staticmethod
    def saturation_count(reset: bool = False) -> int:
        """fp32->fp16 conversions clamped at +-65504 since the last reset (0 = the fp16 activation storage never clipped)."""
        return int(N.lib().b2d_saturation_count(int(reset)))

    def _native_state_dict(self):
        """The reference-keyed state_dict handed to b2d_load_weights (stand-alone Encoder / Decoder runners add placeholders)."""
        return self.state_dict()

    def _release(self):
        if self._h is not None:
            N.lib().b2d_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self._release()
        except Exception:
            pass

    def _ensure(self, batch: int, img_size: int, device):
        if device.type != "cuda":
            raise N.NativeError("DiffusionNet/UNet_downscale run only on CUDA (sm_100a); there is no CPU path. "
                                "Move the inputs to a B200 device.")
        ver = self._weights_version()
        key = (img_size, device.index, bool(self.debug_simt_conv))
        if self._h is not None and (self._h_key != key or self._w_version != ver or batch > self._max_batch):
            self._release()
        if self._h is None:
            L = N.lib()
            self._max_batch = max(batch, self._max_batch)
            cfg = self._config(img_size, self._max_batch)
            h = C.c_void_p()
            with torch.cuda.device(device):
                N.check(L.b2d_create(C.byref(cfg), C.byref(h)))
                self._h = h
                sd = {k: v.detach().to("cpu", torch.float32).contiguous() for k, v in self._native_state_dict().items()
                      if v.dtype.is_floating_point}
                arr = (N.Tensor * len(sd))()
                for i, (k, v) in enumerate(sd.items()):
                    arr[i].name = k.encode()
                    arr[i].data = v.data_ptr()
                    arr[i].ndim = v.dim()
                    for d in range(v.dim()):
                        arr[i].shape[d] = v.shape[d]
                N.check(L.b2d_load_weights(self._h, arr, len(sd)))
            self._h_key, self._w_version = key, ver
            self._cond_key = None
            self._sched_key = None
        return self._h

    @staticmethod
    def _f32c(t, name):
        if t is None:
            return None
        if not t.is_cuda:
            raise N.NativeError(f"{name} must be a CUDA tensor (no CPU path)")
        return t.detach().to(torch.float32).contiguous()

    @staticmethod
    def _tkey(t):
        return None if t is None else (t.data_ptr(), int(t._version), tuple(t.shape))

    def debug_read(self, name: str, batch: int):
        """Bring-up aid: named intermediate activation of the last evaluation as NCHW fp32 (CPU)."""
        buf = torch.empty(batch * 128 * 128 * 64, dtype=torch.float32)
        c, hw = C.c_int32(), C.c_int32()
        N.check(N.lib().b2d_debug_read(self._h, name.encode(), buf.data_ptr(), buf.numel(), C.byref(c), C.byref(hw)))
        n = batch * hw.value * hw.value * c.value
        return buf[:n].reshape(batch, hw.value, hw.value, c.value).permute(0, 3, 1, 2).contiguous()

    def _set_schedule(self, h, betas, alphas, alpha_hat):
        skey = (betas.data_ptr(), int(betas._version), len(betas))
        if skey != self._sched_key:
            b, a, ah = (v.detach().to("cpu", torch.float32).contiguous() for v in (betas, alphas, alpha_hat))
            N.check(N.lib().b2d_set_schedule(h, b.data_ptr(), a.data_ptr(), ah.data_ptr(), len(b)))
            self._sched_key = skey

    def _set_sampler(self, h, ddim=None):
        """Sampler mode of the handle for the next native loop: ``None`` = the reference DDPM loop, ``(timesteps, eta)`` = DDIM
        over that sequence (b2d_set_timesteps).  Every native sampling call sets it, so no mode leaks from one call to the next."""
        if ddim is None:
            N.check(N.lib().b2d_set_timesteps(h, None, 0, 0.0))
            return
        ts, eta = ddim
        arr = (C.c_int32 * len(ts))(*[int(t) for t in ts])
        N.check(N.lib().b2d_set_timesteps(h, arr, len(ts), float(eta)))

    def launch_count(self) -> int:
        return 0 if self._h is None else int(N.lib().b2d_last_launch_count(self._h))


class DiffusionNet(NativeModel):
    """``DiffusionNet(encoder, decoder)`` of modules_DANRA_conditional.py:571-616, evaluated natively.

    ``forward(x, t, y, cond_img, lsm_cond, topo_cond)`` keeps the positional contract the sampler relies on
    (diffusion_DANRA_conditional.py:146)."""

    def __init__(self, encoder: Encoder, decoder: Decoder, lsm_tensor=None, topo_tensor=None, cond_on_img=False,
                 cond_img_dim=None):
        super().__init__()
        self.encoder = encoder
        self.decoder = decoder

    def _config(self, img_size, max_batch):
        e, d = self.encoder, self.decoder
        return N.Config(family=N.FAMILY_R, img_size=img_size, max_batch=max_batch, c_hr=e.hr_channels,
                        c_out=d.output_channels, has_lsm=int(self._has_lsm()), has_topo=int(self._has_topo()),
                        cond_channels=e.cond_channels, num_classes=e.num_classes or 0, n_heads=e.n_heads, attn_ff=0,
                        debug_simt_conv=int(self.debug_simt_conv))

    def _has_lsm(self):
        # modules_DANRA_conditional.py:228 (hasattr(self,'lsm')) / src/unet.py:232 (cond_on_lsm => lsm_cond is passed)
        return hasattr(self.encoder, "lsm") or getattr(self.encoder, "cond_on_lsm", False)

    def _has_topo(self):
        return hasattr(self.encoder, "elevation") or getattr(self.encoder, "cond_on_topo", False)

    def _set_conditioning(self, h, B, y, cond_img, lsm_cond, topo_cond, stream):
        lsm = self._f32c(lsm_cond, "lsm_cond") if self._has_lsm() else None
        topo = self._f32c(topo_cond, "topo_cond") if self._has_topo() else None
        cond = self._f32c(cond_img, "cond_img")
        if self._has_lsm() and lsm is None:
            raise ValueError("model was built with lsm conditioning: lsm_cond is required")
        if self._has_topo() and topo is None:
            raise ValueError("model was built with topography conditioning: topo_cond is required")
        yy = None
        if y is not None:
            if not y.is_cuda:
                raise N.NativeError("y must be a CUDA tensor (no CPU path)")
            yy = y.detach().to(torch.int64).contiguous()
        key = (B, self._tkey(lsm_cond), self._tkey(topo_cond), self._tkey(cond_img), self._tkey(y))
        if key != self._cond_key:
            N.check(N.lib().b2d_set_conditioning(h, N.ptr(lsm), N.ptr(topo), N.ptr(cond), 0, 0, N.ptr(yy), B, stream))
            self._cond_key = key
            # keep the staging copies alive until consumed AND the caller's tensors alive while they key the cache: a freed
            # original's address can be recycled by the caching allocator for the next batch (same ptr/version/shape)
            self._cond_refs = (lsm, topo, cond, yy, lsm_cond, topo_cond, cond_img, y)

    @torch.no_grad()
    def forward(self, x: torch.Tensor, t: torch.Tensor, y: Optional[torch.Tensor] = None,
                cond_img: Optional[torch.Tensor] = None, lsm_cond: Optional[torch.Tensor] = None,
                topo_cond: Optional[torch.Tensor] = None):
        if x.dim() != 4 or x.shape[-1] != x.shape[-2]:
            raise ValueError("x must be [B, C, H, H]")
        B, _, H, _ = x.shape
        h = self._ensure(B, H, x.device)
        xx = self._f32c(x, "x")
        with torch.cuda.device(x.device):
            stream = torch.cuda.current_stream().cuda_stream
            self._set_conditioning(h, B, y, cond_img, lsm_cond, topo_cond, stream)
            out = torch.full((B, self.decoder.output_channels, H, H), float("nan"), device=x.device, dtype=torch.float32)
            th = t.detach().to("cpu", torch.int64).contiguous()
            N.check(N.lib().b2d_forward(h, xx.data_ptr(), th.data_ptr(), out.data_ptr(), B, stream))
        return out

    @torch.no_grad()
    def native_sample(self, x, y, cond_img, lsm_cond, topo_cond, betas, alphas, alpha_hat, noise=None, seed=0,
                      sample_offset=0, noise_scale=1.0, ddim=None):
        """Whole reverse loop on the device (CUDA graph); x is updated in place and returned."""
        B, _, H, _ = x.shape
        h = self._ensure(B, H, x.device)
        if not (x.is_cuda and x.dtype == torch.float32 and x.is_contiguous()):
            raise N.NativeError("x must be a contiguous fp32 CUDA tensor")
        with torch.cuda.device(x.device):
            stream = torch.cuda.current_stream().cuda_stream
            self._set_schedule(h, betas, alphas, alpha_hat)
            self._set_sampler(h, ddim)
            self._set_conditioning(h, B, y, cond_img, lsm_cond, topo_cond, stream)
            nz = self._f32c(noise, "noise")
            N.check(N.lib().b2d_sample(h, x.data_ptr(), N.ptr(nz), int(seed), int(sample_offset), float(noise_scale), B,
                                       stream))
            if nz is not None:
                torch.cuda.current_stream().synchronize()   # nz staging copy must outlive the queued work
        return x

    @torch.no_grad()
    def native_sample_host(self, x_host, y, cond_img, lsm_cond, topo_cond, betas, alphas, alpha_hat, device, noise=None,
                           seed=0, sample_offset=0, noise_scale=1.0, ddim=None):
        """End-to-end entry on HOST tensors (b2d_sample_host): H2D of x_T/conditioning, the whole loop, D2H of x_0."""
        B, _, H, _ = x_host.shape
        device = torch.device(device)
        h = self._ensure(B, H, device)

        def hostc(t, dt=torch.float32):
            if t is None:
                return None
            if t.is_cuda:
                raise ValueError("native_sample_host takes host tensors")
            return t.detach().to(dt).contiguous()

        out = hostc(x_host).clone()
        lsm = hostc(lsm_cond) if self._has_lsm() else None
        topo = hostc(topo_cond) if self._has_topo() else None
        cond, yy, nz = hostc(cond_img), hostc(y, torch.int64), hostc(noise)
        with torch.cuda.device(device):
            self._set_schedule(h, betas, alphas, alpha_hat)
            self._set_sampler(h, ddim)
            self._cond_key = None   # conditioning of the handle is overwritten by this call
            N.check(N.lib().b2d_sample_host(h, out.data_ptr(), N.ptr(lsm), N.ptr(topo), N.ptr(cond), 0, 0, N.ptr(yy),
                                            N.ptr(nz), int(seed), int(sample_offset), float(noise_scale), B))
        return out

    @torch.no_grad()
    def profile_step(self, x, t, y=None, cond_img=None, lsm_cond=None, topo_cond=None, reps=5):
        """Per-launch device times of one eps evaluation (b2d_profile_step) as a list of dicts."""
        B, _, H, _ = x.shape
        h = self._ensure(B, H, x.device)
        xx = self._f32c(x, "x")
        with torch.cuda.device(x.device):
            stream = torch.cuda.current_stream().cuda_stream
            self._set_conditioning(h, B, y, cond_img, lsm_cond, topo_cond, stream)
            torch.cuda.synchronize()
            th = t.detach().to("cpu", torch.int64).contiguous()
            buf = (N.OpProfile * 512)()
            n = C.c_int32()
            N.check(N.lib().b2d_profile_step(h, xx.data_ptr(), th.data_ptr(), B, reps, buf, 512, C.byref(n)))
        return [dict(name=buf[i].name.decode(), klass=buf[i].klass.decode(), flops=buf[i].flops, bytes=buf[i].bytes,
                     ms=buf[i].ms) for i in range(n.value)]


class _HalfRunner(DiffusionNet):
    """Native handle behind a stand-alone ``Encoder`` or ``Decoder``: the other half is a placeholder module (its weights
    are packed but its ops never run), so the same per-batch program serves ``b2d_encoder_forward`` / ``b2d_decoder_forward``."""

    def __init__(self, encoder: Encoder = None, decoder: Decoder = None):
        NativeModel.__init__(self)
        own = encoder if encoder is not None else decoder
        n_heads = own.n_heads
        if encoder is None:
            encoder = Encoder(1, 256, n_heads=n_heads)
            if isinstance(decoder.residual_layers[0].attention, nn.Module) and hasattr(decoder.residual_layers[0].attention, "ff"):
                from . import unet as U
                encoder = U.Encoder(1, 256, n_heads=n_heads, cond_on_lsm=False, cond_on_topo=False)
        if decoder is None:
            decoder = Decoder(512, 1, 256, 64, n_heads=n_heads)
            if hasattr(encoder.attention_layers[0], "ff"):
                from . import unet as U
                decoder = U.Decoder(512, 1, 256, 64, n_heads=n_heads)
        # plain attributes (not registered sub-modules): the stand-alone half must not gain parameters it does not own
        object.__setattr__(self, "encoder", encoder)
        object.__setattr__(self, "decoder", decoder)
        self._attn_ff = int(hasattr(encoder.attention_layers[0], "ff"))
        own_dev = next(own.parameters()).device
        (decoder if own is encoder else encoder).to(own_dev)

    def _config(self, img_size, max_batch):
        cfg = super()._config(img_size, max_batch)
        cfg.attn_ff = self._attn_ff
        return cfg

    def _native_state_dict(self):
        sd = {"encoder." + k: v for k, v in self.encoder.state_dict().items()}
        sd.update({"decoder." + k: v for k, v in self.decoder.state_dict().items()})
        return sd

    def _weights_version(self):
        ts = [t for m in (self.encoder, self.decoder) for t in list(m.parameters()) + list(m.buffers())
              if t.dtype.is_floating_point and t.numel() > 0]
        ident = tuple(int(t._version) for t in ts) + tuple(t.data_ptr() for t in ts) + (self._refresh_epoch,)
        fp = torch.stack(torch._foreach_norm([t.detach() for t in ts])).to("cpu", torch.float64)
        return ident + (fp.numpy().tobytes(),)

    def encode(self, x, t, y, cond_img, lsm_cond, topo_cond):
        if x.dim() != 4 or x.shape[-1] != x.shape[-2]:
            raise ValueError("x must be [B, C, H, H]")
        B, _, H, _ = x.shape
        h = self._ensure(B, H, x.device)
        xx = self._f32c(x, "x")
        with torch.cuda.device(x.device):
            stream = torch.cuda.current_stream().cuda_stream
            self._set_conditioning(h, B, y, cond_img, lsm_cond, topo_cond, stream)
            outs = [torch.full((B, c, H >> (i + 1), H >> (i + 1)), float("nan"), device=x.device, dtype=torch.float32)
                    for i, c in enumerate(FMAP_CHANNELS)]
            ptrs = (C.c_void_p * 5)(*[o.data_ptr() for o in outs])
            th = t.detach().to("cpu", torch.int64).contiguous()
            N.check(N.lib().b2d_encoder_forward(h, xx.data_ptr(), th.data_ptr(), ptrs, B, stream))
        return tuple(outs)

    def decode(self, fmaps, t):
        f1 = fmaps[0]
        B, H = f1.shape[0], f1.shape[-1] * 2
        for i, (f, c) in enumerate(zip(fmaps, FMAP_CHANNELS)):
            if tuple(f.shape) != (B, c, H >> (i + 1), H >> (i + 1)):
                raise ValueError(f"fmap{i + 1} must be [{B}, {c}, {H >> (i + 1)}, {H >> (i + 1)}], got {tuple(f.shape)}")
        h = self._ensure(B, H, f1.device)
        fs = [self._f32c(f, f"fmap{i + 1}") for i, f in enumerate(fmaps)]
        with torch.cuda.device(f1.device):
            stream = torch.cuda.current_stream().cuda_stream
            out = torch.full((B, self.decoder.output_channels, H, H), float("nan"), device=f1.device, dtype=torch.float32)
            ptrs = (C.c_void_p * 5)(*[f.data_ptr() for f in fs])
            th = t.detach().to("cpu", torch.int64).contiguous()
            N.check(N.lib().b2d_decoder_forward(h, ptrs, th.data_ptr(), out.data_ptr(), B, stream))
        return out


# north_star alias: UNet(c_in, c_out, time_dim) style constructor over the same network
def UNet(c_in: int = 1, c_out: int = 1, time_dim: int = 256, lsm: bool = False, topo: bool = False,
         cond_channels: int = 0, num_classes=None, img_size: int = 64, n_heads: int = 4) -> DiffusionNet:
    z = torch.zeros(1, img_size, img_size)
    enc = Encoder(c_in, time_dim, n_heads=n_heads, num_classes=num_classes, lsm_tensor=z if lsm else None,
                  topo_tensor=z.clone() if topo else None, cond_on_img=cond_channels > 0,
                  cond_img_dim=(cond_channels, img_size, img_size) if cond_channels else None)
    dec = Decoder(512, c_out, time_dim, 64, n_heads=n_heads)
    return DiffusionNet(enc, dec)
