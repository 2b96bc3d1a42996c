"""Ensemble generation on top of the native sampler (SURVEY.md §8(f1)).

Mirrors what the reference's generation scripts do around ``DiffusionUtils.sample`` —
``DDPM_DANRA_conditional/generation_DANRA_conditional.py:369-441`` and
``DDPM_clean_application/test/generation_ddpm.py:371-439``: take one evaluation batch ``(img, season, cond), lsm, topo, point``,
sample, bring the fields back to the host and write the ``gen_/eval_/lsm_/cond_/season_/point_samples__*.npz`` bundle (one
positional array each => key ``arr_0``).  The reference draws ONE member per date; here every date gets ``members`` of them and
the whole (date x member) list runs through ``b2d_ensemble_run``: per-date conditioning given once, sub-batches scheduled
natively with pinned double buffers, x_T and z_i drawn on the device keyed by the GLOBAL member index, so the fields are
identical for any ``sub_batch`` and any number of ranks.

``load_checkpoint`` is the ``torch.load(path)['network_params']`` step (generation_DANRA_conditional.py:354-360; written by
``training_DANRA_conditional.py:755-772`` as ``{'network_params', 'optimizer_params'}``).
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import numpy as np
import torch
import torch.distributed as dist

from . import _native as N
from .modules import NativeModel
from .sharding import shard_range

BUNDLE_PARTS = ("gen", "eval", "lsm", "cond", "season", "point")


class EnsembleJob(C.Structure):
    _fields_ = [("n_dates", C.c_int32), ("members", C.c_int32), ("sub_batch", C.c_int32), ("first", C.c_int32),
                ("count", C.c_int32), ("lsm", C.c_void_p), ("topo", C.c_void_p), ("cond", C.c_void_p), ("cond_h", C.c_int32),
                ("cond_w", C.c_int32), ("y", C.c_void_p), ("out", C.c_void_p), ("seed", C.c_uint64), ("noise_scale", C.c_float),
                ("xT_scale", C.c_float)]


class EnsembleStats(C.Structure):
    _fields_ = [("sub_batches", C.c_int32), ("out_pinned", C.c_int32), ("launches", C.c_int64), ("gather_ms", C.c_double),
                ("wall_ms", C.c_double)]


def load_checkpoint(model: torch.nn.Module, path: str, key: str = "network_params", strict: bool = True):
    """``model.load_state_dict(torch.load(path)['network_params'])`` for the reference's ``*.pth.tar`` checkpoints; buffers a
    checkpoint carries for the encoder (``encoder.lsm`` / ``encoder.elevation`` of the iclimate-style models) load like any
    other entry.  Returns the (missing, unexpected) key lists of ``load_state_dict``."""
    ckpt = torch.load(path, map_location="cpu", weights_only=False)
    sd = ckpt[key] if isinstance(ckpt, dict) and key in ckpt else ckpt
    return model.load_state_dict(sd, strict=strict)


def _host_f32(t, name, shape_tail=None):
    if t is None:
        return None
    t = torch.as_tensor(t).detach().to("cpu", torch.float32).contiguous()
    if shape_tail is not None and tuple(t.shape[1:]) != tuple(shape_tail):
        raise ValueError(f"{name}: expected per-date fields of shape [D, {', '.join(map(str, shape_tail))}], got {tuple(t.shape)}")
    return t


@torch.no_grad()
def generate_ensemble(model: NativeModel, diffusion, n_dates: int, members: int, *, season=None, cond_img=None, lsm=None,
                      topo=None, channels_hr: int = 1, img_size: Optional[int] = None, sub_batch: int = 64, seed: int = 0,
                      device="cuda", group=None, gather: bool = True, return_stats: bool = False, steps: Optional[int] = None,
                      eta: float = 0.0, timesteps=None):
    """Sample ``members`` fields for each of ``n_dates`` conditioning sets.

    ``season`` [D] int64, ``cond_img`` [D,C,H,W] (Family D: the low-resolution field [D,C,h,w]), ``lsm`` / ``topo`` [D,1,H,W]:
    HOST tensors, one row per date.  Returns a host tensor [n_dates, members, channels_hr, H, W] (rank-local slice only when
    ``gather=False``).  Under ``torch.distributed`` the flattened member list is cut into contiguous per-rank blocks
    (``sharding.shard_range``) with no data-path collective; one ``all_gather`` of the final fields.

    ``steps`` / ``timesteps`` (with ``eta``) sample every member with ``diffusion.sample_ddim``'s DDIM loop instead of the DDPM
    loop of ``diffusion.sample``; ``None`` for both keeps the DDPM loop."""
    if not isinstance(model, NativeModel):
        raise TypeError("generate_ensemble needs a native model (DiffusionNet / UNet_downscale of this package)")
    device = torch.device(device)
    H = img_size or getattr(diffusion, "img_size", None) or (lsm.shape[-1] if lsm is not None else None) or \
        getattr(model, "img_size", None)
    if H is None:
        raise ValueError("img_size is needed when neither lsm nor the diffusion object carries it")
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    total = n_dates * members
    lo, hi = shard_range(total, world, rank)
    sub_batch = max(1, min(sub_batch, max(hi - lo, 1)))
    ddim = None if (steps is None and timesteps is None) else diffusion._ddim_plan(steps, eta, timesteps)
    model.eval()
    if hasattr(model, "_bind"):            # Family D binds its high-resolution channel count from x
        model._bind(torch.empty(1, channels_hr, H, H))
    h = model._ensure(sub_batch, H, device)
    is_d = model._family == N.FAMILY_D
    lsm_h = None if is_d else _host_f32(lsm, "lsm", (1, H, H))
    topo_h = None if is_d else _host_f32(topo, "topo", (1, H, H))
    cond_h = _host_f32(cond_img, "cond_img")
    y_h = None if season is None else torch.as_tensor(season).detach().to("cpu", torch.int64).contiguous()
    for name, t in (("lsm", lsm_h), ("topo", topo_h), ("cond_img", cond_h), ("season", y_h)):
        if t is not None and t.shape[0] != n_dates:
            raise ValueError(f"{name} must have one row per date ({n_dates}), got {t.shape[0]}")
    scale = 0.005 if getattr(diffusion, "data_scaled", False) else 1.0
    out = torch.empty((hi - lo, channels_hr, H, H), dtype=torch.float32)
    job = EnsembleJob(n_dates=n_dates, members=members, sub_batch=sub_batch, first=lo, count=hi - lo, lsm=N.ptr(lsm_h),
                      topo=N.ptr(topo_h), cond=N.ptr(cond_h), cond_h=cond_h.shape[-2] if (is_d and cond_h is not None) else 0,
                      cond_w=cond_h.shape[-1] if (is_d and cond_h is not None) else 0, y=N.ptr(y_h), out=out.data_ptr(),
                      seed=int(seed), noise_scale=scale, xT_scale=scale)
    stats = EnsembleStats()
    L = N.lib()
    L.b2d_ensemble_run.argtypes = [C.c_void_p, C.POINTER(EnsembleJob), C.POINTER(EnsembleStats)]
    with torch.cuda.device(device):
        model._set_schedule(h, diffusion.betas, diffusion.alphas, diffusion.alpha_hat)
        model._set_sampler(h, ddim)
        model._cond_key = None       # the handle's conditioning is overwritten by the driver
        N.check(L.b2d_ensemble_run(h, C.byref(job), C.byref(stats)))
    if gather and world > 1:
        from .sharding import gather_fields
        out = gather_fields(out.to(device), total, group).cpu()
        lo, hi = 0, total
    res = out.reshape(n_dates, members, channels_hr, H, H) if hi - lo == total else out
    if return_stats:
        return res, dict(sub_batches=stats.sub_batches, out_pinned=bool(stats.out_pinned), launches=int(stats.launches),
                         gather_ms=stats.gather_ms, wall_ms=stats.wall_ms, rank_slice=(lo, hi))
    return res


def bundle_name(model_str, var_str, im_dim_str, cond_str, n_samples):
    """SAVE_NAME of the reference (generation_DANRA_conditional.py:428)."""
    return f"{model_str}__{var_str}__{im_dim_str}__{cond_str}__{n_samples}_samples.npz"


def save_bundle(save_path: str, save_name: str, generated, eval_img=None, eval_lsm=None, eval_cond=None, eval_season=None,
                point=None):
    """The reference's six ``np.savez_compressed(SAVE_PATH + '<part>_samples__' + SAVE_NAME, array)`` calls
    (generation_DANRA_conditional.py:431-436): one positional array per file => key ``arr_0``.  ``generated`` may carry the
    extra member axis [D, M, C, H, W]; parts that are ``None`` are skipped.  Returns the written paths."""
    os.makedirs(save_path, exist_ok=True)
    written = []
    for part, arr in zip(BUNDLE_PARTS, (generated, eval_img, eval_lsm, eval_cond, eval_season, point)):
        if arr is None:
            continue
        a = arr.detach().cpu().numpy() if isinstance(arr, torch.Tensor) else np.asarray(arr)
        p = os.path.join(save_path, f"{part}_samples__{save_name}")
        np.savez_compressed(p, a)
        written.append(p)
    return written
