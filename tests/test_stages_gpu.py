"""Every layer stage of both model families against an fp64 recomputation of that stage alone.

One forward runs on the GPU; then every named activation tap is read back, and each stage is recomputed in fp64 from the
GPU's own fp16 input taps (cast to double) with the state dict in double.  A stage is judged on its own error only: nothing
upstream leaks into it, so an error in one decoder norm or in the time embedding cannot be diluted by the rest of the network
the way it is in the end-to-end eps comparison.  The taps come from the program the batch selects (streaming GEMM with folded
LayerNorm at >= 8192 token rows, norm cluster width, split-K, GroupNorm quarter partials, samples per attention-block CTA),
so the bench batches are run as benchmarked and rows {0, B/2, B-1} are checked; all norms are per sample, so the row slice is
exact.

Gates: relative L2 <= 3e-3 per non-attention stage, <= 4e-3 per attention stage (the op-test gate with P rounded to fp16).
The stem keeps the fp32 state unrounded (hi/lo split) and documents fp16 weights, so it is additionally held to the fp16
rounding of the exact sum computed with those fp16 weights, at a gate of STEM_EXACT_GATE.  That check sees the state's
rounding only where the state dominates the stem's output (the unconditioned cases and x_scale = 300); with conditioning
fields the fp32 conditioning part dominates.

Worst measured error per stage class over all cases, one NVIDIA B200 at its 1000 W power limit:
    stem 3.0e-4 (fp16 rounding check 6.3e-5), encoder stages 5.0e-4, decoder stages 5.1e-4, final layer 6.3e-4,
    Family D inc 4.9e-4, down 7.1e-4, bottleneck 7.6e-4, up 7.4e-4, outc 7.5e-8,
    attention: encoder 3.7e-4, decoder 3.0e-4, Family D 3.3e-4.

Every sample carries its own t (and its own class where the case has classes).  Cases marked with a gain load the weights with
every time projection scaled by TEMB_GAIN, so that the embedding path is not invisible next to the activations; the
``tinyvar`` case gives a quarter of the BatchNorm channels a running variance far below eps (with gamma scaled to keep the
activations in range), where the eps of the BN fold decides the result.
"""
import ctypes as C
import os
import subprocess
import sys

import pytest
import torch

from diffusionmodelscustom_b200 import _native as N
from diffusionmodelscustom_b200.modules import NativeModel
from tests import gpu_util as G
from tests import stage_oracle as S
from tests.cases import D_CASES, R_CASES
from tests.model_util import build_ours_d, build_ours_r, inputs_d, inputs_r

pytestmark = pytest.mark.gpu
GATE = 3e-3
ATTN_GATE = 4e-3
STEM_EXACT_GATE = 1e-4
TEMB_GAIN = 16.0
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

ENC_CH = (64, 64, 128, 256, 512)
DEC_OUT = (256, 128, 64, 64)


def read_tap(net, name, B, C_, hw, rows):
    """NHWC fp16 tap -> NCHW fp64 on the GPU, rows selected.  The host buffer is sized from the stage's known shape."""
    buf = torch.empty(B * hw * hw * C_, dtype=torch.float32)
    c, h = C.c_int32(), C.c_int32()
    N.check(N.lib().b2d_debug_read(net._h, name.encode(), buf.data_ptr(), buf.numel(), C.byref(c), C.byref(h)))
    assert (c.value, h.value) == (C_, hw), (name, c.value, h.value, C_, hw)
    t = buf.reshape(B, hw, hw, C_)[rows].permute(0, 3, 1, 2)
    assert torch.isfinite(t).all(), f"tap {name} is not finite"
    return t.to("cuda", torch.float64)


def _sd64(sd):
    return {k: v.to("cuda", torch.float64) if v.dtype.is_floating_point else v.cuda() for k, v in sd.items()}


def _with_gain(net, sd, gain):
    if gain == 1.0:
        return sd
    sd = {k: (v * gain if ("time_projection" in k or "emb_layer" in k) else v) for k, v in sd.items()}
    net.load_state_dict(sd, strict=True)
    return sd


def _tiny_bn_var(net, sd):
    """A quarter of every encoder BatchNorm's channels get running_var = 1e-6 << eps; gamma is scaled by sqrt((1e-6+eps)/(var+eps))
    so the normalised activations keep their size.  Only there does the eps of the BN fold move the result."""
    sd = dict(sd)
    for k in [k for k in sd if k.endswith(".running_var")]:
        p = k[: -len(".running_var")]
        var, g = sd[k].clone(), sd[p + ".weight"].clone()
        sel = torch.arange(var.numel()) % 4 == 1
        g[sel] = g[sel] * torch.sqrt((1e-6 + 1e-5) / (var[sel] + 1e-5))
        var[sel] = 1e-6
        sd[k], sd[p + ".weight"] = var, g
    net.load_state_dict(sd, strict=True)
    return sd


def _timesteps(B, seed):
    g = torch.Generator().manual_seed(seed)
    t = torch.randperm(997, generator=g)[:B] + 2          # distinct per sample
    t[0] = 999
    if B >= 3:
        t[-1] = 1
    return t


class Checker:
    def __init__(self, tag):
        self.tag, self.errs, self.bad = tag, {}, []

    def __call__(self, stage, out, ref, gate):
        err = G.rel_l2(out, ref)
        self.errs[stage] = err
        if not err <= gate:
            self.bad.append((stage, err, gate))

    def done(self):
        assert not self.bad, (self.tag, self.bad)
        return self.errs


# --------------------------------------------------------------------------------------------------- Family R
def check_family_r(name, batch=None, gain=1.0, tinyvar=False, rows=None, seed=3):
    case = R_CASES[name]
    B = batch or case["batch"]
    H, heads = case["hw"], case.get("n_heads", 4)
    rows = list(range(B)) if rows is None else rows
    net, sd = build_ours_r(case)
    sd = _with_gain(net, sd, gain)
    if tinyvar:
        sd = _tiny_bn_var(net, sd)
    inp, dev = inputs_r(case, B)
    t = _timesteps(B, seed)
    y = None
    if case["num_classes"]:
        y = torch.arange(B) % case["num_classes"]
        dev["y"] = y.cuda()
    x = dev["x"] * case.get("x_scale", 1.0)
    NativeModel.saturation_count(reset=True)
    eps = net(x, t.cuda(), dev["y"], dev["cond"], dev["lsm"], dev["topo"])
    torch.cuda.synchronize()
    assert torch.isfinite(eps).all()
    s = [H, H // 2, H // 4, H // 8, H // 16, H // 32]
    tap = lambda n, c, hw: read_tap(net, n, B, c, hw, rows)
    sd64 = _sd64(sd)
    tr = t[rows].cuda()
    enc, dec = S.family_r_embeddings(sd64, tr, None if y is None else y[rows].cuda(), downscaling=case.get("downscaling", False))
    ck = Checker((name, B, gain, tinyvar))

    # stem: fp64 with the true weights, and exact fp16 rounding of the sum formed with the fp16 state-channel weights
    parts = [x[rows]] + [dev[k][rows] for k in ("lsm", "topo", "cond") if dev[k] is not None]
    xc = torch.cat(parts, dim=1).double()
    f1_pre = tap("f1_pre", 64, s[1])
    ck("stem", f1_pre, S.r_stem(sd64, xc, enc), GATE)
    exact = S.r_stem(sd64, xc, enc, torch.float16, x.shape[1]).half().double()
    ck("stem_fp16_rounding", f1_pre, exact, STEM_EXACT_GATE)

    fm = [tap(f"fmap{k}", ENC_CH[k - 1], s[k]) for k in range(1, 6)]
    ck("enc_attn1", fm[0], S.per_sample(lambda h: S.r_enc_attention(sd64, 0, h, heads), f1_pre), ATTN_GATE)
    for k in range(2, 6):
        pre = tap(f"pre{k}", ENC_CH[k - 1], s[k])
        ck(f"enc_stage{k}", pre, S.r_enc_stage(sd64, k, fm[k - 2], enc), GATE)
        ck(f"enc_attn{k}", fm[k - 1], S.per_sample(lambda h: S.r_enc_attention(sd64, k - 1, h, heads), pre), ATTN_GATE)
    prev = fm[4]
    for i in range(4):
        pre = tap(f"dec{i}_pre", DEC_OUT[i], s[4 - i])
        ck(f"dec{i}", pre, S.r_dec_stage(sd64, i, prev, fm[3 - i], dec), GATE)
        out = tap(f"dec{i}", DEC_OUT[i], s[4 - i])
        ck(f"dec_attn{i}", out, S.per_sample(lambda h: S.r_dec_attention(sd64, i, h, heads), pre), ATTN_GATE)
        prev = out
    ck("final", eps[rows], S.r_final(sd64, prev), GATE)
    assert NativeModel.saturation_count() == 0, "fp16 activation storage clipped"
    return ck.done()


# --------------------------------------------------------------------------------------------------- Family D
def check_family_d(name, batch=None, gain=1.0, rows=None, seed=4):
    case = D_CASES[name]
    B = batch or case["batch"]
    H = case["hw"]
    rows = list(range(B)) if rows is None else rows
    net, sd = build_ours_d(case)
    sd = _with_gain(net, sd, gain)
    inp, dev = inputs_d(case, B)
    t = _timesteps(B, seed)
    NativeModel.saturation_count(reset=True)
    eps = net(dev["x"], t.cuda(), dev["y_lowres"])
    torch.cuda.synchronize()
    assert torch.isfinite(eps).all()
    tap = lambda n, c, hw: read_tap(net, n, B, c, hw, rows)
    sd64 = _sd64(sd)
    emb = S.family_d_embedding(t[rows].cuda())
    ck = Checker((name, B, gain))
    sa = lambda k, h: S.per_sample(lambda v: S.d_sa(sd64, k, v), h)

    y_lr = None if dev["y_lowres"] is None else dev["y_lowres"][rows].double()
    x1 = tap("x1", 64, H)
    ck("inc", x1, S.d_inc(sd64, dev["x"][rows].double(), y_lr, case.get("interp_mode", "bicubic")), GATE)
    xs = [x1]
    for k, (c, hw) in enumerate(((128, H // 2), (256, H // 4), (256, H // 8)), start=1):
        pre = tap(f"x{k + 1}_pre", c, hw)
        ck(f"down{k}", pre, S.d_down(sd64, k, xs[-1], emb), GATE)
        out = tap(f"x{k + 1}", c, hw)
        ck(f"sa{k}", out, sa(k, pre), ATTN_GATE)
        xs.append(out)
    bot = tap("bot", 256, H // 8)
    ck("bot", bot, S.d_bottleneck(sd64, xs[3]), GATE)
    prev = bot
    for k, (c, hw) in enumerate(((128, H // 4), (64, H // 2), (64, H)), start=1):
        pre = tap(f"u{k}_pre", c, hw)
        ck(f"up{k}", pre, S.d_up(sd64, k, prev, xs[3 - k], emb), GATE)
        out = tap(f"u{k}", c, hw)
        ck(f"sa{k + 3}", out, sa(k + 3, pre), ATTN_GATE)
        prev = out
    ck("outc", eps[rows], S.d_outc(sd64, prev), GATE)
    assert NativeModel.saturation_count() == 0, "fp16 activation storage clipped"
    return ck.done()


# --------------------------------------------------------------------------------------------------- cases
R_STAGE_CASES = [(n, None, 1.0, False) for n in R_CASES] + [
    ("full_64_randbn", 3, TEMB_GAIN, False),
    ("cfg3_full_128", 3, TEMB_GAIN, False),
    ("full_64_randbn", 2, 1.0, True),
]
D_STAGE_CASES = [(n, None, 1.0) for n in D_CASES] + [("cfg4_downscale_64", None, TEMB_GAIN)]
# the programs bench.py times, at their benchmarked per-GPU batch
BENCH_PROGRAMS = [("cfg2_lsmtopo_64", 64), ("cfg3_full_128", 32), ("cfg3_full_128", 256), ("cfg5_flexible_128", 128),
                  ("cfg4_downscale_64", 64)]


def _rid(c):
    return f"{c[0]}-B{c[1] or 'case'}" + (f"-gain{c[2]:g}" if c[2] != 1.0 else "") + ("-tinyvar" if len(c) > 3 and c[3] else "")


@pytest.mark.parametrize("name,batch,gain,tinyvar", R_STAGE_CASES, ids=[_rid(c) for c in R_STAGE_CASES])
def test_family_r_stages_vs_fp64(name, batch, gain, tinyvar):
    check_family_r(name, batch, gain, tinyvar)


@pytest.mark.parametrize("name,batch,gain", D_STAGE_CASES, ids=[_rid(c) for c in D_STAGE_CASES])
def test_family_d_stages_vs_fp64(name, batch, gain):
    check_family_d(name, batch, gain)


@pytest.mark.parametrize("name,batch", BENCH_PROGRAMS)
def test_stages_at_bench_batch_vs_fp64(name, batch):
    rows = [0, batch // 2, batch - 1]
    if name in D_CASES:
        check_family_d(name, batch, rows=rows)
    else:
        check_family_r(name, batch, rows=rows)


_FUSED_GN_SCRIPT = r"""
import sys, torch
sys.path.insert(0, sys.argv[1])
from tests import test_stages_gpu as T
from tests.cases import D_CASES
from tests.model_util import build_ours_d, inputs_d
case = D_CASES["cfg4_downscale_64"]
net, _ = build_ours_d(case)
inp, dev = inputs_d(case)
t = torch.full((case["batch"],), 300, dtype=torch.long)
kinds = {p["klass"] for p in net.profile_step(dev["x"], t, dev["y_lowres"], reps=1)}
assert "norm_fused" in kinds, kinds
for c in T.D_STAGE_CASES:
    T.check_family_d(*c)
T.check_family_d("cfg4_downscale_64", 64, rows=[0, 32, 63])
print("ok")
"""


def test_family_d_stages_with_clustered_groupnorm():
    """B2D_FUSED_GN=1 selects the clustered one-pass GroupNorm (norm_fused<1>) wherever a convolution did not already reduce
    the statistics; the switch is read once per process, so the stage checks run in a subprocess with it set."""
    r = subprocess.run([sys.executable, "-c", _FUSED_GN_SCRIPT, ROOT], env=dict(os.environ, B2D_FUSED_GN="1"), capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
