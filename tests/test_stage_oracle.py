"""CPU: the single-stage references of tests/stage_oracle.py, chained stage by stage, reproduce the whole-network oracle of
oracle/ddpm_oracle.py (which is pinned to the reference's goldens), for both model families and every attention flavour."""
import pytest
import torch

from diffusionmodelscustom_b200 import synth
from oracle import ddpm_oracle as O
from tests import stage_oracle as S

TOL = 1e-5


def _close(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm())


@pytest.mark.parametrize("variant", ["plain", "clean", "downscaling"])
def test_family_r_stages_chain_to_the_oracle(variant):
    B, H = 2, 32
    clean, down = variant == "clean", variant == "downscaling"
    c_in, ncls = (1, None) if down else (4, 4)
    sd = synth.synth_state_dict_r(c_in, 1, ncls, (H, H), not down, not down, seed=5, randomize_bn=True, clean=clean)
    inp = synth.synth_inputs(B, H, seed=6, has_lsm=not down, has_topo=not down, has_cond=not down, num_classes=ncls)
    t = torch.tensor([999, 37])
    taps = {}
    eps = O.family_r_forward(sd, inp["x"], t, inp["y"], inp["cond"], inp["lsm"], inp["topo"], n_heads=8 if clean else 4, taps=taps,
                             downscaling=down)
    heads = 8 if clean else 4
    enc, dec = S.family_r_embeddings(sd, t, inp["y"], downscaling=down)
    xc = torch.cat([inp[k] for k in ("x", "lsm", "topo", "cond") if inp.get(k) is not None], dim=1)
    f1 = S.r_enc_attention(sd, 0, S.r_stem(sd, xc, enc), heads)
    assert _close(f1, taps["fmap1"]) < TOL
    for k in range(2, 6):
        fk = S.r_enc_attention(sd, k - 1, S.r_enc_stage(sd, k, taps[f"fmap{k - 1}"], enc), heads)
        assert _close(fk, taps[f"fmap{k}"]) < TOL, k
    prev = taps["fmap5"]
    for i in range(4):
        d = S.r_dec_attention(sd, i, S.r_dec_stage(sd, i, prev, taps[f"fmap{4 - i}"], dec), heads)
        assert _close(d, taps[f"dec{i}"]) < TOL, i
        prev = taps[f"dec{i}"]
    assert _close(S.r_final(sd, prev), eps) < TOL


@pytest.mark.parametrize("mode", ["bicubic", "bilinear", "nearest"])
def test_family_d_stages_chain_to_the_oracle(mode):
    B, H = 2, 32
    sd = synth.synth_state_dict_d(2, 1, seed=7)
    inp = synth.synth_inputs(B, H, seed=8, lowres=5)
    t = torch.tensor([999, 222])
    taps = {}
    eps = O.family_d_forward(sd, inp["x"], t, inp["y_lowres"], interp_mode=mode, taps=taps)
    emb = S.family_d_embedding(t)
    assert _close(S.d_inc(sd, inp["x"], inp["y_lowres"].float(), mode), taps["x1"]) < TOL
    xs = [taps["x1"], taps["x2"], taps["x3"]]
    for k in (1, 2):
        assert _close(S.d_sa(sd, k, S.d_down(sd, k, xs[k - 1], emb)), xs[k]) < TOL, k
    x4 = S.d_sa(sd, 3, S.d_down(sd, 3, xs[2], emb))
    assert _close(S.d_bottleneck(sd, x4), taps["bot"]) < TOL
    prev = taps["bot"]
    for k in (1, 2, 3):
        u = S.d_sa(sd, k + 3, S.d_up(sd, k, prev, xs[3 - k], emb))
        assert _close(u, taps[f"u{k}"]) < TOL, k
        prev = taps[f"u{k}"]
    assert _close(S.d_outc(sd, prev), eps) < TOL
