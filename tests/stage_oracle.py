"""fp64 references of single layer stages of both model families, for tests/test_stages_gpu.py.

Each function recomputes one stage of the forward from that stage's own inputs, so a test can feed it the activations the
GPU stored before the stage and compare with what the GPU stored after it.  Every function is assembled from the pieces of
``oracle/ddpm_oracle.py`` (which stays pinned to the reference's goldens); only the three sinusoidal embeddings are restated
here, because the oracle evaluates them in fp32 as the reference does.  Pass a float64 state dict and float64 tensors: the
pieces are dtype- and device-agnostic, so the references run in fp64 on whatever device the inputs live on.
"""
import torch
import torch.nn.functional as F

from oracle import ddpm_oracle as O


# --------------------------------------------------------------------------------------------------- embeddings in fp64
def _sincos(t, base, channels=256):
    """[sin | cos] layout: Encoder.pos_encoding (base 1000) and UNet_downscale.pos_encoding (base 10000)."""
    t = t.to(torch.float64).unsqueeze(-1)
    inv = 1.0 / (base ** (torch.arange(0, channels, 2, dtype=torch.float64, device=t.device) / channels))
    return torch.cat([torch.sin(t * inv), torch.cos(t * inv)], dim=-1)


def interleaved_embedding(t, dim=256, n=10000):
    """SinusoidalEmbedding: d[2j] = sin(t / n^(2j/dim)), d[2j+1] = cos(...)."""
    div = torch.tensor([n ** (2 * i / dim) for i in range(dim // 2)], dtype=torch.float64, device=t.device)
    e = t.to(torch.float64).unsqueeze(-1) / div
    out = torch.zeros(t.shape[0], dim, dtype=torch.float64, device=t.device)
    out[:, 0::2] = torch.sin(e)
    out[:, 1::2] = torch.cos(e)
    return out


def family_r_embeddings(sd, t, y=None, downscaling=False):
    """(encoder embedding incl. the label embedding, decoder embedding) of Family R."""
    enc = interleaved_embedding(t) if downscaling else _sincos(t, 1000.0)
    if y is not None:
        enc = enc + sd["encoder.label_emb.weight"][y]
    return enc, interleaved_embedding(t)


def family_d_embedding(t):
    return _sincos(t, 10000.0)


def _vec(sd, p, emb):
    return O._tproj(sd, p, emb.to(sd[p + ".1.weight"].dtype))[:, :, None, None]


# --------------------------------------------------------------------------------------------------- Family R
E, D = "encoder.", "decoder."


def attention_kwargs(sd):
    """The clean-application generation names its attention modules mha / ff and adds the FF tail."""
    return dict(mha="mha", ff=True, ffp="ff") if (E + "attention_layers.0.mha.in_proj_weight") in sd else {}


def r_stem(sd, x_cat, enc_emb, x_weight_dtype=None, n_x=None):
    """Encoder.conv1 (8x8, stride 2, pad 3) on [x, lsm, topo, cond] + time projection 0.  ``x_weight_dtype`` rounds the weights
    of the first ``n_x`` (state) channels, to model a kernel that documents fp16 weights on those channels."""
    w = sd[E + "conv1.weight"]
    if x_weight_dtype is not None:
        w = w.clone()
        w[:, :n_x] = w[:, :n_x].to(x_weight_dtype).to(w.dtype)
    return F.conv2d(x_cat, w, None, 2, 3) + _vec(sd, E + "time_projection_layers.0", enc_emb)


def r_enc_attention(sd, level, h, n_heads):
    return O.image_self_attention(sd, f"{E}attention_layers.{level}", h, n_heads, **attention_kwargs(sd))


def r_enc_stage(sd, k, fmap_prev, enc_emb):
    """fmap{k-1} -> pre{k}, k = 2..5: (conv2 -> bn1 -> ReLU for k = 2) -> two BasicBlocks -> + time projection k-1."""
    li = k - 1
    h = fmap_prev
    if k == 2:
        h = F.relu(O._bn_eval(sd, E + "bn1", F.conv2d(h, sd[E + "conv2.weight"], None, 2, 3)))
    for bi in range(2):
        h = O._basic_block(sd, f"{E}layer{li}.{bi}.", h, 2 if (li > 1 and bi == 0) else 1)
    return h + _vec(sd, f"{E}time_projection_layers.{li}", enc_emb)


def r_dec_stage(sd, i, prev, skip, dec_emb):
    """DecoderBlock i up to its attention: ConvT -> IN -> 3x3 conv -> IN -> + skip -> + time projection."""
    p = f"{D}residual_layers.{i}."
    out = F.conv_transpose2d(prev, sd[p + "transpose.weight"], sd[p + "transpose.bias"], stride=2)
    out = F.instance_norm(out, eps=1e-5)
    out = F.conv2d(out, sd[p + "conv.weight"], sd[p + "conv.bias"], 1, 1)
    out = F.instance_norm(out, eps=1e-5)
    return out + skip + _vec(sd, p + "time_projection_layer", dec_emb)


def r_dec_attention(sd, i, h, n_heads):
    return F.relu(O.image_self_attention(sd, f"{D}residual_layers.{i}.attention", h, n_heads, **attention_kwargs(sd)))


def r_final(sd, dec3):
    p = D + "final_layer."
    out = F.conv_transpose2d(dec3, sd[p + "transpose.weight"], sd[p + "transpose.bias"], stride=2)
    out = F.instance_norm(out, eps=1e-5)
    return F.conv2d(out, sd[p + "conv.weight"], sd[p + "conv.bias"], 1, 1)


# --------------------------------------------------------------------------------------------------- Family D
def d_inc(sd, x, y_lowres, interp_mode):
    """Resize of the low-res field to the state's extent, concatenation, inc DoubleConv."""
    if y_lowres is not None:
        yy = F.interpolate(y_lowres, size=[x.shape[-1], x.shape[-2]], mode=interp_mode)
    else:
        yy = torch.zeros_like(x)
    return O._double_conv(sd, "inc", torch.cat([x, yy], dim=1))


def d_down(sd, k, h, emb):
    """Down.forward of down{k}: MaxPool2d(2) -> DoubleConv(res) -> DoubleConv -> + emb_layer."""
    p = f"down{k}"
    h = F.max_pool2d(h, 2)
    h = O._double_conv(sd, p + ".maxpool_conv.1", h, residual=True)
    h = O._double_conv(sd, p + ".maxpool_conv.2", h)
    return h + _vec(sd, p + ".emb_layer", emb)


def d_up(sd, k, h, skip, emb):
    """Up.forward of up{k}: bilinear x2 (align_corners=True) -> cat[skip, x] -> DoubleConv(res) -> DoubleConv -> + emb_layer."""
    p = f"up{k}"
    h = F.interpolate(h, scale_factor=2, mode="bilinear", align_corners=True)
    h = torch.cat([skip, h], dim=1)
    h = O._double_conv(sd, p + ".conv.0", h, residual=True)
    h = O._double_conv(sd, p + ".conv.1", h)
    return h + _vec(sd, p + ".emb_layer", emb)


def d_sa(sd, k, h):
    return O.image_self_attention(sd, f"sa{k}", h, 4, ln="ln", mha="mha", ff=True)


def d_bottleneck(sd, h):
    return O._double_conv(sd, "bot3", O._double_conv(sd, "bot1", h))


def d_outc(sd, u3):
    return F.conv2d(u3, sd["outc.weight"], sd["outc.bias"])


def per_sample(fn, h):
    """Apply a stage one sample at a time.  Attention stages are per sample, and the fp64 scores of a 4096-token map take
    0.5 GiB per sample with 4 heads, so a large batch is never materialised at once."""
    return torch.cat([fn(h[i:i + 1]) for i in range(h.shape[0])])
