"""TEST INFRASTRUCTURE ONLY - fp32 torch restatement of the segmentation forward.

Pinned (tests/test_oracle_vs_reference.py, tests/test_golden.py) against the outputs of the reference modules
themselves: tests/golden/reference_pins.npz and tests/golden/seg_*.npz, produced by scripts/make_reference_golden.py and
scripts/make_golden.py from the *reference* modules.

Follows:
  diarizen/models/eend/model_wavlm_conformer.py:238-264   (wrapper)
  diarizen/models/module/wav2vec2/model.py:68-119          (extract_features)
  diarizen/models/module/wav2vec2/components.py:106-132,182-209 (CNN), :297-308 (projection),
      :366-380 (pos conv), :429-486 + :612-725 (gated rel-pos MHSA), :798-820 (FFN),
      :899-942 (layer wiring), :980-987 + :1004-1024 (transformer)
  diarizen/models/module/conformer.py:27-325               (head)
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional

import torch
import torch.nn.functional as F

from diarizen_b200.archs import (CONV_KERNELS, CONV_STRIDES, HEAD_DIM, MAX_DISTANCE, NUM_BUCKETS,
                                 POS_CONV_GROUPS, POS_CONV_KERNEL, SegArch)


def rel_pos_bucket(rel: torch.Tensor) -> torch.Tensor:
    """components.py:629-666, bidirectional=True."""
    nb = NUM_BUCKETS // 2
    out = (rel > 0).to(torch.long) * nb
    r = rel.abs()
    max_exact = nb // 2
    small = r < max_exact
    large = max_exact + (torch.log(r.float() / max_exact) / math.log(MAX_DISTANCE / max_exact)
                         * (nb - max_exact)).to(torch.long)
    large = torch.min(large, torch.full_like(large, nb - 1))
    return out + torch.where(small, r, large)


def position_bias(embed: torch.Tensor, T: int) -> torch.Tensor:
    """components.py:612-627 -> (H, T, T)."""
    q = torch.arange(T)[:, None]
    k = torch.arange(T)[None, :]
    return embed[rel_pos_bucket(k - q)].permute(2, 0, 1)


def _ln(x, sd, prefix, eps=1e-5):
    return F.layer_norm(x, (x.shape[-1],), sd[prefix + ".weight"], sd[prefix + ".bias"], eps)


def _lin(x, sd, prefix):
    return F.linear(x, sd[prefix + ".weight"], sd[prefix + ".bias"])


def conv_layer(a: SegArch, sd: Dict[str, torch.Tensor], i: int, x: torch.Tensor) -> torch.Tensor:
    """Conv layer i of the feature extractor: (B, C_in, T_in) -> (B, C_i, T_i).  components.py:106-132."""
    pre = "wavlm_model.feature_extractor."
    x = F.conv1d(x, sd[f"{pre}conv_layers.{i}.conv.weight"], stride=CONV_STRIDES[i])
    if a.large:
        x = F.layer_norm(x.transpose(1, 2), (x.shape[1],), sd[f"{pre}conv_layers.{i}.layer_norm.weight"],
                         sd[f"{pre}conv_layers.{i}.layer_norm.bias"]).transpose(1, 2)
    elif i == 0:
        C = x.shape[1]
        x = F.group_norm(x, C, sd[f"{pre}conv_layers.0.layer_norm.weight"],
                         sd[f"{pre}conv_layers.0.layer_norm.bias"])
    return F.gelu(x)


def feature_extractor(a: SegArch, sd: Dict[str, torch.Tensor], wav: torch.Tensor) -> torch.Tensor:
    """(B, N) -> (B, T, C6).  model.py:106-113 + components.py:182-209."""
    pre = "wavlm_model.feature_extractor."
    x = wav
    if a.large:
        x = F.layer_norm(x, x.shape[-1:])
    x = x.unsqueeze(1)
    for i in range(len(CONV_KERNELS)):
        x = conv_layer(a, sd, i, x)
    return x.transpose(1, 2) * sd[pre + "dummy_weight"]


def wavlm_attention_context(a: SegArch, sd, prefix: str, x: torch.Tensor, heads, bias: Optional[torch.Tensor]):
    """components.py:668-725 followed by :429-486 up to the output projection: (B, T, h * 64) attention context of the
    remaining heads, in their order. `x` is the (possibly pre-normed) layer input."""
    B, T, D = x.shape
    H = a.total_heads
    h = len(heads)
    mask = None
    if bias is not None:
        xh = x.view(B, T, H, D // H).permute(0, 2, 1, 3)
        g = _lin(xh, sd, prefix + "gru_rel_pos_linear").view(B, H, T, 2, 4).sum(-1)
        g = torch.sigmoid(g)
        ga, gb = g[..., 0:1], g[..., 1:2]
        gate = ga * (gb * sd[prefix + "gru_rel_pos_const"] - 1.0) + 2.0        # (B,H,T,1)
        mask = (gate * bias.unsqueeze(0))[:, list(heads)]                       # (B,h,T,T)
    q = _lin(x, sd, prefix + "q_proj").view(B, T, h, HEAD_DIM).transpose(1, 2)
    k = _lin(x, sd, prefix + "k_proj").view(B, T, h, HEAD_DIM).permute(0, 2, 3, 1)
    v = _lin(x, sd, prefix + "v_proj").view(B, T, h, HEAD_DIM).transpose(1, 2)
    w = (HEAD_DIM ** -0.5 * q) @ k
    if mask is not None:
        w = w + mask
    w = w - w.max(dim=-1, keepdim=True)[0]
    w = torch.softmax(w, dim=-1)
    return (w @ v).transpose(1, 2).reshape(B, T, h * HEAD_DIM)


def wavlm_attention(a: SegArch, sd, prefix: str, x: torch.Tensor, heads, bias: Optional[torch.Tensor]):
    """components.py:668-725 followed by :429-486. `x` is the (possibly pre-normed) layer input."""
    return _lin(wavlm_attention_context(a, sd, prefix, x, heads, bias), sd, prefix + "out_proj")


def encoder_bias(a: SegArch, sd, T: int) -> Optional[torch.Tensor]:
    """Relative-position bias (H, T, T) shared by every layer; only layer 0 owns the embedding (components.py:1004-1024)."""
    if not a.heads[0]:
        return None
    return position_bias(sd["wavlm_model.encoder.transformer.layers.0.attention.rel_attn_embed.weight"], T)


def pos_conv(a: SegArch, sd, x: torch.Tensor) -> torch.Tensor:
    """Projected features (B, T, D) -> input of layer 0: residual positional convolution (components.py:366-380), then
    the transformer LayerNorm for post-norm models (components.py:1590-1597)."""
    tr = "wavlm_model.encoder.transformer."
    # weight-normed grouped conv: w = g * v / ||v|| over dims (0,1) per tap  (components.py:344)
    v = sd[tr + "pos_conv_embed.conv.parametrizations.weight.original1"]
    g = sd[tr + "pos_conv_embed.conv.parametrizations.weight.original0"]
    w = g * v / v.norm(dim=(0, 1), keepdim=True)
    pc = F.conv1d(x.transpose(1, 2), w, sd[tr + "pos_conv_embed.conv.bias"], padding=POS_CONV_KERNEL // 2,
                  groups=POS_CONV_GROUPS)[..., :-1]
    x = x + F.gelu(pc).transpose(1, 2)
    if not a.large:   # Transformer(layer_norm_first = not encoder_layer_norm_first): components.py:1590-1597
        x = _ln(x, sd, tr + "layer_norm")
    return x


def wavlm_layer(a: SegArch, sd, l: int, x: torch.Tensor, bias: Optional[torch.Tensor]) -> torch.Tensor:
    """Encoder layer l: hidden state l -> hidden state l + 1.  components.py:899-942."""
    L = f"wavlm_model.encoder.transformer.layers.{l}."
    heads = a.heads[l]
    if heads:
        xin = _ln(x, sd, L + "layer_norm") if a.large else x
        x = x + wavlm_attention(a, sd, L + "attention.", xin, heads, bias)
    if a.large:
        if a.ffn[l]:
            y = _ln(x, sd, L + "final_layer_norm")
            y = _lin(F.gelu(_lin(y, sd, L + "feed_forward.intermediate_dense")), sd, L + "feed_forward.output_dense")
            x = x + y
    else:
        x = _ln(x, sd, L + "layer_norm")
        if a.ffn[l]:
            y = _lin(F.gelu(_lin(x, sd, L + "feed_forward.intermediate_dense")), sd, L + "feed_forward.output_dense")
            x = x + y
        x = _ln(x, sd, L + "final_layer_norm")
    return x


def wavlm_encoder(a: SegArch, sd, feats: torch.Tensor, taps: Optional[dict] = None) -> List[torch.Tensor]:
    """(B,T,C6) -> list of L+1 hidden states."""
    en = "wavlm_model.encoder."
    x = _lin(_ln(feats, sd, en + "feature_projection.layer_norm"), sd, en + "feature_projection.projection")
    if taps is not None:
        taps["proj"] = x
    x = pos_conv(a, sd, x)
    ret = [x]
    bias = encoder_bias(a, sd, x.shape[1])
    for l in range(a.num_layers):
        x = wavlm_layer(a, sd, l, x, bias)
        ret.append(x)
    return ret


def conformer_block(a: SegArch, sd, C: str, x: torch.Tensor) -> torch.Tensor:
    """conformer.py:216-257."""
    B, T, A = x.shape

    def ffn(x, p):
        y = _ln(x, sd, C + p + "ln_norm")
        y = _lin(y, sd, C + p + "w_1")
        y = y * torch.sigmoid(y)
        return x + 0.5 * _lin(y, sd, C + p + "w_2")

    x = ffn(x, "ffn1.")
    # MHSA, scores / sqrt(d_k), no positional term (use_posi=False)
    h = a.head_heads
    dk = A // h
    y = _ln(x, sd, C + "mha.ln_norm")
    q = _lin(y, sd, C + "mha.mha.linearQ").view(B, T, h, dk).transpose(1, 2)
    k = _lin(y, sd, C + "mha.mha.linearK").view(B, T, h, dk).transpose(1, 2)
    v = _lin(y, sd, C + "mha.mha.linearV").view(B, T, h, dk).transpose(1, 2)
    att = torch.softmax(q @ k.transpose(-2, -1) / math.sqrt(dk), dim=3)
    y = (att @ v).permute(0, 2, 1, 3).reshape(B, T, h * dk)
    x = x + _lin(y, sd, C + "mha.mha.linearO")
    # conv module
    y = _ln(x, sd, C + "conv.ln_norm").transpose(1, 2)
    y = F.conv1d(y, sd[C + "conv.pointwise_conv1.weight"], sd[C + "conv.pointwise_conv1.bias"])
    y = F.glu(y, dim=1)
    y = F.conv1d(y, sd[C + "conv.depthwise_conv.weight"], sd[C + "conv.depthwise_conv.bias"],
                 padding=(a.head_kernel - 1) // 2, groups=A)
    y = F.batch_norm(y, sd[C + "conv.bn_norm.running_mean"], sd[C + "conv.bn_norm.running_var"],
                     sd[C + "conv.bn_norm.weight"], sd[C + "conv.bn_norm.bias"], training=False, eps=1e-5)
    y = y * torch.sigmoid(y)
    y = F.conv1d(y, sd[C + "conv.pointwise_conv2.weight"], sd[C + "conv.pointwise_conv2.bias"])
    x = x + y.transpose(1, 2)
    x = ffn(x, "ffn2.")
    return _ln(x, sd, C + "ln_norm")


@torch.inference_mode()
def seg_forward(a: SegArch, sd: Dict[str, torch.Tensor], wav: torch.Tensor, taps: Optional[dict] = None):
    """(B, N) fp32 -> (B, T, num_classes) log-probabilities.  model_wavlm_conformer.py:238-264."""
    feats = feature_extractor(a, sd, wav)
    if taps is not None:
        taps["feats"] = feats
    reps = wavlm_encoder(a, sd, feats, taps)
    if taps is not None:
        taps["reps"] = reps
    x = torch.stack(reps, dim=-1)
    x = head_input(sd, F.linear(x, sd["weight_sum.weight"]).squeeze(-1))
    if taps is not None:
        taps["head_in"] = x
    for i in range(a.head_layers):
        x = conformer_block(a, sd, f"conformer.conformer_layer.{i}.", x)
    if taps is not None:
        taps["head_out"] = x
    return classify(sd, x)


def head_input(sd, mix: torch.Tensor) -> torch.Tensor:
    """Weighted layer sum (B, T, D) -> conformer input (B, T, A).  model_wavlm_conformer.py:253-257."""
    return _ln(_lin(mix, sd, "proj"), sd, "lnorm")


def classify(sd, x: torch.Tensor) -> torch.Tensor:
    """Last conformer block output -> powerset log-probabilities.  model_wavlm_conformer.py:258-264."""
    return torch.log_softmax(_lin(x, sd, "classifier"), dim=-1)


def powerset_mapping(num_classes: int = 4, max_set: int = 2) -> torch.Tensor:
    """pa/utils/powerset.py:68-101: rows = powerset classes in order of set size then combinations."""
    import itertools
    rows = []
    for size in range(0, max_set + 1):
        for comb in itertools.combinations(range(num_classes), size):
            r = [0.0] * num_classes
            for c in comb:
                r[c] = 1.0
            rows.append(r)
    return torch.tensor(rows)


def to_multilabel(logp: torch.Tensor) -> torch.Tensor:
    """pa/utils/powerset.py:103-128 (soft=False): argmax -> one-hot -> @ mapping."""
    m = powerset_mapping()
    hard = F.one_hot(torch.argmax(logp, dim=-1), m.shape[0]).float()
    return hard @ m
