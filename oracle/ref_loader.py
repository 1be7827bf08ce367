"""TEST INFRASTRUCTURE ONLY - imports the *reference* modules when /root/reference is mounted.

The reference's `Model` wrapper cannot be imported (pyannote.core & co. are absent, SURVEY.md 8c), so the
wrapper (model_wavlm_conformer.py:238-264) is re-assembled here from the importable reference parts:
`wav2vec2_model`, `ConformerEncoder`.  Used by the scripts that write the golden vectors (scripts/make_golden.py,
scripts/make_reference_golden.py).
"""
from __future__ import annotations

import os
import sys

import torch
import torch.nn as nn

REF = os.environ.get("DIARIZEN_REF", "/root/reference")


def available() -> bool:
    return os.path.isdir(os.path.join(REF, "diarizen"))


def _path():
    if REF not in sys.path:
        sys.path.insert(0, REF)


class RefSegModel(nn.Module):
    """Same submodule names as the reference Model => identical state_dict keys."""

    def __init__(self, arch):
        super().__init__()
        _path()
        from diarizen.models.module.conformer import ConformerEncoder
        from diarizen.models.module.wav2vec2.model import wav2vec2_model
        from diarizen_b200.archs import to_reference_config
        self.wavlm_model = wav2vec2_model(**to_reference_config(arch))
        self.weight_sum = nn.Linear(arch.num_layers + 1, 1, bias=False)
        self.proj = nn.Linear(arch.embed_dim, arch.head_dim_model)
        self.lnorm = nn.LayerNorm(arch.head_dim_model)
        self.conformer = ConformerEncoder(attention_in=arch.head_dim_model, ffn_hidden=arch.head_ffn,
                                          num_head=arch.head_heads, num_layer=arch.head_layers,
                                          kernel_size=arch.head_kernel, dropout=0.1, use_posi=False,
                                          output_activate_function=False)
        self.classifier = nn.Linear(arch.head_dim_model, arch.num_classes)
        self.activation = nn.LogSoftmax(dim=-1)

    def forward(self, waveforms):
        assert waveforms.dim() == 3
        waveforms = waveforms[:, 0, :]
        reps, _ = self.wavlm_model.extract_features(waveforms)
        x = torch.stack(reps, dim=-1)
        x = torch.squeeze(self.weight_sum(x), -1)
        x = self.lnorm(self.proj(x))
        x = self.conformer(x)
        return self.activation(self.classifier(x))


class RefSegModelMC(nn.Module):
    """The reference multi-channel model re-assembled from its importable parts, following
    diarizen/models/eend/model_wavlm_conformer_mc.py:60-95 (modules) and :241-282 (forward): `wav2vec2_model.extract_features_mc`
    with `CrossChannelAttention` fusion modules, channel mean of the 4-D states, layer mix, projection, conformer, classifier.
    Same submodule names as the reference Model => identical state_dict keys."""

    def __init__(self, arch, fusion_dim: int, fusion_heads: int, fusion_layers: int):
        super().__init__()
        _path()
        from diarizen.models.module.conformer import ConformerEncoder
        from diarizen.models.module.utils_mc import CrossChannelAttention
        from diarizen.models.module.wav2vec2.model import wav2vec2_model
        from diarizen_b200.archs import to_reference_config
        self.wavlm_model = wav2vec2_model(**to_reference_config(arch))
        self.weight_sum = nn.Linear(arch.num_layers + 1, 1, bias=False)
        self.proj = nn.Linear(arch.embed_dim, arch.head_dim_model)
        self.lnorm = nn.LayerNorm(arch.head_dim_model)
        self.channel_fusions = nn.ModuleList([CrossChannelAttention(n_units=arch.embed_dim, h_units=fusion_dim, h=fusion_heads)
                                              for _ in range(fusion_layers)])
        self.conformer = ConformerEncoder(attention_in=arch.head_dim_model, ffn_hidden=arch.head_ffn, num_head=arch.head_heads,
                                          num_layer=arch.head_layers, kernel_size=arch.head_kernel, dropout=0.1, use_posi=False,
                                          output_activate_function=False)
        self.classifier = nn.Linear(arch.head_dim_model, arch.num_classes)
        self.activation = nn.LogSoftmax(dim=-1)

    def forward(self, waveforms):
        assert waveforms.dim() == 3
        reps, _ = self.wavlm_model.extract_features_mc(waveforms, channel_fusions=self.channel_fusions)
        reps = [torch.mean(x, 1) if x.dim() == 4 else x for x in reps]
        x = torch.squeeze(self.weight_sum(torch.stack(reps, dim=-1)), -1)
        x = self.conformer(self.lnorm(self.proj(x)))
        out = self.activation(self.classifier(x))
        att = [f.att.reshape(out.shape[0], out.shape[1], *f.att.shape[1:]) for f in self.channel_fusions]
        return out, torch.stack([torch.mean(a, 2) for a in att], 1)     # (B, T, classes), (B, F, T, C, C)
