"""Pins the oracle against the reference modules themselves, through the outputs they produced on the same seeded inputs
(tests/golden/reference_pins.npz, written by scripts/make_reference_golden.py)."""
import json
import os

import numpy as np
import pytest
import torch

from diarizen_b200.archs import get_arch, init_state_dict, param_shapes
from oracle.seg_oracle import seg_forward

PINS = os.path.join(os.path.dirname(__file__), "golden", "reference_pins.npz")


@pytest.mark.parametrize("name,N", [("tiny_base", 16000), ("tiny_large", 16000), ("wavlm_base_s80_md", 24000),
                                    ("wavlm_large_s80_md", 48000)])      # the benchmarked architecture
def test_seg_oracle_equals_reference(name, N):
    z = np.load(PINS)
    a = get_arch(name)
    ref_keys = {k: tuple(int(d) for d in s.split(",") if d) for k, s in (e.split(":") for e in z[f"seg/{name}/state_dict"])}
    assert ref_keys == param_shapes(a), "state_dict layout must match the reference Model"
    sd = init_state_dict(a, seed=4)
    wav = 0.1 * torch.randn(2, N, generator=torch.Generator().manual_seed(9))
    ref = torch.from_numpy(z[f"seg/{name}/logp"])
    assert (seg_forward(a, sd, wav) - ref).abs().max().item() < 1e-5


def test_reference_config_roundtrip():
    from diarizen_b200.archs import arch_from_reference_config
    z = np.load(PINS)
    for name in ("wavlm_base", "wavlm_large", "wavlm_base_s80_md", "wavlm_large_s80_md"):
        a = arch_from_reference_config(json.loads(str(z[f"wavlm_config/{name}"])), name)
        b = get_arch(name)
        assert (a.large, a.conv_channels, a.embed_dim, a.total_heads, a.heads, a.ffn) == \
               (b.large, b.conv_channels, b.embed_dim, b.total_heads, b.heads, b.ffn)
