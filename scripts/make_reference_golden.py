"""Generates tests/golden/reference_pins.npz: what the REFERENCE's own code returns on the inputs of the oracle-pinning
tests (run where the reference tree is available; DIARIZEN_REF points at it).  The tests replay the same inputs through
the oracle and the host code and compare with these outputs, so they run on any machine.

  seg/<arch>/logp, seg/<arch>/state_dict : reference Model (ref_loader.RefSegModel) on seeded weights and audio, and the
                                           layout "<key>:<shape>" of its floating-point state_dict
  wavlm_config/<name>                    : diarizen/models/module/wavlm_config.py get_config(name), as JSON
  receptive_field                        : (size, step, center) of pyannote-audio utils/receptive_field.py for the
                                           WavLM conv stack
  binarize/disc, binarize/rttm           : a {0,1} frame matrix and the RTTM of the reference's Binarize on it
  average_states/<key>                   : diarizen/ckpt_utils.py average_states on the states of test_checkpoints_cli
  vbx/<seed>/...                         : diarizen/clustering/VBx.py vbx_setup (psi, PLDA features of the training
                                           embeddings) and cluster_vbx (gamma, pi) for the test_vbx cases
"""
import importlib.util
import json
import os
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from diarizen_b200.archs import get_arch, init_state_dict  # noqa: E402
from oracle import ref_glue, ref_loader  # noqa: E402
from oracle.pipeline_oracle import filter_embeddings  # noqa: E402
import vbx_util  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "reference_pins.npz")

# the cases of tests/test_oracle_vs_reference.py, tests/test_vbx.py and tests/test_checkpoints_cli.py
SEG_CASES = [("tiny_base", 16000), ("tiny_large", 16000), ("wavlm_base_s80_md", 24000), ("wavlm_large_s80_md", 48000)]
SEG_WEIGHT_SEED, SEG_AUDIO_SEED = 4, 9
WAVLM_CONFIGS = ("wavlm_base", "wavlm_large", "wavlm_base_s80_md", "wavlm_large_s80_md")
VBX_SEEDS = (0, 1, 2)
VBX_PARAMS = ((0.07, 0.8), (0.3, 10.0))


def _module(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def checkpoint_states(n=4):
    g = torch.Generator().manual_seed(0)
    return [{"a.weight": torch.randn(3, 5, generator=g), "a.bias": torch.randn(3, generator=g),
             "bn.num_batches_tracked": torch.tensor(10 + i)} for i in range(n)]


def binarize_input():
    r = np.random.default_rng(0)
    disc = (r.random((4000, 3)) < 0.5).astype(np.float64)
    for k in range(3):                      # runs instead of salt and pepper
        disc[:, k] = np.repeat(r.random(400) < 0.4, 10)
    disc[-1, 0], disc[-2, 0] = 1.0, 0.0     # last frame only: zero-length turn
    return disc


def main():
    assert ref_loader.available() and ref_glue.available(), f"reference tree not found at {ref_loader.REF}"
    out = {}
    for name, N in SEG_CASES:
        a = get_arch(name)
        m = ref_loader.RefSegModel(a).eval()
        out[f"seg/{name}/state_dict"] = np.array(
            [f"{k}:{','.join(map(str, v.shape))}" for k, v in m.state_dict().items() if v.dtype.is_floating_point])
        m.load_state_dict(init_state_dict(a, seed=SEG_WEIGHT_SEED), strict=False)
        wav = 0.1 * torch.randn(2, N, generator=torch.Generator().manual_seed(SEG_AUDIO_SEED))
        with torch.inference_mode():
            out[f"seg/{name}/logp"] = m(wav[:, None]).numpy()
        print(name, out[f"seg/{name}/logp"].shape)

    sys.path.insert(0, ref_loader.REF)
    from diarizen.models.module.wavlm_config import get_config
    for name in WAVLM_CONFIGS:
        out[f"wavlm_config/{name}"] = np.array(json.dumps(get_config(name)))

    ns = ref_glue.load()
    ks, st, pd, dl = [10, 3, 3, 3, 3, 2, 2], [5, 2, 2, 2, 2, 2, 2], [0] * 7, [1] * 7
    rf = ns.receptive_field
    size = rf.multi_conv_receptive_field_size(1, kernel_size=ks, stride=st, padding=pd, dilation=dl)
    step = rf.multi_conv_receptive_field_size(2, kernel_size=ks, stride=st, padding=pd, dilation=dl) - size
    center = rf.multi_conv_receptive_field_center(0, kernel_size=ks, stride=st, padding=pd, dilation=dl)
    out["receptive_field"] = np.array([size, step, center], dtype=np.float64)

    disc = binarize_input()
    swf = ns.core.SlidingWindowFeature(disc, ns.core.SlidingWindow(start=0.0, duration=400 / 16000, step=320 / 16000))
    ann = ns.signal.Binarize(onset=0.5, offset=0.5, min_duration_on=0.0, min_duration_off=0.0)(swf)
    ann.uri = "x"
    out["binarize/disc"] = disc.astype(np.uint8)
    out["binarize/rttm"] = np.array(ann.to_rttm())

    ckpt = _module("ref_ckpt_utils", os.path.join(ref_loader.REF, "diarizen", "ckpt_utils.py"))
    for k, v in ckpt.average_states(checkpoint_states(), torch.device("cpu")).items():
        out[f"average_states/{k}"] = v.numpy()

    vbx = _module("ref_vbx", os.path.join(ref_loader.REF, "diarizen", "clustering", "VBx.py"))
    for seed in VBX_SEEDS:
        emb, seg = vbx_util.make_embeddings(seed)
        train, _, _ = filter_embeddings(emb, seg)
        with tempfile.TemporaryDirectory() as d:
            vbx_util.write_plda(d, seed)
            x_tf, plda_tf, psi = vbx.vbx_setup(d)
        fea = plda_tf(x_tf(train), lda_dim=128)
        out[f"vbx/{seed}/psi"] = psi
        out[f"vbx/{seed}/fea"] = fea
        labels = np.random.default_rng(seed).integers(0, 5, size=len(train))
        for Fa, Fb in VBX_PARAMS:
            gamma, pi = vbx.cluster_vbx(labels, fea, psi[:128], Fa=Fa, Fb=Fb, maxIters=20)
            out[f"vbx/{seed}/{Fa:g}_{Fb:g}/gamma"] = gamma
            out[f"vbx/{seed}/{Fa:g}_{Fb:g}/pi"] = pi
    np.savez_compressed(OUT, **out)
    print(OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    main()
