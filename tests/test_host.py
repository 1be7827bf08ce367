"""Host-side logic that needs no GPU: C ABI exports, architecture tables, result types, waveform decoding,
the relative-position bucket function, and the window sharding / gather used for N > 1 (gloo, world_size 2)."""
import io
import os
import re
import wave

import numpy as np
import pytest
import torch

from diarizen_b200 import _lib
from diarizen_b200.annotation import Annotation, Segment
from diarizen_b200.archs import ARCHS, get_arch, param_shapes

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "diarizen_b200.h")).read()
    declared = set(re.findall(r"\b(dz_[a-z0-9_]+)\s*\(", hdr))
    declared -= {"dz_gemm_desc", "dz_attn_args", "dz_seg_arch"}
    L = _lib.lib()
    missing = [s for s in sorted(declared) if not hasattr(L, s)]
    assert not missing, f"not exported: {missing}"
    assert set(_lib.EXPORTS) <= declared | {"dz_relpos_bucket"}
    assert L.dz_abi_version() == 1


def test_relpos_bucket_matches_oracle():
    from oracle.seg_oracle import rel_pos_bucket
    L = _lib.lib()
    d = torch.arange(-1700, 1701)
    mine = torch.tensor([L.dz_relpos_bucket(int(x)) for x in d])
    assert torch.equal(mine, rel_pos_bucket(d))


def test_no_cuda_means_loud_failure(monkeypatch):
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)     # a host without a CUDA device, also on a GPU machine
    from diarizen_b200.segmentation import SegmentationModel
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        SegmentationModel.random_init("tiny_base")


def test_num_frames_table():
    a = get_arch("wavlm_large_s80_md")
    assert [a.num_frames(n) for n in (16000, 80000, 128000, 256000)] == [49, 249, 399, 799]   # model_wavlm_conformer.py:113-124
    assert a.conv_frames(256000) == [51199, 25599, 12799, 6399, 3199, 1599, 799]


def test_param_shapes_count_parameters():
    # 94.38 M params for the unpruned base encoder stack (SURVEY.md 8c), 63.10 M for large-s80
    def wavlm_params(name):
        return sum(int(np.prod(s)) for k, s in param_shapes(get_arch(name)).items() if k.startswith("wavlm_model."))
    assert abs(wavlm_params("wavlm_base") / 1e6 - 94.38) < 0.05
    assert abs(wavlm_params("wavlm_large_s80_md") / 1e6 - 63.10) < 0.05
    for n in ARCHS:
        assert get_arch(n.upper()).name == n
    with pytest.raises(ValueError):
        get_arch("nope")


def test_annotation_protocol():
    ann = Annotation(uri="sess")
    ann[Segment(1.0, 2.5), 1] = 1
    ann[Segment(0.0, 2.7), 0] = 0
    ann[Segment(1.0, 2.0), 0] = 0
    tracks = list(ann.itertracks(yield_label=True))
    assert [t[0] for t in tracks] == [Segment(0.0, 2.7), Segment(1.0, 2.0), Segment(1.0, 2.5)]
    assert ann.to_rttm().splitlines()[0] == "SPEAKER sess 1 0.000 2.700 <NA> <NA> 0 <NA> <NA>"
    assert Annotation().to_rttm() == "" and ann.labels() == [0, 1]


def test_load_waveform_wav_bytes_and_dict(tmp_path):
    from diarizen_b200.pipeline import load_waveform
    x = (np.sin(np.arange(1600) / 10) * 20000).astype("<i2")
    stereo = np.stack([x, -x], axis=1)
    p = tmp_path / "a.wav"
    for target in (str(p), io.BytesIO()):
        with wave.open(target, "wb") as f:
            f.setnchannels(2); f.setsampwidth(2); f.setframerate(16000); f.writeframes(stereo.tobytes())
        if isinstance(target, io.BytesIO):
            target.seek(0)
        w = load_waveform(target)
        assert w.shape == (1600,) and torch.allclose(w, torch.from_numpy(x.astype(np.float32) / 32768.0))   # channel 0
    assert load_waveform({"waveform": torch.zeros(1, 7), "sample_rate": 16000}).shape == (7,)
    with pytest.raises(TypeError):
        load_waveform(3)


def _shard_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from diarizen_b200.sharding import gather_windows, window_range, window_ranges
    Cn, T = 11, 7
    a, b, per = window_range(Cn, rank, world)
    local = torch.zeros((per, T), dtype=torch.uint8)
    for c in range(a, b):
        local[c - a] = c + 1
    full = gather_windows(local, Cn, world)
    # the packed per-window records of the sharded pipeline: one collective for segmentations + counters + embeddings
    from diarizen_b200.sharding import gather_records
    seg = torch.zeros((per, T, 4), dtype=torch.uint8)
    stats = torch.zeros((per, 4, 2), dtype=torch.int32)
    emb = torch.zeros((per, 4, 5), dtype=torch.float32)
    for c in range(a, b):
        seg[c - a] = c % 2
        stats[c - a] = 1000 * c + torch.arange(8, dtype=torch.int32).view(4, 2)
        emb[c - a] = c + 0.25
    calls = []
    orig = dist.all_gather_into_tensor
    dist.all_gather_into_tensor = lambda *a_, **k_: (calls.append(1), orig(*a_, **k_))[1]
    g = gather_records(seg, stats, emb, Cn, world)
    dist.all_gather_into_tensor = orig
    # uneven split: the clustering rank (root 1 here) takes 40 % of an even share
    rg, per_u = window_ranges(Cn, world, root=1, root_share=0.4)
    ua, ub = rg[rank]
    seg_u = torch.zeros((per_u, T, 4), dtype=torch.uint8); st_u = torch.zeros((per_u, 4, 2), dtype=torch.int32); em_u = torch.zeros((per_u, 4, 5))
    for c in range(ua, ub):
        em_u[c - ua] = c + 0.5
    gu = gather_records(seg_u, st_u, em_u, Cn, world, rg)
    uneven_ok = rg == [(0, 9), (9, 11)] and per_u == 9 and all(float(gu[2][c, 0, 0]) == c + 0.5 for c in range(Cn)) and gu[0].shape[0] == Cn
    ok = (len(calls) == 1 and g[0].shape == (Cn, T, 4) and g[1].dtype == torch.int32 and g[2].dtype == torch.float32
          and all(int(g[0][c].max()) == c % 2 and int(g[1][c, 3, 1]) == 1000 * c + 7 and float(g[2][c, 0, 0]) == c + 0.25 for c in range(Cn)))
    # dispatch policy for several recordings (diarize_many): whole recordings round-robin, the remainder window-sharded with a rotating root
    from diarizen_b200.pipeline import DiariZenPipeline
    log = []

    class Fake(DiariZenPipeline):
        def __init__(self):
            self.rttm_out_dir = None

        def diarize_waveform(self, wav, shard=None, root=0):
            log.append((int(wav[0]), shard, root))
            return {"discrete": np.zeros((3, 1), dtype=np.uint8)} if (shard is False or rank == root) else {}

    outs = Fake().diarize_many([torch.full((4,), float(i)) for i in range(5)], [f"r{i}" for i in range(5)])
    q.put((rank, full.numpy(), ok and uneven_ok, log, [o is not None for o in outs]))
    dist.destroy_process_group()


def test_window_sharding_gloo_world2():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 500
    ps = [ctx.Process(target=_shard_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in ps:
        p.start()
    got = [q.get(timeout=120) for _ in range(2)]
    for p in ps:
        p.join(timeout=60)
    outs = {g[0]: g for g in got}
    expect = np.repeat(np.arange(1, 12, dtype=np.uint8)[:, None], 7, axis=1)
    assert np.array_equal(outs[0][1], expect) and np.array_equal(outs[1][1], expect)
    assert outs[0][2] and outs[1][2], "packed record gather"
    # 5 recordings on 2 ranks: 0..3 whole (rank = index mod 2, no collective), recording 4 sharded with root 4 % 2 = 0
    assert outs[0][3] == [(0, False, 0), (2, False, 0), (4, True, 0)] and outs[1][3] == [(1, False, 0), (3, False, 0), (4, True, 0)]
    assert outs[0][4] == [True, False, True, False, True] and outs[1][4] == [False, True, False, True, False]


def test_load_waveform_resamples_other_rates(tmp_path):
    """(f3) non-16 kHz input goes through torchaudio's resampler like the reference's Audio class."""
    import wave
    import numpy as np
    import torch
    torchaudio = __import__("pytest").importorskip("torchaudio")
    from diarizen_b200.pipeline import load_waveform
    sr = 8000
    t = np.arange(sr) / sr
    x = (0.5 * np.sin(2 * np.pi * 440.0 * t)).astype(np.float32)
    stereo = np.stack([x, -x], axis=1)
    p = tmp_path / "a8k.wav"
    with wave.open(str(p), "wb") as f:
        f.setnchannels(2); f.setsampwidth(2); f.setframerate(sr)
        f.writeframes((stereo * 32767).astype("<i2").tobytes())
    w = load_waveform(str(p))
    assert w.shape == (16000,) and w.dtype == torch.float32
    ref = torchaudio.functional.resample(torch.from_numpy((x * 32767).astype("<i2").astype(np.float32) / 32768.0)[None], sr, 16000)[0]
    assert torch.equal(w, ref)
    # channel 0, 440 Hz preserved
    spec = torch.fft.rfft(w).abs()
    assert int(spec.argmax()) == 440
    w2 = load_waveform({"waveform": torch.from_numpy(x)[None], "sample_rate": sr})
    assert w2.shape == (16000,)


def test_wav_decoder_formats(tmp_path):
    """24-bit PCM, 32-bit float and WAVE_FORMAT_EXTENSIBLE headers (what torchaudio.load accepts and the stdlib `wave` does not)."""
    import io
    import struct
    from diarizen_b200.pipeline import load_waveform
    sr, n = 16000, 800
    x = (0.5 * np.sin(2 * np.pi * 300 * np.arange(n) / sr)).astype(np.float32)

    def riff(fmt, data):
        body = b"WAVE" + b"fmt " + struct.pack("<I", len(fmt)) + fmt + b"LIST" + struct.pack("<I", 4) + b"abcd" + b"data" + struct.pack("<I", len(data)) + data
        return io.BytesIO(b"RIFF" + struct.pack("<I", len(body)) + body)

    i24 = np.round(x * 8388607).astype(np.int32)
    d24 = b"".join(struct.pack("<i", int(v))[:3] for v in i24)
    w = load_waveform(riff(struct.pack("<HHIIHH", 1, 1, sr, sr * 3, 3, 24), d24))
    assert w.shape == (n,) and torch.allclose(w, torch.from_numpy(i24.astype(np.float32) / 8388608.0))
    w = load_waveform(riff(struct.pack("<HHIIHH", 3, 1, sr, sr * 4, 4, 32), x.astype("<f4").tobytes()))
    assert torch.equal(w, torch.from_numpy(x))
    ext = struct.pack("<HHIIHH", 0xFFFE, 2, sr, sr * 4, 4, 16) + struct.pack("<HHI", 22, 16, 3) + struct.pack("<H", 1) + b"\x00" * 14
    st = np.stack([np.round(x * 32767), np.zeros(n)], axis=1).astype("<i2")
    w = load_waveform(riff(ext, st.tobytes()))
    assert w.shape == (n,) and torch.allclose(w, torch.from_numpy(st[:, 0].astype(np.float32) / 32768.0))
    with pytest.raises(ValueError):
        load_waveform(io.BytesIO(b"fLaC" + b"\x00" * 40))
