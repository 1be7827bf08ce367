"""CPU: checkpoint averaging / selection (reference diarizen/ckpt_utils.py, recipes/diar_ssl/infer_avg.py) and the wav.scp
command line (diarizen/pipelines/inference.py:194-368)."""
import os

import numpy as np
import pytest
import torch

from diarizen_b200 import checkpoints, cli

PINS = os.path.join(os.path.dirname(__file__), "golden", "reference_pins.npz")


def _states(n=4):
    g = torch.Generator().manual_seed(0)
    return [{"a.weight": torch.randn(3, 5, generator=g), "a.bias": torch.randn(3, generator=g),
             "bn.num_batches_tracked": torch.tensor(10 + i)} for i in range(n)]


def test_average_states_is_keywise_mean_and_leaves_inputs_alone():
    st = _states()
    keep = [{k: v.clone() for k, v in s.items()} for s in st]
    avg = checkpoints.average_states(st)
    for k in st[0]:
        torch.testing.assert_close(avg[k], torch.stack([s[k].double() for s in keep]).mean(0).to(avg[k].dtype))
        for s, s0 in zip(st, keep):
            assert torch.equal(s[k], s0[k])
    assert avg["bn.num_batches_tracked"].is_floating_point()   # true division, like the reference


def test_average_states_equals_reference():
    """bit-equal to what the reference's average_states returned for _states() (reference_pins.npz)."""
    z = np.load(PINS)
    theirs = {f[len("average_states/"):]: torch.from_numpy(z[f]) for f in z.files if f.startswith("average_states/")}
    ours = checkpoints.average_states(_states())
    assert ours.keys() == theirs.keys()
    for k in ours:
        assert torch.equal(ours[k], theirs[k])


def test_average_checkpoints_from_files(tmp_path):
    st = _states(3)
    paths = []
    for i, s in enumerate(st):
        p = tmp_path / f"epoch_{i:04d}" / "pytorch_model.bin"
        p.parent.mkdir()
        torch.save(s, p)
        paths.append({"bin_path": p} if i % 2 else str(p))
    avg = checkpoints.average_checkpoints(paths)
    torch.testing.assert_close(avg["a.weight"], (st[0]["a.weight"] + st[1]["a.weight"] + st[2]["a.weight"]) / 3)


def _summary(tmp_path, losses, ders):
    f = tmp_path / "val_metric_summary.lst"
    with open(f, "w") as fh:
        for e, (l, d) in enumerate(zip(losses, ders), start=1):
            # the trainer's message (recipes/diar_ssl/trainer_dual_opt.py:124), as collected into the summary file
            fh.write(f"Validation Loss/DER on epoch {e}: {l} / {d}\n")
    return f


def test_metric_summary_and_selection(tmp_path):
    losses = [0.9, 0.5, 0.4, 0.3, 0.35, 0.2, 0.25, 0.6]
    ders = [30.0, 20.0, 18.0, 15.0, 16.0, 12.0, 11.0, 25.0]
    recs = checkpoints.load_metric_summary(_summary(tmp_path, losses, ders), tmp_path / "checkpoints")
    assert [r["epoch"] for r in recs] == list(range(1, 9))
    assert recs[2]["bin_path"] == tmp_path / "checkpoints" / "epoch_0003" / "pytorch_model.bin"
    assert recs[5]["Loss"] == 0.2 and recs[6]["DER"] == 11.0
    best = checkpoints.select_checkpoints(recs, "Loss", "best", 3)
    assert [r["epoch"] for r in best] == [6, 7, 4]
    prev = checkpoints.select_checkpoints(recs, "Loss", "prev", 3)
    assert [r["epoch"] for r in prev] == [4, 5, 6]
    center = checkpoints.select_checkpoints(recs, "DER", "center", 3)     # best DER = epoch 7
    assert [r["epoch"] for r in center] == [6, 7, 8]
    with pytest.raises(AssertionError):
        checkpoints.select_checkpoints(recs, "DER", "center", 5)           # window runs past the last epoch


class _FakePipe:
    calls = []

    def __init__(self, hub, emb, **kw):
        _FakePipe.calls.append(("init", hub, emb, kw))

    def __call__(self, wav, sess_name=None):
        _FakePipe.calls.append(("call", wav, sess_name))


def test_cli_hub_mode_builds_the_reference_config(tmp_path):
    scp = tmp_path / "wav.scp"
    scp.write_text("sessA /data/sessA.wav\nsessB /data/sub/sessB.CH1.wav\n")
    _FakePipe.calls = []
    rc = cli.main(["--in_wav_scp", str(scp), "--diarizen_hub", str(tmp_path), "--embedding_model", "emb.bin",
                   "--clustering_method", "AgglomerativeClustering", "--ahc_threshold", "0.7", "--min_cluster_size", "30",
                   "--no-apply_median_filtering", "--batch_size", "8"], pipeline_factory=_FakePipe)
    assert rc == 0
    init = _FakePipe.calls[0]
    assert init[3]["config_parse"] == {
        "inference": {"args": {"seg_duration": 16, "segmentation_step": 0.1, "batch_size": 8, "apply_median_filtering": False}},
        "clustering": {"args": {"method": "AgglomerativeClustering", "min_speakers": 1, "max_speakers": 20, "ahc_threshold": 0.7,
                                "min_cluster_size": 30}}}
    assert [c[1:] for c in _FakePipe.calls[1:]] == [("/data/sessA.wav", "sessA"), ("/data/sub/sessB.CH1.wav", "sessB")]


def test_cli_experiment_mode_selects_and_passes_checkpoints(tmp_path):
    scp = tmp_path / "wav.scp"
    scp.write_text("s1 /d/s1.wav\n")
    exp = tmp_path / "exp"
    exp.mkdir()
    (exp / "config.toml").write_text("[model]\n[model.args]\nwavlm_src = 'wavlm_base'\n")
    summ = _summary(tmp_path, [0.5, 0.2, 0.3, 0.1, 0.4], [5, 4, 3, 2, 1])
    _FakePipe.calls = []
    cli.main(["-C", str(exp / "config.toml"), "-i", str(scp), "-o", str(tmp_path / "out"), "--embedding_model", "emb.bin",
              "--diarizen_hub", str(tmp_path / "hub"), "--val_metric_summary", str(summ), "--avg_ckpt_num", "2"],
             pipeline_factory=_FakePipe)
    kw = _FakePipe.calls[0][3]
    assert [r["epoch"] for r in kw["segmentation"]] == [4, 2]
    assert kw["segmentation"][0]["bin_path"] == exp / "checkpoints" / "epoch_0004" / "pytorch_model.bin"
    clu = kw["_config"]["clustering"]["args"]
    assert clu["method"] == "VBxClustering" and clu["plda_dir"] == os.path.join(str(tmp_path / "hub"), "plda")
    assert clu["Fa"] == 0.07 and clu["Fb"] == 0.8 and clu["lda_dim"] == 128 and clu["max_iters"] == 20
    assert kw["rttm_out_dir"] == str(tmp_path / "out")
    assert _FakePipe.calls[1] == ("call", "/d/s1.wav", "s1")
