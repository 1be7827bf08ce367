#!/usr/bin/env python
"""Benchmark of the DiariZen inference hot path on B200 (contract: see the task statement).

Default workload (N=1): BASELINE.json configs[1] - WavLM-base-s80 segmentation forward, 5 s / 16 kHz windows,
batch 256 per GPU, synthetic audio, seeded random-init weights.  One "step" = one forward over one batch.
Metric = audio-seconds of window audio processed per wall second (RTF^-1), whole job (all ranks).

  python bench.py --gpus 1 --steps 10 --warmup 3
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
  python bench.py --impl reference         # the reference algorithm on the host cores (oracle port)
  python bench.py --dump-outputs DIR       # also write the last timed step's outputs as DIR/*.npy (to compare builds)
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

SR = 16000
METRIC = "audio-sec/s (RTF^-1)"


def synth_wav(B: int, N: int, seed: int = 1234) -> torch.Tensor:
    g = torch.Generator().manual_seed(seed)
    return (0.1 * torch.randn(B, N, generator=g)).clamp_(-1.0, 1.0)


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return {"hbm": float(p["hbm_gbs"]), "tensor": float(p.get("bf16_tflops_sustained", p["bf16_tflops"])), "src": "measured"}
    except Exception:
        return {"hbm": 6650.0, "tensor": 1400.0, "src": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return None
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return None
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


_THREADS = {}


def pick_threads(arch_name: str, N: int) -> int:
    """torch's intra-op pool degrades badly when oversubscribed on many-core hosts: try a few pool sizes on two
    windows and keep the fastest (that count is what `cores` reports)."""
    key = (arch_name, N)
    if key in _THREADS:
        torch.set_num_threads(_THREADS[key])
        return _THREADS[key]
    from diarizen_b200.archs import get_arch, init_state_dict
    from oracle.seg_oracle import seg_forward
    ncpu = os.cpu_count() or 1
    a = get_arch(arch_name)
    sd = init_state_dict(a, 0)
    wav = synth_wav(2, N)
    best, best_t = None, None
    for n in sorted({min(ncpu, c) for c in (8, 16, 32, 64, ncpu)}):
        torch.set_num_threads(n)
        seg_forward(a, sd, wav[:1])
        t0 = time.perf_counter()
        seg_forward(a, sd, wav)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = n, dt
    _THREADS[key] = best
    torch.set_num_threads(best)
    return best


def cpu_port_rate(arch_name: str, N: int, windows: int, chunk: int, repeats: int = 1):
    """The reference algorithm (oracle port, fp32 torch on the host cores) on a bounded sample."""
    from diarizen_b200.archs import get_arch, init_state_dict
    from oracle.seg_oracle import seg_forward
    cores = pick_threads(arch_name, N)
    a = get_arch(arch_name)
    sd = init_state_dict(a, 0)
    wav = synth_wav(windows, N)
    seg_forward(a, sd, wav[:min(2, windows)])  # warm-up
    best = None
    for _ in range(repeats):
        t0 = time.perf_counter()
        for i in range(0, windows, chunk):
            seg_forward(a, sd, wav[i:i + chunk])
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return windows * N / SR / best, cores, best


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.workload == "pipeline":
        return run_reference_pipeline(args)
    N = int(args.seconds * SR)
    per_step = args.ref_windows
    from diarizen_b200.archs import get_arch, init_state_dict
    from oracle.seg_oracle import seg_forward
    cores = pick_threads(args.arch, N)
    a = get_arch(args.arch)
    sd = init_state_dict(a, 0)
    wav = synth_wav(per_step, N)
    for _ in range(args.warmup):
        seg_forward(a, sd, wav[:max(1, per_step // 4)])
    t0 = time.perf_counter()
    for _ in range(args.steps):
        logp = seg_forward(a, sd, wav)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"logp": logp})
    val = args.steps * per_step * N / SR / dt
    sample = f"{per_step} windows x {args.seconds:g} s per step ({args.steps} steps), fp32 torch oracle port of Model.forward"
    out = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "audio-s/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args), "arch": args.arch, "window_s": args.seconds, "windows_per_step": per_step},
        "cpu_baseline": {"value": val, "unit": "audio-s/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(out)


def run_reference_pipeline(args):
    """Reference arm for the pipeline workload: per step, the oracle port of both network forwards on a bounded number of
    windows (the embedding trunk executed once per (window, speaker) pair as the reference does); stream rate = windows x
    step / time.  Clustering is NOT included in this arm's timed region (it is in cpu_baseline of the main arm)."""
    from diarizen_b200.archs import get_arch, init_resnet_state_dict, init_state_dict
    from oracle.emb_oracle import emb_forward
    from oracle.seg_oracle import seg_forward
    dur = args.seconds
    N = int(dur * SR)
    nw = max(1, args.ref_windows // 8)
    cores = pick_threads(args.arch, N)
    a = get_arch(args.arch)
    sd, esd = init_state_dict(a, 0), init_resnet_state_dict(0)
    wav = synth_wav(nw, N)
    T = a.num_frames(N)
    masks = torch.ones(nw, 1, T)

    def step():
        logp = seg_forward(a, sd, wav)
        for _ in range(4):
            emb = emb_forward(esd, wav, masks)
        return logp, emb
    for _ in range(max(1, args.warmup)):
        seg_forward(a, sd, wav[:1]); emb_forward(esd, wav[:1], masks[:1])
    t0 = time.perf_counter()
    for _ in range(args.steps):
        logp, emb = step()
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"logp": logp, "embeddings": emb})
    val = args.steps * nw * dur * 0.1 / dt
    sample = (f"{nw} windows x {dur:g} s per step ({args.steps} steps): oracle port of Model.forward + 4 ResNet34 passes per window "
              f"(trunk per (window, speaker) pair); stream seconds = windows x {dur * 0.1:g} s step; clustering excluded")
    out = {"impl": "reference", "metric": METRIC, "value": val, "unit": "audio-s/s", "n_gpus": args.gpus, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "f32", "data": "synthetic",
           "config": {"workload": f"{args.arch} full pipeline, {dur:g} s windows / {dur * 0.1:g} s step (BASELINE.json configs[2])", "arch": args.arch,
                      "window_s": dur, "windows_per_step": nw},
           "cpu_baseline": {"value": val, "unit": "audio-s/s", "cores": cores, "kind": "port", "sample": sample},
           "e2e": {"value": val, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(out)


def workload_name(args):
    return f"{args.arch} segmentation forward, {args.seconds:g} s / 16 kHz windows, batch {args.batch} per GPU (BASELINE.json configs[1])"


def classify(step_name: str) -> str:
    n = step_name
    if n.endswith("_attn"):
        return "attention"
    if "_ln" in n or n in ("fp_ln", "tr_ln", "head_ln"):
        return "layernorm"
    if n.startswith("conv0"):
        return "conv0"
    if n in ("wave_stats", "pc_stage", "mix_bf", "mix_last", "classifier") or n.endswith("_mix") or n.endswith("_gate") or n.endswith("_dwconv"):
        return "elementwise"
    return "gemm"


def _source(n: int, s: int, g: torch.Generator) -> torch.Tensor:
    """one synthetic 'speaker': harmonic complex on its own fundamental + coloured noise (spectrally distinct per speaker)"""
    t = torch.arange(n, dtype=torch.float32) / SR
    f0 = (95.0, 170.0, 290.0, 520.0)[s % 4] * (1.0 + 0.07 * (s // 4))
    noise = torch.randn(n, generator=g)
    if s % 2 == 0:
        noise = torch.cat([noise[:1], noise[1:] - 0.9 * noise[:-1]])
    else:
        noise = torch.nn.functional.conv1d(noise[None, None], torch.full((1, 1, 4), 0.25), padding=2)[0, 0, :n]
    x = 0.03 * noise
    for h in range(1, 9):
        x += (0.09 / h ** (0.5 + 0.5 * ((s // 2) % 2))) * torch.sin(2 * math.pi * f0 * h * t + s) * (1 + 0.3 * torch.sin(2 * math.pi * (1.5 + s) * t))
    return x


def synth_meeting(seconds: float, seed: int = 0, speakers: int = 4) -> torch.Tensor:
    """Synthetic 16 kHz mono 'meeting' (seeded): `speakers` spectrally distinct sources taking turns of 12-45 s; one turn in
    five starts 1-3 s before the previous one ends (overlapped speech), one in six is followed by 0.5-2 s of silence."""
    g = torch.Generator().manual_seed(seed)
    n = int(seconds * SR)
    wav = torch.zeros(n)
    pos, prev = 0, -1
    while pos < n:
        s = int(torch.randint(0, speakers, (1,), generator=g))
        if s == prev:
            s = (s + 1) % speakers
        prev = s
        length = int(torch.randint(12 * SR, 45 * SR, (1,), generator=g))
        start = pos
        r = torch.rand(1, generator=g).item()
        if r < 0.2 and pos > 3 * SR:
            start = pos - int(torch.randint(SR, 3 * SR, (1,), generator=g))
        elif r < 0.37:
            start = pos + int(torch.randint(SR // 2, 2 * SR, (1,), generator=g))
        end = min(n, start + length)
        if end > start:
            wav[start:end] += _source(end - start, s, g)
        pos = end
    return wav.clamp_(-1.0, 1.0)


def pipeline_cpu_rate(arch_name: str, seconds_per_window: float, step_s: float, n_seg: int, n_emb: int, emb_np=None, seg_np=None):
    """Reference algorithm on the host cores, bounded sample: oracle segmentation forward on n_seg windows, the embedding
    forward on n_emb windows executed as the reference does (trunk once per (window, speaker) pair: 4x), scipy clustering on
    the embeddings the GPU run produced.  -> (stream audio-s/s, cores, description)."""
    from diarizen_b200.archs import get_arch, init_resnet_state_dict, init_state_dict
    from oracle.emb_oracle import emb_forward
    from oracle.seg_oracle import seg_forward
    N = int(seconds_per_window * SR)
    cores = pick_threads(arch_name, N)
    a = get_arch(arch_name)
    sd = init_state_dict(a, 0)
    esd = init_resnet_state_dict(0)
    wav = synth_wav(max(n_seg, n_emb), N)
    T = a.num_frames(N)
    seg_forward(a, sd, wav[:1])
    t0 = time.perf_counter()
    seg_forward(a, sd, wav[:n_seg])
    t_seg = (time.perf_counter() - t0) / n_seg
    masks = torch.ones(n_emb, 1, T)
    emb_forward(esd, wav[:1], masks[:1])
    t0 = time.perf_counter()
    for _ in range(4):                       # speaker_diarization.py:295-322: one forward per (chunk, speaker)
        emb_forward(esd, wav[:n_emb], masks)
    t_emb = (time.perf_counter() - t0) / n_emb
    t_clu = 0.0
    n_train = 0
    if emb_np is not None and seg_np is not None:
        from oracle import pipeline_oracle as po
        t0 = time.perf_counter()
        try:
            po.cluster_call(emb_np, seg_np, 0.70, 30, 1, 20)
        except Exception:
            pass
        t_clu = time.perf_counter() - t0
        n_train = int(emb_np.shape[0] * emb_np.shape[1])
    per_window = t_seg + t_emb
    return per_window, t_clu, cores, (f"{n_seg} seg windows + {n_emb} windows x 4 embedding passes x {seconds_per_window:g} s, fp32 torch oracle port; "
                                      f"scipy centroid clustering of {n_train} embeddings: {t_clu:.1f} s; {per_window * 1e3:.0f} ms CPU per window")


SEG_KERNEL_OF = (  # step-name pattern -> kernel family the roofline is reported for
    ("_attn", "attention_tc2_kernel"), ("pos_conv", "posconv_tc_kernel"), ("conv0", "conv0_tc_kernel"),
)


def kernel_family(step_name: str) -> str:
    c = classify(step_name)
    if c == "gemm":
        return "posconv_tc_kernel" if step_name == "pos_conv" else "gemm_tc_tma_kernel"
    return {"attention": "attention_tc2_kernel", "layernorm": "layernorm_rows_fast_kernel", "conv0": "conv0_tc_kernel"}.get(c, "elementwise kernels")


def gemm_group(step_name: str) -> str:
    """finer groups inside the GEMM family, so that the line shows how far individual launches are from the peak"""
    n = step_name
    for suf in ("_qkv", "_out", "_ffn1", "_ffn2"):
        if n.endswith(suf) and n[0] == "L":
            return "wavlm" + suf
    if n.startswith("conv") and n[4:].isdigit():
        return "cnn_conv1-6"
    if n[0] == "C":
        return "conformer_head"
    return "other"


def build_hub_dir(root: str, arch_name: str, seed: int, classifier_gain: float, dur: float, batch: int, emb_sd=None) -> str:
    """Synthetic checkpoint FILES in the reference's hub-snapshot layout (diarizen_b200.checkpoints.write_hub_snapshot), so that
    the benchmarked pipeline is constructed through `DiariZenPipeline.from_pretrained(<dir>)` with a `{config, state_dict}` WavLM
    checkpoint - BASELINE.json configs[3]'s loader path (model_wavlm_conformer.py:209-221)."""
    from diarizen_b200.archs import get_arch, init_resnet_state_dict, init_state_dict
    from diarizen_b200.checkpoints import write_hub_snapshot
    arch = get_arch(arch_name)
    write_hub_snapshot(root, arch, init_state_dict(arch, seed, classifier_gain), emb_sd if emb_sd is not None else init_resnet_state_dict(seed),
                       {"seg_duration": dur, "segmentation_step": 0.1, "batch_size": batch, "apply_median_filtering": True},
                       {"method": "AgglomerativeClustering", "min_speakers": 1, "max_speakers": 20, "ahc_criterion": "distance",
                        "ahc_threshold": 0.70, "min_cluster_size": 30})
    return root


def centred_embedding_weights(pipe, wav_dev: torch.Tensor, window: int, T: int, seed: int):
    """Random-init ResNet embeddings are dominated by one common direction (every cosine distance < 0.03), so the clustering
    stage would always see ONE cluster.  The synthetic checkpoint therefore gets its last bias shifted by minus the mean
    embedding of 32 calibration windows: distances between the synthetic speakers then spread over [0.2, 1.8] and the
    agglomerative clustering, small-cluster re-assignment and multi-cluster reconstruction all do real work."""
    from diarizen_b200.archs import init_resnet_state_dict
    n = wav_dev.shape[0]
    starts = torch.linspace(0, n - window - 1, 32).long().tolist()
    w = torch.stack([wav_dev[s:s + window] for s in starts])
    e = pipe._embedding.embed_windows(w, torch.ones((32, 1, T), device=wav_dev.device))[:, 0]
    sd = init_resnet_state_dict(seed)
    sd["resnet.seg_1.bias"] = sd["resnet.seg_1.bias"] - e.mean(dim=0).cpu()
    return sd


def run_pipeline_bench(args, world, rank, local, dist):
    import tempfile
    from diarizen_b200.pipeline import DiariZenPipeline
    seconds = args.minutes * 60.0
    dur = args.seconds
    window = int(dur * SR)

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- model: synthetic checkpoint files in the hub layout, loaded through from_pretrained (configs[2] == configs[3] path) ----
    shared = synth_meeting(seconds, seed=100)              # the ONE recording every mode works on (same on every rank)
    probe = DiariZenPipeline.from_random_init(args.arch, seed=0, seg_duration=dur, batch_size=args.batch, classifier_gain=40.0,
                                              precision=args.precision)
    T = probe._segmentation.num_frames(window)
    emb_sd = centred_embedding_weights(probe, shared[: min(shared.shape[0], 20 * 60 * SR)].cuda(), window, T, seed=0)
    del probe
    hub = tempfile.mkdtemp(prefix=f"dz_hub_r{rank}_")
    build_hub_dir(hub, args.arch, 0, 40.0, dur, args.batch, emb_sd)
    pipe = DiariZenPipeline.from_pretrained(hub, precision=args.precision)
    wav_host = shared.pin_memory()
    wav_dev = wav_host.cuda()
    sharded = dist is not None
    steps = args.steps

    def one(dev_in: bool, shard):
        if dev_in:
            res = pipe.diarize_waveform(wav_dev, shard=shard)
            return pipe.to_annotation(res["discrete"], "bench") if res else None
        return pipe({"waveform": wav_host[None], "sample_rate": SR}, sess_name="bench", shard=shard)

    # ---- headline: device-resident; N > 1 = ONE recording window-sharded over the ranks (strong scaling) ----
    root_share = None
    if sharded and not args.even_split:
        one(True, sharded)
        # the rank that clusters takes a smaller window share, sized from measured stage times, so that with recordings
        # processed back to back (the timed loop) its networks + clustering end together with the other ranks' networks
        root_share = pipe.tune_root_share(wav_dev)
    for _ in range(args.warmup):
        one(True, sharded)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(steps):
        ann = one(True, sharded)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        res = pipe.last             # the dict the last timed diarize_waveform call returned; `ann` is its Annotation
        dump_outputs(args.dump_outputs, {"turns": turns(ann), **{k: res[k] for k in (
            "segmentations", "count", "embeddings", "hard_clusters", "discrete", "centroids") if res.get(k) is not None}})
    # ---- end to end: pinned host waveform in (each rank uploads the span of its own windows), Annotation out on rank 0 ----
    one(False, sharded)
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        ann = one(False, sharded)
    barrier()
    ms_e2e = 1e3 * (time.perf_counter() - t0)
    h2d = float(getattr(pipe, "last_h2d_bytes", 0))
    clocks = sampler.stop() if rank == 0 else None
    # ---- secondary (N > 1): one recording per rank, no collective (the replica mode the previous round reported) ----
    ms_rep = 0.0
    equal = None
    if sharded:
        pipe.diarize_waveform(wav_dev, shard=False)    # untimed: the engines re-plan for the unsharded batch shape
        barrier()
        t0 = time.perf_counter()
        res_un = pipe.diarize_waveform(wav_dev, shard=False)
        barrier()
        ms_rep = 1e3 * (time.perf_counter() - t0)
        if rank == 0:   # the NCCL-sharded result must be the unsharded one
            equal = ann is not None and ann.to_rttm() == pipe.to_annotation(res_un["discrete"], "bench").to_rttm()
    tt = torch.tensor([ms, ms_e2e, ms_rep, h2d], device="cuda", dtype=torch.float64)
    if dist is not None:
        tmax = tt.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = tt.clone()
        dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        ms, ms_e2e, ms_rep, h2d = float(tmax[0]), float(tmax[1]), float(tmax[2]), float(tsum[3])
    if rank != 0:
        return
    # ---- stage times of one recording (separate, synchronising pass; not part of any number above) ----
    stages = None
    if not sharded:
        pipe.collect_timing = True
        pipe.diarize_waveform(wav_dev, shard=False)
        stages = {k: round(v, 2) for k, v in pipe.last["timing"].items()}
        pipe.collect_timing = False
        last = pipe.last
    else:
        last = pipe.last if pipe.last else {}
    Cn, Tn = last["num_chunks"], last["num_frames"]
    peaks = measured_peaks()
    # ---- per-launch device times of one engine call of each network (CUDA events around every launch) ----
    bsz = pipe._planned.get("seg", pipe.engine_windows)      # windows per engine call the recording actually ran with
    wb = wav_dev[: window].repeat(bsz, 1).contiguous()
    pipe._segmentation.profile(wb)
    seg_prof = pipe._segmentation.profile(wb)
    ebs = pipe._planned.get("emb", pipe.engine_emb_windows)
    pipe._embedding.embed_windows(wb[:ebs], torch.ones(ebs, 4, Tn, device="cuda"))
    emb_prof = pipe._embedding.profile()
    n_seg_b, n_emb_b = Cn / bsz, Cn / ebs
    if args.profile_out:
        os.makedirs(os.path.dirname(os.path.abspath(args.profile_out)), exist_ok=True)
        with open(args.profile_out, "w") as f:
            json.dump({"seg": [{"name": n, "ms": m, "flops": fl, "bytes": by} for n, m, fl, by in seg_prof],
                       "emb": [{"name": n, "ms": m, "flops": fl} for n, m, fl in emb_prof],
                       "seg_batches": n_seg_b, "emb_batches": n_emb_b}, f, indent=0)
    fam, classes, groups = {}, {}, {}
    for name, pms, fl, by in seg_prof:
        for table, key in ((fam, kernel_family(name)), (classes, "seg:" + classify(name))):
            c = table.setdefault(key, {"ms": 0.0, "flops": 0.0, "bytes": 0.0, "n": 0})
            c["ms"] += pms * n_seg_b; c["flops"] += fl * n_seg_b; c["bytes"] += by * n_seg_b; c["n"] += 1
        if kernel_family(name) == "gemm_tc_tma_kernel":
            c = groups.setdefault(gemm_group(name), {"ms": 0.0, "flops": 0.0, "n": 0})
            c["ms"] += pms; c["flops"] += fl; c["n"] += 1
    for name, pms, fl in emb_prof:
        is_gemm = ("conv" in name and name != "conv1") or name.endswith("_sc") or name == "seg_1"
        for table, key in ((fam, "gemm_tc_tma_kernel" if is_gemm and "l1b" not in name and "l2b" not in name else ("conv3x3_kernel" if is_gemm else "embedding other")),
                           (classes, "emb:conv_gemm" if is_gemm else "emb:other")):
            c = table.setdefault(key, {"ms": 0.0, "flops": 0.0, "bytes": 0.0, "n": 0})
            c["ms"] += pms * n_emb_b; c["flops"] += fl * n_emb_b; c["n"] += 1
        if is_gemm:
            g = "resnet_" + name.split("b")[0] if name[0] == "l" else "resnet_other"
            c = groups.setdefault(g, {"ms": 0.0, "flops": 0.0, "n": 0})
            c["ms"] += pms; c["flops"] += fl; c["n"] += 1
    total_ms = sum(c["ms"] for c in classes.values())
    dom = max(fam, key=lambda k: fam[k]["ms"])
    d = fam[dom]
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
            traffic = json.load(f)
    except Exception:
        traffic = {}
    if d["flops"] > 0:
        ach = d["flops"] / (d["ms"] * 1e-3) / 1e12
        roof = {"bound": "tensor", "kernel": dom, "achieved": ach, "peak": peaks["tensor"], "unit": "TFLOP/s",
                "frac": ach / peaks["tensor"], "traffic": (traffic.get(dom) or {}).get("bytes_per_launch") if isinstance(traffic.get(dom), dict) else traffic.get(dom),
                "traffic_source": (traffic.get(dom) or {}).get("source") if isinstance(traffic.get(dom), dict) else None,
                "peak_source": peaks["src"] + " (sustained bf16)", "launches_per_recording": round(d["n"] * 1.0, 1),
                "share_of_network_time": d["ms"] / total_ms,
                "how": "sum of algorithmic FLOP of every launch of this kernel / sum of their CUDA-event durations (one engine call per network, events around each launch)"}
    else:
        ach = d["bytes"] / (d["ms"] * 1e-3) / 1e9
        roof = {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peaks["hbm"], "unit": "GB/s", "frac": ach / peaks["hbm"],
                "traffic": None, "peak_source": peaks["src"], "share_of_network_time": d["ms"] / total_ms}
    roof["groups"] = {k: {"launches": v["n"], "ms_per_engine_call": round(v["ms"], 3), "tflops": round(v["flops"] / (v["ms"] * 1e-3) / 1e12, 1),
                          "frac": round(v["flops"] / (v["ms"] * 1e-3) / 1e12 / peaks["tensor"], 3)}
                      for k, v in sorted(groups.items(), key=lambda kv: -kv[1]["ms"])}
    roof["other_kernels"] = {k: ({"ms_per_recording": round(v["ms"], 1), "tflops": round(v["flops"] / (v["ms"] * 1e-3) / 1e12, 1),
                                  "frac": round(v["flops"] / (v["ms"] * 1e-3) / 1e12 / peaks["tensor"], 3)} if v["flops"] > 0 else
                                 {"ms_per_recording": round(v["ms"], 1), "gbs": round(v["bytes"] / (v["ms"] * 1e-3) / 1e9, 1) if v["bytes"] else None,
                                  "frac": round(v["bytes"] / (v["ms"] * 1e-3) / 1e9 / peaks["hbm"], 3) if v["bytes"] else None})
                             for k, v in sorted(fam.items(), key=lambda kv: -kv[1]["ms"]) if k != dom}
    flop_per_audio_s = 136.6e9
    roof["whole_pipeline"] = {"tflops": round(flop_per_audio_s * seconds * steps / (ms * 1e-3) / 1e12 / world, 1),
                              "frac": round(flop_per_audio_s * seconds * steps / (ms * 1e-3) / 1e12 / world / peaks["tensor"], 3),
                              "note": "136.6 GFLOP per audio second (SURVEY.md 8d) x audio seconds / step time, per GPU"}
    breakdown = {k: {"ms_per_recording": round(v["ms"], 2), "share": round(v["ms"] / total_ms, 4),
                     "tflops": round(v["flops"] / (v["ms"] * 1e-3) / 1e12, 1) if v["flops"] else None}
                 for k, v in sorted(classes.items(), key=lambda kv: -kv[1]["ms"])}
    breakdown["networks_total_ms"] = round(total_ms, 1)
    breakdown["whole_recording_ms"] = round(ms / steps, 1)
    if stages:
        breakdown["stages_ms"] = stages
    cpu = None
    if not args.no_cpu_baseline:
        seg_np = last["segmentations"].cpu().numpy().astype("float32")
        per_w, t_clu, cores, desc = pipeline_cpu_rate(args.arch, dur, dur * 0.1, args.cpu_windows, max(1, args.cpu_windows // 2),
                                                      last["embeddings"], seg_np)
        cpu = {"value": seconds / (Cn * per_w + t_clu), "unit": "audio-s/s", "cores": cores, "kind": "port", "sample": desc}
    per_rank_windows = math.ceil(Cn / world)
    launches = (pipe._segmentation.last_launches * math.ceil(per_rank_windows / bsz) + pipe._embedding.last_launches * math.ceil(per_rank_windows / ebs) + 3) * world + 8
    hard = last["hard_clusters"]
    sub = {}
    if world == 1 and not args.no_sub_records:
        try:
            sub["cfg2_seg_base_s80"] = seg_sub_record(args)
        except Exception as e:  # the sub-record must never take the headline down
            sub["cfg2_seg_base_s80"] = {"error": str(e)[:200]}
    out = {
        "metric": METRIC, "value": seconds * steps / (ms * 1e-3), "unit": "audio-s/s", "n_gpus": world,
        "steps": steps, "warmup": args.warmup, "ms_per_step": ms / steps, "higher_is_better": True,
        "scaling": "strong" if world > 1 else "weak",
        "vs_baseline": None,
        "dtype": {"fp16": "fp16 operands, fp32 accumulate", "bf16": "bf16 operands, fp32 accumulate", "bf16x3": "bf16x3 split (fp32-class)"}[args.precision],
        "data": "synthetic (seeded 4-speaker meeting; seeded random-init weights written as checkpoint files in the hub layout, embedding bias centred - see bench.py centred_embedding_weights)",
        "config": {"workload": f"{args.arch} full pipeline (segmentation + ResNet34 embeddings + centroid AHC + reconstruction), ONE "
                               f"{args.minutes:g} min synthetic 16 kHz meeting, {dur:g} s windows / {dur * 0.1:g} s step (BASELINE.json configs[2]; "
                               f"model loaded through from_pretrained(<hub dir>) with a {{config, state_dict}} WavLM checkpoint = configs[3]'s path)",
                   "arch": args.arch, "window_s": dur, "windows_per_recording": Cn, "config_batch_size": args.batch,
                   "engine_windows_per_call": {"segmentation": bsz, "embedding": ebs},
                   "parallelism": (f"one recording window-sharded over {world} ranks ({per_rank_windows} windows each): both networks per rank, ONE NCCL "
                                   f"all-gather of packed uint8 segmentations + int32 frame counters + fp32 embeddings, clustering on rank 0"
                                   if world > 1 else "single GPU"),
                   "root_window_share": root_share,
                   "sharded_rttm_equals_unsharded": equal,
                   "replicas": ({"audio_s_per_s": world * seconds / (ms_rep * 1e-3), "ms": ms_rep,
                                 "note": "secondary: the same recording diarized unsharded on every rank at once (no collective), single shot"} if world > 1 else None),
                   "clusters_found": int(hard.max()) + 1, "speakers_in_output": int(last["discrete"].shape[1]),
                   "training_embeddings": int(((last["embeddings"] == last["embeddings"]).all(-1)).sum()),
                   "l2": "the recording (230 MB/h) and per-batch activations (GBs) exceed the 126 MB L2; no explicit flush"},
        "roofline": roof, "cpu_baseline": cpu,
        "e2e": {"value": seconds * steps / (ms_e2e * 1e-3), "unit": "audio-s/s", "h2d_bytes_per_step": int(h2d),
                "d2h_bytes_per_step": int(last["embeddings"].nbytes + last["discrete"].nbytes + last["hard_clusters"].nbytes),
                "ms_per_step": ms_e2e / steps},
        "gpu_launches": int(launches * steps), "clocks": clocks, "breakdown": breakdown,
    }
    if sub:
        out["sub_records"] = sub
    emit(out)


def run_many_bench(args, world, rank, local, dist):
    """BASELINE.json configs[4] in miniature: R synthetic recordings (seeds 0..R-1) handed to `DiariZenPipeline.diarize_many` -
    whole recordings round-robin over the ranks (each rank clusters its own, no collective), the R mod N left over
    window-sharded with a rotating clustering rank.  Host waveforms in, Annotations out; one step = the whole list."""
    import tempfile
    from diarizen_b200.pipeline import DiariZenPipeline
    seconds, dur, R = args.minutes * 60.0, args.seconds, args.recordings
    window = int(dur * SR)
    recs = [synth_meeting(seconds, seed=i).pin_memory() for i in range(R)]
    probe = DiariZenPipeline.from_random_init(args.arch, seed=0, seg_duration=dur, batch_size=args.batch, classifier_gain=40.0, precision=args.precision)
    T = probe._segmentation.num_frames(window)
    emb_sd = centred_embedding_weights(probe, recs[0].cuda(), window, T, seed=0)
    del probe
    hub = tempfile.mkdtemp(prefix=f"dz_hub_r{rank}_")
    build_hub_dir(hub, args.arch, 0, 40.0, dur, args.batch, emb_sd)
    pipe = DiariZenPipeline.from_pretrained(hub, precision=args.precision)
    names = [f"rec{i:03d}" for i in range(R)]

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
    pipe.diarize_many(recs[:max(world, 1)], names[:max(world, 1)])
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        outs = pipe.diarize_many(recs, names)
    barrier()
    dt = time.perf_counter() - t0
    if args.dump_outputs and rank == 0:      # rows of (recording, start s, end s, speaker label), the Annotations this rank returned
        rows = [np.insert(turns(o), 0, i, axis=1) for i, o in enumerate(outs) if o is not None]
        dump_outputs(args.dump_outputs, {"turns": np.concatenate(rows) if rows else np.zeros((0, 4))})
    done = torch.tensor([sum(o is not None for o in outs)], device="cuda")
    tt = torch.tensor([dt], device="cuda", dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(done)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    if rank != 0:
        return
    dt = float(tt[0])
    emit({"metric": METRIC, "value": R * seconds * args.steps / dt, "unit": "audio-s/s", "n_gpus": world, "steps": args.steps, "warmup": 1,
          "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
          "dtype": {"fp16": "fp16 operands, fp32 accumulate", "bf16": "bf16", "bf16x3": "bf16x3 split (fp32-class)"}[args.precision], "data": "synthetic",
          "config": {"workload": f"{R} x {args.minutes:g} min synthetic recordings through diarize_many (BASELINE.json configs[4] shape), host waveforms in, Annotations out",
                     "arch": args.arch, "recordings": R, "annotations_returned": int(done[0]),
                     "parallelism": f"recordings round-robin over {world} ranks, {R % max(world, 1)} window-sharded with a rotating clustering rank"},
          "e2e": {"value": R * seconds * args.steps / dt, "unit": "audio-s/s", "h2d_bytes_per_step": int(R * seconds * SR * 4), "d2h_bytes_per_step": None},
          "gpu_launches": None})


def seg_sub_record(args):
    """BASELINE.json configs[1] next to the headline: wavlm_base_s80_md, 256 x 5 s windows per step, device resident."""
    from diarizen_b200.segmentation import SegmentationModel
    N, B = 5 * SR, 256
    model = SegmentationModel.random_init("wavlm_base_s80_md", seed=0, precision=args.precision)
    wav = synth_wav(B, N).cuda()
    for _ in range(args.warmup):
        model.hard(wav)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        model.hard(wav)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    return {"workload": "wavlm_base_s80_md segmentation forward, 256 x 5 s windows per step", "ms_per_step": ms,
            "audio_s_per_s": B * 5.0 / (ms * 1e-3), "tflops": 256 * 15.2e9 / (ms * 1e-3) / 1e12,
            "frac_of_tensor_peak": 256 * 15.2e9 / (ms * 1e-3) / 1e12 / measured_peaks()["tensor"]}


DUMP_LIMIT = 64 * 10 ** 6     # bytes, all files of one --dump-outputs directory together


def turns(ann) -> np.ndarray:
    """Annotation -> (turns, 3) float64 rows of start s, end s, speaker label"""
    return np.array([(s.start, s.end, float(lab)) for s, _, lab in ann.itertracks(yield_label=True)], dtype=np.float64).reshape(-1, 3)


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """--dump-outputs: what the timed path returned in its last step, as out_dir/<name>.npy, so that two builds of the
    project can be compared output for output on identical inputs.  float64 stays float64; float32 and integers that
    float32 holds exactly become float32, other integers float64.  Above DUMP_LIMIT bytes in all, every array keeps the
    same fraction of its rows (first axis), drawn with a fixed seed and kept in order; the kept row numbers then go to
    <name>.rows.npy."""
    conv = {}
    for name, a in arrays.items():
        a = a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
        small_int = a.dtype.kind in "biu" and (a.size == 0 or int(np.abs(a.astype(np.int64)).max()) < 2 ** 24)
        conv[name] = a.astype(np.float32 if a.dtype == np.float32 or small_int else np.float64)
    header = 128                                          # bytes of one .npy header (numpy pads it to a multiple of 64)
    cost = sum(a.nbytes + (8 * a.shape[0] if a.ndim else 0) for a in conv.values())   # with the row numbers
    keep = min(1.0, (DUMP_LIMIT - 2 * header * len(conv)) / max(cost, 1))
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(0)
    for name, a in conv.items():
        if keep < 1.0 and a.ndim and a.shape[0] > 1:
            rows = np.sort(rng.choice(a.shape[0], max(1, int(a.shape[0] * keep)), replace=False))
            np.save(os.path.join(out_dir, name + ".rows.npy"), rows.astype(np.float64))
            a = a[rows]
        np.save(os.path.join(out_dir, name + ".npy"), a)


_JSON_OUT = sys.stdout


def emit(obj) -> None:
    """The ONE JSON line of the contract goes to the real stdout; everything else this process prints (the pipeline's
    reference-compatible progress prints, warnings) is routed to stderr by main()."""
    _JSON_OUT.write(json.dumps(obj) + "\n")
    _JSON_OUT.flush()


def main():
    # the ONE JSON line owns the real stdout: keep a private duplicate of file descriptor 1 for it and point fd 1 at stderr, so
    # that C-level writers (NCCL's version banner) cannot put anything else on stdout
    global _JSON_OUT
    try:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)
    except OSError:
        pass
    sys.stdout = sys.stderr
    os.environ.setdefault("NCCL_DEBUG", "WARN")   # keep NCCL's version banner off stdout
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps of every timed loop (default: 3 for pipeline, 5 for pipeline on N > 1, 1 for many, 10 for seg)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--recordings", type=int, default=16, help="--workload many: number of recordings in the list")
    ap.add_argument("--workload", default="pipeline", choices=["pipeline", "seg", "many"],
                    help="pipeline = BASELINE.json configs[2] (large-s80 full pipeline, the metric's configuration); seg = configs[1]")
    ap.add_argument("--arch", default=None)
    ap.add_argument("--seconds", type=float, default=None, help="window length")
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--minutes", type=float, default=60.0, help="recording length of the pipeline workload")
    ap.add_argument("--precision", default="fp16", choices=["fp16", "bf16", "bf16x3"])
    ap.add_argument("--profile-out", default=None, help="write the per-launch table (name, ms, flops, bytes) as JSON")
    ap.add_argument("--attn", default=os.environ.get("DZ_ATTN", "tc"), choices=["tc", "simt"])
    ap.add_argument("--ref-windows", type=int, default=16)
    ap.add_argument("--cpu-windows", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sub-records", action="store_true")
    ap.add_argument("--even-split", action="store_true", help="window-sharded mode: equal window shares (no smaller share for the clustering rank)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the timed path returned in its last step as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.workload in ("pipeline", "many"):
        args.arch = args.arch or "wavlm_large_s80_md"; args.seconds = args.seconds or 16.0; args.batch = args.batch or 32
        args.cpu_windows = args.cpu_windows or 4
    else:
        args.arch = args.arch or "wavlm_base_s80_md"; args.seconds = args.seconds or 5.0; args.batch = args.batch or 256
        args.cpu_windows = args.cpu_windows or 32
    world_env = int(os.environ.get("WORLD_SIZE", "1"))
    if args.steps is None:
        args.steps = (5 if world_env > 1 else 3) if args.workload == "pipeline" else (1 if args.workload == "many" else 10)
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    if args.impl == "reference":
        run_reference(args)
        return

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device (sm_100a); there is no CPU fallback")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    if args.workload == "many":
        run_many_bench(args, world, rank, local, dist)
        if dist is not None:
            dist.barrier()
            dist.destroy_process_group()
        return
    if args.workload == "pipeline":
        run_pipeline_bench(args, world, rank, local, dist)
        if dist is not None:
            dist.barrier()
            dist.destroy_process_group()
        return

    from diarizen_b200.segmentation import SegmentationModel
    N = int(args.seconds * SR)
    B = args.batch
    model = SegmentationModel.random_init(args.arch, seed=0, precision=args.precision, attn_impl=args.attn)
    wav_host = synth_wav(B, N, seed=1234 + rank).pin_memory()
    wav_dev = wav_host.cuda()
    T = model.num_frames(N)

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput ----
    for _ in range(args.warmup):
        model.hard(wav_dev)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        logp, ml = model.hard(wav_dev)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"logp": logp, "multilabel": ml})
    launches = model.last_launches * args.steps
    # ---- end to end through the host entry point (pinned host buffers, H2D + D2H inside) ----
    for _ in range(2):
        model.forward_host(wav_host)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        model.forward_host(wav_host)
    torch.cuda.synchronize()
    ms_e2e = 1e3 * (time.perf_counter() - t0)
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([ms, ms_e2e], device="cuda", dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = float(t[0]), float(t[1])
    audio_per_step = world * B * args.seconds

    if rank == 0:
        peaks = measured_peaks()
        prof = model.profile(wav_dev)
        prof = model.profile(wav_dev)
        if args.profile_out:
            os.makedirs(os.path.dirname(os.path.abspath(args.profile_out)), exist_ok=True)
            with open(args.profile_out, "w") as f:
                json.dump([{"name": n, "ms": m, "flops": fl, "bytes": by} for n, m, fl, by in prof], f, indent=0)
        classes = {}
        for name, pms, fl, by in prof:
            c = classes.setdefault(classify(name), {"ms": 0.0, "flops": 0.0, "bytes": 0.0, "n": 0})
            c["ms"] += pms; c["flops"] += fl; c["bytes"] += by; c["n"] += 1
        total_ms = sum(c["ms"] for c in classes.values())
        dom = max(classes, key=lambda k: classes[k]["ms"])
        d = classes[dom]
        npass = 3 if args.precision == "bf16x3" else 1
        if dom in ("gemm", "attention"):
            ach = d["flops"] / (d["ms"] * 1e-3) / 1e12
            roof = {"bound": "tensor", "kernel": "gemm_tc_tma_kernel / gemm_tc_kernel / posconv_tc_kernel" if dom == "gemm" else "attention_tc2_kernel", "achieved": ach,
                    "peak": peaks["tensor"], "unit": "TFLOP/s", "frac": ach / peaks["tensor"], "traffic": None,
                    "peak_source": peaks["src"] + " (sustained bf16)", "launches_per_step": d["n"],
                    "share_of_step": d["ms"] / total_ms, "tensor_passes": npass}
        else:
            ach = d["bytes"] / (d["ms"] * 1e-3) / 1e9
            roof = {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peaks["hbm"], "unit": "GB/s",
                    "frac": ach / peaks["hbm"], "traffic": None, "peak_source": peaks["src"], "launches_per_step": d["n"],
                    "share_of_step": d["ms"] / total_ms}
        try:
            with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
                tr = json.load(f)
            roof["traffic"] = tr.get(roof["kernel"])
        except Exception:
            pass
        breakdown = {k: {"ms": round(v["ms"], 3), "share": round(v["ms"] / total_ms, 4),
                         "tflops": round(v["flops"] / (v["ms"] * 1e-3) / 1e12, 1) if v["flops"] else None,
                         "gbs": round(v["bytes"] / (v["ms"] * 1e-3) / 1e9, 1) if v["bytes"] else None}
                     for k, v in sorted(classes.items(), key=lambda kv: -kv[1]["ms"])}
        cpu = None
        if not args.no_cpu_baseline:
            rate, cores, secs = cpu_port_rate(args.arch, N, args.cpu_windows, 16)
            cpu = {"value": rate, "unit": "audio-s/s", "cores": cores, "kind": "port",
                   "sample": f"{args.cpu_windows} windows x {args.seconds:g} s, fp32 torch oracle port of Model.forward, {secs:.1f} s of CPU work"}
        out = {
            "metric": METRIC, "value": audio_per_step * args.steps / (ms * 1e-3), "unit": "audio-s/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": {"fp16": "fp16 operands, fp32 accumulate", "bf16": "bf16 operands, fp32 accumulate", "bf16x3": "bf16x3 split (fp32-class)"}[args.precision],
            "data": "synthetic",
            "config": {"workload": workload_name(args), "arch": args.arch, "window_s": args.seconds, "batch_per_gpu": B,
                       "frames_per_window": T, "parallelism": f"dp{world} (windows sharded, no data-path collective)",
                       "l2": "inputs+activations per step (>1 GB) exceed the 126 MB L2; no explicit flush",
                       "attention_impl": args.attn},
            "roofline": roof,
            "cpu_baseline": cpu,
            "e2e": {"value": audio_per_step * args.steps / (ms_e2e * 1e-3), "unit": "audio-s/s",
                    "h2d_bytes_per_step": B * N * 4, "d2h_bytes_per_step": B * T * (model.arch.num_classes * 4 + 4),
                    "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": launches,
            "clocks": clocks,
            "breakdown": breakdown,
        }
        emit(out)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
