// Speaker-embedding engine: WeSpeaker ResNet34 (fbank -> CMN -> conv1 -> 16 BasicBlocks -> masked statistics
// pooling -> Linear 5120 -> 256).  Replaces `PyannoteAudioPretrainedSpeakerEmbedding.__call__`
// (reference: pyannote-audio/pyannote/audio/pipelines/speaker_verification.py:693-705) =
// `WeSpeakerResNet34.forward` (models/embedding/wespeaker/__init__.py:190-204, resnet.py:344-376).
//
// The trunk does not depend on the speaker mask (the mask only enters the pooling), so it runs ONCE per window and
// is pooled with all S (= 4) masks of that window; the reference runs the trunk once per (window, speaker) pair.
//
// HBM layout: activations are zero-bordered NHWC 16-bit planes [b][h = mel][1 + w = frame + 1][C]; every 3x3 / 1x1
// convolution is one tcgen05 GEMM per launch whose k loop walks the input rows of the window (gemm.h, conv2d mode),
// BatchNorm folded into weights + bias, ReLU and the residual add fused in the epilogue.
#include <cmath>
#include <map>
#include <string>
#include <vector>

#include "../../include/diarizen_b200.h"
#include "common.cuh"
#include "emb_kernels.h"
#include "engine_common.h"
#include "gemm.h"

namespace dz {
std::string& tls_error();
int fail(int code, const std::string& msg);
}  // namespace dz
using namespace dz;

static const int NBLOCKS[4] = {3, 4, 6, 3};

struct dz_emb {
  int precision = 2, planes = 1, npass = 1, fp16 = 1, gemm_impl = 0;
  std::map<std::string, std::vector<float>> params;
  bool finalized = false;
  // weights
  DevMem c1_w, c1_scale, c1_shift;
  struct Block { Weight conv1, conv2, sc; bool has_sc = false; int cin = 0, planes = 0, stride = 1; };
  std::vector<Block> blocks;
  Weight seg1;
  DevMem twiddle, window, mel_w, mel_range;
  // plan
  int B = 0, N = 0, S = 0, T = 0, F = 0;
  std::vector<Step> steps;
  std::vector<GemmPlan*> plans;
  std::vector<Conv3Plan*> c3plans;
  std::vector<ConvSPlan*> csplans;
  std::vector<DevMem*> ws;
  DevMem widx;
  const float* cur_wav = nullptr; const float* cur_masks = nullptr; float* cur_out = nullptr;
  float* fb_dev = nullptr;  // tap: fbank
  int last_launches = 0;
  cudaEvent_t done_event = nullptr; cudaStream_t last_stream = nullptr; bool ran = false;
  ~dz_emb() { clear_plan(); if (done_event) cudaEventDestroy(done_event); }
  void clear_plan() {
    for (auto* p : plans) gemm_plan_destroy(p);
    plans.clear();
    for (auto* p : c3plans) conv3x3_c32_plan_destroy(p);
    c3plans.clear();
    for (auto* p : csplans) conv3x3_stream_plan_destroy(p);
    csplans.clear();
    for (auto* w : ws) delete w;
    ws.clear();
    steps.clear();
    B = N = S = T = F = 0;
  }
};

static int emb_finalize(dz_emb* s) {
  g_weight_fp16() = s->fp16;
  auto get = [&](const std::string& k, size_t n, const std::vector<float>*& out) -> int {
    auto it = s->params.find(k);
    if (it == s->params.end()) return fail(DZ_ERR_STATE, "missing parameter " + k);
    if (it->second.size() != n) return fail(DZ_ERR_INVALID, "parameter " + k + " has the wrong size");
    out = &it->second;
    return DZ_OK;
  };
  auto fold_bn = [&](const std::string& bn, int C, std::vector<float>& scale, std::vector<float>& shift) -> int {
    const std::vector<float>*g, *b, *m, *v;
    int r;
    if ((r = get(bn + ".weight", C, g)) || (r = get(bn + ".bias", C, b)) || (r = get(bn + ".running_mean", C, m)) ||
        (r = get(bn + ".running_var", C, v)))
      return r;
    scale.resize(C); shift.resize(C);
    for (int c = 0; c < C; ++c) {
      const double inv = (double)(*g)[c] / std::sqrt((double)(*v)[c] + 1e-5);
      scale[c] = (float)inv;
      shift[c] = (float)((double)(*b)[c] - (double)(*m)[c] * inv);
    }
    return DZ_OK;
  };
  cudaError_t e;
  const std::string P = "resnet.";
  {
    const std::vector<float>* w;
    int r = get(P + "conv1.weight", 32 * 9, w);
    if (r) return r;
    std::vector<float> sc, sh;
    if ((r = fold_bn(P + "bn1", 32, sc, sh))) return r;
    if ((e = upload_vec(s->c1_w, *w)) || (e = upload_vec(s->c1_scale, sc)) || (e = upload_vec(s->c1_shift, sh)))
      return fail(DZ_ERR_CUDA, cudaGetErrorString(e));
  }
  // conv weight [Cout][Cin][kh][kw] * bn scale -> GEMM B [Cout][kh][pad64(kw*Cin)] with element (kw, ci) at kw*Cin + ci
  auto conv_weight = [&](const std::string& wname, const std::string& bn, int Cout, int Cin, int ks, Weight& W) -> int {
    const std::vector<float>* w;
    int r = get(wname, (size_t)Cout * Cin * ks * ks, w);
    if (r) return r;
    std::vector<float> sc, sh;
    if ((r = fold_bn(bn, Cout, sc, sh))) return r;
    const int run = ks * Cin, krun = rup(run, 64);
    std::vector<float> g((size_t)Cout * ks * krun, 0.f);
    for (int co = 0; co < Cout; ++co)
      for (int ci = 0; ci < Cin; ++ci)
        for (int kh = 0; kh < ks; ++kh)
          for (int kw = 0; kw < ks; ++kw)
            g[((size_t)co * ks + kh) * krun + kw * Cin + ci] = (*w)[(((size_t)co * Cin + ci) * ks + kh) * ks + kw] * sc[co];
    cudaError_t ce = make_weight(W, g.data(), 1, Cout, ks * krun, sh.data(), Cout);
    return ce == cudaSuccess ? DZ_OK : fail(DZ_ERR_CUDA, cudaGetErrorString(ce));
  };
  int cin = 32;
  s->blocks.clear();
  s->blocks.reserve(16);
  for (int li = 0; li < 4; ++li) {
    const int planes = 32 << li;
    for (int bi = 0; bi < NBLOCKS[li]; ++bi) {
      s->blocks.emplace_back();
      dz_emb::Block& b = s->blocks.back();
      b.cin = cin; b.planes = planes; b.stride = (bi == 0 && li > 0) ? 2 : 1;
      const std::string bp = P + "layer" + std::to_string(li + 1) + "." + std::to_string(bi) + ".";
      int r;
      if ((r = conv_weight(bp + "conv1.weight", bp + "bn1", planes, cin, 3, b.conv1))) return r;
      if ((r = conv_weight(bp + "conv2.weight", bp + "bn2", planes, planes, 3, b.conv2))) return r;
      b.has_sc = (b.stride != 1 || cin != planes);
      if (b.has_sc && (r = conv_weight(bp + "shortcut.0.weight", bp + "shortcut.1", planes, cin, 1, b.sc))) return r;
      cin = planes;
    }
  }
  {
    const std::vector<float>*w, *b;
    int r;
    if ((r = get(P + "seg_1.weight", (size_t)256 * 5120, w)) || (r = get(P + "seg_1.bias", 256, b))) return r;
    e = make_weight(s->seg1, w->data(), 1, 256, 5120, b->data(), 256);
    if (e != cudaSuccess) return fail(DZ_ERR_CUDA, cudaGetErrorString(e));
  }
  // fbank constants (torchaudio.compliance.kaldi: hamming window, mel banks low 20 Hz .. Nyquist, 80 bins, 512-pt FFT)
  {
    std::vector<float> tw(512), win(400), mel((size_t)80 * 257, 0.f);
    std::vector<int> rng(160);
    for (int k = 0; k < 256; ++k) {
      const double ang = -2.0 * M_PI * k / 512.0;
      tw[2 * k] = (float)std::cos(ang); tw[2 * k + 1] = (float)std::sin(ang);
    }
    for (int i = 0; i < 400; ++i) win[i] = (float)(0.54 - 0.46 * std::cos(2.0 * M_PI * i / 399.0));
    auto melf = [](double f) { return 1127.0 * std::log(1.0 + f / 700.0); };
    const double lo = melf(20.0), hi = melf(8000.0), delta = (hi - lo) / 81.0, binw = 16000.0 / 512.0;
    for (int m = 0; m < 80; ++m) {
      const double left = lo + m * delta, center = lo + (m + 1) * delta, right = lo + (m + 2) * delta;
      int ks = 257, ke = 0;
      for (int k = 0; k < 256; ++k) {
        const double mk = melf(binw * k);
        const double up = (mk - left) / (center - left), down = (right - mk) / (right - center);
        const double v = std::max(0.0, std::min(up, down));
        mel[(size_t)m * 257 + k] = (float)v;
        if (v > 0.0) { ks = std::min(ks, k); ke = std::max(ke, k + 1); }
      }
      if (ke <= ks) { ks = 0; ke = 0; }
      rng[2 * m] = ks; rng[2 * m + 1] = ke;
    }
    auto it = s->params.find("fbank.mel_banks");   // optional override with the host library's own table
    if (it != s->params.end() && it->second.size() == (size_t)80 * 257) {
      mel = it->second;
      for (int m = 0; m < 80; ++m) {
        int ks = 257, ke = 0;
        for (int k = 0; k < 257; ++k) if (mel[(size_t)m * 257 + k] != 0.f) { ks = std::min(ks, k); ke = std::max(ke, k + 1); }
        if (ke <= ks) { ks = 0; ke = 0; }
        rng[2 * m] = ks; rng[2 * m + 1] = ke;
      }
    }
    auto iw = s->params.find("fbank.window");
    if (iw != s->params.end() && iw->second.size() == 400) win = iw->second;
    if ((e = upload_vec(s->twiddle, tw)) || (e = upload_vec(s->window, win)) || (e = upload_vec(s->mel_w, mel)))
      return fail(DZ_ERR_CUDA, cudaGetErrorString(e));
    if ((e = s->mel_range.alloc(rng.size() * 4, false)) || (e = cudaMemcpy(s->mel_range.p, rng.data(), rng.size() * 4, cudaMemcpyHostToDevice)))
      return fail(DZ_ERR_CUDA, cudaGetErrorString(e));
  }
  s->finalized = true;
  s->params.clear();
  return DZ_OK;
}

static int emb_plan(dz_emb* s, int B, int N, int S, int T) {
  s->clear_plan();
  if (N < 400) return fail(DZ_ERR_INVALID, "window shorter than one fbank frame");
  const int F = 1 + (N - 400) / 160;
  const int P = s->planes, FP = s->fp16;
  int err = 0; std::string msg;
  auto buf = [&](size_t bytes, bool zero) -> DevMem* {
    DevMem* m = new DevMem(); s->ws.push_back(m);
    cudaError_t e = m->alloc(bytes, zero);
    if (e != cudaSuccess && !err) { err = DZ_ERR_CUDA; msg = std::string("workspace allocation failed: ") + cudaGetErrorString(e); }
    return m;
  };
  // geometry per stage
  int Hs[4], Ws[4];
  Hs[0] = 80; Ws[0] = F;
  for (int i = 1; i < 4; ++i) { Hs[i] = (Hs[i - 1] - 1) / 2 + 1; Ws[i] = (Ws[i - 1] - 1) / 2 + 1; }
  size_t act_elems = 0;
  for (int i = 0; i < 4; ++i) act_elems = std::max(act_elems, (size_t)B * Hs[i] * (Ws[i] + 2) * (32 << i));
  Planes act[4];
  for (int i = 0; i < 4; ++i) {
    DevMem* m = buf((act_elems + 256) * 2 * P, true);   // borders must be (and stay) zero
    act[i].p = m->as<bf16>(); act[i].plane = (long long)act_elems + 256;
  }
  Conv1Args conv1_args{};
  float* fb = buf((size_t)B * F * 80 * 4, false)->as<float>();
  float* fbm = buf((size_t)B * 80 * 4, false)->as<float>();
  s->fb_dev = fb;
  {
    FbankArgs a{};
    a.N = N; a.F = F; a.twiddle = s->twiddle.as<float2>(); a.window = s->window.as<float>(); a.mel_w = s->mel_w.as<float>();
    a.mel_range = s->mel_range.as<int>(); a.out = fb;
    s->steps.push_back({"fbank", [s, a, B](cudaStream_t st) { FbankArgs aa = a; aa.wav = s->cur_wav; return launch_fbank(aa, B, st); }, 0.0,
                        (double)B * N * 4 + (double)B * F * 80 * 4});
    s->steps.push_back({"fbank_mean", [=](cudaStream_t st) { return launch_fbank_mean(fb, B, F, fbm, st); }, 0.0, (double)B * F * 80 * 4});
    // (the clear of act[0] is inserted below, before conv1, through ensure_geom)
    Conv1Args c{};
    c.fb = fb; c.mean = fbm; c.B = B; c.F = F; c.w = s->c1_w.as<float>(); c.scale = s->c1_scale.as<float>(); c.shift = s->c1_shift.as<float>();
    c.out = act[0].p; c.out_plane = act[0].plane; c.planes = P; c.fp16 = FP;
    conv1_args = c;
  }
  // Zero borders: a buffer is read by the next convolution with geometry (H, W, C); its border columns w = 0 and
  // w = W + 1 must be zero (the interior is fully overwritten by the producer, rows outside [0, H) are never addressed:
  // TMA zero-fills them).  Whenever a buffer is about to be written with a geometry different from the one it last held
  // (stage transitions, and the first use in every forward) only those two columns are cleared.
  long long geom[4] = {-1, -1, -1, -1};
  auto ensure_geom = [&](int bi, int Hh, int Ww, int Cc, const std::string& nm) {
    const long long g = ((long long)Hh << 40) | ((long long)Ww << 16) | Cc;
    if (geom[bi] == g) return;
    geom[bi] = g;
    bf16* p = act[bi].p;
    const long long plane = act[bi].plane;
    const long long rows = (long long)B * Hh;
    const int np = P;
    s->steps.push_back({nm, [=](cudaStream_t st) { return launch_zero_borders(p, plane, np, rows, Ww, Cc, st); }, 0.0,
                        (double)rows * 2 * Cc * 2 * np});
  };
  auto conv = [&](const std::string& nm, Planes in, int Hin, int Win, int Cin, const Weight& W, int ks, int stride, Planes out,
                  const Planes* res, int act) {
    const int pad = ks == 3 ? 1 : 0;
    const int Ho = (Hin + 2 * pad - ks) / stride + 1, Wo = (Win + 2 * pad - ks) / stride + 1, Cout = W.N;
    GemmDesc d = gemm_desc_default();
    d.M = Wo; d.N = Cout; d.K = W.K; d.batches = B * Ho; d.npass = s->npass; d.out_planes = P; d.fp16 = FP;
    d.a = in.p; d.a_plane = in.plane; d.a_rstride = (long long)stride * Cin; d.a_kinner = W.K;
    d.a_hstride = (long long)(Win + 2) * Cin; d.a_bstride = (long long)Hin * (Win + 2) * Cin;
    d.conv_runs = ks; d.conv_run_len = ks * Cin; d.conv_x0 = ks == 3 ? 0 : Cin; d.conv_h0 = -pad; d.conv_hs = stride;
    d.conv_Ho = Ho; d.conv_H = Hin;
    d.b = W.w.p; d.b_plane = W.plane; d.ldb = W.ldb; d.b_gstride = W.gstride; d.bias = W.bias.as<float>();
    d.act = act; d.act_after_res = 1;
    if (res) { d.res16 = res->p; d.res16_plane = res->plane; d.res16_bstride = (long long)(Wo + 2) * Cout; d.ldr16 = Cout; d.res16_row_off = 1; }
    d.out_bf = out.p; d.ob_plane = out.plane; d.ob_bstride = (long long)(Wo + 2) * Cout; d.ldob = Cout; d.out_row_off = 1;
    const double flops = 2.0 * B * Ho * Wo * (double)Cout * ks * ks * Cin;
    if (s->gemm_impl == 1) {
      s->steps.push_back({nm, [d](cudaStream_t st) { return gemm_simt_launch(d, st); }, flops, 0.0});
      return;
    }
    if (ks == 3 && stride == 1 && Cin == Cout && (Cin == 32 || Cin == 64) && P == 1 && s->npass == 1 && act == 3) {
      // layer1 / layer2: resident weights + row-shifted A views instead of the generic implicit GEMM (conv3x3_c32.cu)
      Conv3Args c{};
      c.in = in.p; c.out = out.p; c.res = res ? res->p : nullptr; c.w = W.w.as<bf16>(); c.ldw = W.ldb; c.bias = W.bias.as<float>();
      c.B = B; c.H = Hin; c.W = Win; c.relu = 1; c.fp16 = FP; c.C = Cin;
      Conv3Plan* cp = conv3x3_c32_plan_create(c);
      if (!cp) { if (!err) { err = DZ_ERR_CUDA; msg = "conv3x3 plan '" + nm + "': " + gemm_last_error(); } return; }
      s->c3plans.push_back(cp);
      s->steps.push_back({nm, [cp](cudaStream_t st) { return conv3x3_c32_plan_launch(cp, st); }, flops, 0.0});
      return;
    }
    if (ks == 3 && stride == 1 && Cin == Cout && Cin == 128 && P == 1 && s->npass == 1 && act == 3) {
      // layer3: streamed weights, two output rows per tile, row-shifted A views (conv3x3_c128.cu)
      Conv3Args c{};
      c.in = in.p; c.out = out.p; c.res = res ? res->p : nullptr; c.w = W.w.as<bf16>(); c.ldw = W.ldb; c.bias = W.bias.as<float>();
      c.B = B; c.H = Hin; c.W = Win; c.relu = 1; c.fp16 = FP; c.C = Cin;
      ConvSPlan* cp = conv3x3_stream_plan_create(c);
      if (!cp) { if (!err) { err = DZ_ERR_CUDA; msg = "conv3x3 stream plan '" + nm + "': " + gemm_last_error(); } return; }
      s->csplans.push_back(cp);
      s->steps.push_back({nm, [cp](cudaStream_t st) { return conv3x3_stream_plan_launch(cp, st); }, flops, 0.0});
      return;
    }
    GemmPlan* p = gemm_plan_create(d, 0);
    if (!p) { if (!err) { err = DZ_ERR_CUDA; msg = "gemm plan '" + nm + "': " + gemm_last_error(); } return; }
    s->plans.push_back(p);
    s->steps.push_back({nm, [p](cudaStream_t st) { return gemm_plan_launch(p, st); }, flops, 0.0});
  };
  ensure_geom(0, 80, F, 32, "clr_conv1");
  {
    const Conv1Args c = conv1_args;
    s->steps.push_back({"conv1", [c](cudaStream_t st) { return launch_emb_conv1(c, st); }, 2.0 * B * 80 * F * 9 * 32,
                        (double)B * F * 80 * 4 + (double)B * 80 * (F + 2) * 32 * 2 * P});
  }
  // buffers: x = block input, y = conv1 output, sc = shortcut output, o = block output (rotating)
  int xi = 0;   // index of the buffer holding the current block input
  int curH = 80, curW = F, curC = 32;
  int bidx = 0;
  for (int li = 0; li < 4; ++li) {
    for (int bi = 0; bi < NBLOCKS[li]; ++bi, ++bidx) {
      dz_emb::Block& b = s->blocks[bidx];
      const std::string nm = "l" + std::to_string(li + 1) + "b" + std::to_string(bi);
      const int yi = (xi + 1) & 3, si = (xi + 2) & 3, oi = (xi + 3) & 3;
      const int Ho = (curH - 1) / b.stride + 1, Wo = (curW - 1) / b.stride + 1;
      ensure_geom(yi, Ho, Wo, b.planes, nm + "_clr_y");
      if (b.has_sc) ensure_geom(si, Ho, Wo, b.planes, nm + "_clr_sc");
      ensure_geom(oi, Ho, Wo, b.planes, nm + "_clr_o");
      conv(nm + "_conv1", act[xi], curH, curW, curC, b.conv1, 3, b.stride, act[yi], nullptr, 3);
      const Planes* res = &act[xi];
      if (b.has_sc) {
        conv(nm + "_sc", act[xi], curH, curW, curC, b.sc, 1, b.stride, act[si], nullptr, 0);
        res = &act[si];
      }
      conv(nm + "_conv2", act[yi], Ho, Wo, b.planes, b.conv2, 3, 1, act[oi], res, 3);
      xi = oi; curH = Ho; curW = Wo; curC = b.planes;
    }
  }
  // pooling + final linear
  const int W4 = curW, H4 = curH, C4 = curC;   // 200, 10, 256 for 16 s
  {
    std::vector<int> wi(W4);
    const float scale = (float)T / (float)W4;   // F.interpolate(mode="nearest"): src = min(floor(dst * scale), T - 1)
    for (int w = 0; w < W4; ++w) { int v = (int)floorf((float)w * scale); wi[w] = v < T - 1 ? v : T - 1; }
    cudaError_t e = s->widx.alloc(W4 * 4, false);
    if (e == cudaSuccess) e = cudaMemcpy(s->widx.p, wi.data(), W4 * 4, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) return fail(DZ_ERR_CUDA, cudaGetErrorString(e));
  }
  const int feat = 2 * C4 * H4;
  DevMem* stm = buf(((size_t)B * S * feat + 256) * 2 * P, true);
  Planes stats; stats.p = stm->as<bf16>(); stats.plane = (long long)B * S * feat + 256;
  {
    PoolArgs a{};
    a.x = act[xi].p; a.x_plane = act[xi].plane; a.planes = P; a.fp16 = FP; a.H = H4; a.W = W4; a.C = C4; a.S = S; a.T = T;
    a.widx = s->widx.as<int>(); a.out = stats.p; a.out_plane = stats.plane; a.ldo = feat;
    s->steps.push_back({"stats_pool", [s, a, B](cudaStream_t st) { PoolArgs aa = a; aa.masks = s->cur_masks; return launch_stats_pool(aa, B, st); },
                        0.0, (double)B * H4 * (W4 + 2) * C4 * 2 * P * 2});
    GemmDesc d = gemm_desc_default();
    d.M = B * S; d.N = 256; d.K = feat; d.npass = s->npass; d.out_planes = P; d.fp16 = FP;
    d.a = stats.p; d.a_plane = stats.plane; d.a_rstride = feat; d.a_kinner = feat; d.a_rows_alloc = B * S;
    d.b = s->seg1.w.p; d.b_plane = s->seg1.plane; d.ldb = s->seg1.ldb; d.b_gstride = s->seg1.gstride; d.bias = s->seg1.bias.as<float>();
    d.ldo = 256;
    const double flops = 2.0 * B * S * 256.0 * feat;
    if (s->gemm_impl == 1) {
      s->steps.push_back({"seg_1", [s, d](cudaStream_t st) { GemmDesc dd = d; dd.out_f32 = s->cur_out; return gemm_simt_launch(dd, st); }, flops, 0.0});
    } else {
      // the output pointer changes per call: plan per call is cheap here (one tiny GEMM)
      s->steps.push_back({"seg_1", [s, d](cudaStream_t st) {
        GemmDesc dd = d; dd.out_f32 = s->cur_out;
        GemmPlan* p = gemm_plan_create(dd, 0);
        if (!p) return cudaErrorInvalidValue;
        cudaError_t e = gemm_plan_launch(p, st);
        gemm_plan_destroy(p);
        return e;
      }, flops, 0.0});
    }
  }
  if (err) { s->clear_plan(); return fail(err, msg); }
  s->B = B; s->N = N; s->S = S; s->T = T; s->F = F;
  return DZ_OK;
}

extern "C" {

dz_emb* dz_emb_create(int precision, int gemm_impl) {
  if (precision != 1 && precision != 2 && precision != 3) { fail(DZ_ERR_INVALID, "precision must be 1 (bf16), 2 (fp16) or 3 (bf16x3)"); return nullptr; }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { fail(DZ_ERR_CUDA, "no CUDA device: diarizen_b200 has no CPU fallback"); return nullptr; }
  dz_emb* s = new dz_emb();
  s->precision = precision; s->planes = precision == 3 ? 2 : 1; s->npass = precision == 3 ? 3 : 1; s->fp16 = precision == 2 ? 1 : 0;
  s->gemm_impl = gemm_impl;
  return s;
}
void dz_emb_destroy(dz_emb* s) { delete s; }
int dz_emb_set_param(dz_emb* s, const char* name, const float* host_data, int64_t numel) {
  if (!s || !name || !host_data || numel < 0) return fail(DZ_ERR_INVALID, "bad argument");
  if (s->finalized) return fail(DZ_ERR_STATE, "engine already finalized");
  s->params[name] = std::vector<float>(host_data, host_data + numel);
  return DZ_OK;
}
int dz_emb_finalize(dz_emb* s) {
  if (!s) return fail(DZ_ERR_INVALID, "null handle");
  return s->finalized ? DZ_OK : emb_finalize(s);
}
int dz_emb_num_fbank_frames(int num_samples) { return num_samples < 400 ? 0 : 1 + (num_samples - 400) / 160; }

int dz_emb_forward(dz_emb* s, const float* wav_dev, const float* masks_dev, int B, int N, int S, int T, float* emb_dev, void* stream) {
  if (!s || !wav_dev || !masks_dev || !emb_dev) return fail(DZ_ERR_INVALID, "bad argument");
  if (!s->finalized) return fail(DZ_ERR_STATE, "dz_emb_finalize has not been called");
  if (B <= 0 || S <= 0 || S > 4 || T <= 0) return fail(DZ_ERR_INVALID, "bad shape (1 <= S <= 4)");
  cudaStream_t st = (cudaStream_t)stream;
  if (s->B != B || s->N != N || s->S != S || s->T != T) {
    cudaDeviceSynchronize();
    int r = emb_plan(s, B, N, S, T);
    if (r != DZ_OK) return r;
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) return fail(DZ_ERR_CUDA, std::string("plan failed: ") + cudaGetErrorString(e));
  }
  if (!s->done_event) cudaEventCreateWithFlags(&s->done_event, cudaEventDisableTiming);
  if (s->ran && s->last_stream != st) cudaStreamWaitEvent(st, s->done_event, 0);
  s->cur_wav = wav_dev; s->cur_masks = masks_dev; s->cur_out = emb_dev;
  {
    cudaError_t stale = cudaGetLastError();
    if (stale != cudaSuccess) return fail(DZ_ERR_CUDA, std::string("stale CUDA error before the embedding forward: ") + cudaGetErrorString(stale));
  }
  int n = 0;
  for (auto& step : s->steps) {
    cudaError_t e = step.fn(st);
    if (e != cudaSuccess) return fail(DZ_ERR_CUDA, "launch '" + step.name + "' failed: " + cudaGetErrorString(e) + " " + gemm_last_error());
    ++n;
  }
  s->last_launches = n;
  cudaEventRecord(s->done_event, st);
  s->last_stream = st; s->ran = true;
  return DZ_OK;
}
int dz_emb_last_launches(const dz_emb* s) { return s ? s->last_launches : 0; }
/* debug: copy the fbank features [B][80][F] (mel-major, before mean subtraction) of the last forward */
int64_t dz_emb_tap_fbank(dz_emb* s, float* dst_dev, int64_t capacity) {
  if (!s || !s->fb_dev) return fail(DZ_ERR_STATE, "no forward has run");
  const int64_t n = (int64_t)s->B * s->F * 80;
  if (!dst_dev) return n;
  if (capacity < n) return fail(DZ_ERR_INVALID, "destination too small");
  cudaError_t e = cudaMemcpy(dst_dev, s->fb_dev, n * 4, cudaMemcpyDeviceToDevice);
  return e == cudaSuccess ? n : fail(DZ_ERR_CUDA, cudaGetErrorString(e));
}
int dz_emb_num_steps(const dz_emb* s) { return s ? (int)s->steps.size() : 0; }
int dz_emb_profile(dz_emb* s, float* ms_out, double* flops_out, char* names, int name_stride, int cap, void* stream) {
  if (!s || !s->cur_wav) return fail(DZ_ERR_STATE, "no forward has run");
  cudaStream_t st = (cudaStream_t)stream;
  const int n = (int)s->steps.size();
  if (cap < n) return fail(DZ_ERR_INVALID, "output too small");
  std::vector<cudaEvent_t> ev(n + 1);
  for (auto& e : ev) cudaEventCreate(&e);
  cudaEventRecord(ev[0], st);
  for (int i = 0; i < n; ++i) { s->steps[i].fn(st); cudaEventRecord(ev[i + 1], st); }
  cudaError_t e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) return fail(DZ_ERR_CUDA, cudaGetErrorString(e));
  for (int i = 0; i < n; ++i) {
    cudaEventElapsedTime(&ms_out[i], ev[i], ev[i + 1]);
    if (flops_out) flops_out[i] = s->steps[i].flops;
    if (names) { strncpy(names + (size_t)i * name_stride, s->steps[i].name.c_str(), name_stride - 1); names[(size_t)i * name_stride + name_stride - 1] = 0; }
  }
  for (auto& e1 : ev) cudaEventDestroy(e1);
  return n;
}

}  // extern "C"

extern "C" int dz_conv3x3(const void* in_dev, void* out_dev, const void* res_dev, const void* w_dev, int ldw, const float* bias_dev, int B,
                          int H, int W, int C, int relu, int fp16, void* stream) {
  using namespace dz;
  if (!in_dev || !out_dev || !w_dev || B < 1 || H < 1 || W < 1) return fail(DZ_ERR_INVALID, "bad argument");
  Conv3Args c{};
  c.in = (const bf16*)in_dev; c.out = (bf16*)out_dev; c.res = (const bf16*)res_dev; c.w = (const bf16*)w_dev; c.ldw = ldw; c.bias = bias_dev;
  c.B = B; c.H = H; c.W = W; c.relu = relu; c.fp16 = fp16; c.C = C;
  cudaError_t e;
  if (C == 128) {
    ConvSPlan* p = conv3x3_stream_plan_create(c);
    if (!p) return fail(DZ_ERR_CUDA, std::string("conv3x3 plan: ") + gemm_last_error());
    e = conv3x3_stream_plan_launch(p, (cudaStream_t)stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize((cudaStream_t)stream);
    conv3x3_stream_plan_destroy(p);
  } else if (C == 32 || C == 64) {
    Conv3Plan* p = conv3x3_c32_plan_create(c);
    if (!p) return fail(DZ_ERR_CUDA, std::string("conv3x3 plan: ") + gemm_last_error());
    e = conv3x3_c32_plan_launch(p, (cudaStream_t)stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize((cudaStream_t)stream);
    conv3x3_c32_plan_destroy(p);
  } else {
    return fail(DZ_ERR_INVALID, "dz_conv3x3: C must be 32, 64 or 128");
  }
  if (e != cudaSuccess) return fail(DZ_ERR_CUDA, cudaGetErrorString(e));
  return DZ_OK;
}
