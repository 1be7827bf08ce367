// Segmentation engine: owns the (folded, padded, bf16-plane) weights and the activation workspace of the
// WavLM + Conformer segmentation network and replays the whole forward as a fixed list of kernel launches
// on one CUDA stream.  Replaces `Model.forward` (reference: diarizen/models/eend/model_wavlm_conformer.py:238-264)
// including `Wav2Vec2Model.extract_features` (wav2vec2/model.py:68-119) and the hard powerset decoding that
// `Inference.infer` applies right after it (pyannote-audio/pyannote/audio/core/inference.py:225-226).
//
// HBM layout (per batch of B windows, T frames, D = embed dim; "planes" = bf16 hi [+ lo]):
//   conv activations  planes [B][T_l][Cpad_l]        channels-last so that conv1d(k, s=2) is a strided GEMM view
//   residual stream   fp32   [B*T][Dp]               (x), layer-mix accumulator fp32 [B*T][Dp]
//   GEMM operands     planes [B*T][ld]               written by LayerNorm / GEMM epilogues
//   q|k               planes [B*T][2*h*64], v^T planes [B][h*64][Tp]   (P*V wants keys contiguous)
//   pos-conv staging  planes [B][T+128][16*64]       64 zero rows either side, groups padded to 64 channels
#include <cmath>
#include <functional>
#include <map>
#include <string>
#include <vector>

#include "../../include/diarizen_b200.h"
#include "common.cuh"
#include "gemm.h"
#include "seg_kernels.h"
#include "engine_common.h"

namespace dz {

std::string& tls_error();
int fail(int code, const std::string& msg);

static const int CONV_K[7] = {10, 3, 3, 3, 3, 2, 2};
static const int CONV_S[7] = {5, 2, 2, 2, 2, 2, 2};

int relpos_bucket(int d);  // below

struct Tap { int step; const float* f32; const bf16* bf; long long bf_plane; long long rows; int C; int ld; };

}  // namespace dz

using namespace dz;

struct dz_seg {
  dz_seg_arch arch;
  int precision = 1, planes = 1, npass = 1, fp16 = 0, gemm_impl = 0, attn_impl = 0;
  std::map<std::string, std::vector<float>> params;
  bool finalized = false;

  // weights
  DevMem conv0_w, conv0_gamma, conv0_beta;
  Weight convw[7];                         // [1..6]
  DevMem conv_gamma[7], conv_beta[7];      // large
  DevMem dummy_w, fp_gamma, fp_beta;
  Weight fp_w, pc_w;
  DevMem tr_gamma, tr_beta;
  struct Layer {
    Weight qkv, o, f1, f2;
    DevMem ln1_g, ln1_b, ln2_g, ln2_b, wab, gconst, head_index;
    float ba = 0, bb = 0;
  } layers[DZ_MAX_LAYERS];
  std::vector<float> rel_embed;  // [320][H]
  std::vector<float> mix_w;
  Weight proj_w;
  DevMem lnorm_g, lnorm_b;
  struct CBlock {
    Weight f1a, f1b, f2a, f2b, qkv, o, pw1, pw2;
    DevMem f1_g, f1_b, f2_g, f2_b, mha_g, mha_b, conv_g, conv_b, ln_g, ln_b, dw_w, dw_scale, dw_shift;
  } blocks[8];
  DevMem cls_w, cls_b;

  // plan
  int B = 0, N = 0, T = 0;
  std::vector<Step> steps;
  std::map<std::string, Tap> taps;
  std::vector<GemmPlan*> plans;
  std::vector<AttnPlan*> aplans;
  std::vector<PosConvPlan*> pcplans;
  std::vector<DevMem*> ws;  // workspace buffers
  DevMem bias_tab;
  const float* cur_wav = nullptr;
  float* cur_logp = nullptr;
  uint8_t* cur_ml = nullptr;
  int last_launches = 0;
  // host staging for the end-to-end path
  float* pin_wav = nullptr; float* pin_logp = nullptr; uint8_t* pin_ml = nullptr;
  size_t pin_wav_n = 0, pin_logp_n = 0, pin_ml_n = 0;
  DevMem dev_wav, dev_logp, dev_ml;
  cudaStream_t own_stream = nullptr;
  cudaEvent_t done_event = nullptr;   // recorded after every run: the workspace is shared across streams
  cudaStream_t last_stream = nullptr;
  bool ran = false;

  ~dz_seg() {
    clear_plan();
    if (pin_wav) cudaFreeHost(pin_wav);
    if (pin_logp) cudaFreeHost(pin_logp);
    if (pin_ml) cudaFreeHost(pin_ml);
    if (own_stream) cudaStreamDestroy(own_stream);
    if (done_event) cudaEventDestroy(done_event);
  }
  void clear_plan() {
    for (auto* p : plans) gemm_plan_destroy(p);
    plans.clear();
    for (auto* p : aplans) attention_tc_plan_destroy(p);
    aplans.clear();
    for (auto* p : pcplans) posconv_plan_destroy(p);
    pcplans.clear();
    for (auto* w : ws) delete w;
    ws.clear();
    steps.clear();
    taps.clear();
    B = N = T = 0;
  }
  const std::vector<float>* get(const std::string& k) const {
    auto it = params.find(k);
    return it == params.end() ? nullptr : &it->second;
  }
};

namespace dz {

// components.py:629-666 (bidirectional, 320 buckets, max distance 800) in the same float32 arithmetic.
int relpos_bucket(int d) {
  const int nb = 160, max_exact = 80;
  int out = d > 0 ? nb : 0;
  const int r = d < 0 ? -d : d;
  if (r < max_exact) return out + r;
  const float ratio = (float)r / (float)max_exact;
  const float lg = logf(ratio) / (float)std::log(800.0 / 80.0) * (float)(nb - max_exact);
  int large = max_exact + (int)lg;
  if (large > nb - 1) large = nb - 1;
  return out + large;
}

struct Builder {
  dz_seg* s;
  int err = 0;
  std::string msg;
  const std::vector<float>* need(const std::string& k, size_t n) {
    const std::vector<float>* v = s->get(k);
    if (!v) { if (!err) { err = DZ_ERR_STATE; msg = "missing parameter " + k; } return nullptr; }
    if (v->size() != n) {
      if (!err) { err = DZ_ERR_INVALID; msg = "parameter " + k + " has " + std::to_string(v->size()) + " elements, expected " + std::to_string(n); }
      return nullptr;
    }
    return v;
  }
  void ck(cudaError_t e, const char* what) {
    if (e != cudaSuccess && !err) { err = DZ_ERR_CUDA; msg = std::string(what) + ": " + cudaGetErrorString(e); }
  }
};

static int finalize_impl(dz_seg* s) {
  const dz_seg_arch& a = s->arch;
  g_weight_fp16() = s->fp16;
  Builder b{s};
  const std::string fe = "wavlm_model.feature_extractor.";
  const int D = a.embed_dim, H = a.total_heads;
  // ---- conv stack ----
  {
    const int C0 = a.conv_channels[0];
    auto w = b.need(fe + "conv_layers.0.conv.weight", (size_t)C0 * 10);
    auto g = b.need(fe + "conv_layers.0.layer_norm.weight", C0);
    auto be = b.need(fe + "conv_layers.0.layer_norm.bias", C0);
    if (b.err) return fail(b.err, b.msg);
    b.ck(upload_vec(s->conv0_w, *w), "conv0"); b.ck(upload_vec(s->conv0_gamma, *g), "conv0"); b.ck(upload_vec(s->conv0_beta, *be), "conv0");
  }
  for (int l = 1; l < 7; ++l) {
    const int Ci = a.conv_channels[l - 1], Co = a.conv_channels[l], k = CONV_K[l], Cip = rup(Ci, 8);
    auto w = b.need(fe + "conv_layers." + std::to_string(l) + ".conv.weight", (size_t)Co * Ci * k);
    if (b.err) return fail(b.err, b.msg);
    std::vector<float> r((size_t)Co * k * Cip, 0.f);  // [co][kk*Cip + ci] = w[co][ci][kk]
    for (int co = 0; co < Co; ++co)
      for (int ci = 0; ci < Ci; ++ci)
        for (int kk = 0; kk < k; ++kk) r[(size_t)co * k * Cip + (size_t)kk * Cip + ci] = (*w)[((size_t)co * Ci + ci) * k + kk];
    b.ck(make_weight(s->convw[l], r.data(), 1, Co, k * Cip, nullptr, 0), "conv weight");
    if (a.large) {
      auto g = b.need(fe + "conv_layers." + std::to_string(l) + ".layer_norm.weight", Co);
      auto be = b.need(fe + "conv_layers." + std::to_string(l) + ".layer_norm.bias", Co);
      if (b.err) return fail(b.err, b.msg);
      // zero padded to a multiple of 32 entries: the fused LayerNorm epilogue of the GEMM reads them with unpredicated vector loads
      std::vector<float> gp(rup((int)g->size(), 32), 0.f), bp(rup((int)be->size(), 32), 0.f);
      std::copy(g->begin(), g->end(), gp.begin()); std::copy(be->begin(), be->end(), bp.begin());
      b.ck(upload_vec(s->conv_gamma[l], gp), "conv ln"); b.ck(upload_vec(s->conv_beta[l], bp), "conv ln");
    }
  }
  const int C6 = a.conv_channels[6];
  const std::string en = "wavlm_model.encoder.", tr = en + "transformer.";
  {
    auto dw = b.need(fe + "dummy_weight", C6);
    auto g = b.need(en + "feature_projection.layer_norm.weight", C6);
    auto be = b.need(en + "feature_projection.layer_norm.bias", C6);
    auto w = b.need(en + "feature_projection.projection.weight", (size_t)D * C6);
    auto bi = b.need(en + "feature_projection.projection.bias", D);
    if (b.err) return fail(b.err, b.msg);
    b.ck(upload_vec(s->dummy_w, *dw), "fp"); b.ck(upload_vec(s->fp_gamma, *g), "fp"); b.ck(upload_vec(s->fp_beta, *be), "fp");
    b.ck(make_weight(s->fp_w, w->data(), 1, D, C6, bi->data(), D), "fp weight");
  }
  // ---- pos conv: weight-norm folded (w = g * v / ||v||_(0,1) per tap), groups padded to 64 input channels ----
  {
    const int G = 16, Dg = D / G, KT = 128;
    auto v = b.need(tr + "pos_conv_embed.conv.parametrizations.weight.original1", (size_t)D * Dg * KT);
    auto g = b.need(tr + "pos_conv_embed.conv.parametrizations.weight.original0", KT);
    auto bi = b.need(tr + "pos_conv_embed.conv.bias", D);
    auto lg = b.need(tr + "layer_norm.weight", D);
    auto lb = b.need(tr + "layer_norm.bias", D);
    if (b.err) return fail(b.err, b.msg);
    if (Dg > 64) return fail(DZ_ERR_INVALID, "pos-conv group width > 64 unsupported");
    std::vector<double> nrm(KT, 0.0);
    for (size_t i = 0; i < (size_t)D * Dg; ++i)
      for (int k = 0; k < KT; ++k) { const double x = (*v)[i * KT + k]; nrm[k] += x * x; }
    std::vector<float> scale(KT);
    for (int k = 0; k < KT; ++k) scale[k] = (float)((double)(*g)[k] / std::sqrt(nrm[k]));
    std::vector<float> r((size_t)G * Dg * KT * 64, 0.f);  // [g][n][tap*64 + ci]
    for (int gi = 0; gi < G; ++gi)
      for (int n = 0; n < Dg; ++n)
        for (int ci = 0; ci < Dg; ++ci)
          for (int k = 0; k < KT; ++k)
            r[((size_t)gi * Dg + n) * (KT * 64) + (size_t)k * 64 + ci] = (*v)[(((size_t)gi * Dg + n) * Dg + ci) * KT + k] * scale[k];
    b.ck(make_weight(s->pc_w, r.data(), G, Dg, KT * 64, bi->data(), D), "pos-conv weight");
    b.ck(upload_vec(s->tr_gamma, *lg), "tr ln"); b.ck(upload_vec(s->tr_beta, *lb), "tr ln");
  }
  // ---- encoder layers ----
  for (int l = 0; l < a.num_layers; ++l) {
    auto& L = s->layers[l];
    const std::string P = tr + "layers." + std::to_string(l) + ".";
    const int h = a.num_heads[l];
    if (h > 0) {
      const std::string A = P + "attention.";
      auto wq = b.need(A + "q_proj.weight", (size_t)h * 64 * D); auto bq = b.need(A + "q_proj.bias", h * 64);
      auto wk = b.need(A + "k_proj.weight", (size_t)h * 64 * D); auto bk = b.need(A + "k_proj.bias", h * 64);
      auto wv = b.need(A + "v_proj.weight", (size_t)h * 64 * D); auto bv = b.need(A + "v_proj.bias", h * 64);
      auto wo = b.need(A + "out_proj.weight", (size_t)D * h * 64); auto bo = b.need(A + "out_proj.bias", D);
      auto gw = b.need(A + "gru_rel_pos_linear.weight", 8 * 64); auto gb = b.need(A + "gru_rel_pos_linear.bias", 8);
      auto gc = b.need(A + "gru_rel_pos_const", H);
      if (b.err) return fail(b.err, b.msg);
      if (D / H != 64) return fail(DZ_ERR_INVALID, "head dim must be 64");
      std::vector<float> w((size_t)3 * h * 64 * D), bias(3 * h * 64);
      const float qs = 0.125f;  // head_dim^-0.5, exact power of two (components.py:403,456)
      for (size_t i = 0; i < (size_t)h * 64 * D; ++i) { w[i] = (*wq)[i] * qs; w[(size_t)h * 64 * D + i] = (*wk)[i]; w[(size_t)2 * h * 64 * D + i] = (*wv)[i]; }
      for (int i = 0; i < h * 64; ++i) { bias[i] = (*bq)[i] * qs; bias[h * 64 + i] = (*bk)[i]; bias[2 * h * 64 + i] = (*bv)[i]; }
      b.ck(make_weight(L.qkv, w.data(), 1, 3 * h * 64, D, bias.data(), 3 * h * 64), "qkv");
      b.ck(make_weight(L.o, wo->data(), 1, D, h * 64, bo->data(), D), "out_proj");
      std::vector<float> wab(128, 0.f);
      float ba = 0.f, bb = 0.f;
      for (int j = 0; j < 4; ++j) {
        for (int d = 0; d < 64; ++d) { wab[d] += (*gw)[j * 64 + d]; wab[64 + d] += (*gw)[(4 + j) * 64 + d]; }
        ba += (*gb)[j]; bb += (*gb)[4 + j];
      }
      L.ba = ba; L.bb = bb;
      b.ck(upload_vec(L.wab, wab), "gate"); b.ck(upload_vec(L.gconst, *gc), "gate");
      b.ck(L.head_index.alloc(sizeof(int) * DZ_MAX_HEADS, true), "gate");
      b.ck(cudaMemcpy(L.head_index.p, a.head_index[l], sizeof(int) * h, cudaMemcpyHostToDevice), "gate");
      if (l == 0) {
        auto re = b.need(A + "rel_attn_embed.weight", (size_t)320 * H);
        if (b.err) return fail(b.err, b.msg);
        s->rel_embed = *re;
      }
    }
    auto g1 = b.need(P + "layer_norm.weight", D); auto b1 = b.need(P + "layer_norm.bias", D);
    auto g2 = b.need(P + "final_layer_norm.weight", D); auto b2 = b.need(P + "final_layer_norm.bias", D);
    if (b.err) return fail(b.err, b.msg);
    b.ck(upload_vec(L.ln1_g, *g1), "ln"); b.ck(upload_vec(L.ln1_b, *b1), "ln");
    b.ck(upload_vec(L.ln2_g, *g2), "ln"); b.ck(upload_vec(L.ln2_b, *b2), "ln");
    const int F = a.ffn[l];
    if (F > 0) {
      auto w1 = b.need(P + "feed_forward.intermediate_dense.weight", (size_t)F * D); auto c1 = b.need(P + "feed_forward.intermediate_dense.bias", F);
      auto w2 = b.need(P + "feed_forward.output_dense.weight", (size_t)D * F); auto c2 = b.need(P + "feed_forward.output_dense.bias", D);
      if (b.err) return fail(b.err, b.msg);
      b.ck(make_weight(L.f1, w1->data(), 1, F, D, c1->data(), F), "ffn1");
      b.ck(make_weight(L.f2, w2->data(), 1, D, F, c2->data(), D), "ffn2");
    }
  }
  // ---- head ----
  const int A = a.head_dim_model, F = a.head_ffn, NL = a.num_layers + 1;
  {
    auto mw = b.need("weight_sum.weight", NL);
    auto pw = b.need("proj.weight", (size_t)A * D); auto pb = b.need("proj.bias", A);
    auto lg = b.need("lnorm.weight", A); auto lb = b.need("lnorm.bias", A);
    auto cw = b.need("classifier.weight", (size_t)a.num_classes * A); auto cb = b.need("classifier.bias", a.num_classes);
    if (b.err) return fail(b.err, b.msg);
    s->mix_w = *mw;
    b.ck(make_weight(s->proj_w, pw->data(), 1, A, D, pb->data(), A), "proj");
    b.ck(upload_vec(s->lnorm_g, *lg), "lnorm"); b.ck(upload_vec(s->lnorm_b, *lb), "lnorm");
    b.ck(upload_vec(s->cls_w, *cw), "cls"); b.ck(upload_vec(s->cls_b, *cb), "cls");
  }
  if (a.head_layers > 8) return fail(DZ_ERR_INVALID, "too many conformer blocks");
  const int hh = a.head_heads, dk = A / hh;
  if (dk != 64) return fail(DZ_ERR_INVALID, "conformer head dim must be 64");
  for (int i = 0; i < a.head_layers; ++i) {
    auto& C = s->blocks[i];
    const std::string P = "conformer.conformer_layer." + std::to_string(i) + ".";
    auto ln = [&](const std::string& n, DevMem& g, DevMem& be) {
      auto gg = b.need(P + n + ".weight", A); auto bb = b.need(P + n + ".bias", A);
      if (b.err) return;
      b.ck(upload_vec(g, *gg), "ln"); b.ck(upload_vec(be, *bb), "ln");
    };
    ln("ffn1.ln_norm", C.f1_g, C.f1_b); ln("ffn2.ln_norm", C.f2_g, C.f2_b); ln("mha.ln_norm", C.mha_g, C.mha_b);
    ln("conv.ln_norm", C.conv_g, C.conv_b); ln("ln_norm", C.ln_g, C.ln_b);
    auto lin = [&](const std::string& n, Weight& W, int No, int Ki) {
      auto w = b.need(P + n + ".weight", (size_t)No * Ki); auto bi = b.need(P + n + ".bias", No);
      if (b.err) return;
      b.ck(make_weight(W, w->data(), 1, No, Ki, bi->data(), No), n.c_str());
    };
    lin("ffn1.w_1", C.f1a, F, A); lin("ffn1.w_2", C.f1b, A, F); lin("ffn2.w_1", C.f2a, F, A); lin("ffn2.w_2", C.f2b, A, F);
    lin("mha.mha.linearO", C.o, A, A); lin("conv.pointwise_conv1", C.pw1, 2 * A, A); lin("conv.pointwise_conv2", C.pw2, A, A);
    auto wq = b.need(P + "mha.mha.linearQ.weight", (size_t)A * A); auto bq = b.need(P + "mha.mha.linearQ.bias", A);
    auto wk = b.need(P + "mha.mha.linearK.weight", (size_t)A * A); auto bk = b.need(P + "mha.mha.linearK.bias", A);
    auto wv = b.need(P + "mha.mha.linearV.weight", (size_t)A * A); auto bv = b.need(P + "mha.mha.linearV.bias", A);
    auto dw = b.need(P + "conv.depthwise_conv.weight", (size_t)A * a.head_kernel); auto db = b.need(P + "conv.depthwise_conv.bias", A);
    auto bg = b.need(P + "conv.bn_norm.weight", A); auto bb = b.need(P + "conv.bn_norm.bias", A);
    auto bm = b.need(P + "conv.bn_norm.running_mean", A); auto bv2 = b.need(P + "conv.bn_norm.running_var", A);
    if (b.err) return fail(b.err, b.msg);
    std::vector<float> w((size_t)3 * A * A), bias(3 * A);
    const float qs = 0.125f;  // 1/sqrt(d_k = 64) (conformer.py:59)
    for (size_t j = 0; j < (size_t)A * A; ++j) { w[j] = (*wq)[j] * qs; w[(size_t)A * A + j] = (*wk)[j]; w[(size_t)2 * A * A + j] = (*wv)[j]; }
    for (int j = 0; j < A; ++j) { bias[j] = (*bq)[j] * qs; bias[A + j] = (*bk)[j]; bias[2 * A + j] = (*bv)[j]; }
    b.ck(make_weight(C.qkv, w.data(), 1, 3 * A, A, bias.data(), 3 * A), "head qkv");
    std::vector<float> sc(A), sh(A);
    for (int j = 0; j < A; ++j) {
      const double inv = (double)(*bg)[j] / std::sqrt((double)(*bv2)[j] + 1e-5);
      sc[j] = (float)inv;
      sh[j] = (float)(((double)(*db)[j] - (double)(*bm)[j]) * inv + (double)(*bb)[j]);
    }
    b.ck(upload_vec(C.dw_w, *dw), "dw"); b.ck(upload_vec(C.dw_scale, sc), "dw"); b.ck(upload_vec(C.dw_shift, sh), "dw");
  }
  if (b.err) return fail(b.err, b.msg);
  s->finalized = true;
  s->params.clear();
  return DZ_OK;
}

// ------------------------------------------------------------------------------------------------
// plan: allocate workspace for (B, N) and record the launch list
// ------------------------------------------------------------------------------------------------
struct Planner {
  dz_seg* s;
  int err = 0;
  std::string msg;
  int P;       // planes
  int npass;
  DevMem* buf(size_t bytes, bool zero = false) {
    DevMem* m = new DevMem();
    s->ws.push_back(m);
    cudaError_t e = m->alloc(bytes, zero);
    if (e != cudaSuccess && !err) { err = DZ_ERR_CUDA; msg = std::string("workspace allocation failed: ") + cudaGetErrorString(e); }
    return m;
  }
  Planes planes(size_t elems_per_plane, bool zero = false) {
    DevMem* m = buf(elems_per_plane * 2 * P, zero);
    Planes p; p.p = m->as<bf16>(); p.plane = (long long)elems_per_plane;
    return p;
  }
  void step(const std::string& name, StepFn fn, double flops = 0.0, double bytes = 0.0) { s->steps.push_back({name, fn, flops, bytes}); }
  void tap_f32(const std::string& name, const float* p, long long rows, int C, int ld) {
    s->taps[name] = Tap{(int)s->steps.size(), p, nullptr, 0, rows, C, ld};
  }
  void tap_bf(const std::string& name, Planes p, long long rows, int C, int ld) {
    s->taps[name] = Tap{(int)s->steps.size(), nullptr, p.p, p.plane, rows, C, ld};
  }
  void gemm(const std::string& name, GemmDesc d) {
    d.npass = npass;
    d.out_planes = P;
    d.fp16 = s->fp16;
    const double flops = 2.0 * d.M * (double)d.N * d.K * d.batches * d.groups;  // algorithmic (one pass, valid dims)
    if (s->gemm_impl == 1) {
      step(name, [d](cudaStream_t st) { return gemm_simt_launch(d, st); }, flops);
      return;
    }
    GemmPlan* p = gemm_plan_create(d, 0);
    if (!p) { if (!err) { err = DZ_ERR_CUDA; msg = "gemm plan '" + name + "': " + gemm_last_error(); } return; }
    s->plans.push_back(p);
    step(name, [p](cudaStream_t st) { return gemm_plan_launch(p, st); }, flops);
  }
  // plain linear: A planes [rows][lda] x W -> epilogue
  GemmDesc linear(Planes A, int lda, long long rows, const Weight& W) {
    GemmDesc d = gemm_desc_default();
    d.M = (int)rows; d.N = W.N; d.K = W.K;
    d.a = A.p; d.a_plane = A.plane; d.a_rstride = lda; d.a_kinner = W.K; d.a_rows_alloc = rows;
    d.b = W.w.p; d.b_plane = W.plane; d.ldb = W.ldb; d.b_gstride = W.gstride;
    d.bias = W.bias.as<float>();
    return d;
  }
  void layernorm(const std::string& name, LnArgs a) {
    a.fp16 = s->fp16;
    // algorithmic HBM bytes: read the row once, write each requested output once (mix: read-modify-write)
    double per = 4.0;
    if (a.y_f32) per += 4.0;
    if (a.y_bf) per += 2.0 * a.planes;
    if (a.mix) per += a.mix_init ? 4.0 : 8.0;
    step(name, [a](cudaStream_t st) { return launch_layernorm(a, st); }, 0.0, per * (double)a.rows * a.C);
  }
};

static int plan_impl(dz_seg* s, int B, int N) {
  s->clear_plan();
  const dz_seg_arch& a = s->arch;
  Planner p{s};
  p.P = s->planes; p.npass = s->npass;
  const int FP = s->fp16;
  const int P = s->planes;
  int Tl[7], Cp[7];
  {
    int n = N;
    for (int l = 0; l < 7; ++l) {
      if (n < CONV_K[l]) return fail(DZ_ERR_INVALID, "window too short for the convolution stack");
      n = (n - CONV_K[l]) / CONV_S[l] + 1; Tl[l] = n; Cp[l] = rup(a.conv_channels[l], 8);
    }
  }
  const int T = Tl[6];
  const int D = a.embed_dim, Dp = rup(D, 8), H = a.total_heads;
  const long long R = (long long)B * T;  // rows of the encoder
  const bool large = a.large != 0;

  // ---------------- front end ----------------
  size_t act_elems = 0, f32_elems = 0;
  for (int l = 0; l < 6; ++l) act_elems = std::max(act_elems, (size_t)B * Tl[l] * Cp[l]);
  for (int l = 1; l < 7; ++l) f32_elems = std::max(f32_elems, (size_t)B * Tl[l] * Cp[l]);
  Planes act[2] = {p.planes(act_elems + 64, true), p.planes(act_elems + 64, true)};
  float* convf = p.buf((f32_elems + 64) * 4, true)->as<float>();
  float* wstats = p.buf((size_t)B * 2 * 4)->as<float>();
  double* mom = p.buf((size_t)B * 65 * 8)->as<double>();
  float* coef = p.buf((size_t)B * a.conv_channels[0] * 2 * 4)->as<float>();
  {
    Conv0Args c{};
    c.N = N; c.T0 = Tl[0]; c.C0 = a.conv_channels[0]; c.C0p64 = rup(c.C0, 64);
    if (c.C0p64 > 512) return fail(DZ_ERR_INVALID, "conv0 wider than 512 channels unsupported");
    c.w = s->conv0_w.as<float>(); c.wstats = wstats; c.coef = coef;
    c.gamma = s->conv0_gamma.as<float>(); c.beta = s->conv0_beta.as<float>();
    c.out = act[0].p; c.out_plane = act[0].plane; c.out_bstride = (long long)Tl[0] * Cp[0]; c.ldo = Cp[0]; c.planes = P; c.fp16 = FP;
    const float* g0 = s->conv0_gamma.as<float>(); const float* b0 = s->conv0_beta.as<float>(); const float* w0 = s->conv0_w.as<float>();
    const int C0 = c.C0, T0 = Tl[0];
    if (large) {
      void* wscratch = p.buf(wave_stats_scratch_bytes(B), true)->as<char>();
      p.step("wave_stats", [s, B, N, wstats, wscratch](cudaStream_t st) { return launch_wave_stats(s->cur_wav, B, N, wstats, wscratch, st); });
    } else {
      p.step("conv0_moments", [s, B, N, T0, mom](cudaStream_t st) { return launch_conv0_moments(s->cur_wav, B, N, T0, mom, st); });
      p.step("conv0_gn_coef", [=](cudaStream_t st) { return launch_conv0_gn_coef(mom, w0, g0, b0, B, C0, T0, coef, st); });
    }
    // conv0_tc.cu (tcgen05) runs whenever the tensor-core GEMMs do and it takes the shape (it matches the oracle on the s80
    // configurations at the benchmarked sizes, tests/test_bench_config_gpu.py); otherwise the CUDA-core kernel runs
    const bool c0_tc = s->gemm_impl == 0 && conv0_tc_eligible(c);
    p.step("conv0", [s, c, B, large, c0_tc](cudaStream_t st) {
             Conv0Args cc = c; cc.wav = s->cur_wav;
             return c0_tc ? launch_conv0_tc(cc, B, large, st) : launch_conv0(cc, B, large, st);
           },
           0.0, (double)B * N * 4.0 + (double)B * Tl[0] * Cp[0] * 2.0 * P);
    p.tap_bf("conv0", act[0], (long long)B * Tl[0], a.conv_channels[0], Cp[0]);
  }
  float* feats = convf;  // [B*T][Cp[6]] fp32 after the last conv
  for (int l = 1; l < 7; ++l) {
    const Planes in = act[(l - 1) & 1], out = act[l & 1];
    const Weight& W = s->convw[l];
    GemmDesc d = gemm_desc_default();
    d.M = Tl[l]; d.N = W.N; d.K = W.K; d.batches = B;
    d.a = in.p; d.a_plane = in.plane; d.a_rstride = (long long)CONV_S[l] * Cp[l - 1]; d.a_kinner = W.K;
    d.a_bstride = (long long)Tl[l - 1] * Cp[l - 1]; d.a_rows_alloc = Tl[l];
    d.b = W.w.p; d.b_plane = W.plane; d.ldb = W.ldb; d.b_gstride = W.gstride;
    const bool last = (l == 6);
    if (large && !last && s->gemm_impl == 0 && W.N <= 256) {
      // conv -> LayerNorm(channels) -> GELU in one launch: the accumulator tile holds whole rows (N <= 256), so the
      // normalisation happens on the TMEM row before the 16-bit planes are stored (no fp32 round trip through HBM)
      d.ln_gamma = s->conv_gamma[l].as<float>(); d.ln_beta = s->conv_beta[l].as<float>(); d.ln_eps = 1e-5f; d.act = 1;
      d.out_bf = out.p; d.ob_plane = out.plane; d.ldob = Cp[l]; d.ob_bstride = (long long)Tl[l] * Cp[l]; d.zero_pad_to = Cp[l];
      d.out_planes = P;
      p.gemm("conv" + std::to_string(l), d);
    } else if (large) {
      d.out_f32 = convf; d.ldo = Cp[l]; d.of_bstride = (long long)Tl[l] * Cp[l];
      p.gemm("conv" + std::to_string(l), d);
      LnArgs ln{};
      ln.x = convf; ln.rows = (long long)B * Tl[l]; ln.C = a.conv_channels[l]; ln.ldx = Cp[l];
      ln.gamma = s->conv_gamma[l].as<float>(); ln.beta = s->conv_beta[l].as<float>(); ln.act = 1;
      if (last) { ln.y_f32 = convf; ln.ldy = Cp[l]; }
      else { ln.y_bf = out.p; ln.bf_plane = out.plane; ln.ldb = Cp[l]; ln.planes = P; }
      p.layernorm("conv" + std::to_string(l) + "_ln", ln);
    } else {
      d.act = 1;
      if (last) { d.out_f32 = convf; d.ldo = Cp[l]; d.of_bstride = (long long)Tl[l] * Cp[l]; }
      else { d.out_bf = out.p; d.ob_plane = out.plane; d.ldob = Cp[l]; d.ob_bstride = (long long)Tl[l] * Cp[l]; d.zero_pad_to = Cp[l]; }
      p.gemm("conv" + std::to_string(l), d);
    }
    if (!last) p.tap_bf("conv" + std::to_string(l), out, (long long)B * Tl[l], a.conv_channels[l], Cp[l]);
  }
  p.tap_f32("feats_raw", feats, R, a.conv_channels[6], Cp[6]);

  // ---------------- encoder workspace ----------------
  int hmax = 1, Fmax = 8;
  for (int l = 0; l < a.num_layers; ++l) { hmax = std::max(hmax, a.num_heads[l]); Fmax = std::max(Fmax, a.ffn[l]); }
  const int A = a.head_dim_model, HF = a.head_ffn, hh = a.head_heads;
  hmax = std::max(hmax, hh);
  const int Fp = rup(std::max(std::max(Fmax, HF), 2 * A), 8);
  const int Tp = rup(T, 8);
  float* xres = p.buf((size_t)R * Dp * 4 + 256, true)->as<float>();
  float* mix = p.buf((size_t)R * Dp * 4 + 256, true)->as<float>();
  Planes xbf = p.planes((size_t)R * std::max(Dp, Cp[6]) + 64, true);
  Planes qk = p.planes((size_t)R * 3 * hmax * 64 + 64, true);   // q | k | v columns of every frame row
  Planes ctx = p.planes((size_t)R * hmax * 64 + 64, true);
  Planes mid = p.planes((size_t)R * Fp + 64, true);
  float* gate = p.buf((size_t)B * hmax * T * 4 + 64, true)->as<float>();
  const int PCW = 16 * 64, PCR = T + 128;
  Planes stage = p.planes((size_t)B * PCR * PCW + 64, true);

  // feature projection: LN(feats * dummy_weight) -> Linear
  {
    LnArgs ln{};
    ln.x = feats; ln.rows = R; ln.C = a.conv_channels[6]; ln.ldx = Cp[6];
    ln.prescale = s->dummy_w.as<float>(); ln.gamma = s->fp_gamma.as<float>(); ln.beta = s->fp_beta.as<float>();
    ln.y_bf = xbf.p; ln.bf_plane = xbf.plane; ln.ldb = Cp[6]; ln.planes = P;
    p.layernorm("fp_ln", ln);
    GemmDesc d = p.linear(xbf, Cp[6], R, s->fp_w);
    d.out_f32 = xres; d.ldo = Dp;
    p.gemm("fp_proj", d);
    p.tap_f32("proj", xres, R, D, Dp);
  }
  // positional conv (grouped, k = 128) as 16 batched GEMMs over a zero-padded staging copy
  {
    const int Dg = D / 16;
    p.step("pc_stage", [=](cudaStream_t st) {
      return launch_regroup(xres, R, D, Dp, T, PCR, 64, Dg, 64, stage.p, stage.plane, PCW, P, FP, st);
    });
    const Weight& W = s->pc_w;
    GemmDesc d = gemm_desc_default();
    d.M = T; d.N = Dg; d.K = 128 * 64; d.batches = B; d.groups = 16;
    d.a = stage.p; d.a_plane = stage.plane; d.a_rstride = PCW; d.a_kinner = 64; d.a_kouter = PCW; d.a_gstride = 64;
    d.a_bstride = (long long)PCR * PCW; d.a_rows_alloc = T;
    d.b = W.w.p; d.b_plane = W.plane; d.ldb = W.ldb; d.b_gstride = W.gstride;
    d.bias = W.bias.as<float>(); d.act = 1; d.group_cols = Dg;
    d.residual = xres; d.res_bstride = (long long)T * Dp; d.ldr = Dp;
    d.out_f32 = xres; d.of_bstride = (long long)T * Dp; d.ldo = Dp;
    if (s->npass == 1 && s->gemm_impl == 0 && Dg % 4 == 0) {
      PosConvArgs pa{};
      pa.stage = stage.p; pa.stage_rows = PCR; pa.stage_ld = PCW; pa.w = W.w.as<bf16>(); pa.ldw = W.ldb; pa.w_gstride = W.gstride;
      pa.bias = W.bias.as<float>(); pa.x = xres; pa.ldx = Dp; pa.B = B; pa.T = T; pa.Dg = Dg; pa.fp16 = FP;
      PosConvPlan* pp = posconv_plan_create(pa);
      if (!pp) { if (!p.err) { p.err = DZ_ERR_CUDA; p.msg = std::string("pos-conv plan: ") + gemm_last_error(); } }
      else {
        s->pcplans.push_back(pp);
        p.step("pos_conv", [pp](cudaStream_t st) { return posconv_plan_launch(pp, st); }, 2.0 * (double)R * D * 128 * Dg);
      }
    } else {
      p.gemm("pos_conv", d);
    }
  }
  const std::vector<float>& mw = s->mix_w;
  if (!large) {
    LnArgs ln{};
    ln.x = xres; ln.rows = R; ln.C = D; ln.ldx = Dp; ln.gamma = s->tr_gamma.as<float>(); ln.beta = s->tr_beta.as<float>();
    ln.y_f32 = xres; ln.ldy = Dp; ln.y_bf = xbf.p; ln.bf_plane = xbf.plane; ln.ldb = Dp; ln.planes = P;
    ln.mix = mix; ln.mix_w = mw[0]; ln.mix_src = 2; ln.mix_init = 1;
    p.layernorm("tr_ln", ln);
  }
  p.tap_f32("rep0", xres, R, D, Dp);
  p.tap_bf("xbf", xbf, R, D, Dp);   // 16-bit operand copy of the residual stream (post-norm models read it as the next layer's input)

  // relative-position bias table for this T: tab[hi][d + T - 1] = E[bucket(d)][head]   (layer 0 owns E)
  bool have_bias = a.num_heads[0] > 0;
  std::vector<float> tab_all;  // per layer offset
  std::vector<size_t> tab_off(a.num_layers, 0);
  if (have_bias) {
    for (int l = 0; l < a.num_layers; ++l) {
      tab_off[l] = tab_all.size();
      for (int hi = 0; hi < a.num_heads[l]; ++hi)
        for (int dd = -(T - 1); dd <= T - 1; ++dd) tab_all.push_back(s->rel_embed[(size_t)relpos_bucket(dd) * H + a.head_index[l][hi]]);
    }
    cudaError_t e = upload_vec(s->bias_tab, tab_all);
    if (e != cudaSuccess) return fail(DZ_ERR_CUDA, std::string("bias table: ") + cudaGetErrorString(e));
  }

  auto attention = [&](const std::string& nm, Planes xin, int ldx, const Weight& Wqkv, const Weight& Wo, int h,
                       const float* tab, const float* gatep, float* resid, int ldres) {
    GemmDesc d = p.linear(xin, ldx, R, Wqkv);
    // one plain GEMM: V stays row-major next to q and k (the attention kernel takes it as an MN-major operand), so the
    // projection needs no transposing epilogue
    d.out_bf = qk.p; d.ob_plane = qk.plane; d.ldob = 3 * h * 64;
    p.gemm(nm + "_qkv", d);
    AttnArgs at{};
    at.T = T; at.nheads = h; at.q = qk.p; at.k = qk.p; at.qk_plane = qk.plane; at.ldqk = 3 * h * 64; at.q_col = 0; at.k_col = h * 64;
    at.v = qk.p; at.v_col = 2 * h * 64; at.planes = P; at.bias_tab = tab; at.gate = gatep;
    at.out = ctx.p; at.out_plane = ctx.plane; at.ldo = h * 64; at.out_planes = P; at.fp16 = FP;
    // one-pass modes: attention_tc2_kernel; split-precision mode (hi + lo planes): attention_tc3_kernel (three tensor-core
    // passes per product); attn_impl = 1 keeps the CUDA-core checker kernel
    const int impl = s->attn_impl;
    const double aflops = 4.0 * (double)T * T * 64 * h * B;
    if (impl == 0) {
      AttnPlan* ap = attention_tc_plan_create(at, B);
      if (!ap) { if (!p.err) { p.err = DZ_ERR_CUDA; p.msg = "attention plan '" + nm + "': " + gemm_last_error(); } return; }
      s->aplans.push_back(ap);
      p.step(nm + "_attn", [ap](cudaStream_t st) { return attention_tc_plan_launch(ap, st); }, aflops);
    } else {
      p.step(nm + "_attn", [at, B](cudaStream_t st) { return launch_attention_simt(at, B, st); }, aflops);
    }
    p.tap_bf(nm + "_ctx", ctx, R, h * 64, h * 64);
    GemmDesc o = p.linear(ctx, h * 64, R, Wo);
    o.residual = resid; o.ldr = ldres; o.out_f32 = resid; o.ldo = ldres;
    p.gemm(nm + "_out", o);
  };

  for (int l = 0; l < a.num_layers; ++l) {
    auto& L = s->layers[l];
    const int h = a.num_heads[l], F = a.ffn[l];
    const std::string nm = "L" + std::to_string(l);
    bool mixed = !large;  // post-norm: state l was mixed when it was produced
    if (h > 0) {
      if (large) {
        LnArgs ln{};
        ln.x = xres; ln.rows = R; ln.C = D; ln.ldx = Dp; ln.gamma = L.ln1_g.as<float>(); ln.beta = L.ln1_b.as<float>();
        ln.y_bf = xbf.p; ln.bf_plane = xbf.plane; ln.ldb = Dp; ln.planes = P;
        ln.mix = mix; ln.mix_w = mw[l]; ln.mix_src = 1; ln.mix_init = (l == 0); mixed = true;
        p.layernorm(nm + "_ln1", ln);
      }
      const float* tab = nullptr; const float* gp = nullptr;
      if (have_bias) {
        GateArgs g{};
        g.x = xbf.p; g.x_plane = xbf.plane; g.planes = P; g.rows = R; g.ldx = Dp; g.seq_len = T;
        g.wab = L.wab.as<float>(); g.ba = L.ba; g.bb = L.bb; g.gconst = L.gconst.as<float>();
        g.head_index = L.head_index.as<int>(); g.nheads = h; g.gate = gate; g.fp16 = FP;
        p.step(nm + "_gate", [g](cudaStream_t st) { return launch_gate(g, st); });
        tab = s->bias_tab.as<float>() + tab_off[l]; gp = gate;
      }
      attention(nm, xbf, Dp, L.qkv, L.o, h, tab, gp, xres, Dp);
    }
    if (large) {
      if (F > 0) {
        LnArgs ln{};
        ln.x = xres; ln.rows = R; ln.C = D; ln.ldx = Dp; ln.gamma = L.ln2_g.as<float>(); ln.beta = L.ln2_b.as<float>();
        ln.y_bf = xbf.p; ln.bf_plane = xbf.plane; ln.ldb = Dp; ln.planes = P;
        if (!mixed) { ln.mix = mix; ln.mix_w = mw[l]; ln.mix_src = 1; ln.mix_init = (l == 0); mixed = true; }
        p.layernorm(nm + "_ln2", ln);
      }
      if (!mixed) {
        const float w = mw[l]; const int init = (l == 0); const long long n = R * Dp;
        p.step(nm + "_mix", [=](cudaStream_t st) { return launch_axpy_mix(xres, mix, w, init, n, st); });
      }
    } else {
      LnArgs ln{};
      ln.x = xres; ln.rows = R; ln.C = D; ln.ldx = Dp; ln.gamma = L.ln1_g.as<float>(); ln.beta = L.ln1_b.as<float>();
      ln.y_f32 = xres; ln.ldy = Dp; ln.y_bf = xbf.p; ln.bf_plane = xbf.plane; ln.ldb = Dp; ln.planes = P;
      p.layernorm(nm + "_ln1", ln);
    }
    if (F > 0) {
      GemmDesc d1 = p.linear(xbf, Dp, R, L.f1);
      d1.act = 1; d1.out_bf = mid.p; d1.ob_plane = mid.plane; d1.ldob = rup(F, 8); d1.zero_pad_to = rup(F, 8);
      p.gemm(nm + "_ffn1", d1);
      GemmDesc d2 = p.linear(mid, rup(F, 8), R, L.f2);
      d2.residual = xres; d2.ldr = Dp; d2.out_f32 = xres; d2.ldo = Dp;
      p.gemm(nm + "_ffn2", d2);
    }
    if (!large) {
      LnArgs ln{};
      ln.x = xres; ln.rows = R; ln.C = D; ln.ldx = Dp; ln.gamma = L.ln2_g.as<float>(); ln.beta = L.ln2_b.as<float>();
      ln.y_f32 = xres; ln.ldy = Dp; ln.y_bf = xbf.p; ln.bf_plane = xbf.plane; ln.ldb = Dp; ln.planes = P;
      ln.mix = mix; ln.mix_w = mw[l + 1]; ln.mix_src = 2; ln.mix_init = 0;
      p.layernorm(nm + "_ln2", ln);
    }
    p.tap_f32("rep" + std::to_string(l + 1), xres, R, D, Dp);
  }
  if (large) {
    const float w = mw[a.num_layers]; const long long n = R * Dp; const int init = (a.num_layers == 0);
    p.step("mix_last", [=](cudaStream_t st) { return launch_axpy_mix(xres, mix, w, init, n, st); });
  }
  p.tap_f32("mix", mix, R, D, Dp);

  // ---------------- conformer head ----------------
  float* hx = p.buf((size_t)R * A * 4 + 256, true)->as<float>();
  float* pw1o = p.buf((size_t)R * 2 * A * 4 + 256, true)->as<float>();
  p.step("mix_bf", [=](cudaStream_t st) { return launch_regroup(mix, R, D, Dp, 1, 1, 0, D, D, xbf.p, xbf.plane, Dp, P, FP, st); });
  {
    GemmDesc d = p.linear(xbf, Dp, R, s->proj_w);
    d.out_f32 = hx; d.ldo = A;
    p.gemm("head_proj", d);
    LnArgs ln{};
    ln.x = hx; ln.rows = R; ln.C = A; ln.ldx = A; ln.gamma = s->lnorm_g.as<float>(); ln.beta = s->lnorm_b.as<float>();
    ln.y_f32 = hx; ln.ldy = A;
    p.layernorm("head_ln", ln);
    p.tap_f32("head_in", hx, R, A, A);
  }
  for (int i = 0; i < a.head_layers; ++i) {
    auto& C = s->blocks[i];
    const std::string nm = "C" + std::to_string(i);
    auto ln_to_bf = [&](const std::string& n, DevMem& g, DevMem& be) {
      LnArgs ln{};
      ln.x = hx; ln.rows = R; ln.C = A; ln.ldx = A; ln.gamma = g.as<float>(); ln.beta = be.as<float>();
      ln.y_bf = xbf.p; ln.bf_plane = xbf.plane; ln.ldb = A; ln.planes = P;
      p.layernorm(n, ln);
    };
    auto ffn = [&](const std::string& n, DevMem& g, DevMem& be, const Weight& W1, const Weight& W2) {
      ln_to_bf(n + "_ln", g, be);
      GemmDesc d1 = p.linear(xbf, A, R, W1);
      d1.act = 2; d1.out_bf = mid.p; d1.ob_plane = mid.plane; d1.ldob = rup(HF, 8); d1.zero_pad_to = rup(HF, 8);
      p.gemm(n + "_w1", d1);
      GemmDesc d2 = p.linear(mid, rup(HF, 8), R, W2);
      d2.alpha = 0.5f; d2.residual = hx; d2.ldr = A; d2.out_f32 = hx; d2.ldo = A;
      p.gemm(n + "_w2", d2);
    };
    ffn(nm + "_ffn1", C.f1_g, C.f1_b, C.f1a, C.f1b);
    ln_to_bf(nm + "_mha_ln", C.mha_g, C.mha_b);
    attention(nm + "_mha", xbf, A, C.qkv, C.o, hh, nullptr, nullptr, hx, A);
    ln_to_bf(nm + "_conv_ln", C.conv_g, C.conv_b);
    {
      GemmDesc d = p.linear(xbf, A, R, C.pw1);
      d.out_f32 = pw1o; d.ldo = 2 * A;
      p.gemm(nm + "_pw1", d);
      DwArgs dw{};
      dw.x = pw1o; dw.ldx = 2 * A; dw.T = T; dw.A = A; dw.ksize = a.head_kernel;
      dw.w = C.dw_w.as<float>(); dw.scale = C.dw_scale.as<float>(); dw.shift = C.dw_shift.as<float>();
      dw.out = xbf.p; dw.out_plane = xbf.plane; dw.ldo = A; dw.planes = P; dw.fp16 = FP;
      p.step(nm + "_dwconv", [dw, B](cudaStream_t st) { return launch_glu_dwconv(dw, B, st); });
      GemmDesc d2 = p.linear(xbf, A, R, C.pw2);
      d2.residual = hx; d2.ldr = A; d2.out_f32 = hx; d2.ldo = A;
      p.gemm(nm + "_pw2", d2);
    }
    ffn(nm + "_ffn2", C.f2_g, C.f2_b, C.f2a, C.f2b);
    LnArgs ln{};
    ln.x = hx; ln.rows = R; ln.C = A; ln.ldx = A; ln.gamma = C.ln_g.as<float>(); ln.beta = C.ln_b.as<float>();
    ln.y_f32 = hx; ln.ldy = A;
    p.layernorm(nm + "_ln", ln);
    p.tap_f32(nm + "_out", hx, R, A, A);
  }
  {
    HeadArgs ha{};
    ha.x = hx; ha.rows = R; ha.ldx = A; ha.A = A; ha.NC = a.num_classes; ha.w = s->cls_w.as<float>(); ha.bias = s->cls_b.as<float>();
    p.step("classifier", [s, ha](cudaStream_t st) { HeadArgs h2 = ha; h2.logp = s->cur_logp; h2.multilabel = s->cur_ml; return launch_classifier_head(h2, st); });
  }
  if (p.err) { s->clear_plan(); return fail(p.err, p.msg); }
  s->B = B; s->N = N; s->T = T;
  return DZ_OK;
}

int seg_run(dz_seg* s, const float* wav, int B, int N, float* logp, uint8_t* ml, cudaStream_t st, int upto) {
  if (!s->finalized) return fail(DZ_ERR_STATE, "dz_seg_finalize has not been called");
  if (B <= 0 || N <= 0) return fail(DZ_ERR_INVALID, "bad batch shape");
  if (s->B != B || s->N != N) {
    cudaDeviceSynchronize();  // re-planning frees the workspace earlier launches may still be using
    int r = plan_impl(s, B, N);
    if (r != DZ_OK) return r;
    cudaError_t e = cudaDeviceSynchronize();  // workspace memsets (legacy stream) vs. non-blocking caller streams
    if (e != cudaSuccess) return fail(DZ_ERR_CUDA, std::string("plan failed: ") + cudaGetErrorString(e));
  }
  if (!s->done_event) cudaEventCreateWithFlags(&s->done_event, cudaEventDisableTiming);
  // one workspace per engine: a run on another stream must wait for the previous run to finish
  if (s->ran && s->last_stream != st) cudaStreamWaitEvent(st, s->done_event, 0);
  s->cur_wav = wav; s->cur_logp = logp; s->cur_ml = ml;
  int n = 0;
  for (size_t i = 0; i < s->steps.size(); ++i) {
    if (upto >= 0 && (int)i >= upto) break;
    cudaError_t e = s->steps[i].fn(st);
    if (e != cudaSuccess) return fail(DZ_ERR_CUDA, "launch '" + s->steps[i].name + "' failed: " + cudaGetErrorString(e));
    ++n;
  }
  s->last_launches = n;
  cudaEventRecord(s->done_event, st);
  s->last_stream = st; s->ran = true;
  return DZ_OK;
}

}  // namespace dz

extern "C" {

dz_seg* dz_seg_create(const dz_seg_arch* arch, int precision, int gemm_impl, int attn_impl) {
  if (!arch) { fail(DZ_ERR_INVALID, "null arch"); return nullptr; }
  if (precision != 1 && precision != 2 && precision != 3) { fail(DZ_ERR_INVALID, "precision must be 1 (bf16), 2 (fp16) or 3 (bf16x3)"); return nullptr; }
  if (arch->num_layers > DZ_MAX_LAYERS || arch->total_heads > DZ_MAX_HEADS) { fail(DZ_ERR_INVALID, "architecture exceeds compiled limits"); return nullptr; }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { fail(DZ_ERR_CUDA, "no CUDA device: diarizen_b200 has no CPU fallback"); return nullptr; }
  cudaDeviceProp prop;
  int dev = 0;
  cudaGetDevice(&dev);
  cudaGetDeviceProperties(&prop, dev);
  if (prop.major != 10) { fail(DZ_ERR_CUDA, "diarizen_b200 kernels are built for sm_100a only"); return nullptr; }
  dz_seg* s = new dz_seg();
  s->arch = *arch;
  s->precision = precision;
  s->planes = precision == 3 ? 2 : 1;
  s->npass = precision == 3 ? 3 : 1;
  s->fp16 = precision == 2 ? 1 : 0;
  s->gemm_impl = gemm_impl;
  s->attn_impl = attn_impl;
  return s;
}

void dz_seg_destroy(dz_seg* s) { delete s; }

int dz_seg_set_param(dz_seg* s, const char* name, const float* host_data, int64_t numel) {
  if (!s || !name || !host_data || numel < 0) return fail(DZ_ERR_INVALID, "bad argument");
  if (s->finalized) return fail(DZ_ERR_STATE, "engine already finalized");
  s->params[name] = std::vector<float>(host_data, host_data + numel);
  return DZ_OK;
}

int dz_seg_finalize(dz_seg* s) {
  if (!s) return fail(DZ_ERR_INVALID, "null handle");
  if (s->finalized) return DZ_OK;
  return finalize_impl(s);
}

int dz_seg_num_frames(const dz_seg* s, int num_samples) {
  (void)s;
  int n = num_samples;
  for (int l = 0; l < 7; ++l) {
    if (n < CONV_K[l]) return 0;
    n = (n - CONV_K[l]) / CONV_S[l] + 1;
  }
  return n;
}

/* ---- step-range execution: the hooks the multi-channel model (diarizen_b200/segmentation_mc.py) uses to interleave its channel
 * fusion modules with the layers of this engine (components.py:1026-1070) ---- */
int dz_seg_plan(dz_seg* s, int B, int N) {
  if (!s || !s->finalized) return fail(DZ_ERR_STATE, "dz_seg_finalize has not been called");
  if (s->B == B && s->N == N) return DZ_OK;
  cudaDeviceSynchronize();
  int r = plan_impl(s, B, N);
  if (r != DZ_OK) return r;
  cudaError_t e = cudaDeviceSynchronize();
  return e == cudaSuccess ? DZ_OK : fail(DZ_ERR_CUDA, std::string("plan failed: ") + cudaGetErrorString(e));
}
/* named intermediate of the current plan: device pointer (fp32 rows, or 16-bit planes when *is16 = 1), geometry, and the number of
 * steps after which it holds its value */
int dz_seg_tap_info(dz_seg* s, const char* name, void** ptr, int64_t* plane_elems, int64_t* rows, int* cols, int* ld, int* step, int* is16) {
  if (!s || !name) return fail(DZ_ERR_INVALID, "bad argument");
  auto it = s->taps.find(name);
  if (it == s->taps.end()) return fail(DZ_ERR_INVALID, std::string("unknown tap '") + name + "'");
  const Tap& t = it->second;
  if (ptr) *ptr = t.f32 ? (void*)t.f32 : (void*)t.bf;
  if (plane_elems) *plane_elems = t.bf_plane;
  if (rows) *rows = t.rows;
  if (cols) *cols = t.C;
  if (ld) *ld = t.ld;
  if (step) *step = t.step;
  if (is16) *is16 = t.f32 ? 0 : 1;
  return DZ_OK;
}
/* runs steps [first, last) of the plan for (B, N); wav / logp / multilabel as in dz_seg_forward (only read by the steps that use them) */
int dz_seg_run_steps(dz_seg* s, const float* wav_dev, int B, int N, int first, int last, float* logp_dev, uint8_t* multilabel_dev, void* stream) {
  if (!s) return fail(DZ_ERR_INVALID, "null handle");
  int r = dz_seg_plan(s, B, N);
  if (r != DZ_OK) return r;
  if (last < 0 || last > (int)s->steps.size()) last = (int)s->steps.size();
  if (first < 0 || first > last) return fail(DZ_ERR_INVALID, "bad step range");
  cudaStream_t st = (cudaStream_t)stream;
  if (!s->done_event) cudaEventCreateWithFlags(&s->done_event, cudaEventDisableTiming);
  if (s->ran && s->last_stream != st) cudaStreamWaitEvent(st, s->done_event, 0);
  s->cur_wav = wav_dev; s->cur_logp = logp_dev; s->cur_ml = multilabel_dev;
  for (int i = first; i < last; ++i) {
    cudaError_t e = s->steps[i].fn(st);
    if (e != cudaSuccess) return fail(DZ_ERR_CUDA, "launch '" + s->steps[i].name + "' failed: " + cudaGetErrorString(e));
  }
  s->last_launches = last - first;
  cudaEventRecord(s->done_event, st);
  s->last_stream = st; s->ran = true;
  return DZ_OK;
}

int dz_seg_forward(dz_seg* s, const float* wav_dev, int B, int N, float* logp_dev, uint8_t* multilabel_dev, void* stream) {
  if (!s || !wav_dev) return fail(DZ_ERR_INVALID, "bad argument");
  return seg_run(s, wav_dev, B, N, logp_dev, multilabel_dev, (cudaStream_t)stream, -1);
}

int dz_seg_forward_host(dz_seg* s, const float* wav_host, int B, int N, float* logp_host, uint8_t* multilabel_host) {
  if (!s || !wav_host) return fail(DZ_ERR_INVALID, "bad argument");
  if (!s->own_stream && cudaStreamCreateWithFlags(&s->own_stream, cudaStreamNonBlocking) != cudaSuccess)
    return fail(DZ_ERR_CUDA, "stream creation failed");
  const int T = dz_seg_num_frames(s, N);
  const size_t nw = (size_t)B * N, nl = (size_t)B * T * s->arch.num_classes, nm = (size_t)B * T * 4;
  cudaError_t e = cudaSuccess;
  if (s->pin_wav_n < nw) { if (s->pin_wav) cudaFreeHost(s->pin_wav); e = cudaMallocHost((void**)&s->pin_wav, nw * 4); s->pin_wav_n = nw; if (e == cudaSuccess) e = s->dev_wav.alloc(nw * 4, false); }
  if (e == cudaSuccess && s->pin_logp_n < nl) { if (s->pin_logp) cudaFreeHost(s->pin_logp); e = cudaMallocHost((void**)&s->pin_logp, nl * 4); s->pin_logp_n = nl; if (e == cudaSuccess) e = s->dev_logp.alloc(nl * 4, false); }
  if (e == cudaSuccess && s->pin_ml_n < nm) { if (s->pin_ml) cudaFreeHost(s->pin_ml); e = cudaMallocHost((void**)&s->pin_ml, nm); s->pin_ml_n = nm; if (e == cudaSuccess) e = s->dev_ml.alloc(nm, false); }
  if (e != cudaSuccess) return fail(DZ_ERR_CUDA, std::string("staging allocation failed: ") + cudaGetErrorString(e));
  // caller-pinned buffers are copied from/to directly; pageable ones go through the pinned staging area
  auto is_pinned = [](const void* ptr) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, ptr) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeHost;
  };
  const bool pin_in = is_pinned(wav_host);
  const bool pin_l = logp_host && is_pinned(logp_host), pin_m = multilabel_host && is_pinned(multilabel_host);
  if (!pin_in) memcpy(s->pin_wav, wav_host, nw * 4);
  cudaStream_t st = s->own_stream;
  e = cudaMemcpyAsync(s->dev_wav.p, pin_in ? wav_host : s->pin_wav, nw * 4, cudaMemcpyHostToDevice, st);
  if (e != cudaSuccess) return fail(DZ_ERR_CUDA, std::string("H2D failed: ") + cudaGetErrorString(e));
  int r = seg_run(s, s->dev_wav.as<float>(), B, N, logp_host ? s->dev_logp.as<float>() : nullptr,
                  multilabel_host ? s->dev_ml.as<uint8_t>() : nullptr, st, -1);
  if (r != DZ_OK) return r;
  if (logp_host) cudaMemcpyAsync(pin_l ? logp_host : s->pin_logp, s->dev_logp.p, nl * 4, cudaMemcpyDeviceToHost, st);
  if (multilabel_host) cudaMemcpyAsync(pin_m ? multilabel_host : s->pin_ml, s->dev_ml.p, nm, cudaMemcpyDeviceToHost, st);
  e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) return fail(DZ_ERR_CUDA, std::string("forward failed: ") + cudaGetErrorString(e));
  if (logp_host && !pin_l) memcpy(logp_host, s->pin_logp, nl * 4);
  if (multilabel_host && !pin_m) memcpy(multilabel_host, s->pin_ml, nm);
  return DZ_OK;
}

__global__ void tap_bf_to_f32_kernel(const __nv_bfloat16* p, long long plane, int planes, int fp16, long long rows, int C, int ld, float* dst) {
  const long long n = rows * C;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / C; const int c = (int)(i - r * C);
    float v = from16(p[r * ld + c], fp16);
    if (planes > 1) v += from16(p[plane + r * ld + c], fp16);
    dst[i] = v;
  }
}
__global__ void tap_f32_kernel(const float* p, long long rows, int C, int ld, float* dst) {
  const long long n = rows * C;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / C; const int c = (int)(i - r * C);
    dst[i] = p[r * ld + c];
  }
}

int64_t dz_seg_tap(dz_seg* s, const char* name, float* dst_dev, int64_t capacity) {
  if (!s || !name) return fail(DZ_ERR_INVALID, "bad argument");
  if (s->B == 0 || !s->cur_wav) return fail(DZ_ERR_STATE, "no forward has run");
  auto it = s->taps.find(name);
  if (it == s->taps.end()) return fail(DZ_ERR_INVALID, std::string("unknown tap ") + name);
  const Tap& t = it->second;
  const int64_t n = t.rows * t.C;
  if (!dst_dev) return n;
  if (capacity < n) return fail(DZ_ERR_INVALID, "tap destination too small");
  // replay the forward up to the step that produced the tapped tensor (later steps reuse the buffers)
  int r = seg_run(s, s->cur_wav, s->B, s->N, nullptr, nullptr, 0, t.step);
  if (r != DZ_OK) return r;
  if (t.f32) tap_f32_kernel<<<592, 256>>>(t.f32, t.rows, t.C, t.ld, dst_dev);
  else tap_bf_to_f32_kernel<<<592, 256>>>(t.bf, t.bf_plane, s->planes, s->fp16, t.rows, t.C, t.ld, dst_dev);
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) return fail(DZ_ERR_CUDA, std::string("tap failed: ") + cudaGetErrorString(e));
  return n;
}

int dz_seg_last_launches(const dz_seg* s) { return s ? s->last_launches : 0; }

int dz_seg_num_steps(const dz_seg* s) { return s ? (int)s->steps.size() : 0; }

int dz_seg_step_info(const dz_seg* s, int i, char* name_buf, int name_cap, double* flops, double* bytes) {
  if (s && bytes && i >= 0 && i < (int)s->steps.size()) *bytes = s->steps[i].bytes;
  if (!s || i < 0 || i >= (int)s->steps.size()) return fail(DZ_ERR_INVALID, "bad step index");
  if (name_buf && name_cap > 0) { strncpy(name_buf, s->steps[i].name.c_str(), name_cap - 1); name_buf[name_cap - 1] = 0; }
  if (flops) *flops = s->steps[i].flops;
  return DZ_OK;
}

int dz_seg_profile(dz_seg* s, const float* wav_dev, int B, int N, float* ms_out, int cap, void* stream) {
  if (!s || !wav_dev || !ms_out) return fail(DZ_ERR_INVALID, "bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  int r = seg_run(s, wav_dev, B, N, nullptr, nullptr, st, 0);  // plan only
  if (r != DZ_OK) return r;
  const int n = (int)s->steps.size();
  if (cap < n) return fail(DZ_ERR_INVALID, "ms_out too small");
  std::vector<cudaEvent_t> ev(n + 1);
  for (auto& e : ev) cudaEventCreate(&e);
  s->cur_wav = wav_dev; s->cur_logp = nullptr; s->cur_ml = nullptr;
  cudaEventRecord(ev[0], st);
  for (int i = 0; i < n; ++i) {
    cudaError_t e = s->steps[i].fn(st);
    if (e != cudaSuccess) return fail(DZ_ERR_CUDA, "launch '" + s->steps[i].name + "' failed: " + cudaGetErrorString(e));
    cudaEventRecord(ev[i + 1], st);
  }
  cudaError_t e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) return fail(DZ_ERR_CUDA, std::string("profile failed: ") + cudaGetErrorString(e));
  for (int i = 0; i < n; ++i) cudaEventElapsedTime(&ms_out[i], ev[i], ev[i + 1]);
  for (auto& ev1 : ev) cudaEventDestroy(ev1);
  return n;
}

}  // extern "C"
