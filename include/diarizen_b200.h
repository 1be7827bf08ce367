/* diarizen_b200 C ABI  (libdiarizen_b200.so, sm_100a only)
 *
 * The reference (BUTSpeechFIT/DiariZen) has no FFI of its own: its hot path is Python calling PyTorch
 * (SURVEY.md 8b).  The seam this library sits behind is therefore the three device-side callables of
 * `DiariZenPipeline.__call__` (reference: diarizen/pipelines/inference.py:121-192):
 *
 *   dz_seg_*    replaces  self._segmentation.model(chunks.to(device))          pyannote-audio/pyannote/audio/core/inference.py:213-226
 *                          = Model.forward                                       diarizen/models/eend/model_wavlm_conformer.py:238-264
 *                          + Powerset.to_multilabel (hard)                       pyannote-audio/pyannote/audio/utils/powerset.py:103-128
 *   dz_emb_*    replaces  self._embedding(waveform_batch, masks=mask_batch)    pyannote-audio/pyannote/audio/pipelines/speaker_verification.py:693-705
 *                          = WeSpeakerResNet34.forward                           pyannote-audio/pyannote/audio/models/embedding/wespeaker/__init__.py:190-204
 *   dz_post_* / dz_cluster_*  replace the numpy/scipy stages                     pyannote-audio/pyannote/audio/pipelines/{clustering,speaker_diarization}.py,
 *                                                                                pipelines/utils/diarization.py, core/inference.py:543-666
 *
 * Conventions: plain C, no torch types.  Every pointer named *_dev is a device pointer on the current
 * CUDA device; `stream` is a cudaStream_t passed as void* (NULL = default stream).  Functions return 0 on
 * success and a negative code on failure; dz_last_error() returns a thread-local message.  Nothing in
 * here falls back to the CPU: on a machine without an sm_100 GPU the compute entry points fail.
 * Ownership: the caller owns every buffer it passes; handles own their weights and workspace.
 */
#ifndef DIARIZEN_B200_H_
#define DIARIZEN_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DZ_OK 0
#define DZ_ERR_INVALID (-1)
#define DZ_ERR_CUDA (-2)
#define DZ_ERR_STATE (-3)

const char* dz_last_error(void);
int dz_abi_version(void);

/* ------------------------------------------------------------------------------------------------
 * GEMM descriptor: C = epilogue(A * B^T) over bf16 hi/lo planes (see csrc/gemm.h for the A addressing
 * model that turns conv1d / grouped conv into GEMMs without an im2col copy).
 * ---------------------------------------------------------------------------------------------- */
typedef struct dz_gemm_desc {
  int32_t M, N, K, npass, batches, groups;
  const void* a; /* bf16 */
  int64_t a_plane, a_bstride, a_gstride, a_rstride;
  int32_t a_kinner, fp16; /* fp16: 0 = operands are bfloat16 bits, 1 = IEEE half bits */
  int64_t a_kouter, a_rows_alloc;
  const void* b; /* bf16 [groups][N][ldb] */
  int64_t b_plane, b_gstride;
  int32_t ldb, act;
  const float* bias;
  float alpha;
  int32_t group_cols, out_row_off, ldr;
  const float* residual;
  int64_t res_bstride;
  float* out_f32;
  int64_t of_bstride;
  int32_t ldo, ldob;
  void* out_bf; /* bf16 */
  int64_t ob_plane, ob_bstride;
  int32_t out_planes, zero_pad_to;
  void* out_t; /* bf16 */
  int64_t ot_plane, ot_bstride;
  int32_t ldt, tr_col0, seq_len, act_after_res; /* act_after_res: v = act(alpha*(acc+bias) + residual) */
  /* conv2d mode (conv_runs > 0): A is a zero-bordered NHWC image [b][h][wp][c]; one GEMM "batch" is one output row
   * (b, ho); K runs over conv_runs input rows, each contributing conv_run_len contiguous elements (kw * C). */
  int32_t conv_runs, conv_run_len, conv_x0, conv_h0, conv_hs, conv_Ho, conv_H, _pad2;
  int64_t a_hstride;
  /* residual read from 16-bit planes (same format as the operands) instead of fp32 */
  const void* res16;
  int64_t res16_plane, res16_bstride;
  int32_t ldr16, res16_row_off;
  /* optional row LayerNorm of the accumulator row (over the N valid columns, biased variance) applied before the activation:
   * v = (acc - mean) * rstd * ln_gamma[col] + ln_beta[col].  tcgen05 path only, N <= tile width (256), no bias / residual.
   * Both vectors must be 16-byte aligned and readable, zero padded, up to the next multiple of 32 columns. */
  const float* ln_gamma;
  const float* ln_beta;
  float ln_eps;
  int32_t _pad3;
} dz_gemm_desc;

/* impl: 0 = tcgen05 tensor-core kernel, 1 = CUDA-core checker kernel.  force_bn: 0 auto, or 64/128/256. */
int dz_gemm(const dz_gemm_desc* d, int impl, int force_bn, void* stream);
/* Plan once (tensor maps, launch geometry), launch many times (tcgen05 implementation). */
typedef struct dz_gemm_plan dz_gemm_plan;
dz_gemm_plan* dz_gemm_plan_create(const dz_gemm_desc* d, int force_bn);
int dz_gemm_plan_launch(const dz_gemm_plan* p, void* stream);
void dz_gemm_plan_destroy(dz_gemm_plan* p);

/* ------------------------------------------------------------------------------------------------
 * Element / row kernels of the segmentation path (unit-test surface; the engine calls the same code).
 * ---------------------------------------------------------------------------------------------- */
/* y = act(LayerNorm(x * prescale) * gamma + beta) over the last dim C of x[rows][ldx] (eps 1e-5).
 * Outputs (each optional): fp32 y_f32[rows][ldy]; bf16 planes y_bf[planes][rows][ldb] (pad columns
 * [C, ldb) zeroed).  mix (optional): mix[rows][ldx] = (mix_init ? 0 : mix) + mix_w * (mix_src==1 ? x : y).
 * 1 <= C <= 1024; ldx, ldy multiples of 4 and ldb, bf_plane multiples of 8 (each >= C); DZ_ERR_INVALID otherwise. */
int dz_layernorm(const float* x_dev, int64_t rows, int C, int ldx, const float* prescale_dev, const float* gamma_dev,
                 const float* beta_dev, int act, float* y_f32_dev, int ldy, void* y_bf_dev, int64_t bf_plane,
                 int ldb, int planes, float* mix_dev, float mix_w, int mix_src, int mix_init, int fp16, void* stream);

/* Attention over q|k row-major planes and v^T planes (layout: csrc/seg_kernels.h AttnArgs, same field order).
 *   scores = q.k (+ gate[b][h][q] * bias_tab[h][k - q + T - 1]); softmax over k; out = P v.   q is pre-scaled.
 * impl: 0 = tcgen05 kernel (hi planes only), 1 = CUDA-core kernel (hi + lo planes, fp32). */
typedef struct dz_attn_args {
  int32_t T, nheads;
  const void* q; const void* k; int64_t qk_plane; int32_t ldqk, q_col, k_col, fp16;
  const void* vt; int64_t vt_plane; int32_t ldvt, planes;
  const float* bias_tab; const float* gate;
  void* out; int64_t out_plane; int32_t ldo, out_planes;
  const void* v; int32_t v_col, _pad;   /* optional: V row-major [B*T][ldqk] at column v_col + head*64 (same plane stride as q/k);
                                           when set it replaces the transposed vt (no transposing producer needed) */
} dz_attn_args;
int dz_attention(const dz_attn_args* a, int B, int impl, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Segmentation engine
 * ---------------------------------------------------------------------------------------------- */
#define DZ_MAX_LAYERS 32
#define DZ_MAX_HEADS 16

typedef struct dz_seg_arch {
  int32_t large;            /* 1: layer-norm extractor, pre-norm encoder, waveform normalisation */
  int32_t conv_channels[7];
  int32_t embed_dim, total_heads, num_layers;
  int32_t num_heads[DZ_MAX_LAYERS];                 /* remaining heads per layer (0 = no attention) */
  int32_t head_index[DZ_MAX_LAYERS][DZ_MAX_HEADS];  /* which of the total heads remain */
  int32_t ffn[DZ_MAX_LAYERS];                       /* 0 = no feed-forward */
  int32_t head_dim_model, head_ffn, head_heads, head_layers, head_kernel, num_classes;
} dz_seg_arch;

typedef struct dz_seg dz_seg;

/* precision: 1 = bf16 operands, one tensor-core pass; 2 = fp16 operands (11-bit mantissa, saturating), one pass;
 * 3 = bf16x3 split (hi*hi + lo*hi + hi*lo, fp32-class).  Accumulation, residual stream, LayerNorm, softmax are fp32
 * in every mode.  gemm_impl: 0 tcgen05, 1 CUDA-core.  attn_impl: 0 tcgen05, 1 CUDA-core. */
dz_seg* dz_seg_create(const dz_seg_arch* arch, int precision, int gemm_impl, int attn_impl);
void dz_seg_destroy(dz_seg* s);
/* Parameters are passed by their reference state_dict name (fp32, host memory, C-contiguous). */
int dz_seg_set_param(dz_seg* s, const char* name, const float* host_data, int64_t numel);
/* Folds weight-norm / batch-norm / q-scaling, pads irregular widths, splits to bf16 planes, uploads. */
int dz_seg_finalize(dz_seg* s);
/* Number of output frames for windows of `num_samples` samples (reference: model_wavlm_conformer.py:98-124). */
int dz_seg_num_frames(const dz_seg* s, int num_samples);
/* wav_dev: [B][N] fp32.  logp_dev: [B][T][num_classes] fp32 log-probabilities (may be NULL).
 * multilabel_dev: [B][T][4] uint8 hard powerset decoding (may be NULL). */
int dz_seg_forward(dz_seg* s, const float* wav_dev, int B, int N, float* logp_dev, uint8_t* multilabel_dev, void* stream);
/* Same call with HOST buffers: pinned staging, H2D, forward, D2H inside (the end-to-end path). */
int dz_seg_forward_host(dz_seg* s, const float* wav_host, int B, int N, float* logp_host, uint8_t* multilabel_host);
/* Debug tap: copy a named intermediate of the last forward (fp32) into dst_dev; returns element count or <0. */
int64_t dz_seg_tap(dz_seg* s, const char* name, float* dst_dev, int64_t capacity);
/* Step-range execution for callers that interleave their own device work with the engine's layers (the multi-channel model,
 * diarizen/models/module/wav2vec2/components.py:1026-1070): plan a batch shape, look up a named intermediate of the plan
 * ("rep<l>" = the residual stream after layer l, "mix" = the layer-mix accumulator, "xbf" = its 16-bit operand copy) and run a
 * range of steps. */
int dz_seg_plan(dz_seg* s, int B, int N);
int dz_seg_tap_info(dz_seg* s, const char* name, void** ptr, int64_t* plane_elems, int64_t* rows, int* cols, int* ld, int* step, int* is16);
int dz_seg_run_steps(dz_seg* s, const float* wav_dev, int B, int N, int first, int last, float* logp_dev, uint8_t* multilabel_dev, void* stream);

/* Cross-channel fusion module of the multi-channel model (diarizen/models/module/utils_mc.py:13-64): x (B, C, T, D) fp32, rows
 * ordered (b, c, t), updated in place: x <- LayerNorm(Linear_O(attention over channels(Linear_QKV(x)))) + x.
 * Parameters by the reference's state-dict names: linearQ/K/V/O.{weight,bias}, ln_norm.{weight,bias}. */
typedef struct dz_fusion dz_fusion;
dz_fusion* dz_fusion_create(int D, int hidden, int heads, int precision);
void dz_fusion_destroy(dz_fusion* f);
int dz_fusion_set_param(dz_fusion* f, const char* name, const float* host, int64_t n);
int dz_fusion_finalize(dz_fusion* f);
int dz_fusion_forward(dz_fusion* f, float* x_dev, int B, int C, int T, int ldx, void* xbf_dev, int64_t xbf_plane, int ldb, float* mix_dev,
                      float mix_w, float* att_dev, void* stream);
int dz_rows_to_planes(const float* x_dev, int64_t rows, int C, int ldx, void* out_dev, int64_t plane_elems, int ldo, int planes, int fp16, void* stream);
/* out[(b, t)] = mean over channels of in[(b, c, t)], fp32 rows of width D with leading dimension ld */
int dz_channel_mean(const float* in_dev, float* out_dev, int B, int C, int T, int D, int ld, void* stream);
/* Kernel launches issued by the last dz_seg_forward call. */
int dz_seg_last_launches(const dz_seg* s);
/* Launch list of the current plan: name and algorithmic FLOPs (2*M*N*K for GEMMs, 4*T*T*64*h*B for attention,
 * 0 for bandwidth kernels) and algorithmic HBM bytes (bandwidth kernels) of step i. */
int dz_seg_num_steps(const dz_seg* s);
int dz_seg_step_info(const dz_seg* s, int i, char* name_buf, int name_cap, double* flops, double* bytes);
/* Runs one forward with a CUDA event pair around every launch; ms_out[i] = device time of step i.
 * Returns the number of steps (diagnostic path: events serialise nothing but add ~us per launch). */
int dz_seg_profile(dz_seg* s, const float* wav_dev, int B, int N, float* ms_out, int cap, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Speaker-embedding engine (WeSpeaker ResNet34)
 * ---------------------------------------------------------------------------------------------- */
typedef struct dz_emb dz_emb;
dz_emb* dz_emb_create(int precision, int gemm_impl);
void dz_emb_destroy(dz_emb* s);
/* state_dict names as in the pyannote checkpoint ("resnet.conv1.weight", ...).  Optional "fbank.mel_banks" [80][257]
 * and "fbank.window" [400] override the built-in Kaldi tables. */
int dz_emb_set_param(dz_emb* s, const char* name, const float* host_data, int64_t numel);
int dz_emb_finalize(dz_emb* s);
int dz_emb_num_fbank_frames(int num_samples);
/* wav_dev [B][N] fp32; masks_dev [B][S][T] fp32 (S <= 4 speaker masks per window, T segmentation frames);
 * emb_dev [B][S][256] fp32.  The trunk runs once per window and is pooled with each of the S masks. */
int dz_emb_forward(dz_emb* s, const float* wav_dev, const float* masks_dev, int B, int N, int S, int T, float* emb_dev,
                   void* stream);
int dz_emb_last_launches(const dz_emb* s);
int64_t dz_emb_tap_fbank(dz_emb* s, float* dst_dev, int64_t capacity);
int dz_emb_num_steps(const dz_emb* s);
int dz_emb_profile(dz_emb* s, float* ms_out, double* flops_out, char* names, int name_stride, int cap, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Post-processing and clustering kernels (all buffers on the device; seg is uint8 {0,1} [C][T][S])
 * ---------------------------------------------------------------------------------------------- */
/* scipy.ndimage.median_filter(size=(1,width,1), mode="reflect") on binary data (diarizen/pipelines/inference.py:131-132) */
int dz_median_filter(const uint8_t* in_dev, uint8_t* out_dev, int C, int T, int S, int width, void* stream);
/* count[f] = min(rint(mean over covering chunks of #active speakers), max_count); start[c] = first global frame of chunk c
 * (pipelines/utils/diarization.py:122-157 + core/inference.py:543-666) */
int dz_speaker_count(const uint8_t* seg_dev, const int32_t* start_dev, int C, int T, int S, int F, int max_count,
                     uint8_t* count_dev, void* stream);
/* masks[c][s][t] for the embedding pooling (speaker_diarization.py:271-320); stats[c][s] = (#active frames, #single-speaker frames) */
int dz_embedding_masks(const uint8_t* seg_dev, int C, int T, int S, int min_frames, float* masks_dev, int32_t* stats_dev,
                       void* stream);
/* cluster-wise max, overlap-add sum, per-frame top-count selection (speaker_diarization.py:377-425, diarization.py:193-239);
 * K clusters, Kout >= K output columns (zero-activation padding when a frame's count exceeds K);
 * discrete [F][Kout] uint8, act (optional) [F][Kout] fp32 */
int dz_reconstruct(const uint8_t* seg_dev, const int8_t* hard_dev, const int32_t* start_dev, const uint8_t* count_dev, int C,
                   int T, int S, int K, int Kout, int F, uint8_t* discrete_dev, float* act_dev, void* stream);
/* full symmetric Euclidean distance matrix [N][N] in float64, bit-compatible with scipy pdist on float64(x) */
int dz_pdist(const float* x_dev, int N, int D, double* out_dev, void* stream);
/* scipy linkage(method="centroid") from the distance matrix (destroyed); Z [N-1][4] float64 */
int64_t dz_linkage_workspace_bytes(int N);
int dz_linkage_centroid(double* dist_dev, int N, double* z_dev, void* workspace_dev, void* stream);
/* the same with the kernel chosen explicitly (tests): 0 default, 1 first-generation loop, 2 lazy loop with global-memory state */
int dz_linkage_centroid_variant(double* dist_dev, int N, double* z_dev, void* workspace_dev, void* stream, int variant);
/* Unit-test surface of the stride-1 3x3 convolution kernels of the embedding trunk (conv3x3_c32.cu: C = 32 / 64 with resident
 * weights; conv3x3_c128.cu: C = 128 with streamed weights).  in / out / res: zero-bordered NHWC 16-bit planes [B][H][W+2][C];
 * w: [C][ldw] with element (kh, kw, ci) at kh * rup(3C, 64) + kw * C + ci; out = relu(conv(in) + bias + res). */
int dz_conv3x3(const void* in_dev, void* out_dev, const void* res_dev, const void* w_dev, int ldw, const float* bias_dev, int B, int H,
               int W, int C, int relu, int fp16, void* stream);
/* Flat clusters from the dendrogram of dz_linkage_centroid, selected as AgglomerativeClustering.cluster selects them
 * (pyannote-audio/pyannote/audio/pipelines/clustering.py:418-492): cut at `threshold` (scipy fcluster, criterion "distance");
 * when the number of clusters with >= min_cluster_size members falls outside [min_clusters, max_clusters] (or differs from
 * num_clusters > 0) the cut moves to the merge iteration the reference's search stops at.  labels [N] int32 are
 * scipy's fcluster numbers - 1 (before the small-cluster re-assignment); info [8] int32 = {large clusters, selected
 * iteration or -1, "found only" flag, flat clusters, large clusters at the threshold, target, 0, 0}.
 * force_iteration >= 0 cuts after that merge unconditionally (test hook), -1 otherwise. */
int64_t dz_dendrogram_cut_workspace_bytes(int N);
int dz_dendrogram_cut(const double* z_dev, int N, double threshold, int min_cluster_size, int min_clusters, int max_clusters,
                      int num_clusters, int force_iteration, int32_t* labels_dev, int32_t* info_dev, void* workspace_dev, void* stream);
/* per-chunk constrained assignment maximising the summed soft score (clustering.py:159-173); hard [C][S] int8, -2 = none */
int dz_assign(const double* soft_dev, int C, int S, int K, int8_t* hard_dev, void* stream);

/* VBx: the two halves of one VB-GMM iteration over PLDA-space x-vectors, float64 (diarizen/clustering/VBx.py:86-111).
 * rho = X * sqrt(Phi) [N][D]; G[t] = -0.5 * (|x_t|^2 + D log 2 pi); gamma [N][S]. */
int dz_vbx_model(const double* gamma_dev, const double* rho_dev, const double* phi_dev, int N, int D, int S, double fa_over_fb,
                 double* alpha_dev, double* invl_dev, void* stream);
int dz_vbx_resp(const double* rho_dev, const double* g_dev, const double* alpha_dev, const double* invl_dev, const double* phi_dev,
                const double* pi_dev, int N, int D, int S, double Fa, double* gamma_dev, double* pi_acc_dev, double* logpx_acc_dev,
                void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DIARIZEN_B200_H_ */
