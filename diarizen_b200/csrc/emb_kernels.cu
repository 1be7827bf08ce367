// CUDA-core kernels of the speaker-embedding path: Kaldi-compatible log-mel filterbank (framing, DC removal,
// pre-emphasis, Hamming window, 512-point FFT, mel bins, log), cepstral mean subtraction fused into the first
// 3x3 convolution (C_in = 1 stencil) and the masked statistics pooling (4 speaker masks per trunk output).
// reference: pyannote-audio/pyannote/audio/models/embedding/wespeaker/__init__.py:80-103 (compute_fbank),
//            wespeaker/resnet.py:358 (conv1 + bn1 + relu), resnet.py:49-66 + models/blocks/pooling.py:44-131 (TSTP).
#include "common.cuh"
#include "emb_kernels.h"

namespace dz {

// ------------------------------------------------------------------------------------------------
// K13 fbank: torchaudio.compliance.kaldi.fbank(num_mel_bins=80, frame 25 ms / 10 ms,
// dither 0, hamming, remove_dc_offset, preemphasis 0.97, round_to_power_of_two, use_power, use_log_fbank),
// applied to waveform * 2^15.  The 512-point FFT is organised around the register file:
//  * a warp transforms TWO frames at once (frame f -> real part, frame f + 1 -> imaginary part of one complex sequence;
//    the spectra are separated afterwards as A[k] = (Z[k] + conj Z[N-k]) / 2, B[k] = (Z[k] - conj Z[N-k]) / 2i);
//  * 512 = 8 x 8 x 8: every lane holds 16 complex points and runs two 8-point DFTs per step in registers; between the
//    steps the points cross lanes through shared memory ONCE (two exchanges, not nine butterfly stages), with strides
//    chosen so that every access is bank-conflict free (n = 64 n1 + 8 n2 + n3, k = k1 + 8 k2 + 64 k3:
//    X = sum_n3 W8^{n3 k3} W512^{n3 (k1 + 8 k2)} sum_n2 W8^{n2 k2} W64^{n2 k1} sum_n1 W8^{n1 k1} x);
//  * the per-lane twiddles of both steps are tabulated once per CTA; a CTA walks 64 frames.
// ------------------------------------------------------------------------------------------------
static constexpr int FB_WIN = 400, FB_HOP = 160, FB_NFFT = 512, FB_BINS = 257;
static constexpr int FB2_S = 72;        // exchange row stride (== 8 mod 32)
static constexpr int FB2_Z = 576;       // per-warp floats per component: 8 * 72 = 576 = 512 + 4 * 16 (padded spectrum)
static constexpr int FB2_FRAMES = 64;   // frames per CTA

// in-place 8-point DFT (forward, natural order in and out)
DZ_DEVINL void dft8(float (&r)[8], float (&i)[8]) {
  const float h = 0.70710678118654752440f;
  // stage 1: pairs (0,4) (2,6) (1,5) (3,7)
  const float b0r = r[0] + r[4], b0i = i[0] + i[4], b1r = r[0] - r[4], b1i = i[0] - i[4];
  const float b2r = r[2] + r[6], b2i = i[2] + i[6], b3r = r[2] - r[6], b3i = i[2] - i[6];
  const float b4r = r[1] + r[5], b4i = i[1] + i[5], b5r = r[1] - r[5], b5i = i[1] - i[5];
  const float b6r = r[3] + r[7], b6i = i[3] + i[7], b7r = r[3] - r[7], b7i = i[3] - i[7];
  // stage 2 (-i (x + i y) = y - i x)
  const float c0r = b0r + b2r, c0i = b0i + b2i, c2r = b0r - b2r, c2i = b0i - b2i;
  const float c1r = b1r + b3i, c1i = b1i - b3r, c3r = b1r - b3i, c3i = b1i + b3r;
  const float c4r = b4r + b6r, c4i = b4i + b6i, c6r = b4r - b6r, c6i = b4i - b6i;
  const float c5r = b5r + b7i, c5i = b5i - b7r, c7r = b5r - b7i, c7i = b5i + b7r;
  // stage 3: W8 = (1 - i) / sqrt 2, W8^2 = -i, W8^3 = (-1 - i) / sqrt 2
  const float t5r = h * (c5r + c5i), t5i = h * (c5i - c5r);
  const float t7r = h * (c7i - c7r), t7i = -h * (c7r + c7i);
  r[0] = c0r + c4r; i[0] = c0i + c4i; r[4] = c0r - c4r; i[4] = c0i - c4i;
  r[1] = c1r + t5r; i[1] = c1i + t5i; r[5] = c1r - t5r; i[5] = c1i - t5i;
  r[2] = c2r + c6i; i[2] = c2i - c6r; r[6] = c2r - c6i; i[6] = c2i + c6r;
  r[3] = c3r + t7r; i[3] = c3i + t7i; r[7] = c3r - t7r; i[7] = c3i - t7i;
}

__global__ void __launch_bounds__(256, 3) fbank2_kernel(FbankArgs a) {
  extern __shared__ float smf2[];
  float* win = smf2;                                        // [400] (416 reserved)
  float2* tw1 = reinterpret_cast<float2*>(smf2 + 416);      // [(h * 8 + k1) * 32 + lane]  W64^{n2 k1}
  float2* tw2 = tw1 + 512;                                  // [(h * 8 + k2) * 32 + lane]  W512^{n3 (k1 + 8 k2)}
  float* warp_base = reinterpret_cast<float*>(tw2 + 512);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < FB_WIN; i += blockDim.x) win[i] = a.window[i];
  for (int i = threadIdx.x; i < 512; i += blockDim.x) {
    const int l = i & 31, j = (i >> 5) & 7, h = i >> 8;
    const int pq = l + 32 * h;
    const int e1 = 8 * (pq >> 3) * j;                       // W64^{n2 k1} = W512^{8 n2 k1}, n2 = p >> 3, k1 = j
    const int e2 = (pq & 7) * ((pq >> 3) + 8 * j);          // n3 = q & 7, k1 = q >> 3, k2 = j
    float2 t1 = a.twiddle[e1 & 255], t2 = a.twiddle[e2 & 255];
    if (e1 & 256) { t1.x = -t1.x; t1.y = -t1.y; }
    if (e2 & 256) { t2.x = -t2.x; t2.y = -t2.y; }
    tw1[i] = t1; tw2[i] = t2;
  }
  __syncthreads();
  float* sre = warp_base + warp * (2 * FB2_Z);
  float* sim = sre + FB2_Z;
  const int b = blockIdx.y;
  const float* wav = a.wav + (long long)b * a.N;
  const int f_end = min(a.F, (int)(blockIdx.x + 1) * FB2_FRAMES);
  for (int f = blockIdx.x * FB2_FRAMES + 2 * warp; f < f_end; f += 16) {
    const bool two = f + 1 < a.F;
    // ---- the two frames: sample n = 32 s + lane in slot s (n < 400), DC removal, pre-emphasis, window
    float zr[16], zi[16];
#pragma unroll
    for (int fr = 0; fr < 2; ++fr) {
      const float* src = wav + (long long)(f + (fr && two ? 1 : 0)) * FB_HOP;
      float x[13];
      float sum = 0.f;
#pragma unroll
      for (int sl = 0; sl < 13; ++sl) {
        const int n = 32 * sl + lane;
        x[sl] = (n < FB_WIN) ? src[n] * 32768.0f : 0.f;
        sum += x[sl];
      }
      const float mean = warp_sum(sum) / FB_WIN;
#pragma unroll
      for (int sl = 0; sl < 16; ++sl) {
        float v = 0.f;
        if (sl < 13) {
          const int n = 32 * sl + lane;
          const float up = __shfl_up_sync(0xffffffffu, x[sl], 1);
          const float wrap = __shfl_sync(0xffffffffu, x[sl > 0 ? sl - 1 : 0], 31);
          const float prev = (lane > 0) ? up : (sl > 0 ? wrap : x[0]);
          if (n < FB_WIN) v = ((x[sl] - mean) - 0.97f * (prev - mean)) * win[n];
        }
        if (fr == 0) zr[sl] = v; else zi[sl] = (two ? v : 0.f);
      }
    }
    // ---- step 1: DFT over n1 (slots 2 n1 + h), twiddle W64^{n2 k1}, to shared memory at [k1][p = lane + 32 h]
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      float r8[8], i8[8];
#pragma unroll
      for (int n1 = 0; n1 < 8; ++n1) { r8[n1] = zr[2 * n1 + h]; i8[n1] = zi[2 * n1 + h]; }
      dft8(r8, i8);
#pragma unroll
      for (int k1 = 0; k1 < 8; ++k1) {
        const float2 w = tw1[(h * 8 + k1) * 32 + lane];
        sre[k1 * FB2_S + lane + 32 * h] = r8[k1] * w.x - i8[k1] * w.y;
        sim[k1 * FB2_S + lane + 32 * h] = r8[k1] * w.y + i8[k1] * w.x;
      }
    }
    __syncwarp();
    // ---- step 2: lane owns (k1, n3) = (q >> 3, q & 7), q = lane + 32 h: DFT over n2, twiddle W512^{n3 (k1 + 8 k2)}
    float r2[2][8], i2[2][8];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int q = lane + 32 * h, base = (q >> 3) * FB2_S + (q & 7);
#pragma unroll
      for (int n2 = 0; n2 < 8; ++n2) { r2[h][n2] = sre[base + n2 * 8]; i2[h][n2] = sim[base + n2 * 8]; }
    }
    __syncwarp();
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int q = lane + 32 * h, base = (q >> 3) * FB2_S + (q & 7) * 9;
      dft8(r2[h], i2[h]);
#pragma unroll
      for (int k2 = 0; k2 < 8; ++k2) {
        const float2 w = tw2[(h * 8 + k2) * 32 + lane];
        sre[base + k2] = r2[h][k2] * w.x - i2[h][k2] * w.y;
        sim[base + k2] = r2[h][k2] * w.y + i2[h][k2] * w.x;
      }
    }
    __syncwarp();
    // ---- step 3: lane owns (k1, k2) = (r >> 3, r & 7): DFT over n3 -> Z[k1 + 8 k2 + 64 k3]
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int q = lane + 32 * h, base = (q >> 3) * FB2_S + (q & 7);
#pragma unroll
      for (int n3 = 0; n3 < 8; ++n3) { r2[h][n3] = sre[base + n3 * 9]; i2[h][n3] = sim[base + n3 * 9]; }
    }
    __syncwarp();
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int q = lane + 32 * h;
      dft8(r2[h], i2[h]);
#pragma unroll
      for (int k3 = 0; k3 < 8; ++k3) {
        const int k = (q >> 3) + 8 * (q & 7) + 64 * k3;
        sre[k + 4 * (k >> 5)] = r2[h][k3];            // padded: conflict-free here and in the reads below
        sim[k + 4 * (k >> 5)] = i2[h][k3];
      }
    }
    __syncwarp();
    // ---- power spectra of the two frames (bins 0..256)
    float pa[9], pb[9];
#pragma unroll
    for (int j = 0; j < 9; ++j) {
      const int k = lane + 32 * j;
      pa[j] = 0.f; pb[j] = 0.f;
      if (k < FB_BINS) {
        const int kn = (FB_NFFT - k) & (FB_NFFT - 1);
        const float zkr = sre[k + 4 * (k >> 5)], zki = sim[k + 4 * (k >> 5)];
        const float znr = sre[kn + 4 * (kn >> 5)], zni = sim[kn + 4 * (kn >> 5)];
        const float ar = 0.5f * (zkr + znr), ai = 0.5f * (zki - zni);
        const float br = 0.5f * (zki + zni), bi = 0.5f * (znr - zkr);
        pa[j] = ar * ar + ai * ai;
        pb[j] = br * br + bi * bi;
      }
    }
    __syncwarp();
    float* PA = sre;                     // [257]
    float* PB = sim;
#pragma unroll
    for (int j = 0; j < 9; ++j) {
      const int k = lane + 32 * j;
      if (k < FB_BINS) { PA[k] = pa[j]; PB[k] = pb[j]; }
    }
    __syncwarp();
    // ---- mel bins + log, mel-major output [b][mel][frame]
    float* dst = a.out + (long long)b * 80 * a.F + f;
    for (int m = lane; m < 80; m += 32) {
      const int ks = a.mel_range[2 * m], ke = a.mel_range[2 * m + 1];
      const float* wrow = a.mel_w + m * FB_BINS;
      float acca = 0.f, accb = 0.f;
      for (int k = ks; k < ke; ++k) {
        const float w = __ldg(wrow + k);
        acca = fmaf(PA[k], w, acca);
        accb = fmaf(PB[k], w, accb);
      }
      dst[(long long)m * a.F] = logf(fmaxf(acca, 1.1920928955078125e-07f));
      if (two) dst[(long long)m * a.F + 1] = logf(fmaxf(accb, 1.1920928955078125e-07f));
    }
    __syncwarp();
  }
}

cudaError_t launch_fbank(const FbankArgs& a, int B, cudaStream_t st) {
  dim3 grid((a.F + FB2_FRAMES - 1) / FB2_FRAMES, B);
  const size_t smem = sizeof(float) * (416 + 2 * 512 * 2 + 8 * 2 * FB2_Z);
  fbank2_kernel<<<grid, 256, smem, st>>>(a);
  return cudaGetLastError();
}

// per (window, mel) mean over frames: one warp per contiguous row of the mel-major features.  Lane l sums frames l, l + 32, ...
// in order and the 32 partial sums are combined by the shuffle tree (fp32; the reference's torch.mean uses another order).
__global__ void __launch_bounds__(256) fbank_mean_kernel(const float* __restrict__ fb, int rows, int F, float* __restrict__ mean) {
  const int r = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (r >= rows) return;
  const float* p = fb + (long long)r * F;
  float s = 0.f;
  for (int f = lane; f < F; f += 32) s += p[f];
  s = warp_sum(s);
  if (lane == 0) mean[r] = s / F;
}
cudaError_t launch_fbank_mean(const float* fb, int B, int F, float* mean, cudaStream_t st) {
  fbank_mean_kernel<<<(B * 80 + 7) / 8, 256, 0, st>>>(fb, B * 80, F, mean);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// conv1 (1 -> 32, 3x3, pad 1) on the mean-subtracted fbank + folded BN + ReLU -> zero-bordered NHWC planes
// [b][h = mel][1 + w = frame][32].  One thread per output pixel, 32 channels.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) emb_conv1_kernel(Conv1Args a) {
  __shared__ float w[9 * 32], sc[32], sh[32];
  for (int i = threadIdx.x; i < 288; i += blockDim.x) {
    const int c = i / 9, t = i - c * 9;
    w[t * 32 + c] = a.w[i];   // [tap][c]
  }
  for (int i = threadIdx.x; i < 32; i += blockDim.x) { sc[i] = a.scale[i]; sh[i] = a.shift[i]; }
  __syncthreads();
  const long long total = (long long)a.B * 80 * a.F;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int wf = (int)(i % a.F);
    const long long r = i / a.F;
    const int h = (int)(r % 80), b = (int)(r / 80);
    float in[9];
#pragma unroll
    for (int kh = 0; kh < 3; ++kh)
#pragma unroll
      for (int kw = 0; kw < 3; ++kw) {
        const int hh = h + kh - 1, ww = wf + kw - 1;
        float v = 0.f;
        if (hh >= 0 && hh < 80 && ww >= 0 && ww < a.F) v = a.fb[((long long)b * 80 + hh) * a.F + ww] - a.mean[b * 80 + hh];
        in[kh * 3 + kw] = v;
      }
    bf16* o = a.out + (((long long)b * 80 + h) * (a.F + 2) + wf + 1) * 32;
#pragma unroll
    for (int c8 = 0; c8 < 4; ++c8) {
      uint32_t hw[4], lw[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        float v2[2];
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          const int c = c8 * 8 + e * 2 + q;
          float acc = 0.f;
#pragma unroll
          for (int t = 0; t < 9; ++t) acc = fmaf(in[t], w[t * 32 + c], acc);
          v2[q] = fmaxf(acc * sc[c] + sh[c], 0.f);
        }
        bf16 h0, l0, h1, l1;
        split_bf16(v2[0], h0, l0, a.fp16);
        split_bf16(v2[1], h1, l1, a.fp16);
        hw[e] = (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
        lw[e] = (uint32_t)__bfloat16_as_ushort(l0) | ((uint32_t)__bfloat16_as_ushort(l1) << 16);
      }
      *reinterpret_cast<uint4*>(o + c8 * 8) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
      if (a.planes > 1) *reinterpret_cast<uint4*>(o + a.out_plane + c8 * 8) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
    }
  }
}
// Row kernel, used whenever its three staged rows fit the default 48 KB of shared memory (F up to 4094 frames; the kernel
// above takes longer inputs).  One CTA per (window, mel) output row: the three
// mean-subtracted input rows are staged once in shared memory; a thread owns 8 of the 32 output channels, keeps their 72
// weights (and the folded BatchNorm) in registers for the whole row and walks the frames, so the inner loop is 9 shared-memory
// reads + 72 FMAs per (pixel, channel group) instead of one shared-memory weight read per FMA, there is no 64-bit division per
// pixel, and a warp's stores are 512 contiguous bytes (8 pixels x 4 channel groups x 16 B).  Same tap order per output.
__global__ void __launch_bounds__(256, 2) emb_conv1_rows_kernel(Conv1Args a) {
  extern __shared__ float c1rows[];   // [3][F + 2]: rows h - 1, h, h + 1 minus their means, zero border / zero outside the mel range
  const int F = a.F, W = F + 2;
  const int r = blockIdx.x, b = r / 80, h = r - b * 80;
  for (int i = threadIdx.x; i < 3 * W; i += blockDim.x) {
    const int kh = i / W, x = i - kh * W;
    const int hh = h + kh - 1, ww = x - 1;
    float v = 0.f;
    if (hh >= 0 && hh < 80 && ww >= 0 && ww < F) v = a.fb[((long long)b * 80 + hh) * F + ww] - a.mean[b * 80 + hh];
    c1rows[i] = v;
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, cg = lane & 3, pl = lane >> 2;
  float wr[9][8], sc[8], sh[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
#pragma unroll
    for (int t = 0; t < 9; ++t) wr[t][j] = a.w[(cg * 8 + j) * 9 + t];
    sc[j] = a.scale[cg * 8 + j];
    sh[j] = a.shift[cg * 8 + j];
  }
  __syncthreads();
  bf16* orow = a.out + ((long long)r * W + 1) * 32 + cg * 8;
  for (int wf = warp * 8 + pl; wf < F; wf += 64) {
    float in[9];
#pragma unroll
    for (int kh = 0; kh < 3; ++kh)
#pragma unroll
      for (int kw = 0; kw < 3; ++kw) in[kh * 3 + kw] = c1rows[kh * W + wf + kw];
    uint32_t hw[4], lw[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float v2[2];
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        const int j = e * 2 + q;
        float acc = 0.f;
#pragma unroll
        for (int t = 0; t < 9; ++t) acc = fmaf(in[t], wr[t][j], acc);
        v2[q] = fmaxf(acc * sc[j] + sh[j], 0.f);
      }
      bf16 h0, l0, h1, l1;
      split_bf16(v2[0], h0, l0, a.fp16);
      split_bf16(v2[1], h1, l1, a.fp16);
      hw[e] = (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
      lw[e] = (uint32_t)__bfloat16_as_ushort(l0) | ((uint32_t)__bfloat16_as_ushort(l1) << 16);
    }
    bf16* o = orow + (long long)wf * 32;
    *reinterpret_cast<uint4*>(o) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
    if (a.planes > 1) *reinterpret_cast<uint4*>(o + a.out_plane) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
  }
}
cudaError_t launch_emb_conv1(const Conv1Args& a, cudaStream_t st) {
  const size_t smem = sizeof(float) * 3 * (size_t)(a.F + 2);
  if (smem <= 48 * 1024) {
    emb_conv1_rows_kernel<<<a.B * 80, 256, smem, st>>>(a);
    return cudaGetLastError();
  }
  const long long total = (long long)a.B * 80 * a.F;
  const int grid = (int)min((long long)148 * 16, (total + 255) / 256);
  emb_conv1_kernel<<<grid, 256, 0, st>>>(a);
  return cudaGetLastError();
}

// zero the two border columns (w = 0 and w = W + 1) of a zero-bordered NHWC plane set [B*H][W + 2][C] (+ slack)
__global__ void zero_borders_kernel(bf16* __restrict__ p, long long plane, int planes, long long rows, int W, int C) {
  const long long total = rows * 2 * C;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    const long long r = i / C;
    const long long row = r >> 1;
    const int side = (int)(r & 1);
    const long long o = (row * (W + 2) + (side ? W + 1 : 0)) * C + c;
    p[o] = __float2bfloat16_rn(0.f);
    if (planes > 1) p[plane + o] = __float2bfloat16_rn(0.f);
  }
}
cudaError_t launch_zero_borders(bf16* p, long long plane, int planes, long long rows, int W, int C, cudaStream_t st) {
  const long long total = rows * 2 * C;
  const int grid = (int)min((long long)148 * 8, (total + 255) / 256);
  zero_borders_kernel<<<grid, 256, 0, st>>>(p, plane, planes, rows, W, C);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// K15 masked statistics pooling.  x: zero-bordered NHWC planes [b][h][1 + w][C] (C = 256, h < H = 10);
// masks [b][S][T] -> weights nearest-interpolated to W frames through widx[w];
//   v1 = sum w + 1e-8; mean = sum x w / v1; var = sum (x - mean)^2 w / (v1 - sum w^2 / v1 + 1e-8); std = sqrt(var)
// out planes [b*S + s][2*C*H]: mean at c*H + h, std at C*H + c*H + h ("(dimension channel)" flattening).
// One CTA per (b, h), one thread per channel.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) stats_pool_kernel(PoolArgs a) {
  extern __shared__ float wsm[];  // [S][W]
  const int b = blockIdx.y, h = blockIdx.x, c = threadIdx.x;
  for (int i = threadIdx.x; i < a.S * a.W; i += blockDim.x) {
    const int s = i / a.W, w = i - s * a.W;
    wsm[i] = a.masks[((long long)b * a.S + s) * a.T + a.widx[w]];
  }
  __syncthreads();
  if (c >= a.C) return;
  const bf16* xp = a.x + (((long long)b * a.H + h) * (a.W + 2) + 1) * a.C + c;
  float v1[4] = {0.f, 0.f, 0.f, 0.f}, v2[4] = {0.f, 0.f, 0.f, 0.f}, sx[4] = {0.f, 0.f, 0.f, 0.f};
  for (int w = 0; w < a.W; ++w) {
    float x = from16(xp[(long long)w * a.C], a.fp16);
    if (a.planes > 1) x += from16(xp[a.x_plane + (long long)w * a.C], a.fp16);
#pragma unroll
    for (int s = 0; s < 4; ++s)
      if (s < a.S) { const float wt = wsm[s * a.W + w]; v1[s] += wt; v2[s] += wt * wt; sx[s] += x * wt; }
  }
  float mean[4], dx[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int s = 0; s < 4; ++s) { v1[s] += 1e-8f; mean[s] = sx[s] / v1[s]; }
  for (int w = 0; w < a.W; ++w) {
    float x = from16(xp[(long long)w * a.C], a.fp16);
    if (a.planes > 1) x += from16(xp[a.x_plane + (long long)w * a.C], a.fp16);
#pragma unroll
    for (int s = 0; s < 4; ++s)
      if (s < a.S) { const float dl = x - mean[s]; dx[s] += dl * dl * wsm[s * a.W + w]; }
  }
  const int feat = a.C * a.H;
#pragma unroll
  for (int s = 0; s < 4; ++s) {
    if (s >= a.S) break;
    const float var = dx[s] / (v1[s] - v2[s] / v1[s] + 1e-8f);
    const float sd = sqrtf(var);
    bf16* o = a.out + ((long long)b * a.S + s) * a.ldo;
    bf16 hh, ll;
    split_bf16(mean[s], hh, ll, a.fp16);
    o[c * a.H + h] = hh;
    if (a.planes > 1) o[a.out_plane + c * a.H + h] = ll;
    split_bf16(sd, hh, ll, a.fp16);
    o[feat + c * a.H + h] = hh;
    if (a.planes > 1) o[a.out_plane + feat + c * a.H + h] = ll;
  }
}
cudaError_t launch_stats_pool(const PoolArgs& a, int B, cudaStream_t st) {
  if (a.S > 4 || a.C > 256) return cudaErrorInvalidValue;
  dim3 grid(a.H, B);
  const size_t smem = sizeof(float) * (size_t)a.S * a.W;
  stats_pool_kernel<<<grid, 256, smem, st>>>(a);
  return cudaGetLastError();
}

}  // namespace dz
