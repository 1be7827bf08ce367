// CUDA-core kernels of the segmentation path that are not GEMM-shaped: waveform statistics, the first
// convolution (C_in = 1: a 10-tap stencil, HBM-bound), LayerNorm rows, the relative-position gate,
// the conformer depthwise convolution, the classifier / log-softmax / powerset head.
// Reference call sites are cited per kernel.
#include <cstdint>

#include "common.cuh"
#include "seg_kernels.h"

namespace dz {

// ------------------------------------------------------------------------------------------------
// block reduction helpers
// ------------------------------------------------------------------------------------------------
template <typename T>
DZ_DEVINL T block_sum(T v, T* scratch /* >= 32 */) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = (blockDim.x + 31) >> 5;
  __syncthreads();
  if (l == 0) scratch[w] = v;
  __syncthreads();
  T r = (l < nw) ? scratch[l] : (T)0;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) r += __shfl_xor_sync(0xffffffffu, r, o);
  return r;  // valid in every thread of every warp
}

// ------------------------------------------------------------------------------------------------
// K1 waveform layer-norm statistics (large only).  reference: wav2vec2/model.py:106-113
// stats[b] = (mean, rstd) with biased variance, eps 1e-5.
// ------------------------------------------------------------------------------------------------
// Each window is cut into WS_SLICES slices (one CTA each, 16-byte loads, float64 sums of x and x^2); the last CTA of a window
// to finish adds the slice sums in slice order (deterministic) and writes (mean, rstd).  scratch: [B][WS_SLICES][2] doubles
// followed by [B] tickets (zero before the first launch; the finishing CTA resets its ticket).
static constexpr int WS_SLICES = 16;
__global__ void __launch_bounds__(256) wave_stats_kernel(const float* __restrict__ wav, int N, float* __restrict__ stats,
                                                         double* __restrict__ part, unsigned* __restrict__ ticket) {
  __shared__ double sc[32];
  __shared__ unsigned s_last;
  const int b = blockIdx.y, sl = blockIdx.x;
  const float* x = wav + (long long)b * N;
  const int per = (((N + WS_SLICES - 1) / WS_SLICES) + 3) & ~3;
  const int lo = min(N, sl * per), hi = min(N, lo + per);
  double s = 0.0, q = 0.0;
  if ((((uintptr_t)x) & 15) == 0) {
    const int n4 = (hi - lo) >> 2;
    const float4* x4 = reinterpret_cast<const float4*>(x + lo);
    for (int i = threadIdx.x; i < n4; i += blockDim.x) {
      const float4 v = x4[i];
      s += ((double)v.x + (double)v.y) + ((double)v.z + (double)v.w);
      q += ((double)v.x * v.x + (double)v.y * v.y) + ((double)v.z * v.z + (double)v.w * v.w);
    }
    for (int i = lo + (n4 << 2) + threadIdx.x; i < hi; i += blockDim.x) { const double v = x[i]; s += v; q += v * v; }
  } else {
    for (int i = lo + threadIdx.x; i < hi; i += blockDim.x) { const double v = x[i]; s += v; q += v * v; }
  }
  s = block_sum<double>(s, sc);
  q = block_sum<double>(q, sc);
  if (threadIdx.x == 0) {
    part[((long long)b * WS_SLICES + sl) * 2] = s;
    part[((long long)b * WS_SLICES + sl) * 2 + 1] = q;
    __threadfence();
    s_last = atomicAdd(&ticket[b], 1u) == (unsigned)(WS_SLICES - 1);
  }
  __syncthreads();
  if (s_last && threadIdx.x == 0) {
    __threadfence();
    double ts = 0.0, tq = 0.0;
    for (int i = 0; i < WS_SLICES; ++i) {
      ts += __ldcg(&part[((long long)b * WS_SLICES + i) * 2]);
      tq += __ldcg(&part[((long long)b * WS_SLICES + i) * 2 + 1]);
    }
    const double mean = ts / N;
    const double var = fmax(tq / N - mean * mean, 0.0);
    stats[2 * b] = (float)mean;
    stats[2 * b + 1] = (float)(1.0 / sqrt(var + 1e-5));
    ticket[b] = 0;
  }
}

// ------------------------------------------------------------------------------------------------
// K2a (base): GroupNorm(C0 groups) statistics of conv0 WITHOUT materialising conv0.
// conv0 output y[t,c] = w_c . x[5t:5t+10]  =>  mean_c = w_c . S1 / T0,  E[y^2] = w_c^T S2 w_c / T0 where
// S1[k] = sum_t x[5t+k], S2[k][l] = sum_t x[5t+k] x[5t+l].  65 moments per window, accumulated in fp64.
// reference: components.py:1248-1253 (GroupNorm(num_groups=C0)) applied at components.py:119-121.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) conv0_moments_kernel(const float* __restrict__ wav, int N, int T0,
                                                           double* __restrict__ mom /*[B][65]*/) {
  __shared__ double sc[32];
  const float* x = wav + (long long)blockIdx.x * N;
  double s1[10], s2[55];
#pragma unroll
  for (int k = 0; k < 10; ++k) s1[k] = 0.0;
#pragma unroll
  for (int k = 0; k < 55; ++k) s2[k] = 0.0;
  for (int t = threadIdx.x; t < T0; t += blockDim.x) {
    float xv[10];
#pragma unroll
    for (int k = 0; k < 10; ++k) xv[k] = x[5 * t + k];
    int idx = 0;
#pragma unroll
    for (int k = 0; k < 10; ++k) {
      s1[k] += (double)xv[k];
#pragma unroll
      for (int l = k; l < 10; ++l) s2[idx++] += (double)xv[k] * (double)xv[l];
    }
  }
  double* o = mom + (long long)blockIdx.x * 65;
#pragma unroll
  for (int k = 0; k < 10; ++k) {
    const double r = block_sum<double>(s1[k], sc);
    if (threadIdx.x == 0) o[k] = r;
  }
#pragma unroll
  for (int k = 0; k < 55; ++k) {
    const double r = block_sum<double>(s2[k], sc);
    if (threadIdx.x == 0) o[10 + k] = r;
  }
}

// coef[b][c] = (scale, shift) such that GroupNorm(y)[t,c] = y[t,c]*scale + shift.
__global__ void conv0_gn_coef_kernel(const double* __restrict__ mom, const float* __restrict__ w /*[C0][10]*/,
                                     const float* __restrict__ gamma, const float* __restrict__ beta, int C0, int T0,
                                     float* __restrict__ coef /*[B][C0][2]*/) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  const int b = blockIdx.y;
  if (c >= C0) return;
  const double* m = mom + (long long)b * 65;
  double wv[10];
  for (int k = 0; k < 10; ++k) wv[k] = (double)w[c * 10 + k];
  double mean = 0.0, ey2 = 0.0;
  int idx = 0;
  for (int k = 0; k < 10; ++k) {
    mean += wv[k] * m[k];
    for (int l = k; l < 10; ++l) {
      const double t = wv[k] * wv[l] * m[10 + idx++];
      ey2 += (l == k) ? t : 2.0 * t;
    }
  }
  mean /= T0;
  ey2 /= T0;
  double var = ey2 - mean * mean;
  if (var < 0.0) var = 0.0;
  const double scale = (double)gamma[c] / sqrt(var + 1e-5);
  coef[((long long)b * C0 + c) * 2] = (float)scale;
  coef[((long long)b * C0 + c) * 2 + 1] = (float)((double)beta[c] - mean * scale);
}

// ------------------------------------------------------------------------------------------------
// K2 conv0 (1 -> C0, k = 10, stride 5, no bias) + norm + GELU, channels-last bf16 plane output.
//   LARGE: waveform normalisation on load, LayerNorm over the C0 channels of each time step.
//   base : per-(window, channel) affine from conv0_gn_coef_kernel.
// One warp per time step; lane owns channel pairs (2*lane + 64*i, +1) so stores are 128-byte coalesced.
// reference: components.py:119-122 (conv -> norm -> gelu), :63-70 (LayerNorm with transpose).
// ------------------------------------------------------------------------------------------------
static constexpr int C0_TT = 64;  // time steps per CTA
template <bool LARGE>
__global__ void __launch_bounds__(256) conv0_kernel(Conv0Args a) {
  extern __shared__ float sm0[];
  float* xs = sm0;                       // 5*TT + 5 samples
  float* ws = xs + (5 * C0_TT + 8);      // [10][C0p2]  (C0p2 = channel count padded to 64)
  float* cf = ws + 10 * a.C0p64;         // base: [C0p64][2] scale/shift ; large: gamma/beta
  const int b = blockIdx.y;
  const int t0 = blockIdx.x * C0_TT;
  const float* x = a.wav + (long long)b * a.N;
  float mu = 0.f, rs = 1.f;
  if (LARGE) { mu = a.wstats[2 * b]; rs = a.wstats[2 * b + 1]; }
  for (int i = threadIdx.x; i < 5 * C0_TT + 5; i += blockDim.x) {
    const int s = 5 * t0 + i;
    xs[i] = (s < a.N) ? (x[s] - mu) * rs : 0.f;
  }
  for (int i = threadIdx.x; i < 10 * a.C0p64; i += blockDim.x) {
    const int k = i / a.C0p64, c = i - k * a.C0p64;
    ws[i] = (c < a.C0) ? a.w[c * 10 + k] : 0.f;
  }
  for (int i = threadIdx.x; i < a.C0p64; i += blockDim.x) {
    float p = 0.f, q = 0.f;
    if (i < a.C0) {
      if (LARGE) { p = a.gamma[i]; q = a.beta[i]; }
      else { p = a.coef[((long long)b * a.C0 + i) * 2]; q = a.coef[((long long)b * a.C0 + i) * 2 + 1]; }
    }
    cf[2 * i] = p; cf[2 * i + 1] = q;
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int npair = a.C0p64 / 64;  // pairs per lane (<= 8)
  for (int tt = warp; tt < C0_TT; tt += 8) {
    const int t = t0 + tt;
    if (t >= a.T0) break;
    float xw[10];
#pragma unroll
    for (int k = 0; k < 10; ++k) xw[k] = xs[5 * tt + k];
    float y[16];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float y0 = 0.f, y1 = 0.f;
      if (i < npair) {
        const int c = 2 * lane + 64 * i;
#pragma unroll
        for (int k = 0; k < 10; ++k) {
          const float2 wv = *reinterpret_cast<const float2*>(ws + k * a.C0p64 + c);
          y0 = fmaf(wv.x, xw[k], y0);
          y1 = fmaf(wv.y, xw[k], y1);
        }
      }
      y[2 * i] = y0; y[2 * i + 1] = y1;
    }
    float mean = 0.f, rstd = 1.f;
    if (LARGE) {
      float s = 0.f;
#pragma unroll
      for (int i = 0; i < 16; ++i) s += y[i];  // padded channels contribute exact zeros
      mean = warp_sum(s) / a.C0;
      float q = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        if (i < npair) {
          const int c = 2 * lane + 64 * i;
          if (c < a.C0) { const float dl = y[2 * i] - mean; q += dl * dl; }
          if (c + 1 < a.C0) { const float dl = y[2 * i + 1] - mean; q += dl * dl; }
        }
      }
      rstd = rsqrtf(warp_sum(q) / a.C0 + 1e-5f);
    }
    bf16* oh = a.out + (long long)b * a.out_bstride + (long long)t * a.ldo;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      if (i < npair) {
        const int c = 2 * lane + 64 * i;
        if (c < a.ldo) {
          float v0, v1;
          if (LARGE) {
            v0 = (y[2 * i] - mean) * rstd * cf[2 * c] + cf[2 * c + 1];
            v1 = (y[2 * i + 1] - mean) * rstd * cf[2 * c + 2] + cf[2 * c + 3];
          } else {
            v0 = y[2 * i] * cf[2 * c] + cf[2 * c + 1];
            v1 = y[2 * i + 1] * cf[2 * c + 2] + cf[2 * c + 3];
          }
          v0 = (c < a.C0) ? gelu_erf(v0) : 0.f;
          v1 = (c + 1 < a.C0) ? gelu_erf(v1) : 0.f;
          if (a.planes > 1) {
            bf16 h0, l0, h1, l1;
            split_bf16(v0, h0, l0, a.fp16);
            split_bf16(v1, h1, l1, a.fp16);
            *reinterpret_cast<__nv_bfloat162*>(oh + c) = __halves2bfloat162(h0, h1);
            *reinterpret_cast<__nv_bfloat162*>(oh + a.out_plane + c) = __halves2bfloat162(l0, l1);
          } else {
            *reinterpret_cast<uint32_t*>(oh + c) = a.fp16 ? pack2_16<1>(v0, v1) : pack2_16<0>(v0, v1);
          }
        }
      }
    }
  }
}

size_t wave_stats_scratch_bytes(int B) { return (size_t)B * WS_SLICES * 2 * sizeof(double) + (size_t)B * sizeof(unsigned); }
cudaError_t launch_wave_stats(const float* wav, int B, int N, float* stats, void* scratch, cudaStream_t st) {
  double* part = reinterpret_cast<double*>(scratch);
  unsigned* ticket = reinterpret_cast<unsigned*>(part + (size_t)B * WS_SLICES * 2);
  wave_stats_kernel<<<dim3(WS_SLICES, B), 256, 0, st>>>(wav, N, stats, part, ticket);
  return cudaGetLastError();
}
cudaError_t launch_conv0_moments(const float* wav, int B, int N, int T0, double* mom, cudaStream_t st) {
  conv0_moments_kernel<<<B, 256, 0, st>>>(wav, N, T0, mom);
  return cudaGetLastError();
}
cudaError_t launch_conv0_gn_coef(const double* mom, const float* w, const float* gamma, const float* beta, int B, int C0,
                                 int T0, float* coef, cudaStream_t st) {
  dim3 grid((C0 + 127) / 128, B);
  conv0_gn_coef_kernel<<<grid, 128, 0, st>>>(mom, w, gamma, beta, C0, T0, coef);
  return cudaGetLastError();
}
cudaError_t launch_conv0(const Conv0Args& a, int B, bool large, cudaStream_t st) {
  const size_t smem = sizeof(float) * ((5 * C0_TT + 8) + 10 * a.C0p64 + 2 * a.C0p64 + 4);
  dim3 grid((a.T0 + C0_TT - 1) / C0_TT, B);
  if (large) conv0_kernel<true><<<grid, 256, smem, st>>>(a);
  else conv0_kernel<false><<<grid, 256, smem, st>>>(a);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// K9 LayerNorm over rows (one warp per row, row cached in registers), optional fused prescale, activation,
// fp32 / bf16-plane outputs and layer-mix accumulation (K10: sum_l w_l h_l without torch.stack).
// reference: components.py:63-70, :305, :923-941, :983; conformer.py ln_norm; model_wavlm_conformer.py:235-236,253-257.
// ------------------------------------------------------------------------------------------------
template <int NV>  // float4 chunks per lane: C <= 128 * NV
__global__ void __launch_bounds__(256, 3) layernorm_rows_kernel(LnArgs a) {
  // gamma / beta / prescale staged once per CTA; each warp then walks rows with a grid stride
  extern __shared__ float lnsm[];
  float* sg = lnsm;
  float* sb = sg + NV * 128;
  float* sp = sb + NV * 128;
  for (int i = threadIdx.x; i < NV * 128; i += blockDim.x) {
    sg[i] = i < a.C ? a.gamma[i] : 0.f;
    sb[i] = i < a.C ? a.beta[i] : 0.f;
    sp[i] = (a.prescale != nullptr && i < a.C) ? a.prescale[i] : 1.f;
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool vec = (a.C % 4) == 0;
  for (long long row = (long long)blockIdx.x * 8 + warp; row < a.rows; row += (long long)gridDim.x * 8) {
    const float* xr = a.x + row * a.ldx;
    float v[NV * 4];
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c = (lane + 32 * i) * 4;
      float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
      if (c + 3 < a.C) {
        t = *reinterpret_cast<const float4*>(xr + c);
      } else {
        if (c < a.C) t.x = xr[c];
        if (c + 1 < a.C) t.y = xr[c + 1];
        if (c + 2 < a.C) t.z = xr[c + 2];
      }
      v[4 * i] = t.x; v[4 * i + 1] = t.y; v[4 * i + 2] = t.z; v[4 * i + 3] = t.w;
    }
    if (a.mix != nullptr && a.mix_src == 1) {
      float* mr = a.mix + row * a.ldx;
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        const int c = (lane + 32 * i) * 4;
        if (vec && c + 3 < a.C) {
          float4 m = a.mix_init ? make_float4(0.f, 0.f, 0.f, 0.f) : *reinterpret_cast<const float4*>(mr + c);
          m.x += a.mix_w * v[4 * i]; m.y += a.mix_w * v[4 * i + 1]; m.z += a.mix_w * v[4 * i + 2]; m.w += a.mix_w * v[4 * i + 3];
          *reinterpret_cast<float4*>(mr + c) = m;
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (c + j < a.C) mr[c + j] = (a.mix_init ? 0.f : mr[c + j]) + a.mix_w * v[4 * i + j];
        }
      }
    }
    if (a.prescale != nullptr) {
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        const float4 p4 = *reinterpret_cast<const float4*>(sp + (lane + 32 * i) * 4);
        v[4 * i] *= p4.x; v[4 * i + 1] *= p4.y; v[4 * i + 2] *= p4.z; v[4 * i + 3] *= p4.w;
      }
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < NV * 4; ++i) s += v[i];   // cells beyond C hold exact zeros
    const float mean = warp_sum(s) / a.C;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c = (lane + 32 * i) * 4;
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (c + j < a.C) { const float dl = v[4 * i + j] - mean; q += dl * dl; }
    }
    const float rstd = rsqrtf(warp_sum(q) / a.C + 1e-5f);
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c = (lane + 32 * i) * 4;
      const float4 g4 = *reinterpret_cast<const float4*>(sg + c);
      const float4 b4 = *reinterpret_cast<const float4*>(sb + c);
      const float gg[4] = {g4.x, g4.y, g4.z, g4.w}, bb[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float y = 0.f;
        if (c + j < a.C) y = apply_act((v[4 * i + j] - mean) * rstd * gg[j] + bb[j], a.act);
        v[4 * i + j] = y;
      }
    }
    if (a.mix != nullptr && a.mix_src == 2) {
      float* mr = a.mix + row * a.ldx;
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        const int c = (lane + 32 * i) * 4;
        if (vec && c + 3 < a.C) {
          float4 m = a.mix_init ? make_float4(0.f, 0.f, 0.f, 0.f) : *reinterpret_cast<const float4*>(mr + c);
          m.x += a.mix_w * v[4 * i]; m.y += a.mix_w * v[4 * i + 1]; m.z += a.mix_w * v[4 * i + 2]; m.w += a.mix_w * v[4 * i + 3];
          *reinterpret_cast<float4*>(mr + c) = m;
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (c + j < a.C) mr[c + j] = (a.mix_init ? 0.f : mr[c + j]) + a.mix_w * v[4 * i + j];
        }
      }
    }
    if (a.y_f32 != nullptr) {
      float* yr = a.y_f32 + row * a.ldy;
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        const int c = (lane + 32 * i) * 4;
        if (c + 3 < a.C) {
          *reinterpret_cast<float4*>(yr + c) = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (c + j < a.C) yr[c + j] = v[4 * i + j];
        }
      }
    }
    if (a.y_bf != nullptr) {
      bf16* hr = a.y_bf + row * a.ldb;
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        const int c = (lane + 32 * i) * 4;
        if (c + 3 < a.ldb) {  // ldb % 8 == 0: whole chunk inside the (zero padded) row
          bf16 h[4], l[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) split_bf16(v[4 * i + j], h[j], l[j], a.fp16);
          uint2 hw, lw;
          hw.x = (uint32_t)__bfloat16_as_ushort(h[0]) | ((uint32_t)__bfloat16_as_ushort(h[1]) << 16);
          hw.y = (uint32_t)__bfloat16_as_ushort(h[2]) | ((uint32_t)__bfloat16_as_ushort(h[3]) << 16);
          lw.x = (uint32_t)__bfloat16_as_ushort(l[0]) | ((uint32_t)__bfloat16_as_ushort(l[1]) << 16);
          lw.y = (uint32_t)__bfloat16_as_ushort(l[2]) | ((uint32_t)__bfloat16_as_ushort(l[3]) << 16);
          *reinterpret_cast<uint2*>(hr + c) = hw;
          if (a.planes > 1) *reinterpret_cast<uint2*>(hr + a.bf_plane + c) = lw;
        }
      }
    }
  }
}

// Fast path (C % 4 == 0, which every architecture here satisfies): operand format, plane count and activation are
// compile-time, so the per-element work is ~9 instructions and the kernel sits on the HBM roofline instead of the issue
// limit (the generic kernel above spends ~3x that on uniform-but-dynamic branches).
// A warp normalises R = 8 / NV rows per pass (one row at C = 1024, four at C = 256) so that every lane keeps eight 16-byte
// loads in flight whatever the row length; without the layer mix the kernel fits three CTAs per SM.
template <int NV, int FP16, int TWO, int ACT, int MIX>   // ACT: 0 none, 1 GELU, 2 anything else (dispatch on a.act)
__global__ void __launch_bounds__(256, MIX ? 2 : 3) layernorm_rows_fast_kernel(LnArgs a) {
  constexpr int R = 8 / NV;
  extern __shared__ float lnsm[];
  float* sg = lnsm;
  float* sb = sg + NV * 128;
  float* sp = sb + NV * 128;
  for (int i = threadIdx.x; i < NV * 128; i += blockDim.x) {
    sg[i] = i < a.C ? a.gamma[i] : 0.f;
    sb[i] = i < a.C ? a.beta[i] : 0.f;
    sp[i] = (a.prescale != nullptr && i < a.C) ? a.prescale[i] : 1.f;
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float invC = 1.0f / (float)a.C;
  const bool mix_in = MIX && a.mix_src == 1, mix_out = MIX && a.mix_src == 2;
  const bool has_pre = a.prescale != nullptr;
  const float mw = a.mix_w;
  for (long long row0 = ((long long)blockIdx.x * 8 + warp) * R; row0 < a.rows; row0 += (long long)gridDim.x * 8 * R) {
    float4 v[R][NV];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const long long row = row0 + r;
      const float* xr = a.x + row * a.ldx;
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        const int c = (lane + 32 * i) * 4;
        v[r][i] = (c < a.C && row < a.rows) ? *reinterpret_cast<const float4*>(xr + c) : make_float4(0.f, 0.f, 0.f, 0.f);   // rows are padded to ldx >= rup(C, 4)
        if (c + 3 >= a.C) {   // the chunk that straddles C: the padding columns hold stale data
          if (c + 1 >= a.C) v[r][i].y = 0.f;
          if (c + 2 >= a.C) v[r][i].z = 0.f;
          v[r][i].w = 0.f;
        }
      }
    }
    float4 m[MIX ? R : 1][MIX ? NV : 1];
    if (MIX) {
#pragma unroll
      for (int r = 0; r < R; ++r) {
        const long long row = row0 + r;
        float* mr = a.mix + row * a.ldx;
#pragma unroll
        for (int i = 0; i < NV; ++i) {
          const int c = (lane + 32 * i) * 4;
          m[MIX ? r : 0][MIX ? i : 0] = (!a.mix_init && c < a.C && row < a.rows) ? *reinterpret_cast<const float4*>(mr + c) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
      if (mix_in) {
#pragma unroll
        for (int r = 0; r < R; ++r) {
          const long long row = row0 + r;
          float* mr = a.mix + row * a.ldx;
#pragma unroll
          for (int i = 0; i < NV; ++i) {
            const int c = (lane + 32 * i) * 4;
            float4& mm = m[MIX ? r : 0][MIX ? i : 0];
            mm.x = fmaf(mw, v[r][i].x, mm.x); mm.y = fmaf(mw, v[r][i].y, mm.y);
            mm.z = fmaf(mw, v[r][i].z, mm.z); mm.w = fmaf(mw, v[r][i].w, mm.w);
            if (c < a.C && row < a.rows) *reinterpret_cast<float4*>(mr + c) = mm;
          }
        }
      }
    }
    if (has_pre) {
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        const float4 p4 = *reinterpret_cast<const float4*>(sp + (lane + 32 * i) * 4);
#pragma unroll
        for (int r = 0; r < R; ++r) { v[r][i].x *= p4.x; v[r][i].y *= p4.y; v[r][i].z *= p4.z; v[r][i].w *= p4.w; }
      }
    }
    float s[R], q[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      s[r] = 0.f;
#pragma unroll
      for (int i = 0; i < NV; ++i) s[r] += (v[r][i].x + v[r][i].y) + (v[r][i].z + v[r][i].w);   // cells beyond C hold exact zeros
    }
#pragma unroll
    for (int r = 0; r < R; ++r) s[r] = warp_sum(s[r]) * invC;                                    // mean
#pragma unroll
    for (int r = 0; r < R; ++r) {
      q[r] = 0.f;
      const float mean = s[r];
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        const int c = (lane + 32 * i) * 4;
        if (c < a.C) {
          float4 dd = make_float4(v[r][i].x - mean, v[r][i].y - mean, v[r][i].z - mean, v[r][i].w - mean);
          if (c + 3 >= a.C) {
            if (c + 1 >= a.C) dd.y = 0.f;
            if (c + 2 >= a.C) dd.z = 0.f;
            dd.w = 0.f;
          }
          q[r] = fmaf(dd.x, dd.x, q[r]); q[r] = fmaf(dd.y, dd.y, q[r]); q[r] = fmaf(dd.z, dd.z, q[r]); q[r] = fmaf(dd.w, dd.w, q[r]);
          v[r][i] = dd;
        }
      }
    }
#pragma unroll
    for (int r = 0; r < R; ++r) q[r] = rsqrtf(warp_sum(q[r]) * invC + 1e-5f);                    // 1 / std
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c = (lane + 32 * i) * 4;
      const float4 g4 = *reinterpret_cast<const float4*>(sg + c);
      const float4 b4 = *reinterpret_cast<const float4*>(sb + c);
#pragma unroll
      for (int r = 0; r < R; ++r) {
        const float rstd = q[r];
        float4 y = make_float4(fmaf(v[r][i].x * rstd, g4.x, b4.x), fmaf(v[r][i].y * rstd, g4.y, b4.y),
                               fmaf(v[r][i].z * rstd, g4.z, b4.z), fmaf(v[r][i].w * rstd, g4.w, b4.w));
        if (ACT == 1) { y.x = gelu_erf(y.x); y.y = gelu_erf(y.y); y.z = gelu_erf(y.z); y.w = gelu_erf(y.w); }
        if (ACT == 2) { y.x = apply_act(y.x, a.act); y.y = apply_act(y.y, a.act); y.z = apply_act(y.z, a.act); y.w = apply_act(y.w, a.act); }
        if (c + 3 >= a.C) {   // columns >= C (and whole chunks past C) are written as zeros
          if (c >= a.C) y.x = 0.f;
          if (c + 1 >= a.C) y.y = 0.f;
          if (c + 2 >= a.C) y.z = 0.f;
          y.w = 0.f;
        }
        v[r][i] = y;
      }
    }
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const long long row = row0 + r;
      if (row >= a.rows) break;
      if (mix_out) {
        float* mr = a.mix + row * a.ldx;
#pragma unroll
        for (int i = 0; i < NV; ++i) {
          const int c = (lane + 32 * i) * 4;
          float4& mm = m[MIX ? r : 0][MIX ? i : 0];
          mm.x = fmaf(mw, v[r][i].x, mm.x); mm.y = fmaf(mw, v[r][i].y, mm.y);
          mm.z = fmaf(mw, v[r][i].z, mm.z); mm.w = fmaf(mw, v[r][i].w, mm.w);
          if (c < a.C) *reinterpret_cast<float4*>(mr + c) = mm;
        }
      }
      if (a.y_f32 != nullptr) {
        float* yr = a.y_f32 + row * a.ldy;
#pragma unroll
        for (int i = 0; i < NV; ++i) {
          const int c = (lane + 32 * i) * 4;
          if (c < a.C) *reinterpret_cast<float4*>(yr + c) = v[r][i];
        }
      }
      if (a.y_bf != nullptr) {
        bf16* hr = a.y_bf + row * a.ldb;
#pragma unroll
        for (int i = 0; i < NV; ++i) {
          const int c = (lane + 32 * i) * 4;
          if (c + 3 < a.ldb) {  // ldb % 8 == 0: whole chunk inside the (zero padded) row
            if (TWO) {
              bf16 h[4], l[4];
              split_bf16(v[r][i].x, h[0], l[0], FP16); split_bf16(v[r][i].y, h[1], l[1], FP16);
              split_bf16(v[r][i].z, h[2], l[2], FP16); split_bf16(v[r][i].w, h[3], l[3], FP16);
              uint2 hw, lw;
              hw.x = (uint32_t)__bfloat16_as_ushort(h[0]) | ((uint32_t)__bfloat16_as_ushort(h[1]) << 16);
              hw.y = (uint32_t)__bfloat16_as_ushort(h[2]) | ((uint32_t)__bfloat16_as_ushort(h[3]) << 16);
              lw.x = (uint32_t)__bfloat16_as_ushort(l[0]) | ((uint32_t)__bfloat16_as_ushort(l[1]) << 16);
              lw.y = (uint32_t)__bfloat16_as_ushort(l[2]) | ((uint32_t)__bfloat16_as_ushort(l[3]) << 16);
              *reinterpret_cast<uint2*>(hr + c) = hw;
              *reinterpret_cast<uint2*>(hr + a.bf_plane + c) = lw;
            } else {
              *reinterpret_cast<uint2*>(hr + c) = make_uint2(pack2_16<FP16>(v[r][i].x, v[r][i].y), pack2_16<FP16>(v[r][i].z, v[r][i].w));
            }
          }
        }
      }
    }
  }
}

template <int NV, int FP16, int TWO, int MIX>
static void launch_ln_fast(const LnArgs& a, unsigned grid, cudaStream_t st) {
  const size_t smem = 3 * NV * 128 * sizeof(float);
  if (a.act == 0) layernorm_rows_fast_kernel<NV, FP16, TWO, 0, MIX><<<grid, 256, smem, st>>>(a);
  else if (a.act == 1) layernorm_rows_fast_kernel<NV, FP16, TWO, 1, MIX><<<grid, 256, smem, st>>>(a);
  else layernorm_rows_fast_kernel<NV, FP16, TWO, 2, MIX><<<grid, 256, smem, st>>>(a);
}
template <int NV, int MIX>
static void launch_ln_fast_nv(const LnArgs& a, unsigned grid, cudaStream_t st) {
  const bool two = a.y_bf != nullptr && a.planes > 1;
  if (a.fp16) { if (two) launch_ln_fast<NV, 1, 1, MIX>(a, grid, st); else launch_ln_fast<NV, 1, 0, MIX>(a, grid, st); }
  else { if (two) launch_ln_fast<NV, 0, 1, MIX>(a, grid, st); else launch_ln_fast<NV, 0, 0, MIX>(a, grid, st); }
}

cudaError_t launch_layernorm(const LnArgs& a, cudaStream_t st) {
  // rows must be padded to a multiple of 4 floats; with the layer mix (always D-wide, D % 4 == 0) or a ragged C the
  // chunk straddling C is masked in registers
  const bool fast = (a.ldx % 4) == 0 && a.ldx >= ((a.C + 3) & ~3) && (a.y_f32 == nullptr || (a.ldy % 4 == 0 && a.ldy >= ((a.C + 3) & ~3))) &&
                    (a.mix == nullptr || (a.C % 4) == 0);
  if (fast) {
    if (a.C > 1024) return cudaErrorInvalidValue;
    const int per_cta = 8 * (a.C <= 256 ? 4 : a.C <= 512 ? 2 : 1);                // rows per CTA pass
    const long long want = (a.rows + per_cta - 1) / per_cta;
    const bool mix = a.mix != nullptr;
    const long long cap = 148 * (mix ? 2 : 3) * 4;
    const unsigned grid = (unsigned)(want < cap ? want : cap);
    if (a.C <= 256) { if (mix) launch_ln_fast_nv<2, 1>(a, grid, st); else launch_ln_fast_nv<2, 0>(a, grid, st); }
    else if (a.C <= 512) { if (mix) launch_ln_fast_nv<4, 1>(a, grid, st); else launch_ln_fast_nv<4, 0>(a, grid, st); }
    else { if (mix) launch_ln_fast_nv<8, 1>(a, grid, st); else launch_ln_fast_nv<8, 0>(a, grid, st); }
    return cudaGetLastError();
  }
  const long long want = (a.rows + 7) / 8;
  const unsigned grid = (unsigned)(want < 148 * 8 ? want : 148 * 8);
  if (a.C <= 256) layernorm_rows_kernel<2><<<grid, 256, 3 * 2 * 128 * sizeof(float), st>>>(a);
  else if (a.C <= 512) layernorm_rows_kernel<4><<<grid, 256, 3 * 4 * 128 * sizeof(float), st>>>(a);
  else if (a.C <= 1024) layernorm_rows_kernel<8><<<grid, 256, 3 * 8 * 128 * sizeof(float), st>>>(a);
  else return cudaErrorInvalidValue;
  return cudaGetLastError();
}

// mix = (init ? 0 : mix) + w * x   (flat fp32, n % 4 == 0)
__global__ void axpy_mix_kernel(const float4* __restrict__ x, float4* __restrict__ mix, float w, int init, long long n4) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const float4 xv = x[i];
    float4 m = init ? make_float4(0.f, 0.f, 0.f, 0.f) : mix[i];
    m.x += w * xv.x; m.y += w * xv.y; m.z += w * xv.z; m.w += w * xv.w;
    mix[i] = m;
  }
}
cudaError_t launch_axpy_mix(const float* x, float* mix, float w, int init, long long n, cudaStream_t st) {
  const long long n4 = n / 4;
  const int grid = (int)min((long long)148 * 8, (n4 + 255) / 256);
  axpy_mix_kernel<<<grid, 256, 0, st>>>(reinterpret_cast<const float4*>(x), reinterpret_cast<float4*>(mix), w, init, n4);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// fp32 rows -> bf16 planes with a column regrouping: column c -> (c / gin) * gout + c % gin and a row
// offset per sequence (used to stage the pos-conv input: 64 zero rows either side, 16 groups padded to
// 64 channels).  Pad cells are never written (buffer is zeroed at allocation).
// reference: components.py:366-380 (conv1d padding = 64 over time, groups = 16).
// ------------------------------------------------------------------------------------------------
__global__ void regroup_to_bf16_kernel(const float* __restrict__ x, long long rows, int C, int ldx, int seq_len,
                                       int seq_rows_out, int row_off, int gin, int gout, bf16* __restrict__ out,
                                       long long out_plane, int ldo, int planes, int fp16) {
  const long long total = rows * C;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / C;
    const int c = (int)(i - r * C);
    const long long sb = r / seq_len;
    const int t = (int)(r - sb * seq_len);
    const float v = x[r * ldx + c];
    bf16 h, l;
    split_bf16(v, h, l, fp16);
    const long long o = (sb * seq_rows_out + t + row_off) * ldo + (c / gin) * gout + (c % gin);
    out[o] = h;
    if (planes > 1) out[out_plane + o] = l;
  }
}
// Eight columns per thread (two 16-byte loads, one 16-byte store per plane), one warp per row, one division per row: the
// scalar kernel above pays two 64-bit divisions and 2-byte stores per element (0.36 ms for 77 M elements; this one 0.1 ms).
__global__ void __launch_bounds__(256) regroup_to_bf16_vec8_kernel(const float* __restrict__ x, long long rows, int C, int ldx,
                                                                   int seq_len, int seq_rows_out, int row_off, int gin, int gout,
                                                                   bf16* __restrict__ out, long long out_plane, int ldo, int planes,
                                                                   int fp16) {
  const int cpr = C >> 3, lane = threadIdx.x & 31;
  for (long long r = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); r < rows; r += (long long)gridDim.x * 8) {
    const long long sb = r / seq_len;
    const int t = (int)(r - sb * seq_len);
    const float* xr = x + r * ldx;
    bf16* orow = out + (sb * seq_rows_out + t + row_off) * (long long)ldo;
    for (int k = lane; k < cpr; k += 32) {
      const int c = k << 3;
      const float4 v0 = __ldg(reinterpret_cast<const float4*>(xr + c)), v1 = __ldg(reinterpret_cast<const float4*>(xr + c + 4));
      const float v[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
      uint32_t hw[4], lw[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        bf16 h0, l0, h1, l1;
        split_bf16(v[2 * e], h0, l0, fp16);
        split_bf16(v[2 * e + 1], h1, l1, fp16);
        hw[e] = (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
        lw[e] = (uint32_t)__bfloat16_as_ushort(l0) | ((uint32_t)__bfloat16_as_ushort(l1) << 16);
      }
      const int oc = (c / gin) * gout + (c % gin);
      *reinterpret_cast<uint4*>(orow + oc) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
      if (planes > 1) *reinterpret_cast<uint4*>(orow + out_plane + oc) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
    }
  }
}
cudaError_t launch_regroup(const float* x, long long rows, int C, int ldx, int seq_len, int seq_rows_out, int row_off,
                           int gin, int gout, bf16* out, long long out_plane, int ldo, int planes, int fp16, cudaStream_t st) {
  if (C % 8 == 0 && gin % 8 == 0 && gout % 8 == 0 && ldx % 4 == 0 && ldo % 8 == 0 && out_plane % 8 == 0 &&
      (((uintptr_t)x) & 15) == 0 && (((uintptr_t)out) & 15) == 0) {
    const int grid = (int)min((long long)148 * 8, (rows + 7) / 8);
    regroup_to_bf16_vec8_kernel<<<grid, 256, 0, st>>>(x, rows, C, ldx, seq_len, seq_rows_out, row_off, gin, gout, out, out_plane,
                                                      ldo, planes, fp16);
    return cudaGetLastError();
  }
  const long long total = rows * C;
  const int grid = (int)min((long long)148 * 16, (total + 255) / 256);
  regroup_to_bf16_kernel<<<grid, 256, 0, st>>>(x, rows, C, ldx, seq_len, seq_rows_out, row_off, gin, gout, out, out_plane,
                                               ldo, planes, fp16);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// K7 gated relative-position gate.  For every (row, remaining head):
//   ga = sigmoid(wa_h . x_h + ba), gb = sigmoid(wb_h . x_h + bb), gate = ga * (gb * const_h - 1) + 2
// where x_h is the 64-wide slice of the *layer input* for total-head index h and wa/wb are the sums of the
// first / last four rows of gru_rel_pos_linear (the reference sums the 8 outputs in two groups of 4).
// reference: components.py:702-710.  Output layout gate[b][hi][t] (hi = index among remaining heads).
// ------------------------------------------------------------------------------------------------
// Eight lanes per head (one 16-byte load of 8 channels each), four heads per warp pass, reductions over 8 lanes.
template <bool TWO, int FP16>   // TWO: hi + lo operand planes; FP16: operand format (compile-time conversions)
__global__ void __launch_bounds__(256, TWO ? 2 : 4) relpos_gate_kernel(GateArgs a) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, grp = lane >> 3, sub = lane & 7;
  const long long row = (long long)blockIdx.x * 8 + warp;
  if (row >= a.rows) return;
  const bf16* xr = a.x + row * a.ldx;
  const long long sb = row / a.seq_len;
  const int t = (int)(row - sb * a.seq_len);
  float wa[8], wb[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { wa[j] = a.wab[sub * 8 + j]; wb[j] = a.wab[64 + sub * 8 + j]; }
  const int npass = (a.nheads + 3) >> 2;
  uint4 raw[4], rawl[TWO ? 4 : 1];
#pragma unroll
  for (int it = 0; it < 4; ++it) {               // all loads of the row first (<= 16 remaining heads)
    const int hi = it * 4 + grp;
    raw[it] = make_uint4(0u, 0u, 0u, 0u);
    if (TWO) rawl[TWO ? it : 0] = raw[it];
    if (it < npass && hi < a.nheads) {
      const bf16* hp = xr + a.head_index[hi] * 64 + sub * 8;
      raw[it] = *reinterpret_cast<const uint4*>(hp);
      if (TWO) rawl[TWO ? it : 0] = *reinterpret_cast<const uint4*>(hp + a.x_plane);
    }
  }
#pragma unroll
  for (int it = 0; it < 4; ++it) {
    if (it >= npass) break;
    const int hi = it * 4 + grp;
    const bf16* e = reinterpret_cast<const bf16*>(&raw[it]);
    const bf16* el = reinterpret_cast<const bf16*>(&rawl[TWO ? it : 0]);
    float sa = 0.f, sb2 = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float xv = from16(e[j], FP16);
      if (TWO) xv += from16(el[j], FP16);
      sa = fmaf(wa[j], xv, sa);
      sb2 = fmaf(wb[j], xv, sb2);
    }
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) {
      sa += __shfl_xor_sync(0xffffffffu, sa, o);
      sb2 += __shfl_xor_sync(0xffffffffu, sb2, o);
    }
    if (sub == 0 && hi < a.nheads) {
      const float ga = 1.f / (1.f + expf(-(sa + a.ba))), gb = 1.f / (1.f + expf(-(sb2 + a.bb)));
      a.gate[(sb * a.nheads + hi) * a.seq_len + t] = ga * (gb * a.gconst[a.head_index[hi]] - 1.f) + 2.f;
    }
  }
}
cudaError_t launch_gate(const GateArgs& a, cudaStream_t st) {
  const unsigned grid = (unsigned)((a.rows + 7) / 8);
  if (a.planes > 1) { if (a.fp16) relpos_gate_kernel<true, 1><<<grid, 256, 0, st>>>(a); else relpos_gate_kernel<true, 0><<<grid, 256, 0, st>>>(a); }
  else { if (a.fp16) relpos_gate_kernel<false, 1><<<grid, 256, 0, st>>>(a); else relpos_gate_kernel<false, 0><<<grid, 256, 0, st>>>(a); }
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// CUDA-core attention (checker / bf16x3 mode): one thread per query row, keys streamed through shared
// memory in tiles of 64, online softmax per thread (no cross-thread reductions), fp32 throughout.
//   scores = q.k (+ gate[q] * tab[k - q + T - 1]) ; softmax ; ctx = P V
// q already carries the 1/sqrt(64) scaling (folded into the projection weights).
// reference: components.py:455-480 (+ bias :690-725), conformer.py:48-70.
// ------------------------------------------------------------------------------------------------
static constexpr int AT_Q = 128;
static constexpr int AT_K = 64;
__global__ void __launch_bounds__(AT_Q) attention_simt_kernel(AttnArgs a) {
  extern __shared__ float sma[];
  float* Ks = sma;                    // [64 keys][64 d]
  float* Vs = Ks + AT_K * 64;         // [64 d][64 keys]
  float* tab = Vs + 64 * AT_K;        // [2T-1] bias row of this head (optional)
  const int T = a.T;
  const int hi = blockIdx.y, b = blockIdx.z;
  const int q0 = blockIdx.x * AT_Q;
  const int tq = q0 + threadIdx.x;
  const bool qvalid = tq < T;
  const bool two = a.planes > 1;
  if (a.bias_tab != nullptr)
    for (int i = threadIdx.x; i < 2 * T - 1; i += AT_Q) tab[i] = a.bias_tab[(long long)hi * (2 * T - 1) + i];
  float q[64], o[64];
  {
    const bf16* qp = a.q + ((long long)b * T + (qvalid ? tq : 0)) * a.ldqk + a.q_col + hi * 64;
#pragma unroll
    for (int d = 0; d < 64; ++d) {
      float v = from16(qp[d], a.fp16);
      if (two) v += from16(qp[a.qk_plane + d], a.fp16);
      q[d] = v;
      o[d] = 0.f;
    }
  }
  const float gate = (a.gate != nullptr && qvalid) ? a.gate[((long long)b * a.nheads + hi) * T + tq] : 0.f;
  float mrun = -INFINITY, lrun = 0.f;
  for (int k0 = 0; k0 < T; k0 += AT_K) {
    __syncthreads();
    for (int i = threadIdx.x; i < AT_K * 64; i += AT_Q) {
      const int j = i >> 6, d = i & 63;
      float v = 0.f;
      if (k0 + j < T) {
        const bf16* kp = a.k + ((long long)b * T + k0 + j) * a.ldqk + a.k_col + hi * 64 + d;
        v = from16(*kp, a.fp16);
        if (two) v += from16(kp[a.qk_plane], a.fp16);
      }
      Ks[i] = v;
    }
    for (int i = threadIdx.x; i < 64 * AT_K; i += AT_Q) {
      const int d = i >> 6, j = i & 63;
      float v = 0.f;
      if (k0 + j < T) {
        if (a.v != nullptr) {
          const bf16* vp = a.v + ((long long)b * T + k0 + j) * a.ldqk + a.v_col + hi * 64 + d;
          v = from16(*vp, a.fp16);
          if (two) v += from16(vp[a.qk_plane], a.fp16);
        } else {
          const bf16* vp = a.vt + ((long long)b * a.nheads * 64 + hi * 64 + d) * a.ldvt + k0 + j;
          v = from16(*vp, a.fp16);
          if (two) v += from16(vp[a.vt_plane], a.fp16);
        }
      }
      Vs[i] = v;
    }
    __syncthreads();
#pragma unroll 1
    for (int jc = 0; jc < AT_K; jc += 8) {
      float s[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4* kr = reinterpret_cast<const float4*>(Ks + (jc + j) * 64);
        float acc = 0.f;
#pragma unroll
        for (int d4 = 0; d4 < 16; ++d4) {
          const float4 kv = kr[d4];
          acc = fmaf(q[4 * d4], kv.x, acc);
          acc = fmaf(q[4 * d4 + 1], kv.y, acc);
          acc = fmaf(q[4 * d4 + 2], kv.z, acc);
          acc = fmaf(q[4 * d4 + 3], kv.w, acc);
        }
        const int kk = k0 + jc + j;
        if (a.bias_tab != nullptr && qvalid && kk < T) acc += gate * tab[kk - tq + T - 1];
        s[j] = (kk < T) ? acc : -INFINITY;
      }
      float cm = s[0];
#pragma unroll
      for (int j = 1; j < 8; ++j) cm = fmaxf(cm, s[j]);
      if (cm == -INFINITY) continue;  // whole chunk past the end
      const float mnew = fmaxf(mrun, cm);
      const float corr = __expf(mrun - mnew);  // exp(-inf) = 0 on the first chunk
      lrun *= corr;
      float p[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) { p[j] = __expf(s[j] - mnew); lrun += p[j]; }
#pragma unroll
      for (int d = 0; d < 64; ++d) {
        const float4 v0 = *reinterpret_cast<const float4*>(Vs + d * AT_K + jc);
        const float4 v1 = *reinterpret_cast<const float4*>(Vs + d * AT_K + jc + 4);
        float acc = o[d] * corr;
        acc = fmaf(p[0], v0.x, acc); acc = fmaf(p[1], v0.y, acc); acc = fmaf(p[2], v0.z, acc); acc = fmaf(p[3], v0.w, acc);
        acc = fmaf(p[4], v1.x, acc); acc = fmaf(p[5], v1.y, acc); acc = fmaf(p[6], v1.z, acc); acc = fmaf(p[7], v1.w, acc);
        o[d] = acc;
      }
      mrun = mnew;
    }
  }
  if (qvalid) {
    const float inv = 1.f / lrun;
    bf16* op = a.out + ((long long)b * T + tq) * a.ldo + hi * 64;
#pragma unroll
    for (int d = 0; d < 64; d += 2) {
      bf16 h0, l0, h1, l1;
      split_bf16(o[d] * inv, h0, l0, a.fp16);
      split_bf16(o[d + 1] * inv, h1, l1, a.fp16);
      *reinterpret_cast<__nv_bfloat162*>(op + d) = __halves2bfloat162(h0, h1);
      if (a.out_planes > 1) *reinterpret_cast<__nv_bfloat162*>(op + a.out_plane + d) = __halves2bfloat162(l0, l1);
    }
  }
}
cudaError_t launch_attention_simt(const AttnArgs& a, int B, cudaStream_t st) {
  const size_t smem = sizeof(float) * (AT_K * 64 * 2 + (a.bias_tab ? 2 * a.T - 1 : 0) + 4);
  static bool attr = false;
  if (!attr) {
    cudaFuncSetAttribute(attention_simt_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
    attr = true;
  }
  dim3 grid((a.T + AT_Q - 1) / AT_Q, a.nheads, B);
  attention_simt_kernel<<<grid, AT_Q, smem, st>>>(a);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// Conformer convolution module core: GLU -> depthwise conv (k taps, 'same' padding) -> BatchNorm (eval,
// folded into scale/shift together with the conv bias) -> Swish -> bf16 planes.
// in: [B*T][2A] fp32 (pointwise_conv1 output), out: [B*T][A] bf16 planes.
// reference: conformer.py:205-211.
// ------------------------------------------------------------------------------------------------
static constexpr int DW_TT = 32;
__global__ void __launch_bounds__(256) glu_dwconv_kernel(DwArgs a) {
  extern __shared__ float smd[];  // [(TT + k - 1)][A]
  const int A = a.A, K = a.ksize, half = (K - 1) / 2;
  const int b = blockIdx.y, t0 = blockIdx.x * DW_TT;
  const int nrow = DW_TT + K - 1;
  for (int i = threadIdx.x; i < nrow * A; i += blockDim.x) {
    const int r = i / A, c = i - r * A;
    const int t = t0 + r - half;
    float v = 0.f;
    if (t >= 0 && t < a.T) {
      const float* xr = a.x + ((long long)b * a.T + t) * a.ldx;
      const float g = xr[A + c];
      v = xr[c] / (1.f + expf(-g));
    }
    smd[i] = v;
  }
  __syncthreads();
  for (int c = threadIdx.x; c < A; c += blockDim.x) {
    float w[32];
#pragma unroll
    for (int k = 0; k < 32; ++k) w[k] = (k < K) ? a.w[c * K + k] : 0.f;
    const float sc = a.scale[c], sh = a.shift[c];
    for (int tt = 0; tt < DW_TT; ++tt) {
      const int t = t0 + tt;
      if (t >= a.T) break;
      float acc = 0.f;
#pragma unroll
      for (int k = 0; k < 32; ++k)
        if (k < K) acc = fmaf(w[k], smd[(tt + k) * A + c], acc);
      float y = acc * sc + sh;
      y = y / (1.f + expf(-y));
      bf16 h, l;
      split_bf16(y, h, l, a.fp16);
      const long long o = ((long long)b * a.T + t) * a.ldo + c;
      a.out[o] = h;
      if (a.planes > 1) a.out[a.out_plane + o] = l;
    }
  }
}
// v2, used whenever its shared memory fits in 200 KB (the kernel above takes wider heads): same accumulation order per
// output, fast-intrinsic sigmoids (ncu of the IEEE-division version: 264 instructions per output, most of them the two
// sigmoids); 64 frames per CTA (halo overhead 1.47x instead of 1.94x) and four outputs per thread in flight, which share
// every shared-memory load (0.27 LDS per FMA instead of 1) and break the dependent FMA chain.
static constexpr int DW2_TT = 64;
template <int KS>   // KS > 0: kernel size known at compile time (31 in every shipped configuration) - no per-tap predicates
__global__ void __launch_bounds__(256) glu_dwconv_v2_kernel(DwArgs a) {
  extern __shared__ float smd[];  // [(TT + k - 1)][A]
  const int A = a.A, K = KS > 0 ? KS : a.ksize, half = (K - 1) / 2;
  const int b = blockIdx.y, t0 = blockIdx.x * DW2_TT;
  const int nrow = DW2_TT + K - 1;
  // staging: eight rows' loads are issued before the first shared-memory store (a store per row would otherwise fence the
  // next row's loads behind it: 94 dependent global round trips per CTA)
  const float* __restrict__ xin = a.x;
  for (int c = threadIdx.x; c < A; c += blockDim.x) {
    for (int r0 = 0; r0 < nrow; r0 += 8) {
      float xa[8], xg[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int r = r0 + u, t = t0 + r - half;
        const bool in = r < nrow && t >= 0 && t < a.T;
        const float* xr = xin + ((long long)b * a.T + (in ? t : 0)) * a.ldx;
        xa[u] = in ? __ldg(xr + c) : 0.f;
        xg[u] = in ? __ldg(xr + A + c) : 0.f;
      }
#pragma unroll
      for (int u = 0; u < 8; ++u)     // GLU gate; same fast sigmoid as the GEMM epilogue's swish (rows outside the sequence: 0 / 2 = 0)
        if (r0 + u < nrow) smd[(r0 + u) * A + c] = __fdividef(xa[u], 1.f + __expf(-xg[u]));
    }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < A; c += blockDim.x) {
    float w[32];
#pragma unroll
    for (int k = 0; k < 32; ++k) w[k] = (k < K) ? a.w[c * K + k] : 0.f;
    const float sc = a.scale[c], sh = a.shift[c];
    for (int tt = 0; tt < DW2_TT; tt += 4) {
      if (t0 + tt >= a.T) break;
      float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int k = 0; k < 35; ++k) {            // input row tt + k feeds output tt + u with tap k - u
        if (k < K + 3) {
          const float v = smd[(tt + k) * A + c];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int kk = k - u;
            if (kk >= 0 && kk < 32 && kk < K) acc[u] = fmaf(w[kk < 0 ? 0 : (kk > 31 ? 31 : kk)], v, acc[u]);
          }
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int tq = t0 + tt + u;
        if (tq < a.T) {
          float y = acc[u] * sc + sh;
          y = __fdividef(y, 1.f + __expf(-y));
          bf16 h, l;
          split_bf16(y, h, l, a.fp16);
          const long long o = ((long long)b * a.T + tq) * a.ldo + c;
          a.out[o] = h;
          if (a.planes > 1) a.out[a.out_plane + o] = l;
        }
      }
    }
  }
}

cudaError_t launch_glu_dwconv(const DwArgs& a, int B, cudaStream_t st) {
  if (a.ksize > 32) return cudaErrorInvalidValue;
  const size_t smem2 = sizeof(float) * (size_t)(DW2_TT + a.ksize - 1) * a.A;
  if (smem2 <= 200 * 1024) {
    static size_t attr2 = 0;
    if (smem2 > 48 * 1024 && smem2 > attr2) {
      cudaFuncSetAttribute(glu_dwconv_v2_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2);
      cudaFuncSetAttribute(glu_dwconv_v2_kernel<31>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2);
      attr2 = smem2;
    }
    dim3 grid2((a.T + DW2_TT - 1) / DW2_TT, B);
    if (a.ksize == 31) glu_dwconv_v2_kernel<31><<<grid2, 256, smem2, st>>>(a);
    else glu_dwconv_v2_kernel<0><<<grid2, 256, smem2, st>>>(a);
    return cudaGetLastError();
  }
  const size_t smem = sizeof(float) * (size_t)(DW_TT + a.ksize - 1) * a.A;
  static size_t attr = 0;
  if (smem > 48 * 1024 && smem > attr) {
    cudaFuncSetAttribute(glu_dwconv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    attr = smem;
  }
  dim3 grid((a.T + DW_TT - 1) / DW_TT, B);
  glu_dwconv_kernel<<<grid, 256, smem, st>>>(a);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// K12 head: final LayerNorm of the last conformer block is done by layernorm_rows; this kernel does
// classifier (A -> NC <= 16) + log-softmax + hard powerset decoding (argmax -> multilabel LUT).
// reference: model_wavlm_conformer.py:261-262, pa/utils/powerset.py:103-128, pa/core/inference.py:225-226.
// One warp per frame.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) classifier_head_kernel(HeadArgs a) {
  extern __shared__ float smw[];  // [NC][A] weights + [NC] bias
  for (int i = threadIdx.x; i < a.NC * a.A; i += blockDim.x) smw[i] = a.w[i];
  for (int i = threadIdx.x; i < a.NC; i += blockDim.x) smw[a.NC * a.A + i] = a.bias[i];
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * 8 + warp;
  if (row >= a.rows) return;
  const float* xr = a.x + row * a.ldx;
  float acc[16];
#pragma unroll
  for (int n = 0; n < 16; ++n) acc[n] = 0.f;
  for (int c = lane; c < a.A; c += 32) {
    const float xv = xr[c];
#pragma unroll
    for (int n = 0; n < 16; ++n)
      if (n < a.NC) acc[n] = fmaf(xv, smw[n * a.A + c], acc[n]);
  }
#pragma unroll
  for (int n = 0; n < 16; ++n) acc[n] = warp_sum(acc[n]);
  if (lane == 0) {
    float mx = -INFINITY;
    int arg = 0;
#pragma unroll
    for (int n = 0; n < 16; ++n)
      if (n < a.NC) {
        acc[n] += smw[a.NC * a.A + n];
        if (acc[n] > mx) { mx = acc[n]; arg = n; }  // first maximum, as torch.argmax
      }
    float se = 0.f;
#pragma unroll
    for (int n = 0; n < 16; ++n)
      if (n < a.NC) se += expf(acc[n] - mx);
    const float lse = mx + logf(se);
    if (a.logp != nullptr) {
#pragma unroll
      for (int n = 0; n < 16; ++n)
        if (n < a.NC) a.logp[row * a.NC + n] = acc[n] - lse;
    }
    if (a.multilabel != nullptr) {
      // powerset classes in reference order: {}, {0},{1},{2},{3}, {0,1},{0,2},{0,3},{1,2},{1,3},{2,3}
      const unsigned lut[11] = {0x0, 0x1, 0x2, 0x4, 0x8, 0x3, 0x5, 0x9, 0x6, 0xA, 0xC};
      const unsigned m = (arg < 11) ? lut[arg] : 0u;
      uchar4 o;
      o.x = m & 1; o.y = (m >> 1) & 1; o.z = (m >> 2) & 1; o.w = (m >> 3) & 1;
      *reinterpret_cast<uchar4*>(a.multilabel + row * 4) = o;
    }
  }
}
cudaError_t launch_classifier_head(const HeadArgs& a, cudaStream_t st) {
  if (a.NC > 16) return cudaErrorInvalidValue;
  const size_t smem = sizeof(float) * (size_t)(a.NC * a.A + a.NC);
  classifier_head_kernel<<<(unsigned)((a.rows + 7) / 8), 256, smem, st>>>(a);
  return cudaGetLastError();
}

}  // namespace dz
