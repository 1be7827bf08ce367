// tcgen05 flash attention for sm_100a with the WavLM gated relative-position bias computed on the fly.
//
//   scores[q,k] = Q[q].K[k]  (+ gate[q] * tab[k - q + T - 1])      Q carries the 1/sqrt(64) scaling
//   ctx[q]      = softmax_k(scores[q,:]) . V
//
// One work item = 128 queries of one (window, head); keys are streamed in blocks of 64.
//   warp 4      : TMA producer: the item's Q tile, then K_j (64 keys x 64 d) and V_j (64 keys x 64 d, or V^T_j), 3-stage ring
//   warp 5      : UMMA issuer: S = Q K_j^T (128x64, fp32 in TMEM), then O += P_j V_j (fp32 in TMEM)
//   warps 0..3  : softmax: one query row per thread (= one TMEM lane): tcgen05.ld S -> bias/mask -> running max with
//                 lazy rescaling of O (tcgen05.ld/st only when the max moved by > 8 in log2 units) -> exp2 ->
//                 bf16 P written to shared memory in the 128-byte-swizzled K-major layout the UMMA reads.
// The reference materialises the (B*H, T, T) bias tensor and the full score matrix
// (components.py:695-697, :455-469); here neither ever exists in HBM.
// reference: diarizen/models/module/wav2vec2/components.py:429-486, :668-725; conformer.py:27-71 (no bias).
#include <string>

#include "common.cuh"
#include "gemm.h"
#include "seg_kernels.h"

namespace dz {

bool make_tmap_bf16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_elems,
                    const uint32_t* box);

static constexpr int ABQ = 128;
static constexpr int ABK = 64;
static constexpr int A_THREADS = 192;
static constexpr float LOG2E = 1.4426950408889634f;

struct AttnMaps { CUtensorMap q, k, vt; };

struct AttnPlan {
  AttnArgs a;
  AttnMaps maps;
  int B;
  size_t smem;
  int x3 = 0;                 // split-precision kernel (attention_tc3_kernel)
  CUtensorMap m3[6];          // q hi/lo, k hi/lo, v hi/lo
};

DZ_DEVINL float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// ================================================================================================
// v2: software-pipelined kernel (bf16 or fp16 operands; V row-major or transposed):
//   * two S accumulators in TMEM: S_{j+1} = Q K_{j+1}^T is issued before the softmax of block j finishes, so the tensor
//     pipe and the softmax warps overlap instead of alternating;
//   * two P buffers and a 3-stage K/V ring to go with it;
//   * the softmax denominator comes out of the tensor core: V^T gets a constant 65th row of ones (plus 15 zero rows, N = 80),
//     so O[:,64] = sum_k P[q,k] of exactly the rounded P the numerator uses, and it follows the lazy rescaling for free;
//   * scores are formed relative to the running reference in one FFMA (+ one FFMA for the gated bias), the row maximum uses
//     3-input max, masking runs only in the last key block.
// TMEM: S0 [0,64) S1 [64,128) O [128,208) of a 256-column allocation (2 CTAs/SM = the full 512 columns).
// ================================================================================================
static constexpr int KV_STAGES = 3;
static constexpr int V_STAGE_BYTES = 8192 + 2048;

DZ_DEVINL float fmax3(float a, float b, float c) {
  float r;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
  return r;
}
DZ_DEVINL uint32_t pack16(float lo, float hi, int fp16) {
  uint32_t r;
  if (fp16) asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  else asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}

template <int FP16, int VROW>
__global__ void __launch_bounds__(A_THREADS, 2) attention_tc2_kernel(const __grid_constant__ AttnMaps maps, const AttnArgs a,
                                                                     const int B) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_align1024(smem_raw);
  uint8_t* Qs = smem;                              // 128 x 64, SW128
  uint8_t* Ks = Qs + 16384;                        // KV_STAGES x (64 keys x 64 d)
  uint8_t* Vs = Ks + KV_STAGES * 8192;             // KV_STAGES x (80 rows x 64 keys): 64 d rows + ones row + 15 zero rows
  // VROW: V arrives row-major (64 keys x 64 d per stage, MN-major B operand) and the ones column lives in one shared 8 KB
  // constant block after the stages (second 64-wide N chunk, reached through the descriptor's leading byte offset)
  constexpr int VST = VROW ? 8192 : V_STAGE_BYTES;
  constexpr int VTOT = VROW ? KV_STAGES * 8192 + 8192 : KV_STAGES * V_STAGE_BYTES;
  uint8_t* Vc = Vs + KV_STAGES * 8192;
  uint8_t* Ps = Vs + VTOT;                         // 2 x (128 x 64), SW128
  uint64_t* bars = reinterpret_cast<uint64_t*>(Ps + 2 * 16384);
  uint64_t* q_full = bars;
  uint64_t* q_empty = bars + 1;
  uint64_t* kv_full = bars + 2;    // [3]
  uint64_t* kv_empty = bars + 5;   // [3]
  uint64_t* s_full = bars + 8;     // [2]
  uint64_t* p_ready = bars + 10;   // [2]
  uint64_t* o_ready = bars + 12;   // one phase per key block
  uint64_t* o_final = bars + 13;   // one phase per work item
  uint64_t* o_free = bars + 14;    // one phase per work item (the 4 softmax warps have read O out of TMEM)
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 15);
  float* tab = reinterpret_cast<float*>(bars + 16);  // [2T-1 + 64 pad]

  const int T = a.T;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nblk = (T + ABK - 1) / ABK;
  const int nqt = (T + ABQ - 1) / ABQ;
  const int n_items = B * a.nheads * nqt;   // item = ((head * B) + window) * nqt + query tile: head-major, so that a
                                            // persistent CTA keeps its bias table across consecutive items
  const bool has_bias = a.bias_tab != nullptr;

  if (threadIdx.x == 0) {
    mbar_init(q_full, 1);
    mbar_init(q_empty, 1);
    for (int s = 0; s < KV_STAGES; ++s) { mbar_init(&kv_full[s], 1); mbar_init(&kv_empty[s], 1); }
    mbar_init(&s_full[0], 1); mbar_init(&s_full[1], 1);
    mbar_init(&p_ready[0], 4); mbar_init(&p_ready[1], 4);
    mbar_init(o_ready, 1);
    mbar_init(o_final, 1);
    mbar_init(o_free, 4);
    mbar_fence_init();
    tma_prefetch_desc(&maps.q); tma_prefetch_desc(&maps.k); tma_prefetch_desc(&maps.vt);
  }
  if (warp == 5) tmem_alloc(tmem_ptr, 256);
  {
    // constant tail of every V stage: row 64 = ones (swizzle phase 0: stored as is), rows 65..79 = zeros
    const uint32_t one2 = FP16 ? 0x3C003C00u : 0x3F803F80u;
    if (VROW) {
      // row r (key) of the constant block: column 0 = 1, columns 1..63 = 0; column 0 sits in 16-byte chunk (0 ^ (r & 7))
      for (int i = threadIdx.x; i < 2048; i += A_THREADS) {
        const int r = i >> 5, wd = i & 31;
        reinterpret_cast<uint32_t*>(Vc)[i] = (wd == ((r & 7) << 2)) ? (one2 & 0xFFFFu) : 0u;
      }
    } else {
      for (int i = threadIdx.x; i < KV_STAGES * 512; i += A_THREADS) {
        const int s = i >> 9, wd = i & 511;
        reinterpret_cast<uint32_t*>(Vs + s * V_STAGE_BYTES + 8192)[wd] = wd < 32 ? one2 : 0u;
      }
    }
    fence_proxy_async();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  const uint32_t tmem_O = tmem_base + 128;

  if (warp == 4) {
    if (lane == 0) {
      uint32_t g = 0, n = 0;
      for (int it = blockIdx.x; it < n_items; it += gridDim.x, ++n) {
        const int qt = it % nqt, pair = it / nqt, b = pair % B, hi = pair / B;
        if (n > 0) mbar_wait(q_empty, (n - 1) & 1);   // every S = Q K^T of the previous item has completed
        mbar_expect_tx(q_full, 16384);
        tma_load_3d(Qs, &maps.q, q_full, a.q_col + hi * 64, qt * ABQ, b);
        for (int j = 0; j < nblk; ++j, ++g) {
          const uint32_t s = g % KV_STAGES, use = g / KV_STAGES;
          if (use > 0) mbar_wait(&kv_empty[s], (use - 1) & 1);
          mbar_expect_tx(&kv_full[s], 16384);
          tma_load_3d(Ks + s * 8192, &maps.k, &kv_full[s], a.k_col + hi * 64, j * ABK, b);
          if (VROW) tma_load_3d(Vs + s * VST, &maps.vt, &kv_full[s], a.v_col + hi * 64, j * ABK, b);
          else tma_load_3d(Vs + s * VST, &maps.vt, &kv_full[s], j * ABK, hi * 64, b);
        }
      }
    }
  } else if (warp == 5) {
    if (lane == 0) {
      const uint32_t idesc_s = umma_idesc_bf16(128, 64, FP16);
      const uint32_t idesc_o = umma_idesc_bf16(128, 80, FP16) | (VROW ? (1u << 16) : 0u);   // bit 16: B is MN-major
      const uint32_t qa = smem_u32(Qs);
      uint32_t g = 0, n = 0;
      for (int it = blockIdx.x; it < n_items; it += gridDim.x, ++n) {
        mbar_wait(q_full, n & 1);
        {
          const uint32_t s0 = g % KV_STAGES;
          mbar_wait(&kv_full[s0], (g / KV_STAGES) & 1);
          tc_fence_after();
          const uint32_t ka = smem_u32(Ks + s0 * 8192), ts = tmem_base + (g & 1) * 64;
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_bf16(ts, umma_desc_sw128(qa + k * 32), umma_desc_sw128(ka + k * 32), idesc_s, k > 0);
          umma_commit(&s_full[g & 1]);
          if (nblk == 1) umma_commit(q_empty);
        }
        for (int j = 0; j < nblk; ++j, ++g) {
          if (j + 1 < nblk) {
            // S of the next block: its TMEM buffer was last read by the softmax of block g-1, whose p_ready we have observed
            const uint32_t g1 = g + 1, s1 = g1 % KV_STAGES;
            mbar_wait(&kv_full[s1], (g1 / KV_STAGES) & 1);
            tc_fence_after();
            const uint32_t ka = smem_u32(Ks + s1 * 8192), ts = tmem_base + (g1 & 1) * 64;
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_bf16(ts, umma_desc_sw128(qa + k * 32), umma_desc_sw128(ka + k * 32), idesc_s, k > 0);
            umma_commit(&s_full[g1 & 1]);
            if (j + 2 == nblk) umma_commit(q_empty);   // last read of this item's Q tile
          }
          const uint32_t s = g % KV_STAGES;
          mbar_wait(&p_ready[g & 1], (g >> 1) & 1);
          if (j == 0 && n > 0) mbar_wait(o_free, (n - 1) & 1);   // the previous item's O has been read out of TMEM
          tc_fence_after();
          const uint32_t pa = smem_u32(Ps + (g & 1) * 16384), va = smem_u32(Vs + s * VST);
          if (VROW) {
            const uint32_t lbo = smem_u32(Vc) - va;   // first N chunk (d 0..63) -> second chunk (ones column + 15 zeros)
#pragma unroll
            for (int k = 0; k < 4; ++k)   // 16 keys = 16 rows of 128 B per step
              umma_bf16(tmem_O, umma_desc_sw128(pa + k * 32), umma_desc_sw128_mn(va + k * 2048, lbo), idesc_o, (j > 0 || k > 0) ? 1u : 0u);
          } else {
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_bf16(tmem_O, umma_desc_sw128(pa + k * 32), umma_desc_sw128(va + k * 32), idesc_o, (j > 0 || k > 0) ? 1u : 0u);
          }
          umma_commit(&kv_empty[s]);
          umma_commit(o_ready);
        }
        umma_commit(o_final);
      }
    }
  } else {
    // ---------------- softmax warps: thread <-> query row <-> TMEM lane ----------------
    const int row = threadIdx.x;  // 0..127
    const uint32_t lane_off = (uint32_t)(warp * 32) << 16;
    const int sw = row & 7;
    uint32_t g = 0, n = 0;
    int cur_h = -1;
    for (int it = blockIdx.x; it < n_items; it += gridDim.x, ++n) {
      const int qt = it % nqt, pair = it / nqt, b = pair % B, hi = pair / B;
      const int tq = qt * ABQ + row;
      const bool qvalid = tq < T;
      const float gate = (has_bias && a.gate != nullptr) ? a.gate[((long long)b * a.nheads + hi) * T + (qvalid ? tq : T - 1)] * LOG2E : 0.f;
      if (has_bias && hi != cur_h) {
        asm volatile("bar.sync 1, 128;" ::: "memory");   // everybody is done with the previous head's table
        const float* src = a.bias_tab + (long long)hi * (2 * T - 1);
        for (int i = row; i < 2 * T - 1 + 64; i += 128) tab[i] = (i < 2 * T - 1) ? src[i] : 0.f;
        asm volatile("bar.sync 1, 128;" ::: "memory");
        cur_h = hi;
      }
      const float* trow = tab + (T - 1) - (qvalid ? tq : T - 1);  // trow[k] = tab[k - q + T - 1]
      float m_used = 0.f;   // reference exponent (log2 domain); block 0 always re-references
      for (int j = 0; j < nblk; ++j, ++g) {
        mbar_wait(&s_full[g & 1], (g >> 1) & 1);
        tc_fence_after();
        float r[64];
        {
          uint32_t* ru = reinterpret_cast<uint32_t*>(r);
          const uint32_t ts = tmem_base + (g & 1) * 64 + lane_off;
          tmem_ld_32x32(ts, ru);
          tmem_ld_32x32(ts + 32, ru + 32);
          tmem_ld_wait();
        }
        const int kbase = j * ABK;
        const float negm = -m_used;
        if (has_bias) {
          const float* tr = trow + kbase;
#pragma unroll
          for (int c = 0; c < 64; ++c) r[c] = fmaf(gate, tr[c], fmaf(r[c], LOG2E, negm));
        } else {
#pragma unroll
          for (int c = 0; c < 64; ++c) r[c] = fmaf(r[c], LOG2E, negm);
        }
        if (j == nblk - 1) {
          const int nvalid = T - kbase;
#pragma unroll
          for (int c = 0; c < 64; ++c) r[c] = (c < nvalid) ? r[c] : -INFINITY;
        }
        float mx = fmax3(r[0], r[1], r[2]);
#pragma unroll
        for (int c = 3; c + 1 < 64; c += 2) mx = fmax3(mx, r[c], r[c + 1]);
        mx = fmaxf(mx, r[63]);
        // lazy re-referencing: exponentials stay relative to m_used unless the row maximum moved by more than 2^8
        const bool need = (j == 0) || (mx > 8.0f);
        if (need) {
          m_used += mx;
#pragma unroll
          for (int c = 0; c < 64; ++c) r[c] -= mx;
        }
        if (j > 0 && __any_sync(0xffffffffu, need)) {
          const float corr = need ? ex2(-mx) : 1.0f;
          mbar_wait(o_ready, (g - 1) & 1);   // P V of the previous block has landed in O
          tc_fence_after();
          uint32_t o[32];
#pragma unroll
          for (int hlf = 0; hlf < 2; ++hlf) {
            tmem_ld_32x32(tmem_O + lane_off + hlf * 32, o);
            tmem_ld_wait();
#pragma unroll
            for (int c = 0; c < 32; ++c) o[c] = __float_as_uint(__uint_as_float(o[c]) * corr);
            tmem_st_32x32(tmem_O + lane_off + hlf * 32, o);
          }
          {
            uint32_t o1[16];
            tmem_ld_32x32_x16(tmem_O + lane_off + 64, o1);
            tmem_ld_wait();
            tmem_st_32x32_x1(tmem_O + lane_off + 64, __float_as_uint(__uint_as_float(o1[0]) * corr));
          }
          tmem_st_wait();
        }
        uint8_t* prow = Ps + (g & 1) * 16384 + row * 128;
#pragma unroll
        for (int c8 = 0; c8 < 8; ++c8) {
          uint32_t w[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) w[e] = pack2_16<FP16>(ex2(r[8 * c8 + 2 * e]), ex2(r[8 * c8 + 2 * e + 1]));
          *reinterpret_cast<uint4*>(prow + ((c8 ^ sw) << 4)) = make_uint4(w[0], w[1], w[2], w[3]);
        }
        fence_proxy_async();   // generic-proxy smem writes -> visible to the tensor core (async proxy)
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&p_ready[g & 1]);
      }
      mbar_wait(o_final, n & 1);
      tc_fence_after();
      uint32_t o[64], o1[16];
      tmem_ld_32x32(tmem_O + lane_off, o);
      tmem_ld_32x32(tmem_O + lane_off + 32, o + 32);
      tmem_ld_32x32_x16(tmem_O + lane_off + 64, o1);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(o_free);
      if (qvalid) {
        const float inv = 1.0f / __uint_as_float(o1[0]);
        bf16* op = a.out + ((long long)b * T + tq) * a.ldo + hi * 64;
#pragma unroll
        for (int c8 = 0; c8 < 8; ++c8) {
          uint32_t hw[4], lw[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            bf16 h0, l0, h1, l1;
            split_bf16(__uint_as_float(o[8 * c8 + 2 * e]) * inv, h0, l0, FP16);
            split_bf16(__uint_as_float(o[8 * c8 + 2 * e + 1]) * inv, h1, l1, FP16);
            hw[e] = (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
            lw[e] = (uint32_t)__bfloat16_as_ushort(l0) | ((uint32_t)__bfloat16_as_ushort(l1) << 16);
          }
          *reinterpret_cast<uint4*>(op + 8 * c8) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
          if (a.out_planes > 1) *reinterpret_cast<uint4*>(op + a.out_plane + 8 * c8) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
        }
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 5) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 256);
  }
}

// ================================================================================================
// v3: split-precision (bf16x3, fp32-class) variant of the kernel above for the 1e-3 parity mode - until round 2 that mode fell
// back to the CUDA-core kernel (50 % of its run time).  Operands arrive as bf16 hi + lo planes; both products are
// accumulated as three tensor-core passes into the same fp32 accumulator:
//   S  = Qh Kh^T + Ql Kh^T + Qh Kl^T                      (12 UMMAs of K = 16 per 64-key block)
//   O += Ph Vh + Pl Vh + Ph Vl                            (the softmax warps write P as hi and lo planes)
// The ones column that yields the softmax denominator rides on the two Vh passes (N = 80), so the denominator is
// sum_k (Ph + Pl)[q,k] - exactly the P the numerator uses; the Vl pass runs with N = 64.
// Shared memory: Q 2 x 16 KB, K / V rings 3 x (8 + 8) KB each, ones block 8 KB, P 2 x (16 + 16) KB = 200 KB: one CTA per SM.
// Everything else (persistent head-major work list, S ping-pong in TMEM, lazy rescaling, gated bias from the table) is as above.
// ================================================================================================
struct AttnMaps3 { CUtensorMap q[2], k[2], v[2]; };

__global__ void __launch_bounds__(A_THREADS, 1) attention_tc3_kernel(const __grid_constant__ AttnMaps3 maps, const AttnArgs a,
                                                                     const int B) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_align1024(smem_raw);
  uint8_t* Qs = smem;                              // hi 16 KB | lo 16 KB
  uint8_t* Ks = Qs + 32768;                        // KV_STAGES x (hi 8 KB | lo 8 KB)
  uint8_t* Vs = Ks + KV_STAGES * 16384;            // KV_STAGES x (hi 8 KB | lo 8 KB), row-major V: MN-major B operand
  uint8_t* Vc = Vs + KV_STAGES * 16384;            // ones block (second N chunk of the Vh passes)
  uint8_t* Ps = Vc + 8192;                         // 2 x (hi 16 KB | lo 16 KB)
  uint64_t* bars = reinterpret_cast<uint64_t*>(Ps + 2 * 32768);
  uint64_t* q_full = bars;
  uint64_t* q_empty = bars + 1;
  uint64_t* kv_full = bars + 2;    // [3]
  uint64_t* kv_empty = bars + 5;   // [3]
  uint64_t* s_full = bars + 8;     // [2]
  uint64_t* p_ready = bars + 10;   // [2]
  uint64_t* o_ready = bars + 12;
  uint64_t* o_final = bars + 13;
  uint64_t* o_free = bars + 14;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 15);
  float* tab = reinterpret_cast<float*>(bars + 16);  // [2T-1 + 64 pad]

  const int T = a.T;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nblk = (T + ABK - 1) / ABK;
  const int nqt = (T + ABQ - 1) / ABQ;
  const int n_items = B * a.nheads * nqt;
  const bool has_bias = a.bias_tab != nullptr;

  if (threadIdx.x == 0) {
    mbar_init(q_full, 1);
    mbar_init(q_empty, 1);
    for (int s = 0; s < KV_STAGES; ++s) { mbar_init(&kv_full[s], 1); mbar_init(&kv_empty[s], 1); }
    mbar_init(&s_full[0], 1); mbar_init(&s_full[1], 1);
    mbar_init(&p_ready[0], 4); mbar_init(&p_ready[1], 4);
    mbar_init(o_ready, 1);
    mbar_init(o_final, 1);
    mbar_init(o_free, 4);
    mbar_fence_init();
    for (int i = 0; i < 2; ++i) { tma_prefetch_desc(&maps.q[i]); tma_prefetch_desc(&maps.k[i]); tma_prefetch_desc(&maps.v[i]); }
  }
  if (warp == 5) tmem_alloc(tmem_ptr, 256);
  // ones block: row r (key) has column 0 = 1 (bf16), the rest 0; column 0 sits in 16-byte chunk (0 ^ (r & 7))
  for (int i = threadIdx.x; i < 2048; i += A_THREADS) {
    const int r = i >> 5, wd = i & 31;
    reinterpret_cast<uint32_t*>(Vc)[i] = (wd == ((r & 7) << 2)) ? 0x3F80u : 0u;
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  const uint32_t tmem_O = tmem_base + 128;

  if (warp == 4) {
    if (lane == 0) {
      uint32_t g = 0, n = 0;
      for (int it = blockIdx.x; it < n_items; it += gridDim.x, ++n) {
        const int qt = it % nqt, pair = it / nqt, b = pair % B, hi = pair / B;
        if (n > 0) mbar_wait(q_empty, (n - 1) & 1);
        mbar_expect_tx(q_full, 32768);
        tma_load_3d(Qs, &maps.q[0], q_full, a.q_col + hi * 64, qt * ABQ, b);
        tma_load_3d(Qs + 16384, &maps.q[1], q_full, a.q_col + hi * 64, qt * ABQ, b);
        for (int j = 0; j < nblk; ++j, ++g) {
          const uint32_t s = g % KV_STAGES, use = g / KV_STAGES;
          if (use > 0) mbar_wait(&kv_empty[s], (use - 1) & 1);
          mbar_expect_tx(&kv_full[s], 32768);
          tma_load_3d(Ks + s * 16384, &maps.k[0], &kv_full[s], a.k_col + hi * 64, j * ABK, b);
          tma_load_3d(Ks + s * 16384 + 8192, &maps.k[1], &kv_full[s], a.k_col + hi * 64, j * ABK, b);
          tma_load_3d(Vs + s * 16384, &maps.v[0], &kv_full[s], a.v_col + hi * 64, j * ABK, b);
          tma_load_3d(Vs + s * 16384 + 8192, &maps.v[1], &kv_full[s], a.v_col + hi * 64, j * ABK, b);
        }
      }
    }
  } else if (warp == 5) {
    if (lane == 0) {
      const uint32_t idesc_s = umma_idesc_bf16(128, 64, 0);
      const uint32_t idesc_o80 = umma_idesc_bf16(128, 80, 0) | (1u << 16);   // bit 16: B is MN-major
      const uint32_t idesc_o64 = umma_idesc_bf16(128, 64, 0) | (1u << 16);
      const uint32_t qa = smem_u32(Qs);
      uint32_t g = 0, n = 0;
      // S = Qh Kh^T + Ql Kh^T + Qh Kl^T into TMEM buffer (g & 1)
      auto issue_s = [&](uint32_t gg) {
        const uint32_t s0 = gg % KV_STAGES;
        mbar_wait(&kv_full[s0], (gg / KV_STAGES) & 1);
        tc_fence_after();
        const uint32_t ka = smem_u32(Ks + s0 * 16384), ts = tmem_base + (gg & 1) * 64;
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_bf16(ts, umma_desc_sw128(qa + k * 32), umma_desc_sw128(ka + k * 32), idesc_s, k > 0);
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_bf16(ts, umma_desc_sw128(qa + 16384 + k * 32), umma_desc_sw128(ka + k * 32), idesc_s, 1u);
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_bf16(ts, umma_desc_sw128(qa + k * 32), umma_desc_sw128(ka + 8192 + k * 32), idesc_s, 1u);
        umma_commit(&s_full[gg & 1]);
      };
      for (int it = blockIdx.x; it < n_items; it += gridDim.x, ++n) {
        mbar_wait(q_full, n & 1);
        issue_s(g);
        if (nblk == 1) umma_commit(q_empty);
        for (int j = 0; j < nblk; ++j, ++g) {
          if (j + 1 < nblk) {
            issue_s(g + 1);
            if (j + 2 == nblk) umma_commit(q_empty);   // last read of this item's Q tile
          }
          const uint32_t s = g % KV_STAGES;
          mbar_wait(&p_ready[g & 1], (g >> 1) & 1);
          if (j == 0 && n > 0) mbar_wait(o_free, (n - 1) & 1);
          tc_fence_after();
          const uint32_t pa = smem_u32(Ps + (g & 1) * 32768), va = smem_u32(Vs + s * 16384);
          const uint32_t lbo = smem_u32(Vc) - va;
#pragma unroll
          for (int k = 0; k < 4; ++k)   // Ph Vh (+ ones column)
            umma_bf16(tmem_O, umma_desc_sw128(pa + k * 32), umma_desc_sw128_mn(va + k * 2048, lbo), idesc_o80, (j > 0 || k > 0) ? 1u : 0u);
#pragma unroll
          for (int k = 0; k < 4; ++k)   // Pl Vh (+ ones column)
            umma_bf16(tmem_O, umma_desc_sw128(pa + 16384 + k * 32), umma_desc_sw128_mn(va + k * 2048, lbo), idesc_o80, 1u);
#pragma unroll
          for (int k = 0; k < 4; ++k)   // Ph Vl (64 columns: the denominator must not see it)
            umma_bf16(tmem_O, umma_desc_sw128(pa + k * 32), umma_desc_sw128_mn(va + 8192 + k * 2048, 1024), idesc_o64, 1u);
          umma_commit(&kv_empty[s]);
          umma_commit(o_ready);
        }
        umma_commit(o_final);
      }
    }
  } else {
    // ---------------- softmax warps: thread <-> query row <-> TMEM lane ----------------
    const int row = threadIdx.x;  // 0..127
    const uint32_t lane_off = (uint32_t)(warp * 32) << 16;
    const int sw = row & 7;
    uint32_t g = 0, n = 0;
    int cur_h = -1;
    for (int it = blockIdx.x; it < n_items; it += gridDim.x, ++n) {
      const int qt = it % nqt, pair = it / nqt, b = pair % B, hi = pair / B;
      const int tq = qt * ABQ + row;
      const bool qvalid = tq < T;
      const float gate = (has_bias && a.gate != nullptr) ? a.gate[((long long)b * a.nheads + hi) * T + (qvalid ? tq : T - 1)] * LOG2E : 0.f;
      if (has_bias && hi != cur_h) {
        asm volatile("bar.sync 1, 128;" ::: "memory");
        const float* src = a.bias_tab + (long long)hi * (2 * T - 1);
        for (int i = row; i < 2 * T - 1 + 64; i += 128) tab[i] = (i < 2 * T - 1) ? src[i] : 0.f;
        asm volatile("bar.sync 1, 128;" ::: "memory");
        cur_h = hi;
      }
      const float* trow = tab + (T - 1) - (qvalid ? tq : T - 1);
      float m_used = 0.f;
      for (int j = 0; j < nblk; ++j, ++g) {
        mbar_wait(&s_full[g & 1], (g >> 1) & 1);
        tc_fence_after();
        float r[64];
        {
          uint32_t* ru = reinterpret_cast<uint32_t*>(r);
          const uint32_t ts = tmem_base + (g & 1) * 64 + lane_off;
          tmem_ld_32x32(ts, ru);
          tmem_ld_32x32(ts + 32, ru + 32);
          tmem_ld_wait();
        }
        const int kbase = j * ABK;
        const float negm = -m_used;
        if (has_bias) {
          const float* tr = trow + kbase;
#pragma unroll
          for (int c = 0; c < 64; ++c) r[c] = fmaf(gate, tr[c], fmaf(r[c], LOG2E, negm));
        } else {
#pragma unroll
          for (int c = 0; c < 64; ++c) r[c] = fmaf(r[c], LOG2E, negm);
        }
        if (j == nblk - 1) {
          const int nvalid = T - kbase;
#pragma unroll
          for (int c = 0; c < 64; ++c) r[c] = (c < nvalid) ? r[c] : -INFINITY;
        }
        float mx = fmax3(r[0], r[1], r[2]);
#pragma unroll
        for (int c = 3; c + 1 < 64; c += 2) mx = fmax3(mx, r[c], r[c + 1]);
        mx = fmaxf(mx, r[63]);
        const bool need = (j == 0) || (mx > 8.0f);
        if (need) {
          m_used += mx;
#pragma unroll
          for (int c = 0; c < 64; ++c) r[c] -= mx;
        }
        if (j > 0 && __any_sync(0xffffffffu, need)) {
          const float corr = need ? ex2(-mx) : 1.0f;
          mbar_wait(o_ready, (g - 1) & 1);
          tc_fence_after();
          uint32_t o[32];
#pragma unroll
          for (int hlf = 0; hlf < 2; ++hlf) {
            tmem_ld_32x32(tmem_O + lane_off + hlf * 32, o);
            tmem_ld_wait();
#pragma unroll
            for (int c = 0; c < 32; ++c) o[c] = __float_as_uint(__uint_as_float(o[c]) * corr);
            tmem_st_32x32(tmem_O + lane_off + hlf * 32, o);
          }
          {
            uint32_t o1[16];
            tmem_ld_32x32_x16(tmem_O + lane_off + 64, o1);
            tmem_ld_wait();
            tmem_st_32x32_x1(tmem_O + lane_off + 64, __float_as_uint(__uint_as_float(o1[0]) * corr));
          }
          tmem_st_wait();
        }
        uint8_t* prow = Ps + (g & 1) * 32768 + row * 128;
#pragma unroll
        for (int c8 = 0; c8 < 8; ++c8) {
          uint32_t wh[4], wl[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float p0 = ex2(r[8 * c8 + 2 * e]), p1 = ex2(r[8 * c8 + 2 * e + 1]);
            const uint32_t h2 = pack2_16<0>(p0, p1);                      // bf16 hi pair (p0 in the low half)
            const float h0 = __uint_as_float(h2 << 16), h1 = __uint_as_float(h2 & 0xffff0000u);
            wh[e] = h2;
            wl[e] = pack2_16<0>(p0 - h0, p1 - h1);                        // lo = rn(p - hi)
          }
          *reinterpret_cast<uint4*>(prow + ((c8 ^ sw) << 4)) = make_uint4(wh[0], wh[1], wh[2], wh[3]);
          *reinterpret_cast<uint4*>(prow + 16384 + ((c8 ^ sw) << 4)) = make_uint4(wl[0], wl[1], wl[2], wl[3]);
        }
        fence_proxy_async();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&p_ready[g & 1]);
      }
      mbar_wait(o_final, n & 1);
      tc_fence_after();
      uint32_t o[64], o1[16];
      tmem_ld_32x32(tmem_O + lane_off, o);
      tmem_ld_32x32(tmem_O + lane_off + 32, o + 32);
      tmem_ld_32x32_x16(tmem_O + lane_off + 64, o1);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(o_free);
      if (qvalid) {
        const float inv = 1.0f / __uint_as_float(o1[0]);
        bf16* op = a.out + ((long long)b * T + tq) * a.ldo + hi * 64;
#pragma unroll
        for (int c8 = 0; c8 < 8; ++c8) {
          uint32_t hw[4], lw[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            bf16 h0, l0, h1, l1;
            split_bf16(__uint_as_float(o[8 * c8 + 2 * e]) * inv, h0, l0, 0);
            split_bf16(__uint_as_float(o[8 * c8 + 2 * e + 1]) * inv, h1, l1, 0);
            hw[e] = (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
            lw[e] = (uint32_t)__bfloat16_as_ushort(l0) | ((uint32_t)__bfloat16_as_ushort(l1) << 16);
          }
          *reinterpret_cast<uint4*>(op + 8 * c8) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
          if (a.out_planes > 1) *reinterpret_cast<uint4*>(op + a.out_plane + 8 * c8) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
        }
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 5) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 256);
  }
}

AttnPlan* attention_tc_plan_create(const AttnArgs& a, int B) {
  AttnPlan* p = new AttnPlan();
  p->a = a;
  p->B = B;
  const int T = a.T;
  if (a.planes > 1) {
    // bf16 hi + lo operand planes: the three-pass kernel (row-major V only, bf16 format)
    if (a.v == nullptr || a.fp16) { delete p; return nullptr; }
    uint64_t dims[3] = {(uint64_t)a.ldqk, (uint64_t)T, (uint64_t)B};
    uint64_t str[3] = {1, (uint64_t)a.ldqk, (uint64_t)T * a.ldqk};
    uint32_t boxq[3] = {64, ABQ, 1}, boxk[3] = {64, ABK, 1};
    bool ok = true;
    for (int pl = 0; pl < 2 && ok; ++pl) {
      ok = make_tmap_bf16(&p->m3[0 + pl], a.q + pl * a.qk_plane, 3, dims, str, boxq) &&
           make_tmap_bf16(&p->m3[2 + pl], a.k + pl * a.qk_plane, 3, dims, str, boxk) &&
           make_tmap_bf16(&p->m3[4 + pl], a.v + pl * a.qk_plane, 3, dims, str, boxk);
    }
    if (!ok) { delete p; return nullptr; }
    p->x3 = 1;
    p->smem = 1024 + 32768 + 2 * KV_STAGES * 16384 + 8192 + 2 * 32768 + 128 + sizeof(float) * (size_t)(2 * T - 1 + 64 + 8);
    return p;
  }
  {
    uint64_t dims[3] = {(uint64_t)a.ldqk, (uint64_t)T, (uint64_t)B};
    uint64_t str[3] = {1, (uint64_t)a.ldqk, (uint64_t)T * a.ldqk};
    uint32_t boxq[3] = {64, ABQ, 1}, boxk[3] = {64, ABK, 1};
    if (!make_tmap_bf16(&p->maps.q, a.q, 3, dims, str, boxq) || !make_tmap_bf16(&p->maps.k, a.k, 3, dims, str, boxk)) {
      delete p;
      return nullptr;
    }
  }
  if (a.v != nullptr) {
    uint64_t dims[3] = {(uint64_t)a.ldqk, (uint64_t)T, (uint64_t)B};
    uint64_t str[3] = {1, (uint64_t)a.ldqk, (uint64_t)T * a.ldqk};
    uint32_t box[3] = {64, ABK, 1};
    if (!make_tmap_bf16(&p->maps.vt, a.v, 3, dims, str, box)) { delete p; return nullptr; }
  } else {
    uint64_t dims[3] = {(uint64_t)T, (uint64_t)a.nheads * 64, (uint64_t)B};
    uint64_t str[3] = {1, (uint64_t)a.ldvt, (uint64_t)a.nheads * 64 * a.ldvt};
    uint32_t box[3] = {ABK, 64, 1};
    if (!make_tmap_bf16(&p->maps.vt, a.vt, 3, dims, str, box)) { delete p; return nullptr; }
  }
  p->smem = 1024 + 16384 + KV_STAGES * 8192 + (a.v != nullptr ? KV_STAGES * 8192 + 8192 : KV_STAGES * V_STAGE_BYTES) + 2 * 16384 + 128 +
            sizeof(float) * (size_t)(2 * T - 1 + 64 + 8);
  return p;
}
void attention_tc_plan_destroy(AttnPlan* p) { delete p; }

cudaError_t attention_tc_plan_launch(const AttnPlan* p, cudaStream_t st) {
  if (p->x3) {
    static size_t attr3 = 0;
    if (p->smem > attr3) {
      cudaError_t e = cudaFuncSetAttribute(attention_tc3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p->smem);
      if (e != cudaSuccess) return e;
      attr3 = p->smem;
    }
    static int sms = 0;
    if (!sms) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev); if (sms <= 0) sms = 148; }
    const long long items = (long long)((p->a.T + ABQ - 1) / ABQ) * p->a.nheads * p->B;
    AttnMaps3 m;
    for (int i = 0; i < 2; ++i) { m.q[i] = p->m3[i]; m.k[i] = p->m3[2 + i]; m.v[i] = p->m3[4 + i]; }
    attention_tc3_kernel<<<(unsigned)(items < sms ? items : sms), A_THREADS, p->smem, st>>>(m, p->a, p->B);
    return cudaGetLastError();
  }
  static size_t attr = 0;
  if (p->smem > attr) {
    cudaError_t e = cudaFuncSetAttribute(attention_tc2_kernel<0, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p->smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(attention_tc2_kernel<1, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p->smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(attention_tc2_kernel<0, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p->smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(attention_tc2_kernel<1, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p->smem);
    if (e != cudaSuccess) return e;
    attr = p->smem;
  }
  dim3 grid((p->a.T + ABQ - 1) / ABQ, p->a.nheads, p->B);
  static int slots = 0;
  if (!slots) {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    slots = 2 * sms;   // two resident CTAs per SM (launch bounds, 110 KB of shared memory and 256 TMEM columns each)
  }
  const long long items = (long long)grid.x * grid.y * grid.z;
  const unsigned g = (unsigned)(items < slots ? items : slots);
  const int variant = (p->a.fp16 ? 1 : 0) | (p->a.v != nullptr ? 2 : 0);
  switch (variant) {
    case 0: attention_tc2_kernel<0, 0><<<g, A_THREADS, p->smem, st>>>(p->maps, p->a, p->B); break;
    case 1: attention_tc2_kernel<1, 0><<<g, A_THREADS, p->smem, st>>>(p->maps, p->a, p->B); break;
    case 2: attention_tc2_kernel<0, 1><<<g, A_THREADS, p->smem, st>>>(p->maps, p->a, p->B); break;
    default: attention_tc2_kernel<1, 1><<<g, A_THREADS, p->smem, st>>>(p->maps, p->a, p->B); break;
  }
  return cudaGetLastError();
}

cudaError_t launch_attention_tc(const AttnArgs& a, int B, cudaStream_t st) {
  AttnPlan* p = attention_tc_plan_create(a, B);
  if (!p) return cudaErrorInvalidValue;
  cudaError_t e = attention_tc_plan_launch(p, st);
  attention_tc_plan_destroy(p);
  return e;
}

}  // namespace dz
