// tcgen05 GEMM for sm_100a:  C = epilogue(A * B^T), 16-bit operands (hi/lo planes), fp32 accumulation in TMEM.
//
// Persistent kernel: one CTA per SM walks the 128 x BN output tiles (n fastest, so that the CTAs running
// at the same time share A rows through L2).  Warp roles:
//   warp 0      : TMA producer (one elected lane): A box 128 rows x 64 k, B box BN rows x 64 k, SWIZZLE_128B
//   warp 1      : TMEM allocator + UMMA issuer (one elected lane): 4 x tcgen05.mma (K = 16) per 64-wide k block
//   warps 2..9  : epilogue.  The accumulator is double buffered in TMEM (2 x BN columns) so the epilogue of tile i
//                 overlaps the main loop of tile i+1.  Each epilogue warp owns 32 accumulator rows (its TMEM lane
//                 quarter) and every other 32-column chunk: tcgen05.ld -> registers -> 32x32 transpose through a
//                 private shared-memory patch -> row-wise pass in which a warp touches 128 contiguous bytes of one
//                 output row per instruction (bias / activation / residual / fp32 + 16-bit plane stores), with the
//                 residual loads of 8 rows in flight per warp.
// Pipeline: NSTAGE-deep smem ring with full/empty mbarriers; tcgen05.commit releases a stage back to the
// producer and signals the epilogue.  With npass = 3 the k loop runs three times over
// (A_hi,B_hi), (A_lo,B_hi), (A_hi,B_lo) into the same accumulator.
//
// This kernel replaces the cuBLAS/cuDNN calls behind nn.Linear / nn.Conv1d on the reference hot path
// (reference: diarizen/models/module/wav2vec2/components.py:119 conv1d, :305-306 projection, :374 pos-conv,
//  :455-480 q/k/v/out projections, :805-814 FFN; diarizen/models/module/conformer.py:116-214).
#include <cstdlib>
#include <mutex>
#include <string>

#include "common.cuh"
#include "gemm.h"
#include "gemm_epilogue.cuh"

namespace dz {

static constexpr int BM = 128;
static constexpr int BK = 64;
static constexpr int NUM_EPI_WARPS = 8;
static constexpr int NUM_THREADS = 64 + 32 * NUM_EPI_WARPS;
static constexpr int PATCH_FLOATS = 32 * 36;

template <int BN>
struct TcCfg {
  static constexpr int A_BYTES = BM * BK * 2;
  static constexpr int B_BYTES = BN * BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int NSTAGE = (BN == 256) ? 3 : (BN == 128 ? 5 : 6);
  static constexpr int PATCH_BYTES = NUM_EPI_WARPS * PATCH_FLOATS * 4;
  static constexpr int SMEM = NSTAGE * STAGE_BYTES + PATCH_BYTES + 1024 /*align slack*/ + 256 /*barriers*/;
};

struct TcMaps {
  CUtensorMap a[2];  // hi, lo
  CUtensorMap b[2];
};

struct TileCoord { int m0, n0, g, b; };

DZ_DEVINL TileCoord decode_tile(const GemmDesc& d, int tile, int mt, int nt, int BN) {
  // n (or group) fastest, then m, then batch
  TileCoord c;
  const int ni = tile % nt;
  const int r = tile / nt;
  c.m0 = (r % mt) * BM;
  c.b = r / mt;
  if (d.groups > 1) { c.g = ni; c.n0 = 0; }
  else { c.g = 0; c.n0 = ni * BN; }
  return c;
}

static constexpr int PATCH_LD = 36;  // floats per patch row: 16-byte aligned rows, conflict-free float4 access

DZ_DEVINL float4 act4(float4 v, int act) {
  // one copy of each activation in the instruction stream (the epilogue is instruction-cache sensitive)
  switch (act) {
    case 1: v.x = gelu_erf(v.x); v.y = gelu_erf(v.y); v.z = gelu_erf(v.z); v.w = gelu_erf(v.w); break;
    case 2:
      v.x = __fdividef(v.x, 1.0f + __expf(-v.x)); v.y = __fdividef(v.y, 1.0f + __expf(-v.y));
      v.z = __fdividef(v.z, 1.0f + __expf(-v.z)); v.w = __fdividef(v.w, 1.0f + __expf(-v.w));
      break;
    case 3: v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); break;
    default: break;
  }
  return v;
}

DZ_DEVINL float4 ld_res16(const bf16* rp, long long plane, bool two, int fp16) {
  const uint2 hw = *reinterpret_cast<const uint2*>(rp);
  float4 q;
  q.x = from16(__ushort_as_bfloat16((unsigned short)(hw.x & 0xffff)), fp16);
  q.y = from16(__ushort_as_bfloat16((unsigned short)(hw.x >> 16)), fp16);
  q.z = from16(__ushort_as_bfloat16((unsigned short)(hw.y & 0xffff)), fp16);
  q.w = from16(__ushort_as_bfloat16((unsigned short)(hw.y >> 16)), fp16);
  if (two) {
    const uint2 lw = *reinterpret_cast<const uint2*>(rp + plane);
    q.x += from16(__ushort_as_bfloat16((unsigned short)(lw.x & 0xffff)), fp16);
    q.y += from16(__ushort_as_bfloat16((unsigned short)(lw.x >> 16)), fp16);
    q.z += from16(__ushort_as_bfloat16((unsigned short)(lw.y & 0xffff)), fp16);
    q.w += from16(__ushort_as_bfloat16((unsigned short)(lw.y >> 16)), fp16);
  }
  return q;
}

// Full 32-column chunk (all columns valid and row-major): lane = (row-in-group of 4, 4-column slot); one warp
// instruction covers 4 rows x 128 B.  The fp32 residual rows of the whole chunk are fetched up front (8 x 16 B per lane
// in flight); the row loop itself is kept rolled: code size matters more than loop overhead here.
DZ_DEVINL void epi_rows_fast(const GemmDesc& d, const TileCoord& tc, const float* patch, int lane, int mrow0, int nrows,
                             int ncol0) {
  const int rsub = lane >> 3, c4 = (lane & 7) * 4;
  const int gcol = tc.g * d.group_cols + ncol0 + c4;
  const int fp16 = d.fp16;
  const bool two = d.out_planes > 1;
  float4 res[8];
  const float* resp = d.residual ? d.residual + (long long)tc.b * d.res_bstride + (long long)mrow0 * d.ldr + gcol : nullptr;
  if (resp != nullptr) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int r = 4 * i + rsub;
      res[i] = (r < nrows) ? *reinterpret_cast<const float4*>(resp + r * d.ldr) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
  const bf16* r16 = d.res16 ? (const bf16*)d.res16 + (long long)tc.b * d.res16_bstride +
                                  (long long)(mrow0 + d.res16_row_off) * d.ldr16 + gcol
                            : nullptr;
  float4 bias = make_float4(0.f, 0.f, 0.f, 0.f);
  if (d.bias != nullptr) bias = __ldg(reinterpret_cast<const float4*>(d.bias + gcol));
  float* outp = d.out_f32 ? d.out_f32 + (long long)tc.b * d.of_bstride + (long long)mrow0 * d.ldo + gcol : nullptr;
  bf16* bfp = d.out_bf ? (bf16*)d.out_bf + (long long)tc.b * d.ob_bstride + (long long)(mrow0 + d.out_row_off) * d.ldob + gcol
                       : nullptr;
  const float alpha = d.alpha;
  const int act = d.act;
  const bool after = d.act_after_res != 0;
#pragma unroll 1
  for (int i = 0; i < 8; ++i) {
    const int r = 4 * i + rsub;
    if (r >= nrows) break;
    float4 v = *reinterpret_cast<const float4*>(patch + r * PATCH_LD + c4);
    v.x += bias.x; v.y += bias.y; v.z += bias.z; v.w += bias.w;
    if (!after) v = act4(v, act);
    v.x *= alpha; v.y *= alpha; v.z *= alpha; v.w *= alpha;
    if (resp != nullptr) {
      // res[] is indexed with a loop-variant subscript: keep it in registers through a uniform select chain
      float4 q = res[0];
#pragma unroll
      for (int j = 1; j < 8; ++j) if (i == j) q = res[j];
      v.x += q.x; v.y += q.y; v.z += q.z; v.w += q.w;
    } else if (r16 != nullptr) {
      const float4 q = ld_res16(r16 + r * d.ldr16, d.res16_plane, two, fp16);
      v.x += q.x; v.y += q.y; v.z += q.z; v.w += q.w;
    }
    if (after) v = act4(v, act);
    if (outp != nullptr) *reinterpret_cast<float4*>(outp + r * d.ldo) = v;
    if (bfp != nullptr) {
      bf16 h0, h1, h2, h3, l0, l1, l2, l3;
      split_bf16(v.x, h0, l0, fp16); split_bf16(v.y, h1, l1, fp16);
      split_bf16(v.z, h2, l2, fp16); split_bf16(v.w, h3, l3, fp16);
      uint2 hw;
      hw.x = (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
      hw.y = (uint32_t)__bfloat16_as_ushort(h2) | ((uint32_t)__bfloat16_as_ushort(h3) << 16);
      *reinterpret_cast<uint2*>(bfp + r * d.ldob) = hw;
      if (two) {
        uint2 lw;
        lw.x = (uint32_t)__bfloat16_as_ushort(l0) | ((uint32_t)__bfloat16_as_ushort(l1) << 16);
        lw.y = (uint32_t)__bfloat16_as_ushort(l2) | ((uint32_t)__bfloat16_as_ushort(l3) << 16);
        *reinterpret_cast<uint2*>(bfp + d.ob_plane + r * d.ldob) = lw;
      }
    }
  }
}

// Edge chunk (crosses N, tr_col0 or the zero-pad boundary): element-wise, lane = column.
__device__ __noinline__ void epi_rows_edge(const GemmDesc& d, const TileCoord& tc, const float* patch, int lane, int mrow0,
                                           int nrows, int ncol0, int rm_cols) {
  const int n = ncol0 + lane;
  const int gcol = tc.g * d.group_cols + n;
  const float bias_v = (d.bias != nullptr && n < d.N) ? __ldg(d.bias + gcol) : 0.f;
  for (int r = 0; r < nrows; ++r) {
    const int m = mrow0 + r;
    if (n < d.N) {
      float resv = 0.f;
      if (d.residual != nullptr) resv = d.residual[(long long)tc.b * d.res_bstride + (long long)m * d.ldr + gcol];
      else if (d.res16 != nullptr) {
        const bf16* rp = (const bf16*)d.res16 + (long long)tc.b * d.res16_bstride + (long long)(m + d.res16_row_off) * d.ldr16 + gcol;
        resv = from16(*rp, d.fp16);
        if (d.out_planes > 1) resv += from16(rp[d.res16_plane], d.fp16);
      }
      const float pre = patch[r * PATCH_LD + lane] + bias_v;
      const float v = d.act_after_res ? apply_act(d.alpha * pre + resv, d.act) : d.alpha * apply_act(pre, d.act) + resv;
      if (d.out_f32 != nullptr) d.out_f32[(long long)tc.b * d.of_bstride + (long long)m * d.ldo + gcol] = v;
      if (d.out_bf != nullptr && n < rm_cols) {
        bf16 h, l;
        split_bf16(v, h, l, d.fp16);
        bf16* hp = (bf16*)d.out_bf + (long long)tc.b * d.ob_bstride + (long long)(m + d.out_row_off) * d.ldob + gcol;
        *hp = h;
        if (d.out_planes > 1) hp[d.ob_plane] = l;
      }
    } else if (d.out_bf != nullptr && n < d.zero_pad_to && d.out_t == nullptr) {
      bf16* hp = (bf16*)d.out_bf + (long long)tc.b * d.ob_bstride + (long long)(m + d.out_row_off) * d.ldob + gcol;
      *hp = __float2bfloat16_rn(0.0f);
      if (d.out_planes > 1) hp[d.ob_plane] = __float2bfloat16_rn(0.0f);
    }
  }
}

template <int BN>
__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_tc_kernel(const __grid_constant__ TcMaps maps, const GemmDesc d, const int a_rank5, const int mt, const int nt,
               const int ntiles) {
  using C = TcCfg<BN>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_align1024(smem_raw);
  float* patches = reinterpret_cast<float*>(smem + C::NSTAGE * C::STAGE_BYTES);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + C::NSTAGE * C::STAGE_BYTES + C::PATCH_BYTES);
  uint64_t* empty_bar = full_bar + C::NSTAGE;
  uint64_t* tmem_full = empty_bar + C::NSTAGE;   // [2]
  uint64_t* tmem_empty = tmem_full + 2;          // [2]
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const bool conv2d = d.conv_runs > 0;
  const int kbpr = conv2d ? (d.conv_run_len + BK - 1) / BK : 0;   // k blocks per input row (conv2d)
  const int kblocks = conv2d ? d.conv_runs * kbpr : (d.K + BK - 1) / BK;
  const int iters = kblocks * d.npass;

  if (threadIdx.x == 0) {
    for (int s = 0; s < C::NSTAGE; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(&tmem_full[0], 1); mbar_init(&tmem_full[1], 1);
    mbar_init(&tmem_empty[0], NUM_EPI_WARPS); mbar_init(&tmem_empty[1], NUM_EPI_WARPS);
    mbar_fence_init();
    tma_prefetch_desc(&maps.a[0]);
    tma_prefetch_desc(&maps.b[0]);
  }
  if (warp == 1) tmem_alloc(tmem_ptr, 2 * BN);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    if (lane == 0) {
      int gi = 0;  // global k-iteration counter (ring position)
      for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const TileCoord tc = decode_tile(d, tile, mt, nt, BN);
        for (int it = 0; it < iters; ++it, ++gi) {
          const int s = gi % C::NSTAGE;
          const uint32_t ph = (gi / C::NSTAGE) & 1;
          const int pass = it / kblocks;
          const int kb = it - pass * kblocks;
          mbar_wait(&empty_bar[s], ph ^ 1);
          uint8_t* sa = smem + s * C::STAGE_BYTES;
          uint8_t* sb = sa + C::A_BYTES;
          mbar_expect_tx(&full_bar[s], C::STAGE_BYTES);
          const CUtensorMap* ma = &maps.a[pass == 1 ? 1 : 0];
          const CUtensorMap* mb = &maps.b[pass == 2 ? 1 : 0];
          if (conv2d) {
            // (x in padded row, wo, h, image): tap row `run` of output row ho reads input row hs*ho + h0 + run
            const int run = kb / kbpr, kbr = kb - run * kbpr;
            const int img = tc.b / d.conv_Ho, ho = tc.b - img * d.conv_Ho;
            tma_load_4d(sa, ma, &full_bar[s], d.conv_x0 + kbr * BK, tc.m0, d.conv_hs * ho + d.conv_h0 + run, img);
          } else if (a_rank5) {
            // (k_inner, k_outer, row, group, batch): one k block = one run of a_kinner (=64) elements
            tma_load_5d(sa, ma, &full_bar[s], 0, kb, tc.m0, tc.g, tc.b);
          } else {
            tma_load_3d(sa, ma, &full_bar[s], kb * BK, tc.m0, tc.b);
          }
          tma_load_3d(sb, mb, &full_bar[s], kb * BK, tc.n0, tc.g);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      int gi = 0, tcount = 0;
      for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++tcount) {
        const TileCoord tc = decode_tile(d, tile, mt, nt, BN);
        const int n_valid = min(BN, d.N - tc.n0);
        const uint32_t umma_n = (uint32_t)((n_valid + 15) & ~15);
        const uint32_t idesc = umma_idesc_bf16(BM, umma_n, d.fp16);
        const int acc = tcount & 1;
        const uint32_t tmem_acc = tmem_base + (uint32_t)(acc * BN);
        mbar_wait(&tmem_empty[acc], ((tcount >> 1) & 1) ^ 1);
        tc_fence_after();
        for (int it = 0; it < iters; ++it, ++gi) {
          const int s = gi % C::NSTAGE;
          const uint32_t ph = (gi / C::NSTAGE) & 1;
          const int kb = it % kblocks;
          mbar_wait(&full_bar[s], ph);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + s * C::STAGE_BYTES);
          const uint32_t sb = sa + C::A_BYTES;
          const int krem = conv2d ? d.conv_run_len - (kb % kbpr) * BK : d.K - kb * BK;
          const int ksteps = krem >= BK ? (BK / 16) : ((krem + 15) / 16);
          for (int k = 0; k < ksteps; ++k) {
            const uint64_t adesc = umma_desc_sw128(sa + k * 32);
            const uint64_t bdesc = umma_desc_sw128(sb + k * 32);
            umma_bf16(tmem_acc, adesc, bdesc, idesc, (it > 0 || k > 0) ? 1u : 0u);
          }
          umma_commit(&empty_bar[s]);
        }
        umma_commit(&tmem_full[acc]);
      }
    }
  } else {
    // ---------------- epilogue warps ----------------
    const int ew = warp - 2;         // 0..7
    const int quad = warp & 3;       // TMEM lane quarter this warp may read
    const int half = ew >> 2;        // which alternate 32-column chunks this warp takes
    float* patch = patches + ew * PATCH_FLOATS;
    const int rm_cols = (d.out_t != nullptr) ? d.tr_col0 : d.N;
    int tcount = 0;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++tcount) {
      const TileCoord tc = decode_tile(d, tile, mt, nt, BN);
      const int acc = tcount & 1;
      const uint32_t tmem_acc = tmem_base + (uint32_t)(acc * BN) + ((uint32_t)(quad * 32) << 16);
      const int n_valid = min(BN, d.N - tc.n0);
      const int n_store = max(n_valid, min(BN, d.zero_pad_to - tc.n0));
      const int mrow0 = tc.m0 + quad * 32;
      mbar_wait(&tmem_full[acc], (tcount >> 1) & 1);
      tc_fence_after();
#pragma unroll 1
      for (int c = half * 32; c < n_store; c += 64) {
        uint32_t r[32];
        tmem_ld_32x32(tmem_acc + (uint32_t)c, r);
        tmem_ld_wait();
        const int ncol0 = tc.n0 + c;
        // 32x32 transpose buffer: thread (= accumulator row) writes its 32 columns
        {
          float4* prow = reinterpret_cast<float4*>(patch + lane * PATCH_LD);
#pragma unroll
          for (int j = 0; j < 8; ++j)
            prow[j] = make_float4(__uint_as_float(r[4 * j]), __uint_as_float(r[4 * j + 1]), __uint_as_float(r[4 * j + 2]),
                                  __uint_as_float(r[4 * j + 3]));
        }
        __syncwarp();
        const int nrows = min(32, d.M - mrow0);
        // transposed outputs (v^T): lane <-> row so that consecutive lanes write consecutive frames of one feature
        if (d.out_t != nullptr && ncol0 + 32 > d.tr_col0 && lane < nrows) {
          const int m = mrow0 + lane;
          const int sb = m / d.seq_len, st = m - sb * d.seq_len;
          bf16* tp = (bf16*)d.out_t + (long long)sb * d.ot_bstride + st;
          const float* prow = patch + lane * PATCH_LD;
#pragma unroll 1
          for (int j = 0; j < 32; ++j) {
            const int n = ncol0 + j;
            if (n < d.tr_col0 || n >= d.N) continue;
            float v = prow[j];
            if (d.bias != nullptr) v += __ldg(d.bias + tc.g * d.group_cols + n);
            v = d.alpha * apply_act(v, d.act);
            bf16 h, l;
            split_bf16(v, h, l, d.fp16);
            bf16* q = tp + (long long)(n - d.tr_col0) * d.ldt;
            *q = h;
            if (d.out_planes > 1) q[d.ot_plane] = l;
          }
        }
        // row-major outputs: 4 rows x 128 B per warp instruction
        if (ncol0 < max(rm_cols, d.zero_pad_to) || d.out_f32 != nullptr) {
          if (ncol0 + 32 <= rm_cols) epi_rows_fast(d, tc, patch, lane, mrow0, nrows, ncol0);
          else epi_rows_edge(d, tc, patch, lane, mrow0, nrows, ncol0, rm_cols);
        }
        __syncwarp();
      }
      // all TMEM reads of this accumulator are complete: hand it back to the MMA warp
      tc_fence_before();
      if (lane == 0) mbar_arrive(&tmem_empty[acc]);
    }
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 2 * BN);
  }
}

// ================================================================================================
// TMA-epilogue variant.  Same producer / MMA warps; 4 epilogue warps (one per TMEM lane quarter) work in the
// accumulator's native thread-per-row layout: tcgen05.ld 16 columns -> bias / activation / residual in registers ->
// 16-byte stores into a 128-byte-swizzled shared-memory patch -> one cp.async.bulk.tensor store per 32-row x 128-byte
// sub-tile.  Residual sub-tiles (fp32, or 16-bit planes for the ResNet shortcut) arrive through TMA loads issued one
// span ahead.  No per-element global address arithmetic, no transposition; out-of-range rows / columns are clipped by
// the tensor maps.  mode 0: fp32 output (span = 32 columns); mode 1: 16-bit plane output (span = 64 columns).
// ================================================================================================
struct EpiMaps { CUtensorMap res, res_lo, out, out_lo; };
static constexpr int NUM_EPI2 = 8;                       // two epilogue warps per TMEM lane quarter, alternating spans
static constexpr int NUM_THREADS2 = 64 + 32 * NUM_EPI2;
static constexpr int PATCH2_BYTES = 8192;                // per epilogue warp: 2 x 4 KB (double buffer, or hi|lo planes)

// DEEP (BN = 256 only): a 4th ring stage paid for with single 4 KB store patches.  The ncu captures of round 2 show the
// 16-bit-output GEMMs (QKV, FFN-up, conv stack) with the tensor pipe 23-35 % active and neither DRAM nor issue slots busy:
// with ~1 us of L2 latency the bytes in flight (3 x 48 KB) set the pace, so ring depth is worth more than a double-buffered
// store patch there.  Residual GEMMs keep the double-buffered patches (their residual tiles are prefetched into them).
template <int BN, int DEEP = 0>
struct TcCfg2 {
  static constexpr int STAGE_BYTES = BM * BK * 2 + BN * BK * 2;
  // BN = 64 (narrow outputs: ResNet layer 1/2, conv stack): 4 stages so that two CTAs fit per SM - with so little work
  // per tile, tiles in flight matter more than ring depth.
  static constexpr int NSTAGE = (BN == 128) ? 5 : (DEEP ? 4 : 3);
  static constexpr int PATCH = (BN == 64 || DEEP) ? 4096 : PATCH2_BYTES;   // single 4 KB patch per warp
  static constexpr int SMEM = NSTAGE * STAGE_BYTES + NUM_EPI2 * PATCH + 1024 + 256;
  static constexpr int MIN_CTAS = (BN == 64) ? 2 : 1;
};

DZ_DEVINL float4 unpack4(uint2 w, int fp16) {
  float4 q;
  q.x = from16(__ushort_as_bfloat16((unsigned short)(w.x & 0xffff)), fp16);
  q.y = from16(__ushort_as_bfloat16((unsigned short)(w.x >> 16)), fp16);
  q.z = from16(__ushort_as_bfloat16((unsigned short)(w.y & 0xffff)), fp16);
  q.w = from16(__ushort_as_bfloat16((unsigned short)(w.y >> 16)), fp16);
  return q;
}

// One 32-column group of one accumulator row -> 16-bit (hi [+ lo]) cells of the swizzled store patch; the 16-bit residual
// (TMA-prefetched into the same cells) is added first.  FP16 / TWO are compile-time so that the per-element conversions
// carry no branches (a uniform run-time flag still costs a branch per element once the loop is unrolled).
template <int FP16, int TWO>
DZ_DEVINL void epi_store16(uint8_t* prow, int g, int sw, const float* v, bool has_res, bool relu_after, int nrem) {
#pragma unroll
  for (int h = 0; h < 4; ++h) {   // 4 x 16-byte chunks of 8 columns; chunk index within the 64-column row = 4g + h
    uint4* chi = reinterpret_cast<uint4*>(prow + (((4 * g + h) ^ sw) << 4));
    uint4* clo = reinterpret_cast<uint4*>(prow + 4096 + (((4 * g + h) ^ sw) << 4));
    float e[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) e[c] = v[8 * h + c];
    if (has_res) {
      const uint4 rh = *chi;
      float4 r0 = unpack4(make_uint2(rh.x, rh.y), FP16), r1 = unpack4(make_uint2(rh.z, rh.w), FP16);
      if (TWO) {
        const uint4 rl = *clo;
        const float4 l0 = unpack4(make_uint2(rl.x, rl.y), FP16), l1 = unpack4(make_uint2(rl.z, rl.w), FP16);
        r0.x += l0.x; r0.y += l0.y; r0.z += l0.z; r0.w += l0.w;
        r1.x += l1.x; r1.y += l1.y; r1.z += l1.z; r1.w += l1.w;
      }
      e[0] += r0.x; e[1] += r0.y; e[2] += r0.z; e[3] += r0.w; e[4] += r1.x; e[5] += r1.y; e[6] += r1.z; e[7] += r1.w;
    }
    uint32_t hw[4], lw[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      float x0 = e[2 * c], x1 = e[2 * c + 1];
      if (relu_after) { x0 = fmaxf(x0, 0.f); x1 = fmaxf(x1, 0.f); }
      if (8 * h + 2 * c >= nrem) x0 = 0.f;
      if (8 * h + 2 * c + 1 >= nrem) x1 = 0.f;
      if (TWO) {
        bf16 h0, l0, h1, l1;
        split_bf16(x0, h0, l0, FP16);
        split_bf16(x1, h1, l1, FP16);
        hw[c] = (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
        lw[c] = (uint32_t)__bfloat16_as_ushort(l0) | ((uint32_t)__bfloat16_as_ushort(l1) << 16);
      } else {
        hw[c] = pack2_16<FP16>(x0, x1);
      }
    }
    *chi = make_uint4(hw[0], hw[1], hw[2], hw[3]);
    if (TWO) *clo = make_uint4(lw[0], lw[1], lw[2], lw[3]);
  }
}

// bias + pre-residual activation + scale on 32 accumulator columns held in registers (one code block per activation)
template <int ACT>
DZ_DEVINL void epi_math32(float (&v)[32], const float* __restrict__ bias, float alpha) {
  if (bias != nullptr) {
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const float4 bq = __ldg(reinterpret_cast<const float4*>(bias) + q);
      v[4 * q] += bq.x; v[4 * q + 1] += bq.y; v[4 * q + 2] += bq.z; v[4 * q + 3] += bq.w;
    }
  }
#pragma unroll
  for (int j = 0; j < 32; ++j) {
    float x = v[j];
    if (ACT == 1) x = gelu_erf(x);
    if (ACT == 2) x = __fdividef(x, 1.0f + __expf(-x));
    if (ACT == 3) x = fmaxf(x, 0.f);
    v[j] = x * alpha;
  }
}

template <int BN, int DEEP = 0>
__global__ void __launch_bounds__(NUM_THREADS2, (BN == 64) ? 2 : 1)
gemm_tc_tma_kernel(const __grid_constant__ TcMaps maps, const __grid_constant__ EpiMaps em, const GemmDesc d, const int a_rank5,
                   const int mt, const int nt, const int ntiles, const int mode) {
  using C = TcCfg2<BN, DEEP>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_align1024(smem_raw);
  uint8_t* patches = smem + C::NSTAGE * C::STAGE_BYTES;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(patches + NUM_EPI2 * C::PATCH);
  uint64_t* empty_bar = full_bar + C::NSTAGE;
  uint64_t* tmem_full = empty_bar + C::NSTAGE;   // [2]
  uint64_t* tmem_empty = tmem_full + 2;          // [2]
  uint64_t* res_bar = tmem_empty + 2;            // [8 warps][2 buffers]
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(res_bar + 2 * NUM_EPI2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const bool conv2d = d.conv_runs > 0;
  const int kbpr = conv2d ? (d.conv_run_len + BK - 1) / BK : 0;
  const int kblocks = conv2d ? d.conv_runs * kbpr : (d.K + BK - 1) / BK;
  const int iters = kblocks * d.npass;
  constexpr int A_BYTES = BM * BK * 2;

  if (threadIdx.x == 0) {
    for (int s = 0; s < C::NSTAGE; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    mbar_init(&tmem_full[0], 1); mbar_init(&tmem_full[1], 1);
    mbar_init(&tmem_empty[0], NUM_EPI2); mbar_init(&tmem_empty[1], NUM_EPI2);
    for (int i = 0; i < 2 * NUM_EPI2; ++i) mbar_init(&res_bar[i], 1);
    mbar_fence_init();
    tma_prefetch_desc(&maps.a[0]); tma_prefetch_desc(&maps.b[0]); tma_prefetch_desc(&em.out);
  }
  if (warp == 1) tmem_alloc(tmem_ptr, 2 * BN);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    if (lane == 0) {
      int gi = 0;
      for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const TileCoord tc = decode_tile(d, tile, mt, nt, BN);
        for (int it = 0; it < iters; ++it, ++gi) {
          const int s = gi % C::NSTAGE;
          const uint32_t ph = (gi / C::NSTAGE) & 1;
          const int pass = it / kblocks;
          const int kb = it - pass * kblocks;
          mbar_wait(&empty_bar[s], ph ^ 1);
          uint8_t* sa = smem + s * C::STAGE_BYTES;
          uint8_t* sb = sa + A_BYTES;
          mbar_expect_tx(&full_bar[s], C::STAGE_BYTES);
          const CUtensorMap* ma = &maps.a[pass == 1 ? 1 : 0];
          const CUtensorMap* mb = &maps.b[pass == 2 ? 1 : 0];
          if (conv2d) {
            const int run = kb / kbpr, kbr = kb - run * kbpr;
            const int img = tc.b / d.conv_Ho, ho = tc.b - img * d.conv_Ho;
            tma_load_4d(sa, ma, &full_bar[s], d.conv_x0 + kbr * BK, tc.m0, d.conv_hs * ho + d.conv_h0 + run, img);
          } else if (a_rank5) {
            tma_load_5d(sa, ma, &full_bar[s], 0, kb, tc.m0, tc.g, tc.b);
          } else {
            tma_load_3d(sa, ma, &full_bar[s], kb * BK, tc.m0, tc.b);
          }
          tma_load_3d(sb, mb, &full_bar[s], kb * BK, tc.n0, tc.g);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      int gi = 0, tcount = 0;
      for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++tcount) {
        const TileCoord tc = decode_tile(d, tile, mt, nt, BN);
        const int n_valid = min(BN, d.N - tc.n0);
        const uint32_t idesc = umma_idesc_bf16(BM, (uint32_t)((n_valid + 15) & ~15), d.fp16);
        const int acc = tcount & 1;
        const uint32_t tmem_acc = tmem_base + (uint32_t)(acc * BN);
        mbar_wait(&tmem_empty[acc], ((tcount >> 1) & 1) ^ 1);
        tc_fence_after();
        for (int it = 0; it < iters; ++it, ++gi) {
          const int s = gi % C::NSTAGE;
          const uint32_t ph = (gi / C::NSTAGE) & 1;
          const int kb = it % kblocks;
          mbar_wait(&full_bar[s], ph);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + s * C::STAGE_BYTES);
          const uint32_t sb = sa + A_BYTES;
          const int krem = conv2d ? d.conv_run_len - (kb % kbpr) * BK : d.K - kb * BK;
          const int ksteps = krem >= BK ? (BK / 16) : ((krem + 15) / 16);
          for (int k = 0; k < ksteps; ++k)
            umma_bf16(tmem_acc, umma_desc_sw128(sa + k * 32), umma_desc_sw128(sb + k * 32), idesc, (it > 0 || k > 0) ? 1u : 0u);
          umma_commit(&empty_bar[s]);
        }
        umma_commit(&tmem_full[acc]);
      }
    }
  } else {
    // ---------------- epilogue warps: thread <-> accumulator row; warps (quad, par) take spans s = par (mod 2) ----------------
    const int ew = warp - 2;          // 0..7
    const int quad = warp & 3;        // TMEM lane quarter
    const int par = ew >> 2;          // span parity served by this warp
    uint8_t* pw = patches + ew * C::PATCH;
    uint64_t* rb = res_bar + ew * 2;
    const int SW = mode ? 64 : 32;
    const bool two = d.out_planes > 1;
    const bool has_res = mode ? (d.res16 != nullptr) : (d.residual != nullptr);
    // double-buffered patches unless both planes are needed (hi | lo share the 8 KB) or the patch is the 4 KB one
    const bool dbl = (C::PATCH == PATCH2_BYTES) && !(mode && two);
    const int fp16 = d.fp16;
    const int sw = lane & 7;
    const bool relu_after = d.act_after_res && d.act == 3;
    const int pre_act = d.act_after_res ? 0 : d.act;
    const uint32_t res_bytes = (mode && two) ? 8192u : 4096u;
    const int ncols_out = mode ? max(d.N, d.zero_pad_to) : d.N;
    uint32_t sc = 0;               // spans processed by this warp
    uint32_t use0 = 0, use1 = 0;   // residual loads consumed per buffer (mbarrier phase)
    int tcount = 0;
    auto issue_res = [&](const TileCoord& tc, int col0, int buf) {
      uint8_t* dst = pw + (dbl ? buf * 4096 : 0);
      mbar_expect_tx(&rb[buf], res_bytes);
      const int row0 = tc.m0 + quad * 32 + (mode ? d.res16_row_off : 0);
      tma_load_3d(dst, &em.res, &rb[buf], tc.g * d.group_cols + col0, row0, tc.b);
      if (mode && two) tma_load_3d(dst + 4096, &em.res_lo, &rb[buf], tc.g * d.group_cols + col0, row0, tc.b);
    };
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++tcount) {
      const TileCoord tc = decode_tile(d, tile, mt, nt, BN);
      const int acc = tcount & 1;
      const uint32_t tmem_acc = tmem_base + (uint32_t)(acc * BN) + ((uint32_t)(quad * 32) << 16);
      const int n_store = min(BN, ncols_out - tc.n0);
      const int nspans = (n_store + SW - 1) / SW;
      if (has_res && dbl && lane == 0 && par < nspans) {
        bulk_wait_read<0>();
        issue_res(tc, tc.n0 + par * SW, (int)(sc & 1));
      }
      mbar_wait(&tmem_full[acc], (tcount >> 1) & 1);
      tc_fence_after();
      // Row LayerNorm fused into the epilogue (conv stack of the layer-norm extractor: components.py:119-122): the tile spans
      // the whole output row (N <= BN) and a thread owns one accumulator row, so mean and variance are two thread-local
      // sweeps over its TMEM lane; both warps of a lane quarter compute them (TMEM reads are cheap) and normalise their own spans.
      float ln_mean = 0.f, ln_rstd = 1.f;
      if (d.ln_gamma != nullptr) {
        const int ngrp = (d.N + 31) >> 5;
        float sum = 0.f;
#pragma unroll 1
        for (int g = 0; g < ngrp; ++g) {
          uint32_t r[32];
          tmem_ld_32x32(tmem_acc + (uint32_t)(g * 32), r);
          tmem_ld_wait();
          const int nrem = d.N - g * 32;
          if (nrem >= 32) {
            float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
            for (int j = 0; j < 32; j += 4) { s0 += __uint_as_float(r[j]); s1 += __uint_as_float(r[j + 1]); s2 += __uint_as_float(r[j + 2]); s3 += __uint_as_float(r[j + 3]); }
            sum += (s0 + s1) + (s2 + s3);
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) sum += (j < nrem) ? __uint_as_float(r[j]) : 0.f;
          }
        }
        ln_mean = sum / (float)d.N;
        float ssq = 0.f;
#pragma unroll 1
        for (int g = 0; g < ngrp; ++g) {
          uint32_t r[32];
          tmem_ld_32x32(tmem_acc + (uint32_t)(g * 32), r);
          tmem_ld_wait();
          const int nrem = d.N - g * 32;
          if (nrem >= 32) {
            float q0 = 0.f, q1 = 0.f, q2 = 0.f, q3 = 0.f;
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              const float c0 = __uint_as_float(r[j]) - ln_mean, c1 = __uint_as_float(r[j + 1]) - ln_mean;
              const float c2 = __uint_as_float(r[j + 2]) - ln_mean, c3 = __uint_as_float(r[j + 3]) - ln_mean;
              q0 = fmaf(c0, c0, q0); q1 = fmaf(c1, c1, q1); q2 = fmaf(c2, c2, q2); q3 = fmaf(c3, c3, q3);
            }
            ssq += (q0 + q1) + (q2 + q3);
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) { const float c = __uint_as_float(r[j]) - ln_mean; ssq += (j < nrem) ? c * c : 0.f; }
          }
        }
        ln_rstd = rsqrtf(ssq / (float)d.N + d.ln_eps);
      }
#pragma unroll 1
      for (int s = par; s < nspans; s += 2, ++sc) {
        const int buf = dbl ? (int)(sc & 1) : 0;
        const int col0 = tc.n0 + s * SW;
        if (lane == 0) {
          if (has_res && dbl) {
            if (s + 2 < nspans) { bulk_wait_read<0>(); issue_res(tc, col0 + 2 * SW, buf ^ 1); }
          } else if (has_res) {
            bulk_wait_read<0>();
            issue_res(tc, col0, 0);
          } else if (dbl) {
            bulk_wait_read<1>();   // the store issued two spans ago from this patch has finished reading shared memory
          } else {
            bulk_wait_read<0>();
          }
        }
        __syncwarp();
        if (has_res) {
          const uint32_t u = buf ? use1 : use0;
          mbar_wait(&rb[buf], u & 1);
          if (buf) ++use1; else ++use0;
        }
        uint8_t* prow = pw + (dbl ? buf * 4096 : 0) + lane * 128;
#pragma unroll 1
        for (int g = 0; g < SW / 32; ++g) {
          uint32_t r[32];
          tmem_ld_32x32(tmem_acc + (uint32_t)(s * SW + g * 32), r);
          const int gcol = tc.g * d.group_cols + col0 + g * 32;
          const float* bp = d.bias ? d.bias + gcol : nullptr;
          tmem_ld_wait();
          float v[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
          if (d.ln_gamma != nullptr) {
            // gamma / beta are readable (zero padded) up to the next multiple of 32 columns: vector loads, no predicates
            const float4* gp = reinterpret_cast<const float4*>(d.ln_gamma + gcol);
            const float4* bq = reinterpret_cast<const float4*>(d.ln_beta + gcol);
            const float off = -ln_mean * ln_rstd;
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              const float4 ga = __ldg(gp + q), be = __ldg(bq + q);
              v[4 * q] = fmaf(fmaf(v[4 * q], ln_rstd, off), ga.x, be.x);
              v[4 * q + 1] = fmaf(fmaf(v[4 * q + 1], ln_rstd, off), ga.y, be.y);
              v[4 * q + 2] = fmaf(fmaf(v[4 * q + 2], ln_rstd, off), ga.z, be.z);
              v[4 * q + 3] = fmaf(fmaf(v[4 * q + 3], ln_rstd, off), ga.w, be.w);
            }
          }
          switch (pre_act) {
            case 1: epi_math32<1>(v, bp, d.alpha); break;
            case 2: epi_math32<2>(v, bp, d.alpha); break;
            case 3: epi_math32<3>(v, bp, d.alpha); break;
            default: epi_math32<0>(v, bp, d.alpha); break;
          }
          const int nrem = d.N - (col0 + g * 32);   // valid columns in this group (may be >= 32 or <= 0)
          if (mode == 0) {
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              float4* cell = reinterpret_cast<float4*>(prow + ((q ^ sw) << 4));
              float4 o = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
              if (has_res) { const float4 rq = *cell; o.x += rq.x; o.y += rq.y; o.z += rq.z; o.w += rq.w; }
              if (relu_after) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
              if (4 * q + 3 >= nrem) {
                if (4 * q >= nrem) o.x = 0.f;
                if (4 * q + 1 >= nrem) o.y = 0.f;
                if (4 * q + 2 >= nrem) o.z = 0.f;
                if (4 * q + 3 >= nrem) o.w = 0.f;
              }
              *cell = o;
            }
          } else {
            const int variant = (fp16 ? 1 : 0) | (two ? 2 : 0);
            switch (variant) {
              case 0: epi_store16<0, 0>(prow, g, sw, v, has_res, relu_after, nrem); break;
              case 1: epi_store16<1, 0>(prow, g, sw, v, has_res, relu_after, nrem); break;
              case 2: epi_store16<0, 1>(prow, g, sw, v, has_res, relu_after, nrem); break;
              default: epi_store16<1, 1>(prow, g, sw, v, has_res, relu_after, nrem); break;
            }
          }
        }
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
          const int row0 = tc.m0 + quad * 32;
          const uint8_t* src = pw + (dbl ? buf * 4096 : 0);
          tma_store_3d(&em.out, src, tc.g * d.group_cols + col0, row0, tc.b);
          if (mode && two) tma_store_3d(&em.out_lo, src + 4096, tc.g * d.group_cols + col0, row0, tc.b);
          bulk_commit();
        }
      }
      tc_fence_before();
      if (lane == 0) mbar_arrive(&tmem_empty[acc]);
    }
    if (lane == 0) bulk_wait_all<0>();   // all stores complete before the CTA (and its shared memory) goes away
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 2 * BN);
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static thread_local std::string g_err;
const char* gemm_last_error() { return g_err.c_str(); }

static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

static bool make_tmap_any(CUtensorMap* out, const void* base, int esize, int rank, const uint64_t* dims,
                          const uint64_t* strides_elems, const uint32_t* box) {
  EncodeTiledFn enc = get_encode();
  if (!enc) { g_err = "cuTensorMapEncodeTiled entry point unavailable"; return false; }
  cuuint64_t gdim[5], gstr[4];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) {
    gdim[i] = dims[i]; bx[i] = box[i]; es[i] = 1;
    if (i > 0) {
      gstr[i - 1] = strides_elems[i] * (uint64_t)esize;
      if (gstr[i - 1] % 16 != 0) { g_err = "tensor map stride not a multiple of 16 bytes"; return false; }
    }
  }
  if (reinterpret_cast<uintptr_t>(base) % 16 != 0) { g_err = "tensor map base not 16-byte aligned"; return false; }
  CUresult r = enc(out, esize == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank,
                   const_cast<void*>(base), gdim, gstr, bx, es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { g_err = "cuTensorMapEncodeTiled failed with code " + std::to_string((int)r); return false; }
  return true;
}

bool make_tmap_bf16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_elems,
                    const uint32_t* box) {
  EncodeTiledFn enc = get_encode();
  if (!enc) { g_err = "cuTensorMapEncodeTiled entry point unavailable"; return false; }
  cuuint64_t gdim[5], gstr[4];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) {
    gdim[i] = dims[i];
    bx[i] = box[i];
    es[i] = 1;
    if (i > 0) {
      gstr[i - 1] = strides_elems[i] * 2;
      if (gstr[i - 1] % 16 != 0) { g_err = "tensor map stride not a multiple of 16 bytes"; return false; }
    }
  }
  if (reinterpret_cast<uintptr_t>(base) % 16 != 0) { g_err = "tensor map base not 16-byte aligned"; return false; }
  CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), gdim, gstr, bx, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    g_err = "cuTensorMapEncodeTiled failed with code " + std::to_string((int)r);
    return false;
  }
  return true;
}

// 16-bit tensor map with a selectable swizzle span (32 / 64 / 128 bytes); used by the small-channel convolution kernel
bool make_tmap_sw(CUtensorMap* out, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_elems,
                  const uint32_t* box, int swizzle_bytes) {
  EncodeTiledFn enc = get_encode();
  if (!enc) { g_err = "cuTensorMapEncodeTiled entry point unavailable"; return false; }
  cuuint64_t gdim[5], gstr[4];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) {
    gdim[i] = dims[i];
    bx[i] = box[i];
    es[i] = 1;
    if (i > 0) {
      gstr[i - 1] = strides_elems[i] * 2;
      if (gstr[i - 1] % 16 != 0) { g_err = "tensor map stride not a multiple of 16 bytes"; return false; }
    }
  }
  if (reinterpret_cast<uintptr_t>(base) % 16 != 0) { g_err = "tensor map base not 16-byte aligned"; return false; }
  const CUtensorMapSwizzle sw = swizzle_bytes == 32 ? CU_TENSOR_MAP_SWIZZLE_32B
                                : swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B;
  CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), gdim, gstr, bx, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    g_err = "cuTensorMapEncodeTiled failed with code " + std::to_string((int)r);
    return false;
  }
  return true;
}

struct GemmPlan {
  GemmDesc d;
  TcMaps maps;
  int bn = 128;
  int rank5 = 0;
  int mt = 0, nt = 0, ntiles = 0;
  dim3 grid;
  int tma_epi = 0;   // 1: gemm_tc_tma_kernel
  int epi_mode = 0;  // 0 fp32 output, 1 16-bit plane output
  EpiMaps em;
};

static int sm_count() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

template <int BN>
static cudaError_t launch_bn(const GemmPlan* p, cudaStream_t st) {
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(gemm_tc_kernel<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcCfg<BN>::SMEM);
    if (e != cudaSuccess) return e;
    attr_set = true;
  }
  gemm_tc_kernel<BN><<<p->grid, NUM_THREADS, TcCfg<BN>::SMEM, st>>>(p->maps, p->d, p->rank5, p->mt, p->nt, p->ntiles);
  return cudaGetLastError();
}

template <int BN, int DEEP = 0>
static cudaError_t launch_bn_tma(const GemmPlan* p, cudaStream_t st) {
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(gemm_tc_tma_kernel<BN, DEEP>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcCfg2<BN, DEEP>::SMEM);
    if (e != cudaSuccess) return e;
    attr_set = true;
  }
  gemm_tc_tma_kernel<BN, DEEP><<<p->grid, NUM_THREADS2, TcCfg2<BN, DEEP>::SMEM, st>>>(p->maps, p->em, p->d, p->rank5, p->mt, p->nt,
                                                                                      p->ntiles, p->epi_mode);
  return cudaGetLastError();
}

// The TMA epilogue handles: one group, no transposed output, exactly one of (fp32 | 16-bit plane) outputs, a residual of
// the same kind as the output (or none), and an activation after the residual only when it is ReLU (the one it applies
// after the add).  Everything else takes the generic epilogue.
static bool tma_epilogue_eligible(const GemmDesc& d) {
  static const bool off = (getenv("DZ_GEMM_LEGACY_EPILOGUE") != nullptr);
  if (off && d.ln_gamma == nullptr) return false;
  if (d.groups != 1 || d.out_t != nullptr) return false;
  if (d.act_after_res && d.act != 0 && d.act != 3) return false;
  const bool f = d.out_f32 != nullptr, h = d.out_bf != nullptr;
  if (f == h) return false;
  if (f && (d.res16 != nullptr || (d.ldo % 4) != 0 || (d.residual && (d.ldr % 4) != 0))) return false;
  if (h && (d.residual != nullptr || (d.ldob % 8) != 0 || (d.res16 && (d.ldr16 % 8) != 0))) return false;
  return true;
}

static int choose_bn(const GemmDesc& d) {
  if (d.groups > 1 || d.N <= 64) return 64;
  if (d.N <= 128) return 128;
  // prefer the wider tile (less smem traffic per MAC) unless it leaves a mostly empty tail tile
  const int t256 = (d.N + 255) / 256, t128 = (d.N + 127) / 128;
  const long long pad256 = (long long)t256 * 256 - d.N, pad128 = (long long)t128 * 128 - d.N;
  (void)pad128;
  return (pad256 >= 128) ? 128 : 256;
}

GemmPlan* gemm_plan_create(const GemmDesc& d, int force_bn) {
  GemmPlan* p = new GemmPlan();
  p->d = d;
  p->bn = force_bn ? force_bn : choose_bn(d);
  bool want_tma = tma_epilogue_eligible(d);
  if (want_tma && p->bn == 64 && d.out_bf != nullptr && d.out_planes > 1) {
    // the 4 KB patch of the BN = 64 TMA configuration cannot hold hi + lo planes
    if (force_bn == 0) p->bn = 128; else want_tma = false;
  }
  if (d.groups > 1 && d.N > p->bn) { g_err = "grouped GEMM needs N <= BN"; delete p; return nullptr; }
  if (d.ln_gamma != nullptr) {
    // the fused row LayerNorm needs the whole row in one accumulator tile and the register (TMA-store) epilogue
    if (d.N > 128 && force_bn == 0) p->bn = 256;
    if (d.N > p->bn || !want_tma || d.bias != nullptr || d.residual != nullptr || d.res16 != nullptr || d.ln_beta == nullptr || d.act_after_res) {
      g_err = "fused LayerNorm epilogue needs N <= tile width, one plain output, no bias / residual"; delete p; return nullptr;
    }
  }
  if (d.npass != 1 && d.npass != 3) { g_err = "npass must be 1 or 3"; delete p; return nullptr; }
  p->rank5 = (d.conv_runs == 0 && d.a_kinner != d.K) ? 1 : 0;
  const long long rows_alloc = d.a_rows_alloc > 0 ? d.a_rows_alloc : d.M;
  for (int pl = 0; pl < 2; ++pl) {
    const __nv_bfloat16* abase = (const __nv_bfloat16*)d.a + (pl ? d.a_plane : 0);
    const __nv_bfloat16* bbase = (const __nv_bfloat16*)d.b + (pl ? d.b_plane : 0);
    if (pl == 1 && d.npass == 1) { abase = (const __nv_bfloat16*)d.a; bbase = (const __nv_bfloat16*)d.b; }
    bool ok;
    if (d.conv_runs > 0) {
      const long long row_elems = d.a_hstride;   // padded input row pitch (Wp * C)
      uint64_t dims[4] = {(uint64_t)row_elems, (uint64_t)d.M, (uint64_t)d.conv_H, (uint64_t)(d.batches / d.conv_Ho)};
      uint64_t str[4] = {1, (uint64_t)d.a_rstride, (uint64_t)d.a_hstride, (uint64_t)d.a_bstride};
      uint32_t box[4] = {BK, BM, 1, 1};
      ok = make_tmap_bf16(&p->maps.a[pl], abase, 4, dims, str, box);
    } else if (p->rank5) {
      if (d.a_kinner != BK) { g_err = "rank-5 A operand needs a_kinner == 64"; delete p; return nullptr; }
      uint64_t dims[5] = {(uint64_t)d.a_kinner, (uint64_t)(d.K / d.a_kinner), (uint64_t)rows_alloc,
                          (uint64_t)d.groups, (uint64_t)d.batches};
      uint64_t str[5] = {1, (uint64_t)d.a_kouter, (uint64_t)d.a_rstride, (uint64_t)d.a_gstride, (uint64_t)d.a_bstride};
      uint32_t box[5] = {BK, 1, BM, 1, 1};
      // rows_alloc bounds row + tap: the view is (tap, row) -> row+tap; expose rows so that row+tap stays in the batch
      ok = make_tmap_bf16(&p->maps.a[pl], abase, 5, dims, str, box);
    } else {
      uint64_t dims[3] = {(uint64_t)d.K, (uint64_t)rows_alloc, (uint64_t)d.batches};
      uint64_t str[3] = {1, (uint64_t)d.a_rstride, (uint64_t)(d.batches > 1 ? d.a_bstride : d.a_rstride * rows_alloc)};
      uint32_t box[3] = {BK, BM, 1};
      ok = make_tmap_bf16(&p->maps.a[pl], abase, 3, dims, str, box);
    }
    if (!ok) { delete p; return nullptr; }
    const int kb_total = d.conv_runs > 0 ? d.conv_runs * ((d.conv_run_len + BK - 1) / BK) * BK : d.K;
    uint64_t bdims[3] = {(uint64_t)kb_total, (uint64_t)d.N, (uint64_t)d.groups};
    uint64_t bstr[3] = {1, (uint64_t)d.ldb, (uint64_t)(d.groups > 1 ? d.b_gstride : (long long)d.ldb * d.N)};
    uint32_t bbox[3] = {BK, (uint32_t)p->bn, 1};
    if (!make_tmap_bf16(&p->maps.b[pl], bbase, 3, bdims, bstr, bbox)) { delete p; return nullptr; }
  }
  p->mt = (d.M + BM - 1) / BM;
  p->nt = d.groups > 1 ? d.groups : (d.N + p->bn - 1) / p->bn;
  if (want_tma) {
    p->tma_epi = 1;

    p->epi_mode = d.out_bf != nullptr ? 1 : 0;
    bool ok = true;
    if (p->epi_mode == 0) {
      uint64_t dims[3] = {(uint64_t)d.N, (uint64_t)d.M, (uint64_t)d.batches};
      uint64_t so[3] = {1, (uint64_t)d.ldo, (uint64_t)(d.batches > 1 ? d.of_bstride : (long long)d.ldo * d.M)};
      uint32_t box[3] = {32, 32, 1};
      ok = make_tmap_any(&p->em.out, d.out_f32, 4, 3, dims, so, box);
      p->em.out_lo = p->em.out; p->em.res = p->em.out; p->em.res_lo = p->em.out;
      if (ok && d.residual) {
        uint64_t sr[3] = {1, (uint64_t)d.ldr, (uint64_t)(d.batches > 1 ? d.res_bstride : (long long)d.ldr * d.M)};
        ok = make_tmap_any(&p->em.res, d.residual, 4, 3, dims, sr, box);
      }
    } else {
      const int ncols = d.N > d.zero_pad_to ? d.N : d.zero_pad_to;
      uint64_t dims[3] = {(uint64_t)ncols, (uint64_t)d.M, (uint64_t)d.batches};
      uint64_t so[3] = {1, (uint64_t)d.ldob, (uint64_t)(d.batches > 1 ? d.ob_bstride : (long long)d.ldob * (d.M + d.out_row_off))};
      uint32_t box[3] = {64, 32, 1};
      const __nv_bfloat16* ob = (const __nv_bfloat16*)d.out_bf + (long long)d.out_row_off * d.ldob;
      ok = make_tmap_any(&p->em.out, ob, 2, 3, dims, so, box);
      p->em.out_lo = p->em.out; p->em.res = p->em.out; p->em.res_lo = p->em.out;
      if (ok && d.out_planes > 1) ok = make_tmap_any(&p->em.out_lo, ob + d.ob_plane, 2, 3, dims, so, box);
      if (ok && d.res16) {
        uint64_t rdims[3] = {(uint64_t)d.N, (uint64_t)(d.M + d.res16_row_off), (uint64_t)d.batches};
        uint64_t sr[3] = {1, (uint64_t)d.ldr16, (uint64_t)(d.batches > 1 ? d.res16_bstride : (long long)d.ldr16 * (d.M + d.res16_row_off))};
        ok = make_tmap_any(&p->em.res, d.res16, 2, 3, rdims, sr, box);
        if (ok && d.out_planes > 1) ok = make_tmap_any(&p->em.res_lo, (const __nv_bfloat16*)d.res16 + d.res16_plane, 2, 3, rdims, sr, box);
      }
    }
    if (!ok) { delete p; return nullptr; }
  }
  p->ntiles = p->mt * p->nt * d.batches;
  {
    const int ctas = sm_count() * ((p->tma_epi && p->bn == 64) ? 2 : 1);
    p->grid = dim3(p->ntiles < ctas ? p->ntiles : ctas, 1, 1);
  }
  return p;
}

void gemm_plan_destroy(GemmPlan* p) { delete p; }
const GemmDesc& gemm_plan_desc(const GemmPlan* p) { return p->d; }

cudaError_t gemm_plan_launch(const GemmPlan* p, cudaStream_t st) {
  if (p->tma_epi) {
    switch (p->bn) {
      case 64: return launch_bn_tma<64>(p, st);
      case 128: return launch_bn_tma<128>(p, st);
      case 256: {
        // deep ring when nothing is prefetched into the store patches and one 4 KB patch holds a span (single plane)
        static const bool no_deep = (getenv("DZ_GEMM_NO_DEEP") != nullptr);
        const GemmDesc& d = p->d;
        const bool deep = !no_deep && d.residual == nullptr && d.res16 == nullptr && !(p->epi_mode == 1 && d.out_planes > 1);
        return deep ? launch_bn_tma<256, 1>(p, st) : launch_bn_tma<256, 0>(p, st);
      }
    }
    return cudaErrorInvalidValue;
  }
  switch (p->bn) {
    case 64: return launch_bn<64>(p, st);
    case 128: return launch_bn<128>(p, st);
    case 256: return launch_bn<256>(p, st);
  }
  return cudaErrorInvalidValue;
}

}  // namespace dz
