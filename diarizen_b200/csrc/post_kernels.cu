// Warp-shuffle / shared-memory kernels of the post-processing stages (no tensor cores here):
//   median filter of the binarised segmentations, overlap-add speaker counting, embedding mask selection,
//   cluster-wise reconstruction + per-frame top-count selection, N x N Euclidean distances and the centroid-linkage
//   agglomerative clustering merge loop (both in float64, operation for operation as scipy computes them),
//   constrained (one cluster per local speaker) assignment.
// reference: diarizen/pipelines/inference.py:131-132, pyannote-audio/pyannote/audio/core/inference.py:543-666,
//   pipelines/utils/diarization.py:122-157,193-239, pipelines/speaker_diarization.py:271-320,377-425,
//   pipelines/clustering.py:159-173,404-418 (scipy linkage(method="centroid") on unit-norm embeddings).
#include <string>

#include "../../include/diarizen_b200.h"
#include "common.cuh"
#include "lsap_small.cuh"

namespace dz {
std::string& tls_error();
int fail(int code, const std::string& msg);

// ------------------------------------------------------------------------------------------------
// median filter along frames, window `width` (odd), scipy.ndimage 'reflect' boundary (d c b a | a b c d | d c b a).
// Data are {0,1}: the median is the majority vote.
// ------------------------------------------------------------------------------------------------
__global__ void median_filter_kernel(const uint8_t* __restrict__ in, uint8_t* __restrict__ out, int C, int T, int S, int width) {
  const long long total = (long long)C * T * S;
  const int half = width / 2;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int s = (int)(i % S);
    const long long r = i / S;
    const int t = (int)(r % T);
    const long long c = r / T;
    int cnt = 0;
    for (int k = -half; k <= half; ++k) {
      int tt = t + k;
      // reflect (edge sample repeated); windows longer than the signal keep folding
      while (tt < 0 || tt >= T) tt = tt < 0 ? -tt - 1 : 2 * T - tt - 1;
      cnt += in[(c * T + tt) * S + s];
    }
    out[i] = (cnt * 2 > width) ? 1 : 0;
  }
}

// ------------------------------------------------------------------------------------------------
// speaker count: count[f] = rint(mean over the chunks covering frame f of sum_s seg[c][f - start_c][s]) as uint8.
// start[] is non-decreasing; one thread per output frame gathers its (<= ~10) chunks.
// ------------------------------------------------------------------------------------------------
__global__ void speaker_count_kernel(const uint8_t* __restrict__ seg, const int* __restrict__ start, int C, int T, int S, int F,
                                     int max_count, uint8_t* __restrict__ count) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= F) return;
  // first chunk that can cover f: start_c + T > f ; binary search on the sorted starts
  int lo = 0, hi = C;
  while (lo < hi) { const int mid = (lo + hi) >> 1; if (start[mid] + T > f) hi = mid; else lo = mid + 1; }
  float sum = 0.f, n = 0.f;
  for (int c = lo; c < C && start[c] <= f; ++c) {
    const uint8_t* p = seg + ((long long)c * T + (f - start[c])) * S;
    int a = 0;
    for (int s = 0; s < S; ++s) a += p[s];
    sum += (float)a;
    n += 1.f;
  }
  float v = (n > 0.f) ? rintf(__fdiv_rn(sum, n)) : 0.f;   // np.rint: half to even
  int iv = (int)v;
  if (iv > max_count) iv = max_count;
  count[f] = (uint8_t)iv;
}

// ------------------------------------------------------------------------------------------------
// embedding masks: clean = seg * [sum_s seg < 2]; mask[c][s][:] = clean if sum_t clean > min_frames else seg.
// also active[c][s] = sum_t seg > 0 and clean_count[c][s] = #frames where s is the ONLY active speaker.
// One CTA per chunk.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) embedding_masks_kernel(const uint8_t* __restrict__ seg, int T, int S, int min_frames,
                                                              float* __restrict__ masks, int* __restrict__ stats /*[C][S][2]*/) {
  __shared__ int tot[8], cln[8];
  const int c = blockIdx.x;
  if (threadIdx.x < 8) { tot[threadIdx.x] = 0; cln[threadIdx.x] = 0; }
  __syncthreads();
  const uint8_t* p = seg + (long long)c * T * S;
  int lt[4] = {0, 0, 0, 0}, lc[4] = {0, 0, 0, 0};
  for (int t = threadIdx.x; t < T; t += blockDim.x) {
    int a = 0;
    for (int s = 0; s < S; ++s) a += p[t * S + s];
    for (int s = 0; s < S; ++s) { lt[s] += p[t * S + s]; lc[s] += (a < 2) ? p[t * S + s] : 0; }
  }
  for (int s = 0; s < S; ++s) { atomicAdd(&tot[s], lt[s]); atomicAdd(&cln[s], lc[s]); }
  __syncthreads();
  for (int i = threadIdx.x; i < S * T; i += blockDim.x) {
    const int s = i / T, t = i - s * T;
    int a = 0;
    for (int q = 0; q < S; ++q) a += p[t * S + q];
    const bool use_clean = cln[s] > min_frames;
    const uint8_t v = p[t * S + s];
    masks[((long long)c * S + s) * T + t] = (use_clean && a >= 2) ? 0.f : (float)v;
  }
  if (threadIdx.x < S) { stats[(c * S + threadIdx.x) * 2] = tot[threadIdx.x]; stats[(c * S + threadIdx.x) * 2 + 1] = cln[threadIdx.x]; }
}

// ------------------------------------------------------------------------------------------------
// reconstruct + to_diarization: act[f][k] = sum over chunks covering f of max_{s: hard[c][s]==k} seg[c][f-start_c][s];
// then the count[f] largest activations (stable: lower cluster index wins ties) are switched on.
// One thread per frame, K <= 32.
// ------------------------------------------------------------------------------------------------
__global__ void reconstruct_kernel(const uint8_t* __restrict__ seg, const int8_t* __restrict__ hard, const int* __restrict__ start,
                                   const uint8_t* __restrict__ count, int C, int T, int S, int K, int Kout, int F,
                                   uint8_t* __restrict__ discrete, float* __restrict__ act_out) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= F) return;
  float act[32];
#pragma unroll
  for (int k = 0; k < 32; ++k) act[k] = 0.f;
  int lo = 0, hi = C;
  while (lo < hi) { const int mid = (lo + hi) >> 1; if (start[mid] + T > f) hi = mid; else lo = mid + 1; }
  for (int c = lo; c < C && start[c] <= f; ++c) {
    const uint8_t* p = seg + ((long long)c * T + (f - start[c])) * S;
    unsigned on = 0;   // clusters active in this chunk at this frame (max over local speakers of a 0/1 value)
    for (int s = 0; s < S; ++s) {
      const int k = hard[c * S + s];
      if (k >= 0 && k < 32 && p[s]) on |= 1u << k;
    }
#pragma unroll
    for (int k = 0; k < 32; ++k) act[k] += (float)((on >> k) & 1u);
  }
  const int cnt = min((int)count[f], Kout);
  unsigned chosen = 0;
  for (int i = 0; i < cnt; ++i) {
    int best = -1; float bv = -1.f;
    for (int k = 0; k < Kout; ++k) {
      if ((chosen >> k) & 1u) continue;
      const float v = (k < K) ? act[k] : 0.f;   // columns >= K are the zero padding of diarization.py:222-226
      if (v > bv) { bv = v; best = k; }
    }
    if (best < 0) break;
    chosen |= 1u << best;
  }
  for (int k = 0; k < Kout; ++k) {
    discrete[(long long)f * Kout + k] = (chosen >> k) & 1u;
    if (act_out) act_out[(long long)f * Kout + k] = (k < K) ? act[k] : 0.f;
  }
}

// Same for 32 < K <= 128 clusters (int8 labels allow 127): the per-frame activations live in shared memory ([k][thread],
// conflict-free) instead of registers.  One thread per frame.
__global__ void __launch_bounds__(128) reconstruct_wide_kernel(const uint8_t* __restrict__ seg, const int8_t* __restrict__ hard,
                                                               const int* __restrict__ start, const uint8_t* __restrict__ count, int C,
                                                               int T, int S, int K, int Kout, int F, uint8_t* __restrict__ discrete,
                                                               float* __restrict__ act_out) {
  extern __shared__ float wact[];   // [Kout][128]
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  float* act = wact + threadIdx.x;
  for (int k = 0; k < Kout; ++k) act[k * 128] = 0.f;
  if (f >= F) return;
  int lo = 0, hi = C;
  while (lo < hi) { const int mid = (lo + hi) >> 1; if (start[mid] + T > f) hi = mid; else lo = mid + 1; }
  for (int c = lo; c < C && start[c] <= f; ++c) {
    const uint8_t* p = seg + ((long long)c * T + (f - start[c])) * S;
    for (int s = 0; s < S; ++s) {
      const int k = hard[c * S + s];
      if (k < 0 || k >= K || !p[s]) continue;
      bool dup = false;                       // max over the local speakers of one cluster, not their sum
      for (int q = 0; q < s; ++q) dup |= (hard[c * S + q] == k) && p[q];
      if (!dup) act[k * 128] += 1.f;
    }
  }
  if (act_out)
    for (int k = 0; k < Kout; ++k) act_out[(long long)f * Kout + k] = act[k * 128];
  for (int k = 0; k < Kout; ++k) discrete[(long long)f * Kout + k] = 0;
  const int cnt = min((int)count[f], Kout);
  for (int i = 0; i < cnt; ++i) {
    int best = -1; float bv = -1.f;
    for (int k = 0; k < Kout; ++k) {
      const float v = act[k * 128];
      if (v > bv) { bv = v; best = k; }       // chosen entries are marked -2 below
    }
    if (best < 0) break;
    discrete[(long long)f * Kout + best] = 1;
    act[best * 128] = -2.f;
  }
}

// ------------------------------------------------------------------------------------------------
// Euclidean distance matrix in float64, exactly as scipy.spatial.distance.pdist computes it on the float64 copy of the
// (float32, unit-norm) embeddings: d = sqrt(sum_k (u_k - v_k)^2) accumulated sequentially, no fused multiply-add.
// 32 x 32 tile of pairs per CTA, rows staged in shared memory.  Writes the full symmetric matrix.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) pdist_kernel(const float* __restrict__ X, int N, int D, double* __restrict__ out) {
  extern __shared__ float sx[];   // [2][32][D + 1]
  const int bi = blockIdx.y, bj = blockIdx.x;
  if (bj < bi) return;
  const int ld = D + 1;
  float* A = sx;
  float* B = sx + 32 * ld;
  for (int e = threadIdx.x; e < 32 * D; e += blockDim.x) {
    const int r = e / D, k = e - r * D;
    const int gi = bi * 32 + r, gj = bj * 32 + r;
    A[r * ld + k] = gi < N ? X[(long long)gi * D + k] : 0.f;
    B[r * ld + k] = gj < N ? X[(long long)gj * D + k] : 0.f;
  }
  __syncthreads();
  const int tj = threadIdx.x & 31, ti0 = threadIdx.x >> 5;   // each thread: column tj, rows ti0, ti0+8, ...
  for (int q = 0; q < 4; ++q) {
    const int ti = ti0 + 8 * q;
    const int gi = bi * 32 + ti, gj = bj * 32 + tj;
    if (gi >= N || gj >= N) continue;
    double s = 0.0;
    for (int k = 0; k < D; ++k) {
      const double dl = __dsub_rn((double)A[ti * ld + k], (double)B[tj * ld + k]);
      s = __dadd_rn(s, __dmul_rn(dl, dl));
    }
    const double dist = (gi == gj) ? 0.0 : __dsqrt_rn(s);
    out[(long long)gi * N + gj] = dist;
    out[(long long)gj * N + gi] = dist;
  }
}

// ------------------------------------------------------------------------------------------------
// Centroid-linkage agglomerative clustering (scipy.cluster.hierarchy.linkage(method="centroid")), one persistent CTA.
// Every step merges the globally closest pair of live clusters (x < y slot indices; the merged cluster lives in slot y
// and gets id N + step) and updates the distances with scipy's Lance-Williams expression in float64, evaluated in the
// same order and without fused multiply-add:
//   d(z, x+y) = sqrt((((nx*dxz)*dxz + (ny*dyz)*dyz) - ((nx*ny)*dxy*dxy)/(nx+ny)) / (nx+ny))
// A nearest-neighbour cache (nn[i], nnd[i] over all live j != i) keeps a step at O(N) plus a few row rescans.
// Z row = (min id, max id, distance, size).
// ------------------------------------------------------------------------------------------------
struct ArgMin { double v; int i; };
DZ_DEVINL ArgMin amin(ArgMin a, ArgMin b) { return (b.v < a.v || (b.v == a.v && b.i < a.i)) ? b : a; }
DZ_DEVINL ArgMin block_argmin(ArgMin v, ArgMin* sc) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ArgMin t; t.v = __shfl_xor_sync(0xffffffffu, v.v, o); t.i = __shfl_xor_sync(0xffffffffu, v.i, o);
    v = amin(v, t);
  }
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = blockDim.x >> 5;
  __syncthreads();
  if (l == 0) sc[w] = v;
  __syncthreads();
  ArgMin r = (l < nw) ? sc[l] : ArgMin{INFINITY, 0x7fffffff};
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ArgMin t; t.v = __shfl_xor_sync(0xffffffffu, r.v, o); t.i = __shfl_xor_sync(0xffffffffu, r.i, o);
    r = amin(r, t);
  }
  return r;
}

__global__ void __launch_bounds__(1024) linkage_centroid_kernel(double* __restrict__ Dm, int N, double* __restrict__ Z,
                                                                int* __restrict__ size, int* __restrict__ cid, int* __restrict__ nn,
                                                                double* __restrict__ nnd, int* __restrict__ todo) {
  __shared__ ArgMin sc[32];
  __shared__ int s_ntodo;
  const int tid = threadIdx.x, nt = blockDim.x;
  for (int i = tid; i < N; i += nt) { size[i] = 1; cid[i] = i; }
  __syncthreads();
  // initial nearest neighbours: one warp per row
  for (int i = tid >> 5; i < N; i += nt >> 5) {
    ArgMin best{INFINITY, 0x7fffffff};
    const double* row = Dm + (long long)i * N;
    for (int j = tid & 31; j < N; j += 32)
      if (j != i) best = amin(best, ArgMin{row[j], j});
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      ArgMin t; t.v = __shfl_xor_sync(0xffffffffu, best.v, o); t.i = __shfl_xor_sync(0xffffffffu, best.i, o);
      best = amin(best, t);
    }
    if ((tid & 31) == 0) { nn[i] = best.i; nnd[i] = best.v; }
  }
  __syncthreads();
  for (int step = 0; step < N - 1; ++step) {
    // 1. globally closest pair
    ArgMin best{INFINITY, 0x7fffffff};
    for (int i = tid; i < N; i += nt)
      if (size[i] > 0) best = amin(best, ArgMin{nnd[i], i});
    best = block_argmin(best, sc);
    int x = best.i, y = nn[x];
    if (x > y) { const int t = x; x = y; y = t; }
    const double dxy = Dm[(long long)x * N + y];
    const int nx = size[x], ny = size[y];
    __syncthreads();
    if (tid == 0) {
      const int ix = cid[x], iy = cid[y];
      Z[step * 4 + 0] = (double)min(ix, iy);
      Z[step * 4 + 1] = (double)max(ix, iy);
      Z[step * 4 + 2] = dxy;
      Z[step * 4 + 3] = (double)(nx + ny);
      s_ntodo = 0;
    }
    __syncthreads();
    // 2. Lance-Williams update of row / column y; x dies
    const double nxy = (double)(nx + ny);
    const double cxy = __ddiv_rn(__dmul_rn(__dmul_rn((double)(nx * ny), dxy), dxy), nxy);
    for (int z = tid; z < N; z += nt) {
      if (size[z] == 0 || z == x || z == y) continue;
      const double dxz = Dm[(long long)x * N + z], dyz = Dm[(long long)y * N + z];
      const double t1 = __dmul_rn(__dmul_rn((double)nx, dxz), dxz);
      const double t2 = __dmul_rn(__dmul_rn((double)ny, dyz), dyz);
      const double nd = __dsqrt_rn(__ddiv_rn(__dsub_rn(__dadd_rn(t1, t2), cxy), nxy));
      Dm[(long long)y * N + z] = nd;
      Dm[(long long)z * N + y] = nd;
      // nearest-neighbour maintenance for row z
      const int nz = nn[z];
      if (nz == x || nz == y) {
        todo[atomicAdd(&s_ntodo, 1)] = z;          // its cached neighbour changed: rescan
      } else if (nd < nnd[z]) {
        nn[z] = y; nnd[z] = nd;
      }
    }
    __syncthreads();
    if (tid == 0) { size[x] = 0; size[y] = nx + ny; cid[y] = N + step; todo[s_ntodo++] = y; }
    __syncthreads();
    // 3. rescan the rows whose cached neighbour was invalidated (one warp per row)
    const int ntodo = s_ntodo;
    for (int q = tid >> 5; q < ntodo; q += nt >> 5) {
      const int i = todo[q];
      ArgMin b2{INFINITY, 0x7fffffff};
      const double* row = Dm + (long long)i * N;
      for (int j = tid & 31; j < N; j += 32)
        if (j != i && size[j] > 0) b2 = amin(b2, ArgMin{row[j], j});
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        ArgMin t; t.v = __shfl_xor_sync(0xffffffffu, b2.v, o); t.i = __shfl_xor_sync(0xffffffffu, b2.i, o);
        b2 = amin(b2, t);
      }
      if ((tid & 31) == 0) { nn[i] = b2.i; nnd[i] = b2.v; }
    }
    __syncthreads();
  }
}

// Initial nearest neighbours for every row, on all SMs (one warp per row): the N x N float64 matrix is read once at HBM
// speed here instead of through the single SM that runs the merge loop. Ties go to the lowest column index.
__global__ void __launch_bounds__(256) linkage_nn_init_kernel(const double* __restrict__ Dm, int N, int* __restrict__ nn,
                                                              double* __restrict__ nnd) {
  const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  for (int i = blockIdx.x * wpb + (threadIdx.x >> 5); i < N; i += gridDim.x * wpb) {
    ArgMin best{INFINITY, 0x7fffffff};
    const double* row = Dm + (long long)i * N;
    for (int j0 = lane; j0 < N; j0 += 256) {
      double v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) { const int j = j0 + 32 * u; v[u] = (j < N) ? __ldcs(row + j) : INFINITY; }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int j = j0 + 32 * u;
        if (j < N && j != i) best = amin(best, ArgMin{v[u], j});
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      ArgMin t; t.v = __shfl_xor_sync(0xffffffffu, best.v, o); t.i = __shfl_xor_sync(0xffffffffu, best.i, o);
      best = amin(best, t);
    }
    if (lane == 0) { nn[i] = best.i; nnd[i] = best.v; }
  }
}

// two block-wide argmins behind one pair of barriers
DZ_DEVINL void block_argmin2(ArgMin& a, ArgMin& b, ArgMin* sc) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ArgMin t; t.v = __shfl_xor_sync(0xffffffffu, a.v, o); t.i = __shfl_xor_sync(0xffffffffu, a.i, o);
    a = amin(a, t);
    ArgMin u; u.v = __shfl_xor_sync(0xffffffffu, b.v, o); u.i = __shfl_xor_sync(0xffffffffu, b.i, o);
    b = amin(b, u);
  }
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = blockDim.x >> 5;
  __syncthreads();
  if (l == 0) { sc[w] = a; sc[32 + w] = b; }
  __syncthreads();
  a = (l < nw) ? sc[l] : ArgMin{INFINITY, 0x7fffffff};
  b = (l < nw) ? sc[32 + l] : ArgMin{INFINITY, 0x7fffffff};
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ArgMin t; t.v = __shfl_xor_sync(0xffffffffu, a.v, o); t.i = __shfl_xor_sync(0xffffffffu, a.i, o);
    a = amin(a, t);
    ArgMin u; u.v = __shfl_xor_sync(0xffffffffu, b.v, o); u.i = __shfl_xor_sync(0xffffffffu, b.i, o);
    b = amin(b, u);
  }
}

// The default merge loop for N < 65535 (its slot indices are 16-bit; the kernel above takes larger N): the same arithmetic,
// the same (distance, index) order for the closest pair, organised for one SM's latency and float64 budget:
//  * state (nnd, nn, size, the compact list of live slots and its inverse) in shared memory as 8 + 4 x 2 bytes per slot
//    (N <= ~14 000; beyond that the same code runs on the global workspace); initial neighbours from linkage_nn_init_kernel;
//  * only LIVE slots are visited: the update loop and the row scans walk the compact list, so a step costs O(live), not O(N)
//    (the update is float64-issue-bound: two multiplies, a divide and a square root per live slot);
//  * nnd[z] is a LOWER BOUND when nn[z] == STALE: a row whose cached neighbour was merged away is rescanned only when its
//    bound reaches the top of the selection (the way scipy's own generic algorithm defers its find_min_dist), and not at
//    all if a later merge lands below the bound first - `nd < nnd[z]` then makes the row exact again.  The closest pair
//    is still the exact global minimum with the lowest slot index: every row ordered before it is exact or gets rescanned;
//  * global round trips are batched: all (d(x,z), d(y,z)) pairs of a batch are loaded before the first store (the stores
//    to Dm would otherwise fence each iteration's loads behind the previous one's), row scans keep U loads in flight per
//    thread, d(x,y) is the cached nnd[x], the merged row's neighbour is the block-argmin of the freshly computed distances;
//  * the update loop also carries the minimum of the (updated) bounds of the rows it visits, so the NEXT step's selection is
//    ready after the same pair of barriers; a separate selection pass runs only after a rescan.
constexpr uint16_t kStale = 0xFFFFu;
template <int NT, int U, bool SMEM>
__global__ void __launch_bounds__(NT) linkage_centroid_lazy_kernel(double* __restrict__ Dm, int N, double* __restrict__ Z,
                                                                   int* __restrict__ cid, const int* __restrict__ nn0,
                                                                   double* __restrict__ nnd0, uint16_t* __restrict__ g16,
                                                                   unsigned long long* __restrict__ counters) {
  extern __shared__ double lsm[];
  double* nnd = SMEM ? lsm : nnd0;                                         // [N]
  uint16_t* nn = SMEM ? reinterpret_cast<uint16_t*>(lsm + N) : g16;        // [N]
  uint16_t* size = nn + N;                                                 // [N]
  uint16_t* live = size + N;                                               // [N] compact list of live slots
  uint16_t* pos = live + N;                                                // [N] slot -> position in live
  __shared__ ArgMin sc[64];
  const int tid = threadIdx.x, nt = NT;
  for (int i = tid; i < N; i += nt) {
    size[i] = 1; cid[i] = i; live[i] = (uint16_t)i; pos[i] = (uint16_t)i;
    nn[i] = (uint16_t)nn0[i];
    if (SMEM) nnd[i] = nnd0[i];
  }
  __syncthreads();
  unsigned long long nrescan = 0;
  ArgMin best{INFINITY, 0x7fffffff};
  bool have_best = false;                                                  // best = the selection carried over from the last update
  for (int step = 0; step < N - 1; ++step) {
    const int L = N - step;                                                // live slots
    // 1. closest pair: argmin of the bounds; a stale row at the top is made exact and the selection repeats
    for (;;) {
      if (!have_best) {
        best = ArgMin{INFINITY, 0x7fffffff};
        for (int k = tid; k < L; k += nt) { const int i = live[k]; best = amin(best, ArgMin{nnd[i], i}); }
        best = block_argmin(best, sc);
      }
      have_best = false;
      if (nn[best.i] != kStale) break;
      const int i = best.i;
      const double* row = Dm + (long long)i * N;
      ArgMin b2{INFINITY, 0x7fffffff};
      for (int k0 = tid; k0 < L; k0 += U * nt) {
        double v[U];
        int jj[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int k = k0 + u * nt;
          int j = (k < L) ? (int)live[k] : -1;
          if (j == i) j = -1;
          jj[u] = j;
          v[u] = (j >= 0) ? row[j] : INFINITY;
        }
#pragma unroll
        for (int u = 0; u < U; ++u)
          if (jj[u] >= 0) b2 = amin(b2, ArgMin{v[u], jj[u]});
      }
      b2 = block_argmin(b2, sc);
      if (tid == 0) { nn[i] = (uint16_t)b2.i; nnd[i] = b2.v; ++nrescan; }
      __syncthreads();
    }
    int x = best.i, y = nn[x];
    if (x > y) { const int t = x; x = y; y = t; }
    const double dxy = best.v;                         // == Dm[x][y]: an exact nnd caches exactly the stored distance
    const int nx = size[x], ny = size[y];
    if (tid == nt - 1) {                               // the last warp has the fewest columns: it writes the Z row
      const int ix = cid[x], iy = cid[y];
      Z[step * 4 + 0] = (double)min(ix, iy);
      Z[step * 4 + 1] = (double)max(ix, iy);
      Z[step * 4 + 2] = dxy;
      Z[step * 4 + 3] = (double)(nx + ny);
      cid[y] = N + step;
    }
    // 2. Lance-Williams update of row / column y over the live slots; x dies
    const double nxy = (double)(nx + ny);
    const double cxy = __ddiv_rn(__dmul_rn(__dmul_rn((double)(nx * ny), dxy), dxy), nxy);
    const double* rx = Dm + (long long)x * N;
    double* ry = Dm + (long long)y * N;
    ArgMin ybest{INFINITY, 0x7fffffff}, obest{INFINITY, 0x7fffffff};
    for (int k0 = tid; k0 < L; k0 += U * nt) {
      double dx[U], dy[U];
      int zz[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int k = k0 + u * nt;
        int z = (k < L) ? (int)live[k] : -1;
        if (z == x || z == y) z = -1;
        zz[u] = z;
        dx[u] = (z >= 0) ? rx[z] : 0.0;
        dy[u] = (z >= 0) ? ry[z] : 0.0;
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int z = zz[u];
        if (z < 0) continue;
        const double t1 = __dmul_rn(__dmul_rn((double)nx, dx[u]), dx[u]);
        const double t2 = __dmul_rn(__dmul_rn((double)ny, dy[u]), dy[u]);
        const double nd = __dsqrt_rn(__ddiv_rn(__dsub_rn(__dadd_rn(t1, t2), cxy), nxy));
        ry[z] = nd;
        Dm[(long long)z * N + y] = nd;
        ybest = amin(ybest, ArgMin{nd, z});
        const int nz = nn[z];
        double bound = nnd[z];
        if (nd < bound) {                              // below the row's minimum (or its bound): exact again
          nn[z] = (uint16_t)y; nnd[z] = nd; bound = nd;
        } else if (nz == x || nz == y) {
          nn[z] = kStale;                              // cached neighbour gone: nnd[z] stays as a lower bound
        }
        obest = amin(obest, ArgMin{bound, z});
      }
    }
    // ybest: the merged row's neighbour = min over live z of (d(y,z), z), lowest z on ties; obest: min bound of the other rows
    block_argmin2(ybest, obest, sc);
    best = amin(obest, ArgMin{ybest.v, y});            // next step's selection
    have_best = true;
    if (tid == 0) {
      size[x] = 0; size[y] = (uint16_t)(nx + ny);
      nn[y] = (uint16_t)ybest.i; nnd[y] = ybest.v;
      const int p = pos[x], last = live[L - 1];        // drop x from the live list
      live[p] = (uint16_t)last; pos[last] = (uint16_t)p;
    }
    __syncthreads();
  }
  if (tid == 0 && counters) counters[0] = nrescan;
}

// ------------------------------------------------------------------------------------------------
// Constrained assignment (one distinct cluster per local speaker, maximal total score; clustering.py:159-173): one thread per
// chunk runs the shortest-augmenting-path solver of lsap_small.cuh - scipy's algorithm step for step, so that the many exact
// ties (inactive local speakers share one embedding, hence identical score rows) resolve exactly as in the reference.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(64) assign_kernel(const double* __restrict__ soft, int C, int S, int K, int8_t* __restrict__ hard) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  int8_t h[4];
  lsap_assign_max(soft + (long long)c * S * K, S, K, h);
  for (int s = 0; s < S; ++s) hard[c * S + s] = h[s];
}

}  // namespace dz

using namespace dz;
#define CK_LAUNCH() do { cudaError_t e__ = cudaGetLastError(); if (e__ != cudaSuccess) return fail(DZ_ERR_CUDA, cudaGetErrorString(e__)); } while (0)

extern "C" {

int dz_median_filter(const uint8_t* in_dev, uint8_t* out_dev, int C, int T, int S, int width, void* stream) {
  if (!in_dev || !out_dev || width < 1 || !(width & 1)) return fail(DZ_ERR_INVALID, "bad argument");
  const long long total = (long long)C * T * S;
  median_filter_kernel<<<(int)min((long long)148 * 16, (total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(in_dev, out_dev, C, T, S, width);
  CK_LAUNCH();
  return DZ_OK;
}
int dz_speaker_count(const uint8_t* seg_dev, const int32_t* start_dev, int C, int T, int S, int F, int max_count, uint8_t* count_dev, void* stream) {
  if (!seg_dev || !start_dev || !count_dev) return fail(DZ_ERR_INVALID, "bad argument");
  speaker_count_kernel<<<(F + 255) / 256, 256, 0, (cudaStream_t)stream>>>(seg_dev, start_dev, C, T, S, F, max_count, count_dev);
  CK_LAUNCH();
  return DZ_OK;
}
int dz_embedding_masks(const uint8_t* seg_dev, int C, int T, int S, int min_frames, float* masks_dev, int32_t* stats_dev, void* stream) {
  if (!seg_dev || !masks_dev || !stats_dev || S > 4) return fail(DZ_ERR_INVALID, "bad argument (S <= 4)");
  embedding_masks_kernel<<<C, 256, 0, (cudaStream_t)stream>>>(seg_dev, T, S, min_frames, masks_dev, stats_dev);
  CK_LAUNCH();
  return DZ_OK;
}
int dz_reconstruct(const uint8_t* seg_dev, const int8_t* hard_dev, const int32_t* start_dev, const uint8_t* count_dev, int C, int T,
                   int S, int K, int Kout, int F, uint8_t* discrete_dev, float* act_dev, void* stream) {
  if (!seg_dev || !hard_dev || !start_dev || !count_dev || !discrete_dev || K > 128 || K < 1 || Kout < K || Kout > 255 || S < 1 || S > 8)
    return fail(DZ_ERR_INVALID, "bad argument (1 <= K <= 128, K <= Kout <= 255)");
  if (Kout <= 32) {
    reconstruct_kernel<<<(F + 127) / 128, 128, 0, (cudaStream_t)stream>>>(seg_dev, hard_dev, start_dev, count_dev, C, T, S, K, Kout, F, discrete_dev, act_dev);
  } else {
    const size_t smem = (size_t)Kout * 128 * sizeof(float);
    static size_t attr = 0;
    if (smem > 48 * 1024 && smem > attr) {
      cudaError_t e = cudaFuncSetAttribute(reconstruct_wide_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return fail(DZ_ERR_CUDA, cudaGetErrorString(e));
      attr = smem;
    }
    reconstruct_wide_kernel<<<(F + 127) / 128, 128, smem, (cudaStream_t)stream>>>(seg_dev, hard_dev, start_dev, count_dev, C, T, S, K, Kout, F, discrete_dev, act_dev);
  }
  CK_LAUNCH();
  return DZ_OK;
}
int dz_pdist(const float* x_dev, int N, int D, double* out_dev, void* stream) {
  if (!x_dev || !out_dev || N < 1 || D < 1 || D > 512) return fail(DZ_ERR_INVALID, "bad argument");
  const size_t smem = sizeof(float) * 2 * 32 * (D + 1);
  static size_t attr = 0;
  if (smem > 48 * 1024 && smem > attr) { cudaFuncSetAttribute(pdist_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); attr = smem; }
  dim3 grid((N + 31) / 32, (N + 31) / 32);
  pdist_kernel<<<grid, 256, smem, (cudaStream_t)stream>>>(x_dev, N, D, out_dev);
  CK_LAUNCH();
  return DZ_OK;
}
/* workspace_dev: at least dz_linkage_workspace_bytes(N) bytes */
int64_t dz_linkage_workspace_bytes(int N) { return (int64_t)N * (4 * 4 + 8) + 256; }
/* variant: 0 = the default choice, 1 = first-generation kernel, 2 = lazy kernel with its state in the global workspace (what
   N > ~14 000 runs) - 1 and 2 exist so that the tests can drive every code path at small N */
int dz_linkage_centroid_variant(double* dist_dev, int N, double* z_dev, void* workspace_dev, void* stream, int variant) {
  if (!dist_dev || !z_dev || !workspace_dev || N < 2 || variant < 0 || variant > 2) return fail(DZ_ERR_INVALID, "bad argument");
  char* w = (char*)workspace_dev;
  double* nnd = (double*)w; w += (size_t)N * 8;
  int* cid = (int*)w; w += (size_t)N * 4;
  int* nn = (int*)w; w += (size_t)N * 4;
  char* rest = w;                                          // 8 N bytes: v1's size + todo, or the lazy kernel's 16-bit state
  unsigned long long* counters = (unsigned long long*)(rest + (size_t)N * 8);   // in the 256-byte tail: [0] = row rescans of the last call
  if (variant != 1 && N < 65535) {
    const size_t smem = (size_t)N * (8 + 4 * 2);
    const bool in_smem = smem <= 220 * 1024 && variant != 2;
    // 512 threads x 16 loads in flight: ~10 % faster than 1024 x 8 on every data set tried (cheaper barriers, no spills)
    auto kern = in_smem ? linkage_centroid_lazy_kernel<512, 16, true> : linkage_centroid_lazy_kernel<512, 16, false>;
    static size_t attr = 0;
    if (in_smem && smem > attr) {
      cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return fail(DZ_ERR_CUDA, cudaGetErrorString(e));
      attr = smem;
    }
    linkage_nn_init_kernel<<<min((N + 7) / 8, 148 * 8), 256, 0, (cudaStream_t)stream>>>(dist_dev, N, nn, nnd);
    CK_LAUNCH();
    kern<<<1, 512, in_smem ? smem : 0, (cudaStream_t)stream>>>(dist_dev, N, z_dev, cid, nn, nnd, (uint16_t*)rest, counters);
    CK_LAUNCH();
    return DZ_OK;
  }
  int* size = (int*)rest;
  int* todo = size + N;
  linkage_centroid_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(dist_dev, N, z_dev, size, cid, nn, nnd, todo);
  CK_LAUNCH();
  return DZ_OK;
}
int dz_linkage_centroid(double* dist_dev, int N, double* z_dev, void* workspace_dev, void* stream) {
  return dz_linkage_centroid_variant(dist_dev, N, z_dev, workspace_dev, stream, 0);
}
int dz_assign(const double* soft_dev, int C, int S, int K, int8_t* hard_dev, void* stream) {
  if (!soft_dev || !hard_dev || S < 1 || S > 4 || K < 1 || K > 127) return fail(DZ_ERR_INVALID, "bad argument (S <= 4, K <= 127: labels are int8)");
  assign_kernel<<<(C + 63) / 64, 64, 0, (cudaStream_t)stream>>>(soft_dev, C, S, K, hard_dev);
  CK_LAUNCH();
  return DZ_OK;
}

}  // extern "C"

// ================================================================================================
// VBx (variational Bayes GMM over PLDA-space x-vectors): the two halves of one iteration, float64.
// reference: diarizen/clustering/VBx.py:86-111 (loopProb = 0 branch; the HMM branch is unreachable there).
//   model update  : Ns = sum_t gamma[t,s]; invL[s,d] = 1 / (1 + Fa/Fb * Ns * Phi[d]); alpha[s,d] = Fa/Fb * invL[s,d] * sum_t gamma[t,s] rho[t,d]
//   responsibility: log_p[t,s] = Fa * (rho[t].alpha[s] - 0.5 * sum_d (invL[s,d] + alpha[s,d]^2) Phi[d] + G[t]);
//                   gamma[t,s] = exp(log_p + log(pi_s + 1e-8) - logsumexp_s(...)); pi_new[s] = sum_t gamma[t,s]; logpX = sum_t logsumexp
// ================================================================================================
namespace dz {

__global__ void __launch_bounds__(256) vbx_model_kernel(const double* __restrict__ gamma, const double* __restrict__ rho,
                                                        const double* __restrict__ Phi, int N, int D, int S, double fafb,
                                                        double* __restrict__ alpha, double* __restrict__ invL) {
  __shared__ double sc[32];
  const int s = blockIdx.x;
  double ns = 0.0;
  for (int t = threadIdx.x; t < N; t += blockDim.x) ns += gamma[(long long)t * S + s];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ns += __shfl_xor_sync(0xffffffffu, ns, o);
  if ((threadIdx.x & 31) == 0) sc[threadIdx.x >> 5] = ns;
  __syncthreads();
  ns = 0.0;
  for (int w = 0; w < (blockDim.x >> 5); ++w) ns += sc[w];
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    double acc = 0.0;
    for (int t = 0; t < N; ++t) acc += gamma[(long long)t * S + s] * rho[(long long)t * D + d];
    const double il = 1.0 / (1.0 + fafb * ns * Phi[d]);
    invL[s * D + d] = il;
    alpha[s * D + d] = fafb * il * acc;
  }
}

__global__ void __launch_bounds__(256) vbx_resp_kernel(const double* __restrict__ rho, const double* __restrict__ G,
                                                       const double* __restrict__ alpha, const double* __restrict__ invL,
                                                       const double* __restrict__ Phi, const double* __restrict__ pi, int N, int D,
                                                       int S, double Fa, double* __restrict__ gamma, double* __restrict__ pi_acc,
                                                       double* __restrict__ logpx_acc) {
  extern __shared__ double sh[];   // [S] constant term per speaker, [S] log prior
  double* cst = sh;
  double* lpi = sh + S;
  for (int s = threadIdx.x; s < S; s += blockDim.x) {
    double c = 0.0;
    for (int d = 0; d < D; ++d) c += (invL[s * D + d] + alpha[s * D + d] * alpha[s * D + d]) * Phi[d];
    cst[s] = 0.5 * c;
    lpi[s] = log(pi[s] + 1e-8);
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int t = blockIdx.x * 8 + warp; t < N; t += gridDim.x * 8) {
    const double* r = rho + (long long)t * D;
    double mx = -INFINITY;
    // pass 1: scores (kept in gamma as scratch), running max
    for (int s = 0; s < S; ++s) {
      double dot = 0.0;
      for (int d = lane; d < D; d += 32) dot += r[d] * alpha[s * D + d];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
      const double v = Fa * (dot - cst[s] + G[t]) + lpi[s];
      if (lane == 0) gamma[(long long)t * S + s] = v;
      mx = fmax(mx, v);
    }
    __syncwarp();
    double se = 0.0;
    for (int s = lane; s < S; s += 32) se += exp(gamma[(long long)t * S + s] - mx);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) se += __shfl_xor_sync(0xffffffffu, se, o);
    const double lse = mx + log(se);
    for (int s = lane; s < S; s += 32) {
      const double g = exp(gamma[(long long)t * S + s] - lse);
      gamma[(long long)t * S + s] = g;
      atomicAdd(&pi_acc[s], g);
    }
    if (lane == 0) atomicAdd(logpx_acc, lse);
  }
}

}  // namespace dz

extern "C" {
int dz_vbx_model(const double* gamma_dev, const double* rho_dev, const double* phi_dev, int N, int D, int S, double fa_over_fb,
                 double* alpha_dev, double* invl_dev, void* stream) {
  if (!gamma_dev || !rho_dev || !phi_dev || !alpha_dev || !invl_dev || N < 1 || D < 1 || S < 1) return fail(DZ_ERR_INVALID, "bad argument");
  dz::vbx_model_kernel<<<S, 256, 0, (cudaStream_t)stream>>>(gamma_dev, rho_dev, phi_dev, N, D, S, fa_over_fb, alpha_dev, invl_dev);
  CK_LAUNCH();
  return DZ_OK;
}
/* pi_acc_dev [S] and logpx_acc_dev [1] must be zeroed by the caller; gamma_dev [N][S] is overwritten */
int dz_vbx_resp(const double* rho_dev, const double* g_dev, const double* alpha_dev, const double* invl_dev, const double* phi_dev,
                const double* pi_dev, int N, int D, int S, double Fa, double* gamma_dev, double* pi_acc_dev, double* logpx_acc_dev,
                void* stream) {
  if (!rho_dev || !g_dev || !alpha_dev || !invl_dev || !phi_dev || !pi_dev || !gamma_dev || !pi_acc_dev || !logpx_acc_dev)
    return fail(DZ_ERR_INVALID, "bad argument");
  const int grid = (N + 7) / 8 < 148 * 4 ? (N + 7) / 8 : 148 * 4;
  dz::vbx_resp_kernel<<<grid, 256, sizeof(double) * 2 * S, (cudaStream_t)stream>>>(rho_dev, g_dev, alpha_dev, invl_dev, phi_dev, pi_dev,
                                                                                  N, D, S, Fa, gamma_dev, pi_acc_dev, logpx_acc_dev);
  CK_LAUNCH();
  return DZ_OK;
}
}  // extern "C"
