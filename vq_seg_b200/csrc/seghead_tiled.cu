// Tiled kernels of the VQ segmentation head for any class count K and any feature width D (the per-pixel kernels
// of seghead.cu hold all K chains of a pixel in registers and the prototypes in shared memory: K <= 32, D <= 382).
//
// One register-tiled fp32 contraction core (fma_rows) serves all three kernels.  A block of 256 threads owns a
// 128 x 64 output tile; thread (ta, tb) keeps an 8 x 4 register tile of accumulators; operand tiles of 32 rows are
// staged through shared memory, one after the other in increasing row order.
//   map      : acc[pixel][class] += x[pixel][d] e[class][d], rows = d.  Each accumulator is exactly the exact
//              scorer's chain (exact_chain.cuh, chain_dist2): one fp32 FMA chain in increasing d, restarted at
//              MKL's K-block boundaries, |x|^2 and |e|^2 entering as the last two augmented terms -- the map is an
//              output and stays bit-equal to ATen's CPU cdist.
//   gx       : acc[pixel][dim]  += w[pixel][class] e[class][dim], rows = classes.
//   gE       : acc[dim][class]  += x[pixel][dim] w[pixel][class], rows = pixels (split over blocks, fp32 atomics;
//              deterministic mode: per-split partials with plain stores, added in a fixed order by seghead_slice_sum).
// The backward weight w (g / d, chained through the softmax and the normalisation when the class scores are
// given) is derived on the fly from g, d, the score and four per-pixel scalars: no N x K matrix is materialised.
#include "common.cuh"
#include "kernels.cuh"

namespace vqseg {

constexpr int kTThreads = 256;
constexpr int kTA = 128;             // a extent of a block tile (pixels of the map and of gx, dims of gE)
constexpr int kTB = 64;              // b extent (classes of the map and of gE, dims of gx)
constexpr int kTR = 32;              // contraction rows per staged step
constexpr int kSA = kTA + 4;         // shared row strides: 16-byte aligned rows, 4-way (not 32-way) transposed stores
constexpr int kSB = kTB + 4;

__device__ __forceinline__ int a_index(int ta, int i) { return (i < 4 ? 0 : 64) + 4 * ta + (i & 3); }

// acc[i][j] += a[r][a_index(ta, i)] * b[r][4 tb + j] for r in [r0, r1) in increasing r: per (i, j) one sequential
// fp32 FMA chain.
__device__ __forceinline__ void fma_rows(const float* __restrict__ sa, const float* __restrict__ sb, int r0, int r1,
                                         int ta, int tb, float (&acc)[8][4]) {
#pragma unroll 4
  for (int r = r0; r < r1; ++r) {
    const float4 a0 = *reinterpret_cast<const float4*>(sa + r * kSA + 4 * ta);
    const float4 a1 = *reinterpret_cast<const float4*>(sa + r * kSA + 64 + 4 * ta);
    const float4 b4 = *reinterpret_cast<const float4*>(sb + r * kSB + 4 * tb);
    const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
    const float b[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = __fmaf_rn(a[i], b[j], acc[i][j]);
  }
}

// The rest of chain_dist2 once the products of the open K-block [bs, ..) are in t: that block and any later ones
// (which hold only the augmented terms |x|^2 * 1 and 1 * |e|^2).  kb is normalised (0 < kb <= L).
template <bool IP>
__device__ __forceinline__ float chain_finish(float t, float c, int bs, int D, int kb, float xnorm, float enorm) {
  const int L = IP ? D : D + 2;
  bool first = bs == 0;
  for (int blk = bs; blk < L; blk += kb) {
    const int end = min(blk + kb, L);
    float s = IP ? -t : -2.f * t;                       // exact
    if (!IP && end > D) {
      if (blk <= D) s = __fadd_rn(s, xnorm);            // term D   : |x|^2 * 1
      if (end > D + 1) s = __fadd_rn(s, enorm);         // term D+1 : 1 * |e|^2
    }
    c = first ? s : __fadd_rn(c, s);
    first = false;
    t = 0.f;
  }
  return c;
}

// ---- forward: distance (or similarity) map, argmin / argmax, class counts, fused class scores -----------------------
// A block owns 128 pixels and sweeps all class tiles of 64 for them, so the epilogue can run over complete rows: after
// the last tile it re-reads its own freshly written (L2-resident) map rows for the argmin, the counts and the scores.
// |x|^2 (Euclidean) is accumulated from the staged x tiles during the first class tile in ATen's vectorized_inner_sum
// order (common.cuh, torch_order_sumsq_warp): one 32-dim tile is one "row" of its 32 accumulators; the cascade levels
// live in shared memory ([nlev][32][128]).
template <bool COSINE, bool SPLIT>
__global__ void __launch_bounds__(kTThreads, 2)
seghead_map_tiled_kernel(Rows x, const float* __restrict__ E, int K, int kb, int level_power, int nlev,
                         float* dist, long long oB, long long oP, long long oK, long long* __restrict__ idx_out,
                         unsigned long long* __restrict__ counts, float* __restrict__ score, int smem_counts) {
  extern __shared__ __align__(16) float tm_smem[];
  float* s_a = tm_smem;                                   // [kTR][kSA] x tile (d-major)
  float* s_b = s_a + kTR * kSA;                           // [kTR][kSB] prototype tile (d-major)
  float* s_xn = s_b + kTR * kSB;                          // [kTA] |x|^2
  float* s_en = s_xn + kTA;                               // [kTB] |e|^2 of the class tile
  long long* s_xoff = reinterpret_cast<long long*>(s_en + kTB);   // [kTA] pixel offsets into x
  long long* s_doff = s_xoff + kTA;                       // [kTA] pixel offsets into the maps
  int* s_cnt = reinterpret_cast<int*>(s_doff + kTA);      // [K] block histogram (smem_counts)
  float* s_sq = reinterpret_cast<float*>(s_cnt + (smem_counts ? ((K + 3) & ~3) : 0));   // [nlev][32][kTA]
  const int tid = threadIdx.x, ta = tid & 15, tb = tid >> 4;
  const int D = (int)x.D;
  const long long N = x.n_rows(), n0 = (long long)blockIdx.x * kTA;
  for (int p = tid; p < kTA; p += kTThreads) {
    long long b = 0, pp = 0;
    if (n0 + p < N) split_row(n0 + p, x.P, b, pp);
    s_xoff[p] = b * x.sB + pp * x.sP;
    s_doff[p] = b * oB + pp * oP;
  }
  if (smem_counts)
    for (int k = tid; k < K; k += kTThreads) s_cnt[k] = 0;
  if (!COSINE)
    for (int i = tid; i < nlev * 32 * kTA; i += kTThreads) s_sq[i] = 0.f;
  const bool d_fast = x.sD == 1 && x.sP != 1;             // packed rows: consecutive threads read consecutive dims
  const long long vec_size = D / 8, size_ilp = vec_size / 4;
  const long long lmask = (1ll << level_power) - 1;
  const int bs = ((D - 1) / kb) * kb;                     // K-block that holds the last product
  const int lane = tid & 31, warp = tid >> 5;
  for (int k0 = 0; k0 < K; k0 += kTB) {
    __syncthreads();                                      // previous tile's epilogue is done with s_en
    if (!COSINE) {
      for (int j = warp; j < kTB; j += kTThreads / 32) {  // |e_k|^2 in the same order, one warp per class
        float s = 0.f;
        if (k0 + j < K) {
          const float* row = E + (long long)(k0 + j) * D;
          s = torch_order_sumsq_warp([&](long long q) { const float v = __ldg(row + q); return __fmul_rn(v, v); }, D, lane);
        }
        if (lane == 0) s_en[j] = s;
      }
    }
    float t[8][4], c[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) { t[i][j] = 0.f; c[i][j] = 0.f; }
    for (int d0 = 0; d0 < D; d0 += kTR) {
      float xa[16], eb[8];
#pragma unroll
      for (int m = 0; m < 16; ++m) {
        const int p = d_fast ? (tid >> 5) + 8 * m : tid & 127, r = d_fast ? tid & 31 : (tid >> 7) + 2 * m;
        xa[m] = (n0 + p < N && d0 + r < D) ? __ldg(x.ptr + s_xoff[p] + (long long)(d0 + r) * x.sD) : 0.f;
      }
#pragma unroll
      for (int m = 0; m < 8; ++m) {
        const int j = (tid >> 5) + 8 * m, r = tid & 31;
        eb[m] = (k0 + j < K && d0 + r < D) ? __ldg(E + (long long)(k0 + j) * D + d0 + r) : 0.f;
      }
      __syncthreads();
#pragma unroll
      for (int m = 0; m < 16; ++m) {
        const int p = d_fast ? (tid >> 5) + 8 * m : tid & 127, r = d_fast ? tid & 31 : (tid >> 7) + 2 * m;
        s_a[r * kSA + p] = xa[m];
      }
#pragma unroll
      for (int m = 0; m < 8; ++m) s_b[(tid & 31) * kSB + (tid >> 5) + 8 * m] = eb[m];
      __syncthreads();
      const int R = min(kTR, D - d0);
      if (!COSINE && k0 == 0 && R == kTR) {
        // row d0 / 32 of ATen's sum: accumulator l of pixel p += x[p][d0 + l]^2, then the cascade
        const int p = tid & 127, h = tid >> 7;
        const long long done = d0 / kTR + 1;
#pragma unroll 4
        for (int l = 16 * h; l < 16 * h + 16; ++l) {
          const float v = s_a[l * kSA + p];
          float* a0 = s_sq + l * kTA + p;
          *a0 = __fadd_rn(*a0, __fmul_rn(v, v));
          if ((done & lmask) == 0) {
            float* a1 = a0 + 32 * kTA;
            *a1 = __fadd_rn(*a1, *a0); *a0 = 0.f;
            if ((done & (lmask << level_power)) == 0) {
              float* a2 = a1 + 32 * kTA;
              *a2 = __fadd_rn(*a2, *a1); *a1 = 0.f;
              if ((done & (lmask << (2 * level_power))) == 0) {
                float* a3 = a2 + 32 * kTA;
                *a3 = __fadd_rn(*a3, *a2); *a2 = 0.f;
              }
            }
          }
        }
      }
      for (int r = 0; r < R;) {
        int r1 = R;
        if (SPLIT) {                                      // restart the chains at MKL's K-block boundaries
          const int d = d0 + r;
          if (d > 0 && d % kb == 0) {
            const bool first = d == kb;
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const float s = COSINE ? -t[i][j] : -2.f * t[i][j];
                c[i][j] = first ? s : __fadd_rn(c[i][j], s);
                t[i][j] = 0.f;
              }
          }
          r1 = min(R, (d / kb + 1) * kb - d0);
        }
        fma_rows(s_a, s_b, r, r1, ta, tb, t);
        r = r1;
      }
    }
    if (!COSINE && k0 == 0) {
      // finish |x|^2: fold the cascade, the leftover 8-vectors into accumulators 0..7, the four partial vectors,
      // then 0 + scalar tail + partials in order.  The last (partial) x tile is still staged.
      __syncthreads();
      if (tid < kTA) {
        const int p = tid, dl = ((D - 1) / kTR) * kTR;
        auto acc_of = [&](int l) {
          float a = s_sq[l * kTA + p];
          for (int lv = 1; lv < nlev; ++lv) a = __fadd_rn(a, s_sq[(lv * 32 + l) * kTA + p]);
          if (l < 8)
            for (long long v = size_ilp * 4; v < vec_size; ++v) {
              const float q = s_a[(int)(v * 8 + l - dl) * kSA + p];
              a = __fadd_rn(a, __fmul_rn(q, q));
            }
          return a;
        };
        float f = 0.f;
        for (long long q = vec_size * 8; q < D; ++q) {
          const float v = s_a[(int)(q - dl) * kSA + p];
          f = __fadd_rn(f, __fmul_rn(v, v));
        }
        for (int l = 0; l < 8; ++l) {
          float pl = acc_of(l);
          pl = __fadd_rn(pl, acc_of(l + 8)); pl = __fadd_rn(pl, acc_of(l + 16)); pl = __fadd_rn(pl, acc_of(l + 24));
          f = __fadd_rn(f, pl);
        }
        s_xn[p] = f;
      }
      __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int p = a_index(ta, i);
      if (n0 + p >= N) continue;
      const float xnorm = COSINE ? 0.f : s_xn[p];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int k = k0 + 4 * tb + j;
        if (k >= K) continue;
        const float cc = chain_finish<COSINE>(t[i][j], c[i][j], bs, D, kb, xnorm, COSINE ? 0.f : s_en[4 * tb + j]);
        dist[s_doff[p] + (long long)k * oK] = COSINE ? -cc : __fsqrt_rn(fmaxf(cc, 0.f));
      }
    }
  }
  // ---- epilogue over complete rows: the block's map rows are written (block-visible after the barrier) ----------
  __syncthreads();
  if (tid < kTA && n0 + tid < N) {
    const float* dr = dist + s_doff[tid];
    float best = 0.f, sum = 0.f;
    int best_k = 0;
#pragma unroll 8
    for (int k = 0; k < K; ++k) {
      const float v = dr[(long long)k * oK];
      if (k == 0 || (COSINE ? v > best : v < best)) { best = v; best_k = k; }   // first index wins
      if (!COSINE) sum = __fadd_rn(sum, v);
    }
    if (!COSINE && score) {
      // class scores softmax_k(1 - d_k / sum_j d_j) (vq_segmentation_head.py:245-247); 1 - d / s is monotone in d,
      // so its maximum is the term of the smallest distance
      const float tmax = __fsub_rn(1.f, __fdiv_rn(best, sum));
      float esum = 0.f;
#pragma unroll 8
      for (int k = 0; k < K; ++k) esum += expf(__fsub_rn(1.f, __fdiv_rn(dr[(long long)k * oK], sum)) - tmax);
      float* sr = score + s_doff[tid];
#pragma unroll 8
      for (int k = 0; k < K; ++k)
        sr[(long long)k * oK] = expf(__fsub_rn(1.f, __fdiv_rn(dr[(long long)k * oK], sum)) - tmax) / esum;
    }
    if (idx_out) idx_out[n0 + tid] = best_k;
    if (counts) {
      if (smem_counts) atomicAdd(&s_cnt[best_k], 1);
      else atomicAdd(counts + best_k, 1ull);
    }
  }
  if (counts && smem_counts) {
    __syncthreads();
    for (int k = tid; k < K; k += kTThreads)
      if (s_cnt[k] != 0) atomicAdd(counts + k, (unsigned long long)s_cnt[k]);
  }
}

constexpr int kTiledSmemCountsMax = 4096;    // larger K: the class counts go straight to global atomics

static int ceil_log2(long long v) {
  int cl = 0;
  while ((1ll << cl) < v) ++cl;
  return cl;
}

int launch_seghead_map_tiled(const Rows& x, const float* E, int K, bool cosine, int kb, float* dist, long long oB,
                             long long oP, long long oK, long long* idx, unsigned long long* counts, float* score,
                             cudaStream_t st) {
  const int D = (int)x.D;
  // ATen's cascade geometry (torch_order_sumsq_warp): levels of 2^level_power rows of 32 elements
  const long long size_ilp = D / 32;
  const int level_power = ceil_log2(size_ilp) / 4 > 4 ? ceil_log2(size_ilp) / 4 : 4;
  const long long step = 1ll << level_power;
  int nlev = 1;
  for (long long s = step; nlev < 4 && size_ilp >= s; s *= step) ++nlev;
  const int smem_counts = counts && K <= kTiledSmemCountsMax;
  const size_t smem = (size_t)(kTR * kSA + kTR * kSB + kTA + kTB) * sizeof(float) + 2 * kTA * sizeof(long long) +
                      (smem_counts ? (size_t)((K + 3) & ~3) * sizeof(int) : 0) +
                      (cosine ? 0 : (size_t)nlev * 32 * kTA * sizeof(float));
  const unsigned grid = (unsigned)((x.n_rows() + kTA - 1) / kTA);
  const bool split = kb < (cosine ? D : D + 2);
  auto go = [&](auto kernel, size_t (&state)[kMaxDevices]) -> int {
    int rc = ensure_dynamic_smem(kernel, smem, state);
    if (rc) return rc;
    kernel<<<grid, kTThreads, smem, st>>>(x, E, K, kb, level_power, nlev, dist, oB, oP, oK, idx, counts, score, smem_counts);
    VQSEG_LAUNCH_CHECK();
    return 0;
  };
  static size_t s00[kMaxDevices], s01[kMaxDevices], s10[kMaxDevices], s11[kMaxDevices];
  if (cosine) return split ? go(seghead_map_tiled_kernel<true, true>, s11) : go(seghead_map_tiled_kernel<true, false>, s10);
  return split ? go(seghead_map_tiled_kernel<false, true>, s01) : go(seghead_map_tiled_kernel<false, false>, s00);
}

// ---- backward --------------------------------------------------------------------------------------------------------
// Per-pixel scalars (one float4 per pixel in the caller's workspace):
//   Euclidean: (dot = sum_k g_k s_k, A = (sum_k g_t[k] d_k) / S, 1 / S, sum_k w_k), S = sum_k d_k (score path only for
//              the first three);  cosine: (dot = sum_k g_k sim_k = <xn, gxn>, 1 / max(|x|, 1e-12), 0, 0).
// The weight of one (pixel, class) pair, same algebra as dist_map_bwd_kernel (seghead.cu): with the score,
//   g_t = s (g - dot),  g_d = (A - g_t) / S;  then w = g_d / d (0 where d == 0).
__device__ __forceinline__ float seg_w(float gk, float dv, float sc, const float4& s, bool with_score) {
  if (with_score) {
    const float gt = sc * (gk - s.x);
    gk = (s.y - gt) * s.z;
  }
  return dv == 0.f ? 0.f : __fdiv_rn(gk, dv);
}

__global__ void __launch_bounds__(kTThreads) seghead_bwd_scalars_kernel(Rows x, int K, const float* __restrict__ g,
                                                                        const float* __restrict__ dist, long long oB,
                                                                        long long oP, long long oK,
                                                                        const float* __restrict__ score, int cosine,
                                                                        float4* __restrict__ scal) {
  const long long n = (long long)blockIdx.x * kTThreads + threadIdx.x;
  if (n >= x.n_rows()) return;
  long long b, pp;
  split_row(n, x.P, b, pp);
  const long long o = b * oB + pp * oP;
  if (cosine) {
    float dot = 0.f, ss = 0.f;
    for (int k = 0; k < K; ++k) dot = fmaf(__ldg(g + o + (long long)k * oK), __ldg(dist + o + (long long)k * oK), dot);
    const float* xr = x.ptr + b * x.sB + pp * x.sP;
    for (long long d = 0; d < x.D; ++d) { const float v = __ldg(xr + d * x.sD); ss = fmaf(v, v, ss); }
    scal[n] = make_float4(dot, 1.f / fmaxf(sqrtf(ss), 1e-12f), 0.f, 0.f);
    return;
  }
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  if (score) {
    float dot = 0.f, ssum = 0.f, gtd = 0.f;
    for (int k = 0; k < K; ++k) {
      const long long ok = o + (long long)k * oK;
      dot = fmaf(__ldg(g + ok), __ldg(score + ok), dot);
      ssum += __ldg(dist + ok);
    }
    for (int k = 0; k < K; ++k) {
      const long long ok = o + (long long)k * oK;
      gtd = fmaf(__ldg(score + ok) * (__ldg(g + ok) - dot), __ldg(dist + ok), gtd);
    }
    const float inv = ssum != 0.f ? 1.f / ssum : 0.f;
    s = make_float4(dot, gtd * inv, inv, 0.f);
  }
  float wsum = 0.f;
  for (int k = 0; k < K; ++k) {
    const long long ok = o + (long long)k * oK;
    wsum += seg_w(__ldg(g + ok), __ldg(dist + ok), score ? __ldg(score + ok) : 0.f, s, score != nullptr);
  }
  s.w = wsum;
  scal[n] = s;
}

// gx[n, :] = x[n, :] sum_k w[n, k] - sum_k w[n, k] e_k        (Euclidean)
//          = (gxn - xn <xn, gxn>) / |x|,  gxn = sum_k g[n, k] e_k   (cosine)
// Block tile: 128 pixels x 64 dims, contraction over the classes.
template <bool COSINE>
__global__ void __launch_bounds__(kTThreads, 2)
seghead_bwd_gx_kernel(Rows x, const float* __restrict__ E, int K, const float* __restrict__ g, const float* __restrict__ dist,
                      long long oB, long long oP, long long oK, const float* __restrict__ score,
                      const float4* __restrict__ scal, RowsOut gx) {
  __shared__ __align__(16) float s_a[kTR * kSA];          // [class][pixel] weights
  __shared__ __align__(16) float s_b[kTR * kSB];          // [class][dim] prototypes
  __shared__ long long s_moff[kTA], s_xoff[kTA], s_goff[kTA];
  __shared__ float4 s_scal[kTA];
  const int tid = threadIdx.x, ta = tid & 15, tb = tid >> 4;
  const int D = (int)x.D;
  const long long N = x.n_rows(), n0 = (long long)blockIdx.x * kTA;
  const int dd0 = blockIdx.y * kTB;
  for (int p = tid; p < kTA; p += kTThreads) {
    long long b = 0, pp = 0;
    const bool in = n0 + p < N;
    if (in) split_row(n0 + p, x.P, b, pp);
    s_moff[p] = b * oB + pp * oP;
    s_xoff[p] = b * x.sB + pp * x.sP;
    s_goff[p] = b * gx.sB + pp * gx.sP;
    s_scal[p] = in ? scal[n0 + p] : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  __syncthreads();
  float acc[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  for (int k0 = 0; k0 < K; k0 += kTR) {
    float wa[16], eb[8];
#pragma unroll
    for (int m = 0; m < 16; ++m) {
      const int p = tid & 127, k = k0 + (tid >> 7) + 2 * m;
      float w = 0.f;
      if (n0 + p < N && k < K) {
        const long long o = s_moff[p] + (long long)k * oK;
        w = COSINE ? __ldg(g + o) : seg_w(__ldg(g + o), __ldg(dist + o), score ? __ldg(score + o) : 0.f, s_scal[p], score != nullptr);
      }
      wa[m] = w;
    }
#pragma unroll
    for (int m = 0; m < 8; ++m) {
      const int j = tid & 63, k = k0 + (tid >> 6) + 4 * m;
      eb[m] = (k < K && dd0 + j < D) ? __ldg(E + (long long)k * D + dd0 + j) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int m = 0; m < 16; ++m) s_a[((tid >> 7) + 2 * m) * kSA + (tid & 127)] = wa[m];
#pragma unroll
    for (int m = 0; m < 8; ++m) s_b[((tid >> 6) + 4 * m) * kSB + (tid & 63)] = eb[m];
    __syncthreads();
    fma_rows(s_a, s_b, 0, min(kTR, K - k0), ta, tb, acc);
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int p = a_index(ta, i);
    if (n0 + p >= N) continue;
    const float4 s = s_scal[p];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int d = dd0 + 4 * tb + j;
      if (d >= D) continue;
      const float xv = __ldg(x.ptr + s_xoff[p] + (long long)d * x.sD);
      gx.ptr[s_goff[p] + (long long)d * gx.sD] = COSINE ? (acc[i][j] - (xv * s.y) * s.x) * s.y : xv * s.w - acc[i][j];
    }
  }
}

// gE[k, :] += sum_{n in this block's pixels} w[n, k] (e_k - x[n, :])   (Euclidean)
//          += sum_n g[n, k] xn[n, :]                                    (cosine)
// Block tile: 128 dims x 64 classes, contraction over a range of pixels (grid.z splits the pixels), fp32 atomics.
// DET: split z stores its sum (zeros included) to gE + z K D instead: the caller's partials, or gE itself when
// there is one split.
template <bool COSINE, bool DET>
__global__ void __launch_bounds__(kTThreads, 2)
seghead_bwd_ge_kernel(Rows x, const float* __restrict__ E, int K, const float* __restrict__ g, const float* __restrict__ dist,
                      long long oB, long long oP, long long oK, const float* __restrict__ score,
                      const float4* __restrict__ scal, float* __restrict__ gE, int chunks_per_split) {
  __shared__ __align__(16) float s_a[kTR * kSA];          // [pixel][dim] features
  __shared__ __align__(16) float s_b[kTR * kSB];          // [pixel][class] weights
  __shared__ long long s_xo[kTR], s_mo[kTR];
  __shared__ float4 s_sc[kTR];
  __shared__ float s_ws[kTB];
  const int tid = threadIdx.x, ta = tid & 15, tb = tid >> 4;
  const int D = (int)x.D;
  const long long N = x.n_rows();
  const int dd0 = blockIdx.x * kTA, k0 = blockIdx.y * kTB;
  const long long n_chunks = (N + kTR - 1) / kTR;
  const long long c_begin = (long long)blockIdx.z * chunks_per_split;
  const long long c_end = min(c_begin + chunks_per_split, n_chunks);
  const bool d_fast = x.sD == 1 && x.sP != 1;
  float acc[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  float wsacc = 0.f;
  for (long long ch = c_begin; ch < c_end; ++ch) {
    const long long nb = ch * kTR;
    __syncthreads();                                      // the previous chunk's tiles and offsets are consumed
    if (tid < kTR) {
      long long b = 0, pp = 0;
      const bool in = nb + tid < N;
      if (in) split_row(nb + tid, x.P, b, pp);
      s_xo[tid] = b * x.sB + pp * x.sP;
      s_mo[tid] = b * oB + pp * oP;
      s_sc[tid] = in ? scal[nb + tid] : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    __syncthreads();
    float xa[16], wb[8];
#pragma unroll
    for (int m = 0; m < 16; ++m) {
      const int i = d_fast ? tid & 127 : (tid >> 5) + 8 * m, r = d_fast ? (tid >> 7) + 2 * m : tid & 31;
      float v = (nb + r < N && dd0 + i < D) ? __ldg(x.ptr + s_xo[r] + (long long)(dd0 + i) * x.sD) : 0.f;
      if (COSINE) v *= s_sc[r].y;                         // the prototype gradient works on xn
      xa[m] = v;
    }
#pragma unroll
    for (int m = 0; m < 8; ++m) {
      const int j = (tid >> 5) + 8 * m, r = tid & 31, k = k0 + j;
      float w = 0.f;
      if (nb + r < N && k < K) {
        const long long o = s_mo[r] + (long long)k * oK;
        w = COSINE ? __ldg(g + o) : seg_w(__ldg(g + o), __ldg(dist + o), score ? __ldg(score + o) : 0.f, s_sc[r], score != nullptr);
      }
      wb[m] = w;
    }
#pragma unroll
    for (int m = 0; m < 16; ++m) {
      const int i = d_fast ? tid & 127 : (tid >> 5) + 8 * m, r = d_fast ? (tid >> 7) + 2 * m : tid & 31;
      s_a[r * kSA + i] = xa[m];
    }
#pragma unroll
    for (int m = 0; m < 8; ++m) s_b[(tid & 31) * kSB + (tid >> 5) + 8 * m] = wb[m];
    __syncthreads();
    if (!COSINE && tid < kTB)
      for (int r = 0; r < kTR; ++r) wsacc += s_b[r * kSB + tid];
    fma_rows(s_a, s_b, 0, kTR, ta, tb, acc);
  }
  if (!COSINE && tid < kTB) s_ws[tid] = wsacc;
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int d = dd0 + a_index(ta, i);
    if (d >= D) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = k0 + 4 * tb + j;
      if (k >= K) continue;
      const long long o = (long long)k * D + d;
      const float r = COSINE ? acc[i][j] : __ldg(E + o) * s_ws[4 * tb + j] - acc[i][j];
      if (DET) gE[(long long)blockIdx.z * K * D + o] = r;
      else if (r != 0.f) atomicAdd(gE + o, r);
    }
  }
}

// The pixel split of the gE kernel: ~4 blocks per SM over the (dims x classes) tiles, at most `max_splits` splits.
// (splits, chunks per split) with every split non-empty.
static void ge_split(long long N, int K, int D, long long sms, long long max_splits, long long& splits, long long& cps) {
  const long long tiles = (long long)((D + kTA - 1) / kTA) * ((K + kTB - 1) / kTB);
  const long long n_chunks = (N + kTR - 1) / kTR;
  splits = (4ll * sms + tiles - 1) / tiles;
  if (splits > n_chunks) splits = n_chunks;
  if (splits > 65535) splits = 65535;
  if (splits > max_splits) splits = max_splits;
  cps = (n_chunks + splits - 1) / splits;
  splits = (n_chunks + cps - 1) / cps;
}

// Deterministic mode: the split is a function of the shape alone (a B200's SM count in place of the device's), and
// the partials stay within kSegheadDetPartialBytes.
static void ge_split_det(long long N, int K, int D, long long& splits, long long& cps) {
  ge_split(N, K, D, kSegheadDetSms, seghead_det_max_slices(K, D), splits, cps);
}

size_t seghead_bwd_tiled_workspace_bytes(long long n_rows, int K, int D, bool det) {
  size_t bytes = (size_t)n_rows * sizeof(float4);
  if (det && n_rows > 0 && K > 0 && D > 0) {
    long long splits, cps;
    ge_split_det(n_rows, K, D, splits, cps);
    if (splits > 1) bytes += (size_t)splits * K * D * sizeof(float);
  }
  return bytes;
}

// out[i] = sum_z part[z n + i] over the S slices in a fixed order that depends on S alone: group j of G = min(S, 32)
// adds its run of consecutive slices [j R, (j + 1) R) in ascending order (R = ceil(S / G)), then the G run sums are
// added in ascending j.  (One ascending chain of S dependent loads per element would be latency-bound when K D is
// small and S large: the 3-class head has 96 elements and 2048 slices.)
__global__ void seghead_slice_sum_kernel(const float* __restrict__ part, long long n, int S, int R, float* __restrict__ out) {
  extern __shared__ float ss_run[];                       // [G][32]
  const int e = threadIdx.x & 31, j = threadIdx.x >> 5, G = blockDim.x >> 5;
  const long long i = (long long)blockIdx.x * 32 + e;
  float s = 0.f;
  if (i < n) {
    const int z0 = j * R, z1 = min(z0 + R, S);
    if (z0 < z1) {
      s = part[(long long)z0 * n + i];
#pragma unroll 8
      for (int z = z0 + 1; z < z1; ++z) s = __fadd_rn(s, part[(long long)z * n + i]);
    }
  }
  ss_run[j * 32 + e] = s;
  __syncthreads();
  if (j == 0 && i < n) {
    float t = ss_run[e];
    for (int q = 1; q < G; ++q)
      if (q * R < S) t = __fadd_rn(t, ss_run[q * 32 + e]);
    out[i] = t;
  }
}

int launch_seghead_slice_sum(const float* part, long long n, int S, float* out, cudaStream_t st) {
  const int G = S < 32 ? S : 32, R = (S + G - 1) / G;
  const long long blocks = (n + 31) / 32;
  seghead_slice_sum_kernel<<<(unsigned)blocks, 32 * G, (size_t)G * 32 * sizeof(float), st>>>(part, n, S, R, out);
  VQSEG_LAUNCH_CHECK();
  return 0;
}

int launch_seghead_map_bwd_tiled(const Rows& x, const float* E, int K, bool cosine, const float* g, const float* dist,
                                 long long oB, long long oP, long long oK, const float* score, const RowsOut& gx,
                                 float* gE, bool det, void* ws, cudaStream_t st) {
  const long long N = x.n_rows();
  const int D = (int)x.D;
  float4* scal = static_cast<float4*>(ws);
  seghead_bwd_scalars_kernel<<<(unsigned)((N + kTThreads - 1) / kTThreads), kTThreads, 0, st>>>(
      x, K, g, dist, oB, oP, oK, cosine ? nullptr : score, cosine ? 1 : 0, scal);
  VQSEG_LAUNCH_CHECK();
  const dim3 ggx((unsigned)((N + kTA - 1) / kTA), (unsigned)((D + kTB - 1) / kTB));
  if (cosine) seghead_bwd_gx_kernel<true><<<ggx, kTThreads, 0, st>>>(x, E, K, g, dist, oB, oP, oK, nullptr, scal, gx);
  else seghead_bwd_gx_kernel<false><<<ggx, kTThreads, 0, st>>>(x, E, K, g, dist, oB, oP, oK, score, scal, gx);
  VQSEG_LAUNCH_CHECK();
  long long splits, cps;
  if (det) ge_split_det(N, K, D, splits, cps);
  else ge_split(N, K, D, num_sms(), 65535, splits, cps);
  const dim3 gge((unsigned)((D + kTA - 1) / kTA), (unsigned)((K + kTB - 1) / kTB), (unsigned)splits);
  const float* sc = cosine ? nullptr : score;
  if (!det) {
    if (cosine) seghead_bwd_ge_kernel<true, false><<<gge, kTThreads, 0, st>>>(x, E, K, g, dist, oB, oP, oK, sc, scal, gE, (int)cps);
    else seghead_bwd_ge_kernel<false, false><<<gge, kTThreads, 0, st>>>(x, E, K, g, dist, oB, oP, oK, sc, scal, gE, (int)cps);
    VQSEG_LAUNCH_CHECK();
    return 0;
  }
  float* part = splits > 1 ? reinterpret_cast<float*>(scal + N) : gE;
  if (cosine) seghead_bwd_ge_kernel<true, true><<<gge, kTThreads, 0, st>>>(x, E, K, g, dist, oB, oP, oK, sc, scal, part, (int)cps);
  else seghead_bwd_ge_kernel<false, true><<<gge, kTThreads, 0, st>>>(x, E, K, g, dist, oB, oP, oK, sc, scal, part, (int)cps);
  VQSEG_LAUNCH_CHECK();
  return splits > 1 ? launch_seghead_slice_sum(part, (long long)K * D, (int)splits, gE, st) : 0;
}

}  // namespace vqseg
