// Distance map of the VQ segmentation head (SURVEY.md section 8f rank 3).
//
// Reference call sites (models/modules/vq_segmentation_head.py): EuclideanSegHead.forward
// `torch.cdist(flatten_x, weight, p=2)` + `argmin` + `bincount` (:167-176), CosinesimSegHead.forward
// `einsum('n d, e d -> n e')` + `argmax` (:104-107); the wrapper turns the map into class scores (:243-249), so
// unlike the encoder-side quantizer the full (pixels x classes) map is an OUTPUT and carries gradient
// (torch.cdist backward: grad * (x - e) / d, 0 where d == 0).
//
// Shapes: K = number of classes (3 in the reference configs), D = last decoder width (16..64), N = B*H*W
// pixels (10^5..10^6): HBM-bound, 4ND bytes in, 4NK + 8N out.  One THREAD owns one pixel (consecutive threads =
// consecutive pixels: coalesced for NCHW features); the prototypes sit in shared memory and are read as
// broadcasts; the K chains and the 32 torch-order accumulators of |x|^2 live in registers.  The arithmetic is
// the exact scorer's (exact.cu): one fp32 FMA chain per (pixel, class) in increasing d, the (D+2)-term augmented
// form of ATen's _euclidean_dist, |.|^2 in ATen's CPU summation order -- bit-equal to the CPU reference.
// Limits (loud errors beyond): K <= 32, D + 2 <= 384 (single-chain regime of the CPU GEMM), K*D*4 <= 96 KiB.
#include "common.cuh"
#include "kernels.cuh"

namespace vqseg {

constexpr int kDmThreads = 128;
constexpr int kDmXStride = kDmThreads + 4;     // backward: row stride of the staged x tile (words)

// fl(v*v) summed in ATen's vectorized_inner_sum order for D < 512 (no cascade spill): element j goes to
// accumulator j % 32 for the first (D/32)*32 elements, leftover 8-vectors to accumulators 0..7, then
// p[l] = a[l] + a[l+8] + a[l+16] + a[l+24], then 0 + scalar tail + p[0] + ... + p[7].
struct TorchSumSq {
  float a[32];
  float tail;
  __device__ __forceinline__ void init() {
#pragma unroll
    for (int i = 0; i < 32; ++i) a[i] = 0.f;
    tail = 0.f;
  }
  __device__ __forceinline__ float finish() const {
    float f = tail;
#pragma unroll
    for (int l = 0; l < 8; ++l) {
      float p = a[l];
      p = __fadd_rn(p, a[l + 8]); p = __fadd_rn(p, a[l + 16]); p = __fadd_rn(p, a[l + 24]);
      f = __fadd_rn(f, p);
    }
    return f;
  }
};

// |e_k|^2 in the same order, one warp per prototype (block-cooperative, results in s_en[K])
__device__ __forceinline__ void stage_prototypes(const float* __restrict__ E, int K, int D, float* s_e, float* s_en) {
  for (int i = threadIdx.x; i < K * D; i += blockDim.x) s_e[i] = __ldg(E + i);
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int k = warp; k < K; k += blockDim.x >> 5) {
    const float* row = s_e + k * D;
    const float s = torch_order_sumsq_warp([&](long long j) { float v = row[j]; return __fmul_rn(v, v); }, D, lane);
    if (lane == 0) s_en[k] = s;
  }
  __syncthreads();
}

template <int KMAX, bool COSINE>
__global__ void __launch_bounds__(kDmThreads) dist_map_kernel(Rows x, const float* __restrict__ E, int K,
                                                             float* __restrict__ dist, long long oB, long long oP, long long oK,
                                                             long long* __restrict__ idx_out,
                                                             unsigned long long* __restrict__ counts,
                                                             float* __restrict__ score) {
  extern __shared__ __align__(16) float dm_smem[];
  const int D = (int)x.D;
  float* s_e = dm_smem;                      // [K][D]
  float* s_en = s_e + K * D;                 // [K]
  int* s_cnt = reinterpret_cast<int*>(s_en + K);   // [KMAX]
  if (threadIdx.x < KMAX) s_cnt[threadIdx.x] = 0;
  stage_prototypes(E, K, D, s_e, s_en);
  const long long n_rows = x.n_rows();
  const long long n = (long long)blockIdx.x * kDmThreads + threadIdx.x;
  if (n < n_rows) {
    long long b, pp;
    split_row(n, x.P, b, pp);
    const float* xr = x.ptr + b * x.sB + pp * x.sP;
    TorchSumSq sq;
    sq.init();
    float t[KMAX];
#pragma unroll
    for (int k = 0; k < KMAX; ++k) t[k] = 0.f;
    const int vec_size = D / 8, size_ilp = vec_size / 4;
    auto step = [&](int d, float xv) {
#pragma unroll
      for (int k = 0; k < KMAX; ++k)
        if (k < K) t[k] = __fmaf_rn(xv, s_e[k * D + d], t[k]);
    };
    const bool v4 = (D & 3) == 0;              // prototype rows 16-byte aligned: one LDS.128 feeds four chain steps
    for (int i = 0; i < size_ilp; ++i) {
      float xv[32];
#pragma unroll
      for (int u = 0; u < 32; ++u) xv[u] = __ldg(xr + (long long)(32 * i + u) * x.sD);
      if (v4) {
#pragma unroll
        for (int u = 0; u < 32; u += 4) {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (!COSINE) sq.a[u + j] = __fadd_rn(sq.a[u + j], __fmul_rn(xv[u + j], xv[u + j]));
#pragma unroll
          for (int k = 0; k < KMAX; ++k)
            if (k < K) {                           // (the scalar broadcast loads made the kernel issue-bound: one LDS per FMA)
              const float4 e4 = *reinterpret_cast<const float4*>(s_e + k * D + 32 * i + u);
              t[k] = __fmaf_rn(xv[u], e4.x, t[k]); t[k] = __fmaf_rn(xv[u + 1], e4.y, t[k]);
              t[k] = __fmaf_rn(xv[u + 2], e4.z, t[k]); t[k] = __fmaf_rn(xv[u + 3], e4.w, t[k]);
            }
        }
      } else {
#pragma unroll
        for (int u = 0; u < 32; ++u) {
          if (!COSINE) sq.a[u] = __fadd_rn(sq.a[u], __fmul_rn(xv[u], xv[u]));
          step(32 * i + u, xv[u]);
        }
      }
    }
    for (int v = size_ilp * 4; v < vec_size; ++v) {
      float xv[8];
#pragma unroll
      for (int l = 0; l < 8; ++l) xv[l] = __ldg(xr + (long long)(8 * v + l) * x.sD);
#pragma unroll
      for (int l = 0; l < 8; ++l) {
        if (!COSINE) sq.a[l] = __fadd_rn(sq.a[l], __fmul_rn(xv[l], xv[l]));
        step(8 * v + l, xv[l]);
      }
    }
    for (int d = vec_size * 8; d < D; ++d) {
      const float xv = __ldg(xr + (long long)d * x.sD);
      if (!COSINE) sq.tail = __fadd_rn(sq.tail, __fmul_rn(xv, xv));
      step(d, xv);
    }
    const float xnorm = COSINE ? 0.f : sq.finish();
    float best = 0.f;
    int best_k = 0;
    float* dr = dist + b * oB + pp * oP;
    float dk[KMAX];
#pragma unroll
    for (int k = 0; k < KMAX; ++k) {
      dk[k] = 0.f;
      if (k < K) {
        float v;
        if (COSINE) {
          v = t[k];                                            // similarity: argmax, first index wins
          if (k == 0 || v > best) { best = v; best_k = k; }
        } else {
          float c = -2.f * t[k];                               // exact (power of two)
          c = __fadd_rn(c, xnorm);                             // term D   : |x|^2 * 1
          c = __fadd_rn(c, s_en[k]);                           // term D+1 : 1 * |e|^2
          v = __fsqrt_rn(fmaxf(c, 0.f));
          if (k == 0 || v < best) { best = v; best_k = k; }
        }
        dr[(long long)k * oK] = v;
        dk[k] = v;
      }
    }
    if (!COSINE && score) {
      // class scores of the Euclidean head: softmax_k(1 - d_k / sum_j d_j)   (vq_segmentation_head.py:245-247)
      float sum = 0.f;
#pragma unroll
      for (int k = 0; k < KMAX; ++k) if (k < K) sum = __fadd_rn(sum, dk[k]);
      float tk[KMAX], tmax = -3.0e38f;
#pragma unroll
      for (int k = 0; k < KMAX; ++k) {
        tk[k] = (k < K) ? __fsub_rn(1.f, __fdiv_rn(dk[k], sum)) : -3.0e38f;
        tmax = fmaxf(tmax, tk[k]);
      }
      float esum = 0.f;
#pragma unroll
      for (int k = 0; k < KMAX; ++k) {
        tk[k] = (k < K) ? expf(tk[k] - tmax) : 0.f;
        esum += tk[k];
      }
      float* sr = score + b * oB + pp * oP;
#pragma unroll
      for (int k = 0; k < KMAX; ++k) if (k < K) sr[(long long)k * oK] = tk[k] / esum;
    }
    if (idx_out) idx_out[n] = best_k;
    if (counts) atomicAdd(&s_cnt[best_k], 1);
  }
  __syncthreads();
  if (counts && threadIdx.x < K && s_cnt[threadIdx.x] != 0)
    atomicAdd(counts + threadIdx.x, (unsigned long long)s_cnt[threadIdx.x]);
}

// backward of the Euclidean map: w = g / d (0 where d == 0);  gx[n,:] = sum_k w[n,k] (x[n,:] - e_k);
// gE[k,:] = sum_n w[n,k] (e_k - x[n,:]) = e_k * sum_n w[n,k] - sum_n w[n,k] x[n,:].
// A block owns 128 pixels.  Per chunk of 32 dims every thread (= pixel) loads its 32 values once, writes gx, and
// parks them in a padded smem tile; then thread (k, d) of the block reduces sum_p w[k][p] * x[p][d] over the 128
// pixels straight from shared memory (no shuffles) and issues ONE global atomic per (block, k, d).
// DET: the block walks `tiles_per_block` consecutive tiles instead and keeps its (k, d) sums in its own slice
// gE + blockIdx.x K D with plain stores (thread (k, d) owns the same element in every tile), tiles in ascending order.
template <int KMAX, bool DET>
__global__ void __launch_bounds__(kDmThreads) dist_map_bwd_kernel(Rows x, const float* __restrict__ E, int K,
                                                                 const float* __restrict__ g, const float* __restrict__ dist,
                                                                 long long oB, long long oP, long long oK,
                                                                 RowsOut gx, float* __restrict__ gE,
                                                                 const float* __restrict__ score, int cosine,
                                                                 int tiles_per_block) {
  // cosine != 0: backward of sim[n,k] = <x_n / max(|x_n|, 1e-12), e_k> (CosinesimSegHead, vq_segmentation_head.py:
  // 97-104) instead: w = g;  gxn = sum_k w_k e_k;  gx = (gxn - xn <xn, gxn>) / |x|;  gE[k,:] = sum_n w[n,k] xn[n,:]
  // (`dist` is not read).
  extern __shared__ __align__(16) float dmb_smem[];
  const int D = (int)x.D;
  float* s_e = dmb_smem;                          // [K][D]
  float* s_w = s_e + ((K * D + 3) & ~3);          // [K][128] weights of this block's pixels (16-byte aligned rows)
  float* s_ws = s_w + K * kDmThreads;             // [K] sum_p w[k][p]
  float* s_x = s_ws + KMAX;                       // [32][kDmXStride] tile of x (16-byte aligned rows; KMAX % 4 == 0)
  for (int i = threadIdx.x; i < K * D; i += blockDim.x) s_e[i] = __ldg(E + i);
  const long long n_rows = x.n_rows();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long t0 = DET ? (long long)blockIdx.x * tiles_per_block : blockIdx.x;
  const long long t1 = DET ? min(t0 + tiles_per_block, (n_rows + kDmThreads - 1) / kDmThreads) : t0 + 1;
  float* gEb = DET ? gE + (long long)blockIdx.x * K * D : gE;
  for (long long tile = t0; tile < t1; ++tile) {
    if (DET && tile > t0) __syncthreads();          // the previous tile is done with s_w, s_ws and s_x
    const long long n = tile * kDmThreads + threadIdx.x;
    const bool in = n < n_rows;
    float w[KMAX];
    float wsum = 0.f;
    long long b = 0, pp = 0;
    if (in) split_row(n, x.P, b, pp);
    {
      float gk[KMAX], dv[KMAX];
#pragma unroll
      for (int k = 0; k < KMAX; ++k) {
        gk[k] = 0.f; dv[k] = 0.f;
        if (in && k < K) {
          const long long o = b * oB + pp * oP + (long long)k * oK;
          dv[k] = cosine ? 1.f : __ldg(dist + o);
          gk[k] = __ldg(g + o);
        }
      }
      if (score) {
        // g arrives w.r.t. score = softmax_k(t), t_k = 1 - d_k / s, s = sum_j d_j:
        //   g_t[k] = score_k (g_k - sum_j g_j score_j);   g_d[j] = -g_t[j] / s + (sum_k g_t[k] d_k) / s^2
        float sc[KMAX], dot = 0.f, ssum = 0.f;
#pragma unroll
        for (int k = 0; k < KMAX; ++k) {
          sc[k] = (in && k < K) ? __ldg(score + b * oB + pp * oP + (long long)k * oK) : 0.f;
          dot = fmaf(gk[k], sc[k], dot);
          ssum += dv[k];
        }
        float gtd = 0.f;
#pragma unroll
        for (int k = 0; k < KMAX; ++k) { gk[k] = sc[k] * (gk[k] - dot); gtd = fmaf(gk[k], dv[k], gtd); }
        const float inv = ssum != 0.f ? 1.f / ssum : 0.f;
#pragma unroll
        for (int k = 0; k < KMAX; ++k) gk[k] = (gtd * inv - gk[k]) * inv;
      }
#pragma unroll
      for (int k = 0; k < KMAX; ++k) {
        w[k] = 0.f;
        if (k < K) {
          if (in) w[k] = cosine ? gk[k] : (dv[k] == 0.f ? 0.f : __fdiv_rn(gk[k], dv[k]));
          s_w[k * kDmThreads + threadIdx.x] = w[k];
          wsum += w[k];
        }
      }
    }
    __syncthreads();
    // s_ws[k] = sum over the block's pixels (fixed order: warp tree, then the 4 warp sums)
    for (int k = warp; k < K; k += kDmThreads / 32) {
      float v = s_w[k * kDmThreads + lane] + s_w[k * kDmThreads + 32 + lane] + s_w[k * kDmThreads + 64 + lane] +
                s_w[k * kDmThreads + 96 + lane];
#pragma unroll
      for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0) s_ws[k] = v;
    }
    const float* xr = x.ptr + b * x.sB + pp * x.sP;
    float* gxr = gx.ptr + b * gx.sB + pp * gx.sP;
    float inv_nrm = 1.f, dot = 0.f;
    if (cosine) {
      // |x|^2 and <x, gxn> in one pass over the row (x is read again below: L1 / L2)
      float ss = 0.f, raw = 0.f;
      if (in)
        for (int d = 0; d < D; ++d) {
          const float v = __ldg(xr + (long long)d * x.sD);
          float gxn = 0.f;
#pragma unroll
          for (int k = 0; k < KMAX; ++k)
            if (k < K) gxn = fmaf(w[k], s_e[k * D + d], gxn);
          ss = fmaf(v, v, ss);
          raw = fmaf(v, gxn, raw);
        }
      inv_nrm = 1.f / fmaxf(sqrtf(ss), 1e-12f);
      dot = raw * inv_nrm;                               // <xn, gxn>
    }
    for (int d0 = 0; d0 < D; d0 += 32) {
      float xv[32];
#pragma unroll
      for (int u = 0; u < 32; ++u) xv[u] = (in && d0 + u < D) ? __ldg(xr + (long long)(d0 + u) * x.sD) : 0.f;
      __syncthreads();                               // previous chunk's tile fully consumed (and s_ws visible)
#pragma unroll
      for (int u = 0; u < 32; ++u) {
        if (cosine) xv[u] *= inv_nrm;                // the tile (and the prototype gradient) work on xn
        s_x[u * kDmXStride + threadIdx.x] = xv[u];
      }
      if (in && (D & 3) == 0 && d0 + 32 <= D) {
        // four dims per LDS.128 of a prototype row (same sums in the same order as the scalar loop below)
#pragma unroll
        for (int u = 0; u < 32; u += 4) {
          float a4[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) a4[j] = cosine ? 0.f : xv[u + j] * wsum;
#pragma unroll
          for (int k = 0; k < KMAX; ++k)
            if (k < K) {
              const float4 e4 = *reinterpret_cast<const float4*>(s_e + k * D + d0 + u);
              const float wk = cosine ? w[k] : -w[k];
              a4[0] = fmaf(wk, e4.x, a4[0]); a4[1] = fmaf(wk, e4.y, a4[1]);
              a4[2] = fmaf(wk, e4.z, a4[2]); a4[3] = fmaf(wk, e4.w, a4[3]);
            }
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            float acc = a4[j];
            if (cosine) acc = (acc - xv[u + j] * dot) * inv_nrm;
            gxr[(long long)(d0 + u + j) * gx.sD] = acc;
          }
        }
      } else {
#pragma unroll
        for (int u = 0; u < 32; ++u) {
          if (in && d0 + u < D) {
            float acc = cosine ? 0.f : xv[u] * wsum;   // sum_k w_k (x - e_k) = x sum_k w_k - sum_k w_k e_k
#pragma unroll
            for (int k = 0; k < KMAX; ++k)
              if (k < K) acc = fmaf(cosine ? w[k] : -w[k], s_e[k * D + d0 + u], acc);
            if (cosine) acc = (acc - xv[u] * dot) * inv_nrm;
            gxr[(long long)(d0 + u) * gx.sD] = acc;
          }
        }
      }
      __syncthreads();
      // thread (kk, dd): dd = lane (dim within the chunk), kk = warp, warp + 4, ...
      const int dd = lane;
      if (d0 + dd < D) {
        for (int k = warp; k < K; k += kDmThreads / 32) {
          // 128-bit reads: the weights are a broadcast, a tile row (stride 132 words) is conflict-free per quarter warp
          const float4* wr = reinterpret_cast<const float4*>(s_w + k * kDmThreads);
          const float4* xc = reinterpret_cast<const float4*>(s_x + dd * kDmXStride);
          float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll 8
          for (int p = 0; p < kDmThreads / 4; ++p) {
            const float4 w4 = wr[p], x4 = xc[p];
            a0 = fmaf(w4.x, x4.x, a0); a1 = fmaf(w4.y, x4.y, a1);
            a2 = fmaf(w4.z, x4.z, a2); a3 = fmaf(w4.w, x4.w, a3);
          }
          const float r = cosine ? ((a0 + a1) + (a2 + a3)) : s_e[k * D + d0 + dd] * s_ws[k] - ((a0 + a1) + (a2 + a3));
          if (DET) {
            float* o = gEb + (long long)k * D + d0 + dd;
            *o = tile == t0 ? r : *o + r;
          } else if (r != 0.f) {
            atomicAdd(gE + (long long)k * D + d0 + dd, r);
          }
        }
      }
    }
  }
}

static bool dm_supported(long long K, long long D) {
  return K >= 1 && K <= 32 && D >= 1 && D + 2 <= 384 && (K * D + K * 128 + 32 * 132 + 64) * 4 <= 96 * 1024;
}

template <int KMAX>
static int launch_dm(const Rows& x, const float* E, int K, bool cosine, float* dist, long long oB, long long oP, long long oK,
                     long long* idx, unsigned long long* counts, float* score, cudaStream_t st) {
  const size_t smem = ((size_t)K * x.D + K + KMAX) * sizeof(float);
  const unsigned grid = (unsigned)((x.n_rows() + kDmThreads - 1) / kDmThreads);
  if (cosine) {
    if (smem > 48 * 1024) cudaFuncSetAttribute(dist_map_kernel<KMAX, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
    dist_map_kernel<KMAX, true><<<grid, kDmThreads, smem, st>>>(x, E, K, dist, oB, oP, oK, idx, counts, nullptr);
  } else {
    if (smem > 48 * 1024) cudaFuncSetAttribute(dist_map_kernel<KMAX, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
    dist_map_kernel<KMAX, false><<<grid, kDmThreads, smem, st>>>(x, E, K, dist, oB, oP, oK, idx, counts, score);
  }
  VQSEG_LAUNCH_CHECK();
  return 0;
}

template <int KMAX>
static int launch_dm_bwd(const Rows& x, const float* E, int K, const float* g, const float* dist, long long oB, long long oP,
                         long long oK, const RowsOut& gx, float* gE, const float* score, cudaStream_t st, int cosine = 0) {
  const size_t smem = ((size_t)((K * x.D + 3) & ~3) + (size_t)K * kDmThreads + KMAX + 32 * kDmXStride) * sizeof(float);
  const unsigned grid = (unsigned)((x.n_rows() + kDmThreads - 1) / kDmThreads);
  if (smem > 48 * 1024) cudaFuncSetAttribute(dist_map_bwd_kernel<KMAX, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
  dist_map_bwd_kernel<KMAX, false><<<grid, kDmThreads, smem, st>>>(x, E, K, g, dist, oB, oP, oK, gx, gE, score, cosine, 1);
  VQSEG_LAUNCH_CHECK();
  return 0;
}

// Deterministic backward of the per-pixel kernels: as many slices (blocks) of consecutive 128-pixel tiles as the
// partials' bound allows.
static void dm_det_split(long long n_rows, long long K, long long D, long long& tiles_per_block, long long& slices) {
  const long long tiles = (n_rows + kDmThreads - 1) / kDmThreads;
  const long long max_slices = seghead_det_max_slices(K, D);
  tiles_per_block = (tiles + max_slices - 1) / max_slices;
  slices = (tiles + tiles_per_block - 1) / tiles_per_block;
}

static size_t dm_det_workspace_bytes(long long n_rows, long long K, long long D) {
  long long tpb, slices;
  dm_det_split(n_rows, K, D, tpb, slices);
  return slices > 1 ? (size_t)slices * K * D * sizeof(float) : 0;
}

template <int KMAX>
static int launch_dm_bwd_det(const Rows& x, const float* E, int K, const float* g, const float* dist, long long oB,
                             long long oP, long long oK, const RowsOut& gx, float* gE, const float* score, int cosine,
                             void* ws, cudaStream_t st) {
  const size_t smem = ((size_t)((K * x.D + 3) & ~3) + (size_t)K * kDmThreads + KMAX + 32 * kDmXStride) * sizeof(float);
  long long tpb, slices;
  dm_det_split(x.n_rows(), K, x.D, tpb, slices);
  float* part = slices > 1 ? static_cast<float*>(ws) : gE;
  if (smem > 48 * 1024) cudaFuncSetAttribute(dist_map_bwd_kernel<KMAX, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
  dist_map_bwd_kernel<KMAX, true><<<(unsigned)slices, kDmThreads, smem, st>>>(x, E, K, g, dist, oB, oP, oK, gx, part, score,
                                                                               cosine, (int)tpb);
  VQSEG_LAUNCH_CHECK();
  return slices > 1 ? launch_seghead_slice_sum(part, (long long)K * x.D, (int)slices, gE, st) : 0;
}

}  // namespace vqseg

using namespace vqseg;

extern "C" {

int vqseg_dist_map_f32(const float* x, int64_t B, int64_t P, int64_t D, int64_t sB, int64_t sP, int64_t sD,
                       const float* E, int64_t K, int cosine,
                       float* dist_out, int64_t oB, int64_t oP, int64_t oK,
                       int64_t* idx_out, int64_t* counts_out, float* score_out, void* stream) {
  if (!x || !E || !dist_out || B < 0 || P < 0 || (cosine && score_out)) return VQSEG_EINVAL;
  if (!dm_supported(K, D)) return VQSEG_EUNSUPPORTED;
  int rc = check_arch();
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (counts_out) {
    cudaError_t e = cudaMemsetAsync(counts_out, 0, (size_t)K * sizeof(int64_t), st);
    if (e != cudaSuccess) return (int)e;
  }
  if (B * P == 0) return 0;
  Rows xr{x, B, P, D, sB, sP, sD};
  long long* ix = (long long*)idx_out;
  unsigned long long* cn = (unsigned long long*)counts_out;
  if (K <= 4) return launch_dm<4>(xr, E, (int)K, cosine != 0, dist_out, oB, oP, oK, ix, cn, score_out, st);
  if (K <= 8) return launch_dm<8>(xr, E, (int)K, cosine != 0, dist_out, oB, oP, oK, ix, cn, score_out, st);
  if (K <= 16) return launch_dm<16>(xr, E, (int)K, cosine != 0, dist_out, oB, oP, oK, ix, cn, score_out, st);
  return launch_dm<32>(xr, E, (int)K, cosine != 0, dist_out, oB, oP, oK, ix, cn, score_out, st);
}

int vqseg_dist_map_bwd_f32(const float* g, const float* dist, int64_t oB, int64_t oP, int64_t oK,
                           const float* x, int64_t B, int64_t P, int64_t D, int64_t sB, int64_t sP, int64_t sD,
                           const float* E, int64_t K,
                           float* gx_out, int64_t gxB, int64_t gxP, int64_t gxD, float* gE_out,
                           const float* score, void* stream) {
  if (!g || !dist || !x || !E || !gx_out || !gE_out || B < 0 || P < 0) return VQSEG_EINVAL;
  if (!dm_supported(K, D)) return VQSEG_EUNSUPPORTED;
  int rc = check_arch();
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(gE_out, 0, (size_t)K * D * sizeof(float), st);
  if (e != cudaSuccess) return (int)e;
  if (B * P == 0) return 0;
  Rows xr{x, B, P, D, sB, sP, sD};
  RowsOut gx{gx_out, B, P, D, gxB, gxP, gxD};
  if (K <= 4) return launch_dm_bwd<4>(xr, E, (int)K, g, dist, oB, oP, oK, gx, gE_out, score, st);
  if (K <= 8) return launch_dm_bwd<8>(xr, E, (int)K, g, dist, oB, oP, oK, gx, gE_out, score, st);
  if (K <= 16) return launch_dm_bwd<16>(xr, E, (int)K, g, dist, oB, oP, oK, gx, gE_out, score, st);
  return launch_dm_bwd<32>(xr, E, (int)K, g, dist, oB, oP, oK, gx, gE_out, score, st);
}

int vqseg_sim_map_bwd_f32(const float* g, int64_t oB, int64_t oP, int64_t oK,
                          const float* x, int64_t B, int64_t P, int64_t D, int64_t sB, int64_t sP, int64_t sD,
                          const float* E, int64_t K,
                          float* gx_out, int64_t gxB, int64_t gxP, int64_t gxD, float* gE_out, void* stream) {
  if (!g || !x || !E || !gx_out || !gE_out || B < 0 || P < 0) return VQSEG_EINVAL;
  if (!dm_supported(K, D)) return VQSEG_EUNSUPPORTED;
  int rc = check_arch();
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(gE_out, 0, (size_t)K * D * sizeof(float), st);
  if (e != cudaSuccess) return (int)e;
  if (B * P == 0) return 0;
  Rows xr{x, B, P, D, sB, sP, sD};
  RowsOut gx{gx_out, B, P, D, gxB, gxP, gxD};
  if (K <= 4) return launch_dm_bwd<4>(xr, E, (int)K, g, g, oB, oP, oK, gx, gE_out, nullptr, st, 1);
  if (K <= 8) return launch_dm_bwd<8>(xr, E, (int)K, g, g, oB, oP, oK, gx, gE_out, nullptr, st, 1);
  if (K <= 16) return launch_dm_bwd<16>(xr, E, (int)K, g, g, oB, oP, oK, gx, gE_out, nullptr, st, 1);
  return launch_dm_bwd<32>(xr, E, (int)K, g, g, oB, oP, oK, gx, gE_out, nullptr, st, 1);
}

// -1: bad algo, 0: per-pixel kernels, 1: tiled kernels, VQSEG_EUNSUPPORTED: per-pixel forced beyond its limits.
// The VQSEG_SEGHEAD_DETERMINISTIC bit does not take part in the choice.
static int seghead_kernel(int64_t K, int64_t D, int algo) {
  algo &= ~VQSEG_SEGHEAD_DETERMINISTIC;
  if (algo == VQSEG_SEGHEAD_AUTO) return dm_supported(K, D) ? 0 : 1;
  if (algo == VQSEG_SEGHEAD_PIXEL) return dm_supported(K, D) ? 0 : VQSEG_EUNSUPPORTED;
  if (algo == VQSEG_SEGHEAD_TILED) return 1;
  return -1;
}

int vqseg_seghead_map_f32(const float* x, int64_t B, int64_t P, int64_t D, int64_t sB, int64_t sP, int64_t sD,
                          const float* E, int64_t K, int cosine,
                          float* dist_out, int64_t oB, int64_t oP, int64_t oK,
                          int64_t* idx_out, int64_t* counts_out, float* score_out, int algo, void* stream) {
  if (!x || !E || !dist_out || B < 0 || P < 0 || K < 1 || D < 1 || K > INT32_MAX || D > INT32_MAX ||
      (cosine && score_out) || (algo & VQSEG_SEGHEAD_DETERMINISTIC))
    return VQSEG_EINVAL;
  const int which = seghead_kernel(K, D, algo);
  if (which < 0) return which == -1 ? VQSEG_EINVAL : which;
  if (which == 0)
    return vqseg_dist_map_f32(x, B, P, D, sB, sP, sD, E, K, cosine, dist_out, oB, oP, oK, idx_out, counts_out, score_out, stream);
  int rc = check_arch();
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (counts_out) {
    cudaError_t e = cudaMemsetAsync(counts_out, 0, (size_t)K * sizeof(int64_t), st);
    if (e != cudaSuccess) return (int)e;
  }
  if (B * P == 0) return 0;
  Rows xr{x, B, P, D, sB, sP, sD};
  const long long L = cosine ? D : D + 2;
  const int kb = auto_kblock(L) > 0 ? auto_kblock(L) : (int)L;
  return launch_seghead_map_tiled(xr, E, (int)K, cosine != 0, kb, dist_out, oB, oP, oK, (long long*)idx_out,
                                  (unsigned long long*)counts_out, score_out, st);
}

size_t vqseg_seghead_map_bwd_workspace_bytes(int64_t n_rows, int64_t D, int64_t K, int algo) {
  const int which = seghead_kernel(K, D, algo);
  const bool det = (algo & VQSEG_SEGHEAD_DETERMINISTIC) != 0;
  if (n_rows <= 0 || which < 0) return 0;
  if (which == 0) return det ? dm_det_workspace_bytes(n_rows, K, D) : 0;
  return seghead_bwd_tiled_workspace_bytes(n_rows, (int)K, (int)D, det);
}

int vqseg_seghead_map_bwd_f32(const float* g, const float* map, int64_t oB, int64_t oP, int64_t oK,
                              const float* x, int64_t B, int64_t P, int64_t D, int64_t sB, int64_t sP, int64_t sD,
                              const float* E, int64_t K, int cosine, const float* score,
                              float* gx_out, int64_t gxB, int64_t gxP, int64_t gxD, float* gE_out,
                              int algo, void* ws, size_t ws_bytes, void* stream) {
  if (!g || !map || !x || !E || !gx_out || !gE_out || B < 0 || P < 0 || K < 1 || D < 1 || K > INT32_MAX ||
      D > INT32_MAX || (cosine && score))
    return VQSEG_EINVAL;
  const int which = seghead_kernel(K, D, algo);
  if (which < 0) return which == -1 ? VQSEG_EINVAL : which;
  const bool det = (algo & VQSEG_SEGHEAD_DETERMINISTIC) != 0;
  if (which == 0 && !det) {
    if (cosine) return vqseg_sim_map_bwd_f32(g, oB, oP, oK, x, B, P, D, sB, sP, sD, E, K, gx_out, gxB, gxP, gxD, gE_out, stream);
    return vqseg_dist_map_bwd_f32(g, map, oB, oP, oK, x, B, P, D, sB, sP, sD, E, K, gx_out, gxB, gxP, gxD, gE_out,
                                  score, stream);
  }
  const size_t need = vqseg_seghead_map_bwd_workspace_bytes(B * P, D, K, algo);
  if (ws_bytes < need || (need > 0 && !ws)) return VQSEG_EWORKSPACE;
  int rc = check_arch();
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (!det || B * P == 0) {                        // the deterministic kernels store every element of gE
    cudaError_t e = cudaMemsetAsync(gE_out, 0, (size_t)K * D * sizeof(float), st);
    if (e != cudaSuccess) return (int)e;
  }
  if (B * P == 0) return 0;
  Rows xr{x, B, P, D, sB, sP, sD};
  RowsOut gx{gx_out, B, P, D, gxB, gxP, gxD};
  if (which == 1) return launch_seghead_map_bwd_tiled(xr, E, (int)K, cosine != 0, g, map, oB, oP, oK, score, gx, gE_out, det, ws, st);
  // per-pixel kernels, deterministic (cosine: g stands in for the unread map, as in vqseg_sim_map_bwd_f32)
  const float* dm = cosine ? g : map;
  const int c = cosine != 0;
  if (K <= 4) return launch_dm_bwd_det<4>(xr, E, (int)K, g, dm, oB, oP, oK, gx, gE_out, score, c, ws, st);
  if (K <= 8) return launch_dm_bwd_det<8>(xr, E, (int)K, g, dm, oB, oP, oK, gx, gE_out, score, c, ws, st);
  if (K <= 16) return launch_dm_bwd_det<16>(xr, E, (int)K, g, dm, oB, oP, oK, gx, gE_out, score, c, ws, st);
  return launch_dm_bwd_det<32>(xr, E, (int)K, g, dm, oB, oP, oK, gx, gE_out, score, c, ws, st);
}

}  // extern "C"
