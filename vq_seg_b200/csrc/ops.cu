// HBM-bound kernels of the VQ bottleneck: codebook gather + straight-through estimator + commitment
// loss, its backward, per-code statistics for k-means, and small helpers.
// Reference call sites are cited per kernel (paths relative to the reference root).
#include <climits>
#include <cuda_bf16.h>

#include "common.cuh"

namespace vqseg {

// =================================================================================================
// gather + STE + commitment loss      (vq_img.py:169-170 one_hot+matmul, :236 STE, :239 mse_loss)
// =================================================================================================
// Pixel-contiguous layout (NCHW: sP == 1).  A block owns a 128-pixel x 32-dim tile: codebook rows
// are read along d (coalesced 128 B per code row segment) into a padded smem tile, then x / q are
// streamed along pixels (coalesced).  algorithmic bytes: 4ND (x) + 4ND (q) + 8N (idx) + 4KD (E).
constexpr int kGTile = 32;       // dims per tile (128 x 32 tiles: 2048 blocks at C2, 8 resident per SM -> 1.7 waves;
                                 // 128 x 64 tiles gave 1024 blocks on 888 slots, i.e. a second wave 15 % full)
constexpr int kGPix = 128;       // pixels per tile

// VQSEG_MODE_ROTATE is ORed into a train mode: it changes what is written (c instead of x + (c - x)), not how the code
// is rounded or that x is read
constexpr int base_mode(int mode) { return mode & ~VQSEG_MODE_ROTATE; }
constexpr bool gather_train(int mode) {
  mode = base_mode(mode);
  return mode == VQSEG_MODE_TRAIN || mode == VQSEG_MODE_TRAIN_AMP || mode == VQSEG_MODE_TRAIN_AMP_BF16;
}
// the code as the reference's autocast matmul produces it: rounded (to nearest even) through fp16 / bf16 per mode.
// Signed zeros and infinities pass through, fp32 values beyond the type's range become inf of their sign, and a NaN
// stays a NaN (the canonical one; its sign and payload carry no meaning).
template <int MODE>
__device__ __forceinline__ float round_code(float v) {
  constexpr int M = base_mode(MODE);
  if (M == VQSEG_MODE_TRAIN_AMP || M == VQSEG_MODE_EVAL_AMP) return __half2float(__float2half_rn(v));
  if (M == VQSEG_MODE_TRAIN_AMP_BF16 || M == VQSEG_MODE_EVAL_AMP_BF16) return __bfloat162float(__float2bfloat16_rn(v));
  return v;
}
// pixel p of a tile lives in column (p % 4) * 32 + p / 4: a lane that owns pixels 4*lane .. 4*lane+3 then reads
// columns lane, 32 + lane, 64 + lane, 96 + lane -- conflict-free (straight columns gave 4-way bank conflicts)
__device__ __forceinline__ int gcol(int p) { return ((p & 3) << 5) | (p >> 2); }

// Last-block loss reduction (fused forward): every block publishes its partial, takes a ticket, and the block that
// draws the last one sums all partials in the same fixed order as loss_finalize_kernel -- one launch less.
// The same block also turns the (by then final) per-code counts into the code usage of vq_img.py:173-175.
struct LossTail { int* ticket; float* loss_out; double inv_numel; const unsigned long long* counts; int K; float* usage_out; };
__device__ __forceinline__ void loss_tail(const LossTail& t, const float* partial, int n_partial, int n_blocks) {
  __shared__ double s_dred[256];
  __shared__ int s_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = (atomicAdd(t.ticket, 1) == n_blocks - 1);
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  if (t.loss_out) {
    double s = 0.0;
    for (int i = threadIdx.x; i < n_partial; i += 256) s += (double)__ldcg(partial + i);
    s_dred[threadIdx.x] = s;
    __syncthreads();
    for (int o = 128; o; o >>= 1) {
      if ((int)threadIdx.x < o) s_dred[threadIdx.x] += s_dred[threadIdx.x + o];
      __syncthreads();
    }
    if (threadIdx.x == 0) *t.loss_out = (float)(s_dred[0] * t.inv_numel);
    __syncthreads();
  }
  if (t.usage_out) {
    int z = 0;
    for (int k = threadIdx.x; k < t.K; k += 256) z += (__ldcg(t.counts + k) == 0ull);
    s_dred[threadIdx.x] = (double)z;
    __syncthreads();
    for (int o = 128; o; o >>= 1) {
      if ((int)threadIdx.x < o) s_dred[threadIdx.x] += s_dred[threadIdx.x + o];
      __syncthreads();
    }
    if (threadIdx.x == 0) *t.usage_out = __fmul_rn(100.f, __fdiv_rn((float)s_dred[0], (float)t.K));
  }
}

// VEC: pixel quads are 16-byte aligned and never straddle an image (P % 4 == 0, aligned bases)
template <int MODE, bool VEC>
__global__ void __launch_bounds__(256) gather_ste_pxc_kernel(Rows x, const float* __restrict__ E, int K,
                                                             const long long* __restrict__ idx, RowsOut q,
                                                             float* __restrict__ partial, LossTail tail) {
  __shared__ float tile[kGTile][kGPix + 1];
  __shared__ int s_idx[kGPix];
  __shared__ float s_red[8];
  pdl_wait();                                     // (launched as a programmatic dependent of the assignment's last kernel)
  const int D = (int)x.D;
  const long long n_rows = x.n_rows();
  const long long n0 = (long long)blockIdx.x * kGPix;
  const int d0 = blockIdx.y * kGTile;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr bool kTrain = gather_train(MODE);
  constexpr bool kRot = (MODE & VQSEG_MODE_ROTATE) != 0;     // write c itself; the loss term is (c - x)^2
  if (threadIdx.x < kGPix) {
    long long n = n0 + threadIdx.x;
    long long k = n < n_rows ? idx[n] : 0;
    // element offset of the code row (K * D < 2^31 is checked by the launcher): the gather below then needs one
    // 32-bit add per load instead of a 64-bit multiply -- address arithmetic was a third of this kernel's instructions
    s_idx[threadIdx.x] = (int)(k < 0 ? 0 : (k >= K ? K - 1 : k)) * D;
  }
  __syncthreads();
  // phase 1: gather code row segments (128 B each), lanes along d
  const float* Ed = E + d0 + lane;
#pragma unroll 2
  for (int p0 = warp; p0 < kGPix; p0 += 64) {           // 16 loads in flight per lane before the smem stores
    float v[8][kGTile / 32];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const float* er = Ed + s_idx[p0 + 8 * u];
#pragma unroll
      for (int h = 0; h < kGTile / 32; ++h) {
        const int d = lane + 32 * h;
        v[u][h] = (d0 + d < D) ? __ldg(er + 32 * h) : 0.f;
      }
    }
#pragma unroll
    for (int u = 0; u < 8; ++u)
#pragma unroll
      for (int h = 0; h < kGTile / 32; ++h) tile[lane + 32 * h][gcol(p0 + 8 * u)] = round_code<MODE>(v[u][h]);
  }
  __syncthreads();
  // phase 2: stream pixels; lane owns 4 consecutive pixels, warps take the dims round-robin
  float acc = 0.f;
  const int p4 = lane * 4;
  const long long n = n0 + p4;
  if (VEC) {
    if (n < n_rows) {
      long long b, pp;
      split_row(n, x.P, b, pp);
      const float* xb = kTrain ? x.ptr + b * x.sB + pp : nullptr;
      float* qb = q.ptr + b * q.sB + pp;
      float4 xr[kGTile / 8];
      const float* xd = kTrain ? xb + (long long)(d0 + warp) * x.sD : nullptr;   // rows d0 + warp + 8u: pointer stepping
      float* qd = qb + (long long)(d0 + warp) * q.sD;
      const long long xstep = 8 * x.sD, qstep = 8 * q.sD;
      if (kTrain) {                                        // all row loads in flight before the first use
#pragma unroll
        for (int u = 0; u < kGTile / 8; ++u) {
          const int d = warp + 8 * u;
          xr[u] = (d0 + d < D) ? __ldg(reinterpret_cast<const float4*>(xd + u * xstep))
                               : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
#pragma unroll
      for (int u = 0; u < kGTile / 8; ++u) {
        const int d = warp + 8 * u;
        if (d0 + d < D) {
          float4 e = make_float4(tile[d][lane], tile[d][32 + lane], tile[d][64 + lane], tile[d][96 + lane]);   // = pixels p4 .. p4+3
          float4 o = e;
          if (kTrain) {
            const float4 xv = xr[u];
            if (!kRot) {
              o.x = __fadd_rn(xv.x, __fsub_rn(e.x, xv.x)); o.y = __fadd_rn(xv.y, __fsub_rn(e.y, xv.y));   // x + (q - x)
              o.z = __fadd_rn(xv.z, __fsub_rn(e.z, xv.z)); o.w = __fadd_rn(xv.w, __fsub_rn(e.w, xv.w));
            }
            float f;
            f = __fsub_rn(o.x, xv.x); acc = __fmaf_rn(f, f, acc); f = __fsub_rn(o.y, xv.y); acc = __fmaf_rn(f, f, acc);
            f = __fsub_rn(o.z, xv.z); acc = __fmaf_rn(f, f, acc); f = __fsub_rn(o.w, xv.w); acc = __fmaf_rn(f, f, acc);
          }
          *reinterpret_cast<float4*>(qd + u * qstep) = o;
        }
      }
    }
  } else {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const long long ni = n + i;
      if (ni < n_rows) {
        long long b, pp;
        split_row(ni, x.P, b, pp);
        const float* xb = kTrain ? x.ptr + b * x.sB + pp * x.sP : nullptr;
        float* qb = q.ptr + b * q.sB + pp * q.sP;
        for (int d = warp; d < kGTile; d += 8) {
          if (d0 + d < D) {
            float e = tile[d][32 * i + lane];
            float o = e;
            if (kTrain) {
              float xv = __ldg(xb + (long long)(d0 + d) * x.sD);
              if (!kRot) o = __fadd_rn(xv, __fsub_rn(e, xv));
              float f = __fsub_rn(o, xv);
              acc = __fmaf_rn(f, f, acc);
            }
            qb[(long long)(d0 + d) * q.sD] = o;
          }
        }
      }
    }
  }
  if (partial) {
#pragma unroll
    for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) s_red[warp] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
      float s = 0.f;
#pragma unroll
      for (int w = 0; w < 8; ++w) s += s_red[w];
      partial[(long long)blockIdx.y * gridDim.x + blockIdx.x] = s;
    }
  }
  if (tail.ticket) loss_tail(tail, partial, (int)(gridDim.x * gridDim.y), (int)(gridDim.x * gridDim.y));
}

// Generic strides (row-major samples etc.): one warp per row, lanes along d.
template <int MODE>
__global__ void __launch_bounds__(256) gather_ste_generic_kernel(Rows x, const float* __restrict__ E, int K,
                                                                 const long long* __restrict__ idx, RowsOut q,
                                                                 float* __restrict__ partial, LossTail tail) {
  __shared__ float s_red[8];
  const int D = (int)x.D;
  const long long n_rows = x.n_rows();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float acc = 0.f;
  for (long long n = (long long)blockIdx.x * 8 + warp; n < n_rows; n += (long long)gridDim.x * 8) {
    long long k = idx[n];
    k = k < 0 ? 0 : (k >= K ? K - 1 : k);
    const float* er = E + k * D;
    const float* xr = x.row(n);
    float* qr = q.row(n);
    for (int d = lane; d < D; d += 32) {
      const float e = round_code<MODE>(__ldg(er + d));
      if (!gather_train(MODE)) {
        qr[(long long)d * q.sD] = e;
      } else {
        float xv = __ldg(xr + (long long)d * x.sD);
        float qs = (MODE & VQSEG_MODE_ROTATE) ? e : __fadd_rn(xv, __fsub_rn(e, xv));
        qr[(long long)d * q.sD] = qs;
        float df = __fsub_rn(qs, xv);
        acc = __fmaf_rn(df, df, acc);
      }
    }
  }
  if (partial) {
#pragma unroll
    for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) s_red[warp] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
      float s = 0.f;
#pragma unroll
      for (int w = 0; w < 8; ++w) s += s_red[w];
      partial[blockIdx.x] = s;
    }
  }
  if (tail.ticket) loss_tail(tail, partial, (int)gridDim.x, (int)gridDim.x);
}

// fixed-order final reduction of the per-block partials -> mean
__global__ void __launch_bounds__(256) loss_finalize_kernel(const float* __restrict__ partial, int n_partial,
                                                            double inv_numel, float* __restrict__ loss_out) {
  __shared__ double s_red[256];
  double s = 0.0;
  for (int i = threadIdx.x; i < n_partial; i += 256) s += (double)partial[i];
  s_red[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o; o >>= 1) {
    if (threadIdx.x < o) s_red[threadIdx.x] += s_red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) *loss_out = (float)(s_red[0] * inv_numel);
}

template <int MODE>
static int launch_gather(const Rows& x, const float* E, int K, const long long* idx, const RowsOut& q,
                         float* loss_out, float* partial, size_t partial_cap, cudaStream_t st, int* ticket = nullptr,
                         const unsigned long long* counts = nullptr, float* usage_out = nullptr) {
  const long long n_rows = x.n_rows();
  const bool train = gather_train(MODE);
  const bool want_loss = train && loss_out != nullptr;
  const bool want_usage = ticket && counts && usage_out;
  // ticket (zeroed by the caller): the kernel's last block reduces the loss (and the code usage) itself
  LossTail tail{(want_loss || want_usage) ? ticket : nullptr, want_loss ? loss_out : nullptr,
                1.0 / ((double)n_rows * (double)x.D), counts, K, want_usage ? usage_out : nullptr};
  int n_partial = 0;
  if (x.sP == 1 && q.sP == 1 && (long long)K * x.D < (1ll << 31)) {
    dim3 grid((unsigned)((n_rows + kGPix - 1) / kGPix), (unsigned)((x.D + kGTile - 1) / kGTile));
    n_partial = (int)(grid.x * grid.y);
    if (want_loss && (size_t)n_partial > partial_cap) return VQSEG_EWORKSPACE;
    auto al = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
    const bool vec = (x.P % 4 == 0) && al(q.ptr) && (q.sD % 4 == 0) && (q.sB % 4 == 0) &&
                     (!train || (al(x.ptr) && (x.sD % 4 == 0) && (x.sB % 4 == 0)));
    cudaError_t le;
    if (vec) le = launch_dependent(gather_ste_pxc_kernel<MODE, true>, grid, dim3(256), 0, st, pdl_enabled(), x, E, K, idx, q, want_loss ? partial : nullptr, tail);
    else     le = launch_dependent(gather_ste_pxc_kernel<MODE, false>, grid, dim3(256), 0, st, pdl_enabled(), x, E, K, idx, q, want_loss ? partial : nullptr, tail);
    if (le != cudaSuccess) return (int)le;
  } else {
    long long blocks = (n_rows + 7) / 8;
    long long cap = (long long)num_sms() * 16;
    if (blocks > cap) blocks = cap;
    n_partial = (int)blocks;
    if (want_loss && (size_t)n_partial > partial_cap) return VQSEG_EWORKSPACE;
    gather_ste_generic_kernel<MODE><<<(unsigned)blocks, 256, 0, st>>>(x, E, K, idx, q, want_loss ? partial : nullptr, tail);
  }
  VQSEG_LAUNCH_CHECK();
  if (want_loss && !ticket) {
    loss_finalize_kernel<<<1, 256, 0, st>>>(partial, n_partial, 1.0 / ((double)n_rows * (double)x.D), loss_out);
    VQSEG_LAUNCH_CHECK();
  }
  return 0;
}

// =================================================================================================
// backward w.r.t. x of the training forward (autograd through vq_img.py:236-240)
// gx = g_q + coef * (x - q_ste),  coef = coef_scale * (*coef_dev)
// =================================================================================================
struct View { const float* ptr; long long sB, sP, sD; };
__global__ void __launch_bounds__(256) ste_bwd_kernel(View g, View x, View q, const float* __restrict__ coef_dev,
                                                      float coef_scale, RowsOut o, bool px_fast) {
  const long long total = o.B * o.P * o.D;
  const float coef = coef_dev ? coef_scale * __ldg(coef_dev) : 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    long long b, p, d;
    if (px_fast) { p = i % o.P; long long t = i / o.P; d = t % o.D; b = t / o.D; }
    else         { d = i % o.D; long long t = i / o.D; p = t % o.P; b = t / o.P; }
    float gv = g.ptr ? __ldg(g.ptr + b * g.sB + p * g.sP + d * g.sD) : 0.f;
    float r = gv;
    if (coef_dev) {
      float xv = __ldg(x.ptr + b * x.sB + p * x.sP + d * x.sD);
      float qv = __ldg(q.ptr + b * q.sB + p * q.sP + d * q.sD);
      r = __fmaf_rn(coef, __fsub_rn(xv, qv), gv);
    }
    o.ptr[b * o.sB + p * o.sP + d * o.sD] = r;
  }
}

// same dense layout for all four tensors: flat, vectorised, memory order
__global__ void __launch_bounds__(256) ste_bwd_flat_kernel(const float4* __restrict__ g, const float4* __restrict__ x,
                                                           const float4* __restrict__ q, const float* __restrict__ coef_dev,
                                                           float coef_scale, float4* __restrict__ o, long long n4) {
  const float coef = coef_dev ? coef_scale * __ldg(coef_dev) : 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    float4 r = g ? __ldg(g + i) : make_float4(0.f, 0.f, 0.f, 0.f);
    if (coef_dev) {
      const float4 xv = __ldg(x + i), qv = __ldg(q + i);
      r.x = __fmaf_rn(coef, __fsub_rn(xv.x, qv.x), r.x); r.y = __fmaf_rn(coef, __fsub_rn(xv.y, qv.y), r.y);
      r.z = __fmaf_rn(coef, __fsub_rn(xv.z, qv.z), r.z); r.w = __fmaf_rn(coef, __fsub_rn(xv.w, qv.w), r.w);
    }
    o[i] = r;
  }
}

// =================================================================================================
// backward w.r.t. x of the rotation trick (opt-in extension, no reference counterpart: Fifty et al., arXiv 2410.06424
// §4.2; rotation_trick of lucidrains/vector-quantize-pytorch).  Per row gx = alpha g + beta x + gamma c, with the
// coefficients of vqseg.h from five row sums.  Each sum is eight chains a_l over d = l, l + 8, ... (ascending), combined
// ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7)); all three layout paths below keep that order, so gx is the same
// bits whatever the strides.
// =================================================================================================
constexpr int kRotSums = 5;                     // x.x, c.c, x.c, x.g, c.g
__device__ __forceinline__ void rot_accum(float (&a)[kRotSums], float x, float c, float g) {
  a[0] = __fadd_rn(a[0], __fmul_rn(x, x));
  a[1] = __fadd_rn(a[1], __fmul_rn(c, c));
  a[2] = __fadd_rn(a[2], __fmul_rn(x, c));
  a[3] = __fadd_rn(a[3], __fmul_rn(x, g));
  a[4] = __fadd_rn(a[4], __fmul_rn(c, g));
}
__device__ __forceinline__ float rot_tree(const float (&a)[8]) {
  return __fadd_rn(__fadd_rn(__fadd_rn(a[0], a[1]), __fadd_rn(a[2], a[3])),
                   __fadd_rn(__fadd_rn(a[4], a[5]), __fadd_rn(a[6], a[7])));
}
// (alpha, beta, gamma) from the row sums; a zero x or c row takes the straight-through gradient
__device__ __forceinline__ float3 rot_coefs(const float (&s)[kRotSums], float lam) {
  if (s[0] == 0.f || s[1] == 0.f) return make_float3(1.f, lam, -lam);
  const float nx = __fsqrt_rn(s[0]), nc = __fsqrt_rn(s[1]);
  const float sc = __fdiv_rn(nc, nx);
  const float rho = __fdiv_rn(__fdiv_rn(s[2], nx), nc);
  const float a = __fdiv_rn(s[3], nx), b = __fdiv_rn(s[4], nc);
  const float t = __fadd_rn(1.f, rho);
  const float h = t > 0.f ? __fdiv_rn(__fadd_rn(a, b), t) : 0.f;     // antipodal rows: w = 0, the reflection
  const float beta = __fadd_rn(__fdiv_rn(__fmul_rn(sc, __fsub_rn(__fmul_rn(2.f, b), h)), nx), lam);
  const float gamma = __fsub_rn(-__fdiv_rn(__fmul_rn(sc, h), nc), lam);
  return make_float3(sc, beta, gamma);
}
__device__ __forceinline__ float rot_out(float3 k, float g, float x, float c) {
  return __fadd_rn(__fadd_rn(__fmul_rn(k.x, g), __fmul_rn(k.y, x)), __fmul_rn(k.z, c));
}

// Pixel-contiguous maps (sP == 1): a block owns 32 neighbouring pixels of one image (lane = pixel) and stages chunks of
// up to kRotChunk channels of x, c and g in shared memory (coalesced 128-byte lines); warp w runs the chains of class
// d = w (mod 8), the tree combines them through shared memory, and gx is written from the staged tile when the whole
// row fits (D <= kRotChunk: x, c and g are read from HBM once), else from a second read.
// (Tried: each warp holding its 32 channels of x, c and g in registers instead of the 96 KB tile, 96 loads in flight per
// thread: 70 us against 62 on the config-2 map, and slower on every config-1 layer.)
constexpr int kRotChunk = 256;
__global__ void __launch_bounds__(256) rotate_bwd_px_kernel(View g, View x, View q, const float* __restrict__ coef_dev,
                                                            float coef_scale, RowsOut o, int ch) {
  extern __shared__ float rot_tile[];            // [3][ch][32]: x, c, g
  __shared__ float s_part[kRotSums][8][32];
  __shared__ float s_k[3][32];
  float* tx = rot_tile;
  float* tc = rot_tile + ch * 32;
  float* tg = rot_tile + 2 * ch * 32;
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int D = (int)o.D;
  const float lam = coef_dev ? __fmul_rn(coef_scale, __ldg(coef_dev)) : 0.f;
  const long long groups_per_image = (o.P + 31) / 32;
  for (long long gidx = blockIdx.x; gidx < o.B * groups_per_image; gidx += gridDim.x) {
    const long long b = gidx / groups_per_image, p = (gidx % groups_per_image) * 32 + lane;
    const bool on = p < o.P;
    const long long pp = on ? p : 0;
    const float* xp = x.ptr + b * x.sB + pp * x.sP;
    const float* cp = q.ptr + b * q.sB + pp * q.sP;
    const float* gp = g.ptr ? g.ptr + b * g.sB + pp * g.sP : nullptr;
    float a[kRotSums] = {0.f, 0.f, 0.f, 0.f, 0.f};
    for (int d0 = 0; d0 < D; d0 += ch) {         // ch % 8 == 0: class w stays with warp w across chunks
      const int dn = min(ch, D - d0);
      __syncthreads();
#pragma unroll 4
      for (int j = wib; j < dn; j += 8) {
        const long long d = d0 + j;
        tx[j * 32 + lane] = on ? __ldg(xp + d * x.sD) : 0.f;
        tc[j * 32 + lane] = on ? __ldg(cp + d * q.sD) : 0.f;
        tg[j * 32 + lane] = (on && gp) ? __ldg(gp + d * g.sD) : 0.f;
      }
      __syncthreads();
      for (int j = wib; j < dn; j += 8) rot_accum(a, tx[j * 32 + lane], tc[j * 32 + lane], tg[j * 32 + lane]);
    }
#pragma unroll
    for (int i = 0; i < kRotSums; ++i) s_part[i][wib][lane] = a[i];
    __syncthreads();
    if (wib == 0) {
      float s[kRotSums];
#pragma unroll
      for (int i = 0; i < kRotSums; ++i) {
        float v[8];
#pragma unroll
        for (int w = 0; w < 8; ++w) v[w] = s_part[i][w][lane];
        s[i] = rot_tree(v);
      }
      const float3 k = rot_coefs(s, lam);
      s_k[0][lane] = k.x; s_k[1][lane] = k.y; s_k[2][lane] = k.z;
    }
    __syncthreads();
    const float3 k = make_float3(s_k[0][lane], s_k[1][lane], s_k[2][lane]);
    if (on) {
      float* op = o.ptr + b * o.sB + p * o.sP;
      if (D <= ch) {
        for (int d = wib; d < D; d += 8)
          op[(long long)d * o.sD] = rot_out(k, tg[d * 32 + lane], tx[d * 32 + lane], tc[d * 32 + lane]);
      } else {
        for (int d = wib; d < D; d += 8) {
          const float gv = gp ? __ldg(gp + (long long)d * g.sD) : 0.f;
          op[(long long)d * o.sD] = rot_out(k, gv, __ldg(xp + (long long)d * x.sD), __ldg(cp + (long long)d * q.sD));
        }
      }
    }
  }
}

// Packed rows (sD == 1 of x): eight lanes per row, lane l runs chain l; the butterfly over lanes 1, 2, 4 is the tree.
__global__ void __launch_bounds__(256) rotate_bwd_rows_kernel(View g, View x, View q, const float* __restrict__ coef_dev,
                                                              float coef_scale, RowsOut o) {
  const int l8 = threadIdx.x & 7;
  const long long n = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 3;
  const bool on = n < o.B * o.P;                 // (whole groups of 8 lanes are on or off together)
  const int D = on ? (int)o.D : 0;
  long long b, p;
  split_row(on ? n : 0, o.P, b, p);
  const float* xr = x.ptr + b * x.sB + p * x.sP;
  const float* cr = q.ptr + b * q.sB + p * q.sP;
  const float* gr = g.ptr ? g.ptr + b * g.sB + p * g.sP : nullptr;
  float a[kRotSums] = {0.f, 0.f, 0.f, 0.f, 0.f};
  for (int d = l8; d < D; d += 8)
    rot_accum(a, __ldg(xr + (long long)d * x.sD), __ldg(cr + (long long)d * q.sD), gr ? __ldg(gr + (long long)d * g.sD) : 0.f);
#pragma unroll
  for (int i = 0; i < kRotSums; ++i)
#pragma unroll
    for (int m = 1; m < 8; m <<= 1) a[i] = __fadd_rn(a[i], __shfl_xor_sync(0xffffffffu, a[i], m));
  const float lam = coef_dev ? __fmul_rn(coef_scale, __ldg(coef_dev)) : 0.f;
  const float3 k = rot_coefs(a, lam);
  float* orow = o.ptr + b * o.sB + p * o.sP;
  for (int d = l8; d < D; d += 8) {
    const float gv = gr ? __ldg(gr + (long long)d * g.sD) : 0.f;
    orow[(long long)d * o.sD] = rot_out(k, gv, __ldg(xr + (long long)d * x.sD), __ldg(cr + (long long)d * q.sD));
  }
}

// Any other strides (CNHW-like views with sP > 1 and sD > 1): one thread per row, eight chains in registers.
__global__ void __launch_bounds__(256) rotate_bwd_strided_kernel(View g, View x, View q, const float* __restrict__ coef_dev,
                                                                 float coef_scale, RowsOut o) {
  const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= o.B * o.P) return;
  const int D = (int)o.D;
  long long b, p;
  split_row(n, o.P, b, p);
  const float* xr = x.ptr + b * x.sB + p * x.sP;
  const float* cr = q.ptr + b * q.sB + p * q.sP;
  const float* gr = g.ptr ? g.ptr + b * g.sB + p * g.sP : nullptr;
  float a[kRotSums][8];
#pragma unroll
  for (int i = 0; i < kRotSums; ++i)
#pragma unroll
    for (int l = 0; l < 8; ++l) a[i][l] = 0.f;
  for (int d0 = 0; d0 < D; d0 += 8) {
#pragma unroll
    for (int l = 0; l < 8; ++l) {
      const long long d = d0 + l;
      if (d < D) {
        const float xv = __ldg(xr + d * x.sD), cv = __ldg(cr + d * q.sD), gv = gr ? __ldg(gr + d * g.sD) : 0.f;
        float t[kRotSums] = {a[0][l], a[1][l], a[2][l], a[3][l], a[4][l]};
        rot_accum(t, xv, cv, gv);
#pragma unroll
        for (int i = 0; i < kRotSums; ++i) a[i][l] = t[i];
      }
    }
  }
  float s[kRotSums];
#pragma unroll
  for (int i = 0; i < kRotSums; ++i) s[i] = rot_tree(a[i]);
  const float lam = coef_dev ? __fmul_rn(coef_scale, __ldg(coef_dev)) : 0.f;
  const float3 k = rot_coefs(s, lam);
  float* orow = o.ptr + b * o.sB + p * o.sP;
  for (long long d = 0; d < D; ++d) {
    const float gv = gr ? __ldg(gr + d * g.sD) : 0.f;
    orow[d * o.sD] = rot_out(k, gv, __ldg(xr + d * x.sD), __ldg(cr + d * q.sD));
  }
}

// gE[idx[n], :] += g[n, :]   (eval-mode gather backward; the reference's one_hot matmul gives the
// codebook a gradient only in eval mode, SURVEY.md §8b "autograd contract")
__global__ void __launch_bounds__(256) gather_bwd_codebook_kernel(Rows g, const long long* __restrict__ idx,
                                                                  float* __restrict__ gE, int K) {
  const int D = (int)g.D;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long n_rows = g.n_rows();
  for (long long n = (long long)blockIdx.x * 8 + warp; n < n_rows; n += (long long)gridDim.x * 8) {
    long long k = idx[n];
    if (k < 0 || k >= K) continue;
    const float* gr = g.row(n);
    for (int d = lane; d < D; d += 32) atomicAdd(gE + k * D + d, gr[(long long)d * g.sD]);
  }
}

// =================================================================================================
// per-code statistics      (batched_bincount vq_img.py:22-27,:42; scatter_add_ :47-51)
// =================================================================================================
// fast path: fp32 atomics (RED.ADD.F32), order not fixed.
__global__ void __launch_bounds__(256) code_stats_atomic_kernel(Rows x, const long long* __restrict__ idx, int K,
                                                                unsigned long long* __restrict__ counts,
                                                                float* __restrict__ sums, bool px_fast) {
  const long long n_rows = x.n_rows();
  const int D = (int)x.D;
  const long long total = n_rows * D;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    long long n; int d;
    if (px_fast) {     // consecutive threads -> consecutive pixels of one image at fixed d
      long long p = i % x.P; long long t = i / x.P; d = (int)(t % D); long long b = t / D; n = b * x.P + p;
    } else { d = (int)(i % D); n = i / D; }
    long long k = idx[n];
    if (k < 0 || k >= K) continue;
    atomicAdd(sums + k * D + d, x.row(n)[(long long)d * x.sD]);
    if (d == 0) atomicAdd(counts + k, 1ull);
  }
}

// packed rows: one warp per row, lanes along d, 16-byte vector reductions (red.global.add.v4.f32)
__global__ void __launch_bounds__(256) code_stats_atomic_rows_kernel(const float* __restrict__ x, long long row_stride,
                                                                     long long n_rows, int D,
                                                                     const long long* __restrict__ idx, int K,
                                                                     unsigned long long* __restrict__ counts,
                                                                     float* __restrict__ sums) {
  const int lane = threadIdx.x & 31;
  const long long w0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nw = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long n = w0; n < n_rows; n += nw) {
    const long long k = idx[n];
    if (k < 0 || k >= K) continue;
    const float* xr = x + n * row_stride;
    float* sr = sums + k * D;
    for (int d = 4 * lane; d < D; d += 128) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(xr + d));
      atomicAdd(reinterpret_cast<float4*>(sr + d), v);
    }
    if (lane == 0) atomicAdd(counts + k, 1ull);
  }
}

// deterministic path ---------------------------------------------------------------------------
constexpr int kSortBlock = 1024;   // rows per ranking block

// (1) per-block histogram
__global__ void __launch_bounds__(1024) stats_hist_kernel(const long long* __restrict__ idx, long long n_rows, int K,
                                                          int* __restrict__ hist /* [nblk][K] */) {
  long long n = (long long)blockIdx.x * kSortBlock + threadIdx.x;
  if (n < n_rows) {
    long long k = idx[n];
    if (k >= 0 && k < K) atomicAdd(hist + (long long)blockIdx.x * K + k, 1);
  }
}
// (2) per code: exclusive scan over blocks (in place), total count out
__global__ void __launch_bounds__(256) stats_scan_blocks_kernel(int* __restrict__ hist, int nblk, int K,
                                                                unsigned long long* __restrict__ counts,
                                                                long long* __restrict__ code_total) {
  int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= K) return;
  long long run = 0;
  for (int b = 0; b < nblk; ++b) {
    int h = hist[(long long)b * K + k];
    hist[(long long)b * K + k] = (int)run;     // rows per code < 2^31 per rank
    run += h;
  }
  code_total[k] = run;
  if (counts) atomicAdd(counts + k, (unsigned long long)run);
}
// (2b) the same per (chunk, code): exclusive scan over the chunk's ranking blocks, segment size out (chunk-major)
__global__ void __launch_bounds__(256) stats_scan_chunks_kernel(int* __restrict__ hist, int nblk, int K, int blocks_per_chunk,
                                                                int n_chunks, unsigned long long* __restrict__ counts,
                                                                long long* __restrict__ seg_total) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)n_chunks * K) return;
  const int c = (int)(t / K), k = (int)(t % K);
  const int b1 = min(nblk, (c + 1) * blocks_per_chunk);
  long long run = 0;
  for (int b0 = c * blocks_per_chunk; b0 < b1; b0 += 8) {        // eight loads in flight, then the dependent stores
    int h[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) h[u] = b0 + u < b1 ? hist[(long long)(b0 + u) * K + k] : 0;
#pragma unroll
    for (int u = 0; u < 8; ++u)
      if (b0 + u < b1) { hist[(long long)(b0 + u) * K + k] = (int)run; run += h[u]; }
  }
  seg_total[t] = run;
  if (counts && run) atomicAdd(counts + k, (unsigned long long)run);
}
// (3) exclusive scan over codes / (chunk, code) segments: tiles of 4096 elements, one block each -- tile totals first
// (skipped for a single tile), then every block adds up the totals of the tiles before it and scans its own tile
// (a single block walking config 4's 313 k segments took 160-350 us)
constexpr int kScanTile = 4096;
__global__ void __launch_bounds__(1024) stats_scan_totals_kernel(const long long* __restrict__ in, long long L,
                                                                 long long* __restrict__ tile_tot) {
  __shared__ long long s_warp[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long base = (long long)blockIdx.x * kScanTile + threadIdx.x;
  long long s = 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) s += base + 1024 * i < L ? in[base + 1024 * i] : 0;
#pragma unroll
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) s_warp[warp] = s;
  __syncthreads();
  if (warp == 0) {
    s = s_warp[lane];
#pragma unroll
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) tile_tot[blockIdx.x] = s;
  }
}
__global__ void __launch_bounds__(1024) stats_scan_codes_kernel(const long long* __restrict__ in, long long L,
                                                                long long* __restrict__ out /* L + 1 */,
                                                                const long long* __restrict__ tile_tot) {
  __shared__ long long s_warp[32];
  __shared__ long long s_off;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // offset of this tile = the totals of the tiles before it
  long long o = 0;
  for (long long b = threadIdx.x; b < (long long)blockIdx.x; b += 1024) o += tile_tot[b];
#pragma unroll
  for (int w = 16; w; w >>= 1) o += __shfl_xor_sync(0xffffffffu, o, w);
  if (lane == 0) s_warp[warp] = o;
  __syncthreads();
  if (warp == 0) {
    o = s_warp[lane];
#pragma unroll
    for (int w = 16; w; w >>= 1) o += __shfl_xor_sync(0xffffffffu, o, w);
    if (lane == 0) s_off = o;
  }
  __syncthreads();
  const long long off = s_off;
  // thread t scans elements 4t .. 4t+3 of the tile
  const long long base = (long long)blockIdx.x * kScanTile + 4 * threadIdx.x;
  long long v[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) v[i] = base + i < L ? in[base + i] : 0;
  const long long t = v[0] + v[1] + v[2] + v[3];
  long long inc = t;
#pragma unroll
  for (int w = 1; w < 32; w <<= 1) { const long long u = __shfl_up_sync(0xffffffffu, inc, w); if (lane >= w) inc += u; }
  __syncthreads();                                  // (s_warp is reused)
  if (lane == 31) s_warp[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    const long long wv = s_warp[lane];
    long long winc = wv;
#pragma unroll
    for (int w = 1; w < 32; w <<= 1) { const long long u = __shfl_up_sync(0xffffffffu, winc, w); if (lane >= w) winc += u; }
    s_warp[lane] = winc - wv;
    if (lane == 31 && blockIdx.x == gridDim.x - 1) out[L] = off + winc;
  }
  __syncthreads();
  long long run = off + s_warp[warp] + inc - t;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    if (base + i < L) out[base + i] = run;
    run += v[i];
  }
}
// launcher: `scratch` holds one long long per tile (callers lend the front of `perm`, which the scatter fills later)
static int launch_scan_codes(const long long* in, long long L, long long* out, long long* scratch, cudaStream_t st) {
  const long long tiles = (L + kScanTile - 1) / kScanTile;
  if (tiles > 1) {
    stats_scan_totals_kernel<<<(unsigned)tiles, 1024, 0, st>>>(in, L, scratch);
    VQSEG_LAUNCH_CHECK();
  }
  stats_scan_codes_kernel<<<(unsigned)tiles, 1024, 0, st>>>(in, L, out, scratch);
  VQSEG_LAUNCH_CHECK();
  return 0;
}
// (4) stable scatter: perm[code_start[k] + hist[blk][k] + rank_in_block] = n
// `blocks_per_chunk` > 0: the sort key is (chunk of blocks_per_chunk ranking blocks, code): code_start then holds one
// row of K segment starts per chunk.
__global__ void __launch_bounds__(1024) stats_scatter_kernel(const long long* __restrict__ idx, long long n_rows, int K,
                                                             const int* __restrict__ hist,
                                                             const long long* __restrict__ code_start,
                                                             int* __restrict__ perm, int blocks_per_chunk = 0,
                                                             int* __restrict__ pcode = nullptr) {
  if (blocks_per_chunk > 0) code_start += (long long)(blockIdx.x / blocks_per_chunk) * K;
  extern __shared__ int s_run[];    // K running counters
  for (int k = threadIdx.x; k < K; k += blockDim.x) s_run[k] = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long n = (long long)blockIdx.x * kSortBlock + threadIdx.x;
  long long k = n < n_rows ? idx[n] : -1;
  const bool valid = k >= 0 && k < K;
  const int kk = valid ? (int)k : -1 - lane;            // unique key for invalid lanes
  const unsigned peers = __match_any_sync(0xffffffffu, kk);
  const int rank_in_warp = __popc(peers & ((1u << lane) - 1));
  const int group = __popc(peers);
  const bool leader = rank_in_warp == 0;
  // (the global reads happen BEFORE the turns: inside them their latency was paid 32 times per block, 520 us of
  // config 4's ordered statistics)
  const long long off = valid ? code_start[kk] + hist[(long long)blockIdx.x * K + kk] + rank_in_warp : 0;
  int base = 0;
  for (int w = 0; w < 32; ++w) {          // warps take turns in row order -> stable
    if (warp == w && valid) {
      base = s_run[kk];
      __syncwarp(peers);
      if (leader) s_run[kk] = base + group;
    }
    __syncthreads();
  }
  if (valid) {
    perm[off + base] = (int)n;
    if (pcode) pcode[off + base] = kk;
  }
}
// (4b) the same without the turns, for K up to ~3000: every warp leaves its per-code group sizes in its own row of a
// [32 warps][K] table of 16-bit counters, one pass per code turns the table into exclusive prefixes over the warps
// (the turn-taking version spent 500 us on config 4's 10 M rows: 32 block-wide barriers per 1024 rows)
__global__ void __launch_bounds__(1024) stats_scatter_table_kernel(const long long* __restrict__ idx, long long n_rows, int K,
                                                                   const int* __restrict__ hist,
                                                                   const long long* __restrict__ code_start,
                                                                   int* __restrict__ perm, int blocks_per_chunk,
                                                                   int* __restrict__ pcode) {
  if (blocks_per_chunk > 0) code_start += (long long)(blockIdx.x / blocks_per_chunk) * K;
  extern __shared__ unsigned short s_cnt[];            // [32][Ke], Ke = K rounded up to even
  const int Ke = (K + 1) & ~1;
  for (int i = threadIdx.x; i < 16 * Ke; i += blockDim.x) reinterpret_cast<uint32_t*>(s_cnt)[i] = 0u;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long n = (long long)blockIdx.x * kSortBlock + threadIdx.x;
  long long k = n < n_rows ? idx[n] : -1;
  const bool valid = k >= 0 && k < K;
  const int kk = valid ? (int)k : -1 - lane;            // unique key for invalid lanes
  const unsigned peers = __match_any_sync(0xffffffffu, kk);
  const int rank_in_warp = __popc(peers & ((1u << lane) - 1));
  const long long off = valid ? code_start[kk] + hist[(long long)blockIdx.x * K + kk] + rank_in_warp : 0;
  __syncthreads();
  if (valid && rank_in_warp == 0) s_cnt[warp * Ke + kk] = (unsigned short)__popc(peers);
  __syncthreads();
  for (int c = threadIdx.x; c < K; c += blockDim.x) {
    unsigned run = 0;
#pragma unroll
    for (int w = 0; w < 32; ++w) { const unsigned v = s_cnt[w * Ke + c]; s_cnt[w * Ke + c] = (unsigned short)run; run += v; }
  }
  __syncthreads();
  if (valid) {
    const long long pos = off + s_cnt[warp * Ke + kk];
    perm[pos] = (int)n;
    if (pcode) pcode[pos] = kk;                  // (the unordered sorted-sum kernel reads the code beside the row id)
  }
}
// (5) ordered per-code sums: ascending-row fp32 chain per (k, d).
// Packed rows (sD == 1, B == 1): one warp per (code, 128-dim slab), float4 per lane, 16 rows in flight (the row
// ids of the next batch are fetched lane-parallel and broadcast with shuffles).  The chain of a code is
// inherently sequential (that is what makes it bit-exact), so the critical path is max_k count[k] * latency / 16.
// `big_counts` (optional, with `big_thr`): codes holding more than big_thr rows are left to
// stats_ordered_sum_big_kernel below.
__global__ void __launch_bounds__(256) stats_ordered_sum_rows_kernel(const float* __restrict__ x, long long row_stride,
                                                                     int D, const int* __restrict__ perm,
                                                                     const long long* __restrict__ code_start, int K,
                                                                     float* __restrict__ sums, int n_chunks,
                                                                     const unsigned long long* __restrict__ big_counts,
                                                                     unsigned long long big_thr) {
  const int slabs = (D + 127) / 128;
  const int lane = threadIdx.x & 31;
  const long long wid = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (wid >= (long long)K * slabs) return;
  const int k = (int)(wid / slabs), d = (int)(wid % slabs) * 128 + 4 * lane;
  if (big_counts && big_counts[k] > big_thr) return;
  const bool act = d < D;                       // D % 4 == 0 is guaranteed by the launcher
  float4 s = act ? *reinterpret_cast<const float4*>(sums + (long long)k * D + d) : make_float4(0.f, 0.f, 0.f, 0.f);
  const float* xd = x + (act ? d : 0);
  // n_chunks > 1: the (chunk, code) segments of this code one after the other (packed rows of a flat array: the row
  // ranges are visited in order by every warp, which keeps the accesses of the whole grid within a few ranges)
  long long beg = code_start[k], end = code_start[k + 1];
  int nxt = (beg + lane < end) ? __ldg(perm + beg + lane) : 0;          // row ids of the next 32 rows, one per lane
  for (int c = 0; c < n_chunks; ++c) {
    long long nbeg = 0, nend = 0;
    int nfirst = 0;
    if (c + 1 < n_chunks) {                     // the next segment's bounds and first row ids while this one is summed
      const long long* cs = code_start + (long long)(c + 1) * K + k;
      nbeg = __ldg(cs); nend = __ldg(cs + 1);
      nfirst = (nbeg + lane < nend) ? __ldg(perm + nbeg + lane) : 0;
    }
    long long j = beg;
    while (j < end) {
      const int ids = nxt;
      const long long jn = j + 32;
      nxt = (jn + lane < end) ? __ldg(perm + jn + lane) : 0;
      const int cnt = (int)min((long long)32, end - j);
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        if (16 * h >= cnt) break;
        float4 v[16];
#pragma unroll
        for (int u = 0; u < 16; ++u) {
          // UNCONDITIONAL loads (rows past the end re-read the last valid row and are simply not added): with a
          // predicate on the load the compiler fuses it with the predicated add below and the 16 loads serialise
          const int r = __shfl_sync(0xffffffffu, ids, min(16 * h + u, cnt - 1));
          v[u] = __ldg(reinterpret_cast<const float4*>(xd + (long long)r * row_stride));
        }
#pragma unroll
        for (int u = 0; u < 16; ++u) {
          if (16 * h + u < cnt) {
            s.x = __fadd_rn(s.x, v[u].x); s.y = __fadd_rn(s.y, v[u].y);
            s.z = __fadd_rn(s.z, v[u].z); s.w = __fadd_rn(s.w, v[u].w);
          }
        }
      }
      j = jn;
    }
    beg = nbeg; end = nend; nxt = nfirst;
  }
  if (act) *reinterpret_cast<float4*>(sums + (long long)k * D + d) = s;
}

// Big clusters (more than big_thr rows): a code's (k, d) chains are as long as its cluster and strictly sequential, so
// what bounds them is how fast ONE warp gets through the rows -- 16 rows in flight in registers above, i.e. ~13-25 rows
// per microsecond of memory latency.  Here a warp owns 32 dims of one big code and streams its rows through a
// shared-memory ring with 16-byte cp.async (4-byte requests issue too slowly): sixteen groups of up to 32 rows (128 B
// each) in flight, the row ids themselves requested thirty-two groups ahead; the adds run out of shared memory in row
// order.  One warp per block: four warps on one SM ran at a quarter of the rate each.  Measured (10 M x 512, one cluster
// holding 5-50 % of the rows): 85-100 rows/us per chain against 25-30 before; ncu: memory stalls are gone (long
// scoreboard 2 % of samples), the warp is bound by its own ~180 instructions per 32 rows at ~4 cycles each.
constexpr int kBigGroups = 16, kBigIdsAhead = 32;
struct __align__(16) BigWarpSmem { float rows[kBigGroups][32][32]; int ids[kBigIdsAhead][32]; int cnt[kBigIdsAhead]; };
__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}
__global__ void __launch_bounds__(32) stats_ordered_sum_big_kernel(const float* __restrict__ x, long long row_stride, int D,
                                                                    const int* __restrict__ perm,
                                                                    const long long* __restrict__ seg_start, int K,
                                                                    float* __restrict__ sums, int n_chunks,
                                                                    const unsigned long long* __restrict__ counts,
                                                                    unsigned long long big_thr) {
  extern __shared__ __align__(16) unsigned char big_smem[];
  const int lane = threadIdx.x;
  const int slabs = (D + 31) / 32;
  const int k = (int)(blockIdx.x / slabs);
  if (!(counts[k] > big_thr)) return;
  const int d0 = (int)(blockIdx.x % slabs) * 32;
  const int d = d0 + lane;
  const bool act = d < D;
  BigWarpSmem& sm = *reinterpret_cast<BigWarpSmem*>(big_smem);
  const float* xd = x + (act ? d : 0);
  float s = act ? sums[(long long)k * D + d] : 0.f;
  // generator of id vectors: walks this code's (chunk, code) segments in order, up to 32 rows per vector
  int gc = 0;
  long long gj = seg_start[k], gend = seg_start[k + 1], nb = 0, ne = 0;
  if (n_chunks > 1) { nb = __ldg(seg_start + (long long)K + k); ne = __ldg(seg_start + (long long)K + k + 1); }
  auto generate = [&](int v) {
    while (gj >= gend && gc + 1 < n_chunks) {
      ++gc; gj = nb; gend = ne;
      if (gc + 1 < n_chunks) { nb = __ldg(seg_start + (long long)(gc + 1) * K + k); ne = __ldg(seg_start + (long long)(gc + 1) * K + k + 1); }
    }
    const int cnt = (int)min((long long)32, gend - gj);
    if (lane < cnt) cp_async4(&sm.ids[v % kBigIdsAhead][lane], perm + gj + lane);
    if (lane == 0) sm.cnt[v % kBigIdsAhead] = cnt;
    gj += cnt;
  };
  // a row's 32-dim segment is 128 B = eight 16-byte requests: lane l asks for quad l % 8 of row 4 i + l / 8.
  // (Tried: separate paths without per-row predicates for full vectors and a 32 x 32 -> 64 bit address multiply --
  // fewer instructions, yet 86 rows/us against 98: kept the plain form.)
  const int qd = lane & 7, qr = lane >> 3;
  const bool qact = d0 + 4 * qd < D;
  const float* xq = x + d0 + (qact ? 4 * qd : 0);
  auto issue_rows = [&](int v) {
    const int cnt = sm.cnt[v % kBigIdsAhead];
    const int my = sm.ids[v % kBigIdsAhead][lane];
    float* dst = &sm.rows[v % kBigGroups][qr][4 * qd];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int r = __shfl_sync(0xffffffffu, my, 4 * i + qr);
      if (4 * i + qr < cnt && qact) cp_async16(dst + 128 * i, xq + (long long)r * row_stride);
    }
  };
  for (int v = 0; v < kBigIdsAhead; ++v) generate(v);
  asm volatile("cp.async.commit_group;" ::: "memory");
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncwarp();
  for (int v = 0; v < kBigGroups; ++v) { issue_rows(v); asm volatile("cp.async.commit_group;" ::: "memory"); }
  for (int t = 0;; ++t) {
    asm volatile("cp.async.wait_group %0;" ::"n"(kBigGroups - 1) : "memory");   // group of vector t (rows) and t + 8 (ids) landed
    __syncwarp();
    const int cnt = sm.cnt[t % kBigIdsAhead];
    if (cnt == 0) break;
    const float* src = &sm.rows[t % kBigGroups][0][lane];
    float v[32];
#pragma unroll
    for (int u = 0; u < 32; ++u) v[u] = src[32 * u];
#pragma unroll
    for (int u = 0; u < 32; ++u)
      if (u < cnt) s = __fadd_rn(s, v[u]);
    __syncwarp();                                   // every lane is done with vector t's ids / cnt slots
    issue_rows(t + kBigGroups);
    generate(t + kBigIdsAhead);
    asm volatile("cp.async.commit_group;" ::: "memory");
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  if (act) sums[(long long)k * D + d] = s;
}

// Unordered statistics of LARGE packed inputs (deterministic = 0): the same counting sort, then every warp sums a
// window of 64 consecutive sorted positions x one 128-dim slab in registers and issues one vector RED per code it meets
// (two or three per window instead of one per row).  Rows of one code are spread over as many warps as the code has
// windows, so neither a hot code (same-address atomics: 44 ms for a code owning half of config 4's rows) nor a long
// chain exists: 3.3-3.5 ms whatever the clustering, against 4.6-5.0 ms for one RED per row.
constexpr int kSortedWin = 64;
constexpr long long kSortedMinRows = 1ll << 18;
__global__ void __launch_bounds__(256) stats_sorted_sum_kernel(const float* __restrict__ x, long long row_stride, int D,
                                                               const int* __restrict__ perm, const int* __restrict__ pcode,
                                                               const long long* __restrict__ total_ptr,
                                                               float* __restrict__ sums) {
  const int slabs = (D + 127) / 128;
  const int lane = threadIdx.x & 31;
  const long long wid = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long total = *total_ptr;
  const long long j0 = (wid / slabs) * kSortedWin;
  if (j0 >= total) return;
  const long long j1 = min(j0 + kSortedWin, total);
  const int d = (int)(wid % slabs) * 128 + 4 * lane;
  const bool act = d < D;
  const float* xd = x + (act ? d : 0);
  int cur = -1;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  auto flush = [&]() {
    if (cur >= 0 && act) atomicAdd(reinterpret_cast<float4*>(sums + (long long)cur * D + d), acc);
  };
  for (long long jb = j0; jb < j1; jb += 32) {
    const int cnt = (int)min((long long)32, j1 - jb);
    const int ids = lane < cnt ? __ldg(perm + jb + lane) : 0;
    const int cds = lane < cnt ? __ldg(pcode + jb + lane) : -1;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      if (16 * h >= cnt) break;
      float4 v[16];
#pragma unroll
      for (int u = 0; u < 16; ++u) {                     // unconditional loads (see stats_ordered_sum_rows_kernel)
        const int r = __shfl_sync(0xffffffffu, ids, min(16 * h + u, cnt - 1));
        v[u] = __ldg(reinterpret_cast<const float4*>(xd + (long long)r * row_stride));
      }
#pragma unroll
      for (int u = 0; u < 16; ++u) {
        if (16 * h + u < cnt) {
          const int c = __shfl_sync(0xffffffffu, cds, 16 * h + u);
          if (c != cur) { flush(); cur = c; acc = make_float4(0.f, 0.f, 0.f, 0.f); }
          acc.x += v[u].x; acc.y += v[u].y; acc.z += v[u].z; acc.w += v[u].w;
        }
      }
    }
  }
  flush();
}

// Any strides (NCHW feature maps): one warp per (code, 32-dim slab), lanes along d.
__global__ void __launch_bounds__(256) stats_ordered_sum_kernel(Rows x, const int* __restrict__ perm,
                                                                const long long* __restrict__ code_start, int K,
                                                                float* __restrict__ sums) {
  const int D = (int)x.D;
  const int slabs = (D + 31) / 32;
  const int lane = threadIdx.x & 31;
  const long long wid = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (wid >= (long long)K * slabs) return;
  const int k = (int)(wid / slabs), d = (int)(wid % slabs) * 32 + lane;
  const long long beg = code_start[k], end = code_start[k + 1];
  const bool act = d < D;
  float s = act ? sums[(long long)k * D + d] : 0.f;     // accumulate on top (caller zeroes; ranks chain)
  long long j = beg;
  int nxt = (j + lane < end) ? __ldg(perm + j + lane) : 0;
  while (j < end) {
    const int ids = nxt;
    const long long jn = j + 32;
    nxt = (jn + lane < end) ? __ldg(perm + jn + lane) : 0;
    const int cnt = (int)min((long long)32, end - j);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      float v[16];
#pragma unroll
      for (int u = 0; u < 16; ++u) {
        const int r = __shfl_sync(0xffffffffu, ids, min(16 * h + u, cnt - 1));     // unconditional loads, see above
        long long b, p;
        split_row(r, x.P, b, p);
        v[u] = __ldg(x.ptr + b * x.sB + p * x.sP + (long long)(act ? d : 0) * x.sD);
      }
#pragma unroll
      for (int u = 0; u < 16; ++u)
        if (16 * h + u < cnt) s = __fadd_rn(s, v[u]);
    }
    j = jn;
  }
  if (act) sums[(long long)k * D + d] = s;
}

// means = where(counts==0, means, sums / max(counts,1)) [ + l2norm ]      (vq_img.py:44-45,:53-61)
__global__ void __launch_bounds__(256) kmeans_finalize_kernel(const float* __restrict__ sums,
                                                              const long long* __restrict__ counts,
                                                              float* __restrict__ means, int K, int D, int cosine) {
  const int lane = threadIdx.x & 31;
  const long long k = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (k >= K) return;
  const long long c = counts[k];
  if (c == 0) return;                                   // empty cluster keeps its old mean
  const float cf = __ll2float_rn(c);
  for (int d = lane; d < D; d += 32) means[k * D + d] = __fdiv_rn(sums[k * D + d], cf);
  if (cosine) {
    // l2norm(new_means) on the contiguous (1, K, D) tensor (vq_img.py:53-54): ATen's last-dim order, lanes 0-7
    __syncwarp();
    float nrm = 0.f;
    if (lane < 8) nrm = fmaxf(aten_norm_lastdim8(means + k * D, D, lane), 1e-12f);
    nrm = __shfl_sync(0xffffffffu, nrm, 0);
    for (int d = lane; d < D; d += 32) means[k * D + d] = __fdiv_rn(means[k * D + d], nrm);
  }
}

__global__ void __launch_bounds__(256) code_usage_kernel(const long long* __restrict__ counts, int K, float* out) {
  __shared__ int s_red[256];
  int z = 0;
  for (int k = threadIdx.x; k < K; k += 256) z += counts[k] == 0;
  s_red[threadIdx.x] = z;
  __syncthreads();
  for (int o = 128; o; o >>= 1) { if (threadIdx.x < o) s_red[threadIdx.x] += s_red[threadIdx.x + o]; __syncthreads(); }
  if (threadIdx.x == 0) *out = __fmul_rn(100.f, __fdiv_rn((float)s_red[0], (float)K));   // 100 * (zero / K)
}

__global__ void __launch_bounds__(256) gather_rows_kernel(Rows x, const long long* __restrict__ ids, long long n_ids,
                                                          float* __restrict__ out) {
  const int D = (int)x.D;
  const long long total = n_ids * D;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    long long r = i / D; int d = (int)(i % D);
    long long n = ids[r];
    out[i] = (n >= 0 && n < x.n_rows()) ? x.row(n)[(long long)d * x.sD] : 0.f;
  }
}

__global__ void __launch_bounds__(256) unpack_keys_kernel(const unsigned long long* __restrict__ keys, long long n,
                                                          long long* __restrict__ idx_out, float* __restrict__ dist_out,
                                                          unsigned long long* __restrict__ counts, long long K) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    unsigned long long key = keys[i];
    long long k = (long long)(key & 0xffffffffull);
    if (idx_out) idx_out[i] = k;
    if (dist_out) dist_out[i] = __uint_as_float((unsigned)(key >> 32));
    if (counts && k < K) atomicAdd(counts + k, 1ull);
  }
}

// ---- F.normalize(t, p=2, dim=-1) = t / max(||t||, 1e-12) in ATen's CPU arithmetic (vq_img.py:7-8) --------------------
// Probed on the reference's CPU path (torch 2.11, tests/golden/make_golden_cosine.py and tests/test_layout_rules.py
// pin it).  ATen picks the order by the stride of the reduced dim ALONE, whatever sB, sP and the output's strides are:
//  * sD == 1 (code rows, k-means means, channels-last maps and their batch slices, 1 x 1 maps): ATen's vectorised
//    last-dim reduction: eight lane accumulators a_l += fl(v * v) over elements l, l + 8, ..., summed
//    a_0 + a_1 + ... + a_7 in order, then the D % 8 tail: four separately rounded fl(v * v) adds if at least four
//    remain, fused multiply-adds for the last <= 3;
//  * any other sD (the 'b c h w -> b (h w) c' view of an NCHW map, vq_img.py:232, which is what the cosine codebook
//    normalises, :97) is one sequential chain acc = fl(acc + fl(v * v)) in channel order;
//  * sqrt and the division are IEEE round-to-nearest.
// Eight lanes own a row with sD == 1 (lane l = accumulator l); one thread owns a strided row (pixel-contiguous maps:
// a warp reads 32 neighbouring pixels of one channel).
__global__ void __launch_bounds__(256) l2norm_lastdim_kernel(Rows x, RowsOut out) {
  const int l8 = threadIdx.x & 7;
  const long long n = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 3;
  const bool on = n < x.n_rows();                        // (whole groups of 8 lanes are on or off together)
  const int D = (int)x.D;
  const float* row = x.row(on ? n : 0);
  const float nrm = fmaxf(aten_norm_lastdim8(row, on ? D : 0, l8), 1e-12f);
  if (!on) return;
  float* o = out.row(n);
  for (int d = l8; d < D; d += 8) o[(long long)d * out.sD] = __fdiv_rn(row[d], nrm);   // in place is fine: each element is read by its writer
}

// pixel-contiguous maps (sP == 1): a block owns 32 neighbouring pixels of one image.  All eight warps stage 256
// channels x 32 pixels (coalesced 128-byte lines) in shared memory, warp 0 runs the 32 sequential chains over them
// (lane = pixel), chunk after chunk; then all warps divide (second read of x: L2).  The thread-per-pixel kernel below
// had 32768 threads on the config-2 map, each waiting on 2 x 256 dependent strided loads: 99 us.
__global__ void __launch_bounds__(256) l2norm_px_kernel(Rows x, RowsOut out) {
  __shared__ float tile[256 * 32];
  __shared__ float s_nrm[32];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int D = (int)x.D;
  const long long groups_per_image = (x.P + 31) / 32;
  for (long long gidx = blockIdx.x; gidx < x.B * groups_per_image; gidx += gridDim.x) {
    const long long b = gidx / groups_per_image, p = (gidx % groups_per_image) * 32 + lane;
    const bool on = p < x.P;
    const float* xp = x.ptr + b * x.sB + (on ? p : 0);
    float acc = 0.f;
    for (int d0 = 0; d0 < D; d0 += 256) {
      const int dn = min(256, D - d0);
      __syncthreads();
      for (int j = wib; j < dn; j += 8) tile[j * 32 + lane] = on ? __ldg(xp + (long long)(d0 + j) * x.sD) : 0.f;
      __syncthreads();
      if (wib == 0) {
        int j = 0;
        for (; j + 8 <= dn; j += 8) {                 // loads and squares of 8 terms ahead of the dependent adds
          float q[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) { const float v = tile[(j + u) * 32 + lane]; q[u] = __fmul_rn(v, v); }
#pragma unroll
          for (int u = 0; u < 8; ++u) acc = __fadd_rn(acc, q[u]);
        }
        for (; j < dn; ++j) { const float v = tile[j * 32 + lane]; acc = __fadd_rn(acc, __fmul_rn(v, v)); }
      }
    }
    if (wib == 0) s_nrm[lane] = fmaxf(__fsqrt_rn(acc), 1e-12f);
    __syncthreads();
    const float nrm = s_nrm[lane];
    float* op = out.ptr + b * out.sB + (on ? p : 0) * out.sP;
    if (on) {
      if (D <= 256) {                                  // the whole row is still in the tile
        for (int d = wib; d < D; d += 8) op[(long long)d * out.sD] = __fdiv_rn(tile[d * 32 + lane], nrm);
      } else {
        for (int d = wib; d < D; d += 8) op[(long long)d * out.sD] = __fdiv_rn(__ldg(xp + (long long)d * x.sD), nrm);
      }
    }
  }
}

__global__ void __launch_bounds__(256) l2norm_strided_kernel(Rows x, RowsOut out) {
  const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= x.n_rows()) return;
  const float* xr = x.row(n);
  const int D = (int)x.D;
  float acc = 0.f;
  for (int d = 0; d < D; ++d) { const float v = xr[(long long)d * x.sD]; acc = __fadd_rn(acc, __fmul_rn(v, v)); }
  const float nrm = fmaxf(__fsqrt_rn(acc), 1e-12f);
  float* o = out.row(n);
  for (int d = 0; d < D; ++d) o[(long long)d * out.sD] = __fdiv_rn(xr[(long long)d * x.sD], nrm);
}

static inline unsigned grid_for(long long total, int threads, int waves = 8) {
  long long blocks = (total + threads - 1) / threads;
  long long cap = (long long)num_sms() * waves;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (unsigned)blocks;
}

// =================================================================================================
// EMA codebook update (opt-in extension, SURVEY.md 8f-4; NOT in the reference, which stores `decay` / `eps` unused:
// parity unpinned -- the standard VQ-VAE equations, as in lucidrains/vector-quantize-pytorch from which the
// reference derives):  cluster_size <- decay cluster_size + (1 - decay) counts;  embed_avg <- decay embed_avg +
// (1 - decay) sums;  n = sum(cluster_size);  cs = (cluster_size + eps) / (n + K eps) n;  weight = embed_avg / cs.
// =================================================================================================
// Dead-code expiry (EXPIRE, vqseg_ema_update_expire_f32): a code whose updated cluster_size is < threshold takes the
// next candidate row in ascending k (slot = exclusive prefix of the expired mask), as lucidrains's boolean-mask
// `replace`.  The smoothing's n is summed before any reset, so live codes get exactly what the EXPIRE=false
// instantiation (vqseg_ema_update_f32) writes.
template <bool EXPIRE>
__global__ void __launch_bounds__(256) ema_cluster_kernel(const long long* __restrict__ counts, float* __restrict__ cluster_size,
                                                          int K, float decay, float* __restrict__ total_out,
                                                          float threshold, int* __restrict__ slot,
                                                          long long* __restrict__ expired_out) {
  __shared__ double s_red[256];
  __shared__ int s_warp[2][8];                   // per-warp expired counts, double-buffered: one barrier per 256 codes
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  double s = 0.0;
  int offset = 0;                                // expired codes below this chunk
  auto update = [&](int k) {
    const float cs = __fadd_rn(__fmul_rn(cluster_size[k], decay), __fmul_rn(1.f - decay, (float)counts[k]));
    cluster_size[k] = cs;
    s += (double)cs;
    return cs;
  };
  if constexpr (!EXPIRE) {
    for (int k = threadIdx.x; k < K; k += 256) update(k);
  } else {
    // chunks of 256 codes: thread t still owns k = t, t + 256, ... in increasing order, so s sums in the same order
    for (int k0 = 0; k0 < K; k0 += 256) {
      const int k = k0 + threadIdx.x;
      const bool dead = k < K && update(k) < threshold;
      const unsigned ballot = __ballot_sync(0xffffffffu, dead);
      const int buf = (k0 >> 8) & 1;
      if (lane == 0) s_warp[buf][wid] = __popc(ballot);
      __syncthreads();
      int below = 0, chunk = 0;
#pragma unroll
      for (int w = 0; w < 8; ++w) {
        const int c = s_warp[buf][w];
        below += w < wid ? c : 0;
        chunk += c;
      }
      if (k < K) slot[k] = dead ? offset + below + __popc(ballot & ((1u << lane) - 1u)) : -1;
      offset += chunk;
    }
  }
  s_red[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o; o >>= 1) {
    if ((int)threadIdx.x < o) s_red[threadIdx.x] += s_red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    *total_out = (float)s_red[0];
    if constexpr (EXPIRE) {
      if (expired_out) {
        expired_out[0] = offset;
        expired_out[1] += offset;
      }
    }
  }
}

template <bool EXPIRE>
__global__ void __launch_bounds__(256) ema_embed_kernel(const float* __restrict__ sums, float* __restrict__ cluster_size,
                                                        const float* __restrict__ total, float* __restrict__ embed_avg,
                                                        float* __restrict__ weight, int K, int D, float decay, float eps,
                                                        const int* __restrict__ slot, const float* __restrict__ cand,
                                                        float reset) {
  const int k = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (k >= K) return;
  if constexpr (EXPIRE) {
    const int r = __ldg(slot + k);
    if (r >= 0) {                                // this warp owns code k: nothing else reads or writes its rows
      const float* c = cand + (long long)r * D;
      for (int d = lane; d < D; d += 32) {
        const long long i = (long long)k * D + d;
        const float v = __ldg(c + d);
        weight[i] = v;
        embed_avg[i] = __fmul_rn(v, reset);
      }
      if (lane == 0) cluster_size[k] = reset;
      return;
    }
  }
  const float n = __ldg(total);
  const float cs = __fmul_rn(__fdiv_rn(__fadd_rn(cluster_size[k], eps), __fadd_rn(n, __fmul_rn((float)K, eps))), n);
  for (int d = lane; d < D; d += 32) {
    const long long i = (long long)k * D + d;
    const float ea = __fadd_rn(__fmul_rn(embed_avg[i], decay), __fmul_rn(1.f - decay, sums[i]));
    embed_avg[i] = ea;
    weight[i] = __fdiv_rn(ea, cs);
  }
}

}  // namespace vqseg

using namespace vqseg;

// one pass of the deterministic statistics over a row range (accumulates on top of counts / sums)
// Rows [row0, row0 + n) of a strided (B, P, D) view copied into packed (n, D) rows: 32 x 32 tiles through a padded
// shared-memory transpose (pixel-contiguous NCHW maps: reads coalesced along pixels, writes along dims).  The per-code
// statistics of such maps run on the packed copy: scattering them from the strided layout costs one 32-byte sector per
// 4-byte element (ncu, config-2 map: 765 us atomic / 1328 us ordered against ~25 us for pack + the row kernels).
__global__ void __launch_bounds__(256) pack_rows_kernel(Rows x, long long row0, long long n, float* __restrict__ out) {
  __shared__ float tile[8][32 * 33];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int D = (int)x.D;
  const int n_dchunks = (D + 31) / 32;
  float* t = tile[wib];
  for (long long rt = blockIdx.x; rt * 32 < n; rt += gridDim.x) {
    const long long r = rt * 32 + lane;                          // this lane's row while reading
    const float* xr = x.row(row0 + (r < n ? r : n - 1));
    for (int c = wib; c < n_dchunks; c += 8) {
      const int d0 = c * 32;
      __syncwarp();
#pragma unroll 8
      for (int j = 0; j < 32; ++j) t[j * 33 + lane] = (d0 + j < D) ? __ldg(xr + (long long)(d0 + j) * x.sD) : 0.f;
      __syncwarp();
      if (d0 + lane < D) {
#pragma unroll 8
        for (int i = 0; i < 32; ++i)
          if (rt * 32 + i < n) out[(rt * 32 + i) * D + d0 + lane] = t[lane * 33 + i];
      }
    }
  }
}

static int launch_scatter(const long long* idx, long long n_rows, int K, const int* hist, const long long* code_start,
                          int* perm, int blocks_per_chunk, long long nblk, cudaStream_t st, int* pcode = nullptr) {
  const size_t table = (size_t)32 * ((K + 1) & ~1) * sizeof(unsigned short);
  if (table <= 96 * 1024) {
    static size_t tconf[kMaxDevices] = {0};
    if (int rc = ensure_dynamic_smem(stats_scatter_table_kernel, table, tconf)) return rc;
    stats_scatter_table_kernel<<<(unsigned)nblk, kSortBlock, table, st>>>(idx, n_rows, K, hist, code_start, perm, blocks_per_chunk, pcode);
  } else {
    const size_t smem = (size_t)K * sizeof(int);
    static size_t configured[kMaxDevices] = {0};
    if (int rc = ensure_dynamic_smem(stats_scatter_kernel, smem, configured)) return rc;
    stats_scatter_kernel<<<(unsigned)nblk, kSortBlock, smem, st>>>(idx, n_rows, K, hist, code_start, perm, blocks_per_chunk, pcode);
  }
  VQSEG_LAUNCH_CHECK();
  return 0;
}
static int stats_det_range(const float* x, long long B, long long P, long long D, long long sB, long long sP, long long sD,
                           const int64_t* idx, long long K, int64_t* counts, float* sums, void* ws, cudaStream_t st) {
  const long long n_rows = B * P;
  Rows xr{x, B, P, D, sB, sP, sD};
  const long long nblk = (n_rows + kSortBlock - 1) / kSortBlock;
  char* p = (char*)ws;
  int* hist = (int*)p;                    p += round_up(nblk * K * sizeof(int), 256);
  long long* code_total = (long long*)p;  p += round_up(K * sizeof(long long), 256);
  long long* code_start = (long long*)p;  p += round_up((K + 1) * sizeof(long long), 256);
  int* perm = (int*)p;
  cudaError_t e = cudaMemsetAsync(hist, 0, nblk * K * sizeof(int), st);
  if (e != cudaSuccess) return (int)e;
  stats_hist_kernel<<<(unsigned)nblk, kSortBlock, 0, st>>>((const long long*)idx, n_rows, (int)K, hist);
  VQSEG_LAUNCH_CHECK();
  stats_scan_blocks_kernel<<<(unsigned)((K + 255) / 256), 256, 0, st>>>(hist, (int)nblk, (int)K,
                                                                         (unsigned long long*)counts, code_total);
  VQSEG_LAUNCH_CHECK();
  if (int rc = launch_scan_codes(code_total, K, code_start, reinterpret_cast<long long*>(perm), st)) return rc;
  if (int rc = launch_scatter((const long long*)idx, n_rows, (int)K, hist, code_start, perm, 0, nblk, st)) return rc;
  const bool packed = B == 1 && sD == 1 && D % 4 == 0 && sP % 4 == 0 &&
                      (reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(sums) & 15) == 0;
  if (packed) {
    const long long warps = K * ((D + 127) / 128);
    stats_ordered_sum_rows_kernel<<<(unsigned)((warps * 32 + 255) / 256), 256, 0, st>>>(x, sP, (int)D, perm, code_start,
                                                                                        (int)K, sums, 1, nullptr, 0ull);
  } else {
    const long long warps = K * ((D + 31) / 32);
    stats_ordered_sum_kernel<<<(unsigned)((warps * 32 + 255) / 256), 256, 0, st>>>(xr, perm, code_start, (int)K, sums);
  }
  VQSEG_LAUNCH_CHECK();
  return 0;
}

extern "C" {

size_t vqseg_gather_workspace_bytes(int64_t n_rows, int64_t D) {
  long long tiles = ((n_rows + kGPix - 1) / kGPix) * ((D + kGTile - 1) / kGTile);
  long long generic = (long long)num_sms() * 16;
  long long n = tiles > generic ? tiles : generic;
  return (size_t)round_up(n * sizeof(float), 256);
}

int vqseg_gather_ste_f32(const float* x, int64_t B, int64_t P, int64_t D, int64_t sB, int64_t sP, int64_t sD,
                         const float* E, int64_t K, const int64_t* idx,
                         float* q_out, int64_t qB, int64_t qP, int64_t qD,
                         float* loss_out, int mode, void* ws, size_t ws_bytes, void* stream) {
  if (!E || !idx || !q_out || B < 0 || P < 0 || D <= 0 || K <= 0) return VQSEG_EINVAL;
  const bool train = gather_train(mode);
  if (train && !x) return VQSEG_EINVAL;
  if (B * P == 0) return 0;
  Rows xr{x, B, P, D, sB, sP, sD};
  if (!train) { xr.ptr = nullptr; xr.sB = qB; xr.sP = qP; xr.sD = qD; }
  RowsOut qr{q_out, B, P, D, qB, qP, qD};
  cudaStream_t st = (cudaStream_t)stream;
  float* partial = (float*)ws;
  size_t cap = ws ? ws_bytes / sizeof(float) : 0;
  const long long* ix = (const long long*)idx;
  switch (mode) {
    case VQSEG_MODE_EVAL:      return launch_gather<VQSEG_MODE_EVAL>(xr, E, (int)K, ix, qr, nullptr, partial, cap, st);
    case VQSEG_MODE_EVAL_AMP:  return launch_gather<VQSEG_MODE_EVAL_AMP>(xr, E, (int)K, ix, qr, nullptr, partial, cap, st);
    case VQSEG_MODE_TRAIN:     return launch_gather<VQSEG_MODE_TRAIN>(xr, E, (int)K, ix, qr, loss_out, partial, cap, st);
    case VQSEG_MODE_TRAIN_AMP: return launch_gather<VQSEG_MODE_TRAIN_AMP>(xr, E, (int)K, ix, qr, loss_out, partial, cap, st);
    case VQSEG_MODE_EVAL_AMP_BF16:  return launch_gather<VQSEG_MODE_EVAL_AMP_BF16>(xr, E, (int)K, ix, qr, nullptr, partial, cap, st);
    case VQSEG_MODE_TRAIN_AMP_BF16: return launch_gather<VQSEG_MODE_TRAIN_AMP_BF16>(xr, E, (int)K, ix, qr, loss_out, partial, cap, st);
    case VQSEG_MODE_TRAIN | VQSEG_MODE_ROTATE: return launch_gather<VQSEG_MODE_TRAIN | VQSEG_MODE_ROTATE>(xr, E, (int)K, ix, qr, loss_out, partial, cap, st);
    case VQSEG_MODE_TRAIN_AMP | VQSEG_MODE_ROTATE: return launch_gather<VQSEG_MODE_TRAIN_AMP | VQSEG_MODE_ROTATE>(xr, E, (int)K, ix, qr, loss_out, partial, cap, st);
    case VQSEG_MODE_TRAIN_AMP_BF16 | VQSEG_MODE_ROTATE: return launch_gather<VQSEG_MODE_TRAIN_AMP_BF16 | VQSEG_MODE_ROTATE>(xr, E, (int)K, ix, qr, loss_out, partial, cap, st);
  }
  return VQSEG_EINVAL;
}

// vqseg_gather_ste_f32 for the fused forward: `ticket` (an int the caller has zeroed on this stream) lets the
// kernel's last block reduce the loss, so no separate reduction launch follows
int vqseg_internal_gather_ticket(const float* x, int64_t B, int64_t P, int64_t D, int64_t sB, int64_t sP, int64_t sD,
                                 const float* E, int64_t K, const int64_t* idx,
                                 float* q_out, int64_t qB, int64_t qP, int64_t qD, float* loss_out, int mode,
                                 void* ws, size_t ws_bytes, void* stream, int* ticket,
                                 const int64_t* counts, float* usage_out) {
  if (!E || !idx || !q_out || B < 0 || P < 0 || D <= 0 || K <= 0) return VQSEG_EINVAL;
  const bool train = gather_train(mode);
  if (train && !x) return VQSEG_EINVAL;
  if (B * P == 0) return 0;
  Rows xr{x, B, P, D, sB, sP, sD};
  if (!train) { xr.ptr = nullptr; xr.sB = qB; xr.sP = qP; xr.sD = qD; }
  RowsOut qr{q_out, B, P, D, qB, qP, qD};
  cudaStream_t st = (cudaStream_t)stream;
  float* partial = (float*)ws;
  size_t cap = ws ? ws_bytes / sizeof(float) : 0;
  const long long* ix = (const long long*)idx;
  const unsigned long long* cu = (const unsigned long long*)counts;
  switch (mode) {
    case VQSEG_MODE_EVAL:      return launch_gather<VQSEG_MODE_EVAL>(xr, E, (int)K, ix, qr, nullptr, partial, cap, st, ticket, cu, usage_out);
    case VQSEG_MODE_EVAL_AMP:  return launch_gather<VQSEG_MODE_EVAL_AMP>(xr, E, (int)K, ix, qr, nullptr, partial, cap, st, ticket, cu, usage_out);
    case VQSEG_MODE_TRAIN:     return launch_gather<VQSEG_MODE_TRAIN>(xr, E, (int)K, ix, qr, loss_out, partial, cap, st, ticket, cu, usage_out);
    case VQSEG_MODE_TRAIN_AMP: return launch_gather<VQSEG_MODE_TRAIN_AMP>(xr, E, (int)K, ix, qr, loss_out, partial, cap, st, ticket, cu, usage_out);
    case VQSEG_MODE_EVAL_AMP_BF16:  return launch_gather<VQSEG_MODE_EVAL_AMP_BF16>(xr, E, (int)K, ix, qr, nullptr, partial, cap, st, ticket, cu, usage_out);
    case VQSEG_MODE_TRAIN_AMP_BF16: return launch_gather<VQSEG_MODE_TRAIN_AMP_BF16>(xr, E, (int)K, ix, qr, loss_out, partial, cap, st, ticket, cu, usage_out);
    case VQSEG_MODE_TRAIN | VQSEG_MODE_ROTATE: return launch_gather<VQSEG_MODE_TRAIN | VQSEG_MODE_ROTATE>(xr, E, (int)K, ix, qr, loss_out, partial, cap, st, ticket, cu, usage_out);
    case VQSEG_MODE_TRAIN_AMP | VQSEG_MODE_ROTATE: return launch_gather<VQSEG_MODE_TRAIN_AMP | VQSEG_MODE_ROTATE>(xr, E, (int)K, ix, qr, loss_out, partial, cap, st, ticket, cu, usage_out);
    case VQSEG_MODE_TRAIN_AMP_BF16 | VQSEG_MODE_ROTATE: return launch_gather<VQSEG_MODE_TRAIN_AMP_BF16 | VQSEG_MODE_ROTATE>(xr, E, (int)K, ix, qr, loss_out, partial, cap, st, ticket, cu, usage_out);
  }
  return VQSEG_EINVAL;
}

int vqseg_ste_bwd_f32(const float* g_q, int64_t gB, int64_t gP, int64_t gD,
                      const float* x, int64_t sB, int64_t sP, int64_t sD,
                      const float* q_ste, int64_t qB, int64_t qP, int64_t qD,
                      const float* coef_dev, float coef_scale,
                      float* gx, int64_t oB, int64_t oP, int64_t oD,
                      int64_t B, int64_t P, int64_t D, void* stream) {
  if (!gx || B < 0 || P < 0 || D <= 0) return VQSEG_EINVAL;
  if (coef_dev && (!x || !q_ste)) return VQSEG_EINVAL;
  if (B * P == 0) return 0;
  {
    auto dense = [&](int64_t b, int64_t p, int64_t d) {
      return (p == 1 && d == P && b == D * P) || (d == 1 && p == D && b == P * D);
    };
    auto same = [&](int64_t b, int64_t p, int64_t d) { return b == oB && p == oP && d == oD; };
    auto al = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
    const long long total = B * P * D;
    if (dense(oB, oP, oD) && (!g_q || same(gB, gP, gD)) && (!coef_dev || (same(sB, sP, sD) && same(qB, qP, qD))) &&
        total % 4 == 0 && al(gx) && al(g_q) && al(x) && al(q_ste)) {
      ste_bwd_flat_kernel<<<grid_for(total / 4, 256, 8), 256, 0, (cudaStream_t)stream>>>(
          (const float4*)g_q, (const float4*)x, (const float4*)q_ste, coef_dev, coef_scale, (float4*)gx, total / 4);
      VQSEG_LAUNCH_CHECK();
      return 0;
    }
  }
  View g{g_q, gB, gP, gD}, xv{x, sB, sP, sD}, qv{q_ste, qB, qP, qD};
  RowsOut o{gx, B, P, D, oB, oP, oD};
  bool px_fast = (oP == 1);
  ste_bwd_kernel<<<grid_for(B * P * D, 256, 16), 256, 0, (cudaStream_t)stream>>>(g, xv, qv, coef_dev, coef_scale, o, px_fast);
  VQSEG_LAUNCH_CHECK();
  return 0;
}

int vqseg_rotate_bwd_f32(const float* g_q, int64_t gB, int64_t gP, int64_t gD,
                         const float* x, int64_t sB, int64_t sP, int64_t sD,
                         const float* q, int64_t qB, int64_t qP, int64_t qD,
                         const float* coef_dev, float coef_scale,
                         float* gx, int64_t oB, int64_t oP, int64_t oD,
                         int64_t B, int64_t P, int64_t D, void* stream) {
  if (!gx || !x || !q || B < 0 || P < 0 || D <= 0 || D >= (1ll << 31)) return VQSEG_EINVAL;
  const long long n_rows = B * P;
  if (n_rows == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  View g{g_q, gB, gP, gD}, xv{x, sB, sP, sD}, qv{q, qB, qP, qD};
  RowsOut o{gx, B, P, D, oB, oP, oD};
  // the path follows x's layout (the order of the sums does not depend on it)
  if (sD == 1) {
    rotate_bwd_rows_kernel<<<(unsigned)((n_rows * 8 + 255) / 256), 256, 0, st>>>(g, xv, qv, coef_dev, coef_scale, o);
  } else if (sP == 1) {
    const int ch = (int)(D < kRotChunk ? round_up(D, 8) : kRotChunk);
    const size_t smem = (size_t)3 * ch * 32 * sizeof(float);
    static size_t configured[kMaxDevices] = {0};
    static bool carved[kMaxDevices] = {false};
    if (int rc = ensure_dynamic_smem(rotate_bwd_px_kernel, smem, configured)) return rc;
    if (!carved[current_device()]) {             // 96 KB per block at D >= 256: ask for the large carve-out
      cudaFuncSetAttribute(rotate_bwd_px_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
      carved[current_device()] = true;
    }
    const long long groups = B * ((P + 31) / 32), cap = (long long)num_sms() * 8;
    rotate_bwd_px_kernel<<<(unsigned)(groups < cap ? groups : cap), 256, smem, st>>>(g, xv, qv, coef_dev, coef_scale, o, ch);
  } else {
    rotate_bwd_strided_kernel<<<(unsigned)((n_rows + 255) / 256), 256, 0, st>>>(g, xv, qv, coef_dev, coef_scale, o);
  }
  VQSEG_LAUNCH_CHECK();
  return 0;
}

int vqseg_gather_bwd_codebook_f32(const float* g_q, int64_t B, int64_t P, int64_t D, int64_t gB, int64_t gP, int64_t gD,
                                  const int64_t* idx, float* gE, int64_t K, void* stream) {
  if (!g_q || !idx || !gE || D <= 0 || K <= 0) return VQSEG_EINVAL;
  if (B * P == 0) return 0;
  Rows g{g_q, B, P, D, gB, gP, gD};
  gather_bwd_codebook_kernel<<<grid_for(B * P * 32, 256, 16), 256, 0, (cudaStream_t)stream>>>(g, (const long long*)idx, gE, (int)K);
  VQSEG_LAUNCH_CHECK();
  return 0;
}

// rows per pass of the chunked paths: at most 64 MB of rows (see vqseg_code_stats_f32)
static long long stats_rows_per_chunk(long long D) {
  const long long row_bytes = D * (long long)sizeof(float);
  long long r = (64ll << 20) / row_bytes;
  return r < 4096 ? 4096 : r / 1024 * 1024;
}
static bool stats_sorted_eligible(long long n_rows, long long D, long long K) {
  const long long n_chunks = (n_rows + stats_rows_per_chunk(D) - 1) / stats_rows_per_chunk(D);
  // (K <= 1536: the counting sort costs n_rows / 1024 x K histogram words and needs the table scatter to be cheap)
  return n_rows >= kSortedMinRows && K <= 1536 && n_chunks * K < (1ll << 31);
}
static size_t stats_sort_ws_bytes(long long n_rows, long long D, long long K, int deterministic) {
  if (!deterministic && !stats_sorted_eligible(n_rows, D, K)) return 256;
  long long nblk = (n_rows + kSortBlock - 1) / kSortBlock;
  const long long n_chunks = (n_rows + stats_rows_per_chunk(D) - 1) / stats_rows_per_chunk(D);
  size_t b = 0;
  b += round_up(nblk * K * sizeof(int), 256);                       // hist
  b += round_up(n_chunks * K * sizeof(long long), 256);             // segment sizes per (chunk, code)
  b += round_up((n_chunks * K + 1) * sizeof(long long), 256);       // segment starts
  b += round_up(n_rows * sizeof(int), 256);                         // perm
  if (!deterministic) b += round_up(n_rows * sizeof(int), 256);     // the code of every sorted position (unordered sums)
  return b + 256;
}
size_t vqseg_code_stats_workspace_bytes(int64_t n_rows, int64_t D, int64_t K, int deterministic) {
  // + the packed-row scratch of one chunk (strided inputs are packed chunk by chunk before the row kernels run)
  const long long chunk = n_rows < stats_rows_per_chunk(D) ? n_rows : stats_rows_per_chunk(D);
  return stats_sort_ws_bytes(n_rows, D, K, deterministic) + (size_t)round_up(chunk * D * (long long)sizeof(float), 256);
}

int vqseg_code_stats_f32(const float* x, int64_t B, int64_t P, int64_t D, int64_t sB, int64_t sP, int64_t sD,
                         const int64_t* idx, int64_t K, int64_t* counts, float* sums, int deterministic,
                         void* ws, size_t ws_bytes, void* stream) {
  if (!x || !idx || !counts || !sums || D <= 0 || K <= 0 || B < 0 || P < 0) return VQSEG_EINVAL;
  const long long n_rows = B * P;
  if (n_rows == 0) return 0;
  if (n_rows >= (1ll << 31)) return VQSEG_EUNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  Rows xr{x, B, P, D, sB, sP, sD};
  if (!ws || ws_bytes < vqseg_code_stats_workspace_bytes(n_rows, D, K, deterministic)) return VQSEG_EWORKSPACE;
  const long long rows_per_chunk = stats_rows_per_chunk(D);
  float* scratch = reinterpret_cast<float*>((char*)ws + stats_sort_ws_bytes(n_rows, D, K, deterministic));
  const bool vec_ok = D % 4 == 0 && (reinterpret_cast<uintptr_t>(sums) & 15) == 0;
  const bool flat = sD == 1 && (B == 1 || sB == P * sP);              // one flat range of rows, stride sP
  const bool direct = flat && vec_ok && sP % 4 == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0;
  auto pack = [&](long long r0, long long len) -> int {
    long long blocks = (len + 31) / 32;
    const long long cap = (long long)num_sms() * 8;
    pack_rows_kernel<<<(unsigned)(blocks < cap ? blocks : cap), 256, 0, st>>>(xr, r0, len, scratch);
    VQSEG_LAUNCH_CHECK();
    return 0;
  };
  const bool sorted_fast = !deterministic && direct && stats_sorted_eligible(n_rows, D, K);
  if (!deterministic && !sorted_fast) {
    auto rows_kernel = [&](const float* rows, long long stride, long long len, const int64_t* ix) -> int {
      code_stats_atomic_rows_kernel<<<grid_for(len * 32, 256, 16), 256, 0, st>>>(rows, stride, len, (int)D, (const long long*)ix,
                                                                                 (int)K, (unsigned long long*)counts, sums);
      VQSEG_LAUNCH_CHECK();
      return 0;
    };
    if (direct) return rows_kernel(x, sP, n_rows, idx);
    if (vec_ok) {                                                     // strided (NCHW maps): pack, then vector reductions
      for (long long r0 = 0; r0 < n_rows; r0 += rows_per_chunk) {
        const long long len = n_rows - r0 < rows_per_chunk ? n_rows - r0 : rows_per_chunk;
        if (int rc = pack(r0, len)) return rc;
        if (int rc = rows_kernel(scratch, D, len, idx + r0)) return rc;
      }
      return 0;
    }
    code_stats_atomic_kernel<<<grid_for(n_rows * D, 256, 16), 256, 0, st>>>(xr, (const long long*)idx, (int)K,
                                                                            (unsigned long long*)counts, sums, sP == 1);
    VQSEG_LAUNCH_CHECK();
    return 0;
  }
  if (K * sizeof(int) > 200 * 1024) return VQSEG_EUNSUPPORTED;
  // The ordered sums visit rows grouped by code, i.e. in random order over the whole array: beyond the TLB reach
  // (256 MB of 2 MB pages) every access misses and the chains crawl at ~1.3 us per row.  Row ranges of at most
  // 64 MB are therefore processed one after the other; each (code, d) chain simply continues on top of
  // `sums`, so the summation order -- ascending row id per code -- is unchanged.
  if (direct || vec_ok) {
    // ONE stable counting sort of all row ids by (chunk, code) -- histograms per 1024-row block, a scan per (chunk,
    // code) over the chunk's blocks, a scan over the segments, a stable scatter -- then the ordered sums continue the
    // (code, d) chains range after range on top of `sums`: rows in place (packed rows) in ONE launch whose warps walk
    // the ranges in order (config 4, 10 M rows: 4.1 ms, below the atomic path's 4.6; one launch per range: 6.2 ms;
    // sorting range by range with six small launches each: 22.7 ms); strided maps one pack + one launch per range.
    const long long nblk = (n_rows + kSortBlock - 1) / kSortBlock;
    const int bpc = (int)(rows_per_chunk / kSortBlock);
    const long long n_chunks = (n_rows + rows_per_chunk - 1) / rows_per_chunk;
    char* p = (char*)ws;
    int* hist = (int*)p;                    p += round_up(nblk * K * sizeof(int), 256);
    long long* seg_total = (long long*)p;   p += round_up(n_chunks * K * sizeof(long long), 256);
    long long* seg_start = (long long*)p;   p += round_up((n_chunks * K + 1) * sizeof(long long), 256);
    int* perm = (int*)p;                    p += round_up(n_rows * sizeof(int), 256);
    int* pcode = sorted_fast ? (int*)p : nullptr;
    cudaError_t e = cudaMemsetAsync(hist, 0, nblk * K * sizeof(int), st);
    if (e != cudaSuccess) return (int)e;
    stats_hist_kernel<<<(unsigned)nblk, kSortBlock, 0, st>>>((const long long*)idx, n_rows, (int)K, hist);
    VQSEG_LAUNCH_CHECK();
    stats_scan_chunks_kernel<<<(unsigned)((n_chunks * K + 255) / 256), 256, 0, st>>>(hist, (int)nblk, (int)K, bpc, (int)n_chunks,
                                                                                    (unsigned long long*)counts, seg_total);
    VQSEG_LAUNCH_CHECK();
    if (n_chunks * K >= (1ll << 31)) return VQSEG_EUNSUPPORTED;
    if (int rc = launch_scan_codes(seg_total, n_chunks * K, seg_start, reinterpret_cast<long long*>(perm), st)) return rc;
    if (int rc = launch_scatter((const long long*)idx, n_rows, (int)K, hist, seg_start, perm, bpc, nblk, st, pcode)) return rc;
    if (sorted_fast) {                                                // unordered: windows of sorted positions, one RED per code met
      const long long warps = ((n_rows + kSortedWin - 1) / kSortedWin) * ((D + 127) / 128);
      stats_sorted_sum_kernel<<<(unsigned)((warps * 32 + 255) / 256), 256, 0, st>>>(x, sP, (int)D, perm, pcode,
                                                                                    seg_start + n_chunks * K, sums);
      VQSEG_LAUNCH_CHECK();
      return 0;
    }
    // codes with more than twice the mean share of the rows (and at least 1024: a chain of that length already costs
    // ~40 us through registers) go to the big-cluster kernel; `counts` is final here, so every launch decides alike
    const unsigned long long thr = (unsigned long long)(2 * n_rows / K > 1024 ? 2 * n_rows / K : 1024);
    const bool any_big = (unsigned long long)n_rows > thr;
    const unsigned long long* big_counts = any_big ? (const unsigned long long*)counts : nullptr;
    const size_t bsm = sizeof(BigWarpSmem);
    if (any_big) {
      static size_t bconf[kMaxDevices] = {0};
      if (int rc = ensure_dynamic_smem(stats_ordered_sum_big_kernel, bsm, bconf)) return rc;
    }
    auto sum_launch = [&](const float* base, long long stride, const long long* seg, int nch) -> int {
      const long long warps = K * ((D + 127) / 128);
      stats_ordered_sum_rows_kernel<<<(unsigned)((warps * 32 + 255) / 256), 256, 0, st>>>(base, stride, (int)D, perm, seg, (int)K,
                                                                                          sums, nch, big_counts, thr);
      VQSEG_LAUNCH_CHECK();
      if (any_big) {
        stats_ordered_sum_big_kernel<<<(unsigned)(K * ((D + 31) / 32)), 32, bsm, st>>>(base, stride, (int)D, perm, seg, (int)K,
                                                                                       sums, nch, big_counts, thr);
        VQSEG_LAUNCH_CHECK();
      }
      return 0;
    };
    if (direct) return sum_launch(x, sP, seg_start, (int)n_chunks);   // rows in place: ONE launch walks the ranges in order
    for (long long c = 0; c < n_chunks; ++c) {                        // strided (NCHW maps): pack a range, sum it
      const long long r0 = c * rows_per_chunk;
      const long long len = n_rows - r0 < rows_per_chunk ? n_rows - r0 : rows_per_chunk;
      if (int rc = pack(r0, len)) return rc;
      // perm holds GLOBAL row ids: only rows [r0, r0 + len) are ever addressed through the shifted base
      if (int rc = sum_launch(scratch - r0 * D, D, seg_start + c * K, 1)) return rc;
    }
    return 0;
  }
  // any D, any strides: the generic ordered kernel on the strided view
  if (n_rows <= rows_per_chunk) return stats_det_range(x, B, P, D, sB, sP, sD, idx, K, counts, sums, ws, st);
  if (P <= rows_per_chunk) {                 // whole images per pass
    const long long ipc = rows_per_chunk / P;
    for (long long b0 = 0; b0 < B; b0 += ipc) {
      const long long nb = B - b0 < ipc ? B - b0 : ipc;
      int rc = stats_det_range(x + b0 * sB, nb, P, D, sB, sP, sD, idx + b0 * P, K, counts, sums, ws, st);
      if (rc) return rc;
    }
    return 0;
  }
  for (long long b0 = 0; b0 < B; ++b0)
    for (long long p0 = 0; p0 < P; p0 += rows_per_chunk) {
      const long long len = P - p0 < rows_per_chunk ? P - p0 : rows_per_chunk;
      int rc = stats_det_range(x + b0 * sB + p0 * sP, 1, len, D, sB, sP, sD, idx + b0 * P + p0, K, counts, sums, ws, st);
      if (rc) return rc;
    }
  return 0;
}

int vqseg_kmeans_finalize_f32(const float* sums, const int64_t* counts, float* means_inout, int64_t K, int64_t D,
                              int cosine, void* stream) {
  if (!sums || !counts || !means_inout || K <= 0 || D <= 0) return VQSEG_EINVAL;
  kmeans_finalize_kernel<<<(unsigned)((K * 32 + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      sums, (const long long*)counts, means_inout, (int)K, (int)D, cosine);
  VQSEG_LAUNCH_CHECK();
  return 0;
}

int vqseg_ema_update_f32(const int64_t* counts, const float* sums, float* cluster_size_inout, float* embed_avg_inout,
                         float* weight_out, int64_t K, int64_t D, float decay, float eps, void* ws, void* stream) {
  if (!counts || !sums || !cluster_size_inout || !embed_avg_inout || !weight_out || !ws || K <= 0 || D <= 0) return VQSEG_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  ema_cluster_kernel<false><<<1, 256, 0, st>>>((const long long*)counts, cluster_size_inout, (int)K, decay, (float*)ws,
                                               0.f, nullptr, nullptr);
  VQSEG_LAUNCH_CHECK();
  ema_embed_kernel<false><<<(unsigned)((K * 32 + 255) / 256), 256, 0, st>>>(sums, cluster_size_inout, (const float*)ws,
                                                                           embed_avg_inout, weight_out, (int)K, (int)D,
                                                                           decay, eps, nullptr, nullptr, 0.f);
  VQSEG_LAUNCH_CHECK();
  return 0;
}

// ws: the fp32 n, then one int32 slot per code
static constexpr size_t kExpireSlotOffset = 16;

size_t vqseg_ema_expire_workspace_bytes(int64_t K) {
  return K > 0 ? kExpireSlotOffset + (size_t)K * sizeof(int) : 0;
}

int vqseg_ema_update_expire_f32(const int64_t* counts, const float* sums, float* cluster_size_inout,
                                float* embed_avg_inout, float* weight_out, int64_t K, int64_t D, float decay, float eps,
                                float threshold, float reset, const float* cand_rows, int64_t* expired_out, void* ws,
                                size_t ws_bytes, void* stream) {
  if (!counts || !sums || !cluster_size_inout || !embed_avg_inout || !weight_out || !cand_rows || !ws || K <= 0 ||
      D <= 0 || K > INT_MAX / 32)
    return VQSEG_EINVAL;
  if (ws_bytes < vqseg_ema_expire_workspace_bytes(K)) return VQSEG_EWORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  float* total = (float*)ws;
  int* slot = (int*)((char*)ws + kExpireSlotOffset);
  ema_cluster_kernel<true><<<1, 256, 0, st>>>((const long long*)counts, cluster_size_inout, (int)K, decay, total,
                                              threshold, slot, (long long*)expired_out);
  VQSEG_LAUNCH_CHECK();
  ema_embed_kernel<true><<<(unsigned)((K * 32 + 255) / 256), 256, 0, st>>>(sums, cluster_size_inout, total,
                                                                          embed_avg_inout, weight_out, (int)K, (int)D,
                                                                          decay, eps, slot, cand_rows, reset);
  VQSEG_LAUNCH_CHECK();
  return 0;
}

int vqseg_code_usage(const int64_t* counts, int64_t K, float* usage_out, void* stream) {
  if (!counts || !usage_out || K <= 0) return VQSEG_EINVAL;
  code_usage_kernel<<<1, 256, 0, (cudaStream_t)stream>>>((const long long*)counts, (int)K, usage_out);
  VQSEG_LAUNCH_CHECK();
  return 0;
}

int vqseg_gather_rows_f32(const float* x, int64_t B, int64_t P, int64_t D, int64_t sB, int64_t sP, int64_t sD,
                          const int64_t* row_ids, int64_t n_ids, float* out, void* stream) {
  if (!x || !row_ids || !out || D <= 0) return VQSEG_EINVAL;
  if (n_ids == 0) return 0;
  Rows xr{x, B, P, D, sB, sP, sD};
  gather_rows_kernel<<<grid_for(n_ids * D, 256), 256, 0, (cudaStream_t)stream>>>(xr, (const long long*)row_ids, n_ids, out);
  VQSEG_LAUNCH_CHECK();
  return 0;
}

int vqseg_unpack_keys(const uint64_t* keys, int64_t n, int64_t* idx_out, float* dist_out, int64_t* counts_out,
                      int64_t K, void* stream) {
  if (!keys || n < 0) return VQSEG_EINVAL;
  if (n == 0) return 0;
  unpack_keys_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(
      (const unsigned long long*)keys, n, (long long*)idx_out, dist_out, (unsigned long long*)counts_out, K);
  VQSEG_LAUNCH_CHECK();
  return 0;
}

int vqseg_l2norm_f32(const float* x, int64_t B, int64_t P, int64_t D, int64_t sB, int64_t sP, int64_t sD,
                     float* out, int64_t oB, int64_t oP, int64_t oD, void* stream) {
  if (!x || !out || D <= 0 || B < 0 || P < 0 || D >= (1ll << 31)) return VQSEG_EINVAL;
  if (B * P == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  Rows xr{x, B, P, D, sB, sP, sD};
  RowsOut orow{out, B, P, D, oB, oP, oD};
  if (sD == 1 || D == 1) {
    // the order follows x's reduced dim only (see the kernels above); one term needs no order
    l2norm_lastdim_kernel<<<(unsigned)((B * P * 8 + 255) / 256), 256, 0, st>>>(xr, orow);
  } else {
    if (sP == 1) {
      const long long groups = B * ((P + 31) / 32), cap = (long long)num_sms() * 16;
      static bool carved[kMaxDevices] = {false};        // 32 KB of static shared memory per block: ask for the large carve-out
      if (!carved[current_device()]) {
        cudaFuncSetAttribute(l2norm_px_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        carved[current_device()] = true;
      }
      l2norm_px_kernel<<<(unsigned)(groups < cap ? groups : cap), 256, 0, st>>>(xr, orow);
    } else {
      l2norm_strided_kernel<<<(unsigned)((B * P + 255) / 256), 256, 0, st>>>(xr, orow);
    }
  }
  VQSEG_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"
