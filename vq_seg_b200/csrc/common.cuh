// Shared device/host helpers for libvqseg (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include "../../include/vqseg.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libvqseg is written for sm_100a (B200) only"
#endif

namespace vqseg {

// Logical (B, P, D) view with element strides; row n = b*P + p.
// n = b * P + p with 0 <= p < P.  Row counts stay below 2^31 (checked on entry), so the common case is one 32-bit
// division instead of the 64-bit software routine (fewer instructions; no measurable change in kernel time).
__host__ __device__ inline void split_row(long long n, long long P, long long& b, long long& p) {
  if (((unsigned long long)n | (unsigned long long)P) >> 32) { b = n / P; p = n - b * P; }
  else { const unsigned q = (unsigned)n / (unsigned)P; b = q; p = (unsigned)n - q * (unsigned)P; }
}

struct Rows {
  const float* ptr;
  long long B, P, D, sB, sP, sD;
  __host__ __device__ inline long long n_rows() const { return B * P; }
  __device__ inline const float* row(long long n) const {
    long long b, p;
    split_row(n, P, b, p);
    return ptr + b * sB + p * sP;
  }
};
struct RowsOut {
  float* ptr;
  long long B, P, D, sB, sP, sD;
  __device__ inline float* row(long long n) const {
    long long b, p;
    split_row(n, P, b, p);
    return ptr + b * sB + p * sP;
  }
};

// ---- prepared-codebook blob layout (all offsets 1024-byte aligned) ----------------------------
// [0]    BlobHeader
// [1024] enorm  : K_pad fp32, |e_k|^2 in torch's CPU pow(2).sum(-1) order (pads = +inf marker 3e38)
// [..]   image  : fp16 (-2*s*E) as SWIZZLE_128B K-major tiles of 128 codes x 64 dims (16 KiB each),
//                 ordered [code_block][d_chunk]
// [..]   aug    : per code block a 4 KiB SWIZZLE_NONE tile (128 codes x 16 fp16): cols 0..2 = limbs of s|e|^2/aug_c
// [..]   hash   : K_pad uint64 fingerprints of the fp32 code rows the blob was built from (the codebook guard of the
//                 forward prologue compares them with the live weights, api.cu)
struct BlobHeader {
  uint32_t magic;        // 'VQSB'
  int32_t  K, D, K_pad, D_pad;      // K_pad multiple of 256, D_pad multiple of 64
  float    scale;        // power-of-two prescale s applied to x and E before fp16 rounding
  float    max_enorm;    // max_k |e_k|^2  (fp32, >= true value)
  uint32_t max_enorm_bits;          // written with atomicMax on the float bits
  uint32_t max_abs_bits;            // max |e_kd| bits
  uint64_t off_enorm, off_image, off_aug;
  float    aug_c;        // power of two: s|e_k|^2 = aug_c * (h1 + h2 + h3), three fp16 limbs per code
  uint32_t flags;        // kBlobFlagDeferAll | kBlobFlagIp
  uint32_t max_de2_bits; // max_k |fp16(-2 s e_k) - (-2 s e_k)|^2 : the codebook operand's rounding error, exact
  uint64_t off_hash;
  uint32_t stale;        // guard scratch: set when a row fingerprint differs from the live weights
  uint32_t ticket;       // guard scratch: blocks through the comparison
  uint32_t rebuilds;     // how often the guard had to rebuild the blob (diagnostic)
};
constexpr uint32_t kBlobMagic = 0x42535156u;
constexpr uint32_t kBlobFlagDeferAll = 1u;   // flags bit 0: |e|^2 limbs not representable -> the tensor-core filters defer every row
constexpr uint32_t kBlobFlagIp = 2u;         // flags bit 1: inner-product blob (cosine codebook): no |e|^2 limbs in the score
constexpr int kCodeBlock = 128;     // codes per packed tile
constexpr int kDChunk = 64;         // dims per packed tile (64 fp16 = one 128-byte swizzle row)
constexpr int kTileBytes = kCodeBlock * kDChunk * 2;

__host__ __device__ inline long long round_up(long long a, long long b) { return (a + b - 1) / b * b; }

// ---- torch-CPU-order sum of squares ------------------------------------------------------------
// ATen's CPU sum kernel (aten/src/ATen/native/cpu/SumKernel.cpp, vectorized_inner_sum) reduces a
// contiguous row with 4 ILP accumulators of 8-lane vectors and a 4-level cascade that spills
// every 16 "rows" of 32 elements; element j goes to accumulator t = j % 32.  A warp reproduces it
// with lane t <-> accumulator t.  `sq(j)` must return fl(v_j * v_j).
// All 32 lanes must call this; returns the sum on every lane.
template <typename F>
__device__ inline float torch_order_sumsq_warp(F sq, long long D, int lane) {
  const long long vec_size = D / 8;              // number of 8-wide vectors
  const long long size_ilp = vec_size / 4;       // rows of 4 vectors
  int level_power = 4;
  {
    int cl = 0;
    while ((1ll << cl) < size_ilp) ++cl;         // CeilLog2(size_ilp)
    if (cl / 4 > level_power) level_power = cl / 4;
  }
  const long long level_step = 1ll << level_power, level_mask = level_step - 1;
  float acc0 = 0.f, acc1 = 0.f, acc2 = 0.f, acc3 = 0.f;
  long long i = 0;
  for (; i + level_step <= size_ilp;) {
    for (long long j = 0; j < level_step; ++j, ++i) acc0 = __fadd_rn(acc0, sq(i * 32 + lane));
    // cascade
    acc1 = __fadd_rn(acc1, acc0); acc0 = 0.f;
    if ((i & (level_mask << level_power)) == 0) {
      acc2 = __fadd_rn(acc2, acc1); acc1 = 0.f;
      if ((i & (level_mask << (2 * level_power))) == 0) { acc3 = __fadd_rn(acc3, acc2); acc2 = 0.f; }
    }
  }
  for (; i < size_ilp; ++i) acc0 = __fadd_rn(acc0, sq(i * 32 + lane));
  acc0 = __fadd_rn(acc0, acc1); acc0 = __fadd_rn(acc0, acc2); acc0 = __fadd_rn(acc0, acc3);
  // leftover whole vectors (vec_size % 4) go to partial_sums[0] == lanes 0..7
  for (long long v = size_ilp * 4; v < vec_size; ++v) {
    float s = (lane < 8) ? sq(v * 8 + lane) : 0.f;
    if (lane < 8) acc0 = __fadd_rn(acc0, s);
  }
  // partial_sums[0] += partial_sums[k], k = 1..3   (vector adds, lane l of vector k = lane k*8+l)
  float p = acc0;
  p = __fadd_rn(p, __shfl_sync(0xffffffffu, acc0, (lane & 7) + 8));
  p = __fadd_rn(p, __shfl_sync(0xffffffffu, acc0, (lane & 7) + 16));
  p = __fadd_rn(p, __shfl_sync(0xffffffffu, acc0, (lane & 7) + 24));
  // final_acc = 0 + scalar tail + partials[0..7] sequentially
  float f = 0.f;
  for (long long k = vec_size * 8; k < D; ++k) f = __fadd_rn(f, sq(k));
#pragma unroll
  for (int l = 0; l < 8; ++l) f = __fadd_rn(f, __shfl_sync(0xffffffffu, p, l));
  return f;
}

// ||row|| of a contiguous row in ATen's vectorised last-dim order (see ops.cu, l2norm kernels); 8 lanes cooperate
__device__ __forceinline__ float aten_norm_lastdim8(const float* __restrict__ row, int D, int l8) {
  float a = 0.f;
  const int d8 = D & ~7;
  for (int d = l8; d < d8; d += 8) { const float v = row[d]; a = __fadd_rn(a, __fmul_rn(v, v)); }
  const unsigned gmask = 0xffu << ((threadIdx.x & 31) & ~7);
  float b0 = __shfl_sync(gmask, a, 0, 8);
#pragma unroll
  for (int j = 1; j < 8; ++j) b0 = __fadd_rn(b0, __shfl_sync(gmask, a, j, 8));
  int d = d8;
  if (D - d >= 4) {
#pragma unroll
    for (int j = 0; j < 4; ++j, ++d) { const float v = row[d]; b0 = __fadd_rn(b0, __fmul_rn(v, v)); }
  }
  for (; d < D; ++d) { const float v = row[d]; b0 = __fmaf_rn(v, v, b0); }
  return __fsqrt_rn(b0);
}

__device__ inline float warp_min_f(float v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

inline int check_arch() {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return (int)e;
  int major = 0;
  e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  if (e != cudaSuccess) return (int)e;
  return major == 10 ? 0 : VQSEG_EARCH;
}

// Per-device caches (a process may drive several GPUs: nn.DataParallel, one module per device): the SM count and the
// opt-in dynamic shared-memory limit of a kernel are properties of the CURRENT device.
constexpr int kMaxDevices = 64;
inline int current_device() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) dev = 0;
  return dev;
}
inline int num_sms() {
  static int cached[kMaxDevices] = {0};
  const int dev = current_device();
  if (!cached[dev]) {
    int n = 0;
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    cached[dev] = n > 0 ? n : 148;
  }
  return cached[dev];
}
// cudaFuncAttributeMaxDynamicSharedMemorySize is per device and per function: `state` is the caller's static
// per-device table (one per kernel instantiation) of the size configured so far.
template <typename Kernel>
inline int ensure_dynamic_smem(Kernel kernel, size_t bytes, size_t (&state)[kMaxDevices]) {
  if (bytes <= 48 * 1024) return 0;
  const int dev = current_device();
  if (state[dev] >= bytes) return 0;
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e != cudaSuccess) return (int)e;
  state[dev] = bytes;
  return 0;
}

// ---- programmatic dependent launch (PDL) ------------------------------------------------------------------------------
// A kernel launched with launch_dependent() may become resident while its predecessor in the stream still runs (once
// the predecessor's blocks have executed pdl_trigger() or exited); it must call pdl_wait() before touching anything
// the predecessor writes.  pdl_wait() / pdl_trigger() are no-ops in an ordinary launch.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
template <typename... KArgs, typename... Args>
inline cudaError_t launch_dependent(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl,
                                    Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}
// measured on the config-2 step (A/B, two pairs of runs): 51.9-52.1 us without, 50.5-50.7 us with the rescoring ->
// overflow -> gather chain launched this way (the launch latency of the two small kernels hides behind their
// predecessors); for the big kernels (filter -> rescoring -> gather, round 1) it was slower and is not used
inline bool pdl_enabled() { return true; }

// Slack of the tensor-core filters: how far a code's fp16 score may lie above the row minimum and still be the
// reference's argmin.  |approx - exact| <= |dx| |e^| + |x| |de| (Cauchy-Schwarz on the ACTUAL operand rounding errors,
// both measured: dx by the converters, de by the codebook preparation), two-sided, + the |e|^2 limb residual + the fp32
// accumulation error of the tensor core and of the reference's chain.  The last part in two forms, whichever is
// smaller: (D + 8) 4u (|x| + |e|)^2 (round 1), or -- the reference adds |x|^2 only AFTER the D products
// (_euclidean_dist's term order), so the D-fold error grows with |x||e| and |e|^2 alone --
// (D + 12) 4u |e| (4|x| + |e|) + t2 (|x| + |e|)^2, where t2 = (3 nb + 9) u covers the nb + 1 roundings at the
// magnitude of |x|^2 (two final additions, nb - 1 K-block combines; both sides) and the codes sqrt() merges.  For the
// reference's default codebook init (uniform(-1/K, 1/K), i.e. |e| << |x|) the second form is ~500x tighter: the
// short-lists stay short where the first form sent every row to the overflow kernel (0.8 ms on the config-2 map).
__device__ __forceinline__ float filter_slack(float xn, float dn, float emax, float de_max, float scale, int D, float t2) {
  const float e_s = emax * scale, sum = xn + emax;
  const float chain_a = (float)(D + 8) * 2.4e-7f * sum * sum;
  const float chain_b = (float)(D + 12) * 2.4e-7f * emax * (4.f * xn + emax) + t2 * sum * sum;
  return 2.002f * (dn * 2.002f * e_s + xn * de_max) + scale * fminf(chain_a, chain_b) + 1.0e-6f * e_s * emax;
}

#define VQSEG_LAUNCH_CHECK() do { cudaError_t e__ = cudaGetLastError(); if (e__ != cudaSuccess) return (int)e__; } while (0)

}  // namespace vqseg
