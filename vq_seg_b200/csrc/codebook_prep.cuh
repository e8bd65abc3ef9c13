// Building blocks of the prepared-codebook blob, as device functions over an arbitrary set of cooperating threads:
// the multi-block kernels of vqseg_codebook_prepare_f32 call them with grid-wide ids, the codebook guard of the
// forward prologue (api.cu) calls them from ONE block when it finds that the weights changed behind the cache.
#pragma once
#include "common.cuh"

namespace vqseg {

// 64-bit content fingerprint of one code row (order-sensitive multiply-add over the raw fp32 bits).  All 32 lanes of a
// warp must call; returns the hash on every lane.
__device__ __forceinline__ unsigned long long row_hash_warp(const float* __restrict__ row, int D, int lane) {
  unsigned long long h = 0ull;
  for (int d = lane; d < D; d += 32)
    h += ((unsigned long long)__float_as_uint(row[d]) + 0x9E3779B9ull) * (0x9E3779B97F4A7C15ull * (unsigned long long)(2 * d + 1));
#pragma unroll
  for (int o = 16; o; o >>= 1) h += __shfl_xor_sync(0xffffffffu, h, o);
  return h ^ (h >> 29);
}

// phase 1: |e_k|^2 in torch order, max |e|, max |e|^2, row fingerprints.  Warp `warp` of `n_warps`.
__device__ inline void prep_enorm(const float* __restrict__ E, int K, int D, int K_pad, float* __restrict__ enorm,
                                  BlobHeader* hdr, unsigned long long* __restrict__ hash, int warp, int n_warps, int lane) {
  for (int k = warp; k < K_pad; k += n_warps) {
    if (k >= K) { if (lane == 0) { enorm[k] = 3.0e38f; if (hash) hash[k] = 0ull; } continue; }
    const float* row = E + (long long)k * D;
    const float s = torch_order_sumsq_warp([&](long long j) { float v = row[j]; return __fmul_rn(v, v); }, D, lane);
    float amax = 0.f;
    for (int j = lane; j < D; j += 32) amax = fmaxf(amax, fabsf(row[j]));
#pragma unroll
    for (int o = 16; o; o >>= 1) amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, o));
    const unsigned long long h = hash ? row_hash_warp(row, D, lane) : 0ull;
    if (lane == 0) {
      enorm[k] = s;
      if (hash) hash[k] = h;
      if (hdr) {
        atomicMax(&hdr->max_enorm_bits, __float_as_uint(s));
        atomicMax(&hdr->max_abs_bits, __float_as_uint(amax));
      }
    }
  }
}

// phase 2 (after phase 1 is visible): the fp16 operand image, the scaled norms and their fp16 limbs, header scalars.
// image tile (cb, dc): 128 codes x 64 dims of fp16(-2 * s * e), SWIZZLE_128B K-major:
//   byte = row*128 + ((col/8) ^ (row & 7))*16 + (col % 8)*2
__device__ inline void prep_pack(const float* __restrict__ E, int K, int D, unsigned char* __restrict__ blob,
                                 long long tid, long long n_threads) {
  BlobHeader* hdr = reinterpret_cast<BlobHeader*>(blob);
  const int K_pad = hdr->K_pad, D_pad = hdr->D_pad;
  // power-of-two prescale: max |s e| in [8, 16)
  const uint32_t mbits = hdr->max_abs_bits;
  int ex = (int)((mbits >> 23) & 0xff) - 127;
  if (mbits == 0) ex = 3;
  int se = 3 - ex;
  se = se < -100 ? -100 : (se > 100 ? 100 : se);
  const float s = __uint_as_float((uint32_t)(127 + se) << 23);
  float* enorm_s = reinterpret_cast<float*>(blob + hdr->off_enorm) + K_pad;      // scaled copy after the exact one
  const float* enorm = reinterpret_cast<const float*>(blob + hdr->off_enorm);
  __half* img = reinterpret_cast<__half*>(blob + hdr->off_image);
  const int n_dc = D_pad / kDChunk;
  const long long total = (long long)K_pad * (D_pad / 8);
  for (long long i = tid; i < total; i += n_threads) {
    const int k = (int)(i / (D_pad / 8)), d8 = (int)(i % (D_pad / 8)) * 8;
    __align__(16) __half h[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float v = (k < K && d8 + j < D) ? E[(long long)k * D + d8 + j] : 0.f;
      h[j] = __float2half_rn(-2.f * s * v);
    }
    const int cb = k / kCodeBlock, row = k % kCodeBlock, dc = d8 / kDChunk, c8 = (d8 % kDChunk) / 8;
    unsigned char* tile = reinterpret_cast<unsigned char*>(img) + ((long long)cb * n_dc + dc) * kTileBytes;
    *reinterpret_cast<uint4*>(tile + row * 128 + ((c8 ^ (row & 7)) * 16)) = *reinterpret_cast<const uint4*>(h);
  }
  // |e|^2 limbs for the augmented K step: s|e_k|^2 = c * (h1 + h2 + h3), c a power of two putting the
  // largest norm in [2^13, 2^14) so every limb is a normal/subnormal fp16 with residual <= 2^-24 c
  const float men = __uint_as_float(hdr->max_enorm_bits) * s;
  int ce = (int)((__float_as_uint(men) >> 23) & 0xff) - 127 - 13;
  if (men == 0.f) ce = 0;
  ce = ce < -14 ? -14 : (ce > 15 ? 15 : ce);
  const float c = __uint_as_float((uint32_t)(127 + ce) << 23);
  const float cinv = __uint_as_float((uint32_t)(127 - ce) << 23);
  unsigned char* augbase = blob + hdr->off_aug;
  const bool ip = (hdr->flags & kBlobFlagIp) != 0u;       // inner-product blob: the score is -2 s <x, e> alone
  for (long long kk = tid; kk < K_pad; kk += n_threads) {
    const int k = (int)kk;
    enorm_s[k] = k < K ? enorm[k] * s : 3.0e38f;
    float v = k < K ? (ip ? 0.f : enorm[k] * s * cinv) : 60000.f;
    __half h1, h2, h3;
    if (k < K) {
      if (!(v <= 60000.f)) { atomicOr(&hdr->flags, kBlobFlagDeferAll); v = 60000.f; }
      h1 = __float2half_rn(v);
      const float r1 = v - __half2float(h1);
      h2 = __float2half_rn(r1);
      h3 = __float2half_rn(r1 - __half2float(h2));
    } else {
      h1 = h2 = h3 = __float2half_rn(60000.f);          // pad codes can never come near the row minimum
    }
    const int cb = k / kCodeBlock, row = k % kCodeBlock;
    // SWIZZLE_NONE K-major core matrices: 8 rows x 16 B; byte = (row/8)*256 + khalf*128 + (row%8)*16
    unsigned char* t = augbase + (long long)cb * 4096 + (row >> 3) * 256 + (row & 7) * 16;
    __align__(16) __half lo[8] = {h1, h2, h3, __float2half_rn(0.f), __float2half_rn(0.f), __float2half_rn(0.f),
                                  __float2half_rn(0.f), __float2half_rn(0.f)};
    *reinterpret_cast<uint4*>(t) = *reinterpret_cast<const uint4*>(lo);
    *reinterpret_cast<uint4*>(t + 128) = make_uint4(0u, 0u, 0u, 0u);
  }
  if (tid == 0) {
    hdr->scale = s;
    hdr->max_enorm = __uint_as_float(hdr->max_enorm_bits);
    hdr->aug_c = c;
  }
}

// phase 3 (after phase 2's header scalars are visible): rounding error of the fp16 codebook operand, exact, per code
__device__ inline void prep_rounding(const float* __restrict__ E, int K, int D, unsigned char* __restrict__ blob,
                                     int warp, int n_warps, int lane) {
  BlobHeader* hdr = reinterpret_cast<BlobHeader*>(blob);
  const float s = hdr->scale;
  for (int k = warp; k < K; k += n_warps) {
    float acc = 0.f;
    for (int d = lane; d < D; d += 32) {
      const float v = -2.f * s * E[(long long)k * D + d];
      const float df = __half2float(__float2half_rn(v)) - v;
      acc = fmaf(df, df, acc);
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) atomicMax(&hdr->max_de2_bits, __float_as_uint(acc * 1.0001f));
  }
}

}  // namespace vqseg
