// Fused distance GEMM + argmin on the 5th-gen tensor cores (tcgen05 / TMEM), sm_100a only.
//
// Replaces torch.cdist + torch.argmin (vector_quantizer/vq_img.py:167-168, and :39-41 in kmeans)
// without ever materialising the N x K distance matrix.
//
// The tensor cores evaluate the ranking score  s_k = |e_k|^2 - 2 x.e_k  with fp16 operands and
// fp32 accumulation; that is a FILTER, not the answer.  Every code whose approximate score lies
// within a proven error bound of the row minimum is kept in a per-row short-list, and rows with
// more than one survivor are re-scored by exact.cu with the reference's own fp32 arithmetic.  The
// result therefore equals the exact path bit for bit (DESIGN.md §"why the filter is safe").
//
// Structure (one CTA per SM, persistent over 128-row tiles; unit = 128 rows x 256 codes):
//   warps 0-7   A producers : x (fp32, any strides) -> registers (three chunks of prefetch) -> fp16 ->
//                             SWIZZLE_128B K-major smem tile (128 rows x 64 dims), plus |x|^2 and |fp16(x)-x|^2 per row
//   warps 8-15  epilogue    : one tcgen05.ld pass per accumulator: block min -> running threshold -> bit mask ->
//                             short-list of code indices (two warps per TMEM lane quarter, 128 columns each)
//   warp  16    MMA issuer  : tcgen05.mma.cta_group::1.kind::f16, M=128 N=256 K=16, fp32 accumulators in TMEM;
//                             one extra K=16 step against a constant column adds s |e_k|^2 (three fp16 limbs)
//   warp  17    B loader    : cp.async.bulk (TMA bulk engine) of the pre-packed fp16 (-2 s E) tiles + limb tiles
// Pipelines: smem full/empty mbarriers (3 stages), TMEM full/empty (2 x 256 columns), limb-tile full/empty (2);
// setmaxnreg moves the register budget to the producers (144 / 72 / 40).
#include "tc_common.cuh"
#include "filter_epilogue.cuh"
#include "codebook_prep.cuh"

namespace vqseg {

constexpr int kTileM = 128;           // rows (latent vectors) per tile = UMMA M = TMEM lanes
constexpr int kUnitN = 256;           // codes per unit = UMMA N
constexpr int kStages = 3;
constexpr int kAStageBytes = kTileM * kDChunk * 2;        // 16 KiB
constexpr int kBStageBytes = kUnitN * kDChunk * 2;        // 32 KiB
constexpr int kProducerWarps = 8;
constexpr int kMmaWarp = 16;          // warps 8-15: epilogue, 16: MMA issuer + TMEM alloc, 17: B loader, 18-19: idle
constexpr int kTcThreads = 20 * 32;
constexpr int kXsqBufs = 8;
constexpr int kAugTileBytes = 128 * 16 * 2;               // 4 KiB: 128 codes x 16 fp16, SWIZZLE_NONE core matrices
constexpr uint32_t kIdesc = make_idesc_f16(kTileM, kUnitN);

struct TcSmem {
  // dynamic smem, 1024-aligned base
  static constexpr int off_a = 0;                                             // [kStages] 16 KiB
  static constexpr int off_b = off_a + kStages * kAStageBytes;                // [kStages] 32 KiB
  static constexpr int off_baug = off_b + kStages * kBStageBytes;             // [2] 8 KiB: limb tiles of 256 codes
  static constexpr int off_aaug = off_baug + 2 * 2 * kAugTileBytes;           // 4 KiB
  static constexpr int off_cand = off_aaug + kAugTileBytes;                   // [2 halves][128][cap] code indices
  static constexpr int off_xchg = off_cand + 2 * kTileM * kWorkCandCap * 4;   // [128] {m_run, cnt|overflow} of the upper half
  static constexpr int off_xsq = off_xchg + kTileM * 8;                       // [kXsqBufs][128] float2 {|x|^2, |fp16(x)-x|^2}
  static constexpr int off_bar = off_xsq + kXsqBufs * kTileM * 8;             // mbarriers
  static constexpr int off_tmem = off_bar + 8 * (2 * kStages + 8);
  static constexpr int total = off_tmem + 16 + 1024;   // + slack for the runtime 1024-B alignment
};
static_assert(TcSmem::total <= 232448, "smem budget");


#define VQ_TRACE(role, slot) do { if (a.trace && lane == 0 && (slot) < 256) \
    a.trace[((long long)blockIdx.x * 4 + (role)) * 256 + (slot)] = clock64(); } while (0)

// ---- codebook packing (bodies in codebook_prep.cuh) ------------------------------------------------
__global__ void __launch_bounds__(256) pack_codebook_kernel(const float* __restrict__ E, int K, int D,
                                                            unsigned char* __restrict__ blob) {
  prep_pack(E, K, D, blob, (long long)blockIdx.x * blockDim.x + threadIdx.x, (long long)gridDim.x * blockDim.x);
}
__global__ void __launch_bounds__(256) codebook_rounding_error_kernel(const float* __restrict__ E, int K, int D,
                                                                      unsigned char* __restrict__ blob) {
  prep_rounding(E, K, D, blob, (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5), (int)((gridDim.x * blockDim.x) >> 5),
                (int)(threadIdx.x & 31));
}

// ---- the kernel -----------------------------------------------------------------------------------
// MODE 0: pixel-contiguous float4 loads (NCHW), 1: dim-contiguous float4 (packed rows), 2: scalar, any strides
template <int MODE>
__global__ void __launch_bounds__(kTcThreads, 1) assign_tc_kernel(TcArgs a) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // SWIZZLE_128B needs 1024-B tiles
  const uint32_t sbase = smem_u32(smem);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const BlobHeader* hdr = reinterpret_cast<const BlobHeader*>(a.blob);

  const uint32_t bar_full = sbase + TcSmem::off_bar;                 // [kStages]  8 producer warps + loader (tx)
  const uint32_t bar_empty = bar_full + 8 * kStages;                 // [kStages]  tcgen05.commit
  const uint32_t bar_tfull = bar_empty + 8 * kStages;                // [2]        tcgen05.commit
  const uint32_t bar_tempty = bar_tfull + 16;                        // [2]        8 epilogue warps
  const uint32_t bar_afull = bar_tempty + 16;                        // [2]        |e|^2 limb tile landed (tx)
  const uint32_t bar_aempty = bar_afull + 16;                        // [2]        tcgen05.commit
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + TcSmem::off_tmem);
  float* xsq = reinterpret_cast<float*>(smem + TcSmem::off_xsq);

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) { mbar_init(bar_full + 8 * s, kProducerWarps + 1); mbar_init(bar_empty + 8 * s, 1); }
    for (int b = 0; b < 2; ++b) {
      mbar_init(bar_tfull + 8 * b, 1); mbar_init(bar_tempty + 8 * b, 8);
      mbar_init(bar_afull + 8 * b, 1); mbar_init(bar_aempty + 8 * b, 1);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kMmaWarp) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32((const void*)tmem_slot)), "r"(512u));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int my_tiles = a.n_tiles > (int)blockIdx.x ? (a.n_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
  const int my_units = my_tiles * a.n_cc;

  if (warp < kProducerWarps) {
    // ================= A producers =================
    // lane = quad*8 + g8: dims 8*g8 .. 8*g8+7 of the 64-dim chunk, rows 16*warp + 4*quad + i (i < 4).
    // The 8 lanes of one STS.128 phase share their rows and differ in g8, so the swizzled 16-byte
    // chunks (g8 ^ (row & 7)) land in 8 distinct bank groups: conflict-free with static indexing.
    // Three register buffers rotate over the flat chunk stream: loads run three chunks ahead.
    asm volatile("setmaxnreg.inc.sync.aligned.u32 144;");
    const int g8 = lane & 7, quad = lane >> 3;
    const int r0 = 16 * warp + 4 * quad;
    const int per_tile = a.n_cc * a.n_dc;
    const int total = my_tiles * per_tile;
    const int D = (int)a.x.D;
    const float* rp[4];
    bool rv[4];
    auto decode = [&](int t) {
      const long long n0 = ((long long)blockIdx.x + (long long)t * gridDim.x) * kTileM + r0;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        rv[i] = n0 + i < a.n_rows;
        rp[i] = a.x.row(rv[i] ? n0 + i : 0);
      }
    };
    auto load_chunk = [&](float (&v)[4][8], int dc) {
      const int d0 = dc * kDChunk + 8 * g8;
      if (MODE == 0) {
        const float* p0 = rp[0] + (long long)d0 * a.x.sD;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          float4 f = make_float4(0.f, 0.f, 0.f, 0.f);
          if (rv[0] && d0 + j < D) f = ldg_stream_f4(p0 + (long long)j * a.x.sD);
          v[0][j] = f.x; v[1][j] = f.y; v[2][j] = f.z; v[3][j] = f.w;
        }
      } else if (MODE == 1) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          float4 f0 = make_float4(0.f, 0.f, 0.f, 0.f), f1 = f0;
          if (rv[i] && d0 + 4 <= D) f0 = ldg_stream_f4(rp[i] + d0);
          if (rv[i] && d0 + 8 <= D) f1 = ldg_stream_f4(rp[i] + d0 + 4);
          v[i][0] = f0.x; v[i][1] = f0.y; v[i][2] = f0.z; v[i][3] = f0.w;
          v[i][4] = f1.x; v[i][5] = f1.y; v[i][6] = f1.z; v[i][7] = f1.w;
        }
      } else {
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 8; ++j)
            v[i][j] = (rv[i] && d0 + j < D) ? ldg_stream_f1(rp[i] + (long long)(d0 + j) * a.x.sD) : 0.f;
      }
    };
    int lq = 0, l_dc = 0, l_in = 0, l_t = 0;        // next chunk to load: dim chunk, position in tile, tile
    auto load_next = [&](float (&v)[4][8]) {
      if (lq >= total) return;
      if (l_in == 0) decode(l_t);
      load_chunk(v, l_dc);
      ++lq;
      if (++l_dc == a.n_dc) l_dc = 0;
      if (++l_in == per_tile) { l_in = 0; ++l_t; }
    };
    int sq = 0, s_in = 0, s_t = 0, s_stage = 0;
    uint32_t s_phase = 0;
    float ss[4] = {0.f, 0.f, 0.f, 0.f}, sd[4] = {0.f, 0.f, 0.f, 0.f};
    auto store_next = [&](float (&v)[4][8]) {
      if (sq >= total) return;
      const bool first_pass = s_in < a.n_dc;                 // code chunk 0 of the tile: accumulate the row norms
      if (warp == 0) VQ_TRACE(0, 2 * sq);
      mbar_wait(bar_empty + 8 * s_stage, s_phase ^ 1);
      if (warp == 0) VQ_TRACE(0, 2 * sq + 1);
      unsigned char* at = smem + TcSmem::off_a + s_stage * kAStageBytes;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int r = r0 + i;
        uint32_t pk[4];
#pragma unroll
        for (int j = 0; j < 8; j += 2) {
          __half2 h = __floats2half2_rn(v[i][j], v[i][j + 1]);
          if (first_pass) {
            const float2 hb = __half22float2(h);
            const float e0 = hb.x - v[i][j], e1 = hb.y - v[i][j + 1];
            ss[i] = fmaf(v[i][j], v[i][j], ss[i]); ss[i] = fmaf(v[i][j + 1], v[i][j + 1], ss[i]);
            sd[i] = fmaf(e0, e0, sd[i]); sd[i] = fmaf(e1, e1, sd[i]);
          }
          pk[j >> 1] = *reinterpret_cast<uint32_t*>(&h);
        }
        *reinterpret_cast<uint4*>(at + r * 128 + ((g8 ^ (r & 7)) * 16)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
      }
      if (s_in == a.n_dc - 1) {                              // row norms complete: publish before the arrive
        float2* xs = reinterpret_cast<float2*>(xsq) + (s_t & (kXsqBufs - 1)) * kTileM;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          float v2 = ss[i], e2 = sd[i];
          v2 += __shfl_xor_sync(0xffffffffu, v2, 1); e2 += __shfl_xor_sync(0xffffffffu, e2, 1);
          v2 += __shfl_xor_sync(0xffffffffu, v2, 2); e2 += __shfl_xor_sync(0xffffffffu, e2, 2);
          v2 += __shfl_xor_sync(0xffffffffu, v2, 4); e2 += __shfl_xor_sync(0xffffffffu, e2, 4);
          // |x|^2 and |fp16(x) - x|^2 (inf when an element overflows fp16: the row then goes to the exact pass)
          if (g8 == 0) xs[r0 + i] = make_float2(v2, e2);
          ss[i] = 0.f; sd[i] = 0.f;
        }
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive_relaxed(bar_full + 8 * s_stage);
      ++sq;
      if (++s_stage == kStages) { s_stage = 0; s_phase ^= 1; }
      if (++s_in == per_tile) { s_in = 0; ++s_t; }
    };
    float va[4][8], vb[4][8], vc[4][8];
    load_next(va); load_next(vb); load_next(vc);
    while (sq < total) {
      store_next(va); load_next(va);
      store_next(vb); load_next(vb);
      store_next(vc); load_next(vc);
    }
  } else if (warp < kMmaWarp) {
    // ================= epilogue (8 warps: two per TMEM lane quarter, 128 columns each) =================
    asm volatile("setmaxnreg.dec.sync.aligned.u32 72;");
    const int quarter = warp & 3;
    const int half = (warp - kProducerWarps) >> 2;
    const int r = quarter * 32 + lane;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(quarter * 32) << 16) + half * 128;
    const ShortList<int>::Slots lists(reinterpret_cast<int*>(smem + TcSmem::off_cand), kTileM, half, r);
    float2* xchg = reinterpret_cast<float2*>(smem + TcSmem::off_xchg) + r;
    const FilterBound bound(hdr);
    int u = 0;
    for (int t = 0; t < my_tiles; ++t) {
      const long long n = ((long long)blockIdx.x + (long long)t * gridDim.x) * kTileM + r;
      ShortList<int> sl(lists);
      for (int cc = 0; cc < a.n_cc; ++cc, ++u) {
        const int buf = u & 1;
        if (warp == kProducerWarps) VQ_TRACE(2, 4 * u);
        mbar_wait(bar_tfull + 8 * buf, (uint32_t)(u >> 1) & 1);
        tc_fence_after();
        if (warp == kProducerWarps) VQ_TRACE(2, 4 * u + 1);
        if (cc == 0) {
          // all A chunks of this tile's first unit are in: the row's |x|^2 and |fp16(x)-x|^2 have been published
          const float2 nr = reinterpret_cast<const float2*>(xsq)[(t & (kXsqBufs - 1)) * kTileM + r];
          sl.start(bound, nr.x, nr.y, (int)a.x.D, a.out.slack_t2);
        }
        const uint32_t tb = lane_addr + buf * kUnitN;
#pragma unroll 1
        for (int c = 0; c < 128; c += 32) {
          uint32_t v[32];
          tmem_ld32(tb + c, v);
          sl.scan32(v, cc * kUnitN + half * 128 + c);
        }
        if (warp == kProducerWarps) VQ_TRACE(2, 4 * u + 2);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_tempty + 8 * buf);              // this warp's columns are drained
      }
      sl.finish(half, 1 + quarter, xchg, n < a.n_rows, n, a.out);
    }
  } else {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
    if (warp == kMmaWarp + 1) {
      // ================= B loader (bulk async copies of the pre-packed fp16 tiles) =================
      {   // A-side augmentation tile: columns 0..2 = c (power of two), rest 0; SWIZZLE_NONE core matrices
        const __half cval = __float2half_rn(hdr->aug_c);
        const uint32_t c2 = (uint32_t)__half_as_ushort(cval);
        uint4* aa = reinterpret_cast<uint4*>(smem + TcSmem::off_aaug);
        for (int i = lane; i < kAugTileBytes / 16; i += 32)
          aa[i] = (((i >> 3) & 1) == 0) ? make_uint4(c2 | (c2 << 16), c2, 0u, 0u) : make_uint4(0u, 0u, 0u, 0u);
        fence_proxy_async();
        __syncwarp();
      }
      if (lane == 0) {
        const unsigned char* img = a.blob + hdr->off_image;
        const unsigned char* aug = a.blob + hdr->off_aug;
        int s = 0; uint32_t ph = 0;
        int u = 0;
        for (int t = 0; t < my_tiles; ++t)
          for (int cc = 0; cc < a.n_cc; ++cc, ++u) {
            {   // |e|^2 limb tiles of this unit's 256 codes (2 x 4 KiB), double-buffered by unit parity
              const int b = u & 1;
              mbar_wait(bar_aempty + 8 * b, (((uint32_t)u >> 1) & 1) ^ 1);
              mbar_arrive_expect_tx(bar_afull + 8 * b, 2 * kAugTileBytes);
              bulk_g2s(sbase + TcSmem::off_baug + b * 2 * kAugTileBytes, aug + (long long)(2 * cc) * kAugTileBytes,
                       2 * kAugTileBytes, bar_afull + 8 * b);
            }
            for (int dc = 0; dc < a.n_dc; ++dc) {
              VQ_TRACE(3, 2 * (u * a.n_dc + dc));
              mbar_wait(bar_empty + 8 * s, ph ^ 1);
              VQ_TRACE(3, 2 * (u * a.n_dc + dc) + 1);
              const uint32_t dst = sbase + TcSmem::off_b + s * kBStageBytes;
              mbar_arrive_expect_tx(bar_full + 8 * s, kBStageBytes);
              bulk_g2s(dst, img + ((long long)(2 * cc) * a.n_dc + dc) * kTileBytes, kTileBytes, bar_full + 8 * s);
              bulk_g2s(dst + kTileBytes, img + ((long long)(2 * cc + 1) * a.n_dc + dc) * kTileBytes, kTileBytes, bar_full + 8 * s);
              if (++s == kStages) { s = 0; ph ^= 1; }
            }
          }
      }
    } else if (warp == kMmaWarp) {
      // ================= MMA issuer =================
      const uint64_t aaug = make_desc_noswz(sbase + TcSmem::off_aaug, 128, 256);
      int s = 0; uint32_t ph = 0;
      int it = 0;
      for (int u = 0; u < my_units; ++u) {
        const int buf = u & 1;
        const uint32_t use = (uint32_t)(u >> 1);
        VQ_TRACE(1, 128 + 2 * u);
        mbar_wait(bar_tempty + 8 * buf, (use & 1) ^ 1);     // the epilogue drained this accumulator
        VQ_TRACE(1, 128 + 2 * u + 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + buf * kUnitN;
        for (int dc = 0; dc < a.n_dc; ++dc, ++it) {
          VQ_TRACE(1, 2 * it);
          mbar_wait(bar_full + 8 * s, ph);
          VQ_TRACE(1, 2 * it + 1);
          tc_fence_after();
          if (lane == 0) {
            const uint64_t ad = make_desc(sbase + TcSmem::off_a + s * kAStageBytes);
            const uint64_t bd = make_desc(sbase + TcSmem::off_b + s * kBStageBytes);
#pragma unroll
            for (int k = 0; k < kDChunk / 16; ++k)          // +32 B per K=16 step inside the 128-B swizzle row
              tc_mma_f16(d_tmem, ad + (uint64_t)(2 * k), bd + (uint64_t)(2 * k), kIdesc, (dc | k) ? 1u : 0u);
            tc_commit(bar_empty + 8 * s);                   // smem stage free when these MMAs retire
          }
          __syncwarp();
          if (++s == kStages) { s = 0; ph ^= 1; }
        }
        mbar_wait(bar_afull + 8 * buf, use & 1);            // |e|^2 limbs of this unit's codes
        tc_fence_after();
        if (lane == 0) {
          const uint64_t baug = make_desc_noswz(sbase + TcSmem::off_baug + buf * 2 * kAugTileBytes, 128, 256);
          tc_mma_f16(d_tmem, aaug, baug, kIdesc, 1u);       // + s |e_k|^2 : the accumulator is now the score
          tc_commit(bar_aempty + 8 * buf);
          tc_commit(bar_tfull + 8 * buf);
        }
        __syncwarp();
      }
    }
  }

  // ---- teardown ----
  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u));
  }
}

int launch_pack(const float* E, int K, int D, unsigned char* blob, cudaStream_t st) {
  int blocks = num_sms() * 2;
  pack_codebook_kernel<<<blocks, 256, 0, st>>>(E, K, D, blob);
  VQSEG_LAUNCH_CHECK();
  int rblocks = (K * 32 + 255) / 256;
  if (rblocks > num_sms() * 8) rblocks = num_sms() * 8;
  codebook_rounding_error_kernel<<<rblocks, 256, 0, st>>>(E, K, D, blob);
  VQSEG_LAUNCH_CHECK();
  return 0;
}

template <int MODE>
static int launch_mode(const TcArgs& a, int grid, cudaStream_t st) {
  static size_t configured[kMaxDevices] = {0};
  if (int rc = ensure_dynamic_smem(assign_tc_kernel<MODE>, TcSmem::total, configured)) return rc;
  assign_tc_kernel<MODE><<<grid, kTcThreads, TcSmem::total, st>>>(a);
  VQSEG_LAUNCH_CHECK();
  return 0;
}

int launch_assign_tc(const TcArgs& a, cudaStream_t st) {
  int grid = a.n_tiles < num_sms() ? a.n_tiles : num_sms();
  if (grid <= 0) return 0;
  const bool al16 = (reinterpret_cast<uintptr_t>(a.x.ptr) & 15) == 0 && (a.x.sB & 3) == 0;
  if (al16 && a.x.sP == 1 && (a.x.P & 3) == 0 && (a.x.sD & 3) == 0) return launch_mode<0>(a, grid, st);
  if (al16 && a.x.sD == 1 && (a.x.D & 3) == 0 && (a.x.sP & 3) == 0) return launch_mode<1>(a, grid, st);
  return launch_mode<2>(a, grid, st);
}

}  // namespace vqseg
