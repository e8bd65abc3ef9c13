// Codebook-resident, CTA-pair variant of the fused distance + argmin kernel (tcgen05.cta_group::2).
//
// Same contract as assign_tc.cu (it replaces torch.cdist + torch.argmin, vq_img.py:167-168) for
// codebooks whose fp16 operand image fits the shared memory of TWO SMs:  (K_pad/256) * (D_pad/64) <= 8,
// D_pad <= 256  -- e.g. the headline K=512, D=256.
//
//   * a cluster of 2 CTAs (one TPC) owns 256 rows per tile: each CTA converts and holds its own 128 rows
//     (UMMA M = 256 = 2 x 128 TMEM lanes) and HALF of every 256-code chunk (UMMA N = 256 = 2 x 128 codes),
//     so the whole codebook stays resident (128 KiB per CTA) and every x element is read from HBM once,
//     converted once;
//   * |e_k|^2 enters through one extra K=16 MMA step against a constant column (three fp16 limbs), so the
//     accumulator IS the score and TMEM is never written by the SM;
//   * the next three 64-dim chunks of fp32 rows wait in REGISTERS (3 x 32 regs per producer thread, register
//     budget moved to the producers with setmaxnreg) while the current tile's fp16 operand sits in smem;
//   * the epilogue reads each accumulator exactly once: per 32 columns block-min -> running threshold ->
//     sign-bit mask (one FADD + one funnel shift per score) -> short-list of code indices.
// Roles per CTA (20 warps): 0-7 producers, 8-15 epilogue (two warps per TMEM lane quarter, 128 columns
// each), 16 MMA issuer (leader CTA) + TMEM alloc, 17 codebook loader (cp.async.bulk), 18-19 idle (they
// only donate registers).
#include "tc_common.cuh"
#include "filter_epilogue.cuh"

namespace vqseg {

constexpr int k2Threads = 640;                // 20 warps: 8 producers, 8 epilogue, MMA, loader, 2 idle
constexpr int k2Rows = 128;                 // rows per CTA per tile (pair tile = 256)
constexpr int k2ASlots = 4;                 // A ring = one tile (D_pad <= 256)
constexpr int k2MaxBTiles = 8;              // resident 16 KiB codebook tiles per CTA
constexpr int k2MaxCC = 4;
constexpr int k2XsqBufs = 4;
constexpr int k2AugBytes = 128 * 16 * 2;    // 4 KiB: 128 rows x 16 fp16, SWIZZLE_NONE core matrices
constexpr uint32_t k2Idesc = make_idesc_f16(256, 256);

struct Tc2Smem {
  static constexpr int off_b = 0;                                         // [k2MaxBTiles] 16 KiB
  static constexpr int off_a = off_b + k2MaxBTiles * kTileBytes;           // [k2ASlots] 16 KiB
  static constexpr int off_baug = off_a + k2ASlots * kTileBytes;           // [k2MaxCC] 4 KiB
  static constexpr int off_aaug = off_baug + k2MaxCC * k2AugBytes;         // 4 KiB
  static constexpr int off_cand = off_aaug + k2AugBytes;                   // [2 halves][128][cap] int
  static constexpr int off_xchg = off_cand + 2 * k2Rows * kWorkCandCap * 4; // [128] {m_run, cnt|overflow} of the upper-half warp
  static constexpr int off_xsq = off_xchg + k2Rows * 8;                     // [bufs][128] float2 {|x|^2, |fp16(x)-x|^2}
  static constexpr int off_bar = off_xsq + k2XsqBufs * k2Rows * 8;
  static constexpr int n_bars = 2 * k2ASlots + 4 + 2 * k2MaxCC;
  static constexpr int off_tmem = off_bar + 8 * n_bars;
  static constexpr int total = off_tmem + 16 + 1024;
};
static_assert(Tc2Smem::total <= 232448, "smem budget");


#define VQ2_TRACE(role, slot) do { if (a.trace && lane == 0 && (slot) < 256) \
    a.trace[((long long)blockIdx.x * 4 + (role)) * 256 + (slot)] = clock64(); } while (0)

template <int MODE>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(k2Threads, 1) assign_tc2_kernel(Tc2Args a) {
  extern __shared__ __align__(1024) unsigned char smem_raw2[];
  unsigned char* smem = smem_raw2 + ((1024u - (smem_u32(smem_raw2) & 1023u)) & 1023u);
  const uint32_t sbase = smem_u32(smem);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const BlobHeader* hdr = reinterpret_cast<const BlobHeader*>(a.blob);
  auto gtime = [] { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return (long long)t; };
  if (a.trace && threadIdx.x == 0) { a.trace[((long long)blockIdx.x * 4 + 3) * 256 + 0] = gtime(); a.trace[((long long)blockIdx.x * 4 + 3) * 256 + 4] = clock64(); }

  const uint32_t bar_full = sbase + Tc2Smem::off_bar;                  // [slots]  leader: 16 producer-warp arrivals
  const uint32_t bar_empty = bar_full + 8 * k2ASlots;                  // [slots]  each CTA: 1 (multicast commit)
  const uint32_t bar_tfull = bar_empty + 8 * k2ASlots;                 // [2]      each CTA: 1 (multicast commit)
  const uint32_t bar_tempty = bar_tfull + 16;                          // [2]      leader: 8 epilogue-warp arrivals
  const uint32_t bar_bload = bar_tempty + 16;                          // [k2MaxCC] local bulk-copy completion per code chunk
  const uint32_t bar_bready = bar_bload + 8 * k2MaxCC;                 // [k2MaxCC] leader: 2 (chunk resident in both CTAs)
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + Tc2Smem::off_tmem);
  float* xsq = reinterpret_cast<float*>(smem + Tc2Smem::off_xsq);

  if (threadIdx.x == 0) {
    for (int s = 0; s < k2ASlots; ++s) { mbar_init(bar_full + 8 * s, 16); mbar_init(bar_empty + 8 * s, 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(bar_tfull + 8 * b, 1); mbar_init(bar_tempty + 8 * b, 16); }
    for (int c = 0; c < k2MaxCC; ++c) { mbar_init(bar_bload + 8 * c, 1); mbar_init(bar_bready + 8 * c, 2); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 16) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32((const void*)tmem_slot)), "r"(512u));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (a.trace && threadIdx.x == 0) { a.trace[((long long)blockIdx.x * 4 + 3) * 256 + 1] = gtime(); a.trace[((long long)blockIdx.x * 4 + 3) * 256 + 5] = clock64(); }

  const int n_pairs = (int)gridDim.x >> 1;
  const int pair = (int)blockIdx.x >> 1;
  const int my_tiles = a.n_ptiles > pair ? (a.n_ptiles - 1 - pair) / n_pairs + 1 : 0;
  const uint32_t lead_full = mapa_u32(bar_full, 0);
  const uint32_t lead_tempty = mapa_u32(bar_tempty, 0);

  if (warp < 8) {
    // ================= A producers =================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 144;");
    const int g8 = lane & 7, quad = lane >> 3;
    const int r0 = 16 * warp + 4 * quad;
    const int D = (int)a.x.D;
    const float* rp[4];
    bool rv[4];
    auto decode = [&](int tt) {
      const long long n0 = ((long long)pair + (long long)tt * n_pairs) * 256 + rank * 128 + r0;
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
    float ss[4] = {0.f, 0.f, 0.f, 0.f}, sd[4] = {0.f, 0.f, 0.f, 0.f};
    auto store_chunk = [&](float (&v)[4][8], int dc, int tt) {
      if (warp == 0) VQ2_TRACE(0, 2 * (tt * a.n_dc + dc));
      mbar_wait(bar_empty + 8 * dc, ((uint32_t)tt & 1) ^ 1);        // last tile's MMAs on this slot retired
      if (warp == 0) VQ2_TRACE(0, 2 * (tt * a.n_dc + dc) + 1);
      unsigned char* at = smem + Tc2Smem::off_a + dc * kTileBytes;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int r = r0 + i;
        uint32_t pk[4];
#pragma unroll
        for (int j = 0; j < 8; j += 2) {
          __half2 h = __floats2half2_rn(v[i][j], v[i][j + 1]);
          const float2 hb = __half22float2(h);
          const float e0 = hb.x - v[i][j], e1 = hb.y - v[i][j + 1];
          ss[i] = fmaf(v[i][j], v[i][j], ss[i]); ss[i] = fmaf(v[i][j + 1], v[i][j + 1], ss[i]);
          sd[i] = fmaf(e0, e0, sd[i]); sd[i] = fmaf(e1, e1, sd[i]);
          pk[j >> 1] = *reinterpret_cast<uint32_t*>(&h);
        }
        *reinterpret_cast<uint4*>(at + r * 128 + ((g8 ^ (r & 7)) * 16)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
      }
      if (dc == a.n_dc - 1) {                                        // row norms complete: publish before the arrive
        float2* xs = reinterpret_cast<float2*>(xsq) + (tt & (k2XsqBufs - 1)) * k2Rows;
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
      if (lane == 0) mbar_arrive_cluster_relaxed(lead_full + 8 * dc);        // leader's barrier (remote for rank 1)
    };

    // flat chunk stream q = tt * n_dc + dc; three register buffers rotate, loads run 3 chunks ahead
    const int total = my_tiles * a.n_dc;
    int lq = 0, l_dc = 0, l_tt = 0;               // next chunk to load
    auto load_next = [&](float (&v)[4][8]) {
      if (lq >= total) return;
      if (l_dc == 0) decode(l_tt);
      load_chunk(v, l_dc);
      ++lq;
      if (++l_dc == a.n_dc) { l_dc = 0; ++l_tt; }
    };
    int sq = 0, s_dc = 0, s_tt = 0;               // next chunk to convert + store
    auto store_next = [&](float (&v)[4][8]) {
      if (sq >= total) return;
      store_chunk(v, s_dc, s_tt);
      ++sq;
      if (++s_dc == a.n_dc) { s_dc = 0; ++s_tt; }
    };
    float va[4][8], vb[4][8], vc[4][8];
    load_next(va); load_next(vb); load_next(vc);
    while (sq < total) {
      store_next(va); load_next(va);
      store_next(vb); load_next(vb);
      store_next(vc); load_next(vc);
    }
  } else if (warp < 16) {
    // ================= epilogue =================
    asm volatile("setmaxnreg.dec.sync.aligned.u32 72;");
    const int quarter = warp & 3;                         // TMEM lane quarter this warp may access
    const int half = (warp - 8) >> 2;                     // which 128 of the unit's 256 columns
    const int r = quarter * 32 + lane;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(quarter * 32) << 16) + half * 128;
    const ShortList<int>::Slots lists(reinterpret_cast<int*>(smem + Tc2Smem::off_cand), k2Rows, half, r);
    float2* xchg = reinterpret_cast<float2*>(smem + Tc2Smem::off_xchg) + r;
    const FilterBound bound(hdr);
    int u = 0;
    for (int tt = 0; tt < my_tiles; ++tt) {
      const long long n = ((long long)pair + (long long)tt * n_pairs) * 256 + rank * 128 + r;
      ShortList<int> sl(lists);
      for (int cc = 0; cc < a.n_cc; ++cc, ++u) {
        const int buf = a.n_cc == 1 ? (tt & 1) : cc;
        const uint32_t use = a.n_cc == 1 ? (uint32_t)(tt >> 1) : (uint32_t)tt;
        if (warp == 8) VQ2_TRACE(2, 4 * u);
        mbar_wait(bar_tfull + 8 * buf, use & 1);
        tc_fence_after();
        if (warp == 8) VQ2_TRACE(2, 4 * u + 1);
        if (cc == 0) {
          const float2 nr = reinterpret_cast<const float2*>(xsq)[(tt & (k2XsqBufs - 1)) * k2Rows + r];
          sl.start(bound, nr.x, nr.y, (int)a.x.D, a.out.slack_t2);
        }
        const uint32_t tb = lane_addr + buf * 256;
#pragma unroll 1
        for (int c = 0; c < 128; c += 32) {
          uint32_t v[32];
          tmem_ld32(tb + c, v);
          sl.scan32(v, cc * 256 + half * 128 + c);
        }
        if (warp == 8) VQ2_TRACE(2, 4 * u + 2);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(lead_tempty + 8 * buf);     // this warp's columns are drained
      }
      sl.finish(half, 1 + quarter, xchg, n < a.n_rows, n, a.out);
    }
  } else {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
    if (warp == 17) {
      // ================= codebook loader: this CTA's half of every 256-code chunk stays resident =================
      {   // A-side augmentation tile: column 0..2 = c (power of two), rest 0; SWIZZLE_NONE core matrices
        const __half cval = __float2half_rn(hdr->aug_c);
        const uint32_t c2 = (uint32_t)__half_as_ushort(cval);
        uint4* aa = reinterpret_cast<uint4*>(smem + Tc2Smem::off_aaug);
        for (int i = lane; i < k2AugBytes / 16; i += 32) {
          // 16-byte unit i: group g = i / 16, k-half h = (i / 8) & 1, row-in-group = i & 7
          const bool first_half = ((i >> 3) & 1) == 0;
          aa[i] = first_half ? make_uint4(c2 | (c2 << 16), c2, 0u, 0u) : make_uint4(0u, 0u, 0u, 0u);
        }
        fence_proxy_async();
        __syncwarp();
      }
      if (lane == 0) {
        const unsigned char* img = a.blob + a.off_image;
        const unsigned char* aug = a.blob + a.off_aug;
        const uint32_t bytes = (uint32_t)a.n_dc * kTileBytes + k2AugBytes;
        // code chunk by code chunk: chunk 0 is needed at once, the others only after the first unit, and at
        // kernel start every CTA's codebook load competes with the first x tile for L2 bandwidth
        for (int cc = 0; cc < a.n_cc; ++cc) {
          const int cb = 2 * cc + (int)rank;                       // this CTA's 128 codes of chunk cc
          mbar_arrive_expect_tx(bar_bload + 8 * cc, bytes);
          for (int dc = 0; dc < a.n_dc; ++dc)
            bulk_g2s(sbase + Tc2Smem::off_b + (cc * a.n_dc + dc) * kTileBytes,
                     img + ((long long)cb * a.n_dc + dc) * kTileBytes, kTileBytes, bar_bload + 8 * cc);
          bulk_g2s(sbase + Tc2Smem::off_baug + cc * k2AugBytes, aug + (long long)cb * k2AugBytes, k2AugBytes,
                   bar_bload + 8 * cc);
          mbar_wait(bar_bload + 8 * cc, 0);
          mbar_arrive_cluster(mapa_u32(bar_bready + 8 * cc, 0));
        }
      }
    } else if (warp == 16 && rank == 0) {
      // ================= MMA issuer (leader CTA) =================
      const uint64_t aaug = make_desc_noswz(sbase + Tc2Smem::off_aaug, 128, 256);
      // Dims-outer order: every 64-dim A chunk is multiplied against BOTH 256-code chunks as soon as it lands
      // (the kernel is bound by how fast x arrives, so the MMAs hide under the loads), its smem slot is released
      // at once, and the tile's two accumulators (TMEM columns 0-255 / 256-511) complete together.
      // n_cc == 1: the two TMEM halves alternate between tiles instead.
      for (int tt = 0; tt < my_tiles; ++tt) {
        if (a.n_cc == 2 && tt == my_tiles - 1) {
          // LAST tile, codes-outer: nothing waits for its A slots any more, so code chunk 0 is multiplied against
          // all dim chunks first and its accumulator is handed to the epilogue while chunk 1's MMAs still run
          // (dims-outer would deliver both accumulators together and leave the tensor pipe idle during the drain).
          for (int cc = 0; cc < 2; ++cc) {
            VQ2_TRACE(1, 128 + 2 * (tt * a.n_cc + cc));
            mbar_wait(bar_tempty + 8 * cc, ((uint32_t)tt & 1) ^ 1);
            VQ2_TRACE(1, 128 + 2 * (tt * a.n_cc + cc) + 1);
            if (tt == 0) mbar_wait(bar_bready + 8 * cc, 0);
            tc_fence_after();
            for (int dc = 0; dc < a.n_dc; ++dc) {
              if (cc == 0) {
                VQ2_TRACE(1, 2 * (tt * a.n_dc + dc));
                mbar_wait(bar_full + 8 * dc, (uint32_t)tt & 1);
                VQ2_TRACE(1, 2 * (tt * a.n_dc + dc) + 1);
                tc_fence_after();
              }
              if (lane == 0) {
                const uint64_t ad = make_desc(sbase + Tc2Smem::off_a + dc * kTileBytes);
                const uint64_t bd = make_desc(sbase + Tc2Smem::off_b + (cc * a.n_dc + dc) * kTileBytes);
#pragma unroll
                for (int k = 0; k < kDChunk / 16; ++k)
                  tc_mma_f16_2cta(tmem_base + cc * 256, ad + (uint64_t)(2 * k), bd + (uint64_t)(2 * k), k2Idesc,
                                  (dc | k) ? 1u : 0u);
                if (cc == 1) tc_commit_2cta(bar_empty + 8 * dc);
              }
              __syncwarp();
            }
            if (lane == 0) {
              const uint64_t baug = make_desc_noswz(sbase + Tc2Smem::off_baug + cc * k2AugBytes, 128, 256);
              tc_mma_f16_2cta(tmem_base + cc * 256, aaug, baug, k2Idesc, 1u);   // + s |e_k|^2
              tc_commit_2cta(bar_tfull + 8 * cc);
            }
            __syncwarp();
          }
          continue;
        }
        for (int cc = 0; cc < a.n_cc; ++cc) {
          const int buf = a.n_cc == 1 ? (tt & 1) : cc;
          const uint32_t use = a.n_cc == 1 ? (uint32_t)(tt >> 1) : (uint32_t)tt;
          VQ2_TRACE(1, 128 + 2 * (tt * a.n_cc + cc));
          mbar_wait(bar_tempty + 8 * buf, (use & 1) ^ 1);               // both CTAs' epilogues drained it
          VQ2_TRACE(1, 128 + 2 * (tt * a.n_cc + cc) + 1);
          if (tt == 0) mbar_wait(bar_bready + 8 * cc, 0);                // this code chunk is resident in both CTAs
        }
        tc_fence_after();
        for (int dc = 0; dc < a.n_dc; ++dc) {
          VQ2_TRACE(1, 2 * (tt * a.n_dc + dc));
          mbar_wait(bar_full + 8 * dc, (uint32_t)tt & 1);                // both CTAs' halves of the A chunk landed
          VQ2_TRACE(1, 2 * (tt * a.n_dc + dc) + 1);
          tc_fence_after();
          if (lane == 0) {
            const uint64_t ad = make_desc(sbase + Tc2Smem::off_a + dc * kTileBytes);
            for (int cc = 0; cc < a.n_cc; ++cc) {
              const int buf = a.n_cc == 1 ? (tt & 1) : cc;
              const uint64_t bd = make_desc(sbase + Tc2Smem::off_b + (cc * a.n_dc + dc) * kTileBytes);
#pragma unroll
              for (int k = 0; k < kDChunk / 16; ++k)
                tc_mma_f16_2cta(tmem_base + buf * 256, ad + (uint64_t)(2 * k), bd + (uint64_t)(2 * k), k2Idesc,
                                (dc | k) ? 1u : 0u);
            }
            tc_commit_2cta(bar_empty + 8 * dc);                          // A slot free in both CTAs
          }
          __syncwarp();
        }
        if (lane == 0) {
          for (int cc = 0; cc < a.n_cc; ++cc) {
            const int buf = a.n_cc == 1 ? (tt & 1) : cc;
            const uint64_t baug = make_desc_noswz(sbase + Tc2Smem::off_baug + cc * k2AugBytes, 128, 256);
            tc_mma_f16_2cta(tmem_base + buf * 256, aaug, baug, k2Idesc, 1u);   // + s |e_k|^2
            tc_commit_2cta(bar_tfull + 8 * buf);
          }
        }
        __syncwarp();
      }
    }
  }

  // ---- teardown ----
  if (a.trace && threadIdx.x == 0) { a.trace[((long long)blockIdx.x * 4 + 3) * 256 + 2] = gtime(); a.trace[((long long)blockIdx.x * 4 + 3) * 256 + 6] = clock64(); }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (a.trace && threadIdx.x == 0) { a.trace[((long long)blockIdx.x * 4 + 3) * 256 + 3] = gtime(); a.trace[((long long)blockIdx.x * 4 + 3) * 256 + 7] = clock64(); }
  if (warp == 16) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u));
  }
}

template <int MODE>
static int launch_mode2(const Tc2Args& a, int grid, cudaStream_t st) {
  static size_t configured[kMaxDevices] = {0};
  if (int rc = ensure_dynamic_smem(assign_tc2_kernel<MODE>, Tc2Smem::total, configured)) return rc;
  assign_tc2_kernel<MODE><<<grid, k2Threads, Tc2Smem::total, st>>>(a);
  VQSEG_LAUNCH_CHECK();
  return 0;
}

bool tc2_supported(int n_cc, int n_dc) { return n_dc <= k2ASlots && n_cc <= 2 && n_cc * n_dc <= k2MaxBTiles; }

int launch_assign_tc2(const Tc2Args& a, cudaStream_t st) {
  int pairs = num_sms() / 2;
  if (a.n_ptiles < pairs) pairs = a.n_ptiles;
  if (pairs <= 0) return 0;
  const int grid = 2 * pairs;
  const bool al16 = (reinterpret_cast<uintptr_t>(a.x.ptr) & 15) == 0 && (a.x.sB & 3) == 0;
  if (al16 && a.x.sP == 1 && (a.x.P & 3) == 0 && (a.x.sD & 3) == 0) return launch_mode2<0>(a, grid, st);
  if (al16 && a.x.sD == 1 && (a.x.D & 3) == 0 && (a.x.sP & 3) == 0) return launch_mode2<1>(a, grid, st);
  return launch_mode2<2>(a, grid, st);
}

}  // namespace vqseg
