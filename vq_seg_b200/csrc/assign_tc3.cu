// TMA-fed, codebook-resident, CTA-pair variant of the fused distance + argmin kernel (the headline path).
//
// Same contract as assign_tc2.cu (it replaces torch.cdist + torch.argmin, vq_img.py:167-168) for NCHW feature
// maps -- the 'b c h w -> b (h w) c' view of vq_img.py:232, pixel-contiguous -- whose codebook operand fits the
// shared memory of two SMs ((K_pad/256) * (D_pad/64) <= 8, D_pad <= 256, e.g. the headline K=512, D=256).
//
// What changed against assign_tc2.cu, and why (scripts/dev/bw_bench.cu, profiles/r02_load_paths.md): eight producer
// warps pulling x through registers (LDG.128, 8 x 64 B per request, 24 requests in flight per thread) move a cold
// 32 MiB map in 20 us; one 3-D TMA tensor load per 128-pixel x 32-channel box (16 KiB), issued by two threads into a
// three-stage ring, moves it in 10.4 us -- bytes in flight are not the limit, requests are.  So here
//   * x arrives by cp.async.bulk.tensor.3d (UTMALDG) as fp32 [32 channels][128 pixels] stages;
//   * eight converter warps turn every stage into the fp16 SWIZZLE_128B K-major A operand (lane = pixel: conflict-free
//     LDS.32 down the channels, one conflict-free STS.128 per 8 channels) and accumulate |x|^2, |fp16(x)-x|^2;
//   * the A operand is a 2-slot ring of 64-dim chunks instead of a whole tile (32 KiB), which pays for the staging;
//   * tiles are 128 pixels of ONE image (TMA zero-fills past the image), so 448-pixel maps need no special case;
//   * no setmaxnreg games: nobody holds rows in registers any more.
// MMA issue, TMEM use, the |e|^2 augmentation step and the single-pass mask epilogue are those of assign_tc2.cu.
// Roles per CTA (20 warps): 0-7 converters, 8-15 epilogue, 16 MMA issuer (leader CTA) + TMEM alloc,
// 17 codebook loader (cp.async.bulk) then x loader, 18-19 x loaders (one TMA-issuing thread per stage).
#include <cuda.h>
#include "tc_common.cuh"
#include "filter_epilogue.cuh"

namespace vqseg {

constexpr int k3Threads = 640;
constexpr int k3Rows = 128;                  // pixels per CTA per tile (pair tile = 256)
constexpr int k3ASlots = 2;                  // ring of 64-dim fp16 A chunks
constexpr int k3Stages = 3;                  // ring of fp32 staging boxes
constexpr int k3StageCh = 32;                // channels per box
constexpr int k3StageBytes = k3StageCh * k3Rows * 4;    // 16 KiB
constexpr int k3Issuers = 3;                 // one TMA-issuing thread per stage (each stage barrier has ONE waiter)
constexpr int k3MaxBTiles = 8;               // resident 16 KiB codebook tiles per CTA
constexpr int k3MaxCC = 2;
constexpr int k3AugBytes = 128 * 16 * 2;     // 4 KiB: 128 codes x 16 fp16, SWIZZLE_NONE core matrices
constexpr uint32_t k3Idesc = make_idesc_f16(256, 256);

struct Tc3Smem {
  static constexpr int off_b = 0;                                          // [k3MaxBTiles] 16 KiB
  static constexpr int off_a = off_b + k3MaxBTiles * kTileBytes;            // [k3ASlots] 16 KiB
  static constexpr int off_stage = off_a + k3ASlots * kTileBytes;           // [k3Stages] 16 KiB
  static constexpr int off_baug = off_stage + k3Stages * k3StageBytes;      // [k3MaxCC] 4 KiB
  static constexpr int off_aaug = off_baug + k3MaxCC * k3AugBytes;          // 256 B: ONE 8-row group, reused by all 16 (SBO = 0)
  static constexpr int off_cand = off_aaug + 256;                           // [2 halves][128][cap] uint16
  static constexpr int off_xchg = off_cand + 2 * k3Rows * kWorkCandCap * 2;  // [128] {m_run, cnt|overflow} of the upper-half warp
  static constexpr int off_xsq = off_xchg + k3Rows * 8;                      // [2 tiles][2 groups][128] float2 {|x|^2, |fp16(x)-x|^2}
  static constexpr int off_bar = off_xsq + 2 * 2 * k3Rows * 8;
  static constexpr int n_bars = 2 * k3Stages + 2 * k3ASlots + 4 + 2 * k3MaxCC;
  static constexpr int off_tmem = off_bar + 8 * n_bars;
  static constexpr int total = off_tmem + 16 + 1024;
};
static_assert(Tc3Smem::total <= 232448, "smem budget");
static_assert(k3Issuers == k3Stages, "each stage barrier is waited on by exactly one issuing thread");

#ifdef VQSEG_DEV
#define VQ3_TRACE(role, slot) do { if (a.trace && lane == 0 && (slot) < 240) \
    a.trace[((long long)blockIdx.x * 4 + (role)) * 256 + (slot)] = clock64(); } while (0)
#else
#define VQ3_TRACE(role, slot) do { } while (0)
#endif

__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2, uint32_t bar) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
               ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(bar) : "memory");
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(k3Threads, 1)
assign_tc3_kernel(const __grid_constant__ CUtensorMap tmap, Tc3Args a) {
  extern __shared__ __align__(1024) unsigned char smem_raw3[];
  unsigned char* smem = smem_raw3 + ((1024u - (smem_u32(smem_raw3) & 1023u)) & 1023u);
  const uint32_t sbase = smem_u32(smem);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const BlobHeader* hdr = reinterpret_cast<const BlobHeader*>(a.blob);
#ifdef VQSEG_DEV
  auto stamp = [&](int slot) {               // dev build: {globaltimer, clock64} of thread 0 at four points of the CTA's life
    if (a.trace && threadIdx.x == 0) {
      unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
      a.trace[((long long)blockIdx.x * 4 + 3) * 256 + 240 + 2 * slot] = (long long)t;
      a.trace[((long long)blockIdx.x * 4 + 3) * 256 + 241 + 2 * slot] = clock64();
    }
  };
#else
  auto stamp = [](int) {};
#endif
  stamp(0);

  const uint32_t bar_sfull = sbase + Tc3Smem::off_bar;                 // [stages]  1 + tx bytes (TMA)
  const uint32_t bar_sempty = bar_sfull + 8 * k3Stages;                // [stages]  8 converter warps
  const uint32_t bar_afull = bar_sempty + 8 * k3Stages;                // [slots]   leader: 16 converter-warp arrivals (8 per CTA)
  const uint32_t bar_aempty = bar_afull + 8 * k3ASlots;                // [slots]   each CTA: 1 (multicast commit)
  const uint32_t bar_tfull = bar_aempty + 8 * k3ASlots;                // [2]       each CTA: 1 (multicast commit)
  const uint32_t bar_tempty = bar_tfull + 16;                          // [2]       leader: 16 epilogue-warp arrivals
  const uint32_t bar_bload = bar_tempty + 16;                          // [k3MaxCC] local bulk-copy completion per code chunk
  const uint32_t bar_bready = bar_bload + 8 * k3MaxCC;                 // [k3MaxCC] leader: 2 (chunk resident in both CTAs)
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + Tc3Smem::off_tmem);
  float2* xsq = reinterpret_cast<float2*>(smem + Tc3Smem::off_xsq);

  const int n_pairs = (int)gridDim.x >> 1;
  const int pair = (int)blockIdx.x >> 1;
  const int my_tiles = a.n_ptiles > pair ? (a.n_ptiles - 1 - pair) / n_pairs + 1 : 0;
  const int ops_per_tile = 2 * a.n_dc;                       // 32-channel boxes per tile
  const int total_ops = my_tiles * ops_per_tile;
  // tile tt of this CTA: global tile 2 * (pair + tt * n_pairs) + rank -> (image, first pixel); tiles past the end
  // address image B, which the tensor map zero-fills
  auto tile_coords = [&](int tt, int& img, int& p0) {
    const int t = 2 * (pair + tt * n_pairs) + (int)rank;
    if (t < a.n_tiles) { img = t / a.tiles_per_image; p0 = (t - img * a.tiles_per_image) * k3Rows; }
    else { img = (int)a.B; p0 = 0; }
  };
  auto issue_box = [&](int q, int issuer) {                   // box q goes to the stage its issuer owns
    const int tt = q / ops_per_tile, h = q - tt * ops_per_tile;
    int img, p0;
    tile_coords(tt, img, p0);
    mbar_wait(bar_sempty + 8 * issuer, (((uint32_t)(q / k3Stages)) & 1) ^ 1);
    mbar_arrive_expect_tx(bar_sfull + 8 * issuer, k3StageBytes);
    tma_load_3d(sbase + Tc3Smem::off_stage + issuer * k3StageBytes, &tmap, p0, h * k3StageCh, img, bar_sfull + 8 * issuer);
  };

  if (threadIdx.x == 0) {
    for (int s = 0; s < k3ASlots; ++s) { mbar_init(bar_afull + 8 * s, 16); mbar_init(bar_aempty + 8 * s, 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(bar_tfull + 8 * b, 1); mbar_init(bar_tempty + 8 * b, 16); }
    for (int c = 0; c < k3MaxCC; ++c) { mbar_init(bar_bload + 8 * c, 1); mbar_init(bar_bready + 8 * c, 2); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 16) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32((const void*)tmem_slot)), "r"(512u));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
  }
  if (warp >= 17) {
    // the x pipeline starts BEFORE the CTA / cluster set-up completes: the loader warps initialise the stage barriers
    // among themselves and put the first three boxes in flight (set-up + first-use latency was 3.3 k cycles of an
    // 18 k-cycle kernel before any byte of x was requested)
    if (warp == 17 && lane == 0) {
      for (int s = 0; s < k3Stages; ++s) { mbar_init(bar_sfull + 8 * s, 1); mbar_init(bar_sempty + 8 * s, 8); }
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    asm volatile("bar.sync 9, 96;" ::: "memory");
    if (lane == 0 && warp - 17 < total_ops) issue_box(warp - 17, warp - 17);
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // launched as a programmatic dependent of the prologue kernel (zeroing + codebook guard): everything above -- and the
  // x boxes the loader warps already have in flight -- overlapped it; what reads the blob or accumulates into the
  // outputs waits here (warps 18-19 only ever load x)
  if (warp < 18) pdl_wait();
  // (tried: pdl_trigger() here + the rescoring kernel as a programmatic dependent, so that its blocks take the SMs of
  // pairs that finish early: 47.8-49.0 -> 50.8-51.8 us per step -- not kept)
  stamp(1);

  const uint32_t lead_afull = mapa_u32(bar_afull, 0);
  const uint32_t lead_tempty = mapa_u32(bar_tempty, 0);

  if (warp < 8) {
    // ================= converters: fp32 [32 ch][128 px] stage -> fp16 K-major A chunk half =================
    // EVERY converter warp takes part in EVERY box, in order (lane = pixel 32 * (warp % 4) + lane, warp / 4 = which 16
    // of the box's 32 channels): all mbarrier waits below are then sequential per barrier -- a parity wait can never
    // be two phases behind (two groups taking alternate boxes could drift apart and alias the phase bit).
    const int chh = warp >> 2;
    const int r = 32 * (warp & 3) + lane;
    float ss = 0.f, sd = 0.f;
    for (int q = 0; q < total_ops; ++q) {
      const int tt = q / ops_per_tile, h = q - tt * ops_per_tile;
      const int dc = h >> 1, hh = h & 1;
      const int a_seq = tt * a.n_dc + dc, slot = a_seq & 1;
      const int s = q % k3Stages;
      if (warp == 0) VQ3_TRACE(0, 2 * q);
      mbar_wait(bar_sfull + 8 * s, (uint32_t)(q / k3Stages) & 1);                    // the box has landed
      if (hh == 0) mbar_wait(bar_aempty + 8 * slot, (((uint32_t)a_seq >> 1) & 1) ^ 1);   // the slot's last MMAs retired
      if (warp == 0) VQ3_TRACE(0, 2 * q + 1);
      const float* st = reinterpret_cast<const float*>(smem + Tc3Smem::off_stage + s * k3StageBytes) + (16 * chh) * k3Rows + r;
      unsigned char* arow = smem + Tc3Smem::off_a + slot * kTileBytes + r * 128;
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        float v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = st[(8 * c + j) * k3Rows];
        uint32_t pk[4];
#pragma unroll
        for (int j = 0; j < 8; j += 2) {
          __half2 hv = __floats2half2_rn(v[j], v[j + 1]);
          const float2 hb = __half22float2(hv);
          const float e0 = hb.x - v[j], e1 = hb.y - v[j + 1];
          ss = fmaf(v[j], v[j], ss); ss = fmaf(v[j + 1], v[j + 1], ss);
          sd = fmaf(e0, e0, sd); sd = fmaf(e1, e1, sd);
          pk[j >> 1] = *reinterpret_cast<uint32_t*>(&hv);
        }
        *reinterpret_cast<uint4*>(arow + (((4 * hh + 2 * chh + c) ^ (r & 7)) * 16)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
      }
      if (h == ops_per_tile - 1) {                             // this warp's share of the row norms is complete
        xsq[((tt & 1) * 2 + chh) * k3Rows + r] = make_float2(ss, sd);
        ss = 0.f; sd = 0.f;
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(bar_sempty + 8 * s);                                   // stage free for the next box
        if (hh == 1) mbar_arrive_cluster_relaxed(lead_afull + 8 * slot);   // chunk complete; leader's barrier (remote for rank 1)
      }
    }
  } else if (warp < 16) {
    // ================= epilogue =================
    const int quarter = warp & 3;                         // TMEM lane quarter this warp may access
    const int half = (warp - 8) >> 2;                     // which 128 of the unit's 256 columns
    const int r = quarter * 32 + lane;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(quarter * 32) << 16) + half * 128;
    const ShortList<unsigned short>::Slots lists(reinterpret_cast<unsigned short*>(smem + Tc3Smem::off_cand), k3Rows, half, r);
    float2* xchg = reinterpret_cast<float2*>(smem + Tc3Smem::off_xchg) + r;
    const FilterBound bound(hdr);
    if (warp == 8) {
      // relay: this CTA's half of each code chunk has landed -> tell the leader's MMA issuer (the loader thread goes
      // straight on to issuing x boxes and must not sit in this wait)
      for (int cc = 0; cc < a.n_cc; ++cc) {
        mbar_wait(bar_bload + 8 * cc, 0);
        if (lane == 0) mbar_arrive_cluster(mapa_u32(bar_bready + 8 * cc, 0));
      }
    }
    int u = 0;
    for (int tt = 0; tt < my_tiles; ++tt) {
      int img, p0;
      tile_coords(tt, img, p0);
      const bool in_range = img < (int)a.B && p0 + r < (int)a.P;
      const long long n = (long long)img * a.P + p0 + r;
      ShortList<unsigned short> sl(lists);
      for (int cc = 0; cc < a.n_cc; ++cc, ++u) {
        if (warp == 8) VQ3_TRACE(2, 4 * u);
        mbar_wait(bar_tfull + 8 * cc, (uint32_t)tt & 1);
        tc_fence_after();
        if (warp == 8) VQ3_TRACE(2, 4 * u + 1);
        if (cc == 0) {
          const float2 n0 = xsq[((tt & 1) * 2 + 0) * k3Rows + r], n1 = xsq[((tt & 1) * 2 + 1) * k3Rows + r];
          sl.start(bound, n0.x + n1.x, n0.y + n1.y, (int)a.D, a.out.slack_t2);
        }
        const uint32_t tb = lane_addr + cc * 256;
#pragma unroll 1
        for (int c = 0; c < 128; c += 32) {
          uint32_t v[32];
          tmem_ld32(tb + c, v);
          sl.scan32(v, cc * 256 + half * 128 + c);
        }
        if (warp == 8) VQ3_TRACE(2, 4 * u + 2);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(lead_tempty + 8 * cc);      // this warp's columns are drained
      }
      sl.finish(half, 1 + quarter, xchg, in_range, n, a.out);
    }
  } else if (warp == 16) {
    if (rank == 0 && elect_one()) {
      // ================= MMA issuer (leader CTA): one elected thread, lean instruction stream (tc_common.cuh) ==========
      // The tile's two accumulators (TMEM columns 0-255 / 256-511) ARE the whole tensor memory, so nothing can be
      // double-buffered across tiles.  What can overlap: the first two A chunks of a tile are multiplied against code
      // chunk 0 as soon as accumulator 0 is drained -- while the epilogue still reads accumulator 1 of the previous
      // tile -- and only then against code chunk 1.  The remaining chunks run dims-outer (each chunk against all
      // code chunks, slot released at once).  At the last chunk the accumulators are completed (|e|^2 step + commit)
      // one after the other, so the epilogue starts on the first while the second still computes.
      const uint64_t aaug = make_desc_noswz(sbase + Tc3Smem::off_aaug, 128, 0);
      const uint32_t a_lo0 = desc_lo_sw128(sbase + Tc3Smem::off_a), b_lo0 = desc_lo_sw128(sbase + Tc3Smem::off_b);
      const int n_dc = a.n_dc, n_cc = a.n_cc;
      auto mma_chunk = [&](int cc, int dc, int slot) {
        const uint32_t al = a_lo0 + (uint32_t)slot * (kTileBytes >> 4);
        const uint32_t bl = b_lo0 + (uint32_t)(cc * n_dc + dc) * (kTileBytes >> 4);
        const uint32_t acc = tmem_base + cc * 256;
        tc_mma_f16_2cta_lo(acc, al, bl, k3Idesc, dc ? 1u : 0u);
        tc_mma_f16_2cta_lo(acc, al + 2, bl + 2, k3Idesc, 1u);
        tc_mma_f16_2cta_lo(acc, al + 4, bl + 4, k3Idesc, 1u);
        tc_mma_f16_2cta_lo(acc, al + 6, bl + 6, k3Idesc, 1u);
        if (dc == n_dc - 1) {
          const uint64_t baug = make_desc_noswz(sbase + Tc3Smem::off_baug + cc * k3AugBytes, 128, 256);
          tc_mma_f16_2cta(acc, aaug, baug, k3Idesc, 1u);     // + s |e_k|^2
          tc_commit_2cta(bar_tfull + 8 * cc);
        }
      };
      int a_seq = 0;                                            // running A chunk number: slot = a_seq & 1, phase = a_seq >> 1
      for (int tt = 0; tt < my_tiles; ++tt) {
        const int n_first = n_dc < 2 ? n_dc : 2;
        for (int cc = 0; cc < n_cc; ++cc) {
          VQ3_TRACE(1, 128 + 2 * (tt * n_cc + cc));
          mbar_wait(bar_tempty + 8 * cc, ((uint32_t)tt & 1) ^ 1);          // both CTAs' epilogues drained it
          VQ3_TRACE(1, 128 + 2 * (tt * n_cc + cc) + 1);
          if (tt == 0) mbar_wait(bar_bready + 8 * cc, 0);                  // this code chunk is resident in both CTAs
          tc_fence_after();
          for (int dc = 0; dc < n_first; ++dc) {
            const int sq = a_seq + dc, slot = sq & 1;
            if (cc == 0) {
              VQ3_TRACE(1, 2 * sq);
              mbar_wait(bar_afull + 8 * slot, ((uint32_t)sq >> 1) & 1);    // both CTAs' halves of the A chunk are converted
              VQ3_TRACE(1, 2 * sq + 1);
              tc_fence_after();
            }
            mma_chunk(cc, dc, slot);
            if (cc == n_cc - 1) tc_commit_2cta(bar_aempty + 8 * slot);     // A slot free in both CTAs
          }
        }
        for (int dc = n_first; dc < n_dc; ++dc) {
          const int sq = a_seq + dc, slot = sq & 1;
          VQ3_TRACE(1, 2 * sq);
          mbar_wait(bar_afull + 8 * slot, ((uint32_t)sq >> 1) & 1);
          VQ3_TRACE(1, 2 * sq + 1);
          tc_fence_after();
          for (int cc = 0; cc < n_cc; ++cc) mma_chunk(cc, dc, slot);
          tc_commit_2cta(bar_aempty + 8 * slot);
        }
        a_seq += n_dc;
      }
    }
  } else {
    // ================= loaders (warps 17-19, one issuing thread each) =================
    const int issuer = warp - 17;
    if (warp == 17) {
      // codebook: this CTA's half of every 256-code chunk stays resident
      {   // A-side augmentation rows: columns 0..2 = c (power of two), rest 0; one 8-row group of SWIZZLE_NONE core
          // matrices (K halves 128 B apart) that the descriptor repeats for all 128 rows (stride-byte-offset 0)
        const __half cval = __float2half_rn(hdr->aug_c);
        const uint32_t c2 = (uint32_t)__half_as_ushort(cval);
        uint4* aa = reinterpret_cast<uint4*>(smem + Tc3Smem::off_aaug);
        if (lane < 16) aa[lane] = lane < 8 ? make_uint4(c2 | (c2 << 16), c2, 0u, 0u) : make_uint4(0u, 0u, 0u, 0u);
        fence_proxy_async();
        __syncwarp();
      }
      if (lane == 0) {
        const unsigned char* img = a.blob + a.off_image;
        const unsigned char* aug = a.blob + a.off_aug;
        const uint32_t bytes = (uint32_t)a.n_dc * kTileBytes + k3AugBytes;
        for (int cc = 0; cc < a.n_cc; ++cc) {
          const int cb = 2 * cc + (int)rank;                       // this CTA's 128 codes of chunk cc
          mbar_arrive_expect_tx(bar_bload + 8 * cc, bytes);
          for (int dc = 0; dc < a.n_dc; ++dc)
            bulk_g2s(sbase + Tc3Smem::off_b + (cc * a.n_dc + dc) * kTileBytes,
                     img + ((long long)cb * a.n_dc + dc) * kTileBytes, kTileBytes, bar_bload + 8 * cc);
          bulk_g2s(sbase + Tc3Smem::off_baug + cc * k3AugBytes, aug + (long long)cb * k3AugBytes, k3AugBytes,
                   bar_bload + 8 * cc);
        }
      }
    }
    // x boxes: issuer i owns stage i and issues the boxes q = i, i + 3, ... (a single thread sustains one tensor load
    // per ~1100 cycles, scripts/dev/bw_bench.cu; three keep the ring busy)
    if (lane == 0) {
      for (int q = issuer + k3Issuers; q < total_ops; q += k3Issuers) {
        VQ3_TRACE(3, 2 * q);
        issue_box(q, issuer);
        VQ3_TRACE(3, 2 * q + 1);
      }
    }
  }

  // ---- teardown ----
  stamp(2);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  stamp(3);
  if (warp == 16) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u));
  }
}

// ---- host side ----------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = nullptr;                 // a driver entry point, not a per-device object
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || !p) {
      (void)cudaGetLastError();
      return nullptr;
    }
    fn = (EncodeTiledFn)p;
  }
  return fn;
}

bool tc3_supported(const Rows& x, int n_cc, int n_dc) {
  if (!(n_dc <= 4 && n_cc <= k3MaxCC && n_cc * n_dc <= k3MaxBTiles)) return false;
  if (x.sP != 1 || (reinterpret_cast<uintptr_t>(x.ptr) & 15) != 0) return false;
  if ((x.sD & 3) != 0 || x.sD <= 0) return false;
  if (x.B > 1 && ((x.sB & 3) != 0 || x.sB <= 0)) return false;
  if (x.P >= (1ll << 31) || x.D >= (1ll << 31) || x.B >= (1ll << 31)) return false;
  return encode_tiled_fn() != nullptr;
}

int launch_assign_tc3(const Rows& x, const Tc3Args& a, cudaStream_t st) {
  int pairs = num_sms() / 2;
  if (a.n_ptiles < pairs) pairs = a.n_ptiles;
  if (pairs <= 0) return 0;
  EncodeTiledFn enc = encode_tiled_fn();
  if (!enc) return VQSEG_EUNSUPPORTED;
  // x as a 3-D tensor (pixel, channel, image), fp32; box = 128 pixels x 32 channels x 1 image; out-of-range
  // elements (past the image, past D, the dummy image of an odd tile count) read as zero
  CUtensorMap tmap;
  const cuuint64_t dims[3] = {(cuuint64_t)x.P, (cuuint64_t)x.D, (cuuint64_t)x.B};
  const cuuint64_t strides[2] = {(cuuint64_t)x.sD * 4, (cuuint64_t)(x.B > 1 ? x.sB : x.sD * x.D) * 4};
  const cuuint32_t box[3] = {(cuuint32_t)k3Rows, (cuuint32_t)k3StageCh, 1};
  const cuuint32_t estr[3] = {1, 1, 1};
  CUresult rc = enc(&tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(x.ptr), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (rc != CUDA_SUCCESS) return VQSEG_EUNSUPPORTED;
  static size_t configured[kMaxDevices] = {0};
  if (int e = ensure_dynamic_smem(assign_tc3_kernel, Tc3Smem::total, configured)) return e;
  cudaError_t le = launch_dependent(assign_tc3_kernel, dim3(2 * pairs), dim3(k3Threads), (size_t)Tc3Smem::total, st, pdl_enabled(), tmap, a);
  if (le != cudaSuccess) return (int)le;
  VQSEG_LAUNCH_CHECK();
  return 0;
}

}  // namespace vqseg
