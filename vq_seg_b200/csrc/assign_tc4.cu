// Streaming CTA-pair variant of the fused distance + argmin kernel: any K, D_pad <= 512 -- the k-means shapes
// (config 4: K=1024, D=512; config 5: K=65536, D=256) and every codebook too large to stay resident.
//
// Same contract as assign_tc.cu (it replaces torch.cdist + torch.argmin, vq_img.py:167-168 / :39-41).  What limited
// the single-CTA streaming kernel (assign_tc.cu) was shared-memory/L2 traffic, not the tensor pipe: it re-read and
// re-converted the 128-row x tile for EVERY 256-code chunk and pulled a full 32 KiB codebook stage per 512 MMA
// cycles: ~125 B/clk/SM out of L2 (measured 31-41 % of the tensor peak).  Here
//   * a cluster of 2 CTAs owns 256 rows per tile (UMMA M = 256, cta_group::2) and each CTA loads only ITS half (128
//     codes) of every 256-code chunk: 16 KiB per stage instead of 32;
//   * the fp16 A operand of a tile is converted ONCE and stays resident in an 8-slot ring of 64-dim chunks
//     (128 KiB): one whole tile at D=512 -- its slots are released one by one during the last code chunk, so the
//     next tile's conversion overlaps it -- or two tiles (double-buffered) at D<=256;
//   * the two 256-column accumulators in TMEM alternate between consecutive code chunks, so the epilogue of chunk c
//     overlaps the MMAs of chunk c+1 for the whole run (with the codebook resident, assign_tc3.cu, TMEM holds exactly
//     one tile and nothing overlaps across tiles);
//   * x arrives by TMA tensor loads in both layouts: NCHW maps as [32 ch][128 px] boxes (3-D map), packed rows as
//     [128 rows][32 dims] boxes with the 128-byte swizzle (2-D map), so the converters' reads are conflict-free.
// Roles per CTA (21 warps): 0-7 converters, 8-15 epilogue, 16 MMA issuer (leader CTA) + TMEM alloc, 17 codebook
// loader (cp.async.bulk), 18 relay (local stage landed -> leader's "both halves resident" barrier), 19-20 x loaders.
#include <cuda.h>
#include <string.h>
#include "tc_common.cuh"
#include "filter_epilogue.cuh"

namespace vqseg {

constexpr int k4Threads = 21 * 32;
constexpr int k4Rows = 128;                  // rows per CTA per tile (pair tile = 256)
constexpr int k4ASlots = 8;                  // ring of 64-dim fp16 A chunks (16 KiB each)
constexpr int k4BStages = 3;                 // ring of 128-code x 64-dim codebook stages (16 KiB each)
constexpr int k4XStages = 2;                 // ring of fp32 x boxes (16 KiB each), one issuing thread per stage (power of two)
constexpr int k4BoxDims = 32;                // dims per x box
constexpr int k4XBytes = k4BoxDims * k4Rows * 4;
constexpr int k4AugBytes = 128 * 16 * 2;     // 4 KiB: 128 codes x 16 fp16, SWIZZLE_NONE core matrices
constexpr uint32_t k4Idesc = make_idesc_f16(256, 256);

struct Tc4Smem {
  static constexpr int off_a = 0;                                          // [k4ASlots] 16 KiB
  static constexpr int off_b = off_a + k4ASlots * kTileBytes;               // [k4BStages] 16 KiB
  static constexpr int off_x = off_b + k4BStages * kTileBytes;              // [k4XStages] 16 KiB
  static constexpr int off_baug = off_x + k4XStages * k4XBytes;             // [2] 4 KiB: |e|^2 limb tiles, by unit parity
  static constexpr int off_aaug = off_baug + 2 * k4AugBytes;                // 256 B: ONE 8-row group, reused by all 16 (SBO = 0)
  static constexpr int off_cand = off_aaug + 256;                           // [2 halves][128][cap] uint16
  static constexpr int off_xchg = off_cand + 2 * k4Rows * kWorkCandCap * 2;  // [128] {m_run, cnt|overflow} of the upper-half warp
  static constexpr int off_xsq = off_xchg + k4Rows * 8;                      // [2 tiles][2 halves of a box][128] float2
  static constexpr int off_bar = off_xsq + 2 * 2 * k4Rows * 8;
  static constexpr int n_bars = 2 * k4ASlots + 3 * k4BStages + 2 * k4XStages + 4 + 2 + 2 + k4ASlots;
  static constexpr int off_tmem = off_bar + 8 * n_bars;
  static constexpr int total = off_tmem + 16 + 1024;
};
static_assert(Tc4Smem::total <= 232448, "smem budget");

#ifdef VQSEG_DEV
#define VQ4_TRACE(role, slot) do { if (a.trace && lane == 0 && (slot) < 240) \
    a.trace[((long long)blockIdx.x * 4 + (role)) * 256 + (slot)] = clock64(); } while (0)
#else
#define VQ4_TRACE(role, slot) do { } while (0)
#endif

__device__ __forceinline__ void tma4_load_3d(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2, uint32_t bar) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
               ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(bar) : "memory");
}
__device__ __forceinline__ void tma4_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
               ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(bar) : "memory");
}

// MODE 0: NCHW maps (pixel-contiguous), tiles of 128 pixels of one image; 1: packed rows (dim-contiguous);
// 2: PREPARED samples (vqseg_samples_prepare_f32): the fp16 A chunks already exist in global memory as ready-made
//    SWIZZLE_128B tiles, [row tile][dim chunk] x 16 KiB, and arrive by cp.async.bulk straight into the A ring -- no
//    converter warps, no fp32 staging; the row norms come from the blob.  For inputs that are assigned many times
//    (the Lloyd iterations of k-means: the same samples against new means): the conversion, which bounds the kernel
//    at K ~ 1024 (DESIGN.md 4.0b), is paid once.
template <int MODE>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(k4Threads, 1)
assign_tc4_kernel(const __grid_constant__ CUtensorMap tmap, Tc4Args a) {
  constexpr bool ROWS = MODE != 0;        // row index = tile * 128 + r (no images)
  constexpr bool PRE = MODE == 2;
  extern __shared__ __align__(1024) unsigned char smem_raw4[];
  unsigned char* smem = smem_raw4 + ((1024u - (smem_u32(smem_raw4) & 1023u)) & 1023u);
  const uint32_t sbase = smem_u32(smem);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const BlobHeader* hdr = reinterpret_cast<const BlobHeader*>(a.blob);

  const uint32_t bar_afull = sbase + Tc4Smem::off_bar;                 // [A slots] leader: 16 converter-warp arrivals (8 per CTA)
  const uint32_t bar_aempty = bar_afull + 8 * k4ASlots;                // [A slots] each CTA: 1 (multicast commit after the LAST code chunk)
  const uint32_t bar_bfull = bar_aempty + 8 * k4ASlots;                // [B stages] local: 1 + tx bytes (bulk copies)
  const uint32_t bar_bready = bar_bfull + 8 * k4BStages;               // [B stages] leader: 2 relay arrivals (both halves resident)
  const uint32_t bar_bempty = bar_bready + 8 * k4BStages;              // [B stages] each CTA: 1 (multicast commit)
  const uint32_t bar_xfull = bar_bempty + 8 * k4BStages;               // [X stages] 1 + tx bytes (TMA)
  const uint32_t bar_xempty = bar_xfull + 8 * k4XStages;               // [X stages] 8 converter warps
  const uint32_t bar_tfull = bar_xempty + 8 * k4XStages;               // [2] each CTA: 1 (multicast commit)
  const uint32_t bar_tempty = bar_tfull + 16;                          // [2] leader: 16 epilogue-warp arrivals
  const uint32_t bar_gempty = bar_tempty + 16;                         // [2] each CTA: 1 (multicast commit): limb tile free
  const uint32_t bar_nempty = bar_gempty + 16;                         // [2] local: 8 epilogue warps have read the tile's row norms
  const uint32_t bar_aload = bar_nempty + 16;                          // [A slots] MODE 2, local: 1 + tx bytes (bulk copy of a chunk)
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + Tc4Smem::off_tmem);
  float2* xsq = reinterpret_cast<float2*>(smem + Tc4Smem::off_xsq);

  // A work item is a pair tile (256 rows) x one slice of `a.n_dc` dim chunks.  Normally a slice is the whole row
  // (n_slices == 1).  Split-D mode (few rows, many dims: the 1024- / 2048-channel layers of a model have 2-16 pair
  // tiles for 74 SM pairs) cuts the dims into n_slices slices so that every SM pair has an item; an item then ADDS
  // its partial scores into a[.part_scores] and shortlist_kernel builds the short-lists once all slices have landed.
  const int n_pairs = (int)gridDim.x >> 1;
  const int pair = (int)blockIdx.x >> 1;
  // (Tried: every pair starting its walk over the code chunks at its own offset, so that the pairs do not fetch the same
  // codebook tile at the same moment -- no change at K = 65536: 110.0-110.5 ms against 110.1-111.0.)
  const int n_items = a.n_ptiles * a.n_slices;
  const int my_tiles = n_items > pair ? (n_items - 1 - pair) / n_pairs + 1 : 0;
  const int boxes_per_tile = 2 * a.n_dc;
  const int total_boxes = my_tiles * boxes_per_tile;
  const int my_units = my_tiles * a.n_cc;
  // item tt of this pair = global item pair + tt * n_pairs = (pair tile, slice); this CTA's tile = 2 * pair tile + rank
  auto tile_id = [&](int tt) { return 2 * ((pair + tt * n_pairs) / a.n_slices) + (int)rank; };
  auto slice_of = [&](int tt) { return (pair + tt * n_pairs) % a.n_slices; };
  auto issue_box = [&](int q, int issuer) {                   // box q goes to the stage its issuer owns
    const int tt = q / boxes_per_tile, h = q - tt * boxes_per_tile;
    const int t = tile_id(tt);
    const int dim0 = (slice_of(tt) * boxes_per_tile + h) * k4BoxDims;      // first dim of the box
    mbar_wait(bar_xempty + 8 * issuer, (((uint32_t)(q / k4XStages)) & 1) ^ 1);
    mbar_arrive_expect_tx(bar_xfull + 8 * issuer, k4XBytes);
    const uint32_t dst = sbase + Tc4Smem::off_x + issuer * k4XBytes;
    if (ROWS) {
      // tiles past the end start beyond the last row: the tensor map zero-fills
      tma4_load_2d(dst, &tmap, dim0, t < a.n_tiles ? t * k4Rows : (int)a.n_rows, bar_xfull + 8 * issuer);
    } else {
      int img = (int)a.B, p0 = 0;
      if (t < a.n_tiles) { img = t / a.tiles_per_image; p0 = (t - img * a.tiles_per_image) * k4Rows; }
      tma4_load_3d(dst, &tmap, p0, dim0, img, bar_xfull + 8 * issuer);
    }
  };

  if (threadIdx.x == 0) {
    for (int s = 0; s < k4ASlots; ++s) {
      mbar_init(bar_afull + 8 * s, PRE ? 2 : 16); mbar_init(bar_aempty + 8 * s, 1); mbar_init(bar_aload + 8 * s, 1);
    }
    for (int s = 0; s < k4BStages; ++s) { mbar_init(bar_bfull + 8 * s, 1); mbar_init(bar_bready + 8 * s, 2); mbar_init(bar_bempty + 8 * s, 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(bar_tfull + 8 * b, 1); mbar_init(bar_tempty + 8 * b, 16); mbar_init(bar_gempty + 8 * b, 1); mbar_init(bar_nempty + 8 * b, 8); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 16) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32((const void*)tmem_slot)), "r"(512u));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
  }
  if (warp >= 19 && !PRE) {
    // the x pipeline starts before the CTA / cluster set-up completes (see assign_tc3.cu)
    if (warp == 19 && lane == 0) {
      for (int s = 0; s < k4XStages; ++s) { mbar_init(bar_xfull + 8 * s, 1); mbar_init(bar_xempty + 8 * s, 8); }
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap) : "memory");
    }
    asm volatile("bar.sync 9, 64;" ::: "memory");
    if (lane == 0 && warp - 19 < total_boxes) issue_box(warp - 19, warp - 19);
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // a programmatic dependent of the prologue kernel (zeroing, codebook guard, split-D scratch): the set-up above and
  // the x boxes already in flight overlapped it; the warps that read the blob or write outputs wait here
  if (warp >= 8 && warp < 19) pdl_wait();
  const uint32_t lead_afull = mapa_u32(bar_afull, 0);
  const uint32_t lead_tempty = mapa_u32(bar_tempty, 0);
  const uint32_t lead_bready = mapa_u32(bar_bready, 0);

  if (warp < 8) {
    // ================= converters: fp32 x box -> fp16 K-major A chunk half =================
    // every converter warp takes part in every box, in order (all mbarrier waits sequential per barrier);
    // lane = row 32 * (warp % 4) + lane of the tile, warp / 4 = which 16 of the box's 32 dims
    const int chh = warp >> 2;
    const int r = 32 * (warp & 3) + lane;
    float ss = 0.f, sd = 0.f;
    // loop counters kept incrementally (a division by the runtime box count per box is 20+ dependent instructions)
    int slot = 0; uint32_t apar = 1;                           // A slot of the current chunk, parity of its "empty" phase
    int q = 0;
    const int conv_tiles = PRE ? 0 : my_tiles;                 // (MODE 2: nothing to convert)
    for (int tt = 0; tt < conv_tiles; ++tt)
    for (int h = 0; h < boxes_per_tile; ++h, ++q) {
      const int hh = h & 1;
      const int s = q & (k4XStages - 1);
      if (warp == 0) VQ4_TRACE(0, 2 * q);
      mbar_wait(bar_xfull + 8 * s, (uint32_t)(q / k4XStages) & 1);                   // the box has landed
      if (hh == 0) mbar_wait(bar_aempty + 8 * slot, apar);                          // the slot's last MMAs retired
      if (warp == 0) VQ4_TRACE(0, 2 * q + 1);
      const float* st = reinterpret_cast<const float*>(smem + Tc4Smem::off_x + s * k4XBytes);
      unsigned char* arow = smem + Tc4Smem::off_a + slot * kTileBytes + r * 128;
      // all 16 values first (four LDS.128 / sixteen conflict-free LDS.32 in flight), then the arithmetic with
      // independent accumulators: two warps per scheduler hide little latency, dependent chains would set the pace
      float v[16];
      if (ROWS) {
        // [128 rows][32 dims], 128-byte rows, 16-byte chunk j of row r stored at j ^ (r & 7)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float4 q4 = *reinterpret_cast<const float4*>(st + r * 32 + (((4 * chh + j) ^ (r & 7)) << 2));
          v[4 * j] = q4.x; v[4 * j + 1] = q4.y; v[4 * j + 2] = q4.z; v[4 * j + 3] = q4.w;
        }
      } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = st[(16 * chh + j) * k4Rows + r];
      }
      uint32_t pk[8];
      float s0 = 0.f, s1 = 0.f, d0 = 0.f, d1 = 0.f;
#pragma unroll
      for (int j = 0; j < 16; j += 2) {
        __half2 hv = __floats2half2_rn(v[j], v[j + 1]);
        const float2 hb = __half22float2(hv);
        const float e0 = hb.x - v[j], e1 = hb.y - v[j + 1];
        s0 = fmaf(v[j], v[j], s0); s1 = fmaf(v[j + 1], v[j + 1], s1);
        d0 = fmaf(e0, e0, d0); d1 = fmaf(e1, e1, d1);
        pk[j >> 1] = *reinterpret_cast<uint32_t*>(&hv);
      }
      ss += s0 + s1; sd += d0 + d1;
      *reinterpret_cast<uint4*>(arow + (((4 * hh + 2 * chh) ^ (r & 7)) * 16)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
      *reinterpret_cast<uint4*>(arow + (((4 * hh + 2 * chh + 1) ^ (r & 7)) * 16)) = make_uint4(pk[4], pk[5], pk[6], pk[7]);
      if (h == boxes_per_tile - 1) {                           // this warp's share of the row norms is complete
        // with few dim chunks the A ring holds several tiles: never overwrite norms the epilogue has not read yet
        mbar_wait(bar_nempty + 8 * (tt & 1), (((uint32_t)tt >> 1) & 1) ^ 1);
        xsq[((tt & 1) * 2 + chh) * k4Rows + r] = make_float2(ss, sd);
        ss = 0.f; sd = 0.f;
      }
      if (hh == 1) fence_proxy_async();          // the chunk's A writes (both boxes) -> visible to the tensor core's proxy
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(bar_xempty + 8 * s);                                   // stage free for the next box (reads only: no fence)
        if (hh == 1) mbar_arrive_cluster_relaxed(lead_afull + 8 * slot);   // chunk complete; leader's barrier (remote for rank 1)
      }
      if (hh == 1 && ++slot == k4ASlots) { slot = 0; apar ^= 1u; }
    }
  } else if (warp < 16) {
    // ================= epilogue (8 warps: two per TMEM lane quarter, 128 columns each) =================
    const int quarter = warp & 3;
    const int half = (warp - 8) >> 2;
    const int r = quarter * 32 + lane;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(quarter * 32) << 16) + half * 128;
    const ShortList<unsigned short>::Slots lists(reinterpret_cast<unsigned short*>(smem + Tc4Smem::off_cand), k4Rows, half, r);
    float2* xchg = reinterpret_cast<float2*>(smem + Tc4Smem::off_xchg) + r;
    const FilterBound bound(hdr);
    int u = 0;
    for (int tt = 0; tt < my_tiles; ++tt) {
      const int t = tile_id(tt);
      long long n = -1;                                       // global row of this lane, -1 = none
      if (t < a.n_tiles) {
        if (ROWS) { const long long nn = (long long)t * k4Rows + r; if (nn < a.n_rows) n = nn; }
        else {
          const int img = t / a.tiles_per_image, p0 = (t - img * a.tiles_per_image) * k4Rows;
          if (p0 + r < (int)a.P) n = (long long)img * a.P + p0 + r;
        }
      }
      const bool in_range = n >= 0;
      if (a.part_scores) {
        // ---- split-D mode: add this item's partial scores (and its share of the row norms) to the scratch arrays
        for (int cc = 0; cc < a.n_cc; ++cc, ++u) {
          const int buf = u & 1;
          mbar_wait(bar_tfull + 8 * buf, (uint32_t)(u >> 1) & 1);
          tc_fence_after();
          if (cc == 0) {
            const float2 n0 = xsq[((tt & 1) * 2 + 0) * k4Rows + r], n1 = xsq[((tt & 1) * 2 + 1) * k4Rows + r];
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_nempty + 8 * (tt & 1));
            if (in_range && half == 0) {                               // (split-D mode is never combined with MODE 2)
              atomicAdd(a.part_norms + 2 * n, n0.x + n1.x);
              atomicAdd(a.part_norms + 2 * n + 1, n0.y + n1.y);
            }
          }
          const uint32_t tb = lane_addr + buf * 256;
          float* dst = a.part_scores + (in_range ? n : 0) * (long long)a.K_pad + cc * 256 + half * 128;
#pragma unroll 1
          for (int c = 0; c < 128; c += 32) {
            uint32_t v[32];
            tmem_ld32(tb + c, v);
            if (in_range) {
#pragma unroll
              for (int j = 0; j < 32; j += 4)
                atomicAdd(reinterpret_cast<float4*>(dst + c + j),
                          make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]), __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3])));
            }
          }
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(lead_tempty + 8 * buf);
        }
        continue;
      }
      ShortList<unsigned short> sl(lists);
      for (int cc = 0; cc < a.n_cc; ++cc, ++u) {
        const int buf = u & 1;
        if (warp == 8) VQ4_TRACE(2, 4 * u);
        mbar_wait(bar_tfull + 8 * buf, (uint32_t)(u >> 1) & 1);
        tc_fence_after();
        if (warp == 8) VQ4_TRACE(2, 4 * u + 1);
        if (cc == 0) {
          float2 n0, n1 = make_float2(0.f, 0.f);
          if (PRE) {
            n0 = a.samp_norms[(long long)t * k4Rows + r];               // {|x|^2, |fp16(x) - x|^2} from the prepared blob
          } else {
            n0 = xsq[((tt & 1) * 2 + 0) * k4Rows + r]; n1 = xsq[((tt & 1) * 2 + 1) * k4Rows + r];
          }
          sl.start(bound, n0.x + n1.x, n0.y + n1.y, (int)a.D, a.out.slack_t2);
          __syncwarp();
          if (!PRE && lane == 0) mbar_arrive(bar_nempty + 8 * (tt & 1));  // the converters may reuse this norm buffer
        }
        const uint32_t tb = lane_addr + buf * 256;
#pragma unroll 1
        for (int c = 0; c < 128; c += 32) {
          uint32_t v[32];
          tmem_ld32(tb + c, v);
          sl.scan32(v, cc * 256 + half * 128 + c);
        }
        if (warp == 8) VQ4_TRACE(2, 4 * u + 2);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(lead_tempty + 8 * buf);     // this warp's columns are drained
      }
      sl.finish(half, 1 + quarter, xchg, in_range, n, a.out);
    }
  } else if (warp == 16) {
    if (rank == 0 && elect_one()) {
      // ================= MMA issuer (leader CTA): ONE thread, the leanest instruction stream we can give it ===========
      // (tc_common.cuh "lean MMA issue": every instruction here is ~5 cycles of a 128-cycle MMA slot)
      const uint64_t aaug = make_desc_noswz(sbase + Tc4Smem::off_aaug, 128, 0);
      const uint32_t a_lo0 = desc_lo_sw128(sbase + Tc4Smem::off_a), b_lo0 = desc_lo_sw128(sbase + Tc4Smem::off_b);
      const int n_dc = a.n_dc, n_cc = a.n_cc;
      int slot0 = 0; uint32_t apar0 = 0;                       // first A slot of the current tile and its phase parity
      int bs = 0; uint32_t bpar = 0;                           // codebook stage and its phase parity
      uint32_t tpar = 0;                                       // bit b = parity of the next tempty phase of accumulator b
      int u = 0;
      for (int tt = 0; tt < my_tiles; ++tt) {
        int slot = slot0; uint32_t apar = apar0;
        const bool with_aug = slice_of(tt) == 0;                // |e|^2 enters once per row, with the first slice
        for (int cc = 0; cc < n_cc; ++cc, ++u) {
          const int buf = u & 1;
          const uint32_t acc = tmem_base + buf * 256;
          VQ4_TRACE(1, 128 + 2 * u);
          mbar_wait(bar_tempty + 8 * buf, ((tpar >> buf) & 1) ^ 1);          // both CTAs' epilogues drained this accumulator
          tpar ^= 1u << buf;
          VQ4_TRACE(1, 128 + 2 * u + 1);
          const bool last_cc = cc == n_cc - 1;
          slot = slot0; apar = apar0;
          for (int dc = 0; dc < n_dc; ++dc) {
            if (cc == 0) mbar_wait(bar_afull + 8 * slot, apar);              // both CTAs converted the chunk
            mbar_wait(bar_bready + 8 * bs, bpar);                            // both halves of the stage landed
            tc_fence_after();
            const uint32_t al = a_lo0 + (uint32_t)slot * (kTileBytes >> 4), bl = b_lo0 + (uint32_t)bs * (kTileBytes >> 4);
            tc_mma_f16_2cta_lo(acc, al, bl, k4Idesc, dc ? 1u : 0u);
            tc_mma_f16_2cta_lo(acc, al + 2, bl + 2, k4Idesc, 1u);
            tc_mma_f16_2cta_lo(acc, al + 4, bl + 4, k4Idesc, 1u);
            tc_mma_f16_2cta_lo(acc, al + 6, bl + 6, k4Idesc, 1u);
            if (dc == n_dc - 1) {
              // the limb tile of this unit travelled with its first codebook stage (same barrier)
              const uint64_t baug = make_desc_noswz(sbase + Tc4Smem::off_baug + buf * k4AugBytes, 128, 256);
              if (with_aug) tc_mma_f16_2cta(acc, aaug, baug, k4Idesc, 1u);   // + s |e_k|^2
              tc_commit_2cta(bar_gempty + 8 * buf);
              tc_commit_2cta(bar_tfull + 8 * buf);
            }
            tc_commit_2cta(bar_bempty + 8 * bs);                             // codebook stage free in both CTAs
            if (last_cc) tc_commit_2cta(bar_aempty + 8 * slot);              // A chunk free: the tile's last use of it
            if (++bs == k4BStages) { bs = 0; bpar ^= 1u; }
            if (++slot == k4ASlots) { slot = 0; apar ^= 1u; }
          }
        }
        slot0 = slot; apar0 = apar;
      }
    }
  } else if (warp == 17) {
    // ================= codebook loader: this CTA's half (128 codes) of every 256-code chunk, chunk by chunk ============
    {   // A-side augmentation rows (see assign_tc3.cu): one 8-row group repeated by the descriptor (SBO = 0)
      const __half cval = __float2half_rn(hdr->aug_c);
      const uint32_t c2 = (uint32_t)__half_as_ushort(cval);
      uint4* aa = reinterpret_cast<uint4*>(smem + Tc4Smem::off_aaug);
      if (lane < 16) aa[lane] = lane < 8 ? make_uint4(c2 | (c2 << 16), c2, 0u, 0u) : make_uint4(0u, 0u, 0u, 0u);
      fence_proxy_async();
      __syncwarp();
    }
    if (lane == 0) {
      const unsigned char* img = a.blob + a.off_image;
      const unsigned char* aug = a.blob + a.off_aug;
      int bq = 0;
      for (int u = 0; u < my_units; ++u) {
        const int cc = u % a.n_cc, buf = u & 1;
        const int cb = 2 * cc + (int)rank;                       // this CTA's 128 codes of chunk cc
        const int dc0 = slice_of(u / a.n_cc) * a.n_dc;           // first dim chunk of the item's slice
        for (int dc = 0; dc < a.n_dc; ++dc, ++bq) {
          const int bs = bq % k4BStages;
          mbar_wait(bar_bempty + 8 * bs, (((uint32_t)(bq / k4BStages)) & 1) ^ 1);
          if (dc == 0) {
            mbar_wait(bar_gempty + 8 * buf, (((uint32_t)u >> 1) & 1) ^ 1);             // the limb tile's last reader retired
            mbar_arrive_expect_tx(bar_bfull + 8 * bs, kTileBytes + k4AugBytes);
            bulk_g2s(sbase + Tc4Smem::off_baug + buf * k4AugBytes, aug + (long long)cb * k4AugBytes, k4AugBytes, bar_bfull + 8 * bs);
          } else {
            mbar_arrive_expect_tx(bar_bfull + 8 * bs, kTileBytes);
          }
          bulk_g2s(sbase + Tc4Smem::off_b + bs * kTileBytes, img + ((long long)cb * a.n_dc_total + dc0 + dc) * kTileBytes, kTileBytes,
                   bar_bfull + 8 * bs);
        }
      }
    }
  } else if (warp == 18) {
    // ================= relay: this CTA's half of a stage has landed -> the leader's "both halves" barrier ==============
    const int total_stages = my_units * a.n_dc;
    for (int bq = 0; bq < total_stages; ++bq) {
      const int bs = bq % k4BStages;
      mbar_wait(bar_bfull + 8 * bs, ((uint32_t)(bq / k4BStages)) & 1);
      if (lane == 0) mbar_arrive_cluster(lead_bready + 8 * bs);
      __syncwarp();
    }
  } else {
    // ================= x loaders (warps 19-20): issuer i owns stage i, boxes q = i, i + 2, ... =================
    if (PRE) {
      // MODE 2: warp 19 streams this CTA's ready-made A chunks into the ring, warp 20 tells the leader's MMA issuer
      // when a chunk has landed here (the "full" barrier of a slot then counts the two CTAs)
      if (lane == 0) {
        int slot = 0; uint32_t par = warp == 19 ? 1u : 0u;     // 19: parity of the slot's "empty" phase; 20: of its "landed" phase
        for (int tt = 0; tt < my_tiles; ++tt) {
          const long long t = tile_id(tt);
          for (int dc = 0; dc < a.n_dc; ++dc) {
            if (warp == 19) {
              mbar_wait(bar_aempty + 8 * slot, par);
              mbar_arrive_expect_tx(bar_aload + 8 * slot, kTileBytes);
              bulk_g2s(sbase + Tc4Smem::off_a + slot * kTileBytes, a.samp_img + (t * a.n_dc_total + dc) * kTileBytes, kTileBytes,
                       bar_aload + 8 * slot);
            } else {
              mbar_wait(bar_aload + 8 * slot, par);
              mbar_arrive_cluster(lead_afull + 8 * slot);
            }
            if (++slot == k4ASlots) { slot = 0; par ^= 1u; }
          }
        }
      }
    } else if (lane == 0) {
      const int issuer = warp - 19;
      for (int q = issuer + k4XStages; q < total_boxes; q += k4XStages) issue_box(q, issuer);
    }
  }

  // ---- teardown ----
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 16) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u));
  }
}

// ---- prepared samples (MODE 2): fp16 A tiles + row norms, built once per input --------------------------------------
// image tile (row tile, dc): 128 rows x 64 dims of fp16(x), SWIZZLE_128B K-major like the codebook image:
//   byte = row*128 + ((col/8) ^ (row & 7))*16 + (col % 8)*2;  rows past the end and dims past D are zero
__global__ void __launch_bounds__(256) samples_pack_kernel(Rows x, long long n_rows, long long rows_padded, int D_pad,
                                                           unsigned char* __restrict__ img, float* __restrict__ norms) {
  // thread = (row, group of 8 dims): 32 bytes in, 16 bytes out; the row's |x|^2 and |fp16(x) - x|^2 are reduced over the
  // lanes that share the row (contiguous lanes: a segmented suffix sum by shuffles) and added to `norms` (zeroed)
  const int D = (int)x.D, g8 = D_pad / 8, n_dc = D_pad / kDChunk, lane = threadIdx.x & 31;
  const long long total = rows_padded * g8;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long base = (long long)blockIdx.x * blockDim.x + (threadIdx.x & ~31); base < total; base += stride) {
    const long long i = base + lane;
    const bool valid = i < total;
    const long long n = valid ? i / g8 : -1 - lane;
    const int d8 = valid ? (int)(i % g8) * 8 : 0;
    float ss = 0.f, sd = 0.f;
    if (valid) {
      __align__(16) __half h[8];
      const float* xr = n < n_rows ? x.row(n) : nullptr;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float v = (xr && d8 + j < D) ? __ldg(xr + (long long)(d8 + j) * x.sD) : 0.f;
        h[j] = __float2half_rn(v);
        const float e = __half2float(h[j]) - v;
        ss = fmaf(v, v, ss); sd = fmaf(e, e, sd);
      }
      const long long tile = n / 128;
      const int row = (int)(n % 128), dc = d8 / kDChunk, c8 = (d8 % kDChunk) / 8;
      unsigned char* tp = img + (tile * n_dc + dc) * kTileBytes;
      *reinterpret_cast<uint4*>(tp + row * 128 + ((c8 ^ (row & 7)) * 16)) = *reinterpret_cast<const uint4*>(h);
    }
    const unsigned same = __match_any_sync(0xffffffffu, n);
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const float a = __shfl_down_sync(0xffffffffu, ss, o), b2 = __shfl_down_sync(0xffffffffu, sd, o);
      if (lane + o < 32 && ((same >> (lane + o)) & 1u)) { ss += a; sd += b2; }
    }
    if (valid && n < n_rows && (lane == 0 || !((same >> (lane - 1)) & 1u))) {     // first lane of the row's segment
      atomicAdd(norms + 2 * n, ss);
      atomicAdd(norms + 2 * n + 1, sd);
    }
  }
}
int launch_samples_prepare(const Rows& x, long long rows_padded, int D_pad, unsigned char* img, float2* norms, cudaStream_t st) {
  const long long n_rows = x.n_rows();
  cudaError_t e = cudaMemsetAsync(norms, 0, (size_t)rows_padded * sizeof(float2), st);
  if (e != cudaSuccess) return (int)e;
  long long blocks = (rows_padded * (D_pad / 8) + 255) / 256;
  const long long cap = (long long)num_sms() * 16;
  samples_pack_kernel<<<(unsigned)(blocks < cap ? blocks : cap), 256, 0, st>>>(x, n_rows, rows_padded, D_pad, img,
                                                                               reinterpret_cast<float*>(norms));
  VQSEG_LAUNCH_CHECK();
  return 0;
}

// ---- split-D mode, second step: the short-list of every row over its summed scores ------------------------------------
// One warp per row: the row minimum, the same error bound as the filters' epilogues (from the summed |x|^2 and
// |fp16(x) - x|^2 and the blob's header), the codes within the bound in ascending order.  One survivor: final index;
// otherwise a work record for the rescoring pass (more than kWorkCandCap survivors: "score every code").
__global__ void __launch_bounds__(256) shortlist_kernel(ShortlistArgs a) {
  const FilterBound bound(reinterpret_cast<const BlobHeader*>(a.blob));
  const int lane = threadIdx.x & 31;
  const long long w0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long n = w0; n < a.n_rows; n += nw) {
    const float slack = bound.slack(a.norms[2 * n], a.norms[2 * n + 1], a.D, a.out.slack_t2);
    bool overflow = !(slack < 3.0e38f) || bound.defer_all;
    const float* sc = a.scores + n * (long long)a.K_pad;
    float m = __int_as_float(0x7f800000);
    for (int k = 4 * lane; k < a.K_pad; k += 128) {
      const float4 v = *reinterpret_cast<const float4*>(sc + k);
      m = fminf(m, fminf(fminf(v.x, v.y), fminf(v.z, v.w)));
    }
    m = warp_min_f(m);
    const float thr = m + slack;
    int cnt = 0, mine = -1;                                 // lane l keeps the l-th survivor (l < kWorkCandCap)
    for (int k0 = 0; k0 < a.K_pad && !overflow; k0 += 32) {
      const int k = k0 + lane;
      const bool hit = k < a.out.K && !(thr - sc[k] < 0.f); // the epilogues' sign-bit test: a NaN score is a survivor
      const uint32_t hm = __ballot_sync(0xffffffffu, hit);
      int pos = cnt + __popc(hm & ((1u << lane) - 1));
      // survivor number `pos` goes to lane `pos`
#pragma unroll 1
      for (uint32_t rest = hm; rest;) {
        const int src = __ffs(rest) - 1;
        rest &= rest - 1;
        const int p = __shfl_sync(0xffffffffu, pos, src);
        if (lane == p) mine = k0 + src;
      }
      cnt += __popc(hm);
      if (cnt > kWorkCandCap) overflow = true;
    }
    const int first = __shfl_sync(0xffffffffu, mine, 0);
    if (!overflow && cnt == 1 && !a.out.force_rescore) {
      if (lane == 0) settle_row(a.out, n, first);
    } else {
      defer_row_warp(a.out, n, cnt, overflow, mine, lane);
    }
  }
}

int launch_shortlist(const ShortlistArgs& a, cudaStream_t st) {
  long long blocks = (a.n_rows * 32 + 255) / 256;
  const long long cap = (long long)num_sms() * 8;
  if (blocks > cap) blocks = cap;
  shortlist_kernel<<<(unsigned)blocks, 256, 0, st>>>(a);
  VQSEG_LAUNCH_CHECK();
  return 0;
}

// ---- host side ----------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn4)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                   const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn4 encode_tiled_fn4() {
  static EncodeTiledFn4 fn = nullptr;                // a driver entry point, not a per-device object
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || !p) {
      (void)cudaGetLastError();
      return nullptr;
    }
    fn = (EncodeTiledFn4)p;
  }
  return fn;
}

// 0: not supported; 1: NCHW maps (pixel-contiguous); 2: packed rows (dim-contiguous, one flat row range)
int tc4_layout(const Rows& x, long long K_pad, int n_dc) {      // n_dc: dim chunks per work item (a slice in split-D mode)
  if (n_dc > k4ASlots || n_dc < 1) return 0;
  if (K_pad > 65536) return 0;                                  // short-list entries are 16-bit code ids
  if ((reinterpret_cast<uintptr_t>(x.ptr) & 15) != 0) return 0;
  if (x.P >= (1ll << 31) || x.D >= (1ll << 31) || x.B >= (1ll << 31) || x.n_rows() >= (1ll << 31)) return 0;
  if (!encode_tiled_fn4()) return 0;
  if (x.sP == 1 && x.sD > 0 && (x.sD & 3) == 0 && (x.B == 1 || (x.sB > 0 && (x.sB & 3) == 0))) return 1;
  if (x.sD == 1 && x.sP > 0 && (x.sP & 3) == 0 && (x.B == 1 || x.sB == x.P * x.sP)) return 2;
  return 0;
}

int launch_assign_tc4(const Rows& x, const Tc4Args& a, int layout, cudaStream_t st) {
  int pairs = num_sms() / 2;
  if (a.n_ptiles * a.n_slices < pairs) pairs = a.n_ptiles * a.n_slices;
  if (pairs <= 0) return 0;
  if (layout == 3) {                                           // prepared samples: no tensor map
    CUtensorMap none;
    memset(&none, 0, sizeof(none));
    static size_t configured[kMaxDevices] = {0};
    if (int e = ensure_dynamic_smem(assign_tc4_kernel<2>, Tc4Smem::total, configured)) return e;
    cudaError_t le = launch_dependent(assign_tc4_kernel<2>, dim3(2 * pairs), dim3(k4Threads), (size_t)Tc4Smem::total, st, pdl_enabled(), none, a);
    if (le != cudaSuccess) return (int)le;
    VQSEG_LAUNCH_CHECK();
    return 0;
  }
  EncodeTiledFn4 enc = encode_tiled_fn4();
  if (!enc) return VQSEG_EUNSUPPORTED;
  CUtensorMap tmap;
  const cuuint32_t estr[3] = {1, 1, 1};
  CUresult rc;
  if (layout == 1) {
    // x as a 3-D tensor (pixel, channel, image); box = 128 pixels x 32 channels x 1 image; out-of-range reads as zero
    const cuuint64_t dims[3] = {(cuuint64_t)x.P, (cuuint64_t)x.D, (cuuint64_t)x.B};
    const cuuint64_t strides[2] = {(cuuint64_t)x.sD * 4, (cuuint64_t)(x.B > 1 ? x.sB : x.sD * x.D) * 4};
    const cuuint32_t box[3] = {(cuuint32_t)k4Rows, (cuuint32_t)k4BoxDims, 1};
    rc = enc(&tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(x.ptr), dims, strides, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  } else {
    // x as a 2-D tensor (dim, row); box = 32 dims (128 bytes) x 128 rows, 128-byte swizzle
    const cuuint64_t dims[2] = {(cuuint64_t)x.D, (cuuint64_t)x.n_rows()};
    const cuuint64_t strides[1] = {(cuuint64_t)x.sP * 4};
    const cuuint32_t box[2] = {(cuuint32_t)k4BoxDims, (cuuint32_t)k4Rows};
    rc = enc(&tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(x.ptr), dims, strides, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  }
  if (rc != CUDA_SUCCESS) return VQSEG_EUNSUPPORTED;
  if (layout == 1) {
    static size_t configured[kMaxDevices] = {0};
    if (int e = ensure_dynamic_smem(assign_tc4_kernel<0>, Tc4Smem::total, configured)) return e;
    cudaError_t le = launch_dependent(assign_tc4_kernel<0>, dim3(2 * pairs), dim3(k4Threads), (size_t)Tc4Smem::total, st, pdl_enabled(), tmap, a);
    if (le != cudaSuccess) return (int)le;
  } else {
    static size_t configured[kMaxDevices] = {0};
    if (int e = ensure_dynamic_smem(assign_tc4_kernel<1>, Tc4Smem::total, configured)) return e;
    cudaError_t le = launch_dependent(assign_tc4_kernel<1>, dim3(2 * pairs), dim3(k4Threads), (size_t)Tc4Smem::total, st, pdl_enabled(), tmap, a);
    if (le != cudaSuccess) return (int)le;
  }
  VQSEG_LAUNCH_CHECK();
  return 0;
}

}  // namespace vqseg
