// The short-list rule shared by the tensor-core filters (assign_tc*.cu) and split-D mode's shortlist_kernel: which
// rows a filter settles itself and what it hands to the rescoring pass (exact.cu) as a WorkRec.
//
// An epilogue warp owns one TMEM lane quarter and one half (128 columns) of every 256-code unit; lane = row.  Per row
// and tile it keeps a running minimum of the fp16 scores and the codes within the row's error bound (filter_slack) of
// it, at most kWorkCandCap of them.  At the end of a tile the upper half publishes {minimum, count | -1 overflow |
// -2 unbounded}, the lower half merges it with its own list and writes the row's index, or one work record.
#pragma once
#include "kernels.cuh"

namespace vqseg {

// The row-independent part of the error bound, read from the blob header.  Filters read it before their first
// accumulator wait: its DRAM latency must not sit between "accumulator ready" and "accumulator drained" of the first
// unit, which gates the next MMAs.
struct FilterBound {
  float scale, emax, de_max;
  bool defer_all;           // kBlobFlagDeferAll: the |e|^2 limbs are not representable, no row can be bounded
  __device__ __forceinline__ explicit FilterBound(const BlobHeader* hdr) {
    scale = hdr->scale;
    emax = sqrtf(hdr->max_enorm) * 1.0001f;
    de_max = sqrtf(__uint_as_float(hdr->max_de2_bits)) * 1.0001f;
    defer_all = (hdr->flags & kBlobFlagDeferAll) != 0u;
  }
  // The slack of a row with |x|^2 = x2 and |fp16(x) - x|^2 = dx2 (common.cuh filter_slack).  A row whose slack is not
  // below 3e38, or any row when defer_all is set, cannot be bounded: every code has to be rescored.
  __device__ __forceinline__ float slack(float x2, float dx2, int D, float t2) const {
    return filter_slack(sqrtf(x2) * 1.0001f, sqrtf(dx2) * 1.0001f, emax, de_max, scale, D, t2);
  }
};

__device__ __forceinline__ int work_rec_count(int nc, bool overflow) {
  return (overflow || nc == 0) ? kWorkCandCap + 1 : nc;       // > kWorkCandCap: the rescoring pass scans every code
}

// A row the filter decided: its code index and its count.
__device__ __forceinline__ void settle_row(const FilterOut& o, long long n, int k) {
  o.idx_out[n] = (long long)k + o.code_base;
  if (o.counts_out) atomicAdd(o.counts_out + k, 1ull);
}

// A row handed to the rescoring pass by a warp that owns the row (shortlist_kernel): lane l holds the l-th survivor.
__device__ __forceinline__ void defer_row_warp(const FilterOut& o, long long n, int cnt, bool overflow, int mine, int lane) {
  int slot = 0;
  if (lane == 0) slot = atomicAdd(o.work_count, 1);
  slot = __shfl_sync(0xffffffffu, slot, 0);
  WorkRec* rec = o.work + slot;
  if (lane == 0) { rec->row = (int)n; rec->cnt = work_rec_count(cnt, overflow); }
  if (lane < kWorkCandCap && lane < cnt && !overflow) rec->cand[lane] = mine;
}

// One row's short-list over one half of the columns, for one tile.  Slot: the code-id type of the shared-memory lists
// (unsigned short in the kernels limited to K_pad <= 65536, int in the others).
template <typename Slot>
struct ShortList {
  Slot* cand;               // this half's list
  const Slot* cand_hi;      // the upper half's list (read by the lower half when the halves meet)
  float m_run, slack;
  int cnt;
  bool overflow;            // the list ran over its capacity (cleared when a new minimum drops the list)
  bool bad;                 // the row cannot be bounded at all: every code is rescored

  // Where a row's two lists live in `lists` = [2 halves][rows][kWorkCandCap].  Built once per warp, before the tile
  // loop: the addresses stay out of the loops, as do D and t2, which start() takes from the kernel arguments at use.
  struct Slots {
    Slot* cand; const Slot* cand_hi;
    __device__ __forceinline__ Slots(Slot* lists, int rows, int half, int r) {
      cand = lists + (half * rows + r) * kWorkCandCap;
      cand_hi = lists + (rows + r) * kWorkCandCap;
    }
  };
  __device__ __forceinline__ explicit ShortList(const Slots& s) {
    cand = s.cand; cand_hi = s.cand_hi;
    m_run = __int_as_float(0x7f800000); slack = 0.f; cnt = 0; overflow = false; bad = false;
  }

  // before the first scan of the tile, once the row norms are in
  __device__ __forceinline__ void start(const FilterBound& b, float x2, float dx2, int D, float t2) {
    slack = b.slack(x2, dx2, D, t2);
    if (!(slack < 3.0e38f) || b.defer_all) bad = true;
  }

  // 32 consecutive scores (one tcgen05.ld) of codes col0 .. col0 + 31
  __device__ __forceinline__ void scan32(const uint32_t (&v)[32], int col0) {
    float m0 = __uint_as_float(v[0]), m1 = __uint_as_float(v[1]);
#pragma unroll
    for (int j = 0; j < 32; j += 4) {
      m0 = fminf(m0, fminf(__uint_as_float(v[j]), __uint_as_float(v[j + 2])));
      m1 = fminf(m1, fminf(__uint_as_float(v[j + 1]), __uint_as_float(v[j + 3])));
    }
    const float m_new = fminf(m_run, fminf(m0, m1));
    if (m_run > m_new + slack) { cnt = 0; overflow = false; }   // every earlier entry (listed or dropped) scored >= the old minimum
    m_run = m_new;
    const float thr = m_run + slack;
    // bit (31 - j) of ~mk <=> v[j] <= thr: one FADD + one funnel shift per score, four independent chains
    uint32_t mka = 0u, mkb = 0u, mkc = 0u, mkd = 0u;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      mka = __funnelshift_l(__float_as_uint(thr - __uint_as_float(v[j])), mka, 1);
      mkb = __funnelshift_l(__float_as_uint(thr - __uint_as_float(v[j + 8])), mkb, 1);
      mkc = __funnelshift_l(__float_as_uint(thr - __uint_as_float(v[j + 16])), mkc, 1);
      mkd = __funnelshift_l(__float_as_uint(thr - __uint_as_float(v[j + 24])), mkd, 1);
    }
    uint32_t mk = ~((mka << 24) | ((mkb & 0xffu) << 16) | ((mkc & 0xffu) << 8) | (mkd & 0xffu));
    if (overflow || bad) mk = 0u;
    while (mk) {
      const int j = __clz(mk);
      mk &= ~(0x80000000u >> j);
      if (cnt < kWorkCandCap) cand[cnt++] = (Slot)(col0 + j);
      else { overflow = true; mk = 0u; }
    }
  }

  // Tile done: the two column halves of each row meet through `xchg` between two named barriers of the lane quarter's
  // 64 threads (`bar_id`); the lower half settles row n or writes its work record.  The second barrier frees the lists
  // and `xchg` for the next tile.
  __device__ __forceinline__ void finish(int half, int bar_id, float2* xchg, bool in_range, long long n, const FilterOut& o) {
    if (half == 1) *xchg = make_float2(m_run, __int_as_float(bad ? -2 : (overflow ? -1 : cnt)));
    asm volatile("bar.sync %0, 64;" ::"r"(bar_id) : "memory");
    if (half == 0) resolve(*xchg, in_range, n, o);
    asm volatile("bar.sync %0, 64;" ::"r"(bar_id) : "memory");
  }

 private:
  __device__ __forceinline__ void resolve(const float2 hi, bool in_range, long long n, const FilterOut& o) {
    const int lane = threadIdx.x & 31;
    int cnt1 = __float_as_int(hi.y);
    const float m = fminf(m_run, hi.x);
    bool ov1 = cnt1 == -1;
    if (cnt1 == -2) bad = true;
    // a half whose own minimum is out of range contributes nothing (all its entries scored >= that minimum)
    if (m_run > m + slack) { cnt = 0; overflow = false; }
    if (hi.x > m + slack) { cnt1 = 0; ov1 = false; }
    if (cnt1 < 0) cnt1 = 0;
    overflow = overflow || ov1 || bad;
    const int tot = overflow ? 0 : cnt + cnt1;
    const int last = (!overflow && tot == 1) ? (cnt == 1 ? (int)cand[0] : (int)cand_hi[0]) : 0;
    const bool unique = !overflow && tot == 1 && !o.force_rescore && last < o.K;
    if (in_range && unique) settle_row(o, n, last);
    const bool flagged = in_range && !unique;
    const uint32_t fm = __ballot_sync(0xffffffffu, flagged);
    if (fm) {                                            // one atomic per warp on the work counter
      int base = 0;
      if (lane == 0) base = atomicAdd(o.work_count, __popc(fm));
      base = __shfl_sync(0xffffffffu, base, 0);
      if (flagged) {
        int* rec = reinterpret_cast<int*>(o.work + (base + __popc(fm & ((1u << lane) - 1))));
        int nc = 0;
        if (!overflow) {
          for (int e = 0; e < cnt; ++e) { int k = cand[e]; if (k < o.K && nc < kWorkCandCap) rec[4 + nc++] = k; else if (k < o.K) overflow = true; }
          for (int e = 0; e < cnt1; ++e) { int k = cand_hi[e]; if (k < o.K && nc < kWorkCandCap) rec[4 + nc++] = k; else if (k < o.K) overflow = true; }
        }
        rec[0] = (int)n;
        rec[1] = work_rec_count(nc, overflow);
      }
    }
  }
};

}  // namespace vqseg
