// Launch interface between the C ABI layer (api.cu) and the kernel translation units: argument structs and
// launchers, defined once here.
#pragma once
#include "common.cuh"

namespace vqseg {

// One undecided row handed from a tensor-core filter to the rescoring pass: the row id and the short-list of codes
// whose approximate score lies within the proven error bound of the row minimum.  cnt > kWorkCandCap means "the
// short-list overflowed: score every code".  48 bytes, 16-byte aligned: one coalesced fetch per record.
constexpr int kWorkCandCap = 8;
struct alignas(16) WorkRec { int row; int cnt; int pad0; int pad1; int cand[kWorkCandCap]; };

// What a tensor-core filter writes (filter_epilogue.cuh): the index and count of every row it decides, one WorkRec per
// row it leaves to the rescoring pass.
struct FilterOut {
  int K;
  long long* idx_out; unsigned long long* counts_out; long long code_base;
  int force_rescore;              // 1 -> every row goes to the exact pass (sharded mode needs exact distances)
  float slack_t2;                 // coefficient of the |x|^2-magnitude roundings in the filter's slack (common.cuh filter_slack)
  WorkRec* work; int* work_count;
};

// ---- exact.cu: exact fp32 scorer (brute force over all codes, or the rescoring pass over the filter's short-lists)
constexpr int kOvfSplitCap = 512;   // overflow rows up to which each row's codes are split over several blocks
struct ExactArgs {
  Rows x;
  const float* E; int K;
  const float* enorm;
  int kblock;
  int ip;               // 1: inner-product mode (cosine codebook): argmax <x, e>, plain D-term chain (exact_chain.cuh)
  // candidate mode (null -> all rows x all codes)
  const WorkRec* work; const int* work_count;         // undecided rows + device counter
  int* ovf_rows; int* ovf_count;                      // rows whose short-list overflowed: deferred to overflow_rows_kernel
  unsigned long long* ovf_keys; int* ovf_tickets;     // kOvfSplitCap packed (score, code) minima + block tickets: few overflow rows are split over blocks
  long long* idx_out; unsigned long long* counts_out; unsigned long long* key_out; long long code_base;
  long long* trace;     // dev tool: [0] min start ns, [1] max end ns
};
int launch_enorm(const float* E, int K, int D, int K_pad, float* enorm, BlobHeader* hdr, unsigned long long* hash,
                 cudaStream_t st);
int launch_exact(const ExactArgs& a, long long max_work, cudaStream_t st);

// ---- assign_tc.cu: single-CTA streaming tcgen05 filter, and the codebook packer
struct TcArgs {
  Rows x;
  const unsigned char* blob;      // prepared codebook
  long long n_rows;
  int n_tiles, n_cc, n_dc;        // tiles of 128 rows, code chunks of 256, dim chunks of 64
  FilterOut out;
  long long* trace;               // optional (dev tool): [cta][role][256] clock64 stamps
};
int launch_pack(const float* E, int K, int D, unsigned char* blob, cudaStream_t st);
int launch_assign_tc(const TcArgs& a, cudaStream_t st);

// ---- assign_tc2.cu: CTA-pair, codebook-resident tcgen05 filter
struct Tc2Args {
  Rows x;
  const unsigned char* blob;
  long long n_rows;
  int n_ptiles, n_cc, n_dc;       // pair tiles of 256 rows, code chunks of 256, dim chunks of 64
  int K_pad;
  unsigned long long off_image, off_aug, off_enorm;
  FilterOut out;
  long long* trace;
};
bool tc2_supported(int n_cc, int n_dc);
int launch_assign_tc2(const Tc2Args& a, cudaStream_t st);

// ---- assign_tc3.cu: TMA-fed CTA-pair, codebook-resident tcgen05 filter (pixel-contiguous / NCHW inputs)
struct Tc3Args {
  long long B, P, D;              // logical (B, P, D) view; memory is pixel-contiguous (sP == 1)
  long long n_rows;
  const unsigned char* blob;
  int n_tiles, tiles_per_image;   // tiles of 128 pixels, never straddling an image
  int n_ptiles, n_cc, n_dc;       // pair tiles (two tiles), code chunks of 256, dim chunks of 64
  int K_pad;
  unsigned long long off_image, off_aug, off_enorm;
  FilterOut out;
  long long* trace;
};
bool tc3_supported(const Rows& x, int n_cc, int n_dc);
int launch_assign_tc3(const Rows& x, const Tc3Args& a, cudaStream_t st);

// ---- assign_tc4.cu: TMA-fed CTA-pair STREAMING tcgen05 filter (any K <= 65536, D_pad <= 512; NCHW maps or packed rows)
struct Tc4Args {
  long long B, P, D;              // logical (B, P, D) view
  long long n_rows;
  const unsigned char* blob;
  int n_tiles, tiles_per_image;   // tiles of 128 rows (NCHW: 128 pixels of one image)
  int n_ptiles, n_cc, n_dc;       // pair tiles (two tiles), code chunks of 256, dim chunks of 64 PER WORK ITEM
  int n_slices, n_dc_total;       // split-D mode: dim slices per row (1 = off), dim chunks of the whole row
  float* part_scores;             // split-D mode: [n_rows][K_pad] partial scores, zeroed by the prologue (else null)
  float* part_norms;              //               [n_rows][2] {|x|^2, |fp16(x) - x|^2}
  const unsigned char* samp_img;  // MODE 2 (prepared samples): fp16 A tiles [row tile][dim chunk] x 16 KiB
  const float2* samp_norms;       //                            [padded rows] {|x|^2, |fp16(x) - x|^2}
  int K_pad;
  unsigned long long off_image, off_aug, off_enorm;
  FilterOut out;
  long long* trace;
};
// split-D mode's second step: per row the short-list over the summed scores (same rule as the filters' epilogues)
struct ShortlistArgs {
  const float* scores; const float* norms; long long n_rows; int K_pad, D;
  const unsigned char* blob;
  FilterOut out;
};
int launch_shortlist(const ShortlistArgs& a, cudaStream_t st);
int tc4_layout(const Rows& x, long long K_pad, int n_dc);   // 0: unsupported, 1: NCHW maps, 2: packed rows
int launch_assign_tc4(const Rows& x, const Tc4Args& a, int layout, cudaStream_t st);    // layout 3: prepared samples
int launch_samples_prepare(const Rows& x, long long rows_padded, int D_pad, unsigned char* img, float2* norms, cudaStream_t st);

// MKL's sgemm K-blocking as probed on the reference CPU path (DESIGN.md §parity): one chain up to
// 384 terms, two halves up to 768, 384-blocks beyond.  0: one chain.
inline int auto_kblock(long long L) {
  if (L <= 384) return 0;
  if (L <= 768) return (int)((L + 1) / 2);
  return 384;
}

// ---- seghead_tiled.cu: register-tiled map and backward of the segmentation head (any K, any D)
// kb: the chain's K-block, normalised (0 < kb <= D + 2, or <= D for cosine).  Outputs as in vqseg_seghead_map_f32;
// counts must be zeroed by the caller.
int launch_seghead_map_tiled(const Rows& x, const float* E, int K, bool cosine, int kb, float* dist, long long oB,
                             long long oP, long long oK, long long* idx, unsigned long long* counts, float* score,
                             cudaStream_t st);
// Deterministic backward (VQSEG_SEGHEAD_DETERMINISTIC): the pixels are cut into slices of consecutive rows whose
// number is a function of (n_rows, K, D) alone; each slice's (K, D) partial is stored with plain stores and the
// partials are added in a fixed order (launch_seghead_slice_sum).  The split uses a B200's SM count as a constant, and
// the partials never take more than kSegheadDetPartialBytes.
constexpr long long kSegheadDetSms = 148;
constexpr long long kSegheadDetPartialBytes = 32ll << 20;
inline long long seghead_det_max_slices(long long K, long long D) {
  const long long m = kSegheadDetPartialBytes / (K * D * (long long)sizeof(float));
  return m > 1 ? m : 1;
}
size_t seghead_bwd_tiled_workspace_bytes(long long n_rows, int K, int D, bool det);
// gE must be zeroed by the caller unless det (every element is stored); cosine: dist is the similarity map
int launch_seghead_map_bwd_tiled(const Rows& x, const float* E, int K, bool cosine, const float* g, const float* dist,
                                 long long oB, long long oP, long long oK, const float* score, const RowsOut& gx,
                                 float* gE, bool det, void* ws, cudaStream_t st);
// out[i] = the sum of part[z n + i] over z < S, in an order that depends on S alone
int launch_seghead_slice_sum(const float* part, long long n, int S, float* out, cudaStream_t st);

}  // namespace vqseg
