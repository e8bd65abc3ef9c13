// C ABI entry points for codebook preparation and nearest-code assignment (see include/vqseg.h).
#include "common.cuh"
#include "kernels.cuh"
#include "codebook_prep.cuh"
#include <string.h>

namespace vqseg {

__global__ void blob_init_kernel(BlobHeader* h, int K, int D, int K_pad, int D_pad, unsigned long long off_enorm,
                                 unsigned long long off_image, unsigned long long off_aug, unsigned long long off_hash,
                                 int ip) {
  h->off_aug = off_aug; h->aug_c = 1.f; h->flags = ip ? kBlobFlagIp : 0u; h->max_de2_bits = 0u;
  h->magic = kBlobMagic; h->K = K; h->D = D; h->K_pad = K_pad; h->D_pad = D_pad;
  h->scale = 1.f; h->max_enorm = 0.f; h->max_enorm_bits = 0u; h->max_abs_bits = 0u;
  h->off_enorm = off_enorm; h->off_image = off_image; h->off_hash = off_hash;
  h->stale = 0u; h->ticket = 0u; h->rebuilds = 0u;
}

int rvq_stage_gather(const float* r, int64_t B, int64_t P, int64_t D, int64_t sB, int64_t sP, int64_t sD,
                     const float* x, int64_t xB, int64_t xP, int64_t xD, const float* E, int64_t K, const int64_t* idx,
                     float* q, int64_t qB, int64_t qP, int64_t qD, float* r_next, float* acc,
                     float* layer_mse, float* layer_usage, const int64_t* counts, int layer, int n_layers, float weight,
                     float* loss_out, float* usage_out, int mode, void* ws, size_t ws_bytes, cudaStream_t st, int* ticket);

extern "C" int vqseg_internal_gather_ticket(const float* x, int64_t B, int64_t P, int64_t D, int64_t sB, int64_t sP, int64_t sD,
                                            const float* E, int64_t K, const int64_t* idx,
                                            float* q_out, int64_t qB, int64_t qP, int64_t qD, float* loss_out, int mode,
                                            void* ws, size_t ws_bytes, void* stream, int* ticket,
                                            const int64_t* counts, float* usage_out);

// Prologue of every assignment: ONE launch that
//   (a) zeroes what the kernels behind it accumulate into -- the work counter and the tickets, and for the fused
//       forward the per-code counts and the loss (three memset nodes cost 3 us more per step in a CUDA graph);
//   (b) guards the prepared-codebook cache: `weight.data.copy_()` / `.data.mul_()` (k-means init, mean-teacher
//       updates, vq_img.py:189) change the codebook without bumping the tensor version the host-side cache is keyed
//       on, so every warp re-hashes code rows and compares with the fingerprints the blob was built from; the last
//       block through (ticket) rebuilds the blob in place if any row differs.  One block, because a grid-wide
//       rebuild needs grid barriers; it is the rare path (a rebuild per weight change, ~50 us at K=512, D=256).
//   (c) checks that the blob was built for the metric of this call (inner-product blobs carry no |e|^2 limbs) and
//       rebuilds it for the other metric otherwise.
__global__ void __launch_bounds__(256) assign_prologue_kernel(unsigned long long* counts, int n_counts, float* loss, int* work4,
                                                              const float* __restrict__ E, int K, int D, unsigned char* blob,
                                                              int ip, float4* zero16 = nullptr, long long n_zero16 = 0) {
  pdl_trigger();     // the filter behind may become resident: it sets up and requests x while this kernel runs
  // (d) split-D mode of the streaming filter: its partial-score scratch starts from zero
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_zero16; i += (long long)gridDim.x * blockDim.x)
    zero16[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  if (blockIdx.x == 0) {
    for (int k = threadIdx.x; k < n_counts; k += blockDim.x) counts[k] = 0ull;
    if (threadIdx.x == 0) { if (loss) *loss = 0.f; work4[0] = 0; work4[1] = 0; work4[2] = 0; work4[3] = 0; }
  }
  if (!blob) return;
  BlobHeader* hdr = reinterpret_cast<BlobHeader*>(blob);
  const unsigned long long* hash = reinterpret_cast<const unsigned long long*>(blob + hdr->off_hash);
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  bool differ = ((hdr->flags & kBlobFlagIp) != 0u) != (ip != 0);
  for (int k = blockIdx.x * 8 + wib; k < K; k += gridDim.x * 8) {
    const unsigned long long h = row_hash_warp(E + (long long)k * D, D, lane);
    differ |= (h != hash[k]);
  }
  if (differ && lane == 0) atomicOr(&hdr->stale, 1u);
  __shared__ int s_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = (atomicAdd(&hdr->ticket, 1u) == gridDim.x - 1);
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  const bool stale = *reinterpret_cast<volatile uint32_t*>(&hdr->stale) != 0u;
  if (stale) {
    if (threadIdx.x == 0) { hdr->flags = ip ? kBlobFlagIp : 0u; hdr->max_de2_bits = 0u; hdr->max_enorm_bits = 0u; hdr->max_abs_bits = 0u; }
    __threadfence(); __syncthreads();
    prep_enorm(E, K, D, hdr->K_pad, reinterpret_cast<float*>(blob + hdr->off_enorm), hdr,
               reinterpret_cast<unsigned long long*>(blob + hdr->off_hash), wib, 8, lane);
    __threadfence(); __syncthreads();
    prep_pack(E, K, D, blob, threadIdx.x, blockDim.x);
    __threadfence(); __syncthreads();
    prep_rounding(E, K, D, blob, wib, 8, lane);
    __threadfence(); __syncthreads();
  }
  if (threadIdx.x == 0) { hdr->ticket = 0u; hdr->stale = 0u; if (stale) hdr->rebuilds += 1u; }
}

#ifdef VQSEG_DEV
long long* g_dev_trace = nullptr;            // developer build only (libvqseg_dev.so): clock stamps of the pipeline roles
#endif
static long long* dev_trace() {
#ifdef VQSEG_DEV
  return g_dev_trace;
#else
  return nullptr;
#endif
}
}  // namespace vqseg

using namespace vqseg;

// optional per-call profiling: the CALLER's four cudaEvent_t, recorded on `stream` around the filter ([0], [1]) and
// the rescoring kernel ([2], [3]).  No library state.
static void prof_record(void* const* ev, int i, cudaStream_t st) {
  if (!ev || !ev[i]) return;
  // inside a stream capture the record must be an EXTERNAL event node, or the event cannot be read after a replay
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(st, &cs) != cudaSuccess) { (void)cudaGetLastError(); cs = cudaStreamCaptureStatusNone; }
  const unsigned flags = cs == cudaStreamCaptureStatusActive ? cudaEventRecordExternal : cudaEventRecordDefault;
  if (cudaEventRecordWithFlags((cudaEvent_t)ev[i], st, flags) != cudaSuccess) (void)cudaGetLastError();   // never poison the launch checks
}

extern "C" {

int vqseg_version(void) { return VQSEG_VERSION; }

#ifdef VQSEG_DEV
void vqseg_debug_set_trace(void* dev_buf) { g_dev_trace = (long long*)dev_buf; }
#endif

const char* vqseg_error_string(int code) {
  switch (code) {
    case 0: return "ok";
    case VQSEG_EINVAL: return "vqseg: invalid argument";
    case VQSEG_EWORKSPACE: return "vqseg: workspace too small";
    case VQSEG_EUNSUPPORTED: return "vqseg: shape not supported by the requested algorithm";
    case VQSEG_EARCH: return "vqseg: device is not sm_100 (B200)";
  }
  if (code > 0) return cudaGetErrorString((cudaError_t)code);
  return "vqseg: unknown error";
}

static void blob_geometry(int64_t K, int64_t D, long long* K_pad, long long* D_pad, size_t* off_enorm, size_t* off_image,
                          size_t* total, size_t* off_aug = nullptr, size_t* off_hash = nullptr) {
  *K_pad = round_up(K, 256);
  *D_pad = round_up(D, kDChunk);
  *off_enorm = 1024;
  *off_image = *off_enorm + (size_t)round_up(2 * *K_pad * sizeof(float), 1024);
  size_t aug = *off_image + (size_t)(*K_pad / kCodeBlock) * (size_t)(*D_pad / kDChunk) * kTileBytes;
  if (off_aug) *off_aug = aug;
  size_t hash = aug + (size_t)(*K_pad / kCodeBlock) * 4096;
  if (off_hash) *off_hash = hash;
  *total = hash + (size_t)round_up(*K_pad * sizeof(unsigned long long), 1024);
}

size_t vqseg_codebook_blob_bytes(int64_t K, int64_t D) {
  if (K <= 0 || D <= 0) return 0;
  long long kp, dp; size_t oe, oi, tot;
  blob_geometry(K, D, &kp, &dp, &oe, &oi, &tot);
  return tot;
}

static int codebook_prepare(const float* E, int64_t K, int64_t D, void* blob, size_t blob_bytes, void* stream, int ip);

int vqseg_codebook_prepare_f32(const float* E, int64_t K, int64_t D, void* blob, size_t blob_bytes, void* stream) {
  return codebook_prepare(E, K, D, blob, blob_bytes, stream, 0);
}

int vqseg_codebook_prepare_ip_f32(const float* E, int64_t K, int64_t D, void* blob, size_t blob_bytes, void* stream) {
  return codebook_prepare(E, K, D, blob, blob_bytes, stream, 1);
}

static int codebook_prepare(const float* E, int64_t K, int64_t D, void* blob, size_t blob_bytes, void* stream, int ip) {
  if (!E || !blob || K <= 0 || D <= 0 || K >= (1ll << 30) || D >= (1ll << 20)) return VQSEG_EINVAL;
  long long kp, dp; size_t oe, oi, tot, oa, oh;
  blob_geometry(K, D, &kp, &dp, &oe, &oi, &tot, &oa, &oh);
  if (blob_bytes < tot) return VQSEG_EWORKSPACE;
  if ((reinterpret_cast<uintptr_t>(blob) & 1023) != 0) return VQSEG_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  unsigned char* b = (unsigned char*)blob;
  blob_init_kernel<<<1, 1, 0, st>>>((BlobHeader*)b, (int)K, (int)D, (int)kp, (int)dp, oe, oi, oa, oh, ip);
  VQSEG_LAUNCH_CHECK();
  int rc = launch_enorm(E, (int)K, (int)D, (int)kp, (float*)(b + oe), (BlobHeader*)b, (unsigned long long*)(b + oh), st);
  if (rc) return rc;
  return launch_pack(E, (int)K, (int)D, b, st);
}

// ---- prepared samples: [0, 256) header | norms float2[rows_padded] | image (1024-aligned) ------------------------------
static void samples_geometry(long long n_rows, long long D, long long* rows_padded, long long* D_pad, size_t* off_img, size_t* total) {
  *rows_padded = round_up(n_rows, 256);                 // whole PAIR tiles: the second CTA of the last pair finds zeros
  *D_pad = round_up(D, kDChunk);
  *off_img = (size_t)round_up(256 + *rows_padded * 8, 1024);
  *total = *off_img + (size_t)(*rows_padded) * (size_t)(*D_pad) * 2;
}
size_t vqseg_samples_blob_bytes(int64_t n_rows, int64_t D) {
  if (n_rows <= 0 || D <= 0) return 0;
  long long rp, dp; size_t oi, tot;
  samples_geometry(n_rows, D, &rp, &dp, &oi, &tot);
  return tot;
}
int vqseg_samples_prepare_f32(const float* x, int64_t B, int64_t P, int64_t D, int64_t sB, int64_t sP, int64_t sD,
                              void* blob, size_t blob_bytes, void* stream) {
  if (!x || !blob || B <= 0 || P <= 0 || D <= 0 || B * P >= (1ll << 31)) return VQSEG_EINVAL;
  long long rp, dp; size_t oi, tot;
  samples_geometry(B * P, D, &rp, &dp, &oi, &tot);
  if (blob_bytes < tot) return VQSEG_EWORKSPACE;
  if ((reinterpret_cast<uintptr_t>(blob) & 1023) != 0) return VQSEG_EINVAL;
  Rows xr{x, B, P, D, sB, sP, sD};
  return launch_samples_prepare(xr, rp, (int)dp, (unsigned char*)blob + oi, reinterpret_cast<float2*>((unsigned char*)blob + 256),
                                (cudaStream_t)stream);
}

// split-D mode (few rows, many dims) sums partial scores in an [n_rows][K_pad] fp32 scratch (+ 2 floats per row):
// only problems whose scratch stays below 32 MB are eligible
static size_t splitd_scratch_bytes(long long n_rows, long long K) {
  const long long kp = round_up(K, 256);
  const long long bytes = n_rows * kp * 4;
  if (n_rows <= 0 || bytes > (32ll << 20)) return 0;
  return (size_t)round_up(bytes, 256) + (size_t)round_up(n_rows * 8, 256);
}

constexpr size_t kOvfScratchBytes = (size_t)kOvfSplitCap * (sizeof(unsigned long long) + sizeof(int)) + 2048;   // 8 KiB
size_t vqseg_assign_workspace_bytes(int64_t n_rows, int64_t D, int64_t K, int algo) {
  (void)D; (void)algo;
  size_t b = 256 + kOvfScratchBytes;                                  // work counter + tickets, minima / tickets of split overflow rows
  b += (size_t)round_up(n_rows * (long long)sizeof(WorkRec), 256);    // one record per undecided row (worst case: all)
  b += (size_t)round_up(n_rows * (long long)sizeof(int), 256);        // rows whose short-list overflowed (worst case: all)
  b += (size_t)round_up(round_up(K, 256) * sizeof(float), 256);       // enorm when no blob is given
  b += splitd_scratch_bytes(n_rows, K);                               // split-D mode: partial scores + row norms
  return b;
}

static int assign_internal(const float* x, int64_t B, int64_t P, int64_t D, int64_t sB, int64_t sP, int64_t sD,
                           const float* E, int64_t K, void* blob,
                           int64_t* idx_out, int64_t* counts_out, uint64_t* best_key_out,
                           int64_t code_base, int kblock, int algo, void* ws, size_t ws_bytes, void* stream,
                           void* const* prof_events, float* zero_loss, bool zero_counts, const void* samples = nullptr) {
  if (!x || !E || B < 0 || P < 0 || D <= 0 || K <= 0) return VQSEG_EINVAL;
  if (!idx_out && !best_key_out) return VQSEG_EINVAL;
  const int ip = (algo & VQSEG_METRIC_IP) ? 1 : 0;
  algo &= ~VQSEG_METRIC_IP;
  if (ip && best_key_out) return VQSEG_EUNSUPPORTED;       // packed keys order distances, not signed inner products
  const long long n_rows = B * P;
  if (n_rows == 0) return 0;
  if (n_rows >= (1ll << 31) || K >= (1ll << 31) - 1 || D >= (1ll << 20)) return VQSEG_EUNSUPPORTED;
  if (!ws || ws_bytes < vqseg_assign_workspace_bytes(n_rows, D, K, algo)) return VQSEG_EWORKSPACE;
  int rc = check_arch();
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (kblock == 0) kblock = auto_kblock(ip ? D : D + 2);

  char* p = (char*)ws;
  int* work_count = (int*)p;   p += 256;                       // [0] undecided rows, [1] overflow rows, [2] gather ticket, [3] spare
  unsigned long long* ovf_keys = (unsigned long long*)p; int* ovf_tickets = (int*)(p + kOvfSplitCap * sizeof(unsigned long long));
  p += kOvfScratchBytes;
  WorkRec* work = (WorkRec*)p; p += round_up(n_rows * (long long)sizeof(WorkRec), 256);
  int* ovf_rows = (int*)p;     p += round_up(n_rows * (long long)sizeof(int), 256);
  float* enorm_ws = (float*)p; p += round_up(round_up(K, 256) * sizeof(float), 256);
  float* part_scores = splitd_scratch_bytes(n_rows, K) ? (float*)p : nullptr;
  float* part_norms = part_scores ? (float*)(p + round_up(n_rows * round_up(K, 256) * 4, 256)) : nullptr;

  bool use_tc = false;
  if (algo == VQSEG_ALGO_AUTO) use_tc = blob != nullptr && n_rows >= 64 && K >= 32;
  else if (algo == VQSEG_ALGO_EXACT) use_tc = false;
  else if (algo >= VQSEG_ALGO_TC && algo <= VQSEG_ALGO_TC_STREAM_PAIR) { if (!blob) return VQSEG_EINVAL; use_tc = true; }
  else return VQSEG_EINVAL;

  Rows xr{x, B, P, D, sB, sP, sD};
  long long kp = 0, dp = 0;
  size_t oe = 0, oi = 0, tot = 0, oa = 0;
  int n_cc = 0, n_dc = 0, kernel = 0, lay4 = 0, slice_dc = 0, n_slices = 1;
  const bool force = (best_key_out != nullptr || idx_out == nullptr);
  if (use_tc) {
    blob_geometry(K, D, &kp, &dp, &oe, &oi, &tot, &oa);
    n_cc = (int)(kp / 256); n_dc = (int)(dp / kDChunk);
    const bool can3 = tc3_supported(xr, n_cc, n_dc), can2 = tc2_supported(n_cc, n_dc);
    lay4 = tc4_layout(xr, kp, n_dc);
    const int pairs = num_sms() / 2;
    // codebook-resident kernels when the codebook fits two SMs; else the streaming pair kernel when its TMA layouts
    // apply and there is at least one pair tile per SM pair to amortise the A conversion; else the single-CTA kernel
    const long long ptiles4 = lay4 == 1 ? (B * ((P + 127) / 128) + 1) / 2 : ((n_rows + 127) / 128 + 1) / 2;
    kernel = can3 ? 3 : (can2 ? 2 : ((lay4 && 4 * ptiles4 >= pairs) ? 4 : 1));
    // ... unless the single-CTA kernel would leave most of the GPU idle (fewer pair tiles than a quarter of the SM
    // pairs; or more than 512 dims, which the pair kernel cannot hold as one tile): then the pair kernel in split-D
    // mode, when the score scratch is small.  Slices as LARGE as still give half the SM pairs an item: every slice
    // adds N x K_pad float atomics (measured: ~1.9 us per million + ~12 us fixed).
    if (kernel == 1 && part_scores && (algo == VQSEG_ALGO_AUTO || algo == VQSEG_ALGO_TC)) {
      for (int sd_ = 8; sd_ >= 2; --sd_) {
        if (n_dc % sd_ || n_dc / sd_ < 2) continue;
        const int lay = tc4_layout(xr, kp, sd_);
        if (!lay) break;
        const long long tiles = lay == 1 ? B * ((P + 127) / 128) : (n_rows + 127) / 128;
        if (2 * ((tiles + 1) / 2) * (n_dc / sd_) >= pairs || sd_ == 2) { slice_dc = sd_; n_slices = n_dc / sd_; lay4 = lay; kernel = 5; break; }
      }
    }
    // prepared samples (vqseg_samples_prepare_f32): the streaming pair kernel reads its A operand ready-made
    if (samples && n_dc <= 8 && kp <= 65536 && (algo == VQSEG_ALGO_AUTO || algo == VQSEG_ALGO_TC || algo == VQSEG_ALGO_TC_STREAM_PAIR)) {
      kernel = 4; lay4 = 3; n_slices = 1;
    }
    if (algo == VQSEG_ALGO_TC_STREAM) kernel = 1;
    if (algo == VQSEG_ALGO_TC_STREAM_PAIR) { if (!lay4) return VQSEG_EUNSUPPORTED; kernel = 4; }
    if (algo == VQSEG_ALGO_TC_PAIR) { if (!can2) return VQSEG_EUNSUPPORTED; kernel = 2; }
    if (algo == VQSEG_ALGO_TC_TMA) { if (!can3) return VQSEG_EUNSUPPORTED; kernel = 3; }
  }

  // prologue: zeroing + (when a prepared codebook is used) the guard that rebuilds a stale blob in place
  {
    int guard_blocks = use_tc ? (int)((K + 7) / 8 < 2 * num_sms() ? (K + 7) / 8 : 2 * num_sms()) : 1;
    long long n_zero16 = 0;
    if (kernel == 5) {
      n_zero16 = (long long)(splitd_scratch_bytes(n_rows, K) / 16);
      guard_blocks = 2 * num_sms();
    }
    assign_prologue_kernel<<<guard_blocks, 256, 0, st>>>(zero_counts ? (unsigned long long*)counts_out : nullptr,
                                                         zero_counts ? (int)K : 0, zero_loss, work_count, E, (int)K, (int)D,
                                                         use_tc ? (unsigned char*)blob : nullptr, ip,
                                                         reinterpret_cast<float4*>(part_scores), n_zero16);
    VQSEG_LAUNCH_CHECK();
  }

  const float* enorm = nullptr;
  if (use_tc) {
    enorm = (const float*)((const char*)blob + oe);
  } else {
    rc = launch_enorm(E, (int)K, (int)D, (int)K, enorm_ws, nullptr, nullptr, st);
    if (rc) return rc;
    enorm = enorm_ws;
  }

  ExactArgs ea;
  memset(&ea, 0, sizeof(ea));
  ea.x = xr; ea.E = E; ea.K = (int)K; ea.enorm = enorm; ea.kblock = kblock; ea.ip = ip;
  ea.idx_out = (long long*)idx_out; ea.counts_out = (unsigned long long*)counts_out;
  ea.key_out = (unsigned long long*)best_key_out; ea.code_base = code_base;
  if (!use_tc) return launch_exact(ea, n_rows, st);

  // (3 nb + 9) u: nb = K-blocks of the reference chain the exact scorer restates (filter_slack, common.cuh)
  const long long chain_len = ip ? D : D + 2;
  const long long kb_eff = (kblock <= 0 || kblock > chain_len) ? chain_len : kblock;
  const float slack_t2 = (float)(3 * ((chain_len + kb_eff - 1) / kb_eff) + 9) * 5.97e-8f;
  const FilterOut out{(int)K, (long long*)idx_out, (unsigned long long*)counts_out, code_base, force ? 1 : 0, slack_t2,
                      work, work_count};
  prof_record(prof_events, 0, st);
  if (kernel == 3) {
    Tc3Args t3;
    memset(&t3, 0, sizeof(t3));
    t3.B = B; t3.P = P; t3.D = D; t3.n_rows = n_rows; t3.blob = (const unsigned char*)blob;
    t3.tiles_per_image = (int)((P + 127) / 128);
    t3.n_tiles = (int)(B * t3.tiles_per_image);
    t3.n_ptiles = (t3.n_tiles + 1) / 2; t3.n_cc = n_cc; t3.n_dc = n_dc;
    t3.K_pad = (int)kp; t3.off_image = oi; t3.off_aug = oa; t3.off_enorm = oe;
    t3.out = out;
    t3.trace = dev_trace();
    rc = launch_assign_tc3(xr, t3, st);
  } else if (kernel == 4 || kernel == 5) {
    Tc4Args t4;
    memset(&t4, 0, sizeof(t4));
    t4.B = B; t4.P = P; t4.D = D; t4.n_rows = n_rows; t4.blob = (const unsigned char*)blob;
    if (lay4 == 1) { t4.tiles_per_image = (int)((P + 127) / 128); t4.n_tiles = (int)(B * t4.tiles_per_image); }
    else { t4.tiles_per_image = 0; t4.n_tiles = (int)((n_rows + 127) / 128); }
    if (lay4 == 3) {
      long long rp, dpp; size_t soi, stot;
      samples_geometry(n_rows, D, &rp, &dpp, &soi, &stot);
      t4.samp_img = (const unsigned char*)samples + soi;
      t4.samp_norms = reinterpret_cast<const float2*>((const unsigned char*)samples + 256);
    }
    t4.n_ptiles = (t4.n_tiles + 1) / 2; t4.n_cc = n_cc; t4.n_dc = n_dc;
    t4.n_slices = 1; t4.n_dc_total = n_dc;
    if (kernel == 5) {                              // split-D mode: partial scores into the scratch, short-lists afterwards
      t4.n_dc = slice_dc; t4.n_slices = n_slices;
      t4.part_scores = part_scores; t4.part_norms = part_norms;
    }
    t4.K_pad = (int)kp; t4.off_image = oi; t4.off_aug = oa; t4.off_enorm = oe;
    t4.out = out;
    t4.trace = dev_trace();
    rc = launch_assign_tc4(xr, t4, lay4, st);
    if (!rc && kernel == 5) {
      ShortlistArgs sl;
      memset(&sl, 0, sizeof(sl));
      sl.scores = part_scores; sl.norms = part_norms; sl.n_rows = n_rows; sl.K_pad = (int)kp; sl.D = (int)D;
      sl.blob = (const unsigned char*)blob;
      sl.out = out;
      rc = launch_shortlist(sl, st);
    }
  } else if (kernel == 2) {
    Tc2Args t2;
    memset(&t2, 0, sizeof(t2));
    t2.x = xr; t2.blob = (const unsigned char*)blob; t2.n_rows = n_rows;
    t2.n_ptiles = (int)((n_rows + 255) / 256); t2.n_cc = n_cc; t2.n_dc = n_dc;
    t2.K_pad = (int)kp; t2.off_image = oi; t2.off_aug = oa; t2.off_enorm = oe;
    t2.out = out;
    t2.trace = dev_trace();
    rc = launch_assign_tc2(t2, st);
  } else {
    TcArgs ta;
    memset(&ta, 0, sizeof(ta));
    ta.x = xr; ta.blob = (const unsigned char*)blob; ta.n_rows = n_rows;
    ta.n_tiles = (int)((n_rows + 127) / 128); ta.n_cc = n_cc; ta.n_dc = n_dc;
    ta.out = out;
    ta.trace = dev_trace();
    rc = launch_assign_tc(ta, st);
  }
  prof_record(prof_events, 1, st);
  if (rc) return rc;
  ea.work = work; ea.work_count = work_count;
  ea.ovf_keys = ovf_keys; ea.ovf_tickets = ovf_tickets;
  ea.ovf_rows = ovf_rows; ea.ovf_count = work_count + 1;               // ([1] is zeroed by the prologue with the counter)
  ea.trace = dev_trace() ? dev_trace() + 148 * 4 * 256 : nullptr;      // dev tool: 8 int64 after the filter's trace area
  prof_record(prof_events, 2, st);
  rc = launch_exact(ea, n_rows, st);
  prof_record(prof_events, 3, st);
  return rc;
}

int vqseg_assign_f32(const float* x, int64_t B, int64_t P, int64_t D, int64_t sB, int64_t sP, int64_t sD,
                     const float* E, int64_t K, void* blob,
                     int64_t* idx_out, int64_t* counts_out, uint64_t* best_key_out,
                     int64_t code_base, int kblock, int algo, void* ws, size_t ws_bytes, void* stream,
                     void* const* prof_events) {
  return assign_internal(x, B, P, D, sB, sP, sD, E, K, blob, idx_out, counts_out, best_key_out, code_base, kblock, algo,
                         ws, ws_bytes, stream, prof_events, nullptr, false);
}

int vqseg_assign_prepared_f32(const float* x, int64_t B, int64_t P, int64_t D, int64_t sB, int64_t sP, int64_t sD,
                              const void* samples, const float* E, int64_t K, void* blob,
                              int64_t* idx_out, int64_t* counts_out, int algo, void* ws, size_t ws_bytes, void* stream,
                              void* const* prof_events) {
  if (!samples || !blob) return VQSEG_EINVAL;
  return assign_internal(x, B, P, D, sB, sP, sD, E, K, blob, idx_out, counts_out, nullptr, 0, 0, algo,
                         ws, ws_bytes, stream, prof_events, nullptr, false, samples);
}

size_t vqseg_forward_workspace_bytes(int64_t n_rows, int64_t D, int64_t K) {
  return (size_t)round_up(vqseg_assign_workspace_bytes(n_rows, D, K, 0), 256) + vqseg_gather_workspace_bytes(n_rows, D);
}

int vqseg_vq_forward_f32(const float* x, int64_t B, int64_t P, int64_t D, int64_t sB, int64_t sP, int64_t sD,
                         const float* E, int64_t K, void* blob,
                         int64_t* idx_out, int64_t* counts_out, float* usage_out,
                         float* q_out, int64_t qB, int64_t qP, int64_t qD, float* loss_out,
                         int mode, int algo, int kblock, void* ws, size_t ws_bytes, void* stream,
                         void* const* prof_events) {
  if (!counts_out || K <= 0 || B < 0 || P < 0) return VQSEG_EINVAL;
  if (B * P != 0 && (!idx_out || !q_out)) return VQSEG_EINVAL;   // (empty tensors have null data pointers)
  if (algo & VQSEG_METRIC_IP) return VQSEG_EINVAL;               // the cosine codebook looks up l2norm(x) but gathers against x
  const size_t wa = (size_t)round_up(vqseg_assign_workspace_bytes(B * P, D, K, algo), 256);
  if (B * P != 0 && (!ws || ws_bytes < wa + vqseg_gather_workspace_bytes(B * P, D))) return VQSEG_EWORKSPACE;
  if (B * P == 0) {                                              // nothing to launch: outputs of an empty batch
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(counts_out, 0, (size_t)K * sizeof(int64_t), st);
    if (e == cudaSuccess && loss_out) e = cudaMemsetAsync(loss_out, 0, sizeof(float), st);
    if (e != cudaSuccess) return (int)e;
    return usage_out ? vqseg_code_usage(counts_out, K, usage_out, stream) : 0;     // no code is used: 100 %
  }
  int rc = assign_internal(x, B, P, D, sB, sP, sD, E, K, blob, idx_out, counts_out, nullptr, 0, kblock, algo, ws, wa, stream,
                           prof_events, loss_out, true);   // the prologue zeroes counts, loss, work counter and tickets
  if (rc) return rc;
  // the first 256 bytes of the assignment workspace hold {work counter, -, gather ticket, -}, all zeroed above; the
  // gather's last block reduces the loss and turns the (final) counts into the code usage
  return vqseg_internal_gather_ticket(x, B, P, D, sB, sP, sD, E, K, idx_out, q_out, qB, qP, qD, loss_out, mode,
                                      (char*)ws + wa, ws_bytes - wa, stream, (int*)ws + 2, counts_out, usage_out);
}

size_t vqseg_rvq_stage_workspace_bytes(int64_t n_rows, int64_t D, int64_t K) {
  return vqseg_forward_workspace_bytes(n_rows, D, K);
}

int vqseg_rvq_stage_f32(const float* r, int64_t B, int64_t P, int64_t D, int64_t sB, int64_t sP, int64_t sD,
                        const float* rn, int64_t nB, int64_t nP, int64_t nD,
                        const float* x, int64_t xB, int64_t xP, int64_t xD,
                        const float* E, int64_t K, void* blob,
                        int64_t* idx_out, int64_t* counts,
                        float* q, int64_t qB, int64_t qP, int64_t qD, float* r_next, float* acc,
                        float* layer_mse, float* layer_usage, float* loss_out, float* usage_out,
                        int layer, int n_layers, float weight, int mode, int algo,
                        void* ws, size_t ws_bytes, void* stream) {
  if (!counts || !layer_mse || !layer_usage || K <= 0 || B < 0 || P < 0 || D <= 0) return VQSEG_EINVAL;
  if (n_layers < 1 || layer < 0 || layer >= n_layers) return VQSEG_EINVAL;
  if (mode < VQSEG_MODE_EVAL || mode > VQSEG_MODE_EVAL_AMP_BF16) return VQSEG_EINVAL;     // (no VQSEG_MODE_ROTATE)
  if (algo & VQSEG_METRIC_IP) return VQSEG_EINVAL;               // the metric follows from `rn`
  const bool train = mode == VQSEG_MODE_TRAIN || mode == VQSEG_MODE_TRAIN_AMP || mode == VQSEG_MODE_TRAIN_AMP_BF16;
  const bool last = layer == n_layers - 1;
  cudaStream_t st = (cudaStream_t)stream;
  int64_t* counts_l = counts + (int64_t)layer * K;
  if (B * P == 0) {                                              // an empty batch: no code is used, no loss
    cudaError_t e = cudaMemsetAsync(counts_l, 0, (size_t)K * sizeof(int64_t), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(layer_mse + layer, 0, sizeof(float), st);
    if (e == cudaSuccess && last && loss_out) e = cudaMemsetAsync(loss_out, 0, sizeof(float), st);
    if (e != cudaSuccess) return (int)e;
    int rc = vqseg_code_usage(counts_l, K, layer_usage + layer, stream);
    if (!rc && last && usage_out) rc = vqseg_code_usage(counts, (int64_t)n_layers * K, usage_out, stream);
    return rc;
  }
  if (!r || !idx_out || !q || (!last && !r_next) || (train && last && !x)) return VQSEG_EINVAL;
  const size_t wa = (size_t)round_up(vqseg_assign_workspace_bytes(B * P, D, K, algo), 256);
  if (!ws || ws_bytes < wa + vqseg_gather_workspace_bytes(B * P, D)) return VQSEG_EWORKSPACE;
  // the lookup: r itself (Euclidean) or its normalised rows (inner product); the prologue zeroes this layer's counts and
  // m_l, the work counter and the tickets
  const float* lx = rn ? rn : r;
  int rc = assign_internal(lx, B, P, D, rn ? nB : sB, rn ? nP : sP, rn ? nD : sD, E, K, blob, idx_out, counts_l, nullptr, 0, 0,
                           algo | (rn ? VQSEG_METRIC_IP : 0), ws, wa, stream, nullptr, layer_mse + layer, true);
  if (rc) return rc;
  return rvq_stage_gather(r, B, P, D, sB, sP, sD, x, xB, xP, xD, E, K, idx_out, q, qB, qP, qD, last ? nullptr : r_next, acc,
                          layer_mse, layer_usage, counts, layer, n_layers, weight, loss_out, usage_out, mode,
                          (char*)ws + wa, ws_bytes - wa, st, (int*)ws + 2);
}

}  // extern "C"
