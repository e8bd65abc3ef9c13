/*
 * vqseg.h -- C ABI of libvqseg.so: the B200 (sm_100a) kernels behind VQ_SEG's VectorQuantizer.
 *
 * The reference (chaeyeongyun/VQ_SEG) is pure PyTorch: its "FFI" for this path is the torch ops
 * that vector_quantizer/vq_img.py calls.  Each entry point below names the reference call sites
 * it replaces (file:line relative to the reference root).  Host code binds these with ctypes
 * (vq_seg_b200/_native.py); INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Conventions
 *   - every function returns 0 on success, a positive cudaError_t, or a negative VQSEG_E* code;
 *   - all pointers are DEVICE pointers unless the name ends in _host; tensors stay owned by the
 *     caller, the kernels borrow them;
 *   - no cudaMalloc, no host synchronisation and no global state inside (except per-device caches of
 *     cudaFuncSetAttribute calls / the SM count); everything is enqueued on `stream`;
 *   - latent vectors are described as a logical (B, P, D) array with ELEMENT strides
 *     (sB, sP, sD): NCHW feature maps are (B, H*W, C) with sB=C*H*W, sP=1, sD=H*W (the view made
 *     by `rearrange(x,'b c h w -> b (h w) c')`, vq_img.py:232); packed row-major samples are
 *     B=1, sP=D, sD=1.  Row id n = b*P + p.
 *   - indices and counts are int64 (what torch.argmin / torch.bincount return).
 */
#ifndef VQSEG_H_
#define VQSEG_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VQSEG_VERSION 100            /* 0.1.0 */

#define VQSEG_EINVAL    (-1)         /* bad argument (null pointer, negative size, ...)          */
#define VQSEG_EWORKSPACE (-2)        /* workspace too small: call vqseg_*_workspace_bytes        */
#define VQSEG_EUNSUPPORTED (-3)      /* shape not supported by the requested algorithm           */
#define VQSEG_EARCH     (-4)         /* device is not sm_100 (Blackwell B200)                    */

/* assign algorithms */
#define VQSEG_ALGO_AUTO   0          /* tensor-core filter + exact rescoring when the shape allows */
#define VQSEG_ALGO_EXACT  1          /* exact fp32 scorer on every (row, code) pair                */
#define VQSEG_ALGO_TC     2          /* tcgen05 fp16 filter + exact fp32 rescoring; the kernel is chosen by shape/layout: */
#define VQSEG_ALGO_TC_STREAM 3       /*   ... the single-CTA streaming kernel (any K, D, strides)                  */
#define VQSEG_ALGO_TC_PAIR   4       /*   ... the codebook-resident CTA-pair kernel, x through registers (any strides) */
#define VQSEG_ALGO_TC_TMA    5       /*   ... the codebook-resident CTA-pair kernel, x by TMA tensor loads (NCHW maps) */
#define VQSEG_ALGO_TC_STREAM_PAIR 6  /*   ... the streaming CTA-pair kernel, x by TMA (NCHW maps or packed rows, D <= 512) */
#define VQSEG_METRIC_IP  0x100       /* OR into `algo`: inner-product metric -- idx = FIRST argmax_k <x_n, e_k> with the fp32 sum
                                        evaluated as ATen's CPU matmul does (the cosine codebook, vq_img.py:104-107, and
                                        `samples @ means^T` + argmax in kmeans, :37-41); x and E are used as given
                                        (callers normalise them with vqseg_l2norm_f32); best_key_out is not supported */
/* 3-6 force one kernel (VQSEG_EUNSUPPORTED if the shape does not fit it): the tests cover all three on the same inputs */

/* gather modes */
#define VQSEG_MODE_EVAL        0     /* quantize = E[idx]                          (vq_img.py:170)     */
#define VQSEG_MODE_TRAIN       1     /* quantize = x + (E[idx] - x), two roundings (vq_img.py:236)     */
#define VQSEG_MODE_TRAIN_AMP   2     /* as TRAIN with E[idx] rounded through fp16 (autocast matmul)    */
#define VQSEG_MODE_EVAL_AMP    3
#define VQSEG_MODE_TRAIN_AMP_BF16 4  /* as TRAIN with E[idx] rounded through bf16 (autocast matmul)   */
#define VQSEG_MODE_EVAL_AMP_BF16  5  /* as EVAL with E[idx] rounded through bf16 (autocast matmul)    */
#define VQSEG_MODE_ROTATE   0x10     /* OR into a TRAIN mode (opt-in rotation trick, see vqseg_rotate_bwd_f32): quantize = c,
                                        the code after the mode's rounding (bit-equal to the matching EVAL mode's output),
                                        not x + (c - x); the loss is mean((c - x)^2) with the same fixed reduction.  With an
                                        EVAL mode, or with any other unknown bit, the gather returns VQSEG_EINVAL. */

int         vqseg_version(void);
const char* vqseg_error_string(int code);

/* ---- codebook preparation --------------------------------------------------------------------
 * Replaces the per-call `x2.pow(2).sum(-1)` + operand building inside torch.cdist
 * (ATen _euclidean_dist, reached from vq_img.py:167 and :39).  Fills an opaque, reusable
 * "prepared codebook" blob: fp32 |e_k|^2 in torch's CPU summation order, max |e_k|, the fp16
 * power-of-two prescale and the fp16 (-2 * s * E) image laid out as tcgen05 SWIZZLE_128B K-major
 * shared-memory tiles (one bulk copy per pipeline stage), and a 64-bit fingerprint per code row.
 * The blob is a CACHE: every assignment that is given one first compares those fingerprints with
 * the live E (its prologue kernel) and rebuilds the blob in place when a row changed, so results
 * never depend on a stale image (weight.data.copy_ / mul_ do not bump torch's version counter).
 * Re-running this after a known change just moves the rebuild off the assignment's critical path. */
size_t vqseg_codebook_blob_bytes(int64_t K, int64_t D);
int    vqseg_codebook_prepare_f32(const float* E, int64_t K, int64_t D,
                                  void* blob, size_t blob_bytes, void* stream);
/* the same for VQSEG_METRIC_IP assignments (no |e_k|^2 term in the score).  A blob built for the other metric is
 * detected and rebuilt by the assignment's prologue, like a stale one. */
int    vqseg_codebook_prepare_ip_f32(const float* E, int64_t K, int64_t D,
                                     void* blob, size_t blob_bytes, void* stream);

/* ---- nearest-code assignment -----------------------------------------------------------------
 * Replaces `torch.cdist(flatten_x, weight, p=2)` + `torch.argmin(distance, -1)`
 * (vq_img.py:167-168) and `-torch.cdist` + `torch.argmax` inside kmeans (vq_img.py:39-41).
 * The N x K distance matrix is never written.  idx_out[n] is the FIRST index minimising
 * sqrt(max(|x|^2 - 2 x.e + |e|^2, 0)) evaluated in fp32 exactly as ATen's CPU path does
 * (one FMA chain over the D+2 augmented terms, split every `kblock` terms; see DESIGN.md).
 * counts_out (nullable, K int64, must be zeroed by the caller) receives bincount(idx)
 * (vq_img.py:173 / batched_bincount :22-27).  code_base is added to every written index and
 * best_key_out (nullable, N uint64) receives (float_bits(dist) << 32 | global index) for the
 * codebook-sharded mode (min-reduce across ranks keeps the lowest index on ties).            */
size_t vqseg_assign_workspace_bytes(int64_t n_rows, int64_t D, int64_t K, int algo);
int    vqseg_assign_f32(const float* x, int64_t B, int64_t P, int64_t D,
                        int64_t sB, int64_t sP, int64_t sD,
                        const float* E, int64_t K, void* blob,
                        int64_t* idx_out, int64_t* counts_out, uint64_t* best_key_out,
                        int64_t code_base, int kblock, int algo,
                        void* ws, size_t ws_bytes, void* stream, void* const* prof_events);
/* prof_events (nullable): four cudaEvent_t owned by the caller; the call records [0],[1] around the tensor-core
 * filter kernel and [2],[3] around the rescoring kernel on `stream` (bench.py's roofline line).  No library state. */

/* ---- prepared samples: for inputs that are assigned many times (the Lloyd iterations of kmeans, vq_img.py:35-61:
 * the same samples against new means every iteration).  vqseg_samples_prepare_f32 builds, once, the fp16 operand of
 * the tensor-core filter as ready-made shared-memory tiles plus the per-row norms of its error bound;
 * vqseg_assign_prepared_f32 is vqseg_assign_f32 whose filter streams those tiles instead of converting x on the fly
 * (D <= 512, K <= 65536; otherwise `samples` is ignored).  x is still needed: the exact rescoring reads it.  Results are
 * identical to vqseg_assign_f32's.  The blob must be 1024-byte aligned. */
size_t vqseg_samples_blob_bytes(int64_t n_rows, int64_t D);
int    vqseg_samples_prepare_f32(const float* x, int64_t B, int64_t P, int64_t D,
                                 int64_t sB, int64_t sP, int64_t sD,
                                 void* samples_blob, size_t blob_bytes, void* stream);
int    vqseg_assign_prepared_f32(const float* x, int64_t B, int64_t P, int64_t D,
                                 int64_t sB, int64_t sP, int64_t sD,
                                 const void* samples_blob, const float* E, int64_t K, void* blob,
                                 int64_t* idx_out, int64_t* counts_out, int algo,
                                 void* ws, size_t ws_bytes, void* stream, void* const* prof_events);

/* unpack the keys of the sharded mode after the cross-rank min: idx = key & 0xffffffff           */
int    vqseg_unpack_keys(const uint64_t* keys, int64_t n, int64_t* idx_out, float* dist_out,
                         int64_t* counts_out, int64_t K, void* stream);

/* ---- gather + straight-through estimator + commitment loss -----------------------------------
 * Replaces `F.one_hot(idx) -> matmul(onehot.float(), weight)` (vq_img.py:169-170), the STE
 * `x + (quantize - x).detach()` (:236) and `F.mse_loss(quantize.detach(), x)` (:239).
 * q_out has the same (B,P,D) logical shape with its own strides.  loss_out (nullable) receives
 * sum((q_ste - x)^2) / (B*P*D) as ONE fp32 (deterministic two-stage reduction through `ws`).   */
size_t vqseg_gather_workspace_bytes(int64_t n_rows, int64_t D);
int    vqseg_gather_ste_f32(const float* x, int64_t B, int64_t P, int64_t D,
                            int64_t sB, int64_t sP, int64_t sD,
                            const float* E, int64_t K, const int64_t* idx,
                            float* q_out, int64_t qB, int64_t qP, int64_t qD,
                            float* loss_out, int mode, void* ws, size_t ws_bytes, void* stream);

/* ---- the whole VectorQuantizer.forward in one call -------------------------------------------------
 * vqseg_assign_f32 + vqseg_code_usage + vqseg_gather_ste_f32 enqueued back to back (vq_img.py:228-244 minus the
 * k-means hook): one host call instead of three, for latency-bound feature-map sizes.  counts_out is zeroed
 * here.  ws must hold vqseg_forward_workspace_bytes.  Outputs as in the individual calls.               */
size_t vqseg_forward_workspace_bytes(int64_t n_rows, int64_t D, int64_t K);
int    vqseg_vq_forward_f32(const float* x, int64_t B, int64_t P, int64_t D,
                            int64_t sB, int64_t sP, int64_t sD,
                            const float* E, int64_t K, void* blob,
                            int64_t* idx_out, int64_t* counts_out, float* usage_out,
                            float* q_out, int64_t qB, int64_t qP, int64_t qD, float* loss_out,
                            int mode, int algo, int kblock, void* ws, size_t ws_bytes, void* stream,
                            void* const* prof_events);

/* ---- backward of the training forward w.r.t. x -----------------------------------------------
 * Replaces autograd through vq_img.py:236-240:  gx = g_q + coef * (x - q_ste), with
 * coef = g_loss * commitment_weight * 2 / numel read from device memory (coef_dev, 1 float) so no
 * host sync is needed.  g_q may be null (treated as zeros), coef_dev may be null (no loss term).
 * q_ste may be null (treated as zeros: gx = fma(coef, x, g_q), the residual VQ backward with x = A below).
 * All tensors share the (B,P,D) logical shape; each has its own strides.                        */
int    vqseg_ste_bwd_f32(const float* g_q, int64_t gB, int64_t gP, int64_t gD,
                         const float* x, int64_t sB, int64_t sP, int64_t sD,
                         const float* q_ste, int64_t qB, int64_t qP, int64_t qD,
                         const float* coef_dev, float coef_scale,
                         float* gx, int64_t oB, int64_t oP, int64_t oD,
                         int64_t B, int64_t P, int64_t D, void* stream);

/* ---- backward w.r.t. x of the rotation trick: OPT-IN EXTENSION, no reference counterpart ------------------------
 * Fifty et al., "Restructuring Vector Quantization with the Rotation Trick" (arXiv 2410.06424, §4.2); rotation_trick of
 * lucidrains/vector-quantize-pytorch.  For the forward of a TRAIN | VQSEG_MODE_ROTATE gather (quantize = c), per row n
 * with x the input, c the SAVED quantize (never E[idx]: the EMA update may have rewritten E in between), g = g_q (0 when
 * g_q is null) and lam = coef_scale * (*coef_dev) (0 when coef_dev is null; the convention of vqseg_ste_bwd_f32):
 *   gx = s (g - 2 (w.g) w + 2 (q^.g) u) + lam (x - c), the gradient of quantize = s (x - 2 (x.w) w + 2 (x.u) q^) with
 *        u = x/|x|, q^ = c/|c|, w = (u + q^)/|u + q^| and s = |c|/|x| held constant (the forward value is c), plus the
 *        commitment term.  Evaluated in fp32 with IEEE sqrt and division and no contraction as:
 *   xx, cc, xc, xg, cg = row sums of x*x, c*c, x*c, x*g, c*g, each as eight chains a_l = fl(fl(p_d) + a_l) over
 *        d = l, l+8, l+16, ... ascending (l = 0..7), then ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
 *   xx == 0 or cc == 0:  alpha = 1, beta = lam, gamma = -lam  (the straight-through gradient);
 *   else  nx = sqrt(xx), nc = sqrt(cc), s = nc / nx, rho = (xc / nx) / nc, a = xg / nx, b = cg / nc, t = 1 + rho,
 *         h = (a + b) / t if t > 0 else 0  (antipodal rows: the reflection),
 *         alpha = s, beta = ((s (2b - h)) / nx) + lam, gamma = (-((s h) / nc)) - lam;
 *   gx_d = ((alpha g_d) + (beta x_d)) + (gamma c_d).
 * The order of the sums does not depend on the strides: gx is bit-identical for every layout of the inputs and the
 * output and from run to run (no atomics).  Arguments as in vqseg_ste_bwd_f32; x and q are required.  16 N D bytes. */
int    vqseg_rotate_bwd_f32(const float* g_q, int64_t gB, int64_t gP, int64_t gD,
                            const float* x, int64_t sB, int64_t sP, int64_t sD,
                            const float* q, int64_t qB, int64_t qP, int64_t qD,
                            const float* coef_dev, float coef_scale,
                            float* gx, int64_t oB, int64_t oP, int64_t oD,
                            int64_t B, int64_t P, int64_t D, void* stream);

/* ---- residual vector quantization: OPT-IN EXTENSION, no reference counterpart (ResidualVQ of
 * lucidrains/vector-quantize-pytorch; parity unpinned).  Q codebooks E_0 .. E_{Q-1} quantize x, then what the first left,
 * and so on.  x is the (B, P, D) view of the input map, w the commitment weight, rho the gather mode's rounding of the
 * code (identity in TRAIN / EVAL, fp16 or bf16 round-to-nearest-even in the AMP modes); every operation is a separately
 * rounded fp32 operation with no contraction, and "ascending" means l = 0, 1, ...:
 *   r_0 = x;  for l = 0 .. Q-1:
 *     idx_l = the lookup of r_l: Euclidean, the first argmin of vqseg_assign_f32; cosine (rn given), the first argmax of
 *             l2norm(r_l) . E_l^T (vqseg_assign_f32 with VQSEG_METRIC_IP on rn = l2norm(r_l), E_l already renormalised)
 *     c_l   = rho(E_l[idx_l]);   S = c_l if l == 0 else S + c_l
 *     TRAIN:           q_l = r_l + (c_l - r_l);  m_l = mean((q_l - r_l)^2) with the gather's fixed two-stage reduction
 *                      (exactly what vqseg_gather_ste_f32 writes as the loss for input r_l in the TRAIN mode)
 *     TRAIN, acc given: A = (r_l - q_l) if l == 0 else A + (r_l - q_l)
 *     r_{l+1} = r_l - c_l   (l < Q-1, in TRAIN and EVAL alike)
 * Outputs: quantize = x + (S - x) in TRAIN, S in EVAL; loss L = w m_0, then L + w m_l ascending (TRAIN); code usage
 * 100 * (Z / (Q K)) with Z the number of (l, k) pairs with a zero count.  With Q = 1 all of it is vqseg_vq_forward_f32.
 * Gradient (TRAIN): gx = fma(coef, A, g) with coef = g_loss * w * 2 / (B P D): vqseg_ste_bwd_f32 with x = A and a null
 * q_ste.  The codebooks get none; in EVAL gE_l[k] = sum over the rows with idx_l = k of g (vqseg_gather_bwd_codebook_f32).
 *
 * vqseg_rvq_stage_f32 runs stage `layer` of `n_layers` with ONE host call: the launches of vqseg_vq_forward_f32 (the
 * assignment prologue and guard, filter, rescoring and overflow rows) with the stage kernel in the gather's place.  Per
 * element the stage kernel reads r_l, the code and S (layer > 0) and writes S (into q), r_{l+1} (into r_next, unless this
 * is the last stage), A (into acc, TRAIN only, nullable) and, in the last TRAIN stage, quantize over S from x (any strides).
 * q, r_next and acc share q's strides; (D*P, 1, P) (NCHW memory order) lets the next stage take the same TMA-fed filter as
 * stage 0.  r: r_l (any strides); rn: null (Euclidean) or l2norm(r_l) for the cosine lookup; idx_out: B*P int64 (this
 * layer's slice); counts: (Q, K) int64, row `layer` zeroed and filled here; layer_mse / layer_usage: (Q,) floats, entry
 * `layer` written (m_l, 0 in EVAL; and the layer's usage); the last stage also writes loss_out (nullable: L from
 * layer_mse[0 .. Q-1] and w in TRAIN, 0 in EVAL) and usage_out (nullable) from all Q count rows.  mode: a TRAIN or EVAL mode without
 * VQSEG_MODE_ROTATE; algo: as vqseg_assign_f32 without VQSEG_METRIC_IP.  ws: vqseg_rvq_stage_workspace_bytes.
 * An empty batch (B * P == 0) writes zero counts, m_l = 0, usage 100 and loss 0.                                       */
size_t vqseg_rvq_stage_workspace_bytes(int64_t n_rows, int64_t D, int64_t K);
int    vqseg_rvq_stage_f32(const float* r, int64_t B, int64_t P, int64_t D, int64_t sB, int64_t sP, int64_t sD,
                           const float* rn, int64_t nB, int64_t nP, int64_t nD,
                           const float* x, int64_t xB, int64_t xP, int64_t xD,
                           const float* E, int64_t K, void* blob,
                           int64_t* idx_out, int64_t* counts,
                           float* q, int64_t qB, int64_t qP, int64_t qD, float* r_next, float* acc,
                           float* layer_mse, float* layer_usage, float* loss_out, float* usage_out,
                           int layer, int n_layers, float weight, int mode, int algo,
                           void* ws, size_t ws_bytes, void* stream);
/* S of the restatement above from a (Q, B, P) int64 index array (idx[l][b][p]) and the Q codebooks packed (Q, K, D), in one
 * launch for any Q >= 1: out = c_0, then out + c_l ascending, with the rounding of `mode` (an EVAL mode).  Bit-equal to
 * the EVAL quantize of the same indices.  out: (B, P, D) with any strides.                                              */
int    vqseg_rvq_decode_f32(const int64_t* idx, int64_t Q, int64_t B, int64_t P, const float* E, int64_t K, int64_t D,
                            float* out, int64_t oB, int64_t oP, int64_t oD, int mode, void* stream);

/* gradient of the eval-mode gather w.r.t. the codebook: gE[idx[n], :] += g_q[n, :]              */
int    vqseg_gather_bwd_codebook_f32(const float* g_q, int64_t B, int64_t P, int64_t D,
                                     int64_t gB, int64_t gP, int64_t gD,
                                     const int64_t* idx, float* gE, int64_t K, void* stream);

/* ---- per-code statistics (k-means update) ----------------------------------------------------
 * Replaces batched_bincount (vq_img.py:22-27, :42) and
 * `new_means.scatter_add_(1, repeat(buckets,'h n -> h n d'), samples)` (:47-51).
 * counts (K int64) and sums (K*D fp32) must be zeroed by the caller (so ranks can accumulate).
 * deterministic=1: per-code sums are accumulated in ascending row order, one fp32 chain per
 * (code, d) -- the order of the reference's sequential CPU scatter_add_ -- via a stable counting
 * sort (clusters far above the mean size stream through a shared-memory ring, one warp per 32 dims);
 * deterministic=0: order not fixed -- vector fp32 reductions per row, or, for packed inputs of
 * 2^18 rows and more with K <= 1536, the same sort followed by register sums over windows of 64 sorted rows
 * (one reduction per code met: no hot addresses whatever the clustering).  The workspace size
 * depends on the mode: always ask vqseg_code_stats_workspace_bytes.                              */
size_t vqseg_code_stats_workspace_bytes(int64_t n_rows, int64_t D, int64_t K, int deterministic);
int    vqseg_code_stats_f32(const float* x, int64_t B, int64_t P, int64_t D,
                            int64_t sB, int64_t sP, int64_t sD,
                            const int64_t* idx, int64_t K,
                            int64_t* counts, float* sums, int deterministic,
                            void* ws, size_t ws_bytes, void* stream);

/* means = where(counts == 0, means, sums / max(counts,1))  [then l2norm rows if cosine]
 * (vq_img.py:44-45, :53-61).                                                                    */
int    vqseg_kmeans_finalize_f32(const float* sums, const int64_t* counts, float* means_inout,
                                 int64_t K, int64_t D, int cosine, void* stream);

/* code_usage = 100 * (#counts == 0) / K as one fp32 (vq_img.py:174-175)                         */
int    vqseg_code_usage(const int64_t* counts, int64_t K, float* usage_out, void* stream);

/* rows[i,:] = x[row_ids[i], :] packed (K,D): initial k-means means (sample_vectors, vq_img.py:10-17) */
int    vqseg_gather_rows_f32(const float* x, int64_t B, int64_t P, int64_t D,
                             int64_t sB, int64_t sP, int64_t sD,
                             const int64_t* row_ids, int64_t n_ids, float* out, void* stream);

/* ---- cosine codebook helper (CosinesimCodebook, vq_img.py:93-107) -----------------------------
 * out[b,p,:] = x[b,p,:] / max(|x[b,p,:]|, 1e-12)  (F.normalize, vq_img.py:7-8,:97,:100,:54) in ATen's CPU
 * arithmetic, whose summation order follows the stride of x's reduced dim alone: sD == 1 (code rows, k-means means,
 * channels-last maps and their batch slices, 1 x 1 maps) is reduced in ATen's vectorised last-dim order, any other sD
 * (the 'b c h w -> b (h w) c' view of an NCHW map the cosine codebook normalises) as one sequential chain; IEEE sqrt
 * and division.  Any sB and sP are accepted.  `out` may have any strides, which do not change the order (same layout
 * as x keeps NCHW maps TMA-loadable), and may alias x when the strides are equal (in-place renormalisation of the
 * codebook, vq_img.py:100).
 * The lookup itself (einsum + argmax, vq_img.py:104-107) is vqseg_assign_f32 with VQSEG_METRIC_IP. */
int    vqseg_l2norm_f32(const float* x, int64_t B, int64_t P, int64_t D,
                        int64_t sB, int64_t sP, int64_t sD,
                        float* out, int64_t oB, int64_t oP, int64_t oD, void* stream);

/* ---- EMA codebook update: OPT-IN EXTENSION, no reference counterpart (the reference stores `decay` and `eps`,
 * vq_img.py:150-151,199-200, and never reads them: there is no EMA, so parity is unpinned). Standard VQ-VAE
 * equations: cluster_size <- decay*cluster_size + (1-decay)*counts; embed_avg <- decay*embed_avg + (1-decay)*sums;
 * n = sum(cluster_size); cs = (cluster_size + eps) / (n + K*eps) * n; weight = embed_avg / cs.  counts / sums come
 * from vqseg_code_stats_f32 (all-reduced by the caller in data-parallel training).  ws: >= 4 bytes.           */
int    vqseg_ema_update_f32(const int64_t* counts, const float* sums, float* cluster_size_inout,
                            float* embed_avg_inout, float* weight_out, int64_t K, int64_t D,
                            float decay, float eps, void* ws, void* stream);

/* ---- EMA update with dead-code expiry: OPT-IN EXTENSION, no reference counterpart (threshold_ema_dead_code of
 * lucidrains/vector-quantize-pytorch, expire_codes_ / replace).  The update of vqseg_ema_update_f32, then:
 *   expired[k] = cluster_size[k] < threshold   (strict fp32 comparison on the cluster sizes just updated);
 *   the r-th expired code in ascending k takes candidate row r of cand_rows ((K, D) packed: the caller samples K rows
 *   of the batch, randperm(N)[:K] for N >= K, else randint(0, N, (K,))):
 *     weight[k] = cand[r];  embed_avg[k] = cand[r] * reset (one fp32 multiply);  cluster_size[k] = reset.
 * The Laplace smoothing uses n = sum(cluster_size) BEFORE any reset, so every output of a code that did not expire is
 * bit-identical to what vqseg_ema_update_f32 writes on the same inputs.  expired_out (nullable) = int64 [last, total]:
 * [0] is set to this call's expired count and [1] accumulates it (counters for logging without a host sync).
 * Two launches like vqseg_ema_update_f32; K < 2^26.  ws: >= vqseg_ema_expire_workspace_bytes(K).              */
size_t vqseg_ema_expire_workspace_bytes(int64_t K);
int    vqseg_ema_update_expire_f32(const int64_t* counts, const float* sums, float* cluster_size_inout,
                                   float* embed_avg_inout, float* weight_out, int64_t K, int64_t D,
                                   float decay, float eps, float threshold, float reset,
                                   const float* cand_rows, int64_t* expired_out,
                                   void* ws, size_t ws_bytes, void* stream);

/* ---- VQ segmentation head (models/modules/vq_segmentation_head.py) ------------------------------
 * The head classifies every decoder pixel by its distance to K class prototypes and RETURNS the distance map.
 * dist_out[b, p, k] (element strides oB, oP, oK; (K*P, 1, P) gives the (B, K, H, W) score layout directly):
 *   cosine == 0: torch.cdist(flatten_x, weight, p=2)  (EuclideanSegHead.forward :167), bit-equal to ATen's CPU
 *                result; idx = first argmin (:168);
 *   cosine != 0: einsum('n d, e d -> n e') over rows the caller has already l2-normalised
 *                (CosinesimSegHead.forward :104); idx = first argmax (:107).
 * counts_out (nullable) = bincount(idx, K) (:174), zeroed by the call.  K <= 32, D <= 382, K*D small enough for
 * shared memory (VQSEG_EUNSUPPORTED otherwise: a segmentation head has K = classes, D = last decoder width;
 * vqseg_seghead_map_f32 below takes any K and D).
 * score_out (nullable, Euclidean only, same strides): the wrapper's class scores softmax_k(1 - d_k / sum_j d_j)
 * (VQSegmentationHead.forward :243-247 with the default nn.Softmax2d activation), written by the same kernel.  */
int    vqseg_dist_map_f32(const float* x, int64_t B, int64_t P, int64_t D, int64_t sB, int64_t sP, int64_t sD,
                          const float* E, int64_t K, int cosine,
                          float* dist_out, int64_t oB, int64_t oP, int64_t oK,
                          int64_t* idx_out, int64_t* counts_out, float* score_out, void* stream);
/* backward of the Euclidean map (autograd of torch.cdist, p=2): with w = g / dist (0 where dist == 0),
 *   gx[n,:] = sum_k w[n,k] (x[n,:] - e_k),   gE[k,:] = sum_n w[n,k] (e_k - x[n,:])   (gE zeroed by the call;
 * accumulated with fp32 atomics: sums within 1e-5 relative, not bit-reproducible -- vqseg_seghead_map_bwd_f32 with
 * VQSEG_SEGHEAD_DETERMINISTIC is).  g and dist share strides.
 * score (nullable): when given, g is the gradient w.r.t. score_out and the kernel first chains it through the
 * softmax and the 1 - d / sum(d) normalisation.                                                           */
int    vqseg_dist_map_bwd_f32(const float* g, const float* dist, int64_t oB, int64_t oP, int64_t oK,
                              const float* x, int64_t B, int64_t P, int64_t D, int64_t sB, int64_t sP, int64_t sD,
                              const float* E, int64_t K,
                              float* gx_out, int64_t gxB, int64_t gxP, int64_t gxD, float* gE_out,
                              const float* score, void* stream);
/* backward of the cosine similarity map (vqseg_dist_map_f32 with cosine = 1 on x, i.e. CosinesimSegHead's
 * l2norm(x) @ weight^T, models/modules/vq_segmentation_head.py:97-104): g is the gradient w.r.t. the map (same strides
 * as the map); gx = (gxn - xn <xn, gxn>) / |x| with gxn = g @ E, gE[k,:] = sum_n g[n,k] xn[n,:].  Same limits as the map. */
int    vqseg_sim_map_bwd_f32(const float* g, int64_t oB, int64_t oP, int64_t oK,
                             const float* x, int64_t B, int64_t P, int64_t D,
                             int64_t sB, int64_t sP, int64_t sD,
                             const float* E, int64_t K,
                             float* gx_out, int64_t gxB, int64_t gxP, int64_t gxD, float* gE_out, void* stream);

/* ---- segmentation head for any class count and feature width ------------------------------------------------
 * Same outputs and arithmetic as vqseg_dist_map_f32 (Euclidean map bit-equal to ATen's CPU cdist, including MKL's
 * K-blocked chains for D + 2 > 384; cosine: the plain D-term chain over caller-normalised rows) for any K >= 1 and
 * D >= 1.  `algo` picks the kernel:
 *   VQSEG_SEGHEAD_AUTO  : the per-pixel kernels of vqseg_dist_map_f32 where their limits hold (K <= 32, D <= 382:
 *                         the reference's 3-class heads), the tiled kernels otherwise;
 *   VQSEG_SEGHEAD_PIXEL : the per-pixel kernels only (VQSEG_EUNSUPPORTED beyond their limits);
 *   VQSEG_SEGHEAD_TILED : the register-tiled kernels (a block owns 128 pixels x 64 classes per step).
 * No workspace; counts_out (nullable) is zeroed by the call.                                                      */
#define VQSEG_SEGHEAD_AUTO   0
#define VQSEG_SEGHEAD_PIXEL  1
#define VQSEG_SEGHEAD_TILED  2
/* OR into the algo of vqseg_seghead_map_bwd_workspace_bytes / vqseg_seghead_map_bwd_f32 (the forward map rejects it
 * with VQSEG_EINVAL): gE bit-reproducible, see below.                                                             */
#define VQSEG_SEGHEAD_DETERMINISTIC 0x100
int    vqseg_seghead_map_f32(const float* x, int64_t B, int64_t P, int64_t D, int64_t sB, int64_t sP, int64_t sD,
                             const float* E, int64_t K, int cosine,
                             float* dist_out, int64_t oB, int64_t oP, int64_t oK,
                             int64_t* idx_out, int64_t* counts_out, float* score_out, int algo, void* stream);
/* backward of vqseg_seghead_map_f32.  cosine == 0: as vqseg_dist_map_bwd_f32 (`map` = the distance map, `score`
 * nullable); cosine != 0: as vqseg_sim_map_bwd_f32 with `map` = the similarity map (the tiled kernels take
 * <xn, gxn> = sum_k g_k sim_k from it), score must be null.  g and map share strides.  ws must hold
 * vqseg_seghead_map_bwd_workspace_bytes of the same algo.
 * Without VQSEG_SEGHEAD_DETERMINISTIC gE_out is zeroed by the call and accumulated with fp32 atomics (not
 * bit-reproducible); the workspace is 16 bytes per pixel for the tiled kernels, 0 for the per-pixel ones.
 * With it gE_out is a function of the inputs and of (B*P, K, D) alone -- not of the device's SM count, the launch
 * timing, the stream or the strides of x: the pixels are cut into S slices of consecutive rows (S from the shape
 * only), each slice's (K, D) partial sum is formed in the kernel's fixed in-block order with tiles in ascending
 * order and stored with plain stores, and the S partials are added in a fixed order that depends on S alone.  The
 * workspace adds S*K*D*4 bytes of partials when S > 1, never more than 32 MiB.  gx is the same either way. */
size_t vqseg_seghead_map_bwd_workspace_bytes(int64_t n_rows, int64_t D, int64_t K, int algo);
int    vqseg_seghead_map_bwd_f32(const float* g, const float* map, int64_t oB, int64_t oP, int64_t oK,
                                 const float* x, int64_t B, int64_t P, int64_t D, int64_t sB, int64_t sP, int64_t sD,
                                 const float* E, int64_t K, int cosine, const float* score,
                                 float* gx_out, int64_t gxB, int64_t gxP, int64_t gxD, float* gE_out,
                                 int algo, void* ws, size_t ws_bytes, void* stream);


#ifdef __cplusplus
}
#endif
#endif  /* VQSEG_H_ */
