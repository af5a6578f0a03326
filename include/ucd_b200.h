/*
 * ucd_b200 C ABI - the drop-in boundary of the B200-native UCD distillation-loss hot path.
 *
 * One shared library (ucd_b200/libucd_b200.so), extern "C", plain pointers and sizes, no torch
 * types.  Every pointer is a DEVICE pointer unless its name ends in _host.  Every entry point is
 * asynchronous on `stream` (a cudaStream_t passed as void*), allocates nothing, keeps no global
 * mutable state, reads no environment variable and returns 0 on success or a negative UCD_E* code; the message of the last
 * failure on the calling thread is available from ucd_last_error().
 *
 * Each function names the reference interface (file:line under the UCD tree) it replaces.  The
 * reference is pure PyTorch, so "FFI binding" means the ctypes stubs in ucd_b200/_lib.py; see
 * INTEGRATION.md for the loss-module classes a maintainer swaps in.
 */
#ifndef UCD_B200_H
#define UCD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define UCD_OK 0
#define UCD_EINVAL (-1)   /* bad argument (shape, alignment, unsupported size) */
#define UCD_ECUDA (-2)    /* a CUDA runtime call or launch failed */
#define UCD_ENOSUP (-3)   /* valid request this build does not support yet */

#define UCD_REDUCTION_NONE 0
#define UCD_REDUCTION_MEAN 1
#define UCD_REDUCTION_SUM 2

/* feature width of the pixel embeddings (DeepLab head_channels, segmentation_module.py:23,45) */
#define UCD_FEAT_DIM 256
/* rows/columns of one similarity tile; all packed buffers are padded to multiples of it */
#define UCD_TILE 128

int ucd_version(void);
const char* ucd_last_error(void);
/* 1 if a CUDA device of compute capability 10.x is present, else 0 (no other side effects). */
int ucd_device_ok(void);

/* ------------------------------------------------------------------------------------------
 * Unbiased cross-entropy   (utils/loss.py:96-109, alt utils/loss_new.py:89-115)
 *   x      [B,C,HW] fp32 logits (NCHW contiguous)       y [B,HW] int64 labels, REMAPPED IN PLACE
 *   loss_px[B,HW]   per-pixel loss (reduction 'none')   (y < old_cl -> 0, like loss.py:104-105)
 *   lse_all [B,HW]  saved log-sum-exp over all channels;  lse_old [B,HW] or NULL: the same over the first old_cl
 *                   channels (not needed by the backward: at label-0 pixels loss_px IS lse_all - lse_old)
 *   stats  float[2] : {sum of per-pixel losses, number of non-ignored pixels} (for mean/sum)
 * ---------------------------------------------------------------------------------------- */
int ucd_unce_fwd(const float* x, int64_t* y, float* loss_px, float* lse_all, float* lse_old,
                 float* stats /*or NULL*/, float* scratch /*float[ucd_reduce_scratch_floats()], with stats*/,
                 int B, int C, int old_cl, int64_t HW, int ignore_index, void* stream);
/* dx = g * dloss/dx.  g_px [B,HW] per-pixel upstream gradient or NULL; then the upstream gradient is
 * the scalar *g_scalar (device) times g_mul (host), and with mean_over_valid != 0 it is additionally
 * divided by stats[1] (nll_loss 'mean' semantics).
 * accumulate != 0 (here and in ucd_unkd_bwd / ucd_kd_bwd): dx += ... instead of dx = ...: the second of two losses
 * on the same logits (train.py:116 and :133 both consume `outputs`) adds into the first one's gradient buffer, which
 * replaces autograd's own full-size add kernel (8 % of the drop-in step) by one extra read of dx. */
int ucd_unce_bwd(const float* x, const int64_t* y, const float* lse_all,
                 const float* bkg_gap /* [B,HW]: lse_all - lse_old at the pixels whose (remapped) label is 0, anything
                 elsewhere - the forward's loss_px as it stands */,
                 const float* g_px, const float* g_scalar, float g_mul, const float* stats,
                 int mean_over_valid, float* dx, int accumulate, int B, int C, int old_cl, int64_t HW,
                 int ignore_index, void* stream);

/* ------------------------------------------------------------------------------------------
 * Unbiased knowledge distillation   (utils/loss.py:148-184, alt utils/loss_new.py:216-263)
 *   x [B,C,HW] new logits, t [B,C_old,HW] old logits, mask [B,HW] fp32 or NULL
 *   out_px [B,HW] = -loss_px (written when non-NULL; what reduction 'none' returns)
 *   stats float[1] = sum over pixels of loss_px (caller negates / divides)
 *   lse3 [3,B,HW] saved {lse_all(x), lse_bkg(x over {0} U new), lse(alpha t)}
 *   scratch: float[ucd_reduce_scratch_floats()]
 * ---------------------------------------------------------------------------------------- */
int ucd_unkd_fwd(const float* x, const float* t, const float* mask, float alpha, float* out_px,
                 float* stats, float* lse3, float* scratch, int B, int C, int C_old, int64_t HW,
                 void* stream);
/* dx = upstream * d(-loss_px)/dx; upstream is g_px[B,HW] if non-NULL else *g_scalar * g_mul. */
int ucd_unkd_bwd(const float* x, const float* t, const float* mask, float alpha, const float* lse3,
                 const float* g_px, const float* g_scalar, float g_mul, float* dx, int accumulate, int B, int C,
                 int C_old, int64_t HW, void* stream);
size_t ucd_reduce_scratch_floats(void);

/* Sibling distillation losses on the same kernels (SURVEY.md section 8(f) row N3).  `variant`:
 *   0  UnbiasedKnowledgeDistillationLoss (identical to ucd_unkd_*)
 *   1  KnowledgeDistillationLoss (utils/loss.py:112-136): log-softmax over the first C_old of the C channels of x,
 *      mean over those channels; dx of the remaining channels is written as 0
 *   2  MaskKnowledgeDistillationLoss (utils/loss.py:218-256): variant 0 with the pixel weight [mask == 0] */
int ucd_kd_fwd(const float* x, const float* t, const float* mask, float alpha, float* out_px, float* stats,
               float* lse3, float* scratch, int B, int C, int C_old, int64_t HW, int variant, float stats_scale,
               void* stream);   /* stats[0] = stats_scale * sum_px(weight * l_px): -1/(B*HW) gives the 'mean' loss */
int ucd_kd_bwd(const float* x, const float* t, const float* mask, float alpha, const float* lse3,
               const float* g_px, const float* g_scalar, float g_mul, float* dx, int accumulate, int B, int C,
               int C_old, int64_t HW, int variant, void* stream);
/* UNCE + UNKD backward in one pass (both losses consume the same `outputs`, train.py:116 and :133): the sum of what
 * ucd_unce_bwd and ucd_kd_bwd (variant 0 or 2) would write, with x read and dx written once.  lse_all is the statistic
 * both forwards saved (log-sum-exp over all C channels); lse3 as saved by ucd_kd_fwd. */
int ucd_unce_unkd_bwd(const float* x, const int64_t* y, const float* lse_all, const float* bkg_gap /* as above */,
                      const float* ce_g_px, const float* ce_g_scalar, float ce_g_mul, const float* ce_stats,
                      int mean_over_valid, int old_cl, int ignore_index, const float* t, const float* mask,
                      float alpha, const float* lse3, const float* kd_g_px, const float* kd_g_scalar, float kd_g_mul,
                      int kd_variant, float* dx, int accumulate, int B, int C, int C_old, int64_t HW, void* stream);
/* MaskCrossEntropy's pixel weight (utils/loss.py:207-211): mask[b,p] = 1 if argmax_c t_old[b,c,p] == 0 or
 * labels[b,p] > old_cl, else 0.  t_old [B,C_old,HW] fp32, labels [B,HW] int64, mask [B,HW] fp32. */
int ucd_bkg_mask(const float* t_old, const int64_t* labels, float* mask, int B, int C_old, int64_t HW,
                 int old_cl, void* stream);

/* ------------------------------------------------------------------------------------------
 * Bilinear logit upsample, align_corners=False   (segmentation_module.py:133)
 *   in [N,h,w] -> out [N,H,W]   (N = B*C planes), and its adjoint.
 * ---------------------------------------------------------------------------------------- */
int ucd_upsample_bilinear_fwd(const float* in, float* out, int64_t planes, int h, int w, int H, int W,
                              void* stream);
int ucd_upsample_bilinear_bwd(const float* gout, float* gin, int64_t planes, int h, int w, int H, int W,
                              void* stream);
/* Prediction without the upsample: pred [B,H,W] int64 = argmax over the C channels of what
 * ucd_upsample_bilinear_fwd writes for lr [B,C,h,w], bit for bit (same taps and operation order; ties go to the first
 * maximal channel, NaN counts as maximal, as torch.argmax).  No [B,C,H,W] tensor is written or allocated.
 * Upsampling only (H >= h, W >= w): downscaling returns UCD_EINVAL. */
int ucd_upsample_argmax(const float* lr, int64_t* pred, int B, int C, int h, int w, int H, int W, void* stream);
/* ucd_unce_unkd_bwd contracted with the adjoint of ucd_upsample_bilinear_fwd: when the logits x [B,C,H,W] are the
 * upsample of lr [B,C,h,w], d_lr [B,C,h,w] = upsample_adjoint(dx) of the dx ucd_unce_unkd_bwd would write (same
 * per-element values; the adjoint's summation order is its own).  dx is never written: one read-only pass over x, t,
 * the labels and the saved planes.  d_lr is overwritten.  Deterministic.  UCD_ENOSUP (nothing launched) unless the
 * shape is one the sweep-form adjoint takes: H % h == 0, W % w == 0, (W / w) % 8 == 0, W / 4 a multiple of 32 and
 * <= 256, all planes 16-byte aligned; the caller then takes ucd_unce_unkd_bwd + ucd_upsample_bilinear_bwd. */
int ucd_unce_unkd_bwd_lowres(const float* x, const int64_t* y, const float* lse_all, const float* bkg_gap,
                             const float* ce_g_px, const float* ce_g_scalar, float ce_g_mul, const float* ce_stats,
                             int mean_over_valid, int old_cl, int ignore_index, const float* t, const float* mask,
                             float alpha, const float* lse3, const float* kd_g_px, const float* kd_g_scalar,
                             float kd_g_mul, int kd_variant, float* d_lr, int B, int C, int C_old, int h, int w, int H,
                             int W, void* stream);

/* ------------------------------------------------------------------------------------------
 * N1 (SURVEY.md 8f), opt-in: upsample + unbiased CE + unbiased KD fused, from the LOW-RES logits
 *   (segmentation_module.py:133 + utils/loss.py:96-109 + :148-184 as wired by train.py:116,133).
 * The full-resolution logits are never written.  lr [B,C,h,w], lr_old [B,C_old,h,w], labels [B,H,W] int64
 * (remapped in place like ucd_unce_fwd).  Outputs: sums[3] = {sum_px ce_px, #non-ignored pixels, sum_px kd_px}
 * with kd_px = -loss_px of the KD term, and (need_grad) the unit gradients g_ce, g_kd [B,C,h,w] of the two sums
 * with respect to lr.  Cross-block sums go through `workspace` (ucd_seg_fused_workspace_floats floats, 16 B
 * aligned) and are added in a fixed order: bit-identical from run to run.
 * CE-only form (the base step, which has no old model): C_old == 0 with lr_old == NULL.  Only the CE is computed,
 * g_kd is neither read nor written (may be NULL) and alpha is ignored; sums[2] = 0.  With old_cl == 0 the CE is plain
 * cross-entropy (the background branch needs old_cl > 0).
 * ---------------------------------------------------------------------------------------- */
size_t ucd_seg_fused_workspace_floats(int B, int C, int C_old, int h, int w, int H, int W);
int ucd_seg_fused_fwd(const float* lr, const float* lr_old, int64_t* labels, float* g_ce, float* g_kd,
                      float* sums, float* workspace, size_t workspace_floats, int B, int C, int C_old, int h,
                      int w, int H, int W, int old_cl, int ignore_index, float alpha, int need_grad,
                      void* stream);

/* ------------------------------------------------------------------------------------------
 * Contrastive prep   (utils/loss.py:258-395 v2 branch == utils/utils.py:256-397)
 *
 * Step 1 (labels):  per low-res pixel p=(b,y,x): label_n = clamp(trunc(bilinear(labels))),
 *   pseudo = argmax_c l_po, mix, flags (bit0 anchor, bit1 pseudo, bit2 GT-new), the rank of the pixel
 *   among anchors / pseudos, and counts = {N_a, N_o, min_new, n_px}.
 * Step 2 (pack): writes, for anchors (from f_n) and pseudo pixels (from f_o):
 *   - unit-norm fp32 rows  anchor_f32 [N_a,256], contrast_f32 [N_a+N_o,256] (reference order b,y,x)
 *   - bf16 tiles for the tensor-core sweeps: feat_tiles [T][32][128][8], prob_tiles [T][Kp/8][128][8]
 *     (softmax of l_po), lab_tiles [T][128] (-1 = padding), T = ucd_con_max_tiles(n_px)
 *   - row metadata: row_ref [n_px] (class-sorted anchor row -> reference row), inv_norm [n_px]
 * Layout of a tile: element (row r, feature k) at ((k/8)*128 + r)*8 + k%8  (UMMA no-swizzle
 * canonical layout, K-major for S=A*C^T and MN-major for V=E*C from the same bytes).
 * ---------------------------------------------------------------------------------------- */
int64_t ucd_con_max_tiles(int64_t n_px);          /* ceil(2*n_px/128)+1 */
int ucd_con_prob_kpad(int C_old);                 /* C_old rounded up to a multiple of 16 */
int ucd_con_num_bins(int max_label, int C_old);   /* label bins of the class sort: max(max_label, C_old-1)+1 */
int64_t ucd_con_px_meta_ints(int64_t n_px);       /* int32 count of px_meta (7 planes of n_px) */
int64_t ucd_con_blk_meta_ints(int64_t n_px, int nb);
/* px_meta planes: 0 label_n | 1 mix | 2 flags | 3,4 rank of the pixel among the anchors / pseudos of its
 * 256-pixel block in pixel order | 5,6 the same rank among pixels of the SAME label (class-sorted order).
 * blk_meta: per-block exclusive offsets for both orders.  counts = {N_a, N_o, min_new, n_px}. */
int ucd_con_prep_labels(const int64_t* labels, const float* l_po, int B, int C_old, int h, int w,
                        int H, int W, int max_label, int32_t* px_meta, int32_t* blk_meta, int32_t* counts,
                        int32_t* counts_host /* optional: device-accessible (mapped, pinned) HOST int32[4] that receives
                        a copy of counts from the kernel itself - a host that needs N_a / N_o for tensor shapes then
                        waits on an event instead of queueing a D2H copy behind other transfers; NULL to skip */,
                        void* stream);
/* fp32 rows / labels are written in the reference's row order (pixel order b,y,x); the bf16 tiles are
 * written CLASS-SORTED (stable counting sort by label, anchors first, then pseudo columns) so that most
 * tiles hold a single label; row_ref[sorted anchor row] = reference row.  tile_range [max_tiles][2] =
 * min/max valid label per tile. */
int ucd_con_prep_pack(const float* f_n, const float* f_o, const float* l_po, const int32_t* px_meta,
                      int32_t* blk_meta, const int32_t* counts, int B, int C_old, int h, int w, int max_label,
                      float* anchor_f32, float* contrast_f32, void* la, void* lc,
                      int label_bytes /* element size of la / lc: 1 (int8, max_label <= 127) or 4 (int32) */,
                      void* feat_tiles, void* prob_tiles, int32_t* lab_tiles, int32_t* tile_range,
                      int32_t* row_range /*[ceil(n_px/128)][2], anchors only*/, int32_t* row_ref, float* inv_norm,
                      int64_t max_tiles, void* stream);
/* adjoint of the anchor gather + F.normalize: df_n[b,:,y,x] = (g - (g.a)a) * inv_norm for anchors, 0 else */
int ucd_con_prep_bwd(const float* g_anchor, const float* anchor_f32, const float* inv_norm,
                     const int32_t* px_meta, const int32_t* blk_meta, float* df_n, int B, int h, int w,
                     void* stream);
/* Feature hand-off in bf16 (SURVEY.md N2; replaces the fp32 features that segmentation_module.py:86-107 hands to
 * utils/loss.py:363-366): f_n / f_o are the head's NCHW features as bf16 (e.g. a head under autocast), read as they
 * are - no fp32 copy of the two feature maps; everything else as ucd_con_prep_pack.  The adjoint writes df_n in bf16. */
int ucd_con_prep_pack_bf16(const void* f_n, const void* f_o, const float* l_po, const int32_t* px_meta,
                           int32_t* blk_meta, const int32_t* counts, int B, int C_old, int h, int w, int max_label,
                           float* anchor_f32, float* contrast_f32, void* la, void* lc, int label_bytes,
                           void* feat_tiles, void* prob_tiles, int32_t* lab_tiles, int32_t* tile_range,
                           int32_t* row_range, int32_t* row_ref, float* inv_norm, int64_t max_tiles, void* stream);
int ucd_con_prep_bwd_bf16(const float* g_anchor, const float* anchor_f32, const float* inv_norm,
                          const int32_t* px_meta, const int32_t* blk_meta, void* df_n, int B, int h, int w,
                          void* stream);
/* min/max valid (>= 0) label of every 128-entry tile; with n_limit != NULL only entries [0, *n_limit) count */
int ucd_con_tile_ranges(const int32_t* lab_tiles, int64_t n_tiles, const int32_t* n_limit, int32_t* tile_range,
                        void* stream);
/* compat path of PixelConLossV2.forward with caller-supplied dense tensors: fp32 rows -> bf16 tiles */
int ucd_con_pack_rows(const float* rows, const int32_t* labels, int64_t n, void* feat_tiles,
                      int32_t* lab_tiles, int64_t max_tiles, void* stream);

/* Pixel-to-pixel branches of pre_contrastive_pixel (utils/loss.py:273-289, f_o and/or l_po absent): every pixel of
 * f [B,256,h,w] becomes a unit-norm row (F.normalize, eps 1e-12) of rows [B*h*w, 256] in (b,y,x) order;
 * inv_norm [B*h*w] is saved for the adjoint df = (g - (g.a) a) * inv_norm scattered back to [B,256,h,w]. */
int ucd_rows_normalize_fwd(const float* f, float* rows, float* inv_norm, int B, int h, int w, void* stream);
int ucd_rows_normalize_bwd(const float* g_rows, const float* rows, const float* inv_norm, float* df, int B, int h,
                           int w, void* stream);

/* ------------------------------------------------------------------------------------------
 * PixelConLossV2   (utils/loss.py:412-466), fused: the N_a x N_c matrices are never materialised.
 *
 * Columns (the contrast set) come as `n_chunks` chunks (one per rank after the all-gather) of
 * `chunk_tiles` tiles each; chunk_counts [n_chunks][2] = {N_a, N_o} of that rank (device), the chunk
 * holds N_a+N_o valid columns.  Rows (anchors) come as their own tile pointers (row block rb = tile rb;
 * in the fused path they alias the first tiles of the local chunk), *n_rows of them are valid.
 * tile_range / row_range: [tile][2] min/max valid label per column tile / row tile (ucd_con_tile_ranges);
 * sweep 2 skips column tiles whose range misses the row block's range (no equal-label pair possible).
 * self_tile0: column tile that holds row block 0 itself (row i of block rb is column i of tile
 * self_tile0+rb - the reference's `eye` on the first N_a columns, loss.py:437), or -1.
 * p_mode: 0 = P is None, 1 = joint probability pA.pC^T from the prob tiles with the GT-new override
 * (both labels >= *min_new -> 1, loss.py:380-393), 2 = dense fp32 P [N_a, ldp] (single chunk).
 *
 * ucd_con_fwd runs sweep 1 (row max, negative sum, positive count, V = sum_neg exp(s) c), the
 * combine, sweep 2 (loss terms, T, U) and the finalize; it writes
 *   out float[3]  = {sum_i loss_i over rows with num_i != 0, number of such rows, their ratio (= the loss)}
 *   grad_unit [max_row_tiles*128, 256] = d(sum_i loss_i)/d a_i   (scaled by g/M in ucd_con_bwd)
 * ---------------------------------------------------------------------------------------- */
/* plan_row_tiles (here and in ucd_con_fwd, same value): row tiles expected to hold anchors, 0 = max_row_tiles.  Only a
 * planning hint (column splits are chosen for that many row blocks); results do not depend on it beyond summation
 * order.  Used by hosts that size for the worst case because they do not read N_a back (sync-free path). */
size_t ucd_con_workspace_bytes(int64_t max_row_tiles, int64_t max_col_tiles, int64_t plan_row_tiles,
                               int64_t local_col_tiles /* chunk_tiles for a two-part run (part 1 + part 2), else 0 */);
/* Column arrays and the exchange payload.  chunk_stride_bytes == 0: feat_tiles / prob_tiles / lab_tiles / tile_range are
 * [n_chunks][chunk_tiles][...] arrays of their own and chunk_counts is [n_chunks][2].  chunk_stride_bytes > 0: every
 * rank ships ONE contiguous payload (header {N_a, N_o, min_new, n_px}, tile ranges, label tiles, probability tiles,
 * feature tiles; ucd_b200/losses.py::payload_layout) and the all-gathered buffer is [n_chunks][chunk_stride_bytes];
 * the five pointers address the sub-arrays of chunk 0 (part 1: of chunk `local_chunk`), chunk c lies c * stride bytes
 * further, and min_new points at chunk 0's header entry (the kernel takes the minimum over all chunks: no MIN
 * all-reduce).  part: 0 = everything in one call; 1 = only sweep 1 over the LOCAL chunk (pointers address that chunk
 * alone, e.g. the rank's own payload while the all-gather is still in flight); 2 = sweep 1 over the other chunks, the
 * combine, sweep 2 over all chunks and the finalize (pointers address the gathered buffer).  Parts 1 and 2 must be
 * called with the same n_chunks / chunk_tiles / max_row_tiles / plan_row_tiles / workspace. */
int ucd_con_fwd(const void* feat_tiles, const void* prob_tiles, const int32_t* lab_tiles,
                const int32_t* chunk_counts, int n_chunks, int64_t chunk_tiles, int64_t chunk_stride_bytes,
                int local_chunk, int part, const void* row_feat_tiles,
                const void* row_prob_tiles, const int32_t* row_lab_tiles, const int32_t* n_rows,
                const int32_t* tile_range, const int32_t* row_range, int64_t self_tile0, const int32_t* min_new, int p_mode, int kpad, const float* dense_p,
                int64_t ldp, float inv_temperature, int need_grad, float* out, float* grad_unit,
                void* workspace, size_t workspace_bytes, int64_t max_row_tiles, int64_t plan_row_tiles,
                void* stream);
/* Gradient of PixelConLossV2 with respect to the contrast features, utils/loss.py:445-466 (the reference back-propagates
 * into contrast_feature whenever it carries a graph; SURVEY.md Appendix A.2, column side):
 *   G_ij = dL/ds_ij = -kappa_i w_ij neg_i / den_ij (positive pair) | +kappa_i T_i exp(s_ij) (negative pair) | 0 (j is i)
 *   grad_unit [chunk_tiles*128, 256] = d(sum_i loss_i)/d c_j = (1/tau) sum_i (M G_ij) a_i,   kappa_i = [num_i != 0]/(M num_i)
 * (rows >= N_c are 0; scaled by g / out[1] in ucd_con_bwd with n_rows = device {N_c}, row_ref = NULL).  Call it after
 * ucd_con_fwd (part 0, any need_grad) on the same workspace, sized by ucd_con_contrast_grad_workspace_bytes with the
 * forward's max_row_tiles / chunk_tiles / plan_row_tiles, with the forward's column and row arguments: it reads the
 * forward's statistics (row max, neg, num, T) and runs a transposed third sweep (contrast tiles as rows, anchor tiles
 * streamed) that forms G pair by pair and accumulates G^T A on the tensor cores.  Single-chunk layout only
 * (n_chunks = 1, chunk_stride_bytes = 0), p_mode 0 or 2, self_tile0 0 or -1; anything else is UCD_EINVAL.  The self
 * pair (anchor i, column i) is never a positive; it is a negative when its two labels differ, as in the forward. */
size_t ucd_con_contrast_grad_workspace_bytes(int64_t max_row_tiles, int64_t chunk_tiles, int64_t plan_row_tiles);
int ucd_con_contrast_grad(const void* feat_tiles, const int32_t* lab_tiles, const int32_t* chunk_counts, int n_chunks,
                          int64_t chunk_tiles, int64_t chunk_stride_bytes, const void* row_feat_tiles,
                          const int32_t* row_lab_tiles, const int32_t* n_rows, const int32_t* tile_range,
                          const int32_t* row_range, int64_t self_tile0, int p_mode, const float* dense_p, int64_t ldp,
                          float inv_temperature, float* grad_unit, void* workspace, size_t workspace_bytes,
                          int64_t max_row_tiles, int64_t plan_row_tiles, void* stream);
/* Self-contrast losses of utils/loss_new.py on the same sweeps (SURVEY.md row N3):
 *   mode 0  PixelConLoss (v1), loss_new.py:354-400:  s = F F^T / tau, unshifted exponentials,
 *           loss = mean_{num_i != 0} -(1/num_i) sum_j mp_ij [s_ij - log(exp(s_ij) + neg_j)]
 *   mode 1  SupConLoss, loss_new.py:263-352 (labels or SimCLR; contrast_mode 'all': n_anchor = n, 'one': the first
 *           n_anchor rows are the anchors), kappa = temperature / base_temperature
 * on n rows packed by ucd_con_pack_rows (feat / lab tiles; tile_range from ucd_con_tile_ranges; counts = device
 * {n, 0}; n_rows = device {n}).  Both losses back-propagate through BOTH operands of F F^T: the forward runs sweep 1
 * (row max, negative sum, positive count), sweep 2 over the equal-label tiles (row terms), a per-pixel coefficient
 * kernel and - with need_grad - a third sweep that forms H = G + G^T pair by pair and accumulates H F on the tensor cores.
 *   out float[3] = {sum of the row losses, rows in the mean, their ratio (= the loss)}
 *   grad_unit [n, 256] = d(sum of row losses)/dF (scaled by g / out[1] in ucd_con_bwd, row_ref = NULL) */
size_t ucd_selfcon_workspace_bytes(int64_t tiles /* ceil(n / 128) */);
int ucd_selfcon_fwd(const void* feat_tiles, const int32_t* lab_tiles, const int32_t* tile_range, const int32_t* counts,
                    const int32_t* n_rows, int64_t n, int64_t n_anchor, int mode, float inv_temperature, float kappa,
                    int need_grad, float* out, float* grad_unit, void* workspace, size_t workspace_bytes, void* stream);
/* d_anchor[row_ref[i],:] = (*g_scalar) * g_mul / out[1] * grad_unit[i,:] for i < min(*n_rows, max_rows);
 * row_ref NULL = identity */
int ucd_con_bwd(const float* grad_unit, const float* out, const float* g_scalar, float g_mul,
                const int32_t* n_rows, const int32_t* row_ref, float* d_anchor, int64_t max_rows, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* UCD_B200_H */
