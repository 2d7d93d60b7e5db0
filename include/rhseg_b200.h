/*
 * rhseg_b200 — C-ABI of the B200-native restrictive-hierarchy head / loss / metric path.
 *
 * The reference (Banksylel/Restrictive-Hierarchical-Semantic-Segmentation) has no FFI: its
 * boundary is the Python API of Models/models.py, Metrics/losses.py and
 * Metrics/performance_metrics.py.  The functions below are what a binding for that path
 * binds; each one cites the reference lines it replaces (paths relative to the reference
 * root).  INTEGRATION.md shows the ctypes stub.
 *
 * Conventions
 *   - plain pointers and sizes only; the CALLER owns every buffer (PyTorch allocates them);
 *   - every entry point is stateless, stream-ordered on `stream` (a cudaStream_t passed as
 *     void*), never synchronises, never allocates, and is CUDA-graph capturable;
 *   - tensors are fp32 NCHW.  Feature / logit / probability tensors are contiguous; target
 *     tensors may be channel slices of a wider tensor, so they carry batch and channel
 *     strides (in elements) and a contiguous H*W plane;
 *   - return value: 0 on success, a negative RHSEG_ERR_* for argument errors, or a positive
 *     cudaError_t from the launch.  Nothing throws.
 *   - accumulators that cross thread blocks are fp64 (loss statistics, FiLM pool sums,
 *     weight-gradient sums) or int64 (confusion matrix).
 */
#ifndef RHSEG_B200_H
#define RHSEG_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RHSEG_ABI_VERSION 1
#define RHSEG_MAX_K 16           /* channels per level the table format holds            */
#define RHSEG_KERNEL_MAX_K 8     /* channels per level the fused kernels are built for    */
#define RHSEG_TABLE_INTS (4 + 5 * RHSEG_MAX_K)
#define RHSEG_EVAL_PREZEROED 1   /* rhseg_level_eval / rhseg_head_level_fwd_eval flag       */
#define RHSEG_EVAL_COMPOSED 0x40 /* rhseg_head_level_fwd_eval flag: validation evaluation     */
/* Feature element type flag of rhseg_head_level_fwd (zero_psum), rhseg_head_level_fwd_eval (flags),
 * rhseg_head_conv_bwd (zero_sums) and rhseg_head_conv_bwd_params (flags): set, feats (and dfeats) are
 * bf16 [B,C,Hf,Wf], 2-byte aligned (autocast-trained donors); clear, fp32.  Each bf16 value is converted
 * to fp32 exactly; every other tensor and every sum keeps its type, and dfeats is formed in fp32 and
 * rounded to bf16 (nearest even) once, when stored.  So the results equal the fp32 path's on the
 * upcast features.                                                                             */
#define RHSEG_FEATS_BF16 0x10
/* Feature layout flag of the same four calls: set, feats (and dfeats) are channels-last, [B,Hf,Wf,C] in
 * memory (what a donor converted with torch.channels_last returns); clear, [B,C,Hf,Wf].  Combines with
 * RHSEG_FEATS_BF16.  Requires C * element size to be a multiple of 16 bytes and a 16-byte aligned
 * feats (and dfeats) base (every pixel then starts on a 16-byte granule), and in the conv backward at
 * most 4096 bytes per pixel; a call that misses one returns RHSEG_ERR_UNSUPPORTED.  Every other tensor
 * keeps its layout.  Full-resolution logits and probabilities are formed in the [B,C,Hf,Wf] kernels'
 * order, and dfeats too for the same dz; see DESIGN.md 3.8 for when they are bit-identical.  The
 * low-resolution logits of upsampled heads and the fp64 sums agree to rounding.                */
#define RHSEG_FEATS_NHWC 0x20
/* Logit element type flag, OR-ed into the `flags` of rhseg_level_eval, the `act_mode` of rhseg_head_dz_fullres_fused and
 * the `logits_input` of rhseg_loss_stats and rhseg_loss_bwd: set, the logits (outs) are bf16 and dz / dz_out is written
 * as bf16 (a flat head run under bf16 autocast); clear, both are fp32.  Each bf16 logit is converted to fp32 exactly
 * when it is loaded; every other tensor and every sum keeps its type, and the gradient is formed in fp32 and rounded to
 * bf16 (nearest even) once, when stored.  So the results equal the fp32 path's on the upcast logits.  Only the flat
 * model's calls take it: rhseg_level_eval at the root level (child 0, no parent targets, prev_idx or idx_out) and
 * rhseg_head_dz_fullres_fused with RHSEG_ACT_ZEROS; any other combination returns RHSEG_ERR_UNSUPPORTED.          */
#define RHSEG_LOGITS_BF16 0x80
#define RHSEG_NSTAT 5            /* per (sample, class) loss statistics, see loss_stats   */
#define RHSEG_MAX_LEVELS 8       /* tree depth rhseg_step_finalize handles in one launch  */
#define RHSEG_STITCH_MAX_LEAVES 16 /* leaf channels of a flat model rhseg_stitch_levels reads */
#define RHSEG_STITCH_MAX_OUT 32    /* tree nodes (output channels) it writes                 */
/* Optional hint OR-ed into the `act_mode` (grouped levels) and `child` arguments: every parent group of the
 * level has exactly `gsz` channels (the reference's trees: one group of 4, 2 or 3; two groups of 2).  The kernels
 * then run code with the group layout fixed at compile time; 0 (no hint) reads the layout from the level table.
 * A hint that contradicts the table gives wrong results: pass what rhseg_tree_compile_level's table says.   */
#define RHSEG_GROUP_HINT(gsz) ((int)(gsz) << 8)
#define RHSEG_GROUP_HINT_OF(arg) (((arg) >> 8) & 0xff)

enum {
  RHSEG_OK = 0,
  RHSEG_ERR_ARG = -1,         /* null pointer / non-positive size / bad stride           */
  RHSEG_ERR_UNSUPPORTED = -2, /* K outside [1, RHSEG_KERNEL_MAX_K] etc.                  */
  RHSEG_ERR_TREE = -3         /* malformed level description                             */
};

/* activation modes of one level (Models/models.py:269, :282-300) */
enum {
  RHSEG_ACT_SIGMOID = 0, /* level 0: P = sigmoid(z)                                      */
  RHSEG_ACT_GROUPED = 1, /* level >0: per-parent softmax, P_c = P_parent * Q_c           */
  RHSEG_ACT_ZEROS = 2    /* level >0 without any group: probabilities are zeros          */
};

int rhseg_abi_version(void);
const char* rhseg_status_string(int status);
/* SM count / compute capability of the current device (grid sizing, sm_100a check). */
int rhseg_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ---------------------------------------------------------------------------------------
 * (1) class tree -> index tables.  Replaces build_hierarchy_indices / get_level_classes /
 * the child_groups construction and the per-forward string lookups
 * (Models/models.py:38-54, :82-98, :229-238, :293, :789; Metrics/losses.py:168).
 *
 * Host function.  `parent_ch[k]` is the channel (in level L-1) of the parent of channel k
 * of level L, or -1 for every channel of level 0.  Children of one parent must be
 * contiguous (they are, by construction of the reference's level lists).  Fills `table`
 * (RHSEG_TABLE_INTS int32, layout below); the caller uploads it to the device once.
 *   [0] K  [1] G (#groups)  [2] K_prev  [3] activation mode
 *   [4 + k]                 parent_ch[k]
 *   [4 + MAX_K + k]         group_of[k]
 *   [4 + 2*MAX_K + g]       group_start[g]
 *   [4 + 3*MAX_K + g]       group_len[g]
 *   [4 + 4*MAX_K + g]       group_parent[g]   (channel in level L-1)
 * --------------------------------------------------------------------------------------- */
int rhseg_tree_compile_level(const int32_t* parent_ch, int K, int K_prev, int32_t* table);

/* ---------------------------------------------------------------------------------------
 * (2) head, forward.  One level = FiLM (Models/models.py:58-77) folded into the 1x1 head
 * conv (:177-184, :268, :280, :765, :775), optional bilinear align_corners=True upsample
 * (:766, :776), sigmoid / restrictive per-parent softmax / composition / concat
 * (:269, :288-302, :767, :784-796).
 * --------------------------------------------------------------------------------------- */

/* FiLM fold: cond = prev_psum / n_pix; [gamma|beta] = film_w . cond + film_b;
 * eff_w[b,k,c] = head_w[k,c] * gamma[b,c]; eff_b[b,k] = head_b[k] + sum_c head_w[k,c] beta[b,c].
 * film_w == NULL (level 0): eff_w[b] = head_w, eff_b[b] = head_b, gamma_beta untouched.
 *   head_w [K,C], head_b [K], film_w [2C,K_prev], film_b [2C], prev_psum [B,K_prev] fp64,
 *   gamma_beta [B,2C] out, eff_w [B,K,C] out, eff_b [B,K] out.                            */
int rhseg_film_fold(const float* head_w, const float* head_b, const float* film_w, const float* film_b,
                    const double* prev_psum, double n_pix, int B, int C, int K, int K_prev,
                    float* gamma_beta, float* eff_w, float* eff_b, void* stream);

/* Level forward.  feats [B,C,Hf,Wf]; eff_w/eff_b from rhseg_film_fold; prev_probs
 * [B,K_prev,H,W] (NULL at level 0); table = device copy of the level table.
 * (H,W) == (Hf,Wf): conv + activation fused in one pass over the features.
 * otherwise: conv at (Hf,Wf) into z_lo [B,K,Hf,Wf] (caller workspace), then one hi-res pass
 * doing upsample + activation.
 * Outputs: logits [B,K,H,W], probs [B,K,H,W], psum [B,K] fp64 = sum over pixels of probs
 * (accumulated with atomics: zeroed here when zero_psum != 0, otherwise the caller passes a
 * zeroed buffer; it is the FiLM pool of the next level).                                  */
int rhseg_head_level_fwd(const void* feats, const float* eff_w, const float* eff_b,
                         const float* prev_probs, const int32_t* table,
                         int B, int C, int Hf, int Wf, int H, int W, int K, int K_prev, int act_mode,
                         float* z_lo, float* logits, float* probs, double* psum, int zero_psum,
                         void* stream);
/* zero_psum bit 1 (value 2): z_lo was zeroed by the caller (one fill for all levels); without it the
 * low-res pass zeroes z_lo itself whenever pixel tiles are split between CTAs.
 * zero_psum bit 2 (value 4): eff_w / eff_b are ONE [K,C] / [K] pair shared by all samples (a level without
 * FiLM, i.e. level 0: pass the head's own weight and bias, no rhseg_film_fold launch).
 * zero_psum & RHSEG_FEATS_BF16: feats holds bf16 values (see RHSEG_FEATS_BF16).
 * zero_psum & RHSEG_FEATS_NHWC: feats is channels-last (see RHSEG_FEATS_NHWC).                */

/* Level forward of an UPSAMPLED head (HRNet) fused with rhseg_level_eval: the hi-res pass that
 * interpolates and activates the logits also evaluates them against the ternary targets while
 * they are in registers.  Arguments = rhseg_head_level_fwd (psum must be zeroed by the caller) +
 * rhseg_level_eval (child is derived from act_mode).  Returns RHSEG_ERR_UNSUPPORTED for heads at
 * feature resolution: call the two functions separately there.                              */
int rhseg_head_level_fwd_eval(const void* feats, const float* eff_w, const float* eff_b,
                              const float* prev_probs, const int32_t* table,
                              int B, int C, int Hf, int Wf, int H, int W, int K, int K_prev, int act_mode,
                              float* z_lo, float* logits, float* probs, double* psum,
                              const float* targets, long t_bstride, long t_cstride,
                              const float* parent_targets, long pt_bstride, long pt_cstride,
                              const unsigned char* prev_idx, void* out_words, unsigned char* idx_out,
                              int flags, void* stream);
/* flags & RHSEG_EVAL_COMPOSED: the pass evaluates what rhseg_level_eval_composed evaluates (the reference's test(),
 * train.py:324-339) instead of the training evaluation: the confusion matrix of ProcessClasses over the composed
 * probabilities against the raw targets, and on grouped levels the consistency sums of the probabilities against
 * prev_probs, the parent probabilities the activation reads anyway.  parent_targets, prev_idx and idx_out are
 * ignored.  Shapes the band kernel does not take run rhseg_level_eval_composed after the forward.               */

/* ---------------------------------------------------------------------------------------
 * (2') head, backward (what autograd does for the reference; closed forms in DESIGN.md).
 * --------------------------------------------------------------------------------------- */

/* Activation backward at output resolution.
 *   dz_total = dz_in + d(probs path)/dz, where the gradient arriving at the probabilities is
 *   dP[b,k,n] = g_uniform[b,k] * inv_npix  (FiLM pool of the next level; NULL -> 0)
 *             + dp_pix[b,k,n] for channels whose bit is set in pix_mask (NULL/0 -> none).
 * For grouped levels also accumulates dL/dP_parent into dp_prev[b, parent, n] (+=, caller
 * pre-initialises; NULL -> skipped).  dz_in may be NULL (-> 0).  dz_out must not alias.   */
int rhseg_head_act_bwd(const float* logits, const float* prev_probs, const int32_t* table,
                       const float* dz_in, const double* g_uniform, double inv_npix,
                       const float* dp_pix, uint32_t pix_mask,
                       int B, int K, int K_prev, int H, int W, int act_mode,
                       float* dz_out, float* dp_prev, void* stream);

/* Adjoint of the bilinear align_corners=True upsample: dz_hi [B,K,H,W] -> dz_lo [B,K,Hf,Wf]
 * (deterministic, separable).  Three kernels, fastest first:
 *   flags & RHSEG_DZ_PREZEROED (caller zeroed dz_lo), W % 4 == 0, upsampling: ONE band kernel, each CTA
 *     reduces a band of hi-res rows along x and y in shared memory and adds its few low-res rows into
 *     dz_lo (at most two CTAs feed a row, so the fp32 result does not depend on their order);
 *   tmp != NULL (workspace [B,K,H,Wf] fp32), W % 4 == 0: halo-free row kernel + y-reduction kernel;
 *   otherwise the shared-memory tiled kernel.                                               */
#define RHSEG_DZ_PREZEROED 1
int rhseg_upsample_adjoint(const float* dz_hi, int B, int K, int Hf, int Wf, int H, int W,
                           float* dz_lo, float* tmp, int flags, void* stream);

/* Fused hi-res backward for upsampled heads (HRNet): forms per hi-res pixel
 *   dz_hi = d(g_ce*CE + g_dice*Dice)/dz  (closed form from logits, targets, coef of
 *           rhseg_loss_finalize)  +  activation backward of rhseg_head_act_bwd (g_uniform, dp_pix)
 * and applies the upsample adjoint in the same kernel, so dz_hi is never materialised.
 * Result dz_lo [B,K,Hf,Wf]; dp_prev (+=) as in rhseg_head_act_bwd.  tmp / flags as in
 * rhseg_upsample_adjoint.                                                                  */
int rhseg_head_dz_lowres_fused(const float* logits, const float* targets, long t_bstride, long t_cstride,
                               const float* coef, const float* g_ce, const float* g_dice,
                               const float* prev_probs, const int32_t* table, const double* g_uniform,
                               double inv_npix, const float* dp_pix, uint32_t pix_mask,
                               int B, int K, int K_prev, int Hf, int Wf, int H, int W, int act_mode,
                               float* dz_lo, float* dp_prev, float* tmp, int flags, void* stream);

/* 1x1 conv backward at feature resolution: dfeats[b,c,n] = sum_k eff_w[b,k,c] dz[b,k,n];
 * S[b,k,c] = sum_n dz[b,k,n] feats[b,c,n]; s[b,k] = sum_n dz[b,k,n]  (fp64, accumulated with
 * atomics: zeroed here when zero_sums != 0, otherwise the caller passes zeroed buffers).
 * dfeats may be NULL (features do not require grad).
 * zero_sums bit 0: zero S / s here; bit 1 (value 2): eff_w is one [K,C] matrix shared by all samples;
 * RHSEG_FEATS_BF16: feats and dfeats are bf16; RHSEG_FEATS_NHWC: feats and dfeats are channels-last.      */
int rhseg_head_conv_bwd(const void* feats, const float* dz, const float* eff_w,
                        int B, int C, int K, int n_pix,
                        void* dfeats, double* S, double* s, int zero_sums, void* stream);

/* rhseg_head_conv_bwd followed by rhseg_head_param_grads.  Arguments: those of the two functions; flags = zero_sums of
 * rhseg_head_conv_bwd | 4 when g_prev is zero on entry (part of a larger zero fill; otherwise it is zeroed here);
 * n_pix_out = H*W of the output (the FiLM pool size); ticket = a device counter that is zero on entry (left zero).
 * Two forms, same results: a level WITHOUT FiLM (film_w == NULL: d_head_w = sum_b S_b, d_head_b = sum_b s_b) of a
 * narrow donor (B*C*K <= 4096) is ONE launch, the sums being formed by the conv kernel's last CTA; every other level
 * is the conv kernel + the 12-CTA parameter kernel behind a programmatic dependent launch.                         */
int rhseg_head_conv_bwd_params(const void* feats, const float* dz, const float* eff_w, int B, int C, int K,
                               int n_pix, void* dfeats, double* S, double* s, int flags, const float* head_w,
                               const float* film_w, const float* gamma_beta, const double* prev_psum,
                               double n_pix_out, int K_prev, float* d_head_w, float* d_head_b, float* d_film_w,
                               float* d_film_b, double* g_prev, unsigned* ticket, void* stream);

/* Parameter gradients of one level from S / s (all sums over the batch):
 *   d_head_w [K,C], d_head_b [K]; and when film_w != NULL: d_film_w [2C,K_prev],
 *   d_film_b [2C], g_prev [B,K_prev] fp64 = film_w^T [dgamma|dbeta]  (the uniform gradient
 *   w.r.t. the previous level's pooled probabilities, before the 1/n_pix).
 * gamma_beta [B,2C] and prev_psum [B,K_prev] are the forward's.  g_prev is accumulated with
 * atomics: zeroed here unless g_prev_zeroed != 0 (the caller passes a zeroed buffer).        */
int rhseg_head_param_grads(const double* S, const double* s, const float* head_w,
                           const float* film_w, const float* gamma_beta, const double* prev_psum,
                           double n_pix, int B, int C, int K, int K_prev,
                           float* d_head_w, float* d_head_b, float* d_film_w, float* d_film_b,
                           double* g_prev, int g_prev_zeroed, void* stream);

/* ---------------------------------------------------------------------------------------
 * (3) hierarchical loss.  Replaces CrossEntropyLoss / SoftDiceLoss (Metrics/losses.py:16-134)
 * and hierarchical_consistency_loss (:150-177).
 * --------------------------------------------------------------------------------------- */

/* One pass over (outs, targets): per (sample, class) statistics, fp64 [B,K,RHSEG_NSTAT]:
 *   [0] sum_m t*lp   [1] |m|   [2] sum_m p*t   [3] sum_m p   [4] sum_m t,   m = (t != -1)
 * logits_input != 0: lp = log_softmax(outs), p = softmax(outs) over the K channels;
 * otherwise lp = p = outs (the modules' logits_input=False mode).  Zeroes `stats` first.
 * logits_input & RHSEG_LOGITS_BF16: outs is bf16 (either mode).
 * targets: element (b,k,n) at targets[b*t_bstride + k*t_cstride + n].                    */
int rhseg_loss_stats(const void* outs, const float* targets, long t_bstride, long t_cstride,
                     int B, int K, int n_pix, int logits_input, double* stats, void* stream);

/* Scalars from the statistics (one tiny launch):
 *   out[0] = CE   (losses.py:95-119: per class -w*S0/cnt, class mean, NaN sample -> 1, batch mean)
 *   out[1] = Dice (losses.py:23-66: per sample 1-(2I+smooth)/(U+smooth), NaN samples dropped;
 *            0 when none is left)      out[2] = number of non-NaN dice samples
 *   out[3] = number of non-NaN CE samples.      weights [K] fp32 (class_weight).
 * Also writes coef [B,K,3] fp32 = (dCE/dstat0, dDice/dstat2, dDice/dstat3) per (sample, class),
 * the closed-form backward coefficients rhseg_loss_bwd consumes (zero for dropped samples). */
int rhseg_loss_finalize(const double* stats, const float* weights, int B, int K, double smooth,
                        float* out4, float* coef, void* stream);

/* d(g_ce*CE + g_dice*Dice)/d outs -> dz [B,K,n_pix] (written, not accumulated).
 * g_ce / g_dice are DEVICE scalars (autograd's upstream gradients; NULL -> 0).            */
int rhseg_loss_bwd(const void* outs, const float* targets, long t_bstride, long t_cstride,
                   const float* coef, const float* g_ce, const float* g_dice,
                   int B, int K, int n_pix, int logits_input, void* dz, void* stream);
/* logits_input & RHSEG_LOGITS_BF16: outs and dz are bf16.                                  */

/* Consistency term of one (level, parent-group set): for each group g of `table`,
 * sums[g] = sum_{b,n} | sum_{c in g} cur[b,c,n] - prev[b,parent(g),n] |  (fp64, zeroed here).
 * The caller divides by B*n_pix and averages over all pairs (losses.py:172-177).          */
int rhseg_consistency_sums(const float* cur, const float* prev, const int32_t* table,
                           int B, int K, int K_prev, int n_pix, double* sums, void* stream);

/* ---------------------------------------------------------------------------------------
 * (4) metrics.  Replaces ProcessClasses + the torchmetrics calls of the five wrappers
 * (Metrics/performance_metrics.py:27-141) and the train-loop prediction glue
 * (train.py:206-231, predictEval.py:409-422).
 * --------------------------------------------------------------------------------------- */

/* Confusion matrix of one level, int64 [nc,nc] (row = target class, col = predicted class),
 * nc = K (child == 0) or K+1 (child != 0: class 0 = "no channel positive", rows with target
 * class 0 are dropped = torchmetrics ignore_index=0).  argmax = first maximum, NaN wins.
 * probs / targets both strided like targets above.  Zeroes `conf` first.                  */
int rhseg_confusion_matrix(const float* probs, long p_bstride, long p_cstride,
                           const float* targets, long t_bstride, long t_cstride,
                           int B, int K, int n_pix, int child, int64_t* conf, void* stream);

/* Per-class ratios from a confusion matrix, torchmetrics arithmetic (int64 -> fp32, ratio,
 * zero denominator -> 0).  out5 [5,nc] fp32 rows: F1/Dice, Jaccard/IoU, Accuracy (= per-class
 * recall, average=None), Precision, Recall.  (performance_metrics.py:62-66, :82-86, ...)   */
int rhseg_metric_ratios(const int64_t* conf, int nc, float* out5, void* stream);

/* Train-path prediction (train.py:206-231): onehot = one_hot(argmax(softmax(logits)))
 * zeroed where target == -1; eval_t = target with -1 -> 0.  Either output may be NULL.
 * pred_idx (int32 [B,n_pix], argmax index, optional) may be NULL.                         */
int rhseg_predict_onehot(const float* logits, const float* targets, long t_bstride, long t_cstride,
                         int B, int K, int n_pix, float* onehot, float* eval_t, int32_t* pred_idx,
                         void* stream);

/* Fused metrics straight from logits + ternary targets (SURVEY.md row f1): identical result
 * to rhseg_predict_onehot followed by rhseg_confusion_matrix, without the one-hot tensors. */
int rhseg_confusion_from_logits(const float* logits, const float* targets, long t_bstride, long t_cstride,
                                int B, int K, int n_pix, int child, int64_t* conf, void* stream);

/* Same fused gradient for full-resolution heads (UNet): dz_out [B,K,n_pix] written once. */
int rhseg_head_dz_fullres_fused(const void* logits, const float* targets, long t_bstride, long t_cstride,
                                const float* coef, const float* g_ce, const float* g_dice,
                                const float* prev_probs, const int32_t* table, const double* g_uniform,
                                double inv_npix, const float* dp_pix, uint32_t pix_mask,
                                int B, int K, int K_prev, int n_pix, int act_mode,
                                void* dz_out, float* dp_prev, void* stream);
/* act_mode & RHSEG_LOGITS_BF16: logits and dz_out are bf16 (RHSEG_ACT_ZEROS only).          */

/* All levels of one training step from the rhseg_level_eval workspaces (stored back to back in
 * level order), one launch:  out[0] = total = sum_L (CE_L + Dice_L) + consistency
 * (train.py:132-149), out[1] = consistency, out[2+4L .. 2+4L+3] = rhseg_loss_finalize's out4 of
 * level L, followed by each level's [5,nc_L] ratio block of rhseg_metric_ratios computed from the
 * workspace's confusion matrix; coef_all = the levels' [B,K_L,3] backward coefficients back to back.
 * weights_all = the levels' class weights back to back; K_per_level / groups_per_level are HOST
 * arrays (groups_per_level[0] is ignored).  summary (optional, fp64 [2 + 4*n_levels + sum nc_L^2]):
 * the ADDITIVE per-rank quantities a batch-sharded job all-reduces: B, consistency*B, per level
 * (sum_b CE_b, sum_valid Dice_b, #valid dice samples, #non-NaN CE samples), then the confusion
 * counts as fp64.                                                                           */
int rhseg_step_finalize(const void* eval_words, const float* weights_all, int B, int n_levels,
                        const int32_t* K_per_level, const int32_t* groups_per_level, double smooth,
                        long n_pix, unsigned level_mask, float* out, float* coef_all, double* summary, void* stream);
/* level_mask: bit L set = level L's CE + Dice enter the total (train.get_loss's level-pretrain curriculum,
 * train.py:125-134, skips levels L > cur_epoch // pretrain_epoch; their per-level values, metrics and the consistency
 * term are still reported, as the reference does).  All ones = every level.                                      */

/* Data-parallel gradient factors (SURVEY.md 8(e); reference semantics Metrics/losses.py:64-66, :117-119: CE is a mean
 * over all samples of the GLOBAL batch, Dice over the GLOBAL number of non-NaN samples).  local / global = this rank's
 * rhseg_step_finalize summary and its SUM over ranks; g = the upstream gradient (device scalar, NULL -> 1).
 *   out[2L]   = g * world * B_local / B_global             (-> g_ce   of rhseg_head_dz_*_fused at level L)
 *   out[2L+1] = g * world * n_valid_local[L] / n_valid_global[L]   (-> g_dice; 0 when no sample is valid anywhere)
 * so that the mean over ranks of the per-rank gradients equals the single-process gradient on the concatenated batch. */
int rhseg_dp_grad_scales(const double* local_summary, const double* global_summary, int n_levels, int world,
                         const float* g, float* out, void* stream);

/* Fused per-level TRAINING evaluation (train.py:206-239 for one level in one pass): loss
 * statistics + train-path prediction + confusion matrix of the masked one-hot prediction +
 * consistency sums of the masked one-hot predictions against the previous level's.
 *   parent_targets: the previous level's target slice (strided), prev_idx: its prediction index
 *   map (uint8 [B,n_pix]) as written by this function for that level; both NULL at level 0.
 *   out_words (8-byte words, zeroed here):
 *     [B*K*RHSEG_NSTAT fp64 statistics][RHSEG_MAX_K fp64 consistency sums][nc*nc int64 confusion]
 *   idx_out: uint8 [B,n_pix] prediction index map (NULL when no deeper level needs it).
 *   flags: RHSEG_EVAL_PREZEROED = the caller already zeroed out_words (one fill for all levels);
 *          RHSEG_LOGITS_BF16 = logits are bf16 (level 0 only).
 *   child: 0 / 1, optionally | RHSEG_GROUP_HINT(gsz).                                          */
int rhseg_level_eval(const void* logits, const float* targets, long t_bstride, long t_cstride,
                     const float* parent_targets, long pt_bstride, long pt_cstride,
                     const unsigned char* prev_idx, const int32_t* table, int B, int K, int n_pix,
                     int child, void* out_words, unsigned char* idx_out, int flags, void* stream);

/* Fused per-level VALIDATION evaluation: what the reference's test() computes for one level
 * (train.py:324-339), which differs from the training evaluation above:
 *   - confusion: ProcessClasses (first maximum, NaN wins, the prepended "nothing positive" channel on
 *     child levels) over the COMPOSED probabilities `probs` against the RAW ternary targets; child levels
 *     drop target class 0, level 0 counts every pixel;
 *   - consistency: per group g of `table`, sum over pixels of |sum_{c in g} probs_c - prev_probs[parent(g)]|
 *     on the real probabilities, without an ignore mask (rhseg_consistency_sums' sums), so that
 *     rhseg_step_finalize turns them into the test() term unchanged;
 *   - statistics: rhseg_level_eval's CE/Dice statistics of `logits`.
 * No prediction index map is read or written.
 *   logits, probs [B,K,n_pix] contiguous; prev_probs [B,K_prev,n_pix] contiguous (NULL: no consistency
 *   sums; ignored at level 0); targets strided as everywhere.  out_words, flags and child as in
 *   rhseg_level_eval (child: 0 / 1, optionally | RHSEG_GROUP_HINT(gsz)).  A bulk-copy pipeline serves
 *   16-byte aligned planes with n_pix % 4 == 0 and target strides that are multiples of 4; any other
 *   shape takes a one-pixel-per-thread kernel with the same results.                            */
int rhseg_level_eval_composed(const float* logits, const float* probs, const float* prev_probs,
                              const float* targets, long t_bstride, long t_cstride, const int32_t* table,
                              int B, int K, int K_prev, int n_pix, int child, void* out_words, int flags,
                              void* stream);

/* Flat -> hierarchy stitching (predictEval.py:85-185, :381-388): `leaves` [B,n_leaves,n_pix] are the
 * flat model's leaf channels (predictions or targets); `out` [B,n_out,n_pix] gets one channel per tree
 * node in level order: masks[o] bit 31 set = copy leaf channel (the single low bit set), clear = union
 * (any > 0 -> 1.0) of the leaf channels whose low bits are set.  masks is a HOST array.          */
int rhseg_stitch_levels(const float* leaves, int B, int n_leaves, int n_pix, const uint32_t* masks,
                        int n_out, float* out, void* stream);

/* out [B, c_image+K, n_pix] = cat([image [B,c_image,n_pix], logits [B,K,n_pix]], dim=1).  Stand-alone
 * utility (north_star item 2): the reference itself never concatenates (SURVEY F1), so nothing in
 * the forward path calls it.                                                                    */
int rhseg_concat_image_logits(const float* image, int c_image, const float* logits, int K, int B, int n_pix,
                              float* out, void* stream);

/* Ternary targets as int8 ({1, 0, -1}; Data/dataset.py:227-265 only ever produces these three values) -> the fp32
 * tensor the path reads: out[i] = (float) in[i], n elements, both pointers 16-byte aligned.  Lets a caller ship the
 * wide target tensor over PCIe at a quarter of its fp32 size (FusedHierStep accepts int8 targets).                 */
int rhseg_targets_i8_to_f32(const signed char* in, long n, float* out, void* stream);

/* Data-parallel exchange buffer (no reference counterpart: train.py:201-241 is single-process; the
 * batch shards over ranks and ONE all-reduce of a packed fp64 buffer carries the step summary and
 * the head / FiLM parameter gradients, SURVEY.md 8(e)).
 * rhseg_pack_f64:   out[off_k + i] = (double) srcs[k][i]   for n <= 32 fp32 device tensors of
 *                   counts[k] elements, back to back in list order (one launch).
 * rhseg_unpack_f32: dsts[k][i] = (float)(in[off_k + i] * scale)   the inverse, with the averaging
 *                   factor folded in.  srcs / dsts / counts are HOST arrays (of device pointers).   */
int rhseg_pack_f64(const void* const* srcs, const long* counts, int n, double* out, void* stream);
int rhseg_unpack_f32(const double* in, double scale, void* const* dsts, const long* counts, int n, void* stream);

/* One-shot all-reduce (SUM) of the exchange buffer over NVLink peer memory: single node, one process
 * per GPU, replaces the NCCL all-reduce of the ~100 KB buffer (pure latency) by ONE kernel: it converts
 * the rank's contribution to fp64, pushes every element into each peer's receive area as a
 * self-validating 16-byte record {lo32, epoch, hi32, epoch}, polls its own memory for the peers'
 * records and adds them in rank order (bit-identical results on every rank; one NVLink one-way
 * latency; no fences, flags or barriers).  CUDA-graph capturable (the epoch lives in device memory).
 *   rhseg_xchg_create : allocates this rank's receive area (2 * world * capacity * 16 bytes) and returns
 *                       its CUDA IPC handle (RHSEG_XCHG_HANDLE_BYTES bytes) for the peers.
 *   rhseg_xchg_connect: maps the peers' areas; handles = world * RHSEG_XCHG_HANDLE_BYTES bytes in rank
 *                       order (gathered by the host, e.g. torch.distributed.all_gather).
 *   rhseg_xchg_all_reduce: out[0..n_sum) = sum_r summary_r ; out[n_sum + off_k + i] = sum_r (double)
 *                       srcs_r[k][i]  (srcs / counts as in rhseg_pack_f64; out may alias summary;
 *                       n_sum + sum counts <= capacity).  Every rank calls it with the same sizes, in
 *                       the same order.
 *   rhseg_xchg_status : 0, or 1 (sticky) when a wait for a peer timed out.  A timeout is a hard failure: that exchange
 *                       and every later one of the context writes NaN into the WHOLE result, so the loss and the
 *                       gradients poison visibly instead of the replicas diverging; the host raises at its next sync
 *                       point (dist.PeerExchange.check).  Synchronises the device.
 *   rhseg_xchg_set_timeout_ms: wait limit per exchange, default 30 s (RHSEG_XCHG_TIMEOUT_MS), 0 = wait for ever like an
 *                       NCCL all-reduce.  Applies to launches (and graph captures) made after the call.
 * World size <= 16.                                                                               */
#define RHSEG_XCHG_HANDLE_BYTES 64
int rhseg_xchg_create(long capacity, int world, void** ctx_out, unsigned char* handle_out);
int rhseg_xchg_connect(void* ctx, int rank, const unsigned char* handles);
int rhseg_xchg_all_reduce(void* ctx, const double* summary, long n_sum, const void* const* srcs,
                          const long* counts, int n, double* out, void* stream);
int rhseg_xchg_status(void* ctx, int* status_out);
int rhseg_xchg_set_timeout_ms(void* ctx, long ms);
int rhseg_xchg_destroy(void* ctx);

#ifdef __cplusplus
}
#endif
#endif /* RHSEG_B200_H */
