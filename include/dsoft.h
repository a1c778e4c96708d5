/*
 * dsoft.h - C ABI of the B200-native DINO-Soft loss path (libdsoft.so).
 *
 * The reference (nickxir12/Refining-CLIP-via-Dinov2-representations) is pure Python; the interface this
 * library sits under is the loss module `ClipLossWithDINOEnhancements`
 * (reference src/open_clip/loss.py:190-607) together with `gather_features` (loss.py:23-81) and
 * `compute_student_tau` (loss.py:166-175).  The Python mirror of that module
 * (refining-clip-via-dinov2-representations_b200/loss.py) binds these symbols through ctypes; see
 * INTEGRATION.md for the stub.
 *
 * Conventions
 *   - every pointer named *_dev is a CUDA device pointer on the current device;
 *   - `stream` is a cudaStream_t passed as void*; all work is stream-ordered and host-sync free;
 *   - functions return 0 on success, a cudaError_t value (>0) or a DSOFT_E* code (<0) on failure;
 *     dsoft_last_error() gives the message for the calling thread;
 *   - there is no CPU path: calls fail with DSOFT_ENODEV when the device is not sm_100.
 */
#ifndef DSOFT_H_
#define DSOFT_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DSOFT_VERSION 260 /* 0.2.6: SigLIP loss (DSOFT_F_SIGLIP, dsoft_siglip_*), later extended without a number
                             change by DistillClipLoss (DSOFT_F_DISTILL, dsoft_distill_*: additions only, nothing
                             existing changed), by kNN top-k (dsoft_knn_scratch_bytes, dsoft_knn_topk:
                             additions only) and by embedding geometry (dsoft_geometry_scratch_bytes,
                             dsoft_geometry: additions only); 0.2.5: retrieval ranks
                             (dsoft_retrieval_ranks); 0.2.4: weighted plans accept the fused
                             backward (no DSOFT_F_GMAT); 0.2.3: weighted
                             CE branch at world > 1 (phases 5 / 6, dsoft_plan_lse_rows, dsoft_plan_wsigma_info) */

/* error codes */
#define DSOFT_EINVAL (-1)  /* bad argument / unsupported shape            */
#define DSOFT_ENODEV (-2)  /* no sm_100 device / driver entry point missing */
#define DSOFT_ETMA (-3)    /* cuTensorMapEncodeTiled failed               */

/* dsoft_shape_t.flags */
#define DSOFT_F_SOFT 1u        /* image-image KL-teacher term enabled (loss.py:356-384)            */
#define DSOFT_F_TEXT 2u        /* text-text KL term enabled (loss.py:387-397)                      */
#define DSOFT_F_SOFT_LOCAL 4u  /* soft terms over the local b x b block only (reference at W>1)    */
#define DSOFT_F_ROW_ONLY 8u    /* gather_with_grad=False: gathered columns carry no gradient       */
#define DSOFT_F_GMAT 16u       /* two-phase backward: the similarity tiles are recomputed by the forward
                                  kernels' main loop, written out as fp16 logit-gradient matrices (scratch:
                                  2 bytes per element of the local [b x columns] blocks), and the feature
                                  gradients come from plain M=256 x N=256 gradient GEMMs.  Same results as
                                  the fused backward, faster when the scratch memory can be spared.       */

#define DSOFT_F_WEIGHTED 32u    /* denominator-modulated ("weighted") CE branch, loss.py:416-471 + diagnostics
                                  479-595: DINO-dissimilarity offsets on the CLIP logits.  Both backward forms:
                                  with DSOFT_F_GMAT one fp16 logit-gradient matrix per direction (world 1: one),
                                  without it the fused backward, whose two CLIP launches (bwd clip image / text
                                  rows) then also recompute the DINO tile.  world > 1 (the reference only runs
                                  it on one rank): this rank's rows of the global B x B problem, beta from the
                                  row stds of all B rows - see dsoft_plan_wsigma_info.  Such plans never share
                                  soft tiles (DSOFT_SYM_W). */
#define DSOFT_F_WSYM 64u        /* weight_text_symmetry: modulate the text direction too (loss.py:449-463) */
#define DSOFT_F_SIGLIP 128u     /* SigLIP sigmoid loss (open_clip SigLipLoss) instead of the DINO-Soft terms: only
                                  with Dp = Dd = 0 and no other flag (else DSOFT_EINVAL); runs through
                                  dsoft_siglip_forward / dsoft_siglip_backward, which dsoft_forward /
                                  dsoft_backward refuse.  dsoft_pack and the gathered layout are unchanged. */
#define DSOFT_F_DISTILL 256u    /* DistillClipLoss (open_clip) instead of the DINO-Soft terms: Dd = the teacher width
                                  and Dp = Dd; the packed row is image | text | teacher image | teacher text (dsoft_pack's
                                  student and DINO arguments carry the teacher).  The only other flag it takes is
                                  DSOFT_F_ROW_ONLY at world > 1 (else DSOFT_EINVAL); runs through
                                  dsoft_distill_forward / dsoft_distill_backward, which dsoft_forward /
                                  dsoft_backward refuse. */

/* element types accepted by dsoft_pack */
#define DSOFT_DT_F32 0
#define DSOFT_DT_BF16 1
#define DSOFT_DT_F16 2

/* Problem description. b = local batch, B = world*b = global batch.
 * Replaces the shape information the reference reads off its tensors in
 * ClipLossWithDINOEnhancements.forward (loss.py:301-302, 324-325). */
typedef struct dsoft_shape {
  int32_t b;      /* local rows per rank                                            */
  int32_t world;  /* world size W                                                   */
  int32_t rank;   /* this rank                                                      */
  int32_t D;      /* CLIP embedding dim (image and text), multiple of 8             */
  int32_t Dp;     /* student dim after the projection head; 0 = no projection       */
  int32_t Dd;     /* DINO feature dim; 0 = no DINO features                         */
  uint32_t flags; /* DSOFT_F_*                                                      */
  float teacher_temp; /* tau_t  (loss.py:368)                                       */
  float text_temp;    /* tau_txt (loss.py:391)                                      */
  float rho;          /* weighted CE: beta = rho * median(row std) / c_clip (loss.py:418, 443) */
  float c_clip;       /* weighted CE: clamp of the centred dissimilarity (loss.py:419)  */
} dsoft_shape_t;

typedef struct dsoft_plan dsoft_plan_t; /* opaque: packed layout, tile/split schedule, workspace map */

int dsoft_version(void);
const char* dsoft_last_error(void);

/* Plan life cycle (host only; no device work). */
int dsoft_plan_create(const dsoft_shape_t* shape, dsoft_plan_t** out);
void dsoft_plan_destroy(dsoft_plan_t* plan);

/* Sizes the caller must allocate (device memory):
 *   gathered : [B, row_elems] bf16 - packed image|text|student|dino embeddings of all ranks; the local
 *              block (rows rank*b ..) is written by dsoft_pack, the rest by the caller's all-gather
 *              (this is the buffer `gather_features` loss.py:23-81 would have produced, in bf16);
 *   state    : small per-call state that must survive from forward to backward;
 *   scratch  : partial statistics / partial gradients (and, with DSOFT_F_GMAT, the fp16 logit-gradient
 *              matrices), free to reuse after each call.  dsoft_forward only touches the first
 *              dsoft_plan_forward_scratch_bytes of it. */
size_t dsoft_plan_gathered_row_elems(const dsoft_plan_t* plan);
size_t dsoft_plan_gathered_bytes(const dsoft_plan_t* plan);
size_t dsoft_plan_state_bytes(const dsoft_plan_t* plan);
size_t dsoft_plan_scratch_bytes(const dsoft_plan_t* plan);
size_t dsoft_plan_forward_scratch_bytes(const dsoft_plan_t* plan);
/* Algorithmic FLOPs of one fwd+bwd evaluation for this rank (SURVEY.md 8(d) formula / world). */
double dsoft_plan_algorithmic_flops(const dsoft_plan_t* plan);
/* FLOPs of the tile-kernel launches of one fwd+bwd for this rank, in dsoft_profile_read order (n >= 7;
 * 9 slots are filled when available): fwd clip i->t, fwd clip t->i, fwd soft, bwd clip (image rows), bwd
 * clip (text rows) - of a weighted plan the fused weighted CE kernel, CLIP and DINO products -, bwd student,
 * bwd text, [7] CLIP logit-gradient kernel(s), [8] soft logit-gradient kernel
 * (the last two only with DSOFT_F_GMAT, where slots 3..6 are the gradient GEMMs).  `algorithmic` follows
 * SURVEY.md 8(d) (each distinct product once, no recompute); `executed` is what the tensor cores really do
 * (tile recompute included). */
int dsoft_plan_kernel_flops(const dsoft_plan_t* plan, double* algorithmic, double* executed, int n);
/* Number of CUDA kernels dsoft_forward / dsoft_backward launch (for bench.py's gpu_launches). */
int dsoft_plan_launches_forward(const dsoft_plan_t* plan);
int dsoft_plan_launches_backward(const dsoft_plan_t* plan);

/* Round the local embeddings to bf16 and write them into rows [rank*b, rank*b+b) of `gathered`.
 * student_dev may be NULL when Dp == 0; dino_dev may be NULL when Dd == 0 - or when the caller writes the DINO
 * columns itself with dsoft_gather_rows (device feature table).  ld* are row strides in elements.  Replaces the
 * operand preparation of loss.py:313, 330-347, 358-359, 392. */
int dsoft_pack(const dsoft_plan_t* plan, const void* image_dev, int image_dtype, int64_t ld_image,
               const void* text_dev, int text_dtype, int64_t ld_text, const void* student_dev,
               int student_dtype, int64_t ld_student, const void* dino_dev, int dino_dtype,
               int64_t ld_dino, void* gathered_dev, void* stream);

/* Projection head, forward (replaces `self.image_to_dino_proj(image_features)` under train.py's bf16 autocast,
 * loss.py:214-238 + 322-330): Linear(D -> Dp) when hidden_dim == 0 (w2/b2/hidden unused), else
 * Linear(D -> hidden_dim) + ReLU + Linear(hidden_dim -> Dp).  Runs on the tcgen05 tile kernel with bias, ReLU and the
 * bf16 rounding in the epilogue.  Input: the image columns of this rank's rows of `gathered` (written by dsoft_pack,
 * which must be called with student_dev == NULL); output: the student columns of the same rows (no separate student
 * tensor, no pack pass) and, for the MLP, hidden_dev [b][hidden_dim] bf16 (the ReLU output, needed by the caller's
 * backward).  Weights: bf16, nn.Linear layout ([out][in], row-major); biases fp32 (may be NULL).  All dims multiples
 * of 8, pointers 16-byte aligned.  LayerNorm / residual heads (loss.py:229-232, 331-343) stay with the caller. */
int dsoft_head_forward(const dsoft_plan_t* plan, void* gathered_dev, const void* w1_dev, const float* b1_dev,
                       const void* w2_dev, const float* b2_dev, int32_t hidden_dim, void* hidden_dev, void* stream);

/* Symmetric soft tiles across ranks (world > 1, global soft scope, gather_with_grad, DSOFT_F_GMAT, no
 * DSOFT_F_WEIGHTED, local batch a multiple of 512 and a per-rank block of more than 2^28 similarity entries;
 * environment DSOFT_SYM_W=0 switches it off, DSOFT_SYM_W=1 drops the size condition but never applies to weighted
 * plans).  The teacher / student / text Gram matrices are
 * symmetric, so each pair of row blocks is computed by ONE of its two ranks, and what belongs to the other rank's
 * rows is exchanged by the caller - the reduce-scatter of the gathered-feature gradients that `gather_features`
 * implies (loss.py:59-64, `_AllGather.backward`), restricted to the soft terms:
 *   dsoft_forward_phase(.., 4)   operand statistics (scalars, norms)
 *   dsoft_forward_phase(.., 1)   soft tile kernel + column reductions
 *   caller: the column sums [6][b] of every primed block k >= 1 go to rank (rank + k) % world, the received ones are
 *           added to the first b columns (dsoft_plan_symw_info gives offsets and sizes)
 *   dsoft_forward_phase(.., 3)   CLIP tile kernels; needs phase 4 only and touches nothing phase 1 or the exchange
 *                                touch, so the caller may run it on another stream next to them
 *   dsoft_forward_phase(.., 2)   finalize (losses, log-sum-exps): after phases 1 and 3 and the exchange
 *   dsoft_backward_phase(.., 4)  statistics relayout, fp16 gradient operands
 *   dsoft_backward_phase(.., 1)  soft logit-gradient kernel + its gradient GEMMs, incl. the transposed products
 *   caller: rows [(k-1) b, k b) of the transposed products go to rank (rank + k) % world, the received ones are added
 *           to this rank's own partial sums (split 0)
 *   dsoft_backward_phase(.., 3)  CLIP logit-gradient kernels + gradient GEMMs (as above: after phase 4, beside 1)
 *   dsoft_backward_phase(.., 2)  finalize (chain rule, outputs): after phases 1 and 3 and the exchange
 * Every call of one pass takes the same arguments.
 * dsoft_forward / dsoft_backward refuse such a plan.  Arguments as for dsoft_forward / dsoft_backward. */
int dsoft_plan_symw_info(const dsoft_plan_t* plan, long long* out12, int n);

/* Weighted CE branch at world > 1 (DSOFT_F_WEIGHTED): beta is the median of the row stds of ALL B rows, one value on
 * every rank, so the forward pauses once for the caller's exchange of the row stds:
 *   dsoft_forward_phase(.., 5)   everything up to the weighted row statistics (row stds into `state`)
 *   caller: all-gather the row-std block in place - rank r's [b x ndir] floats at state + out3[0] + r * out3[1]
 *   dsoft_forward_phase(.., 6)   median, modulated log-sum-exps, diagnostics, losses
 * dsoft_forward refuses such a plan (world 1 accepts both forms).  dsoft_plan_wsigma_info: out3 = {offset of the
 * block in `state` (floats), floats per rank, directions per row (2 with DSOFT_F_WSYM)}, all zero for other plans.
 * lse_local of such a plan has dsoft_plan_lse_rows() rows: the five log-sum-exps, then per modulated direction
 * c, lse~ (log2) and A of the rows, which the backward's column side needs from every rank (one all-gather with the
 * log-sum-exps, as before).  dsoft_plan_lse_rows returns 5 for every other plan. */
int dsoft_plan_wsigma_info(const dsoft_plan_t* plan, long long* out3, int n);
int dsoft_plan_lse_rows(const dsoft_plan_t* plan);
int dsoft_forward_phase(const dsoft_plan_t* plan, const void* gathered_dev, const float* logit_scale_dev,
                        const float* lambdas, void* state_dev, void* scratch_dev, float* lse_local_dev,
                        float* losses_dev, float* dbg_dev, void* stream, int phase);
int dsoft_backward_phase(const dsoft_plan_t* plan, const void* gathered_dev, const void* state_dev, void* scratch_dev,
                         const float* lse_all_dev, const float* gout_dev, const float* lambdas, float* d_image_dev,
                         float* d_text_dev, float* d_student_dev, float* d_scale_dev, void* stream, int phase);

/* CLIP-blind pair statistics (replaces the cs / ds matrices, masks and counts of
 * src/open_clip_train/helpers.py:221-285, `_pair_stats`).  Over the pairs i < j of n L2-normalised rows:
 *   counts_dev[2 k + 0] += #{cs_ij >= cmin[k]},  counts_dev[2 k + 1] += #{cs_ij >= cmin[k] and ds_ij <= dmax[k]}
 * (k < n_thr <= 8; cmin / dmax are HOST arrays; counts_dev = NULL skips the counting) and every pair with
 * cs_ij - ds_ij >= gap_floor is appended to cand_dev as 4 x 32 bit {int i, int j, float cs, float ds} (order
 * unspecified; *cand_count_dev counts ALL qualifying pairs, only the first cand_cap are stored; cand_cap = 0 skips the
 * collection).  The caller zeroes counts_dev and *cand_count_dev.  cs = clip_a . clip_b^T, ds = dino_a . dino_b^T,
 * bf16 operands [n][k] row-major with fp32 accumulation: pass a == b for bf16 features, or the split pair
 * a = [hi | lo | hi], b = [hi | hi | lo] (k = 3 d) for fp32 features at ~1e-5 cosine accuracy. */
int dsoft_pair_stats(const void* clip_a_dev, const void* clip_b_dev, int32_t k_clip, const void* dino_a_dev,
                     const void* dino_b_dev, int32_t k_dino, int32_t n, const float* cmin, const float* dmax,
                     int32_t n_thr, unsigned long long* counts_dev, float gap_floor, void* cand_dev,
                     uint32_t cand_cap, uint32_t* cand_count_dev, void* stream);

/* Retrieval ranks of open_clip's get_clip_metrics (open_clip_train/train.py) without the [n_img x n_txt] logit
 * matrix.  s_ij = <img_i, txt_j> (bf16 operands [n][k] row-major, fp32 accumulation, features used as given); t(j) =
 * text_image_dev[j], the image caption j belongs to (NULL: t(j) = j, which needs n_img == n_txt).
 *   rank_img_dev[i] = #{j : t(j) != i, s_ij > p_i},  p_i = max over the captions of image i of s_ij
 *   rank_txt_dev[j] = #{i : i != t(j), s_ij > s_t(j),j}
 * i.e. the 0-based position of the (first) positive in a descending sort, ties counted in the query's favour (strict
 * >).  The positives s_t(j),j and p_i come from an fp32 pre-pass over the same operands; the tile pass masks the
 * positives themselves, so a positive never counts against its own query.  Pass a == b-style split operands
 * img = [hi | lo | hi], txt = [hi | hi | lo] (k = 3 d) for fp32 features at ~1e-5 score accuracy, as for
 * dsoft_pair_stats.  Every map entry must lie in [0, n_img) and every image must have a caption (not checked on
 * the device: an entry out of range makes that caption count nothing, an image without caption gets rank n_txt).  Both rank arrays are written (no zeroing by the caller).  Operands and scratch 16-byte
 * aligned, k a multiple of 8; scratch_dev holds dsoft_retrieval_scratch_bytes(n_img, n_txt) bytes, O(n_img + n_txt).
 * Asynchronous on `stream`, no host synchronisation (graph-capturable). */
size_t dsoft_retrieval_scratch_bytes(int32_t n_img, int32_t n_txt);
int dsoft_retrieval_ranks(const void* img_dev, const void* txt_dev, int32_t k, int32_t n_img, int32_t n_txt,
                          const int32_t* text_image_dev, int32_t* rank_img_dev, int32_t* rank_txt_dev,
                          void* scratch_dev, void* stream);

/* kNN top-k (the neighbour search of DINO's knn_classifier) without the [n_q x n_k] score matrix.
 *   s_ij = <q_i, k_j> * key_scale_dev[j] * query_scale_dev[i]   (bf16 operands [n][width] row-major, fp32
 *   accumulation; a NULL scale is 1; pass 1/||k_j|| and 1/||q_i|| for cosine scores, so that the operands are never
 *   re-rounded after a normalisation)
 * values_dev [n_q][k] fp32 / indices_dev [n_q][k] int32: row i holds the k largest s_ij over j < n_k by decreasing
 * value, equal values by increasing key index (stable and deterministic).  Exact for any key order: the tile pass keeps
 * the best 32 (k <= 32) or 64 keys of every 128-column strip of every column split per query, and a merge selects the
 * top-k of those lists.  Both scales are applied before any comparison, so the order is that of the returned values.
 * Pass split operands q = [hi | lo | hi], k = [hi | hi | lo] (width = 3 d) for fp32 features, as for
 * dsoft_retrieval_ranks.  1 <= k <= 64 and k <= n_k (else DSOFT_EINVAL); operands and scratch 16-byte aligned, width
 * a multiple of 8; the scales hold n_k and n_q fp32 (any alignment).  scratch_dev holds
 * dsoft_knn_scratch_bytes(n_q, n_k, k) bytes for the current device, O(n_q k + n_k) (0: invalid arguments or no
 * sm_100 device).  Asynchronous on `stream`, no host synchronisation (graph-capturable). */
size_t dsoft_knn_scratch_bytes(int32_t n_q, int32_t n_k, int32_t k);
int dsoft_knn_topk(const void* q_dev, const void* k_dev, int32_t width, int32_t n_q, int32_t n_k, int32_t k,
                   const float* key_scale_dev, const float* query_scale_dev, float* values_dev, int32_t* indices_dev,
                   void* scratch_dev, void* stream);

/* Embedding geometry (Wang & Isola's uniformity and alignment, cosine histograms) without an [n_a x n_b] matrix.
 *   cos_ij = <a_i, b_j> * b_scale_dev[j] * a_scale_dev[i]   (bf16 operands [n][width] row-major, fp32 accumulation, a
 *   NULL scale is 1; pass 1/||row|| of the values the kernel multiplies for cosines)
 * One set: n_b = 0, the pairs i < j of the n_a >= 2 rows; b_dev is the column operand of the same rows (NULL: a_dev)
 * and the column scale is a_scale_dev.  Two sets: n_a, n_b >= 1; t(j) = text_image_dev[j], the row of a that column j
 * belongs to (NULL: t(j) = j, which needs n_a == n_b); the positives are the pairs (t(j), j), the negatives all others.
 * Split operands a = [hi | lo | hi], b = [hi | hi | lo] (width = 3 d) serve fp32 / fp16 features, as for
 * dsoft_knn_topk.
 *   sums_dev (fp64 [2], written): [0] = sum over the one set's pairs, or the negatives, of 2^(kappa (cos - 1)) with
 *     kappa = 2 t log2(e), i.e. exp(2 t (cos - 1)); 0 when t == 0 (0 <= t <= 20, else DSOFT_EINVAL)
 *     [1] = two sets: sum over the positives of max(2 - 2 cos, 0)^(alpha / 2) (alpha > 0); one set: 0
 *   hist_dev (uint64, written; may be NULL when bins == 0): [bins + 2] per histogram, the bins equal-width over
 *     [lo, hi) with the last one closed (numpy.histogram's convention), then the counts below lo and above hi.  One
 *     set: one histogram over the pairs; two sets: [0] the positives, [1] the negatives.  0 <= bins <= 256.
 *   pos_cos_dev (fp32 [n_b], or NULL; two sets only): the positives' cosines.
 * The positives come from an fp32 pre-pass over the same operands, and the tile pass masks them, so each is counted
 * once.  Map entries must lie in [0, n_a) (not checked on the device: a column whose entry is out of range counts
 * nothing).  Both sums reduce fixed-size fp64 partials in a fixed order: repeated calls are bit-identical.
 * Operands and scratch 16-byte aligned, width a multiple of 8; scratch_dev holds dsoft_geometry_scratch_bytes(n_a,
 * n_b, bins) bytes for the current device, O(n_a + n_b) (0: invalid arguments or no sm_100 device).  Asynchronous on
 * `stream`, no host synchronisation (graph-capturable). */
size_t dsoft_geometry_scratch_bytes(int32_t n_a, int32_t n_b, int32_t bins);
int dsoft_geometry(const void* a_dev, const void* b_dev, int32_t width, int32_t n_a, int32_t n_b,
                   const float* a_scale_dev, const float* b_scale_dev, const int32_t* text_image_dev, float t,
                   float alpha, float lo, float hi, int32_t bins, double* sums_dev, unsigned long long* hist_dev,
                   float* pos_cos_dev, void* scratch_dev, void* stream);

/* SigLIP sigmoid loss of a DSOFT_F_SIGLIP plan (open_clip SigLipLoss).  z_ij = s <I_i, T_j> + beta over the bf16
 * image | text columns of `gathered` (fp32 accumulation, s and beta applied in fp32), l_ij = +1 for j == i (global
 * index), -1 otherwise:
 *   loss = (1/b) sum_{i in this rank's rows} sum_{j < B} softplus(-l_ij z_ij)
 * dsoft_siglip_forward: logit_scale_dev = s (already exp'd), logit_bias_dev = beta (NULL: 0), both one fp32 on the
 *   device.  loss_dev: one fp32.  g_dev: NULL for a forward without gradient, else dsoft_siglip_g_bytes(plan) bytes
 *   (16-byte aligned) that receive this rank's fp16 logit-gradient matrix G 2^14 (G = d loss / d z times b, blocked
 *   layout), 2 bytes per element of the [b x B] row block.  The forward also leaves the sums of G x and G in `state`.
 *   Scratch: dsoft_plan_forward_scratch_bytes.
 * dsoft_siglip_backward: the same gathered / state and g_dev of the forward; gout_dev = the upstream gradient of the
 *   loss (one fp32).  Outputs fp32, 16-byte aligned: d_image [b][D] and d_text [b][D] = the derivative of the SUM of
 *   all ranks' losses with respect to this rank's rows (what an all-gather with gradient delivers), d_scale [1] and
 *   d_bias [1] (NULL: skipped) = the derivative of this rank's own loss; this assumes the same s, beta and upstream
 *   gradient on every rank.  Scratch: dsoft_plan_scratch_bytes (at world > 1 it holds the text rows' G, another
 *   2 b B bytes, computed here).  No statistic crosses ranks: the backward needs no collective.
 * Profile slots: 0 = forward tile kernel, 3 / 4 = the gradient GEMMs (image / text rows), 7 = the text rows' G kernel
 * (world > 1).  Both calls are asynchronous on `stream`, make no host synchronisation and can be captured in a graph. */
size_t dsoft_siglip_g_bytes(const dsoft_plan_t* plan);
int dsoft_siglip_forward(const dsoft_plan_t* plan, const void* gathered_dev, const float* logit_scale_dev,
                         const float* logit_bias_dev, void* state_dev, void* scratch_dev, void* g_dev, float* loss_dev,
                         void* stream);
int dsoft_siglip_backward(const dsoft_plan_t* plan, const void* gathered_dev, const void* state_dev, void* scratch_dev,
                          const void* g_dev, const float* gout_dev, float* d_image_dev, float* d_text_dev,
                          float* d_scale_dev, float* d_bias_dev, void* stream);

/* DistillClipLoss of a DSOFT_F_DISTILL plan (open_clip DistillClipLoss with local_loss).  x = s <I_i, T_j> (student),
 * t = s_t <I_t_i, T_t_j> (teacher) over the bf16 columns of `gathered` (fp32 accumulation); p / q = their soft-maxes
 * over this rank's rows of both directions (image rows x all B texts, text rows x all B images):
 *   contrastive = 1/2 [mean_i CE(x_i., i) + mean_j CE(x_.j, j)]     (global index of the positive)
 *   distill     = 1/2 [mean_i (lse(x_i.) - sum_j q_ij x_ij) + mean_j (lse(x_.j) - sum_i q_ij x_ij)]
 * dsoft_distill_forward: logit_scale_dev = s, dist_logit_scale_dev = s_t (both already exp'd, one fp32 each on the
 *   device).  losses_dev: [2] fp32 = contrastive, distill.  stats_dev: [4][b] fp32, this rank's row statistics -
 *   the log-sum-exps (log2 units) of the student and teacher logits of its image rows, then of its text rows.
 *   Scratch: dsoft_plan_forward_scratch_bytes.
 * dsoft_distill_backward: the same gathered / state.  stats_all_dev: the [W][4][b] concatenation of every rank's
 *   stats_dev (the caller all-gathers them; world 1: the forward's stats_dev); with DSOFT_F_ROW_ONLY this rank's
 *   [4][b] alone.  g_dev: dsoft_distill_g_bytes(plan) bytes (16-byte aligned) for the fp16 logit-gradient matrix of a
 *   [b x B] row block (world > 1: used by both directions in turn).  gout_dev: [2] fp32 upstream gradients g_c, g_d
 *   of the two losses.  Outputs fp32, 16-byte aligned: d_image [b][D] and d_text [b][D] = the derivative of the SUM of
 *   all ranks' losses with respect to this rank's rows (what an all-gather with gradient delivers; DSOFT_F_ROW_ONLY:
 *   of this rank's loss only, the gathered copies being constants), d_scale [1] = the derivative of this rank's own
 *   loss with respect to s; this assumes the same s, s_t and upstream gradients on every rank.  The teacher gets no
 *   gradient.  Scratch: dsoft_plan_scratch_bytes.
 * Profile slots: 0 / 1 = forward tile kernel (image / text rows), 7 = logit-gradient kernel, 3 / 4 = the gradient
 * GEMMs (image / text rows).  Both calls are asynchronous on `stream`, make no host synchronisation and can be
 * captured in a graph. */
size_t dsoft_distill_g_bytes(const dsoft_plan_t* plan);
int dsoft_distill_forward(const dsoft_plan_t* plan, const void* gathered_dev, const float* logit_scale_dev,
                          const float* dist_logit_scale_dev, void* state_dev, void* scratch_dev, float* stats_dev,
                          float* losses_dev, void* stream);
int dsoft_distill_backward(const dsoft_plan_t* plan, const void* gathered_dev, const void* state_dev, void* scratch_dev,
                           const float* stats_all_dev, void* g_dev, const float* gout_dev, float* d_image_dev,
                           float* d_text_dev, float* d_scale_dev, void* stream);

/* Column (in elements) of the DINO block inside a packed row: where dsoft_gather_rows must write when the caller
 * fills the DINO columns of `gathered` itself (dsoft_pack with dino_dev == NULL). */
size_t dsoft_plan_dino_col_offset(const dsoft_plan_t* plan);

/* Device-resident DINO feature table: out[i, :] = table[indices[i], :] for i < n, converted to out_dtype, with
 * the index range check done ON THE DEVICE.  Replaces the reference's per-step CPU gather from a pinned table,
 * H2D copy and `.item()` range check (src/open_clip_train/main.py:693-741, src/open_clip_train/train.py:250-280).
 * `out_dev` may be a plain [n, cols] matrix or the DINO columns of the packed `gathered` buffer (out_dev =
 * gathered + (rank*b) * row_elems + dsoft_plan_dino_col_offset, ld_out = row_elems, out_dtype = DSOFT_DT_BF16), so
 * that the gather feeds the loss kernels directly.  Rows with an index outside [0, n_rows) are written as zeros
 * and recorded in status_dev (4 x int64, sticky across calls, initialise to {0, INT64_MAX, INT64_MIN, -1}):
 * [0] number of bad indices, [1] smallest index seen, [2] largest index seen, [3] one bad index value.
 * cols must be a multiple of 8; table rows and out rows 16-byte aligned. */
int dsoft_gather_rows(const void* table_dev, int table_dtype, int64_t ld_table, int64_t n_rows, int32_t cols,
                      const int64_t* indices_dev, int32_t n, void* out_dev, int out_dtype, int64_t ld_out,
                      long long* status_dev, void* stream);

/* Forward statistics pass.  logit_scale_dev: one fp32 (already exp'd, reference model.py:571).
 * lambdas (HOST, 4 floats): {lambda_original, lambda_soft, text_lambda, lambda_weighted} (loss.py:387-388,
 * 417, 474).  Outputs: lse_local_dev [dsoft_plan_lse_rows][b] fp32 (rows 0..4: log2-domain row log-sum-exps:
 * clip i->t, clip t->i, teacher, student, text) and losses_dev[6] = {classic_loss, soft_imgimg, soft_texttext,
 * soft = imgimg + text_lambda * texttext, total = lambda_original * classic + lambda_soft * soft
 * + lambda_weighted * weighted, weighted_loss} (loss.py:317-319, 383, 396-397, 466, 473-477), the first three
 * already divided by b.  With DSOFT_F_WEIGHTED, dbg_dev (32 floats, may be NULL to skip the diagnostics pass)
 * receives the reference's diagnostic scalars (loss.py:479-595): [0,1] pc_err img/txt, [2,3] diag_max, [4..6]
 * delta_img max/mean/std, [7..9] delta_txt, [10,11] l1_prob_shift, [12,13] corr_rhat_dprob, [14..17] ce_img_base,
 * ce_txt_base, ce_img_mod, ce_txt_mod, [18..21] pos/neg_frac img, pos/neg_frac txt, [22,23] beta img/txt,
 * [24] rho, [25] c_clip.  beta stays on the device: no host synchronisation (the reference calls .item()).
 * At world > 1 the losses and diagnostics are this rank's row block (means over its b rows; beta global). */
int dsoft_forward(const dsoft_plan_t* plan, const void* gathered_dev, const float* logit_scale_dev,
                  const float* lambdas_host, void* state_dev, void* scratch_dev, float* lse_local_dev,
                  float* losses_dev, float* dbg_dev, void* stream);

/* Backward pass.  lse_all_dev [world][dsoft_plan_lse_rows][b] = all ranks' lse_local (all-gathered by the caller when
 * world > 1).  gout_dev[6] = upstream gradients of the six forward outputs (the chain rule through
 * `soft` and `total` is applied on the device with the same lambdas).  Outputs (fp32):
 * d_image [b][D], d_text [b][D], d_student [b][Dp] (ignored when Dp == 0), d_logit_scale [1].
 * Gradients follow the reference's per-rank convention (sum over ranks' losses == W x gradient of the
 * global mean loss; SURVEY.md "Gradient scaling"). */
int dsoft_backward(const dsoft_plan_t* plan, const void* gathered_dev, const void* state_dev,
                   void* scratch_dev, const float* lse_all_dev, const float* gout_dev,
                   const float* lambdas_host, float* d_image_dev, float* d_text_dev, float* d_student_dev,
                   float* d_logit_scale_dev, void* stream);

/* Optional timing of the tile kernels with CUDA events on the launching stream (bench.py roofline).
 * dsoft_profile_read synchronises the device, returns summed milliseconds and launch counts per kernel
 * kind since the last read, and resets the recorder.  9 slots: the 7 kinds above (with DSOFT_F_GMAT slots
 * 3..6 are the gradient GEMMs; without it slots 3 / 4 of a weighted plan are the fused weighted CE kernel) followed by the CLIP (2 launches) and the soft logit-gradient kernels. */
int dsoft_profile_enable(int on);
int dsoft_profile_read(double* ms_sum, int* counts, int n);

/* The independent tile kernels of one pass (3 forward, 4 backward) are launched on internal side streams
 * forked from / joined back into `stream`, so the next kernel's CTAs fill the partially empty last wave of
 * the previous one; callers still see plain stream-ordered semantics, and stream capture records a
 * fork/join graph.  on = 0 launches them serially on `stream` (also forced while dsoft_profile_enable(1) is
 * active so that per-kernel durations are isolated), on = 1 always forks, on < 0 (default, or the
 * DSOFT_CONCURRENCY=0/1 variable unset) forks only for small per-rank blocks, where it pays. */
int dsoft_set_concurrency(int on);
/* What the launches of `plan` will do right now: 0 = serial on `stream`, 1 = forked lanes, 2 = serial because the
 * recorder is on (a caller that overlaps the phases of a DSOFT_SYM_W plan on its own streams must not do so then). */
int dsoft_plan_concurrency(const dsoft_plan_t* plan);

/* Test / bring-up helper: C[M][N] (fp32) = A[M][K] . B[N][K]^T with bf16 operands through the same
 * TMA + tcgen05 tile path the loss kernels use (128 x 128 tiles). */
int dsoft_selftest_gemm(const void* a_bf16_dev, const void* b_bf16_dev, float* c_dev, int M, int N,
                        int K, void* stream);

/* Test / bring-up helper: out[M][F] (fp32) = fp16(A . B^T) . V with A [M][K], B [N][K] bf16 and
 * V [N][F] fp16: the backward data path (tile -> fp16 G tile in swizzled shared memory -> second tcgen05
 * GEMM with an MN-major fp16 operand) without any soft-max arithmetic. */
int dsoft_selftest_chain(const void* a_bf16_dev, const void* b_bf16_dev, const void* v_fp16_dev,
                         float* out_dev, int M, int N, int K, int F, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DSOFT_H_ */
