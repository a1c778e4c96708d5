// DINO-Soft streaming row-block kernels for sm_100a (tcgen05 + TMEM + TMA).
//
// One CTA owns a block of 128 rows (TMEM lanes) of the B x B similarity matrices and streams column tiles of
// them:
//   * forward ("stats") kernels reduce every tile to per-row soft-max statistics; nothing of size B x B is
//     written to HBM;
//   * two-phase backward, phase 1 (MODE_CLIP_G / MODE_SOFT_G of the forward kernel): the tile is recomputed and
//     turned into the fp16 logit-gradient tile G, which is streamed to HBM in a blocked layout for the gradient
//     GEMMs of dsoft_gy.cuh (2 bytes per matrix element instead of recomputing per feature chunk);
//   * fused backward (dsoft_bwd_kernel, fallback when the G matrices do not fit): G stays in shared memory and
//     is fed straight back into the tensor core as the A operand of dX += G . Y.
//
// Reference semantics being reproduced (file:line in /root/reference/src/open_clip/loss.py):
//   CLIP logits / CE ............ get_logits 254-274, forward 313-319
//   teacher / student / text KL .. forward 356-397
// Warp roles (12 warps): 0 = TMA producer, 1 = tcgen05.mma issuer, 2 = TMEM allocator,
// 3 = idle (fused backward: DSMEM sender), 4..11 = epilogue (warp w owns TMEM lanes 32*(w%4).., column half
// (w-4)/4).
#pragma once

#include <type_traits>

#include "dsoft_ptx.cuh"

namespace dsoft {

constexpr int BM = 128;                  // rows per CTA == TMEM lanes
constexpr int BN = 128;                  // columns per similarity tile
constexpr int BK = 64;                   // bf16 per 128-byte swizzled smem row
constexpr int TILE_BYTES = BM * BK * 2;  // one TMA box: 128 rows x 128 B = 16 KiB
constexpr int NUM_THREADS = 384;
constexpr int EPI_WARP0 = 4;
constexpr int NUM_EPI_THREADS = 256;
constexpr int TMEM_COLS = 512;
constexpr int F_STAGES = 6;      // forward operand ring (A+B boxes per stage)
constexpr int F_SLOTS = 4;       // forward S-tile slots in TMEM (4 x 128 columns)
constexpr int B_STAGES = 4;      // backward operand ring
constexpr int B_SLOTS = 2;       // backward S-tile slots (2 x 128 columns) + 256 accumulator columns
constexpr int CHUNK_F = 256;     // gradient features accumulated in TMEM per pass
constexpr int ACC_COL = 256;     // TMEM column where the gradient accumulator starts
constexpr float NEG_BIG = -1.0e30f;  // masked logit (finite: 0 * NEG_BIG stays 0)
constexpr float M_FLOOR = -1.0e4f;   // initial running max (log2 units); real logits are far above

constexpr int MODE_CLIP = 0;
constexpr int MODE_SOFT = 1;
constexpr int MODE_RAW = 2;  // bring-up: forward stores the raw tile, backward uses G = raw dot products
constexpr int MODE_CLIP_G = 3;  // forward main loop, epilogue writes the fp16 logit-gradient tile (two-phase bwd)
constexpr int MODE_SOFT_G = 4;
// denominator-modulated ("weighted") CE branch, loss.py:416-471 + diagnostics 479-595: CLIP + DINO tiles
constexpr int MODE_WCE_STAT = 5;
constexpr int MODE_WCE_LSE = 6;
constexpr int MODE_WCE_DBG = 7;
constexpr int MODE_WCE_G = 8;
constexpr int MODE_WCE_X = 9;  // fused backward (dsoft_bwd_kernel) of the same logit gradient: no G matrix in HBM
constexpr int MODE_SOFT_SYM16 = 13;  // forward soft statistics, upper block triangle + column reductions, on a
                                     // 16x256b TMEM load shape (4 rows per thread: short butterflies)
constexpr int MODE_LINEAR = 11;   // projection head layer: out = act(A . W^T + bias) as bf16 (loss.py:214-238, 322-347)
constexpr int MODE_PAIRS = 12;    // CLIP-blind pair statistics (open_clip_train/helpers.py:221-285): threshold counts
                                  // and candidate pairs over the upper triangle of two Gram matrices
constexpr int MODE_CLIP_SYM = 10; // forward CLIP statistics of BOTH directions from one pass over I . T^T: row
                                  // log-sum-exp partials as MODE_CLIP + per-warp column partials (the text -> image
                                  // direction is the transpose: loss.py:267/273 recomputes it)
constexpr int MODE_RANKS = 14;    // retrieval ranks (open_clip get_clip_metrics): per image and per caption, the number
                                  // of non-positive scores of I . T^T above its positive, over the full rectangle
constexpr int MODE_SIGLIP = 15;   // SigLIP sigmoid loss (open_clip SigLipLoss): per pair loss and logit gradient from the
                                  // pair's own logit; writes the fp16 G tile (scaled by 2^SIG_GK) and row partials
constexpr int SIG_GK = 14;        // SigLIP G is stored as G * 2^14: |G| < 1, and sigma down to 2^-28 stays normal fp16
constexpr int MODE_DIST_FWD = 16; // DistillClipLoss (open_clip): student and teacher row statistics of one direction
                                  // from two products per tile (student logits, teacher logits)
constexpr int MODE_DIST_G = 17;   // DistillClipLoss logit gradient of one direction's rows, both directions' terms
constexpr int MODE_TOPK = 18;     // kNN top-k (DINO knn_classifier): per query row and 128-column strip of a column
constexpr int MODE_TOPK32 = 19;   // split, the 64 (MODE_TOPK32: 32) best (score, key index) in registers
__host__ __device__ constexpr int topk_list(int mode) { return mode == MODE_TOPK32 ? 32 : 64; }
constexpr int MODE_GEOM = 20;     // embedding geometry (Wang & Isola uniformity, cosine histograms): per pair of a Gram
                                  // matrix of scaled rows, one exponential and one histogram count
constexpr int GEOM_BINS_MAX = 256;  // histogram bins; each epilogue warp counts into [bins + 2] (below, above) in smem

// scalar block computed on device by prep_scalars_kernel (no host sync on logit_scale)
enum {
  SC_SCALE = 0,     // logit scale s
  SC_SCALE_L2 = 1,  // s * log2(e)
  SC_ITS = 2,       // 1/tau_s            (compute_student_tau, loss.py:166-175)
  SC_ITS_L2 = 3,    // log2(e)/tau_s
  SC_ITT = 4,       // 1/tau_t            (teacher_temp, loss.py:368-369)
  SC_ITT_L2 = 5,
  SC_ITX = 6,       // 1/tau_txt          (text_student_temp, loss.py:391-393)
  SC_ITX_L2 = 7,
  SC_RMIN_T = 8,    // min_j 1/||text_j||    (atomicMin by rinv_kernel; +inf until then)
  SC_RMIN_Z = 9,    // min_j 1/||student_j||
  SC_RMIN_D = 10,   // min_j 1/||dino_j||
  SC_WCE_IGK = 11,  // weighted CE backward: 1/gk (SC_WCE_GK)
  SC_TICKET_F = 12, // (int) blocks of finalize_fwd_kernel that are done: the last one reduces the row losses
  SC_TICKET_B = 13, // (int) same for finalize_bwd_kernel
  SC_C_CLIP = 14,   // reference exponent c of the factorised CLIP logit gradients (lse_prepare_kernel)
  SC_FAST_CLIP = 15,// 1.0: all CLIP log-sum-exps lie within 200 log2 units -> one exponential per pair
  SC_WBETA = 16,    // [2] beta = rho * median(row std) / c_clip of the weighted CE, image / text direction
  SC_WBETA2 = 18,   // [2] beta * log2(e)
  SC_SIG_BIAS = 20, // SigLIP: logit bias beta (0 without one)
  SC_SIG_GX = 21,   // SigLIP: sum over this rank's pairs of G x (d logit_scale, before gout / b), by the forward
  SC_SIG_G = 22,    // SigLIP: sum of G (d logit_bias, before gout / b)
  SC_TICKET_S = 23, // (int) SigLIP finalize tickets (forward, backward)
  SC_DST_TSCALE_L2 = 24, // DistillClipLoss: teacher scale s_t * log2(e)
  SC_DST_GC = 25,   // DistillClipLoss backward: g_c * gk (contrastive upstream gradient times the G scale)
  SC_DST_GD = 26,   // g_d * gk (distill upstream gradient times the G scale)
  SC_DST_GK = 27,   // gk: power-of-two scale of the fp16 G (2^14 while |g_c| + |g_d| <= 1)
  SC_DST_SPD = 28,  // sum over this rank's rows of both directions of (sum_j p x - x_ii), by the forward
  SC_DST_SPQ = 29,  // sum over the same rows of (sum_j p x - sum_j q x)
  SC_TICKET_DST = 30, // (int) DistillClipLoss forward finalize ticket
  SC_WCE_GK = 31,   // weighted CE backward: gk, power-of-two scale of its fp16 logit gradient (wce_gscale_kernel)
  SC_COUNT = 32
};

struct TileMaps {
  CUtensorMap m[4];  // 0 = image, 1 = text, 2 = student, 3 = dino; box = 64 features x 128 rows, SW128
  CUtensorMap g[2];  // logit-gradient modes: the blocked fp16 G matrices (gout[0], gout[1]) as 64 columns x
                     // (row blocks * K tiles * 128) rows, box = 64 columns x 32 rows, SW128: TMA STORES of the
                     // epilogue warps' staged 32-row strips
};

struct FwdParams {
  int nprod;        // products per tile: clip 1; soft 2 (teacher, student) or 3 (+ text)
  int a_map[3];     // tensor map of the row-side operand of product p
  int b_map[3];     // tensor map of the column-side operand of product p
  int kchunks[3];   // ceil(K_p / 64)
  int row0;         // global index of local row 0 (rank * b)
  int b;            // local rows
  int col0;         // first global column in scope
  int ncols;        // number of columns in scope
  int ntiles;       // ceil(ncols / bn)
  int tiles_per_split;
  int npart;        // nsplit * 2 (two column halves per split)
  int bn;           // columns per tile: 256 (one N=256 MMA per K step, 2 TMEM slots); 128 only in the self test
  int resident;     // single product with K <= 512: the row block's operand stays in smem (8 boxes),
                    // only the column operand streams through a ring of 16 KiB stages
  const float* scal;
  const float* rinv[3];  // per product: inverse L2 norms by global index (soft only)
  float* part;           // partial statistics [nstat][npart][b]
  float* diag;           // clip: raw dot product on the diagonal [b]
  // ---- logit-gradient modes (MODE_CLIP_G / MODE_SOFT_G: first phase of the two-phase backward)
  const float* lse_row[3];  // per product: LSE (log2) of this rank's rows (soft: 0 teacher, 1 student, 2 text)
  const float* lse_col[3];  // clip, exact form: LSE by global column (the OTHER direction's)
  const float* colfac[3];   // per product, by global column: 2^(c - lse_col) of the factorised logit gradients
                            // (soft teacher in the exact form: lse_col itself), written by lse_prepare_kernel;
                            // zero (exact: +1e30) when the column-side terms are dropped
  int fast_t;               // soft G: teacher in the factorised form (log2(e)/tau_t <= 60)
  __half* gout[2];          // fp16 logit gradients, blocked [row block][64-col K tile][128 rows][64 cols]:
                            // clip -> gout[0]; soft -> gout[0] student, gout[1] text
  int g_pitch;              // columns of G (multiple of 64 >= ncols)
  int row_only;             // clip, exact form: gather_with_grad == False drops the column-side terms
  float* ds_part;           // clip: d(logit_scale) row partials [npart][b]
  // ---- weighted-CE modes (MODE_WCE_*): one rank's [b x B] row block (row0 = rank * b, col0 = 0)
  int ncolvec;              // per-column vectors staged per tile: colvec[0 .. ncolvec)
  const float* colvec[6];   // [0] 1/||dino_j||; G mode, by global column, of the OTHER direction: [1] lse,
                            // [2] lse~, [3] c', [4] A'
  const float* wrow[4];     // per row: [0] lse of the unmodified logits (log2), [1] c_a, [2] lse~ (log2), [3] A_a
  int wdir;                 // 0: image rows x text columns, 1: text rows x image columns
  int wsym;                 // G mode: the column-side direction is modulated (image rows: weight_text_symmetry,
                            // loss.py:449-463; text rows: always)
  int wrow_plain;           // G mode: the row-side direction is the classic CE (text rows without weight_text_symmetry)
  int wsplit;               // G mode, world > 1: the d(logit_scale) row partial takes the row-side term only (the
                            // text rows' launch holds the rest), and row_only drops the column-side term
  float wcc;                // c_clip
  const float* wgout;       // G mode: upstream gradients [6] (device)
  // ---- symmetric forward (MODE_SOFT_SYM16): column partials [6][cp_rows = 4 * row blocks][cp_pitch]
  float* colpart;
  int cp_rows, cp_pitch;
  // ---- one-pass CLIP forward (MODE_CLIP_SYM): column partials (reference exponent, sum) [cp_rows][cp_pitch] each,
  // and a lower bound of every row's / column's log-sum-exp: the raw diagonal dot product by global index
  float* colM;
  float* colS;
  const float* dbound;
  // ---- pair statistics (MODE_PAIRS): products [0] CLIP Gram, [1] DINO Gram of L2-normalised rows, pairs i < j
  int pr_nthr;                    // threshold pairs (<= 8)
  float pr_cmin[8], pr_dmax[8];   // count cs >= cmin, and cs >= cmin && ds <= dmax
  unsigned long long* pr_counts;  // [8][2] (clip-high, blind), or null: skip the counting
  float pr_gap_floor;             // pairs with cs - ds >= floor are appended to pr_cand (i, j, cs, ds)
  float4* pr_cand;
  unsigned int pr_cand_cap;
  unsigned int* pr_cand_count;    // total number of qualifying pairs (may exceed the capacity)
  // ---- projection-head layer (MODE_LINEAR): out[li][j] = act(dot + bias[j]) -> bf16, j < ncols (multiple of 8)
  __nv_bfloat16* lin_out;
  int lin_ld;             // row stride of out in elements (multiple of 8)
  const float* lin_bias;  // [ncols] or null
  int lin_relu;
  float wlam[2];            // G mode: lambda_original, lambda_weighted
  int tri;                  // soft G, world == 1: the matrices are symmetric -> only the 256-column tiles from the
                            // row pair's own diagonal tile (index rb / 2) onwards are computed and stored, scaled
                            // symmetrically; the gradient GEMM reads the missing part from the transposed blocks
  int ds_both;              // clip, world == 1: one launch serves both directions (the text rows' matrix is the
                            // transpose), so the row partial also takes the column-side term
  // ---- symmetric soft kernels across ranks (world > 1, DSOFT_SYM_W): column coordinates are "primed" - relative
  // to this rank's first row, so that its diagonal block comes first - and wrap around the global batch
  int wrap;                 // 0, or B: global column of primed tile t = (col0 + t * 256) mod wrap  (col0 == row0)
  int rb_half, ntiles_a;    // row blocks rb < rb_half own the primed tiles [diagonal, ntiles_a) only, the others
                            // [diagonal, ntiles): the contested half block of the rank pair (r, r + W/2)
  // ---- retrieval ranks (MODE_RANKS): rows = images (b = n_img), columns = captions (ncols = n_txt); colvec[0] =
  // the caption's threshold s_t(j),j (+inf past n_txt), colvec[1] = t(j) as int bits (rk_mapped only)
  const float* rk_p;        // per image: p_i = max over its captions of s_ij
  int* rk_img;              // += #{j : t(j) != i, s_ij > p_i}   (caller-zeroed)
  int* rk_txt;              // += #{i : i != t(j), s_ij > s_t(j),j}
  int rk_mapped;            // 0: t(j) = j (the positives are the diagonal), 1: t(j) from colvec[1]
  // ---- kNN top-k (MODE_TOPK, MODE_TOPK32): rows = queries (b = n_q), columns = keys (ncols = n_k); colvec[0] = the
  // key scale (1/||k_j||, or 1), padded to whole tiles
  const float* tk_qscale;   // per query: 1/||q_i||, or null (1)
  float* tk_val;            // [npart][b][topk_list(MODE)] partial lists, by decreasing score (ties: increasing index)
  int* tk_idx;              // their key indices (INT_MAX in slots no key filled)
  // ---- embedding geometry (MODE_GEOM): cos_ij = <a_i, b_j> * colvec[0][j] * gm_rscale[i]; one set (tri): the pairs
  // i < j; two sets: every pair but the positives (t(j) == i: colvec[1] as int bits when gm_mapped, else j == i)
  const float* gm_rscale;   // per row: 1/||a_i||
  int gm_mapped;
  float gm_kappa;           // 2 t log2(e): the pair adds 2^(kappa (cos - 1)); 0: no uniformity sum
  int gm_bins;              // 0: no histogram
  float gm_lo, gm_hi, gm_bscale;         // bin = floor((cos - lo) * bscale), bscale = bins / (hi - lo)
  unsigned long long* gm_hist;           // [bins + 2]: the bins, below lo, above hi (+= per CTA)
  double* gm_part;          // [CTAs]: this CTA's sum of the exponentials, by blockIdx.y * gridDim.x + blockIdx.x
};

struct BwdParams {
  int nprod;       // clip 1; soft 2 (teacher, then student-or-text)
  int a_map[2];
  int b_map[2];
  int kchunks[2];
  int dout;        // feature width of the gradient
  int row0, b, col0, ncols, ntiles, tiles_per_split, nsplit;
  int chunk0;      // first feature chunk of this launch (cluster rank c handles chunk0 + c)
  int row_only;    // gather_with_grad == False: gathered columns are constants
  int want_ds;     // clip: also accumulate the d(logit_scale) row term
  const float* scal;
  int tau_idx;             // soft: SC_ITS_L2 or SC_ITX_L2
  const float* lse_row;    // clip: this direction's row LSE (log2), local rows
  const float* lse_col;    // clip: other direction's LSE by global column (padded)
  const float* lse_t_row;  // soft: teacher LSE, local rows
  const float* lse_t_col;  // soft: teacher LSE by global column
  const float* lse_y_row;  // soft: student/text LSE, local rows
  const float* lse_y_col;
  const float* rinv_d;     // by global index
  const float* rinv_y;
  float* acc_part;         // [nsplit][b][dout] fp32
  float* ds_part;          // [nsplit * C * 2][b]
  // ---- weighted CE (MODE_WCE_X): products [0] CLIP (row side = direction wdir), [1] DINO; the fields mean what the
  // MODE_WCE_G fields of FwdParams mean (rinv_d: 1/||dino|| by global index, read for rows and columns)
  const float* wrow[4];    // per local row: [0] lse (log2), [1] c_a, [2] lse~ (log2), [3] A_a
  const float* wcol[4];    // by global column, of the OTHER direction: [0] lse, [1] lse~, [2] c', [3] A'
  int wdir, wsym, wrow_plain, wsplit;
  float wcc;
  float wlam[2];           // lambda_original, lambda_weighted
  const float* wgout;      // upstream gradients [6] (device)
};

// Weighted CE logit gradient of one pair (row a of direction wdir, column j), MODE_WCE_G and MODE_WCE_X:
//   g  = g_c (e1 + e2) + g_w (gimg + gtxt),  d CE~_a / d x_aj = p~_aj - beta A_a p_aj (r_aj - c_a)  (j != a)
//   gr = this row's own loss terms (world > 1 or the fused backward: the other direction's launch holds the rest)
// e1 / gimg are the row side's classic / modulated terms, e2 / gtxt the column side's (the other direction's entry of
// the same pair, statistics by column); x is the CLIP logit in log2 units, r the DINO dissimilarity.  The switches
// (wrow_plain, wsym, wsplit, row_only) are read from the kernel parameters P (FwdParams or BwdParams) at each use, as
// the kernel-parameter bank costs no registers.  g_c and g_w arrive multiplied by gk = scal[SC_WCE_GK], so that g and
// gr are the pair's entry times gk (|g gk| < 2^15 at any upstream gradient); the finalize kernel divides gk out.
struct WceRowK {
  float lse, c, lset, aa;      // row side: lse, c_a, lse~, A_a
  float beta, beta2;           // row side: beta, beta log2(e)
  float beta_t, beta2_t;       // column side
  float cc, gcl, gwt;          // c_clip, g_c gk, g_w gk
};
struct WcePair { float g, gr; };
template <class Params>
__device__ __forceinline__ WcePair wce_pair(const Params& P, const WceRowK& k, float x, float r, float lse_j,
                                            float lset_j, float c_j, float aa_j) {
  const float za = r - k.c;
  const float e1 = fast_exp2(x - k.lse);
  float gimg = e1;  // row-side direction (the image direction unless wdir == 1)
  if (!P.wrow_plain) {
    const float pt = fast_exp2(fmaf(k.beta2, fminf(fmaxf(za, -k.cc), k.cc), x) - k.lset);
    gimg = pt - k.beta * k.aa * e1 * za;
  }
  float e2 = fast_exp2(x - lse_j);
  float gtxt = e2;
  if (P.wsym) {
    const float zj = r - c_j;
    const float ptj = fast_exp2(fmaf(k.beta2_t, fminf(fmaxf(zj, -k.cc), k.cc), x) - lset_j);
    gtxt = ptj - k.beta_t * aa_j * e2 * zj;
  }
  if (P.wsplit && P.row_only) e2 = gtxt = 0.f;  // gathered columns carry no gradient
  WcePair o;
  o.g = k.gcl * (e1 + e2) + k.gwt * (gimg + gtxt);
  o.gr = P.wsplit ? k.gcl * e1 + k.gwt * gimg : o.g;
  return o;
}

__device__ __forceinline__ uint8_t* align_1024(uint8_t* p) {
  uintptr_t a = reinterpret_cast<uintptr_t>(p);
  return reinterpret_cast<uint8_t*>((a + 1023) & ~static_cast<uintptr_t>(1023));
}

// S tile (128 x n, K = 64 slice; n = 128 or 256 columns): 4 tcgen05.mma of K=16, both operands K-major
// SW128 (a 256-column B operand is two stacked 128-row boxes = 32 contiguous 8-row swizzle groups).
__device__ __forceinline__ void issue_s_stage(uint32_t tmem_d, uint32_t a_smem, uint32_t b_smem,
                                              bool first_stage, int n = BN) {
  const uint32_t idesc = make_idesc_bf16(BM, n, 0, 0);
  const uint64_t ad = make_smem_desc(a_smem, 16, 1024);
  const uint64_t bd = make_smem_desc(b_smem, 16, 1024);
#pragma unroll
  for (int kk = 0; kk < BK / 16; ++kk) {
    // advancing 16 elements (32 B) inside the 128 B swizzle row: +2 in the (addr >> 4) field
    umma_bf16(tmem_d, ad + 2 * kk, bd + 2 * kk, idesc, (first_stage && kk == 0) ? 0u : 1u);
  }
}

// Packed fp32 pairs (sm_100 FFMA2 / FMUL2 / FADD2: one issue slot and one pass through the FMA pipe for two lanes'
// worth of work).  The epilogues are issue-bound (two epilogue warps per scheduler next to the MMA stream), so their
// element loops are written over column PAIRS.
__device__ __forceinline__ float2 pk(float a, float b) { return make_float2(a, b); }
__device__ __forceinline__ float2 pk1(float a) { return make_float2(a, a); }
__device__ __forceinline__ float2 pk_mul(float2 a, float2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ float2 pk_add(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 pk_fma(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ float2 pk_exp2(float2 a) { return make_float2(fast_exp2(a.x), fast_exp2(a.y)); }

// Column sums over the 32 rows of a warp: every lane holds x[k] = the value of ITS row in column k; lane l returns
// sum over the lanes of x[l].  Butterfly: a stage keeps the half of the columns that matches the lane's bit and
// swaps the other half with the partner lane (31 shuffles; fixed order, so the result is deterministic).
__device__ __forceinline__ float warp_colsum32(float (&x)[32], int lane) {
#define DSOFT_CS_STAGE(O)                                                                   \
  {                                                                                         \
    const bool up = (lane & O) != 0;                                                        \
    _Pragma("unroll") for (int i = 0; i < O; i += 2) {                                      \
      const float send0 = up ? x[i] : x[i + O], send1 = up ? x[i + 1] : x[i + 1 + O];       \
      const float keep0 = up ? x[i + O] : x[i], keep1 = up ? x[i + 1 + O] : x[i + 1];       \
      const float2 r = pk_add(pk(keep0, keep1), pk(__shfl_xor_sync(0xffffffffu, send0, O),  \
                                                   __shfl_xor_sync(0xffffffffu, send1, O))); \
      x[i] = r.x;                                                                           \
      x[i + 1] = r.y;                                                                       \
    }                                                                                       \
  }
  DSOFT_CS_STAGE(16) DSOFT_CS_STAGE(8) DSOFT_CS_STAGE(4) DSOFT_CS_STAGE(2)
#undef DSOFT_CS_STAGE
  {
    const bool up = (lane & 1) != 0;
    const float send = up ? x[0] : x[1];
    const float keep = up ? x[1] : x[0];
    x[0] = keep + __shfl_xor_sync(0xffffffffu, send, 1);
  }
  return x[0];
}

// Column sums for the 16x256b fragment layout: lane (g = lane / 4, c2 = lane % 4) holds x[2 j + e] = the sum over ITS
// four rows of column 8 j + 2 c2 + e of a 32-column chunk; the sum over the eight row groups g comes out of three
// butterfly stages (7 shuffles).  Lane (g, c2) returns the total of column 8 (g / 2) + 2 c2 + (g % 2).
__device__ __forceinline__ float warp_colsum8(float2 (&x)[4], int lane) {
  float v[8] = {x[0].x, x[0].y, x[1].x, x[1].y, x[2].x, x[2].y, x[3].x, x[3].y};
  {
    const bool up = (lane & 16) != 0;
#pragma unroll
    for (int k = 0; k < 4; k += 2) {
      const float s0 = up ? v[k] : v[k + 4], s1 = up ? v[k + 1] : v[k + 5];
      const float k0 = up ? v[k + 4] : v[k], k1 = up ? v[k + 5] : v[k + 1];
      const float2 r = pk_add(pk(k0, k1), pk(__shfl_xor_sync(0xffffffffu, s0, 16), __shfl_xor_sync(0xffffffffu, s1, 16)));
      v[k] = r.x;
      v[k + 1] = r.y;
    }
  }
  {
    const bool up = (lane & 8) != 0;
    const float s0 = up ? v[0] : v[2], s1 = up ? v[1] : v[3];
    const float k0 = up ? v[2] : v[0], k1 = up ? v[3] : v[1];
    const float2 r = pk_add(pk(k0, k1), pk(__shfl_xor_sync(0xffffffffu, s0, 8), __shfl_xor_sync(0xffffffffu, s1, 8)));
    v[0] = r.x;
    v[1] = r.y;
  }
  {
    const bool up = (lane & 4) != 0;
    const float s0 = up ? v[0] : v[1];
    const float k0 = up ? v[1] : v[0];
    v[0] = k0 + __shfl_xor_sync(0xffffffffu, s0, 4);
  }
  return v[0];
}

// Column maxima over the 32 rows of a warp, same butterfly as warp_colsum32
__device__ __forceinline__ float warp_colmax32(float (&x)[32], int lane) {
#define DSOFT_CM_STAGE(O)                                               \
  {                                                                     \
    const bool up = (lane & O) != 0;                                    \
    _Pragma("unroll") for (int i = 0; i < O; ++i) {                     \
      const float send = up ? x[i] : x[i + O];                          \
      const float keep = up ? x[i + O] : x[i];                          \
      x[i] = fmaxf(keep, __shfl_xor_sync(0xffffffffu, send, O));        \
    }                                                                   \
  }
  DSOFT_CM_STAGE(16) DSOFT_CM_STAGE(8) DSOFT_CM_STAGE(4) DSOFT_CM_STAGE(2) DSOFT_CM_STAGE(1)
#undef DSOFT_CM_STAGE
  return x[0];
}

// SigLIP pair terms (MODE_SIGLIP).  z = s x + beta, l = +1 for the positive pair, -1 otherwise:
//   loss = softplus(-l z) = max(-l z, 0) + log1p(e),  e = 2^(-|z| log2 e)  (the one MUFU op per pair)
//   G = d loss / d z = -l sigma(-l z),  sigma(t) = r (t >= 0) or e r (t < 0),  r = 1 / (1 + e)
// r and log1p(e) run on the FMA pipe: lg2.approx of 1 + e loses ~1e-3 of the typical negative's term (e ~ 5e-5 at
// s = 10, beta = -10) to the rounding of 1 + e, and the CLIP logit-gradient kernel was MUFU-bound at one ex2 per
// pair.  r: quadratic on [1, 2] (1e-2) + two Newton steps, 1.8e-7; log1p(e) = e P7(e), 3.2e-7 relative on [0, 1].
__device__ __forceinline__ float2 sig_rcp1p(float2 e) {
  const float2 y = pk_add(e, pk1(1.f));
  float2 r = pk_fma(pk_fma(y, pk1(0.32323232f), pk1(-1.45454545f)), y, pk1(2.12121212f));
#pragma unroll
  for (int k = 0; k < 2; ++k) r = pk_fma(r, pk_fma(pk(-y.x, -y.y), r, pk1(1.f)), r);
  return r;
}
__device__ __forceinline__ float2 sig_log1p(float2 e) {
  float2 q = pk_fma(e, pk1(-0.00837115291506052f), pk1(0.04349390044808388f));
  q = pk_fma(q, e, pk1(-0.1068500280380249f));
  q = pk_fma(q, e, pk1(0.1768747717142105f));
  q = pk_fma(q, e, pk1(-0.24474774301052094f));
  q = pk_fma(q, e, pk1(0.3327192962169647f));
  q = pk_fma(q, e, pk1(-0.49997174739837646f));
  q = pk_fma(q, e, pk1(0.9999997615814209f));
  return pk_mul(q, e);
}
// two pairs at once; pos.x / pos.y: the pair is a positive.  Returns the loss terms, G in g.
__device__ __forceinline__ float2 siglip_pair2(float2 z, bool pos_x, bool pos_y, float2& g) {
  const float L2E = 1.4426950408889634f;
  const float2 e = pk_exp2(pk_mul(pk(fabsf(z.x), fabsf(z.y)), pk1(-L2E)));
  const float2 r = sig_rcp1p(e);
  const float2 er = pk_mul(e, r);
  const float tx = pos_x ? -z.x : z.x, ty = pos_y ? -z.y : z.y;  // -l z
  const float sx = tx >= 0.f ? r.x : er.x, sy = ty >= 0.f ? r.y : er.y;
  g = pk(pos_x ? -sx : sx, pos_y ? -sy : sy);
  return pk_add(pk(fmaxf(tx, 0.f), fmaxf(ty, 0.f)), sig_log1p(e));
}

// ================================================================================================
// Forward: per-row soft-max statistics
// ================================================================================================
//  MODE_CLIP partials (2): running max m (log2 units), sum 2^(x-m)        [+ diag dot product]
//  MODE_SOFT partials (7): teacher m, Zt, Aq=sum w*q, Ap=sum w*p, Ar=sum w*r, student Zs, text Ztt
//  (w = 2^(q-m); student/text use the fixed maximum log2(e)/tau, reached on the diagonal.)
// The kernel runs as clusters of two CTAs (consecutive row blocks) that drive cta_group::2 MMAs (M = 256): each
// CTA loads its own 128 rows of the row-side operand and HALF of the column-side tile, the leader issues one MMA for
// both.
//
// Tile width.  What bounds these kernels is the L2 -> SM operand stream (~6300 B/clk for the whole chip, i.e.
// ~42 B/clk per SM): an M=256 x N=128 pair tile with a streamed row operand pulls 24 KiB per CTA per 64-deep K
// step = 96 B/clk at the full MMA rate (round 1: 49 % tensor activity, 11.3 TB/s from L2), an M=256 x N=256 tile
// 32 KiB per twice the math = 64 B/clk (the gradient GEMM's ratio: 93 %).  All modes therefore run 256-column
// tiles: two TMEM slots of 256 columns, every epilogue thread owns one row x 128 columns of each product.  The
// soft epilogues keep the teacher strip of those 128 columns in registers across the student and text products
// (w / E below); setmaxnreg moves the registers the producer / MMA / allocator warps do not need to the two
// epilogue warpgroups (56 / 216 per thread).
//
// Epilogue warps.  Eight (two per TMEM lane quadrant, 128-column strips) everywhere except MODE_CLIP_SYM, whose
// epilogue is a chain of short dependent steps (chunk maximum -> warp reduction -> exponentials -> 5-stage shuffle
// butterfly): with two warps per scheduler it issued 23 % of the time and took 8200 clocks per tile against 5700 of
// MMA time.  It runs SIXTEEN epilogue warps (four per quadrant, 64-column strips, 640 threads per CTA, <= 96
// registers) so that four warps per scheduler hide each other's latencies.  (Tried for MODE_CLIP_G as well, with
// 32-column half-box G stores so that the staging strips still fit: 1.17 ms against 1.04 ms - dropped.)

// Per-column vectors the producer stages per tile for the epilogue (bulk copies into shared memory, COL_BUFS tiles
// deep, read as shared-memory broadcasts instead of dependent global loads per 32-column chunk)
enum FwdCols {
  COLS_NONE,
  COLS_RINV,         // P.rinv[p] per product: inverse column norms
  COLS_RINV_COLFAC,  // P.rinv[p] and P.colfac[p] (at vector 3 + p): the soft logit gradient
  COLS_COLVEC        // P.colvec[0 .. ncolvec)
};
struct FwdMode {
  int stages;     // operand ring depth in 32 KiB stages, with the column buffers (and the G strips) behind the ring;
                  // 0: as deep as the shared memory allows (see the kernel)
  int g_stage;    // the G staging strips start at g_stage * 32 KiB, behind the ring (modes that write G)
  FwdCols cols;
  bool writes_g;  // streams fp16 logit-gradient tiles through TMA stores (maps.g, L2 policies)
  bool regsplit;  // setmaxnreg hand-over (40 / 232) from the producer / MMA / allocator warps to the epilogue; the
                  // ranks, distill, kNN and geometry epilogues fit the even split (168 registers) without spills
  int epi_warps;
};
__host__ __device__ constexpr FwdMode fwd_mode(int mode) {
  switch (mode) {
    case MODE_SOFT:
    case MODE_SOFT_SYM16: return {6, 6, COLS_RINV, false, true, 8};
    case MODE_SOFT_G: return {5, 5, COLS_RINV_COLFAC, true, true, 8};
    case MODE_WCE_STAT:
    case MODE_WCE_LSE:
    case MODE_WCE_DBG:
    case MODE_PAIRS: return {6, 6, COLS_COLVEC, false, true, 8};
    case MODE_WCE_G: return {5, 5, COLS_COLVEC, true, true, 8};
    case MODE_RANKS:
    case MODE_TOPK:
    case MODE_TOPK32:
    case MODE_GEOM:
    case MODE_DIST_FWD: return {6, 6, COLS_COLVEC, false, false, 8};
    case MODE_DIST_G: return {5, 5, COLS_COLVEC, true, false, 8};
    case MODE_CLIP_G:
    case MODE_SIGLIP: return {0, 6, COLS_NONE, true, false, 8};
    case MODE_CLIP_SYM: return {0, 6, COLS_NONE, false, false, 16};
    default: return {0, 6, COLS_NONE, false, false, 8};  // MODE_CLIP, MODE_RAW, MODE_LINEAR
  }
}
__host__ __device__ constexpr int fwd_epi_warps(int mode) { return fwd_mode(mode).epi_warps; }

// Histogram slot of a cosine (MODE_GEOM and the positives' pre-pass): bins equal-width over [lo, hi), the last one
// closed (numpy.histogram's convention); nb: below lo, nb + 1: above hi
__device__ __forceinline__ int geom_bin(float x, float lo, float hi, float bscale, int nb) {
  return x < lo ? nb : (x > hi ? nb + 1 : min(static_cast<int>((x - lo) * bscale), nb - 1));
}
__host__ __device__ constexpr int fwd_threads(int mode) { return 32 * (EPI_WARP0 + fwd_epi_warps(mode)); }

template <int MODE, int CG>
__global__ void __launch_bounds__(fwd_threads(MODE), 1)
dsoft_fwd_kernel(const __grid_constant__ TileMaps maps, const __grid_constant__ FwdParams P) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align_1024(smem_raw);
  static_assert(CG == 2, "the forward kernel runs as CTA pairs");
  constexpr FwdMode kM = fwd_mode(MODE);
  constexpr int kEpiThreads = 32 * kM.epi_warps;
  // epilogue families (the shared part below reads only kM)
  constexpr bool kWce = (MODE >= MODE_WCE_STAT && MODE <= MODE_WCE_G);
  constexpr bool kDist = (MODE == MODE_DIST_FWD || MODE == MODE_DIST_G);
  // streaming mode: stages of (A box | B boxes); resident mode: 8 A boxes, then B-only stages
  const bool resident = P.resident != 0;
  const int bn = P.bn;
  const int brows = bn / CG;  // column-operand rows this CTA stages per tile
  const int boxr = 64;        // rows per TMA box (maps are built accordingly)
  const int box_bytes = boxr * 128;
  const int stage_bytes = (resident ? 0 : TILE_BYTES) + brows * 128;
  // Ring depth.  Modes with column vectors: 6 stages of 32 KiB with the staged vectors behind them (logit-gradient
  // modes: 5 stages, the G staging strips right behind them).  The others: as many stages as fit (at most 8); the
  // logit-gradient ones stop at the G staging strips (g_stage * 2 boxes of 16 KiB: streaming stages take two boxes,
  // resident ones one box of the 256-column tile behind the 8 resident boxes).
  static_assert(!kM.writes_g || kM.stages == 0 || kM.stages == kM.g_stage, "G strips right behind the ring");
  const int nstages = kM.stages ? kM.stages
                                : min(kM.writes_g ? (resident ? 2 * kM.g_stage - 8 : kM.g_stage) : 8,
                                      (resident ? 6 : 14) * TILE_BYTES / stage_bytes);
  // G staging: one 4 KiB strip (32 rows x 64 columns fp16, 128-byte swizzle) per epilogue warp.  A strip is written
  // with conflict-free 16-byte shared stores and leaves through ONE TMA tensor store; per-thread 32-byte global
  // stores (32 different lines per warp instruction) kept the L1TEX pipe at 78 % and the tensor pipe at 62 %.
  uint8_t* gstage = smem + kM.g_stage * 2 * TILE_BYTES;
  const int nslots = TMEM_COLS / bn;  // 4 x 128 or 2 x 256 columns
  uint8_t* ring = resident ? smem + 8 * TILE_BYTES : smem;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + F_STAGES * 2 * TILE_BYTES + 2 * TILE_BYTES);
  uint64_t* ring_full = bars;        // [8]  (the leader's copy collects both CTAs' bytes)
  uint64_t* ring_empty = bars + 8;   // [8]
  uint64_t* s_full = bars + 16;
  uint64_t* s_empty = s_full + F_SLOTS;  // (the leader's copy collects both CTAs' epilogues)
  uint64_t* a_full = s_empty + F_SLOTS;
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(a_full + 1);
  // the per-column vectors of a tile (kM.cols; 256 columns each) are staged by the producer with bulk copies,
  // COL_BUFS tiles deep.  The epilogue reads them as shared-memory broadcasts instead of dependent global loads per
  // 32-column chunk.
  constexpr int COL_VECS = 6, COL_BUFS = 2, CT = 256;
  float* colbuf = reinterpret_cast<float*>(smem + 6 * 2 * TILE_BYTES);            // [COL_BUFS][COL_VECS][256]
  uint64_t* col_full = reinterpret_cast<uint64_t*>(colbuf + COL_BUFS * COL_VECS * CT);  // [COL_BUFS]
  uint64_t* col_empty = col_full + COL_BUFS;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int rb = blockIdx.x;
  const int split = blockIdx.y;
  // triangular mode (soft G, world == 1, 256-column tiles): a row pair only computes the tiles from its own
  // diagonal tile onwards.  Column chunks are aligned from the END of the row for every row pair, so that the
  // CTAs of one chunk index (launched next to each other) stream the same column tiles at the same time and
  // share them in L2; a pair's lowest chunk is cut at its diagonal tile and the chunks left of it are empty
  int t0 = split * P.tiles_per_split;
  int t1 = min(t0 + P.tiles_per_split, P.ntiles);
  if (P.tri) {
    const int tend = (rb < P.rb_half) ? P.ntiles_a : P.ntiles;  // both CTAs of a pair lie in the same half
    t1 = tend - split * P.tiles_per_split;
    t0 = max(t1 - P.tiles_per_split, rb >> 1);  // may be >= t1: nothing to do
  }
  // global column of the first column of (primed) tile t; without wrap the two coincide up to col0
  auto gcol = [&](int t) { return P.wrap ? (P.col0 + t * P.bn) % P.wrap : P.col0 + t * P.bn; };
  const int prank = rb & 1;  // rank in the pair (== cluster rank)
  const bool leader = prank == 0;

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < 4; ++i) tma_prefetch_desc(&maps.m[i]);
    if constexpr (kM.writes_g) {
      tma_prefetch_desc(&maps.g[0]);
      tma_prefetch_desc(&maps.g[1]);
    }
    for (int i = 0; i < 8; ++i) {
      mbar_init(smem_u32(&ring_full[i]), 1);
      mbar_init(smem_u32(&ring_empty[i]), 1);
    }
    for (int i = 0; i < F_SLOTS; ++i) {
      mbar_init(smem_u32(&s_full[i]), 1);
      mbar_init(smem_u32(&s_empty[i]), CG * kEpiThreads);
    }
    mbar_init(smem_u32(a_full), 1);
    if constexpr (kM.cols != COLS_NONE) {
      for (int i = 0; i < COL_BUFS; ++i) {
        mbar_init(smem_u32(&col_full[i]), 1);
        mbar_init(smem_u32(&col_empty[i]), NUM_EPI_THREADS);
      }
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc_cg<CG>(smem_u32(tmem_holder), TMEM_COLS);
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  // the register hand-over sits INSIDE the role branches: ptxas budgets the code dominated by a setmaxnreg with
  // its value (placed before the branch it compiled the whole kernel, epilogues included, for 56 registers)
  if (warp < EPI_WARP0) {
  if constexpr (kM.regsplit) setmaxnreg_dec<40>();
  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer (warp-uniform loop)
    int stage = 0;
    uint32_t phase = 0;
    // logit-gradient modes: the operands must survive the G store stream in L2
    const uint64_t pol_keep = kM.writes_g ? l2_policy_evict_last() : 0ull;
    auto load = [&](uint32_t dst, const CUtensorMap* m, uint32_t bar_local, int c0, int c1) {
      // fwd_mode(MODE), not kM: nvcc rejects a member of the enclosing constexpr local in this lambda's if constexpr
      if constexpr (fwd_mode(MODE).writes_g) tma_load_2d_2sm_hint(dst, m, mapa_shared(bar_local, 0), c0, c1, pol_keep);
      else tma_load_2d_2sm(dst, m, mapa_shared(bar_local, 0), c0, c1);
    };
    if (resident && elect_one()) {
      const uint32_t af = smem_u32(a_full);
      if (leader) mbar_arrive_expect_tx(af, CG * P.kchunks[0] * TILE_BYTES);
      for (int kc = 0; kc < P.kchunks[0]; ++kc)
        for (int i = 0; i < BM / boxr; ++i)
          load(smem_u32(smem + kc * TILE_BYTES + i * box_bytes), &maps.m[P.a_map[0]], af, kc * BK,
               P.row0 + rb * BM + i * boxr);
    }
    __syncwarp();
    for (int t = t0; t < t1; ++t) {
      if constexpr (kM.cols != COLS_NONE) {
        const int n = t - t0;
        const int cb = n % COL_BUFS;
        mbar_wait(smem_u32(&col_empty[cb]), ((static_cast<uint32_t>(n / COL_BUFS)) & 1) ^ 1);
        if (elect_one()) {
          const uint32_t full = smem_u32(&col_full[cb]);
          const int nvec = kM.cols == COLS_COLVEC ? P.ncolvec : (kM.cols == COLS_RINV_COLFAC ? 2 : 1) * P.nprod;
          mbar_arrive_expect_tx(full, nvec * CT * 4);
          float* dst = colbuf + cb * COL_VECS * CT;
          const size_t c0 = static_cast<size_t>(gcol(t));  // CT == bn == 256 in the modes with column vectors
          if constexpr (kM.cols == COLS_COLVEC) {
            for (int k = 0; k < P.ncolvec; ++k) bulk_copy_g2s(smem_u32(dst + k * CT), P.colvec[k] + c0, CT * 4, full);
          } else {
            for (int p = 0; p < P.nprod; ++p) {
              bulk_copy_g2s(smem_u32(dst + p * CT), P.rinv[p] + c0, CT * 4, full);
              if constexpr (kM.cols == COLS_RINV_COLFAC)
                bulk_copy_g2s(smem_u32(dst + (3 + p) * CT), P.colfac[p] + c0, CT * 4, full);
            }
          }
        }
        __syncwarp();
      }
      for (int p = 0; p < P.nprod; ++p) {
        const CUtensorMap* am = &maps.m[P.a_map[p]];
        const CUtensorMap* bm = &maps.m[P.b_map[p]];
        for (int kc = 0; kc < P.kchunks[p]; ++kc) {
          mbar_wait(smem_u32(&ring_empty[stage]), phase ^ 1);
          if (elect_one()) {
            const uint32_t full = smem_u32(&ring_full[stage]);
            const uint32_t dst = smem_u32(ring + stage * stage_bytes);
            if (leader) mbar_arrive_expect_tx(full, CG * stage_bytes);  // both CTAs' boxes land on this barrier
            uint32_t bdst = dst;
            if (!resident) {
              for (int i = 0; i < BM / boxr; ++i)
                load(dst + i * box_bytes, am, full, kc * BK, P.row0 + rb * BM + i * boxr);
              bdst += TILE_BYTES;
            }
            for (int i = 0; i < brows / boxr; ++i)
              load(bdst + i * box_bytes, bm, full, kc * BK, gcol(t) + prank * brows + i * boxr);
          }
          __syncwarp();
          if (++stage == nstages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (leader CTA only)
    if (leader) {
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      const uint32_t idesc = make_idesc_bf16(BM * CG, bn, 0, 0);
      if (resident) {
        mbar_wait(smem_u32(a_full), 0);
        tc_fence_after();
      }
      for (int t = t0; t < t1; ++t) {
        for (int p = 0; p < P.nprod; ++p, ++it) {
          const int slot = it % nslots;
          const uint32_t use = static_cast<uint32_t>(it / nslots);
          mbar_wait(smem_u32(&s_empty[slot]), (use & 1) ^ 1);
          tc_fence_after();
          const uint32_t tmem_d = tmem_base + slot * bn;
          for (int kc = 0; kc < P.kchunks[p]; ++kc) {
            mbar_wait(smem_u32(&ring_full[stage]), phase);
            tc_fence_after();
            if (elect_one()) {
              const uint32_t st_smem = smem_u32(ring + stage * stage_bytes);
              const uint32_t a_smem = resident ? smem_u32(smem + kc * TILE_BYTES) : st_smem;
              const uint32_t b_smem = resident ? st_smem : st_smem + TILE_BYTES;
              const uint64_t ad = make_smem_desc(a_smem, 16, 1024);
              const uint64_t bd = make_smem_desc(b_smem, 16, 1024);
#pragma unroll
              for (int kk = 0; kk < BK / 16; ++kk)
                umma_cg<CG>(tmem_d, ad + 2 * kk, bd + 2 * kk, idesc, (kc == 0 && kk == 0) ? 0u : 1u);
              umma_commit_cg<CG>(smem_u32(&ring_empty[stage]));
              if (kc == P.kchunks[p] - 1) umma_commit_cg<CG>(smem_u32(&s_full[slot]));
            }
            __syncwarp();
            if (++stage == nstages) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  }
  } else {
    // ------------------------------------------------------------------ epilogue
    if constexpr (kM.regsplit) setmaxnreg_inc<232>();
    const int q = warp & 3;
    const int half = (warp - EPI_WARP0) >> 2;
    const int row = q * 32 + lane;
    const int li = rb * BM + row;  // local row
    const int gi = P.row0 + li;    // global index of this row
    const int gw0 = P.row0 + rb * BM + q * 32;  // first global row of this warp (diagonal test, warp-uniform)
    const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const int sp = split * 2 + half;
    float v[32];
    // ---- G staging (logit-gradient modes): this warp's strip, its swizzled row, and the TMA store of a finished
    // 64-column box.  Strip reuse: the issuing lane waits until its previous store has read the strip.
    const uint64_t pol_stream = kM.writes_g ? l2_policy_evict_first() : 0ull;  // G tiles: written once, read once later
    const uint32_t gs_base = smem_u32(gstage) + static_cast<uint32_t>(warp - EPI_WARP0) * 4096u;
    const uint32_t gs_row = gs_base + static_cast<uint32_t>(lane) * 128u;
    const int gsw = lane & 7;
    auto stage_begin = [&]() {  // before the first write of a box
      if (lane == 0) bulk_wait_group_read<0>();
      __syncwarp();
    };
    auto stage_put32 = [&](const uint32_t (&w16)[16], int chalf) {  // 32 fp16 pairs = columns chalf * 32 .. + 32
#pragma unroll
      for (int k4 = 0; k4 < 4; ++k4)
        st_shared_v4(gs_row + (((chalf * 4 + k4) ^ gsw) << 4), w16[4 * k4], w16[4 * k4 + 1], w16[4 * k4 + 2],
                     w16[4 * k4 + 3]);
    };
    auto stage_store = [&](const CUtensorMap* gm, int box_row) {  // after the second half of a box is written
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        tma_store_2d_hint(gm, gs_base, 0, box_row, pol_stream);
        bulk_commit_group();
      }
    };
    auto release_slot = [&](int slot) {  // the MMA issuer lives in the pair's leader
      // relaxed: a .release arrive is a MEMBAR that waits for every earlier memory operation of the thread (ncu:
      // "membar" was the top stall of the soft epilogue, and with the G stores in flight it serialised the G
      // kernels).  The barrier only hands back TMEM, whose reads are complete (tcgen05.wait::ld) and ordered by
      // fence::before_thread_sync.
      mbar_arrive_cluster_relaxed(mapa_shared(smem_u32(&s_empty[slot]), 0));
    };

    if constexpr (MODE == MODE_RAW) {
      int it = 0;
      for (int t = t0; t < t1; ++t, ++it) {
        const int slot = it % nslots;
        const uint32_t use = static_cast<uint32_t>(it / nslots);
        mbar_wait(smem_u32(&s_full[slot]), use & 1);
        tc_fence_after();
#pragma unroll 1
        for (int c = 0; c < bn / 64; ++c) {
          const int jrel0 = t * bn + half * (bn / 2) + c * 32;
          tmem_ld32(lane_addr + slot * bn + half * (bn / 2) + c * 32, v);
          if (li < P.b) {
#pragma unroll
            for (int e = 0; e < 32; ++e)
              if (jrel0 + e < P.ncols) P.part[static_cast<size_t>(li) * P.ncols + jrel0 + e] = v[e];
          }
        }
        tc_fence_before();
        release_slot(slot);
      }
    } else if constexpr (MODE == MODE_CLIP) {
      const float s2 = P.scal[SC_SCALE_L2];
      const float2 s22 = pk1(s2);
      float m = M_FLOOR, sum = 0.f, dg = 0.f;
      bool have_dg = false;
      int it = 0;
      for (int t = t0; t < t1; ++t, ++it) {
        const int slot = it % nslots;
        const uint32_t use = static_cast<uint32_t>(it / nslots);
        mbar_wait(smem_u32(&s_full[slot]), use & 1);
        tc_fence_after();
#pragma unroll 1
        for (int c = 0; c < bn / 64; ++c) {
          const int jrel0 = t * bn + half * (bn / 2) + c * 32;
          const int gj0 = P.col0 + jrel0;
          tmem_ld32(lane_addr + slot * bn + half * (bn / 2) + c * 32, v);
          if (gi >= gj0 && gi < gj0 + 32) {
#pragma unroll
            for (int e = 0; e < 32; ++e)
              if (gj0 + e == gi) dg = v[e];
            have_dg = true;
          }
          float x[32];
#pragma unroll
          for (int e = 0; e < 32; e += 2) {
            const float2 xx = pk_mul(pk(v[e], v[e + 1]), s22);
            x[e] = xx.x;
            x[e + 1] = xx.y;
          }
          if (jrel0 + 32 > P.ncols) {
#pragma unroll
            for (int e = 0; e < 32; ++e)
              if (jrel0 + e >= P.ncols) x[e] = NEG_BIG;
          }
          float cm[4] = {x[0], x[1], x[2], x[3]};
#pragma unroll
          for (int e = 4; e < 32; ++e) cm[e & 3] = fmaxf(cm[e & 3], x[e]);
          const float mnew = fmaxf(m, fmaxf(fmaxf(cm[0], cm[1]), fmaxf(cm[2], cm[3])));
          const float2 nm2 = pk1(-mnew);
          float2 acc[2] = {pk1(0.f), pk1(0.f)};
#pragma unroll
          for (int e = 0; e < 32; e += 2)
            acc[(e >> 1) & 1] = pk_add(acc[(e >> 1) & 1], pk_exp2(pk_add(pk(x[e], x[e + 1]), nm2)));
          sum = sum * fast_exp2(m - mnew) + ((acc[0].x + acc[0].y) + (acc[1].x + acc[1].y));
          m = mnew;
        }
        tc_fence_before();
        release_slot(slot);
      }
      if (li < P.b) {
        P.part[(0 * P.npart + sp) * P.b + li] = m;
        P.part[(1 * P.npart + sp) * P.b + li] = sum;
        if (have_dg && P.diag) P.diag[li] = dg;
      }
    } else if constexpr (MODE == MODE_PAIRS) {
      // ---------------------------------------------------------------- CLIP-blind pair statistics
      // helpers.py:221-285 (_pair_stats): cs = Z Z^T, ds = D D^T for L2-normalised rows, over the pairs i < j:
      // how many have cs >= cmin, how many of those have ds <= dmax ("blind": CLIP calls them similar, DINOv2 does
      // not), and the pairs with the largest gap cs - ds.  Upper block triangle only (P.tri); the CLIP tile waits
      // in registers for the DINO tile; counts are exact integers (warp sum -> one 64-bit atomic per warp at the
      // end); candidates above the gap floor are appended through one warp-aggregated atomic per chunk.
      float xq[128];
      unsigned int chi[8], cbl[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) chi[k] = cbl[k] = 0u;
      const bool live_row = li < P.b;
      const bool counting = P.pr_counts != nullptr;
      const float floor_gap = P.pr_gap_floor;
      int it = 0;
      for (int t = t0; t < t1; ++t, it += 2) {
        const int jt0 = t * CT + half * 128;
        const int cb = (t - t0) % COL_BUFS;
        mbar_wait(smem_u32(&col_full[cb]), static_cast<uint32_t>((t - t0) / COL_BUFS) & 1);
        {  // ---- CLIP Gram tile -> xq
          const int slot = it % 2;
          mbar_wait(smem_u32(&s_full[slot]), static_cast<uint32_t>(it / 2) & 1);
          tc_fence_after();
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            tmem_ld32(lane_addr + slot * CT + half * 128 + c * 32, v);
#pragma unroll
            for (int e = 0; e < 32; ++e) xq[c * 32 + e] = v[e];
          }
          tc_fence_before();
          release_slot(slot);
        }
        {  // ---- DINO Gram tile
          const int slot = (it + 1) % 2;
          mbar_wait(smem_u32(&s_full[slot]), static_cast<uint32_t>((it + 1) / 2) & 1);
          tc_fence_after();
#pragma unroll 1
          for (int c = 0; c < 4; ++c) {
            const int jrel0 = jt0 + c * 32;
            tmem_ld32(lane_addr + slot * CT + half * 128 + c * 32, v);
            if (c == 3) {
              tc_fence_before();
              release_slot(slot);
            }
            // pairs i < j only; the whole chunk is out when its last column is not right of the warp's first row
            if (jrel0 + 31 <= gw0 || jrel0 >= P.ncols) continue;  // warp-uniform
            const bool edge = jrel0 <= gw0 + 31 || jrel0 + 32 > P.ncols || !live_row ||
                              rb * BM + q * 32 + 32 > P.b;      // warp-uniform: some entries need the mask
#pragma unroll
            for (int e = 0; e < 32; ++e) {
              // the chunk's CLIP values sit at a runtime offset of xq: select them with a static index
              const float cs = (c == 0) ? xq[e] : (c == 1) ? xq[32 + e] : (c == 2) ? xq[64 + e] : xq[96 + e];
              const float ds = v[e];
              const bool ok = !edge || (jrel0 + e > gi && jrel0 + e < P.ncols && live_row);
              if (counting) {
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                  if (k < P.pr_nthr) {
                    const bool hi = ok && cs >= P.pr_cmin[k];
                    chi[k] += hi ? 1u : 0u;
                    cbl[k] += (hi && ds <= P.pr_dmax[k]) ? 1u : 0u;
                  }
                }
              }
              const bool cand = ok && (cs - ds) >= floor_gap;
              const unsigned int mask = __ballot_sync(0xffffffffu, cand);
              if (mask) {
                unsigned int base = 0;
                const int leader = __ffs(mask) - 1;
                if (lane == leader) base = atomicAdd(P.pr_cand_count, __popc(mask));
                base = __shfl_sync(0xffffffffu, base, leader);
                if (cand) {
                  const unsigned int idx = base + __popc(mask & ((1u << lane) - 1u));
                  if (idx < P.pr_cand_cap)
                    P.pr_cand[idx] = make_float4(__int_as_float(gi), __int_as_float(jrel0 + e), cs, ds);
                }
              }
            }
          }
        }
        mbar_arrive(smem_u32(&col_empty[cb]));
      }
      if (counting) {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          if (k < P.pr_nthr) {
            const unsigned int a = __reduce_add_sync(0xffffffffu, chi[k]);
            const unsigned int bsum = __reduce_add_sync(0xffffffffu, cbl[k]);
            if (lane == 0) {
              if (a) atomicAdd(P.pr_counts + 2 * k + 0, static_cast<unsigned long long>(a));
              if (bsum) atomicAdd(P.pr_counts + 2 * k + 1, static_cast<unsigned long long>(bsum));
            }
          }
        }
      }
    } else if constexpr (MODE == MODE_RANKS) {
      // ---------------------------------------------------------------- retrieval ranks
      // open_clip get_clip_metrics as counts over s = I . T^T (rows = images, columns = captions): a pair (i, j) is
      // the positive when t(j) == i (1:1: the diagonal, warp-uniform per 32 x 32 chunk); every other pair counts
      //   for image i   when s_ij > p_i       (row count, a register across this CTA's tiles, one atomic at the end)
      //   for caption j when s_ij > thr_j     (ballot over the warp's 32 rows, summed over the CTA's 4 warps of a
      //                                        column strip in shared memory, one atomic per column and tile)
      // Integer sums: the result does not depend on the order of the atomics.  colsum is double-buffered by tile
      // parity, so one named barrier per tile separates the shared sums of a tile from their flush.
      int* colsum = reinterpret_cast<int*>(smem + 6 * 2 * TILE_BYTES + 16384);  // [2][256], behind colbuf
      const int et = threadIdx.x - 32 * EPI_WARP0;                              // 0 .. 255
      colsum[et] = 0;
      colsum[CT + et] = 0;
      named_bar_sync(1, NUM_EPI_THREADS);
      const bool live_row = li < P.b;
      const float prow = live_row ? P.rk_p[li] : 0.f;
      const bool mapped = P.rk_mapped != 0;
      unsigned int rcount = 0;
      int it = 0;
      for (int t = t0; t < t1; ++t, ++it) {
        const int slot = it % nslots;
        const int cb = it % COL_BUFS;
        mbar_wait(smem_u32(&col_full[cb]), static_cast<uint32_t>(it / COL_BUFS) & 1);
        mbar_wait(smem_u32(&s_full[slot]), static_cast<uint32_t>(it / nslots) & 1);
        tc_fence_after();
        const float* thr = colbuf + cb * COL_VECS * CT;
        const int* tmap = reinterpret_cast<const int*>(thr + CT);
        int* csum = colsum + (it & 1) * CT;
#pragma unroll 1
        for (int c = 0; c < 4; ++c) {
          const int jt = half * 128 + c * 32;  // column in the tile
          const int gj0 = t * CT + jt;
          tmem_ld32(lane_addr + slot * CT + jt, v);
          if (c == 3) {
            tc_fence_before();
            release_slot(slot);
          }
          if (gj0 >= P.ncols) continue;                 // warp-uniform
          const bool ragged = gj0 + 32 > P.ncols;      // warp-uniform
          unsigned int mine = 0;
          if (mapped) {
#pragma unroll
            for (int e = 0; e < 32; ++e) {
              const bool other = tmap[jt + e] != gi && (!ragged || gj0 + e < P.ncols);
              rcount += (other && v[e] > prow) ? 1u : 0u;
              const unsigned int bal = __ballot_sync(0xffffffffu, other && live_row && v[e] > thr[jt + e]);
              if (lane == e) mine = __popc(bal);
            }
          } else {
            const bool diag = gj0 == gw0;  // warp-uniform: rows and chunks are both 32-aligned
#pragma unroll
            for (int e = 0; e < 32; ++e) {
              const bool other = !(diag && lane == e) && (!ragged || gj0 + e < P.ncols);
              rcount += (other && v[e] > prow) ? 1u : 0u;
              const unsigned int bal = __ballot_sync(0xffffffffu, other && live_row && v[e] > thr[jt + e]);
              if (lane == e) mine = __popc(bal);
            }
          }
          if (mine) atomicAdd(csum + jt + lane, static_cast<int>(mine));
        }
        mbar_arrive(smem_u32(&col_empty[cb]));
        named_bar_sync(1, NUM_EPI_THREADS);
        const int s = csum[et];
        if (s) {
          atomicAdd(P.rk_txt + t * CT + et, s);  // s > 0 only for columns < ncols (thr = +inf past them)
          csum[et] = 0;
        }
      }
      if (live_row && rcount) atomicAdd(P.rk_img + li, static_cast<int>(rcount));
    } else if constexpr (MODE == MODE_TOPK || MODE == MODE_TOPK32) {
      // ---------------------------------------------------------------- kNN top-k
      // s_ij = <q_i, k_j> (rows = queries, columns = keys) times the staged key scale and this row's query scale.
      // Each thread keeps the KL best (score, key index) of its row and 128-column strip in registers, sorted by
      // decreasing score.  Keys reach a thread in increasing index order, so a score enters only when it is strictly
      // above the list's last entry, and a listed equal score stays ahead of it: ties keep the smaller key index.
      // One compare per score builds the chunk's survivor mask (usually empty once the list has filled).  A chunk
      // with survivors is parked in this thread's slice of shared memory, which frees u[] for the insertion; each
      // survivor is read back and inserted with static list indices only, so the list never leaves the registers.
      // Chunks are CW columns wide, 16 for a 32-entry list and 8 for a 64-entry one: next to the 2 KL list registers,
      // wider chunks do not fit the even register split (168) without spills.  Both scales are applied here, before
      // any comparison, so that the lists and the merge order exactly the values that are returned.
      constexpr int KL = topk_list(MODE);
      constexpr int CW = KL == 64 ? 8 : 16;
      float tv[KL], u[CW];
      int ti[KL];
#pragma unroll
      for (int k = 0; k < KL; ++k) {
        tv[k] = __int_as_float(static_cast<int>(0xff800000u));  // -inf: no score is below it
        ti[k] = 0x7fffffff;
      }
      const float qs = (P.tk_qscale && li < P.b) ? P.tk_qscale[li] : 1.f;
      // 256-column tiles: two TMEM slots and two column buffers, both picked by the parity of the tile's position
      for (int t = t0; t < t1; ++t) {
        const int n = t - t0, par = n & 1;
        mbar_wait(smem_u32(&col_full[par]), static_cast<uint32_t>(n >> 1) & 1);
        mbar_wait(smem_u32(&s_full[par]), static_cast<uint32_t>(n >> 1) & 1);
        tc_fence_after();
        const float* ks = colbuf + par * COL_VECS * CT + half * 128;
        const uint32_t taddr = lane_addr + par * CT + half * 128;
        const int gcol0 = t * CT + half * 128;
#pragma unroll 1
        for (int c = 0; c < 128 / CW; ++c) {
          const int gj0 = gcol0 + c * CW;
          if constexpr (CW == 16) tmem_ld16(taddr + c * CW, u);
          else tmem_ld8(taddr + c * CW, u);
          if (c == 128 / CW - 1) {
            tc_fence_before();
            release_slot(par);
          }
          if (gj0 >= P.ncols) continue;  // warp-uniform
          const float lo = tv[KL - 1];
          unsigned int m = 0;
#pragma unroll
          for (int e = 0; e < CW; ++e) {
            u[e] = (u[e] * ks[c * CW + e]) * qs;
            m |= (u[e] > lo) ? (1u << e) : 0u;
          }
          if (gj0 + CW > P.ncols) m &= (1u << (P.ncols - gj0)) - 1u;  // columns past n_k never enter
          float* stash = reinterpret_cast<float*>(smem + 6 * 2 * TILE_BYTES + 16384)  // [256][CW], behind colbuf
                         + (threadIdx.x - 32 * EPI_WARP0) * CW;
          if (m) {
#pragma unroll
            for (int e = 0; e < CW; e += 4)
              reinterpret_cast<float4*>(stash)[e / 4] = make_float4(u[e], u[e + 1], u[e + 2], u[e + 3]);
          }
          while (m) {
            const int e = __ffs(m) - 1;
            m &= m - 1u;
            const float x = stash[e];
            const int xj = gj0 + e;
            // new[i] = old[i-1] if old[i-1] < x, else x if old[i] < x, else old[i] (a no-op when x <= old[KL-1])
#pragma unroll
            for (int i = KL - 1; i > 0; --i) {
              const bool up = tv[i - 1] < x, here = tv[i] < x;
              tv[i] = up ? tv[i - 1] : (here ? x : tv[i]);
              ti[i] = up ? ti[i - 1] : (here ? xj : ti[i]);
            }
            if (tv[0] < x) {
              tv[0] = x;
              ti[0] = xj;
            }
          }
        }
        mbar_arrive(smem_u32(&col_empty[par]));
      }
      if (li < P.b) {
        const size_t o = (static_cast<size_t>(sp) * P.b + li) * KL;
        float4* dv = reinterpret_cast<float4*>(P.tk_val + o);
        int4* di = reinterpret_cast<int4*>(P.tk_idx + o);
#pragma unroll
        for (int k = 0; k < KL / 4; ++k) {
          dv[k] = make_float4(tv[4 * k], tv[4 * k + 1], tv[4 * k + 2], tv[4 * k + 3]);
          di[k] = make_int4(ti[4 * k], ti[4 * k + 1], ti[4 * k + 2], ti[4 * k + 3]);
        }
      }
    } else if constexpr (MODE == MODE_GEOM) {
      // ---------------------------------------------------------------- embedding geometry
      // cos = <a_i, b_j> times the staged column scale and this row's scale, over the pairs in scope: one set (P.tri,
      // upper block triangle) the pairs i < j, two sets every pair but the positives (masked as in MODE_RANKS).  Per
      // pair, 2^(kappa (cos - 1)) goes into fp32 sums per tile (at most 128 terms <= 1 per thread), promoted to fp64
      // across tiles: a thread sees 10^5 - 10^6 terms, and one fp32 sum would lose ~1e-3 relative.  The exponent's
      // maximum is 0 (cos <= 1), so no running maximum is needed.  And one count goes into this warp's histogram in
      // shared memory.  At the end the CTA writes its fp64 sum to its own slot, which a finalize kernel reduces in a
      // fixed order (no float atomics: bit-identical across calls), and adds its histogram, summed over the warps, to
      // the 64-bit counters.  A warp's 32-bit counters take at most 32 x 128 columns per tile of its split.
      static_assert(8 * (GEOM_BINS_MAX + 2) * 4 + 8 * 8 <= 16384, "histograms behind colbuf, in front of the barriers");
      const int nb = P.gm_bins, nh = nb + 2;
      const int et = threadIdx.x - 32 * EPI_WARP0;                                       // 0 .. 255
      uint32_t* hist = reinterpret_cast<uint32_t*>(smem + 6 * 2 * TILE_BYTES + 16384);  // [8][nh], behind colbuf
      double* wsum = reinterpret_cast<double*>(hist + 8 * (GEOM_BINS_MAX + 2));         // [8]
      for (int k = et; k < 8 * nh; k += NUM_EPI_THREADS) hist[k] = 0u;
      named_bar_sync(1, NUM_EPI_THREADS);
      uint32_t* whist = hist + (warp - EPI_WARP0) * nh;
      const bool live_row = li < P.b;
      const bool rows_edge = rb * BM + q * 32 + 32 > P.b;  // warp-uniform: some rows of the warp are past b
      const float rs = (P.gm_rscale && live_row) ? P.gm_rscale[li] : 1.f;
      const float kap = P.gm_kappa, lo = P.gm_lo, hi = P.gm_hi, bscale = P.gm_bscale;
      const bool tri = P.tri != 0, mapped = P.gm_mapped != 0;
      double usum = 0.0;
      // 256-column tiles: two TMEM slots and two column buffers, both picked by the parity of the tile's position
      for (int t = t0; t < t1; ++t) {
        const int n = t - t0, par = n & 1;
        mbar_wait(smem_u32(&col_full[par]), static_cast<uint32_t>(n >> 1) & 1);
        mbar_wait(smem_u32(&s_full[par]), static_cast<uint32_t>(n >> 1) & 1);
        tc_fence_after();
        const float* cs = colbuf + par * COL_VECS * CT + half * 128;
        const int* tmap = reinterpret_cast<const int*>(cs + CT);
        const uint32_t taddr = lane_addr + par * CT + half * 128;
        float tsum[2] = {0.f, 0.f};
#pragma unroll 1
        for (int c = 0; c < 4; ++c) {
          const int gj0 = t * CT + half * 128 + c * 32;
          tmem_ld32(taddr + c * 32, v);
          if (c == 3) {
            tc_fence_before();
            release_slot(par);
          }
          if (gj0 >= P.ncols || (tri && gj0 + 31 <= gw0)) continue;  // warp-uniform: no pair of the chunk in scope
          // warp-uniform: some entries need the mask (rows and chunks are both 32-aligned: gj0 == gw0 holds the diagonal)
          const bool edge = rows_edge || gj0 + 32 > P.ncols || (tri ? gj0 <= gw0 + 31 : gj0 == gw0);
#pragma unroll
          for (int e = 0; e < 32; ++e) {
            const int gj = gj0 + e;
            const float x = (v[e] * cs[c * 32 + e]) * rs;
            bool ok = !edge || (live_row && gj < P.ncols && (tri ? gj > gi : (mapped || gj != gi)));
            if (mapped) ok = ok && tmap[c * 32 + e] != gi;
            if (kap != 0.f) tsum[e & 1] += ok ? fast_exp2(fmaf(kap, x, -kap)) : 0.f;
            if (nb && ok) atomicAdd(whist + geom_bin(x, lo, hi, bscale, nb), 1u);
          }
        }
        usum += static_cast<double>(tsum[0] + tsum[1]);
        mbar_arrive(smem_u32(&col_empty[par]));
      }
#pragma unroll
      for (int o = 16; o; o >>= 1) usum += __shfl_xor_sync(0xffffffffu, usum, o);
      if (lane == 0) wsum[warp - EPI_WARP0] = usum;
      named_bar_sync(1, NUM_EPI_THREADS);
      if (et == 0) {
        double s = 0.0;
        for (int w = 0; w < 8; ++w) s += wsum[w];
        P.gm_part[blockIdx.y * gridDim.x + blockIdx.x] = s;
      }
      if (nb) {
        for (int k = et; k < nh; k += NUM_EPI_THREADS) {
          uint32_t s = 0u;
          for (int w = 0; w < 8; ++w) s += hist[w * nh + k];
          if (s) atomicAdd(P.gm_hist + k, static_cast<unsigned long long>(s));
        }
      }
    } else if constexpr (MODE == MODE_LINEAR) {
      // ---------------------------------------------------------------- projection-head layer
      // Row operand = the samples (image rows of the packed buffer, or the hidden activations), column operand =
      // the rows of the weight matrix [out features][K] (nn.Linear's layout is K-major already).  The epilogue adds
      // the bias, applies the ReLU of the hidden layer and rounds to bf16 - the dtype torch.autocast gives the
      // reference's nn.Linear outputs (train.py:285) and the dtype of the student operand of the Gram kernels:
      // the second layer writes straight into the student columns of the packed buffer.
      const bool relu = P.lin_relu != 0;
      int it = 0;
      for (int t = t0; t < t1; ++t, ++it) {
        const int slot = it % nslots;
        const uint32_t use = static_cast<uint32_t>(it / nslots);
        mbar_wait(smem_u32(&s_full[slot]), use & 1);
        tc_fence_after();
#pragma unroll 1
        for (int c = 0; c < 4; ++c) {
          const int jrel0 = t * 256 + half * 128 + c * 32;
          tmem_ld32(lane_addr + slot * 256 + half * 128 + c * 32, v);
          if (c == 3) {
            tc_fence_before();
            release_slot(slot);
          }
          if (li < P.b && jrel0 < P.ncols) {
            __nv_bfloat16* orow = P.lin_out + static_cast<size_t>(li) * P.lin_ld + jrel0;
#pragma unroll
            for (int e8 = 0; e8 < 4; ++e8) {
              if (jrel0 + e8 * 8 < P.ncols) {
                float bb[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
                if (P.lin_bias) {
                  const float4 b0 = __ldg(reinterpret_cast<const float4*>(P.lin_bias + jrel0 + e8 * 8));
                  const float4 b1 = __ldg(reinterpret_cast<const float4*>(P.lin_bias + jrel0 + e8 * 8 + 4));
                  bb[0] = b0.x; bb[1] = b0.y; bb[2] = b0.z; bb[3] = b0.w;
                  bb[4] = b1.x; bb[5] = b1.y; bb[6] = b1.z; bb[7] = b1.w;
                }
                uint32_t w[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  float x0 = v[e8 * 8 + 2 * k] + bb[2 * k], x1 = v[e8 * 8 + 2 * k + 1] + bb[2 * k + 1];
                  if (relu) { x0 = fmaxf(x0, 0.f); x1 = fmaxf(x1, 0.f); }
                  w[k] = pack_bf16x2(x0, x1);
                }
                *reinterpret_cast<uint4*>(orow + e8 * 8) = make_uint4(w[0], w[1], w[2], w[3]);
              }
            }
          }
        }
      }
    } else if constexpr (MODE == MODE_CLIP_SYM) {
      // ---------------------------------------------------------------- one-pass CLIP forward
      // The text -> image logits are the transpose of the image -> text ones (loss.py:266-273), so one pass over
      // x = s log2e (I . T^T) yields both soft-max denominators: row sums as in MODE_CLIP, and per column the sum
      // over the 32 rows of this warp (warp_colsum32), written as a partial (reference exponent, sum) per
      // (warp row, column); clip_colreduce_kernel combines the partials of all row blocks into the column LSEs.
      // ONE exponential per pair serves both sums: e = 2^(x - R) with R = the maximum of the warp's 32 x 32 chunk.
      // A term that is flushed to zero by the fp32 range (x < R - 126) is harmless as long as the log-sum-exp of
      // its row and of its column is not far below R.  Both have an a-priori lower bound - the diagonal logit
      // x_aa, from the dot products rinv_kernel computes next to the norms (P.dbound) - so the test
      //   R - 80 <= min(bound of the warp's rows, bound of the chunk's columns)
      // is warp-uniform and costs nothing; a chunk that fails it (logit scale near 100 next to a badly matched
      // pair) takes the exact path: row sums against the row's own chunk maximum, column sums against per-column
      // maxima (butterfly maximum, second exponential).
      // Sixteen epilogue warps: warp w owns TMEM lanes 32 (w % 4) .. and the 64-column strip (w - 4) / 4 of the tile.
      const int strip = (warp - EPI_WARP0) >> 2;
      const int sp4 = split * 4 + strip;  // P.npart == 4 * nsplit
      const float s2 = P.scal[SC_SCALE_L2];
      const float as2 = fabsf(s2);
      const bool live_row = li < P.b;
      const bool real_block = rb * BM < P.b;
      const bool tail_rows = rb * BM + q * 32 + 32 > P.b;  // warp-uniform: some rows of this warp are past b
      const float row_lo = warp_min_f32(live_row ? P.dbound[gi] * s2 : 3.0e38f);
      float m = M_FLOOR, sum = 0.f, dg = 0.f;
      bool have_dg = false;
      const size_t cp_off = static_cast<size_t>(rb * 4 + q) * P.cp_pitch;
      float* cM = P.colM + cp_off;
      float* cS = P.colS + cp_off;
      // column bounds of the two chunks, fetched one tile ahead (one coalesced load per chunk and warp)
      float bcur[2] = {0.f, 0.f}, bnxt[2] = {0.f, 0.f};
      if (t0 < t1) {
        bnxt[0] = __ldg(P.dbound + P.col0 + t0 * 256 + strip * 64 + lane);
        bnxt[1] = __ldg(P.dbound + P.col0 + t0 * 256 + strip * 64 + 32 + lane);
      }
      int it = 0;
      for (int t = t0; t < t1; ++t, ++it) {
        const int slot = it % nslots;
        const uint32_t use = static_cast<uint32_t>(it / nslots);
        bcur[0] = bnxt[0];
        bcur[1] = bnxt[1];
        if (t + 1 < t1) {
          bnxt[0] = __ldg(P.dbound + P.col0 + (t + 1) * 256 + strip * 64 + lane);
          bnxt[1] = __ldg(P.dbound + P.col0 + (t + 1) * 256 + strip * 64 + 32 + lane);
        }
        mbar_wait(smem_u32(&s_full[slot]), use & 1);
        tc_fence_after();
        // one copy of the chunk code (no unrolling: the instruction cache matters more than the TMEM latency,
        // which the four warps per scheduler hide); the slot goes back once the second chunk is in registers
#pragma unroll 1
        for (int c = 0; c < 2; ++c) {
          const int jrel0 = t * 256 + strip * 64 + c * 32;
          const int gj0 = P.col0 + jrel0;
          tmem_ld32(lane_addr + slot * 256 + strip * 64 + c * 32, v);
          if (c == 1) {
            tc_fence_before();
            release_slot(slot);
          }
          const float lo = fminf(row_lo, s2 * warp_min_f32(c ? bcur[1] : bcur[0]));
          if (gi >= gj0 && gi < gj0 + 32) {
#pragma unroll
            for (int e = 0; e < 32; ++e)
              if (gj0 + e == gi) dg = v[e];
            have_dg = true;
          }
          if (s2 < 0.f) {  // never in training (the model passes exp(logit_scale)); keeps x = v * as2 below
#pragma unroll
            for (int e = 0; e < 32; ++e) v[e] = -v[e];
          }
          if (jrel0 + 32 > P.ncols || tail_rows) {  // ragged columns, rows past b: out of every sum (warp-uniform)
#pragma unroll
            for (int e = 0; e < 32; ++e)
              if (jrel0 + e >= P.ncols || !live_row) v[e] = NEG_BIG;
          }
          float cm[4] = {v[0], v[1], v[2], v[3]};
#pragma unroll
          for (int e = 4; e < 32; ++e) cm[e & 3] = fmaxf(cm[e & 3], v[e]);
          // this row's chunk maximum in log2 units
          const float mo = fmaxf(fmaxf(fmaxf(cm[0], cm[1]), fmaxf(cm[2], cm[3])) * as2, M_FLOOR);
          const float mw = warp_max_f32(mo);
          float ref = mw, csum, cmax = mw;
          if (mw - 80.f <= lo) {
            float2 acc[2] = {pk1(0.f), pk1(0.f)};
            const float2 as22 = pk1(as2), nmw2 = pk1(-mw);
#pragma unroll
            for (int e = 0; e < 32; e += 2) {
              const float2 ex = pk_exp2(pk_fma(pk(v[e], v[e + 1]), as22, nmw2));
              v[e] = ex.x;
              v[e + 1] = ex.y;
              acc[(e >> 1) & 1] = pk_add(acc[(e >> 1) & 1], ex);
            }
            csum = (acc[0].x + acc[0].y) + (acc[1].x + acc[1].y);
          } else {
            ref = mo;
            float x[32], acc = 0.f;
#pragma unroll
            for (int e = 0; e < 32; ++e) {
              x[e] = v[e] * as2;
              acc += fast_exp2(x[e] - mo);
              v[e] = x[e];
            }
            csum = acc;
            cmax = fmaxf(warp_colmax32(x, lane), M_FLOOR);
#pragma unroll
            for (int e = 0; e < 32; ++e) v[e] = fast_exp2(v[e] - __shfl_sync(0xffffffffu, cmax, e));
          }
          const float mnew = fmaxf(m, ref);
          sum = sum * fast_exp2(m - mnew) + csum * fast_exp2(ref - mnew);
          m = mnew;
          const float cs = warp_colsum32(v, lane);
          if (real_block) {
            cM[jrel0 + lane] = cmax;
            cS[jrel0 + lane] = cs;
          }
        }
      }
      if (li < P.b) {
        P.part[(0 * P.npart + sp4) * P.b + li] = m;
        P.part[(1 * P.npart + sp4) * P.b + li] = sum;
        if (have_dg && P.diag) P.diag[li] = dg;
      }
    } else if constexpr (MODE == MODE_CLIP_G) {
      // G_aj = 2^(x - lse_row_a) + 2^(x - lse_col_j), j != a (the diagonal entry incl. its -2 one-hot part and
      // the s/(2b) factor are applied in fp32 by finalize_bwd_kernel); ds_a = sum_j 2^(x - lse_row_a) dot_aj.
      // Fast form (SC_FAST_CLIP, set on the device when the log-sum-exps of all rows and columns lie within 200
      // log2 units of each other): G_aj = 2^(x - c) (2^(c - lse_row_a) + 2^(c - lse_col_j)), ONE exponential per
      // pair; the column factors are precomputed by lse_prepare_kernel.  The exact two-exponential form bounded
      // this kernel at the MUFU rate (2 x 128 ex2 per thread and tile = the MMA time of the tile).
      const float s2 = P.scal[SC_SCALE_L2];
      const float la = P.lse_row[0][min(li, P.b - 1)];
      const bool fast = P.scal[SC_FAST_CLIP] != 0.f;
      const float cref = P.scal[SC_C_CLIP];
      const float fr = fast ? exp2f(cref - la) : 0.f;
      const float* colv = fast ? P.colfac[0] : P.lse_col[0];  // per column: 2^(c - lse_col) or lse_col
      const bool row_only = P.row_only != 0;  // exact form only: the fast form's column factors are zero then
      const bool real_block = rb * BM < P.b;  // the odd pair member past the last row block owns no G rows
      const bool live_row = li < P.b;         // rows past b are K entries of the transposed GEMM: keep them zero
      const bool ds_both = P.ds_both != 0;
      float dsacc = 0.f;
      float2 dsacc2 = pk1(0.f);  // fast form: even / odd columns
      const float2 s22 = pk1(s2), ncref2 = pk1(-cref), fr2 = pk1(fr);
      // per-column values: lane l fetches columns 4l .. 4l+3 of this warp's 128-column strip ONE TILE AHEAD (a
      // single coalesced 16-byte load per lane and tile) and the warp broadcasts them with shuffles.  Eight
      // broadcast loads per 32-column chunk, one chunk ahead, left the epilogue waiting on L2 (long-scoreboard
      // stalls right after every chunk boundary); launched with bn == 256 only
      float4 ccur = make_float4(0.f, 0.f, 0.f, 0.f), cnxt = ccur;
      if (t0 < t1) cnxt = ldg_nc_v4_volatile(colv + P.col0 + t0 * 256 + half * 128 + 4 * lane);
      int it = 0;
      for (int t = t0; t < t1; ++t, ++it) {
        const int slot = it % nslots;
        const uint32_t use = static_cast<uint32_t>(it / nslots);
        ccur = cnxt;
        if (t + 1 < t1) cnxt = ldg_nc_v4_volatile(colv + P.col0 + (t + 1) * 256 + half * 128 + 4 * lane);
        mbar_wait(smem_u32(&s_full[slot]), use & 1);
        tc_fence_after();
        // TMEM loads run one 32-column chunk ahead of the arithmetic (two register buffers)
        uint32_t rA[32], rB[32];
        tmem_ld32_nowait(lane_addr + slot * 256 + half * 128, rA);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const int jrel0 = t * 256 + half * 128 + c * 32;
          const int gj0 = P.col0 + jrel0;
          uint32_t(&rcur)[32] = (c & 1) ? rB : rA;
          uint32_t(&rnxt)[32] = (c & 1) ? rA : rB;
          tmem_ld_wait(rcur);
          if (c < 3) {
            tmem_ld32_nowait(lane_addr + slot * 256 + half * 128 + (c + 1) * 32, rnxt);
          } else {  // every value of this slot is in registers: hand it back before the last chunk's arithmetic
            tc_fence_before();
            release_slot(slot);
          }
#pragma unroll
          for (int e = 0; e < 32; ++e) v[e] = __uint_as_float(rcur[e]);
          float4 cur[8];  // this chunk's 32 column values: column 4 e4 + k lives in lane c * 8 + e4, component k
#pragma unroll
          for (int e4 = 0; e4 < 8; ++e4) {
            cur[e4].x = __shfl_sync(0xffffffffu, ccur.x, c * 8 + e4);
            cur[e4].y = __shfl_sync(0xffffffffu, ccur.y, c * 8 + e4);
            cur[e4].z = __shfl_sync(0xffffffffu, ccur.z, c * 8 + e4);
            cur[e4].w = __shfl_sync(0xffffffffu, ccur.w, c * 8 + e4);
          }
          // masking (diagonal, ragged columns, rows past b) only where a chunk can need it: warp-uniform
          const bool need_mask = (gw0 < gj0 + 32 && gj0 < gw0 + 32) || jrel0 + 32 > P.ncols || !real_block ||
                                 rb * BM + q * 32 + 32 > P.b;
          float g[32];
          if (fast) {
#pragma unroll
            for (int e4 = 0; e4 < 8; ++e4) {
              const float fc[4] = {cur[e4].x, cur[e4].y, cur[e4].z, cur[e4].w};
#pragma unroll
              for (int k = 0; k < 4; k += 2) {
                const int e = 4 * e4 + k;
                const float2 vv = pk(v[e], v[e + 1]);
                const float2 ex = pk_exp2(pk_fma(vv, s22, ncref2));
                const float2 gg = pk_mul(ex, pk_add(fr2, pk(fc[k], fc[k + 1])));
                dsacc2 = pk_fma(ds_both ? gg : pk_mul(ex, fr2), vv, dsacc2);  // ragged columns carry dot = 0
                g[e] = gg.x;
                g[e + 1] = gg.y;
              }
            }
          } else {
#pragma unroll
            for (int e4 = 0; e4 < 8; ++e4) {
              const float ll[4] = {cur[e4].x, cur[e4].y, cur[e4].z, cur[e4].w};
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const int e = 4 * e4 + k;
                const float x2 = v[e] * s2;
                const float e1 = fast_exp2(x2 - la);
                const float e2 = row_only ? 0.f : fast_exp2(x2 - ll[k]);
                dsacc = fmaf(ds_both ? e1 + e2 : e1, v[e], dsacc);
                g[e] = e1 + e2;
              }
            }
          }
          if (need_mask) {
#pragma unroll
            for (int e = 0; e < 32; ++e)
              if (gj0 + e == gi || jrel0 + e >= P.ncols || !live_row) g[e] = 0.f;
          }
          if (real_block && jrel0 + 32 <= P.g_pitch) {  // warp-uniform (the pitch is a multiple of 64 columns)
            uint32_t w16[16];
#pragma unroll
            for (int k = 0; k < 16; ++k) w16[k] = pack_f16x2(g[2 * k], g[2 * k + 1]);
            if ((c & 1) == 0) stage_begin();
            stage_put32(w16, c & 1);
            if (c & 1)
              stage_store(&maps.g[0], (rb * (P.g_pitch >> 6) + (jrel0 >> 6)) * BM + q * 32);
          }
        }
      }
      if (lane == 0) bulk_wait_group<0>();  // the stores have landed before the CTA may exit
      if (li < P.b) P.ds_part[sp * P.b + li] = dsacc + (dsacc2.x + dsacc2.y);
    } else if constexpr (MODE == MODE_SIGLIP) {
      // SigLIP (siglip_pair2): z = s x + beta per pair, positive where global row == global column.  The G tile
      // (G 2^SIG_GK, fp16) goes to gout[0] unless that is null (no gradient wanted); the row partials sum loss, G x
      // and G into part[3][npart][b] unless part is null (the text rows' launch at world > 1 only writes G).
      const float2 s22 = pk1(P.scal[SC_SCALE]), b22 = pk1(P.scal[SC_SIG_BIAS]);
      const bool want_g = P.gout[0] != nullptr;
      const bool real_block = rb * BM < P.b;  // the odd pair member past the last row block owns no G rows
      const bool live_row = li < P.b;         // rows past b are K entries of the transposed GEMM: keep them zero
      float2 lacc = pk1(0.f), gxacc = pk1(0.f), gacc = pk1(0.f);
      int it = 0;
      for (int t = t0; t < t1; ++t, ++it) {
        const int slot = it % nslots;
        const uint32_t use = static_cast<uint32_t>(it / nslots);
        mbar_wait(smem_u32(&s_full[slot]), use & 1);
        tc_fence_after();
        uint32_t rA[32], rB[32];
        tmem_ld32_nowait(lane_addr + slot * 256 + half * 128, rA);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const int jrel0 = t * 256 + half * 128 + c * 32;
          const int gj0 = P.col0 + jrel0;
          uint32_t(&rcur)[32] = (c & 1) ? rB : rA;
          uint32_t(&rnxt)[32] = (c & 1) ? rA : rB;
          tmem_ld_wait(rcur);
          if (c < 3) {
            tmem_ld32_nowait(lane_addr + slot * 256 + half * 128 + (c + 1) * 32, rnxt);
          } else {
            tc_fence_before();
            release_slot(slot);
          }
#pragma unroll
          for (int e = 0; e < 32; ++e) v[e] = __uint_as_float(rcur[e]);
          // positives, ragged columns, rows past b: only in the chunks that can hold them (warp-uniform)
          const bool need_mask = (gw0 < gj0 + 32 && gj0 < gw0 + 32) || jrel0 + 32 > P.ncols || !real_block ||
                                 rb * BM + q * 32 + 32 > P.b;
          float g[32];
          if (!need_mask) {
#pragma unroll
            for (int e = 0; e < 32; e += 2) {
              const float2 vv = pk(v[e], v[e + 1]);
              float2 gg;
              lacc = pk_add(lacc, siglip_pair2(pk_fma(vv, s22, b22), false, false, gg));
              gxacc = pk_fma(gg, vv, gxacc);
              gacc = pk_add(gacc, gg);
              g[e] = gg.x;
              g[e + 1] = gg.y;
            }
          } else {
#pragma unroll
            for (int e = 0; e < 32; e += 2) {
              const bool ok0 = live_row && jrel0 + e < P.ncols, ok1 = live_row && jrel0 + e + 1 < P.ncols;
              const float2 vv = pk(v[e], v[e + 1]);
              float2 gg;
              float2 ll = siglip_pair2(pk_fma(vv, s22, b22), gj0 + e == gi, gj0 + e + 1 == gi, gg);
              gg = pk(ok0 ? gg.x : 0.f, ok1 ? gg.y : 0.f);
              ll = pk(ok0 ? ll.x : 0.f, ok1 ? ll.y : 0.f);
              lacc = pk_add(lacc, ll);
              gxacc = pk_fma(gg, vv, gxacc);
              gacc = pk_add(gacc, gg);
              g[e] = gg.x;
              g[e + 1] = gg.y;
            }
          }
          if (want_g && real_block && jrel0 + 32 <= P.g_pitch) {  // warp-uniform (the pitch is a multiple of 64)
            uint32_t w16[16];
            const float sk = static_cast<float>(1 << SIG_GK);
#pragma unroll
            for (int k = 0; k < 16; ++k) w16[k] = pack_f16x2(g[2 * k] * sk, g[2 * k + 1] * sk);
            if ((c & 1) == 0) stage_begin();
            stage_put32(w16, c & 1);
            if (c & 1)
              stage_store(&maps.g[0], (rb * (P.g_pitch >> 6) + (jrel0 >> 6)) * BM + q * 32);
          }
        }
      }
      if (lane == 0) bulk_wait_group<0>();  // the stores have landed before the CTA may exit
      if (P.part && live_row) {
        const int st = P.npart * P.b;
        P.part[0 * st + sp * P.b + li] = lacc.x + lacc.y;
        P.part[1 * st + sp * P.b + li] = gxacc.x + gxacc.y;
        P.part[2 * st + sp * P.b + li] = gacc.x + gacc.y;
      }
    } else if constexpr (MODE == MODE_SOFT_G) {
      // G_aj = [(2^(p-ls_a) + 2^(p-ls_j)) - (2^(q-lt_a) + 2^(q-lt_j))] * mant(1/||y_j||), j != a, for the
      // student (-> gout[0]) and the text term (-> gout[1]) from ONE teacher tile.
      //  * student / text: p - ls = (p - M) + (M - ls) with the fixed maximum M = log2(e)/tau (reached on the
      //    diagonal, so M <= ls <= M + log2 B): 2^(p-M) (2^(M-ls_a) + 2^(M-ls_j)), one exponential per pair;
      //  * teacher: the same form with M_t = log2(e)/tau_t when M_t <= 60 (fast_t, decided on the host from
      //    tau_t: every exponent then stays inside fp32), else the exact two-exponential form;
      //  the column factors 2^(M - l_j) (teacher exact form: l_j itself) come staged from lse_prepare_kernel, which
      //  writes zeros (exact form: +1e30) when the column-side terms are dropped (gather_with_grad == False).
      //  * the fp16 gradient operand row is y_j * 2^floor(log2(1/||y_j||)) (exact), so G carries the remaining
      //    mantissa of 1/||y_j|| in [1, 2) of its COLUMN; world == 1 (tri): also that of its ROW, which makes the
      //    stored matrix symmetric - the gradient GEMM reads the blocks left of the diagonal transposed from the
      //    same matrix and finalize_bwd_kernel divides the row factor out again.
      const int lic = min(li, P.b - 1);
      const float cq = P.rinv[0][gi] * P.scal[SC_ITT_L2];
      const float mt = P.scal[SC_ITT_L2];
      const float lt = P.lse_row[0][lic];
      const bool fast_t = P.fast_t != 0;
      const float frt = fast_t ? exp2f(mt - lt) : 0.f;
      const float2 cq2 = pk1(cq), nmt2 = pk1(-mt), nfrt2 = pk1(-frt);
      const bool real_block = rb * BM < P.b;
      const bool live_row = li < P.b;  // rows past b are K entries of the transposed gradient GEMM: keep them zero
      float E[128];  // -(teacher terms) of this thread's 128 columns, kept across the student / text products
      int it = 0;
      for (int t = t0; t < t1; ++t, it += P.nprod) {
        const int jt0 = t * CT + half * 128;
        // this tile's column vectors (staged by the producer): [p] inverse norms, [3 + p] column factors
        const int cb = (t - t0) % COL_BUFS;
        mbar_wait(smem_u32(&col_full[cb]), static_cast<uint32_t>((t - t0) / COL_BUFS) & 1);
        const float* cv = colbuf + cb * COL_VECS * CT + half * 128;
        {
          const int slot = (it + 0) % 2;
          mbar_wait(smem_u32(&s_full[slot]), static_cast<uint32_t>((it + 0) / 2) & 1);
          tc_fence_after();
          uint32_t rA[32], rB[32];  // TMEM loads run one chunk ahead of the arithmetic
          tmem_ld32_nowait(lane_addr + slot * CT + half * 128, rA);
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            uint32_t(&rcur)[32] = (c & 1) ? rB : rA;
            uint32_t(&rnxt)[32] = (c & 1) ? rA : rB;
            tmem_ld_wait(rcur);
            if (c < 3) {
              tmem_ld32_nowait(lane_addr + slot * CT + half * 128 + (c + 1) * 32, rnxt);
            } else {
              tc_fence_before();
              release_slot(slot);
            }
#pragma unroll
            for (int e = 0; e < 32; ++e) v[e] = __uint_as_float(rcur[e]);
            const float4* rc = reinterpret_cast<const float4*>(cv + 0 * CT + c * 32);
            const float4* lc = reinterpret_cast<const float4*>(cv + 3 * CT + c * 32);
#pragma unroll
            for (int e4 = 0; e4 < 8; ++e4) {
              const float4 r4 = rc[e4];
              const float4 l4 = lc[e4];
              const float rr[4] = {r4.x, r4.y, r4.z, r4.w};
              const float ll[4] = {l4.x, l4.y, l4.z, l4.w};
#pragma unroll
              for (int k = 0; k < 4; k += 2) {
                const int e = 4 * e4 + k;
                if (fast_t) {  // -2^(q - M_t) (2^(M_t - lt_a) + 2^(M_t - lt_j))
                  const float2 ex = pk_exp2(pk_fma(pk(v[e], v[e + 1]), pk_mul(cq2, pk(rr[k], rr[k + 1])), nmt2));
                  const float2 r = pk_mul(ex, pk_add(nfrt2, pk(-ll[k], -ll[k + 1])));
                  E[c * 32 + e] = r.x;
                  E[c * 32 + e + 1] = r.y;
                } else {
#pragma unroll
                  for (int u = 0; u < 2; ++u) {
                    const float q2 = v[e + u] * cq * rr[k + u];
                    E[c * 32 + e + u] = -(fast_exp2(q2 - lt) + fast_exp2(q2 - ll[k + u]));
                  }
                }
              }
            }
          }
        }
        for (int p = 1; p < P.nprod; ++p) {
          const int slot = (it + p) % 2;
          mbar_wait(smem_u32(&s_full[slot]), static_cast<uint32_t>((it + p) / 2) & 1);
          tc_fence_after();
          const float my = P.scal[(p == 1) ? SC_ITS_L2 : SC_ITX_L2];
          const float ry = P.rinv[p][gi];
          const float cy = ry * my;
          const float fry = exp2f(my - P.lse_row[p][lic]);
          const float rowf = P.tri ? mant12(ry) : 1.f;
          const float2 cy2 = pk1(cy), nmy2 = pk1(-my), fry2 = pk1(fry), rowf2 = pk1(rowf);
          uint32_t rA[32], rB[32];
          tmem_ld32_nowait(lane_addr + slot * CT + half * 128, rA);
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const int jrel0 = jt0 + c * 32;
            const int gj0 = P.col0 + jrel0;
            uint32_t(&rcur)[32] = (c & 1) ? rB : rA;
            uint32_t(&rnxt)[32] = (c & 1) ? rA : rB;
            tmem_ld_wait(rcur);
            if (c < 3) {
              tmem_ld32_nowait(lane_addr + slot * CT + half * 128 + (c + 1) * 32, rnxt);
            } else {
              tc_fence_before();
              release_slot(slot);
            }
#pragma unroll
            for (int e = 0; e < 32; ++e) v[e] = __uint_as_float(rcur[e]);
            const bool need_mask = (gw0 < gj0 + 32 && gj0 < gw0 + 32) || jrel0 + 32 > P.ncols || !real_block ||
                                   rb * BM + q * 32 + 32 > P.b;
            const float4* rc = reinterpret_cast<const float4*>(cv + p * CT + c * 32);
            const float4* lc = reinterpret_cast<const float4*>(cv + (3 + p) * CT + c * 32);
            uint32_t w16[16];
#pragma unroll
            for (int e4 = 0; e4 < 8; ++e4) {
              const float4 r4 = rc[e4];
              const float4 l4 = lc[e4];
              const float rr[4] = {r4.x, r4.y, r4.z, r4.w};
              const float ll[4] = {l4.x, l4.y, l4.z, l4.w};
              float g4[4];
#pragma unroll
              for (int k = 0; k < 4; k += 2) {
                const int e = 4 * e4 + k;
                const float2 rk = pk(rr[k], rr[k + 1]);
                const float2 ex = pk_exp2(pk_fma(pk(v[e], v[e + 1]), pk_mul(cy2, rk), nmy2));
                // symmetric in (a, j) when world == 1
                float2 g = pk_fma(ex, pk_add(fry2, pk(ll[k], ll[k + 1])), pk(E[c * 32 + e], E[c * 32 + e + 1]));
                if (need_mask) {
                  if ((gj0 + e == gi) || (jrel0 + e >= P.ncols) || !live_row) g.x = 0.f;
                  if ((gj0 + e + 1 == gi) || (jrel0 + e + 1 >= P.ncols) || !live_row) g.y = 0.f;
                }
                g = pk_mul(g, pk_mul(rowf2, pk(mant12(rk.x), mant12(rk.y))));
                g4[k] = g.x;
                g4[k + 1] = g.y;
              }
              w16[2 * e4 + 0] = pack_f16x2(g4[0], g4[1]);
              w16[2 * e4 + 1] = pack_f16x2(g4[2], g4[3]);
            }
            if (real_block && jrel0 + 32 <= P.g_pitch) {  // warp-uniform (the pitch is a multiple of 64 columns)
              if ((c & 1) == 0) stage_begin();
              stage_put32(w16, c & 1);
              if (c & 1)
                stage_store(&maps.g[p - 1], (rb * (P.g_pitch >> 6) + (jrel0 >> 6)) * BM + q * 32);
            }
          }
        }
        mbar_arrive(smem_u32(&col_empty[cb]));
      }
      if (lane == 0) bulk_wait_group<0>();  // the stores have landed before the CTA may exit
    } else if constexpr (kWce) {
      // ---------------------------------------------------------------- denominator-modulated CE, loss.py:416-471
      // Products per 256-column tile: [0] CLIP logits x (row operand = image rows, or text rows for the text
      // direction), [1] DINO cosine -> dissimilarity r = 1 - clamp(cos), r_aa = 0 (loss.py:424-429).  The rows are
      // this rank's block [row0, row0 + b) of the global B x B problem, the columns all of it (col0 == 0), so the
      // diagonal of local row li sits at column row0 + li.  World size 1 is the reference's square problem.
      //   STAT : c_a = sum_j p_aj r_aj with p = soft-max of the UNMODIFIED row (loss.py:434-435), and the row sums
      //          of x and x^2 behind the row std of the logits (loss.py:440-441)
      //   LSE  : log-sum-exp of x~ = x + beta clamp(r - c_a, +-c_clip) (diagonal unshifted, loss.py:445-447) and
      //          A_a = sum_{j != a} p~_aj [ |r_aj - c_a| <= c_clip ] (the share of the row that feels d c_a)
      //   DBG  : the row statistics behind the reference's diagnostics (loss.py:479-595)
      //   G    : the fp16 logit gradient of  g_c * classic CE  +  g_w * weighted CE, times gk (SC_WCE_GK), for
      //          BOTH directions in one matrix (rows = image, columns = text; the text direction's entry is the
      //          transposed one and reads its row statistics per column):
      //          d CE~_a / d x_ak = p~_ak - delta_ak - beta A_a p_ak (r_ak - c_a).
      //          World > 1: one launch per direction (wdir = row side); the column side reads the other
      //          direction's all-gathered row statistics by global column, as MODE_CLIP_G does.
      const int lic = min(li, P.b - 1);
      const float s2 = P.scal[SC_SCALE_L2];
      const float rda = P.colvec[0][min(gi, P.ncols - 1)];
      const float cc = P.wcc;
      const float beta2 = (MODE == MODE_WCE_STAT) ? 0.f : P.scal[SC_WBETA2 + P.wdir];
      const float lse_a = (MODE == MODE_WCE_LSE) ? 0.f : P.wrow[0][lic];
      const float c_a = (MODE == MODE_WCE_STAT) ? 0.f : P.wrow[1][lic];
      const float lset_a = (MODE == MODE_WCE_DBG || MODE == MODE_WCE_G) ? P.wrow[2][lic] : 0.f;
      const bool real_block = rb * BM < P.b;
      const bool live_row = li < P.b;
      float xq[128];  // this thread's 128 CLIP logits (log2 units), kept while the DINO tile arrives
      // accumulators (meaning per mode, see the stores at the end)
      float acc[11];
#pragma unroll
      for (int k = 0; k < 11; ++k) acc[k] = 0.f;
      float mrun = M_FLOOR;
      // G mode: upstream gradients and the text direction's knobs
      WceRowK wk{};
      if constexpr (MODE == MODE_WCE_G) {
        wk.lse = lse_a;
        wk.c = c_a;
        wk.lset = lset_a;
        wk.aa = P.wrow[3][lic];
        wk.beta = P.scal[SC_WBETA + P.wdir];  // row-side direction
        wk.beta2 = beta2;
        wk.beta_t = P.scal[SC_WBETA + 1 - P.wdir];
        wk.beta2_t = P.scal[SC_WBETA2 + 1 - P.wdir];
        wk.cc = cc;
        wk.gcl = (P.wgout[0] + P.wlam[0] * P.wgout[4]) * P.scal[SC_WCE_GK];
        wk.gwt = (P.wgout[5] + P.wlam[1] * P.wgout[4]) * P.scal[SC_WCE_GK];
      }
      int it = 0;
      for (int t = t0; t < t1; ++t, it += 2) {
        const int jt0 = t * CT + half * 128;
        const int cb = (t - t0) % COL_BUFS;
        mbar_wait(smem_u32(&col_full[cb]), static_cast<uint32_t>((t - t0) / COL_BUFS) & 1);
        const float* cv = colbuf + cb * COL_VECS * CT + half * 128;
        {  // ---- CLIP tile -> xq
          const int slot = it % 2;
          mbar_wait(smem_u32(&s_full[slot]), static_cast<uint32_t>(it / 2) & 1);
          tc_fence_after();
          uint32_t rA[32], rB[32];
          tmem_ld32_nowait(lane_addr + slot * CT + half * 128, rA);
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            uint32_t(&rcur)[32] = (c & 1) ? rB : rA;
            uint32_t(&rnxt)[32] = (c & 1) ? rA : rB;
            tmem_ld_wait(rcur);
            if (c < 3) {
              tmem_ld32_nowait(lane_addr + slot * CT + half * 128 + (c + 1) * 32, rnxt);
            } else {
              tc_fence_before();
              release_slot(slot);
            }
#pragma unroll
            for (int e = 0; e < 32; ++e) xq[c * 32 + e] = __uint_as_float(rcur[e]) * s2;
          }
        }
        {  // ---- DINO tile -> r, then the mode's arithmetic per 32-column chunk
          const int slot = (it + 1) % 2;
          mbar_wait(smem_u32(&s_full[slot]), static_cast<uint32_t>((it + 1) / 2) & 1);
          tc_fence_after();
          uint32_t rA[32], rB[32];
          tmem_ld32_nowait(lane_addr + slot * CT + half * 128, rA);
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const int jrel0 = jt0 + c * 32;
            uint32_t(&rcur)[32] = (c & 1) ? rB : rA;
            uint32_t(&rnxt)[32] = (c & 1) ? rA : rB;
            tmem_ld_wait(rcur);
            if (c < 3) {
              tmem_ld32_nowait(lane_addr + slot * CT + half * 128 + (c + 1) * 32, rnxt);
            } else {
              tc_fence_before();
              release_slot(slot);
            }
            const bool has_diag = gw0 < jrel0 + 32 && jrel0 < gw0 + 32;  // warp-uniform
            const bool ragged = jrel0 + 32 > P.ncols;
            const float4* rc = reinterpret_cast<const float4*>(cv + 0 * CT + c * 32);
            float r[32];
#pragma unroll
            for (int e4 = 0; e4 < 8; ++e4) {
              const float4 q4 = rc[e4];
              const float rr[4] = {q4.x, q4.y, q4.z, q4.w};
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const int e = 4 * e4 + k;
                const float cosv = __uint_as_float(rcur[e]) * rda * rr[k];
                r[e] = 1.f - fminf(fmaxf(cosv, -1.f), 1.f);
              }
            }
            if (has_diag) {
#pragma unroll
              for (int e = 0; e < 32; ++e)
                if (jrel0 + e == gi) r[e] = 0.f;
            }
            if constexpr (MODE == MODE_WCE_STAT) {
#pragma unroll
              for (int e = 0; e < 32; ++e) {
                const float x = xq[c * 32 + e];
                const bool live = !ragged || jrel0 + e < P.ncols;
                const float p = live ? fast_exp2(x - lse_a) : 0.f;
                acc[0] = fmaf(p, r[e], acc[0]);
                acc[1 + (e & 1)] += live ? x : 0.f;          // two partial sums each: shorter dependency chains
                acc[3 + (e & 1)] = fmaf(live ? x : 0.f, x, acc[3 + (e & 1)]);
              }
            } else if constexpr (MODE == MODE_WCE_LSE) {
              float xt[32];
              float cm = NEG_BIG;
#pragma unroll
              for (int e = 0; e < 32; ++e) {
                const float z = r[e] - c_a;
                const bool dg = has_diag && jrel0 + e == gi;
                float x = xq[c * 32 + e] + (dg ? 0.f : beta2 * fminf(fmaxf(z, -cc), cc));
                if (ragged && jrel0 + e >= P.ncols) x = NEG_BIG;
                xt[e] = x;
                cm = fmaxf(cm, x);
              }
              const float mnew = fmaxf(mrun, cm);
              const float alpha = fast_exp2(mrun - mnew);
              mrun = mnew;
              float s0 = 0.f, s1 = 0.f;
#pragma unroll
              for (int e = 0; e < 32; ++e) {
                const float ex = fast_exp2(xt[e] - mnew);
                const bool ind = fabsf(r[e] - c_a) <= cc && !(has_diag && jrel0 + e == gi);
                s0 += ex;
                s1 += ind ? ex : 0.f;
              }
              acc[0] = fmaf(acc[0], alpha, s0);
              acc[1] = fmaf(acc[1], alpha, s1);
            } else if constexpr (MODE == MODE_WCE_DBG) {
#pragma unroll
              for (int e = 0; e < 32; ++e) {
                const bool dg = has_diag && jrel0 + e == gi;
                const bool live = !ragged || jrel0 + e < P.ncols;
                const float x = xq[c * 32 + e];
                const float rh = fminf(fmaxf(r[e] - c_a, -cc), cc);
                const float xm = x + (dg ? 0.f : beta2 * rh);
                const float p = live ? fast_exp2(x - lse_a) : 0.f;
                const float pt = live ? fast_exp2(xm - lset_a) : 0.f;
                const float dp = pt - p;
                const float rl = live ? rh : 0.f;
                const float ro = dg ? 0.f : rl;  // off-diagonal share
                acc[0] = fmaf(p, rl, acc[0]);       // sum p r^        (pc_err)
                acc[1] += fabsf(dp);                // sum |dp|        (l1 shift)
                acc[2] += rl;                       // sum r^
                acc[3] = fmaf(rl, rl, acc[3]);      // sum r^^2
                acc[4] += dp;                       // sum dp
                acc[5] = fmaf(dp, dp, acc[5]);      // sum dp^2
                acc[6] = fmaf(rl, dp, acc[6]);      // sum r^ dp
                acc[7] += fabsf(ro);                // sum |r^| off-diagonal (delta mean)
                acc[8] = fmaf(ro, ro, acc[8]);      // sum r^^2 off-diagonal (delta std)
                acc[9] = fmaxf(acc[9], fabsf(ro));  // max |r^| off-diagonal (delta max)
                acc[10] += (ro > 0.f) ? 1.f : 0.f;  // count r^ > 0 off-diagonal
              }
            } else {  // MODE_WCE_G
              const float4* l1c = reinterpret_cast<const float4*>(cv + 1 * CT + c * 32);  // lse_ti by column
              const float4* l2c = reinterpret_cast<const float4*>(cv + 2 * CT + c * 32);  // lse~ (text dir)
              const float4* ccc = reinterpret_cast<const float4*>(cv + 3 * CT + c * 32);  // c' (text dir)
              const float4* aac = reinterpret_cast<const float4*>(cv + 4 * CT + c * 32);  // A' (text dir)
              const bool need_mask = has_diag || ragged || !real_block || rb * BM + q * 32 + 32 > P.b;
              uint32_t w16[16];
#pragma unroll
              for (int e4 = 0; e4 < 8; ++e4) {
                const float4 a4 = l1c[e4], b4 = l2c[e4], c4 = ccc[e4], d4 = aac[e4];
                const float lti[4] = {a4.x, a4.y, a4.z, a4.w}, ltt[4] = {b4.x, b4.y, b4.z, b4.w};
                const float cj[4] = {c4.x, c4.y, c4.z, c4.w}, aj[4] = {d4.x, d4.y, d4.z, d4.w};
                float g4[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  const int e = 4 * e4 + k;
                  const float x = xq[c * 32 + e];
                  const WcePair wp = wce_pair(P, wk, x, r[e], lti[k], ltt[k], cj[k], aj[k]);
                  float g = wp.g;
                  float gr = wp.gr;  // this rank's own loss terms
                  if (need_mask && ((jrel0 + e == gi) || (jrel0 + e >= P.ncols) || !live_row)) g = gr = 0.f;
                  acc[0] = fmaf(gr, x, acc[0]);  // d(logit_scale) row term in log2 units of x (off-diagonal part)
                  g4[k] = g;
                }
                w16[2 * e4 + 0] = pack_f16x2(g4[0], g4[1]);
                w16[2 * e4 + 1] = pack_f16x2(g4[2], g4[3]);
              }
              if (real_block && jrel0 + 32 <= P.g_pitch) {
                if ((c & 1) == 0) stage_begin();
                stage_put32(w16, c & 1);
                if (c & 1) stage_store(&maps.g[0], (rb * (P.g_pitch >> 6) + (jrel0 >> 6)) * BM + q * 32);
              }
            }
          }
        }
        mbar_arrive(smem_u32(&col_empty[cb]));
      }
      if constexpr (MODE == MODE_WCE_G) {
        if (lane == 0) bulk_wait_group<0>();
        if (li < P.b) P.ds_part[sp * P.b + li] = acc[0] / s2;  // back to raw dot-product units (still times gk)
      } else if (li < P.b) {
        const int o = sp * P.b + li;
        const int st = P.npart * P.b;
        if constexpr (MODE == MODE_WCE_STAT) {
          P.part[0 * st + o] = acc[0];
          P.part[1 * st + o] = acc[1] + acc[2];
          P.part[2 * st + o] = acc[3] + acc[4];
        } else if constexpr (MODE == MODE_WCE_LSE) {
          P.part[0 * st + o] = mrun;
          P.part[1 * st + o] = acc[0];
          P.part[2 * st + o] = acc[1];
        } else {
#pragma unroll
          for (int k = 0; k < 11; ++k) P.part[k * st + o] = acc[k];
        }
      }
    } else if constexpr (kDist) {
      // ---------------------------------------------------------------- DistillClipLoss (open_clip)
      // Products per 256-column tile: [0] student logits x = s <row, col> (image rows x text columns, or text rows x
      // image columns), [1] teacher logits t = s_t <row_t, col_t> of the same pairs; both in log2 units.  The rows are
      // this rank's block [row0, row0 + b), the columns all B; the diagonal of local row li is column row0 + li.
      // Both TMEM slots of a tile are read chunk by chunk side by side (holding the student strip in registers while
      // the teacher tile arrives, as the weighted-CE modes do, does not fit the register budget without spills).
      //   FWD: per row, with online maxima (neither diagonal bounds its row): student m, sum 2^(x-m), sum 2^(x-m) (x-m);
      //        teacher m_t, sum 2^(t-m_t) and sum 2^(t-m_t) (x-m) (relative to the CURRENT student maximum, so that
      //        the distill term comes out as a difference of small numbers) -> part[6][npart][b]; the raw diagonal dot
      //        products -> diag[0 / 1][b] (student / teacher).
      //   G  : (2b gk) dL/dx off the diagonal, without the diagonal's one-hot term (applied in fp32 afterwards):
      //          a_c (p_r + p_c) + a_d ((p_r - q_r) + (p_c - q_c)),   a_c = g_c gk, a_d = g_d gk
      //        p_r / q_r from this row's student / teacher lse (wrow[0 / 1]), p_c / q_c from the column's (the other
      //        direction's row statistics by global column, colvec[0 / 1]); row_only drops the column side.
      const int lic = min(li, P.b - 1);
      const float s2 = P.scal[SC_SCALE_L2], st2 = P.scal[SC_DST_TSCALE_L2];
      const bool real_block = rb * BM < P.b;
      const bool live_row = li < P.b;
      float ms = M_FLOOR, ss = 0.f, ps = 0.f, mt = M_FLOOR, stt = 0.f, qa = 0.f, dgx = 0.f, dgt = 0.f;
      bool have_dg = false;
      float lse_r = 0.f, lset_r = 0.f, ac = 0.f, ad = 0.f;
      if constexpr (MODE == MODE_DIST_G) {
        lse_r = P.wrow[0][lic];
        lset_r = P.wrow[1][lic];
        ac = P.scal[SC_DST_GC];
        ad = P.scal[SC_DST_GD];
      }
      int it = 0;
      for (int t = t0; t < t1; ++t, it += 2) {
        const int jt0 = t * CT + half * 128;
        const int cb = (t - t0) % COL_BUFS;
        mbar_wait(smem_u32(&col_full[cb]), static_cast<uint32_t>((t - t0) / COL_BUFS) & 1);
        const float* cv = colbuf + cb * COL_VECS * CT + half * 128;
        const int slot_x = it % 2, slot_t = (it + 1) % 2;
        mbar_wait(smem_u32(&s_full[slot_x]), static_cast<uint32_t>(it / 2) & 1);
        mbar_wait(smem_u32(&s_full[slot_t]), static_cast<uint32_t>((it + 1) / 2) & 1);
        tc_fence_after();
#pragma unroll 1
        for (int c = 0; c < 4; ++c) {
          const int jrel0 = jt0 + c * 32;
          uint32_t rX[32], rT[32];
          tmem_ld32_nowait(lane_addr + slot_x * CT + half * 128 + c * 32, rX);
          tmem_ld32_nowait(lane_addr + slot_t * CT + half * 128 + c * 32, rT);
          tmem_ld_wait(rX);
          tmem_ld_wait(rT);
          if (c == 3) {
            tc_fence_before();
            release_slot(slot_x);
            release_slot(slot_t);
          }
          const bool has_diag = gw0 < jrel0 + 32 && jrel0 < gw0 + 32;  // warp-uniform
          const bool ragged = jrel0 + 32 > P.ncols;
          if constexpr (MODE == MODE_DIST_FWD) {
            if (has_diag) {
#pragma unroll
              for (int e = 0; e < 32; ++e)
                if (jrel0 + e == gi) {
                  dgx = __uint_as_float(rX[e]);  // raw dot products: the finalize scales them as below
                  dgt = __uint_as_float(rT[e]);
                  have_dg = true;
                }
            }
            float cm = NEG_BIG, cmt = NEG_BIG;
#pragma unroll
            for (int e = 0; e < 32; ++e) {
              float x = __uint_as_float(rX[e]) * s2, tt = __uint_as_float(rT[e]) * st2;
              if (ragged && jrel0 + e >= P.ncols) x = tt = NEG_BIG;
              rX[e] = __float_as_uint(x);
              rT[e] = __float_as_uint(tt);
              cm = fmaxf(cm, x);
              cmt = fmaxf(cmt, tt);
            }
            const float mnew = fmaxf(ms, cm);
            const float dl = mnew - ms;
            const float al = fast_exp2(-dl);
            ps = al * fmaf(-dl, ss, ps);  // sum 2^(x-m) (x-m) relative to the new maximum
            ss *= al;
            qa = fmaf(-dl, stt, qa);      // sum 2^(t-m_t) (x-m): the student reference moves
            ms = mnew;
            const float mtn = fmaxf(mt, cmt);
            const float alt = fast_exp2(mt - mtn);
            stt *= alt;
            qa *= alt;
            mt = mtn;
            float2 sacc = pk1(0.f), pacc = pk1(0.f), tacc = pk1(0.f), qacc = pk1(0.f);
#pragma unroll
            for (int e = 0; e < 32; e += 2) {
              const float2 d = pk_add(pk(__uint_as_float(rX[e]), __uint_as_float(rX[e + 1])), pk1(-ms));
              const float2 ex = pk_exp2(d);
              const float2 w = pk_exp2(pk_add(pk(__uint_as_float(rT[e]), __uint_as_float(rT[e + 1])), pk1(-mt)));
              sacc = pk_add(sacc, ex);
              pacc = pk_fma(ex, d, pacc);
              tacc = pk_add(tacc, w);
              qacc = pk_fma(w, d, qacc);
            }
            ss += sacc.x + sacc.y;
            ps += pacc.x + pacc.y;
            stt += tacc.x + tacc.y;
            qa += qacc.x + qacc.y;
          } else {  // MODE_DIST_G
            const float4* lsc = reinterpret_cast<const float4*>(cv + 0 * CT + c * 32);  // column's student lse
            const float4* ltc = reinterpret_cast<const float4*>(cv + 1 * CT + c * 32);  // column's teacher lse
            const bool need_mask = has_diag || ragged || !real_block || rb * BM + q * 32 + 32 > P.b;
            uint32_t w16[16];
#pragma unroll
            for (int e4 = 0; e4 < 8; ++e4) {
              float4 l4 = make_float4(0.f, 0.f, 0.f, 0.f), m4 = l4;
              if (!P.row_only) {
                l4 = lsc[e4];
                m4 = ltc[e4];
              }
              const float lcol[4] = {l4.x, l4.y, l4.z, l4.w}, tcol[4] = {m4.x, m4.y, m4.z, m4.w};
              float g4[4];
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const int e = 4 * e4 + k;
                const float x = __uint_as_float(rX[e]) * s2;
                const float tt = __uint_as_float(rT[e]) * st2;
                const float pr = fast_exp2(x - lse_r);
                const float qr = fast_exp2(tt - lset_r);
                float psum = pr, dpq = pr - qr;  // p - q formed in fp32
                if (!P.row_only) {
                  const float pc = fast_exp2(x - lcol[k]);
                  const float qc = fast_exp2(tt - tcol[k]);
                  psum += pc;
                  dpq += pc - qc;
                }
                float g = fmaf(ac, psum, ad * dpq);
                if (need_mask && ((jrel0 + e == gi) || (jrel0 + e >= P.ncols) || !live_row)) g = 0.f;
                g4[k] = g;
              }
              w16[2 * e4 + 0] = pack_f16x2(g4[0], g4[1]);
              w16[2 * e4 + 1] = pack_f16x2(g4[2], g4[3]);
            }
            if (real_block && jrel0 + 32 <= P.g_pitch) {
              if ((c & 1) == 0) stage_begin();
              stage_put32(w16, c & 1);
              if (c & 1) stage_store(&maps.g[0], (rb * (P.g_pitch >> 6) + (jrel0 >> 6)) * BM + q * 32);
            }
          }
        }
        mbar_arrive(smem_u32(&col_empty[cb]));
      }
      if constexpr (MODE == MODE_DIST_G) {
        if (lane == 0) bulk_wait_group<0>();  // the stores have landed before the CTA may exit
      } else if (live_row) {
        const int o = sp * P.b + li;
        const int st = P.npart * P.b;
        P.part[0 * st + o] = ms;
        P.part[1 * st + o] = ss;
        P.part[2 * st + o] = ps;
        P.part[3 * st + o] = mt;
        P.part[4 * st + o] = stt;
        P.part[5 * st + o] = qa;
        if (have_dg) {
          P.diag[li] = dgx;
          P.diag[P.b + li] = dgt;
        }
      }
    } else if constexpr (MODE == MODE_SOFT_SYM16) {
      // ---------------------------------------------------------------- symmetric forward, 16x256b TMEM loads
      // The teacher, student and text Gram matrices are symmetric, so a row pair only computes the tiles from its
      // own diagonal tile onwards (P.tri).  A tile right of the diagonal also holds, transposed, the entries the
      // rows of its COLUMN block need: every quantity is summed over the 32 rows of a warp per column and written
      // as a column partial [k][rb * 4 + q][column]; soft_colreduce_kernel adds those to the row partials.  All
      // exponentials use FIXED maxima (teacher: log2(e)/tau_t, valid because fast_t bounds it by 60; student /
      // text: log2(e)/tau, reached on the diagonal), so row and column partials share one reference and no running
      // maximum has to be reconciled.  Exponent arguments come out of ONE fma: arg = dot * (row factor * column
      // factor) - M, with M = NEG_BIG for a dead row (rows past b: 2^arg = 0 without a select, so they never reach
      // the column sums).  The weighted sums are kept relative to the fixed maxima, sum w (q - M_t) etc.;
      // finalize_fwd adds M * Zt back.
      // Register layout: tcgen05.ld 16x256b gives every thread FOUR rows (g, g + 8, g + 16, g + 24 of the warp's 32;
      // g = lane / 4) and, per 32-column chunk, the columns 8 j + 2 c2 + {0, 1} (j = 0..3, c2 = lane % 4).  The
      // column sums over the warp's rows then start with three in-register adds per column and need a three-stage
      // butterfly over the eight row groups (warp_colsum8: 7 shuffles + 14 selects per quantity and chunk) instead of
      // the five-stage one over 32 lanes that the 32x32b shape needs (31 + 62).  Row sums: every thread accumulates
      // its four rows per product and tile, the four lanes of a row group combine them (two xor stages) and lane c2
      // keeps row g + 8 c2, so the persistent accumulators stay one row per thread.
      const float mt2 = P.scal[SC_ITT_L2], ms2 = P.scal[SC_ITS_L2], mx2 = P.scal[SC_ITX_L2];
      const int g = lane >> 2, c2 = lane & 3;
      const int wrow0 = rb * BM + q * 32;  // first local row of this warp
      int lrow[4];
      float rq[4], rz[4], rx[4];  // inverse norms of the thread's rows: DINO, student, text
      const bool has_text = P.nprod == 3;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        lrow[i] = wrow0 + g + 8 * i;
        const int gr = P.row0 + lrow[i];
        rq[i] = P.rinv[0][gr];
        rz[i] = P.rinv[1][gr];
        rx[i] = has_text ? P.rinv[2][gr] : 0.f;
      }
      float zt = 0.f, aq = 0.f, ap = 0.f, ar = 0.f, zs = 0.f, zx = 0.f;  // row g + 8 c2
      float w[128];  // teacher weights of the thread's 4 rows x 32 columns: [chunk c][half h][8 j + 4 rs + ... ]
      const size_t cp_stride = static_cast<size_t>(P.cp_rows) * P.cp_pitch;
      float* cp_row = P.colpart + static_cast<size_t>(rb * 4 + q) * P.cp_pitch;
      const int mycol = 8 * (g >> 1) + 2 * c2 + (g & 1);  // the column of a chunk whose sum warp_colsum8 returns here
      // sum over the two columns of a pair, then over the four lanes of the row group; lane c2 takes row c2
      auto row_take = [&](const float2 (&a)[4]) {
        float r[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          r[i] = a[i].x + a[i].y;
          r[i] += __shfl_xor_sync(0xffffffffu, r[i], 1);
          r[i] += __shfl_xor_sync(0xffffffffu, r[i], 2);
        }
        return c2 == 0 ? r[0] : (c2 == 1 ? r[1] : (c2 == 2 ? r[2] : r[3]));
      };
      int it = 0;
      for (int t = t0; t < t1; ++t, it += P.nprod) {
        const int jt0 = t * CT + half * 128;
        const bool ragged = jt0 + 128 > P.ncols;
        const bool offdiag = t > (rb >> 1);  // this tile also serves the rows of its column block
        const int cb = (t - t0) % COL_BUFS;
        mbar_wait(smem_u32(&col_full[cb]), static_cast<uint32_t>((t - t0) / COL_BUFS) & 1);
        const float* cv = colbuf + cb * COL_VECS * CT + half * 128;
        // one product of the tile; kT: the teacher product (writes w, masks its diagonal), else student / text
        auto product = [&](auto kT_, const int p) {
          constexpr bool kT = decltype(kT_)::value;
          const int slot = (it + p) % 2;
          mbar_wait(smem_u32(&s_full[slot]), static_cast<uint32_t>((it + p) / 2) & 1);
          tc_fence_after();
          const float mfix = kT ? mt2 : ((p == 1) ? ms2 : mx2);
          float2 fr[4], bias[4];  // per row: (1 / norm) * log2(e) / tau, and -M (dead row: -1e30, so 2^arg = 0)
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            fr[i] = pk1((kT ? rq[i] : ((p == 1) ? rz[i] : rx[i])) * mfix);
            bias[i] = pk1(lrow[i] < P.b ? -mfix : NEG_BIG);
          }
          float2 a0[4], a1[4];  // per row: sum of the exponentials, sum of w * arg
#pragma unroll
          for (int i = 0; i < 4; ++i) a0[i] = a1[i] = pk1(0.f);
          const uint32_t tbase = lane_addr + slot * CT + half * 128;
          uint32_t rA[16], rB[16];
          tmem_ld16x256_nowait(tbase, rA);
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const int jrel0 = jt0 + c * 32;
            const bool rag = ragged && jrel0 + 32 > P.ncols;
            // the teacher diagonal (column == local row, primed coordinates) can only lie in a chunk that overlaps
            // the warp's rows; diagonal tiles always take the masked path (cheap: one tile per row pair)
            const bool need_mask = (kT && ((wrow0 < jrel0 + 32 && jrel0 < wrow0 + 32) || !offdiag)) || rag;
            float2 cs0[4], cs1[4];  // per column pair j: sums over the thread's four rows
#pragma unroll
            for (int j = 0; j < 4; ++j) cs0[j] = cs1[j] = pk1(0.f);
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              uint32_t(&rcur)[16] = (h == 0) ? rA : rB;
              uint32_t(&rnxt)[16] = (h == 0) ? rB : rA;
              tmem_ld_wait16(rcur);
              if (h == 0) {
                tmem_ld16x256_nowait(tbase + (16u << 16) + c * 32, rnxt);
              } else if (c < 3) {
                tmem_ld16x256_nowait(tbase + (c + 1) * 32, rnxt);
              } else {
                tc_fence_before();
                release_slot(slot);
              }
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const float2 rr = *reinterpret_cast<const float2*>(cv + p * CT + c * 32 + 8 * j + 2 * c2);
                const int col = jrel0 + 8 * j + 2 * c2;
#pragma unroll
                for (int rs = 0; rs < 2; ++rs) {
                  const int i = 2 * h + rs;
                  const int wi = c * 32 + h * 16 + 4 * j + 2 * rs;
                  const float2 arg = pk_fma(pk(__uint_as_float(rcur[4 * j + 2 * rs]),
                                               __uint_as_float(rcur[4 * j + 2 * rs + 1])),
                                            pk_mul(fr[i], rr), bias[i]);
                  float2 ex = pk_exp2(arg);
                  if (need_mask) {  // ragged columns; teacher: the diagonal (loss.py:376-377)
                    if (col >= P.ncols || (kT && col == lrow[i])) ex.x = 0.f;
                    if (col + 1 >= P.ncols || (kT && col + 1 == lrow[i])) ex.y = 0.f;
                  }
                  float2 wa;
                  if constexpr (kT) {
                    w[wi] = ex.x;
                    w[wi + 1] = ex.y;
                    wa = pk_mul(ex, arg);
                  } else {
                    wa = pk_mul(pk(w[wi], w[wi + 1]), arg);  // w is zero on masked entries and in dead rows
                  }
                  a0[i] = pk_add(a0[i], ex);
                  a1[i] = pk_add(a1[i], wa);
                  cs0[j] = pk_add(cs0[j], ex);
                  cs1[j] = pk_add(cs1[j], wa);
                }
              }
            }
            if (offdiag) {  // warp-uniform
              const float s0 = warp_colsum8(cs0, lane);
              const float s1 = warp_colsum8(cs1, lane);
              // column partial quantities: [0] teacher sum, [1] sum w q, [2] sum w p, [3] sum w r,
              // [4] student sum, [5] text sum
              const int k0 = kT ? 0 : ((p == 1) ? 4 : 5);
              const int k1 = kT ? 1 : ((p == 1) ? 2 : 3);
              cp_row[k0 * cp_stride + jrel0 + mycol] = s0;
              cp_row[k1 * cp_stride + jrel0 + mycol] = s1;
            }
          }
          const float t0s = row_take(a0), t1s = row_take(a1);
          if (kT) { zt += t0s; aq += t1s; } else if (p == 1) { zs += t0s; ap += t1s; } else { zx += t0s; ar += t1s; }
        };
        product(std::true_type{}, 0);
        for (int p = 1; p < P.nprod; ++p) product(std::false_type{}, p);
        mbar_arrive(smem_u32(&col_empty[cb]));
      }
      const int myrow = wrow0 + g + 8 * c2;
      if (myrow < P.b) {  // same partial layout as MODE_SOFT; the maximum is the fixed one
        const int o = sp * P.b + myrow;
        const int st = P.npart * P.b;
        P.part[0 * st + o] = mt2;
        P.part[1 * st + o] = zt;
        P.part[2 * st + o] = aq;
        P.part[3 * st + o] = ap;
        P.part[4 * st + o] = ar;
        P.part[5 * st + o] = zs;
        P.part[6 * st + o] = zx;
      }
    } else {
      const float cq = P.rinv[0][gi] * P.scal[SC_ITT_L2];
      const float cp = P.rinv[1][gi] * P.scal[SC_ITS_L2];
      const float ms2 = P.scal[SC_ITS_L2];
      const bool has_text = P.nprod == 3;
      const float cr = has_text ? P.rinv[2][gi] * P.scal[SC_ITX_L2] : 0.f;
      const float mx2 = P.scal[SC_ITX_L2];
      float m = M_FLOOR, zt = 0.f, aq = 0.f, ap = 0.f, ar = 0.f, zs = 0.f, zx = 0.f;
      float w[128];  // teacher weights 2^(q - m) of this thread's 128 columns, kept across the three products
      int it = 0;
      for (int t = t0; t < t1; ++t, it += P.nprod) {
        const int jt0 = t * CT + half * 128;  // first column (relative to col0) of this thread's 128 columns
        const bool ragged = jt0 + 128 > P.ncols;
        // this tile's inverse column norms per product, staged by the producer
        const int cb = (t - t0) % COL_BUFS;
        mbar_wait(smem_u32(&col_full[cb]), static_cast<uint32_t>((t - t0) / COL_BUFS) & 1);
        const float* cv = colbuf + cb * COL_VECS * CT + half * 128;
        // ---- teacher: q (log2 units) for all 128 columns, then ONE running-max update for the tile; the
        // TMEM slot goes back to the MMA issuer as soon as the values are in registers
        {
          const int slot = (it + 0) % 2;
          mbar_wait(smem_u32(&s_full[slot]), static_cast<uint32_t>((it + 0) / 2) & 1);
          tc_fence_after();
          uint32_t rA[32], rB[32];  // TMEM loads run one chunk ahead of the arithmetic
          tmem_ld32_nowait(lane_addr + slot * CT + half * 128, rA);
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            uint32_t(&rcur)[32] = (c & 1) ? rB : rA;
            uint32_t(&rnxt)[32] = (c & 1) ? rA : rB;
            tmem_ld_wait(rcur);
            if (c < 3) {
              tmem_ld32_nowait(lane_addr + slot * CT + half * 128 + (c + 1) * 32, rnxt);
            } else {
              tc_fence_before();
              release_slot(slot);
            }
#pragma unroll
            for (int e = 0; e < 32; ++e) v[e] = __uint_as_float(rcur[e]);
            const float4* rc = reinterpret_cast<const float4*>(cv + c * 32);
#pragma unroll
            for (int e4 = 0; e4 < 8; ++e4) {
              const float4 r = rc[e4];
              w[c * 32 + 4 * e4 + 0] = v[4 * e4 + 0] * cq * r.x;
              w[c * 32 + 4 * e4 + 1] = v[4 * e4 + 1] * cq * r.y;
              w[c * 32 + 4 * e4 + 2] = v[4 * e4 + 2] * cq * r.z;
              w[c * 32 + 4 * e4 + 3] = v[4 * e4 + 3] * cq * r.w;
            }
          }
          const int gj0 = P.col0 + jt0;
          if (ragged || (gw0 < gj0 + 128 && gj0 < gw0 + 32)) {  // warp-uniform
#pragma unroll
            for (int e = 0; e < 128; ++e)
              if (jt0 + e >= P.ncols || gj0 + e == gi) w[e] = NEG_BIG;  // teacher diag masked: loss.py:376-377
          }
          float cm[4] = {w[0], w[1], w[2], w[3]};
#pragma unroll
          for (int e = 4; e < 128; ++e) cm[e & 3] = fmaxf(cm[e & 3], w[e]);
          const float mnew = fmaxf(m, fmaxf(fmaxf(cm[0], cm[1]), fmaxf(cm[2], cm[3])));
          const float alpha = fast_exp2(m - mnew);
          m = mnew;
          float a0[4] = {0.f, 0.f, 0.f, 0.f}, a1[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
          for (int e = 0; e < 128; ++e) {
            const float q2 = w[e];
            const float we = fast_exp2(q2 - mnew);
            a0[e & 3] += we;
            a1[e & 3] = fmaf(we, q2, a1[e & 3]);
            w[e] = we;
          }
          zt = zt * alpha + ((a0[0] + a0[1]) + (a0[2] + a0[3]));
          aq = aq * alpha + ((a1[0] + a1[1]) + (a1[2] + a1[3]));
          ap *= alpha;
          ar *= alpha;
        }
        // ---- student (p = 1) and text (p = 2, loss.py:387-397): sum w*p and the fixed-max exp sum
        for (int p = 1; p < P.nprod; ++p) {
          const int slot = (it + p) % 2;
          mbar_wait(smem_u32(&s_full[slot]), static_cast<uint32_t>((it + p) / 2) & 1);
          tc_fence_after();
          const float cs = (p == 1) ? cp : cr;
          const float mfix = (p == 1) ? ms2 : mx2;
          float b0[4] = {0.f, 0.f, 0.f, 0.f}, b1[4] = {0.f, 0.f, 0.f, 0.f};
          uint32_t rA[32], rB[32];
          tmem_ld32_nowait(lane_addr + slot * CT + half * 128, rA);
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const int jrel0 = jt0 + c * 32;
            uint32_t(&rcur)[32] = (c & 1) ? rB : rA;
            uint32_t(&rnxt)[32] = (c & 1) ? rA : rB;
            tmem_ld_wait(rcur);
            if (c < 3) {
              tmem_ld32_nowait(lane_addr + slot * CT + half * 128 + (c + 1) * 32, rnxt);
            } else {
              tc_fence_before();
              release_slot(slot);
            }
#pragma unroll
            for (int e = 0; e < 32; ++e) v[e] = __uint_as_float(rcur[e]);
            const float4* rc = reinterpret_cast<const float4*>(cv + p * CT + c * 32);
            const bool rag = ragged && jrel0 + 32 > P.ncols;
#pragma unroll
            for (int e4 = 0; e4 < 8; ++e4) {
              const float4 r = rc[e4];
              const float rr[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const int e = 4 * e4 + k;
                float p2 = v[e] * cs * rr[k];
                if (rag && jrel0 + e >= P.ncols) p2 = NEG_BIG;
                b0[k] += fast_exp2(p2 - mfix);
                b1[k] = fmaf(w[c * 32 + e], p2, b1[k]);
              }
            }
          }
          const float zsum = (b0[0] + b0[1]) + (b0[2] + b0[3]);
          const float asum = (b1[0] + b1[1]) + (b1[2] + b1[3]);
          if (p == 1) { zs += zsum; ap += asum; } else { zx += zsum; ar += asum; }
        }
        mbar_arrive(smem_u32(&col_empty[cb]));
      }
      if (li < P.b) {
        const int o = sp * P.b + li;
        const int st = P.npart * P.b;
        P.part[0 * st + o] = m;
        P.part[1 * st + o] = zt;
        P.part[2 * st + o] = aq;
        P.part[3 * st + o] = ap;
        P.part[4 * st + o] = ar;
        P.part[5 * st + o] = zs;
        P.part[6 * st + o] = zx;
      }
    }
  }

  tc_fence_before();
  cluster_sync_all();
  if (warp == 2) tmem_dealloc_cg<CG>(tmem_base, TMEM_COLS);
}

// ================================================================================================
// Backward: recompute tile -> G (fp16, smem) -> accumulate G . Y in TMEM
// ================================================================================================
//  MODE_CLIP: G_aj = 2^(x - lse_row_a) + 2^(x - lse_col_j), j != a   (the diagonal entry incl. its
//             -2 one-hot part and the s/(2b) factor are applied in fp32 by the finalize kernel)
//  MODE_SOFT: G_aj = [(2^(p-ls_a) + 2^(p-ls_j)) - (2^(q-lt_a) + 2^(q-lt_j))] / (||y_j|| sigma), j != a
//             (diagonal dropped: it is parallel to y_a and vanishes in the normalise backward)
//  MODE_WCE_X: G_aj = the weighted CE entry of MODE_WCE_G (wce_pair, times gk) for the rows of one direction, from a
//             CLIP tile and a DINO tile per column tile (diagonal dropped, applied in fp32 by the finalize kernel); one
//             launch per direction, each with the row-side d(logit_scale) term only (wsplit), as MODE_CLIP
//  row_only drops the *_j (column-side) terms: gathered features are constants (gather_with_grad=0).
//  G is stored as fp16 (10-bit mantissa) and multiplied with an EXACT fp16 copy of the gradient operand
//  (bf16 features times a power of two sigma): bf16 G costs 8x the rounding error, mixed fp16 x bf16
//  operands are not accepted by tcgen05.mma, and a rounded (normalised) operand would put the same
//  error into every row's gradient.
//
//  The gradient of a 128-row block is [128 x Dout] fp32; only 256 of its columns fit in TMEM next to the
//  S tiles.  The Dout/256 feature chunks of one (row block, column split) are therefore the CTAs of one
//  thread-block CLUSTER (C <= 3): CTA c owns accumulator columns [256c, 256c+256), computes the S tile
//  and G only for the column tiles t = t0 + r*C + c ("its" tile of round r), and ships that fp16 G tile
//  to the other CTAs with a DSMEM bulk copy (cp.async.bulk.shared::cluster).  Every CTA then multiplies
//  all C tiles of the round with its own feature chunk of Y.  No S tile is ever recomputed per chunk.
//
//  shared memory (7 slabs of 32 KiB): G[C] | one operand ring of 7 - C stages.  A ring stage holds either
//  an S-operand pair (A box | B box, 64 features) or a gradient-operand half tile (64 j x 256 features);
//  the TMA producer fills stages in exactly the order the MMA issuer consumes them, so every phase of the
//  kernel has the whole ring (up to 192 KiB) in flight.
//  warps: 0 = TMA producer, 1 = MMA issuer, 2 = TMEM alloc, 3 = G sender, 4..11 = epilogue
constexpr int X_MAXC = 3;
constexpr int SLAB = 2 * TILE_BYTES;   // 32 KiB
constexpr int X_SLABS = 7;
constexpr int X_MAXSTAGES = 6;

template <int MODE>
__global__ void __launch_bounds__(NUM_THREADS, 1)
dsoft_bwd_kernel(const __grid_constant__ TileMaps maps, const __grid_constant__ CUtensorMap vmap,
                 const __grid_constant__ BwdParams P) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align_1024(smem_raw);
  const int csize = gridDim.x;           // cluster size == feature chunks handled by this launch
  const int crank = blockIdx.x;          // == %cluster_ctarank
  const int ns = X_SLABS - csize;        // operand ring stages (6 / 5 / 4)
  uint8_t* g_smem = smem;                          // csize slabs: G tile of producer k at slab k
  uint8_t* s_smem = smem + csize * SLAB;           // ns slabs
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + X_SLABS * SLAB);
  uint64_t* ring_full = bars;           // [6]
  uint64_t* ring_empty = bars + 6;      // [6]
  uint64_t* s_full = bars + 12;         // [2]
  uint64_t* s_empty = bars + 14;        // [2]
  uint64_t* g_written = bars + 16;      // own G tile stored (256 epilogue arrivals)
  uint64_t* g_in = bars + 17;           // [3] G tile of producer k landed (tx bytes)
  uint64_t* g_free = bars + 20;         // own G tile consumed by all C CTAs (multicast commits)
  uint64_t* acc_full = bars + 21;
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(bars + 22);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int rb = blockIdx.y;
  const int split = blockIdx.z;
  const int chunk = P.chunk0 + crank;
  const int t0 = split * P.tiles_per_split;
  const int t1 = min(t0 + P.tiles_per_split, P.ntiles);
  const int nrounds = (t1 - t0 + csize - 1) / csize;
  const int f0 = chunk * CHUNK_F;                            // first gradient feature of this CTA
  const int nfb = min(4, (P.dout - f0 + BK - 1) / BK);       // 64-feature boxes of this CTA

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < 4; ++i) tma_prefetch_desc(&maps.m[i]);
    tma_prefetch_desc(&vmap);
    for (int i = 0; i < X_MAXSTAGES; ++i) {
      mbar_init(smem_u32(&ring_full[i]), 1);
      mbar_init(smem_u32(&ring_empty[i]), 1);
    }
    for (int i = 0; i < B_SLOTS; ++i) {
      mbar_init(smem_u32(&s_full[i]), 1);
      mbar_init(smem_u32(&s_empty[i]), NUM_EPI_THREADS);
    }
    mbar_init(smem_u32(g_written), NUM_EPI_THREADS);
    for (int i = 0; i < X_MAXC; ++i) mbar_init(smem_u32(&g_in[i]), 1);
    mbar_init(smem_u32(g_free), csize);
    mbar_init(smem_u32(acc_full), 1);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc(smem_u32(tmem_holder), TMEM_COLS);
  tc_fence_before();
  cluster_sync_all();  // peers' mbarriers must exist before any DSMEM copy / multicast commit reaches them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer (one ring, MMA order)
    int stage = 0;
    uint32_t phase = 0;
    auto load_grad_operands = [&](int r) {  // Y16 half tiles for the gradient GEMMs of round r
      for (int k = 0; k < csize; ++k) {
        const int t = t0 + r * csize + k;
        if (t >= t1) break;
        for (int h = 0; h < 2; ++h) {
          mbar_wait(smem_u32(&ring_empty[stage]), phase ^ 1);
          if (elect_one()) {
            const uint32_t full = smem_u32(&ring_full[stage]);
            const uint32_t dst = smem_u32(s_smem + stage * SLAB);
            mbar_arrive_expect_tx(full, nfb * (TILE_BYTES / 2));
            for (int fb = 0; fb < nfb; ++fb)
              tma_load_2d(dst + fb * (TILE_BYTES / 2), &vmap, full, f0 + fb * BK, P.col0 + t * BN + h * 64);
          }
          __syncwarp();
          if (++stage == ns) { stage = 0; phase ^= 1; }
        }
      }
    };
    for (int r = 0; r < nrounds; ++r) {
      const int t = t0 + r * csize + crank;
      if (t < t1) {
        for (int p = 0; p < P.nprod; ++p) {
          const CUtensorMap* am = &maps.m[P.a_map[p]];
          const CUtensorMap* bm = &maps.m[P.b_map[p]];
          for (int kc = 0; kc < P.kchunks[p]; ++kc) {
            mbar_wait(smem_u32(&ring_empty[stage]), phase ^ 1);
            if (elect_one()) {
              const uint32_t full = smem_u32(&ring_full[stage]);
              const uint32_t a_dst = smem_u32(s_smem + stage * SLAB);
              mbar_arrive_expect_tx(full, 2 * TILE_BYTES);
              tma_load_2d(a_dst, am, full, kc * BK, P.row0 + rb * BM);
              tma_load_2d(a_dst + TILE_BYTES, bm, full, kc * BK, P.col0 + t * BN);
            }
            __syncwarp();
            if (++stage == ns) { stage = 0; phase ^= 1; }
          }
        }
      }
      if (r > 0) load_grad_operands(r - 1);
    }
    load_grad_operands(nrounds - 1);
  } else if (warp == 3) {
    // ------------------------------------------------------------------ G sender (DSMEM bulk copies)
    if (csize > 1) {
      const uint32_t src = smem_u32(g_smem + crank * SLAB);
      for (int r = 0; r < nrounds; ++r) {
        if (t0 + r * csize + crank >= t1) break;
        mbar_wait(smem_u32(g_written), static_cast<uint32_t>(r) & 1);
        if (elect_one()) {
          for (int k = 0; k < csize; ++k) {
            if (k == crank) continue;
            bulk_copy_to_peer(mapa_shared(src, k), src, SLAB, mapa_shared(smem_u32(&g_in[crank]), k));
          }
        }
        __syncwarp();
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (warp-uniform loop)
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    bool first_grad = true;
    const uint32_t idesc_g = make_idesc_bf16(BM, nfb * BK, 0, 1, 1);  // fp16: A = G (K-major), B = Y16 (MN-major)
    const uint32_t tmem_acc = tmem_base + ACC_COL;
    if (elect_one()) {
      for (int k = 0; k < csize; ++k)
        if (k != crank && t0 + k < t1) mbar_arrive_expect_tx(smem_u32(&g_in[k]), SLAB);
    }
    __syncwarp();
    auto issue_grads = [&](int r) {
      for (int k = 0; k < csize; ++k) {
        if (t0 + r * csize + k >= t1) break;
        if (k == crank) {
          mbar_wait(smem_u32(g_written), static_cast<uint32_t>(r) & 1);
        } else {
          mbar_wait(smem_u32(&g_in[k]), static_cast<uint32_t>(r) & 1);
          // re-arm for the next round now: producer k cannot send before this CTA's commit below
          if (t0 + (r + 1) * csize + k < t1 && elect_one()) mbar_arrive_expect_tx(smem_u32(&g_in[k]), SLAB);
          __syncwarp();
        }
        tc_fence_after();
        const uint32_t g_addr = smem_u32(g_smem + k * SLAB);
        for (int h = 0; h < 2; ++h) {
          mbar_wait(smem_u32(&ring_full[stage]), phase);
          tc_fence_after();
          if (elect_one()) {
            const uint32_t v_addr = smem_u32(s_smem + stage * SLAB);
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
              // A: G[128 rows, 16 j] in K-block h; B: Y16[16 j, 64*nfb features] MN-major (8 KiB boxes)
              const uint64_t ad = make_smem_desc(g_addr + h * TILE_BYTES + kk * 32, 16, 1024);
              const uint64_t bd = make_smem_desc(v_addr + kk * 2048, TILE_BYTES / 2, 1024);
              umma_bf16(tmem_acc, ad, bd, idesc_g, (first_grad && h == 0 && kk == 0) ? 0u : 1u);
            }
            umma_commit(smem_u32(&ring_empty[stage]));
            if (h == 1) {
              if (csize > 1)
                umma_commit_mc(smem_u32(g_free), static_cast<uint16_t>(1u << k));  // tell producer k
              else
                umma_commit(smem_u32(g_free));
            }
          }
          __syncwarp();
          if (++stage == ns) { stage = 0; phase ^= 1; }
        }
        first_grad = false;
      }
    };
    for (int r = 0; r < nrounds; ++r) {
      const int t = t0 + r * csize + crank;
      if (t < t1) {
        for (int p = 0; p < P.nprod; ++p, ++it) {
          const int slot = it % B_SLOTS;
          const uint32_t use = static_cast<uint32_t>(it / B_SLOTS);
          mbar_wait(smem_u32(&s_empty[slot]), (use & 1) ^ 1);
          tc_fence_after();
          const uint32_t tmem_d = tmem_base + slot * BN;
          for (int kc = 0; kc < P.kchunks[p]; ++kc) {
            mbar_wait(smem_u32(&ring_full[stage]), phase);
            tc_fence_after();
            if (elect_one()) {
              const uint32_t a_smem = smem_u32(s_smem + stage * SLAB);
              issue_s_stage(tmem_d, a_smem, a_smem + TILE_BYTES, kc == 0);
              umma_commit(smem_u32(&ring_empty[stage]));
              if (kc == P.kchunks[p] - 1) umma_commit(smem_u32(&s_full[slot]));
            }
            __syncwarp();
            if (++stage == ns) { stage = 0; phase ^= 1; }
          }
        }
      }
      if (r > 0) issue_grads(r - 1);  // keeps the tensor pipe busy while this round's epilogue runs
    }
    issue_grads(nrounds - 1);
    if (elect_one()) umma_commit(smem_u32(acc_full));
    __syncwarp();
  } else if (warp >= EPI_WARP0) {
    // ------------------------------------------------------------------ epilogue
    const int q = warp & 3;
    const int half = (warp - EPI_WARP0) >> 2;
    const int row = q * 32 + lane;
    const int li = rb * BM + row;
    const int lic = min(li, P.b - 1);  // clamped index for per-row constant loads
    const int gi = P.row0 + li;
    const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const uint32_t g_row = smem_u32(g_smem + crank * SLAB) + half * TILE_BYTES + row * 128;
    const int sw = row & 7;
    const bool row_only = P.row_only != 0;
    float v[32];
    float dsacc = 0.f;

    float c_a = 0.f, c_b = 0.f, l_a = 0.f, l_b = 0.f;
    if constexpr (MODE == MODE_RAW) {
      c_a = 1.f;
    } else if constexpr (MODE == MODE_CLIP) {
      c_a = P.scal[SC_SCALE_L2];
      l_a = P.lse_row[lic];
    } else if constexpr (MODE == MODE_WCE_X) {
      c_a = P.scal[SC_SCALE_L2];
      c_b = P.rinv_d[gi];
    } else {
      c_a = P.rinv_d[gi] * P.scal[SC_ITT_L2];  // teacher
      l_a = P.lse_t_row[lic];
      c_b = P.rinv_y[gi] * P.scal[P.tau_idx];  // student / text
      l_b = P.lse_y_row[lic];
    }
    WceRowK wk{};
    if constexpr (MODE == MODE_WCE_X) {
      wk.lse = P.wrow[0][lic];
      wk.c = P.wrow[1][lic];
      wk.lset = P.wrow[2][lic];
      wk.aa = P.wrow[3][lic];
      wk.beta = P.scal[SC_WBETA + P.wdir];
      wk.beta2 = P.scal[SC_WBETA2 + P.wdir];
      wk.beta_t = P.scal[SC_WBETA + 1 - P.wdir];
      wk.beta2_t = P.scal[SC_WBETA2 + 1 - P.wdir];
      wk.cc = P.wcc;
      wk.gcl = (P.wgout[0] + P.wlam[0] * P.wgout[4]) * P.scal[SC_WCE_GK];
      wk.gwt = (P.wgout[5] + P.wlam[1] * P.wgout[4]) * P.scal[SC_WCE_GK];
    }

    // 32 fp32 -> fp16, 4 x 16-byte swizzled stores into the K-major SW128 A-operand layout
    auto store_g = [&](const float (&g)[32], int c) {
#pragma unroll
      for (int k4 = 0; k4 < 4; ++k4) {
        const uint32_t w0 = pack_f16x2(g[8 * k4 + 0], g[8 * k4 + 1]);
        const uint32_t w1 = pack_f16x2(g[8 * k4 + 2], g[8 * k4 + 3]);
        const uint32_t w2 = pack_f16x2(g[8 * k4 + 4], g[8 * k4 + 5]);
        const uint32_t w3 = pack_f16x2(g[8 * k4 + 6], g[8 * k4 + 7]);
        const int chunk16 = c * 4 + k4;
        st_shared_v4(g_row + ((chunk16 ^ sw) << 4), w0, w1, w2, w3);
      }
    };

    int it = 0;
    for (int r = 0; r < nrounds; ++r, it += P.nprod) {
      const int t = t0 + r * csize + crank;
      if (t >= t1) break;
      const int slot0 = it % B_SLOTS;
      const int jt0 = t * BN + half * 64;  // first column (relative to col0) of this thread's 64 columns

      if constexpr (MODE == MODE_WCE_X) {
        // ---- CLIP tile first: the raw dot products stay in registers and the TMEM slot is handed back at once,
        // as in MODE_SOFT
        float Xd[64];
        const int slot1 = (it + 1) % B_SLOTS;
        mbar_wait(smem_u32(&s_full[slot0]), static_cast<uint32_t>(it / B_SLOTS) & 1);
        tc_fence_after();
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          tmem_ld32(lane_addr + slot0 * BN + half * 64 + c * 32, v);
#pragma unroll
          for (int e = 0; e < 32; ++e) Xd[c * 32 + e] = v[e];
        }
        tc_fence_before();
        mbar_arrive(smem_u32(&s_empty[slot0]));
        // ---- DINO tile: r = 1 - clamp(cos), then the pair's weighted logit gradient (MODE_WCE_G's arithmetic)
        mbar_wait(smem_u32(&s_full[slot1]), static_cast<uint32_t>((it + 1) / B_SLOTS) & 1);
        tc_fence_after();
        if (r > 0) mbar_wait(smem_u32(g_free), static_cast<uint32_t>(r - 1) & 1);
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          const int jrel0 = jt0 + c * 32;
          const int gj0 = P.col0 + jrel0;
          float g[32];
          tmem_ld32(lane_addr + slot1 * BN + half * 64 + c * 32, v);
          const float4* rc = reinterpret_cast<const float4*>(P.rinv_d + gj0);
          const float4* l1c = reinterpret_cast<const float4*>(P.wcol[0] + gj0);
          const float4* l2c = reinterpret_cast<const float4*>(P.wcol[1] + gj0);
          const float4* ccc = reinterpret_cast<const float4*>(P.wcol[2] + gj0);
          const float4* aac = reinterpret_cast<const float4*>(P.wcol[3] + gj0);
#pragma unroll
          for (int e4 = 0; e4 < 8; ++e4) {
            const float4 r4 = __ldg(rc + e4), a4 = __ldg(l1c + e4), b4 = __ldg(l2c + e4);
            const float4 c4 = __ldg(ccc + e4), d4 = __ldg(aac + e4);
            const float rr[4] = {r4.x, r4.y, r4.z, r4.w};
            const float lj[4] = {a4.x, a4.y, a4.z, a4.w}, ltj[4] = {b4.x, b4.y, b4.z, b4.w};
            const float cj[4] = {c4.x, c4.y, c4.z, c4.w}, aj[4] = {d4.x, d4.y, d4.z, d4.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const int e = 4 * e4 + k;
              const float rd = 1.f - fminf(fmaxf(v[e] * c_b * rr[k], -1.f), 1.f);
              const float dot = Xd[c * 32 + e];
              const WcePair wp = wce_pair(P, wk, dot * c_a, rd, lj[k], ltj[k], cj[k], aj[k]);
              // diagonal (r_aa = 0: applied in fp32 by finalize_bwd_kernel) and ragged columns dropped
              const bool dead = (gj0 + e == gi) || (jrel0 + e >= P.ncols);
              dsacc = fmaf(dead ? 0.f : wp.gr, dot, dsacc);
              g[e] = dead ? 0.f : wp.g;
            }
          }
          store_g(g, c);
        }
        tc_fence_before();
        mbar_arrive(smem_u32(&s_empty[slot1]));
      } else if constexpr (MODE == MODE_SOFT) {
        // ---- teacher tile first: E = -(2^(q-lt_a) + 2^(q-lt_j)) stays in registers and the TMEM slot is
        // handed back at once, so the next tile's teacher MMAs overlap the rest of this epilogue
        float E[64];
        const int slot1 = (it + 1) % B_SLOTS;
        mbar_wait(smem_u32(&s_full[slot0]), static_cast<uint32_t>(it / B_SLOTS) & 1);
        tc_fence_after();
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          const int gj0 = P.col0 + jt0 + c * 32;
          tmem_ld32(lane_addr + slot0 * BN + half * 64 + c * 32, v);
          const float4* rc = reinterpret_cast<const float4*>(P.rinv_d + gj0);
          const float4* lc = reinterpret_cast<const float4*>(P.lse_t_col + gj0);
#pragma unroll
          for (int e4 = 0; e4 < 8; ++e4) {
            const float4 r4 = __ldg(rc + e4);
            const float4 l4 = __ldg(lc + e4);
            const float rr[4] = {r4.x, r4.y, r4.z, r4.w};
            const float ll[4] = {l4.x, l4.y, l4.z, l4.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const int e = 4 * e4 + k;
              const float q2 = v[e] * c_a * rr[k];
              const float e1 = fast_exp2(q2 - l_a);
              const float e2 = row_only ? 0.f : fast_exp2(q2 - ll[k]);
              E[c * 32 + e] = -(e1 + e2);
            }
          }
        }
        tc_fence_before();
        mbar_arrive(smem_u32(&s_empty[slot0]));
        // ---- student / text tile
        mbar_wait(smem_u32(&s_full[slot1]), static_cast<uint32_t>((it + 1) / B_SLOTS) & 1);
        tc_fence_after();
        if (r > 0) mbar_wait(smem_u32(g_free), static_cast<uint32_t>(r - 1) & 1);
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          const int jrel0 = jt0 + c * 32;
          const int gj0 = P.col0 + jrel0;
          float g[32];
          tmem_ld32(lane_addr + slot1 * BN + half * 64 + c * 32, v);
          const float4* rc = reinterpret_cast<const float4*>(P.rinv_y + gj0);
          const float4* lc = reinterpret_cast<const float4*>(P.lse_y_col + gj0);
#pragma unroll
          for (int e4 = 0; e4 < 8; ++e4) {
            const float4 r4 = __ldg(rc + e4);
            const float4 l4 = __ldg(lc + e4);
            const float rr[4] = {r4.x, r4.y, r4.z, r4.w};
            const float ll[4] = {l4.x, l4.y, l4.z, l4.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const int e = 4 * e4 + k;
              const float p2 = v[e] * c_b * rr[k];
              const float e1 = fast_exp2(p2 - l_b);
              const float e2 = row_only ? 0.f : fast_exp2(p2 - ll[k]);
              // the fp16 operand row is y_j * 2^floor(log2(1/||y_j||)) (exact), so G carries the remaining
              // mantissa of 1/||y_j|| in [1, 2); diagonal (teacher masked, student parallel to y_a) and ragged
              // columns dropped
              const bool dead = (gj0 + e == gi) || (jrel0 + e >= P.ncols);
              g[e] = dead ? 0.f : (E[c * 32 + e] + (e1 + e2)) * mant12(rr[k]);
            }
          }
          store_g(g, c);
        }
        tc_fence_before();
        mbar_arrive(smem_u32(&s_empty[slot1]));
      } else {
        mbar_wait(smem_u32(&s_full[slot0]), static_cast<uint32_t>(it / B_SLOTS) & 1);
        tc_fence_after();
        // previous own G tile consumed by every CTA of the cluster (local and remote copies are free)
        if (r > 0) mbar_wait(smem_u32(g_free), static_cast<uint32_t>(r - 1) & 1);
#pragma unroll 1
        for (int c = 0; c < 2; ++c) {
          const int jrel0 = jt0 + c * 32;
          const int gj0 = P.col0 + jrel0;
          float g[32];
          tmem_ld32(lane_addr + slot0 * BN + half * 64 + c * 32, v);
          if constexpr (MODE == MODE_RAW) {
#pragma unroll
            for (int e = 0; e < 32; ++e) g[e] = v[e];
          } else {
            const float4* lc = reinterpret_cast<const float4*>(P.lse_col + gj0);
#pragma unroll
            for (int e4 = 0; e4 < 8; ++e4) {
              const float4 l4 = __ldg(lc + e4);
              const float ll[4] = {l4.x, l4.y, l4.z, l4.w};
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const int e = 4 * e4 + k;
                const float x2 = v[e] * c_a;
                const float e1 = fast_exp2(x2 - l_a);
                const float e2 = row_only ? 0.f : fast_exp2(x2 - ll[k]);
                dsacc = fmaf(e1, v[e], dsacc);
                g[e] = e1 + e2;
              }
            }
            if (gi >= gj0 && gi < gj0 + 32) {
              // the diagonal entry (p_aa close to 1 once trained) is applied in fp32 by finalize_bwd_kernel
#pragma unroll
              for (int e = 0; e < 32; ++e)
                if (gj0 + e == gi) g[e] = 0.f;
            }
          }
          if (jrel0 + 32 > P.ncols) {
#pragma unroll
            for (int e = 0; e < 32; ++e)
              if (jrel0 + e >= P.ncols) g[e] = 0.f;
          }
          store_g(g, c);
        }
        tc_fence_before();
        mbar_arrive(smem_u32(&s_empty[slot0]));
      }
      fence_proxy_async_smem();
      mbar_arrive(smem_u32(g_written));
    }

    // ---- drain the accumulator: TMEM -> fp32 partial gradient
    mbar_wait(smem_u32(acc_full), 0);
    tc_fence_after();
    {
      float* dst = P.acc_part + (static_cast<size_t>(split) * P.b + li) * P.dout + f0;
      const int nvalid = min(nfb * BK, P.dout - f0);
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        const int cf = half * 128 + c * 32;
        if (cf >= nfb * BK) break;  // warp-uniform
        tmem_ld32(lane_addr + ACC_COL + cf, v);
        if (li < P.b) {
          if (cf + 32 <= nvalid) {
#pragma unroll
            for (int e4 = 0; e4 < 8; ++e4)
              *reinterpret_cast<float4*>(dst + cf + 4 * e4) =
                  make_float4(v[4 * e4], v[4 * e4 + 1], v[4 * e4 + 2], v[4 * e4 + 3]);
          } else {
#pragma unroll
            for (int e = 0; e < 32; ++e)
              if (cf + e < nvalid) dst[cf + e] = v[e];
          }
        }
      }
    }
    // d(logit_scale) row term: this CTA saw only its own column tiles -> one partial per (split, cluster
    // rank, half); written by the CTAs of the first chunk group only
    if ((MODE == MODE_CLIP || MODE == MODE_WCE_X) && P.want_ds && P.chunk0 == 0 && li < P.b)
      P.ds_part[((split * csize + crank) * 2 + half) * P.b + li] = dsacc;
  }

  tc_fence_before();
  cluster_sync_all();  // nobody leaves while a peer may still copy into / signal this CTA
  if (warp == 2) tmem_dealloc(tmem_base, TMEM_COLS);
}

constexpr int FWD_SMEM_BYTES = F_STAGES * 2 * TILE_BYTES + 2 * TILE_BYTES + 1024 + 256;  // 7 slabs
constexpr int BWD_SMEM_BYTES = X_SLABS * SLAB + 1024 + 256;

}  // namespace dsoft
