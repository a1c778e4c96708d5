// C ABI of libdsoft.so (see include/dsoft.h): plan/schedule, TMA descriptor construction, the small
// memory-bound helper kernels (pack, norms, scalars, finalize) and the launches of the tcgen05 tile
// kernels in dsoft_kernels.cuh.
#include "../../include/dsoft.h"

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>

#include "dsoft_kernels.cuh"
#include "dsoft_gy.cuh"

using namespace dsoft;

// ------------------------------------------------------------------------------------------------
// error plumbing
// ------------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

#define CUDA_TRY(expr)                                                                     \
  do {                                                                                     \
    cudaError_t e__ = (expr);                                                              \
    if (e__ != cudaSuccess)                                                                \
      return fail(static_cast<int>(e__), "%s failed: %s (%s:%d)", #expr,                   \
                  cudaGetErrorString(e__), __FILE__, __LINE__);                            \
  } while (0)

// ------------------------------------------------------------------------------------------------
// plan
// ------------------------------------------------------------------------------------------------
struct SplitPlan {
  int nsplit = 1;
  int tps = 1;  // tiles per split
};

struct dsoft_plan {
  dsoft_shape_t sh;
  int B;           // global batch
  int Bcol;        // padded length of per-column fp32 vectors
  int have_soft, have_text, have_proj, soft_local, row_only;
  int fwd_sym;         // world == 1 and fast_t: the soft forward computes the upper block triangle only
  int clip_sym;        // world == 1: one CLIP forward pass serves both directions (MODE_CLIP_SYM)
  // world > 1, global soft scope (DSOFT_SYM_W): the soft Gram matrices are symmetric, so every pair of row blocks
  // is computed by ONE of its two ranks.  Rank r owns, in column coordinates relative to its own first row
  // ("primed"), the blocks [0, W/2) - its diagonal block first - plus half of the contested block W/2 (ranks below
  // W/2: all of its columns for the rows b/2.., the others: its first b/2 columns for all rows).  The column
  // sums of the forward statistics and the transposed gradient products that belong to other ranks' rows leave
  // through two exchanges driven by the caller (dsoft_forward_phase / dsoft_backward_phase).
  int sym_w;
  int sw_ncols_a, sw_rb_half;  // row blocks < sw_rb_half own the primed columns [.., sw_ncols_a), the rest s_ncols
  size_t sc_accR3, sc_accR4;   // transposed products for other ranks' rows: [s_ncols - b][Dz] / [s_ncols - b][D]
  size_t sc_clipM, sc_clipS, sc_lse_ti, st_dbound;
  SplitPlan f_sym;     // its (triangular) column chunks
  size_t sc_colpart, sc_colsum;
  int weighted, wsym;  // denominator-modulated CE branch (loss.py:416-471); world > 1: this rank's row block
  int wnd;             // directions with a row std (1, or 2 with weight_text_symmetry)
  int lse_rows;        // per-row statistics rows of lse_local: 5, weighted world > 1 5 + 3 wnd (c, lse~, A)
  size_t st_wsig;      // weighted, world > 1: row std [B][wnd] by global row (all-gathered by the caller)
  SplitPlan f_wce;     // column split of its tile passes
  int Dz;          // student width (Dp or D)
  // packed row layout (elements)
  int offI, offT, offZ, offD, row_elems;
  int num_sms;
  // column scopes
  int ntiles_g;               // clip / global scope, 128-column tiles (fused backward)
  int s_col0, s_ncols, ntiles_s;  // soft scope; ntiles_s counts 256-column tiles (forward / logit-gradient kernels)
  int ntiles_s128;            // soft scope in 128-column tiles (fused backward)
  int fast_t;                 // teacher logit gradients in the factorised form (log2(e)/tau_t <= 60)
  SplitPlan f_clip, f_soft, b_clip, b_stu, b_txt;
  int nch_clip, nch_stu, nch_txt;
  // state layout (float offsets)
  size_t st_scal, st_rinv_t, st_rinv_z, st_rinv_d, st_diag, st_lsecols, st_colfac, st_lsestat, st_wstat, st_total;
  // scratch layout (float offsets)
  size_t sc_wpart, sc_wrows;  // weighted CE: split partials [11][npart][b], per-row results [2][WR_N][b]
  size_t sc_pc_it, sc_pc_ti, sc_ps, sc_rowloss, sc_acc1, sc_acc2, sc_acc3, sc_acc4, sc_ds1, sc_ds2,
      sc_dsrow, sc_v16, sc_total;
  // fp16 gradient-operand buffer [B][v_row]: text | image | normalised student | normalised text
  int v_offT, v_offI, v_offZn, v_offTn, v_row;
  // DSOFT_F_GMAT: two-phase backward through fp16 logit-gradient matrices in scratch
  int gmat;
  int pitch_c, pitch_s;  // columns of the CLIP / soft G matrices: multiples of 64
  size_t sc_Gci, sc_Gct, sc_Gs, sc_Gx, sc_fwd_total;
  SplitPlan g_clip, g_stu, g_txt;  // K splits of the gradient GEMMs (tps = K steps per split)
  SplitPlan g_clip_t;              // world == 1: dT = G^T . I, K runs over G's rows
  int clip_tr;                     // world == 1 two-phase: one CLIP logit-gradient matrix serves both directions
  // DSOFT_F_SIGLIP: SigLIP sigmoid loss on the image | text columns of `gathered` (its own state / scratch layout)
  int siglip;
  size_t sg_part, sg_blk;  // forward scratch: row partials [3][npart][b], per-block sums [3][blocks]
  size_t sg_Gt;            // backward scratch, world > 1: the text rows' fp16 G [bpad][pitch_c]
  // DSOFT_F_DISTILL: DistillClipLoss on image | text | teacher image | teacher text (the student and DINO slots)
  int distill;
  size_t st_ddiag;         // state: raw diagonal dot products [2 directions][student, teacher][b]
  size_t dl_part, dl_blk;  // forward scratch: row partials [2 directions][6][npart][b], per-block sums [4][blocks]
  size_t dl_col;           // backward scratch: the column side's statistics by global column [4][Bcol]
};

static int ceil_div(int a, int b) { return (a + b - 1) / b; }
// feature chunks are processed by clusters of at most X_MAXC CTAs; nch chunks -> `groups` launches
static int chunk_groups(int nch) { return ceil_div(nch, X_MAXC); }
static int chunk_cluster(int nch) { return ceil_div(nch, chunk_groups(nch)); }
static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Choose the column split so that (row blocks x splits x chunks) CTAs fill the SMs in whole waves.
// cost ~ waves x (tiles per CTA + fixed prologue/drain overhead expressed in tiles).
static SplitPlan choose_split(int row_blocks, int nchunk, int ntiles, int num_sms) {
  SplitPlan best;
  double best_cost = 1e300;
  const int max_split = std::min(ntiles, 64);
  for (int ns = 1; ns <= max_split; ++ns) {
    const int tps = ceil_div(ntiles, ns);
    const int ns_eff = ceil_div(ntiles, tps);
    const long ctas = static_cast<long>(row_blocks) * nchunk * ns_eff;
    const long waves = (ctas + num_sms - 1) / num_sms;
    const double cost = static_cast<double>(waves) * (tps + 1.5);
    if (cost < best_cost - 1e-9) {
      best_cost = cost;
      best.nsplit = ns_eff;
      best.tps = tps;
    }
  }
  return best;
}

// K split of a gradient GEMM: `tiles` CTA pairs per split on num_sms / 2 pair slots.  Cost model: whole waves of
// pair slots x (K steps per CTA + a fixed prologue / drain overhead in K steps); e.g. 96 tiles (b = 8192, Dout = 768)
// on 74 slots run as 2 waves unsplit (the second 30 % full) but as 4 full waves with a 3-way split.
// Every extra split also costs one more [b x Dout] fp32 partial to write and to read back in finalize_bwd (~2.5 TB/s
// there), expressed in K-step times of a CTA pair (512 clocks ~ 0.27 us).
static SplitPlan choose_gy_split(int tiles, int ksteps, int num_sms, int b, int dout) {
  const double split_penalty = static_cast<double>(b) * dout / 84375.0;
  const int slots = std::max(1, num_sms / 2);
  const int max_ns = std::min(32, std::max(1, ksteps / 4));  // at least 4 K steps (256 columns) per split
  int best = 1;
  double best_cost = 1e300;
  for (int ns = 1; ns <= max_ns; ++ns) {
    const int tps = ceil_div(ksteps, ns);
    const int ns_eff = ceil_div(ksteps, tps);
    const long waves = (static_cast<long>(tiles) * ns_eff + slots - 1) / slots;
    const double cost = static_cast<double>(waves) * (tps + 8.0) + split_penalty * (ns_eff - 1);
    if (cost < 0.95 * best_cost) {  // more splits only for a clear gain (the model is coarse)
      best_cost = cost;
      best = ns_eff;
    }
  }
  SplitPlan sp;
  sp.tps = ceil_div(ksteps, best);
  sp.nsplit = ceil_div(ksteps, sp.tps);
  return sp;
}

extern "C" int dsoft_version(void) { return DSOFT_VERSION; }
extern "C" const char* dsoft_last_error(void) { return g_err; }

static int query_num_sms(int* out) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return fail(DSOFT_ENODEV, "cudaGetDevice: %s", cudaGetErrorString(e));
  int major = 0, sms = 0;
  CUDA_TRY(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  if (major != 10)
    return fail(DSOFT_ENODEV, "libdsoft needs an sm_100 (B200) device, found compute capability %d.x",
                major);
  *out = sms;
  return 0;
}

extern "C" int dsoft_plan_create(const dsoft_shape_t* sh, dsoft_plan_t** out) {
  if (!sh || !out) return fail(DSOFT_EINVAL, "null argument");
  if (sh->b <= 0 || sh->world <= 0 || sh->rank < 0 || sh->rank >= sh->world)
    return fail(DSOFT_EINVAL, "bad b/world/rank (%d/%d/%d)", sh->b, sh->world, sh->rank);
  if (sh->D <= 0 || sh->D % 8 || sh->Dp < 0 || sh->Dp % 8 || sh->Dd < 0 || sh->Dd % 8)
    return fail(DSOFT_EINVAL, "feature dims must be positive multiples of 8 (D=%d Dp=%d Dd=%d)", sh->D,
                sh->Dp, sh->Dd);
  if (sh->world > 1 && sh->b % 8)
    return fail(DSOFT_EINVAL, "local batch must be a multiple of 8 when world > 1 (b=%d)", sh->b);
  const bool soft = (sh->flags & DSOFT_F_SOFT) != 0;
  if (soft && sh->Dd == 0) return fail(DSOFT_EINVAL, "DSOFT_F_SOFT needs Dd > 0");
  if ((sh->flags & DSOFT_F_TEXT) && !soft) return fail(DSOFT_EINVAL, "DSOFT_F_TEXT needs DSOFT_F_SOFT");
  if (soft && !(sh->teacher_temp > 0.f)) return fail(DSOFT_EINVAL, "teacher_temp must be > 0");
  if ((sh->flags & DSOFT_F_TEXT) && !(sh->text_temp > 0.f))
    return fail(DSOFT_EINVAL, "text_temp must be > 0");
  if (sh->flags & DSOFT_F_WEIGHTED) {
    // world > 1 (the reference fails there, loss.py:423-446): this rank's row block of the global B x B problem,
    // beta from the row stds of all B rows (dsoft_forward_phase 5, exchange, 6)
    if (sh->Dd == 0) return fail(DSOFT_EINVAL, "DSOFT_F_WEIGHTED needs Dd > 0");
    if (!(sh->c_clip > 0.f)) return fail(DSOFT_EINVAL, "c_clip must be > 0");
  }
  if ((sh->flags & DSOFT_F_SIGLIP) && (sh->flags != DSOFT_F_SIGLIP || sh->Dp != 0 || sh->Dd != 0))
    return fail(DSOFT_EINVAL, "DSOFT_F_SIGLIP takes no other flag and needs Dp = Dd = 0");
  if (sh->flags & DSOFT_F_DISTILL) {
    const uint32_t other = sh->flags & ~(DSOFT_F_DISTILL | (sh->world > 1 ? DSOFT_F_ROW_ONLY : 0u));
    if (other)
      return fail(DSOFT_EINVAL, "DSOFT_F_DISTILL takes no other flag than DSOFT_F_ROW_ONLY at world > 1 (flags %u)",
                  sh->flags);
    if (sh->Dd <= 0 || sh->Dp != sh->Dd)
      return fail(DSOFT_EINVAL, "DSOFT_F_DISTILL needs Dp = Dd > 0, the teacher width (Dp=%d Dd=%d)", sh->Dp, sh->Dd);
  }
  if (static_cast<long>(sh->b) * sh->world > (1L << 30)) return fail(DSOFT_EINVAL, "batch too large");
  if (sh->D > 2048 || sh->Dp > 2048) return fail(DSOFT_EINVAL, "feature dims above 2048 are not supported");

  int sms = 0;
  int rc = query_num_sms(&sms);
  if (rc) return rc;

  dsoft_plan* p = new (std::nothrow) dsoft_plan();
  if (!p) return fail(DSOFT_EINVAL, "out of host memory");
  p->sh = *sh;
  p->num_sms = sms;
  p->B = sh->b * sh->world;
  p->Bcol = ceil_div(p->B, 2 * BN) * 2 * BN + 2 * BN;  // 256-column tiles may start anywhere up to B - 8
  p->have_soft = soft;
  p->have_text = (sh->flags & DSOFT_F_TEXT) != 0;
  p->have_proj = soft && sh->Dp > 0;
  p->weighted = (sh->flags & DSOFT_F_WEIGHTED) != 0;
  p->wsym = p->weighted && (sh->flags & DSOFT_F_WSYM) != 0;
  p->wnd = p->wsym ? 2 : 1;
  p->lse_rows = (p->weighted && sh->world > 1) ? 5 + 3 * p->wnd : 5;
  p->soft_local = (sh->flags & DSOFT_F_SOFT_LOCAL) != 0 && sh->world > 1;
  p->row_only = (sh->flags & DSOFT_F_ROW_ONLY) != 0 && sh->world > 1;
  p->Dz = p->have_proj ? sh->Dp : sh->D;

  p->offI = 0;
  p->offT = sh->D;
  p->offZ = p->have_proj ? 2 * sh->D : 0;
  p->offD = 2 * sh->D + (p->have_proj ? sh->Dp : 0);
  p->row_elems = p->offD + ((soft || p->weighted) ? sh->Dd : 0);

  const int rbs = ceil_div(sh->b, BM);
  p->ntiles_g = ceil_div(p->B, BN);
  p->s_col0 = p->soft_local ? sh->rank * sh->b : 0;
  p->s_ncols = p->soft_local ? sh->b : p->B;
  {
    // DSOFT_SYM_W: 0 = never, 1 = whenever the plan allows it, unset = only for per-rank blocks above 2^28 similarity
    // entries.  Below that the step is a few milliseconds of short kernels and the two extra exchanges (about 25
    // small torch / NCCL calls per step) cost the eager step more than the halved soft tiles save: global batch 32768
    // on 8 GPUs 2.56 ms with the shared tiles against 2.47 ms without (4 GPUs: 5.29 against 4.41 ms; replayed as a
    // CUDA graph 4.20 ms), on 2 GPUs 7.4 ms against 8.85 ms.  DESIGN.md section 6.
    const char* e = getenv("DSOFT_SYM_W");
    const bool big = static_cast<double>(sh->b) * p->B > 268435456.0;
    // weighted plans never share soft tiles (their forward has its own exchange)
    p->sym_w = soft && sh->world > 1 && !p->soft_local && !p->row_only && (sh->flags & DSOFT_F_GMAT) && !p->weighted &&
               1.4426950408889634 / sh->teacher_temp <= 60.0 && sh->b % 512 == 0 &&
               (e ? e[0] != '0' : big);
    p->sw_ncols_a = 0;
    p->sw_rb_half = 0;
    if (p->sym_w) {
      const int W = sh->world, r = sh->rank, b = sh->b;
      const int nfull = (W % 2) ? (W + 1) / 2 : W / 2;
      p->s_col0 = r * b;
      p->s_ncols = p->sw_ncols_a = nfull * b;
      if (W % 2 == 0) {
        if (r < W / 2) {
          p->s_ncols = (nfull + 1) * b;
          p->sw_rb_half = (b / 2) / BM;
        } else {
          p->s_ncols = p->sw_ncols_a = nfull * b + b / 2;
        }
      }
    }
  }
  p->ntiles_s = ceil_div(p->s_ncols, 2 * BN);
  p->ntiles_s128 = ceil_div(p->s_ncols, BN);
  p->fast_t = soft && (1.4426950408889634 / sh->teacher_temp <= 60.0);
  p->nch_clip = ceil_div(sh->D, CHUNK_F);
  p->nch_stu = ceil_div(p->Dz, CHUNK_F);
  p->nch_txt = ceil_div(sh->D, CHUNK_F);
  p->f_clip = choose_split(rbs, 1, ceil_div(p->B, 2 * BN), sms);  // forward CLIP kernel uses 256-column tiles
  p->f_soft = choose_split(rbs, 1, p->ntiles_s, sms);
  p->f_wce = choose_split(rbs, 1, ceil_div(p->B, 2 * BN), sms);
  {
    // symmetric forward: needs one rank (the row block is the whole square), the fixed teacher maximum, and more
    // than one row pair (otherwise there is nothing to save)
    p->fwd_sym = soft && (sh->world == 1 || p->sym_w) && p->fast_t && rbs > 2;
    p->f_sym.tps = std::max(4, ceil_div(p->ntiles_s, 10));
    p->f_sym.nsplit = ceil_div(p->ntiles_s, p->f_sym.tps);
  }
  {
    // one-pass CLIP forward: the row block must be the whole square (one rank); DSOFT_CLIP_SYM=0 keeps two passes
    const char* e = getenv("DSOFT_CLIP_SYM");
    p->clip_sym = sh->world == 1 && rbs > 2 && !(e && e[0] == '0');
  }
  p->b_clip = choose_split(rbs, p->nch_clip, p->ntiles_g, sms);
  p->b_stu = choose_split(rbs, p->nch_stu, p->ntiles_s128, sms);
  p->b_txt = choose_split(rbs, p->nch_txt, p->ntiles_s128, sms);
  p->gmat = (sh->flags & DSOFT_F_GMAT) != 0;
  p->pitch_c = ceil_div(p->B, 64) * 64;
  p->pitch_s = ceil_div(p->s_ncols, 64) * 64;
  if (p->gmat) {
    const int pairs = ceil_div(rbs, 2);
    p->g_clip = choose_gy_split(pairs * ceil_div(sh->D, GY_N), p->pitch_c / 64, sms, sh->b, sh->D);
    p->g_stu = choose_gy_split(pairs * ceil_div(p->Dz, GY_N), p->pitch_s / 64, sms, sh->b, p->Dz);
    p->g_txt = choose_gy_split(pairs * ceil_div(sh->D, GY_N), p->pitch_s / 64, sms, sh->b, sh->D);
    p->clip_tr = sh->world == 1;
    p->g_clip_t = choose_gy_split(pairs * ceil_div(sh->D, GY_N), rbs * 2, sms, sh->b, sh->D);
  }

  // ---- state (floats)
  size_t o = 0;
  auto take = [&](size_t n) { size_t r = o; o = align_up(o + n, 64); return r; };
  if (sh->flags & DSOFT_F_SIGLIP) {
    // state: the scalar block (s, beta, the forward's sums of G x and G).  Forward scratch: the row partials.
    // Backward scratch: the gradient GEMMs' split partials, the fp16 text | image operands and, at world > 1, the
    // text rows' G.  The image rows' G is the caller's (dsoft_siglip_g_bytes).
    const int pairs = ceil_div(rbs, 2);
    p->siglip = 1;
    p->clip_tr = sh->world == 1;
    p->g_clip = choose_gy_split(pairs * ceil_div(sh->D, GY_N), p->pitch_c / 64, sms, sh->b, sh->D);
    p->g_clip_t = choose_gy_split(pairs * ceil_div(sh->D, GY_N), rbs * 2, sms, sh->b, sh->D);
    p->st_scal = take(SC_COUNT);
    p->st_total = o;
    o = 0;
    p->sg_part = take(static_cast<size_t>(3) * 2 * p->f_clip.nsplit * sh->b);
    p->sg_blk = take(static_cast<size_t>(3) * ceil_div(sh->b, 128));
    p->sc_fwd_total = o;
    const size_t ns_t = p->clip_tr ? p->g_clip_t.nsplit : p->g_clip.nsplit;
    p->sc_acc1 = take(static_cast<size_t>(p->g_clip.nsplit) * sh->b * sh->D);
    p->sc_acc2 = take(ns_t * sh->b * sh->D);
    p->v_offT = 0;
    p->v_offI = sh->D;
    p->v_row = 2 * sh->D;
    p->sc_v16 = take(static_cast<size_t>(p->B) * p->v_row / 2 + 1);
    p->sg_Gt = take(p->clip_tr ? 0 : static_cast<size_t>(rbs) * BM * p->pitch_c / 2);
    p->sc_total = o;
    *out = p;
    return 0;
  }
  if (sh->flags & DSOFT_F_DISTILL) {
    // packed row: image | text | teacher image | teacher text (dsoft_pack's student and DINO slots).  State: the
    // scalar block and the diagonal dot products.  Forward scratch: the row partials of both directions.  Backward
    // scratch: the column-side statistics, the gradient GEMMs' split partials and the fp16 text | image operands.
    // The logit-gradient matrix is the caller's (dsoft_distill_g_bytes); at world > 1 the text rows reuse it.
    const int pairs = ceil_div(rbs, 2);
    p->distill = 1;
    p->Dz = sh->Dd;
    p->offZ = 2 * sh->D;
    p->offD = 2 * sh->D + sh->Dd;
    p->row_elems = 2 * sh->D + 2 * sh->Dd;
    p->clip_tr = sh->world == 1;
    p->g_clip = choose_gy_split(pairs * ceil_div(sh->D, GY_N), p->pitch_c / 64, sms, sh->b, sh->D);
    p->g_clip_t = choose_gy_split(pairs * ceil_div(sh->D, GY_N), rbs * 2, sms, sh->b, sh->D);
    p->st_scal = take(SC_COUNT);
    p->st_ddiag = take(static_cast<size_t>(4) * sh->b);
    p->st_total = o;
    o = 0;
    p->dl_part = take(static_cast<size_t>(2) * 6 * 2 * p->f_wce.nsplit * sh->b);
    p->dl_blk = take(static_cast<size_t>(4) * ceil_div(2 * sh->b, 128));
    p->sc_fwd_total = o;
    const size_t ns_t = p->clip_tr ? p->g_clip_t.nsplit : p->g_clip.nsplit;
    p->dl_col = take(static_cast<size_t>(4) * p->Bcol);
    p->sc_acc1 = take(static_cast<size_t>(p->g_clip.nsplit) * sh->b * sh->D);
    p->sc_acc2 = take(ns_t * sh->b * sh->D);
    p->v_offT = 0;
    p->v_offI = sh->D;
    p->v_row = 2 * sh->D;
    p->sc_v16 = take(static_cast<size_t>(p->B) * p->v_row / 2 + 1);
    p->sc_total = o;
    *out = p;
    return 0;
  }
  p->st_scal = take(SC_COUNT);
  p->st_rinv_t = take(p->Bcol);
  p->st_rinv_z = take(p->Bcol);
  p->st_rinv_d = take(p->Bcol);
  p->st_diag = take(sh->b);
  p->st_dbound = take(p->Bcol);
  p->st_lsecols = take(static_cast<size_t>(5) * p->Bcol);
  p->st_colfac = take(static_cast<size_t>(5) * p->Bcol);
  p->st_lsestat = take(2 * 64);
  p->st_wstat = take(p->weighted ? static_cast<size_t>(8) * p->Bcol : 0);
  p->st_wsig = take(p->weighted && sh->world > 1 ? static_cast<size_t>(p->wnd) * p->B : 0);
  p->st_total = o;

  // ---- scratch (floats)
  o = 0;
  const size_t b = sh->b;
  p->sc_pc_it = take(2 * (p->clip_sym ? 4 : 2) * p->f_clip.nsplit * b);
  p->sc_pc_ti = take(2 * 2 * p->f_clip.nsplit * b);
  p->sc_ps = take(soft ? 7 * 2 * std::max(p->f_soft.nsplit, p->fwd_sym ? p->f_sym.nsplit : 0) * b : 0);
  p->sc_colpart = take(p->fwd_sym ? static_cast<size_t>(6) * (4 * rbs) * p->Bcol : 0);
  p->sc_colsum = take(p->fwd_sym ? static_cast<size_t>(6) * p->Bcol : 0);
  p->sc_clipM = take(p->clip_sym ? static_cast<size_t>(4 * rbs) * p->Bcol : 0);
  p->sc_clipS = take(p->clip_sym ? static_cast<size_t>(4 * rbs) * p->Bcol : 0);
  p->sc_lse_ti = take(p->clip_sym ? p->Bcol : 0);
  p->sc_rowloss = take(3 * b);
  p->sc_wpart = take(p->weighted ? 11 * 2 * p->f_wce.nsplit * b : 0);
  p->sc_wrows = take(p->weighted ? 2 * 10 * b : 0);
  p->sc_fwd_total = o;  // the forward only needs the statistics partials above
  const size_t ns_c = p->gmat ? std::max(p->g_clip.nsplit, p->g_clip_t.nsplit) : p->b_clip.nsplit;
  const size_t ns_s = p->gmat ? p->g_stu.nsplit : p->b_stu.nsplit;
  const size_t ns_x = p->gmat ? p->g_txt.nsplit : p->b_txt.nsplit;
  p->sc_acc1 = take(ns_c * b * sh->D);
  p->sc_acc2 = take(ns_c * b * sh->D);
  p->sc_acc3 = take(soft ? ns_s * b * p->Dz : 0);
  p->sc_acc4 = take(p->have_text ? ns_x * b * sh->D : 0);
  p->sc_accR3 = take(p->sym_w ? static_cast<size_t>(p->s_ncols - sh->b) * p->Dz : 0);
  p->sc_accR4 = take(p->sym_w && p->have_text ? static_cast<size_t>(p->s_ncols - sh->b) * sh->D : 0);
  const size_t nds_g = 2 * std::max(p->f_clip.nsplit, p->weighted ? p->f_wce.nsplit : 0);
  p->sc_ds1 = take(p->gmat ? nds_g * b : 2 * X_MAXC * p->b_clip.nsplit * b);
  p->sc_ds2 = take(p->gmat ? nds_g * b : 2 * X_MAXC * p->b_clip.nsplit * b);
  p->sc_dsrow = take(b);
  if (p->gmat) {
    const size_t bpad = static_cast<size_t>(rbs) * BM;  // blocked layout holds whole 128-row blocks
    p->sc_Gci = take(bpad * p->pitch_c / 2);
    p->sc_Gct = take(p->clip_tr ? 0 : bpad * p->pitch_c / 2);
    p->sc_Gs = take(soft ? bpad * p->pitch_s / 2 : 0);
    p->sc_Gx = take(p->have_text ? bpad * p->pitch_s / 2 : 0);
  }
  p->v_offT = 0;
  p->v_offI = sh->D;
  p->v_offZn = 2 * sh->D;
  p->v_offTn = 2 * sh->D + (soft ? p->Dz : 0);
  p->v_row = p->v_offTn + (p->have_text ? sh->D : 0);
  p->sc_v16 = take(static_cast<size_t>(p->B) * p->v_row / 2 + 1);
  p->sc_total = o;

  *out = p;
  return 0;
}

extern "C" void dsoft_plan_destroy(dsoft_plan_t* plan) { delete plan; }

extern "C" size_t dsoft_plan_gathered_row_elems(const dsoft_plan_t* p) { return p ? p->row_elems : 0; }
extern "C" size_t dsoft_plan_gathered_bytes(const dsoft_plan_t* p) {
  return p ? static_cast<size_t>(p->B) * p->row_elems * 2 : 0;
}
extern "C" size_t dsoft_plan_state_bytes(const dsoft_plan_t* p) { return p ? p->st_total * 4 : 0; }
extern "C" size_t dsoft_plan_scratch_bytes(const dsoft_plan_t* p) { return p ? p->sc_total * 4 : 0; }
extern "C" size_t dsoft_plan_forward_scratch_bytes(const dsoft_plan_t* p) { return p ? p->sc_fwd_total * 4 : 0; }

extern "C" double dsoft_plan_algorithmic_flops(const dsoft_plan_t* p) {
  if (!p) return 0.0;
  if (p->siglip) return 2.0 * p->sh.b * p->B * (3.0 * p->sh.D);  // I . T^T, G . T, G^T . I
  if (p->distill) {  // forward: both products per direction; G: both products once (world 1) or per direction
    const double pr = p->sh.D + p->sh.Dd;
    return 2.0 * p->sh.b * p->B * (2.0 * pr + (p->clip_tr ? 1.0 : 2.0) * pr + 2.0 * p->sh.D);
  }
  // SURVEY.md 8(d): F_alg = 2 B^2 (3D + 2Dp + Dd [+ 2D]) for the whole job; this rank's share is 1/W.
  const double b = p->sh.b, cols_c = p->B, cols_s = p->sym_w ? p->B : p->s_ncols;
  double f = 2.0 * b * cols_c * (3.0 * p->sh.D);
  if (p->have_soft) f += 2.0 * b * cols_s * (2.0 * p->Dz + p->sh.Dd);
  if (p->have_text) f += 2.0 * b * cols_s * (2.0 * p->sh.D);
  return f;
}
// Per tile-kernel FLOP accounting (index = profile kind): algorithmic share per SURVEY 8(d) and the FLOPs
// the kernel really executes (recompute per 256-feature chunk included).  Both for this rank.
extern "C" int dsoft_plan_kernel_flops(const dsoft_plan_t* p, double* algorithmic, double* executed, int n) {
  if (!p || !algorithmic || !executed || n < 7) return fail(DSOFT_EINVAL, "need 7 slots");
  const double b = p->sh.b, Bc = p->B, Bs = p->sym_w ? p->B : p->s_ncols, D = p->sh.D, Dz = p->Dz, Dd = p->sh.Dd;
  const double sw = p->sym_w ? 0.5 : 1.0;  // symmetric ownership across ranks: half of the soft tiles per rank
  for (int k = 0; k < n; ++k) algorithmic[k] = executed[k] = 0.0;
  if (p->siglip) {  // [0] forward tile kernel, [3] / [4] gradient GEMMs, [7] world > 1: the text rows' G kernel
    algorithmic[0] = executed[0] = algorithmic[3] = executed[3] = algorithmic[4] = executed[4] = 2.0 * b * Bc * D;
    if (n > 7 && !p->clip_tr) executed[7] = 2.0 * b * Bc * D;
    return 0;
  }
  if (p->distill) {  // [0] / [1] forward image / text rows, [3] / [4] gradient GEMMs, [7] the logit-gradient kernel
    algorithmic[0] = executed[0] = algorithmic[1] = executed[1] = 2.0 * b * Bc * (D + Dd);
    algorithmic[3] = executed[3] = algorithmic[4] = executed[4] = 2.0 * b * Bc * D;
    if (n > 7) algorithmic[7] = executed[7] = (p->clip_tr ? 1.0 : 2.0) * 2.0 * b * Bc * (D + Dd);
    return 0;
  }
  // forward CLIP: the two directions are exact transposes -> one algorithmic product, two executed
  algorithmic[0] = algorithmic[1] = b * Bc * D;
  executed[0] = executed[1] = 2.0 * b * Bc * D;
  if (p->clip_sym) {  // one pass: the product is computed once
    algorithmic[0] = 2.0 * b * Bc * D;
    algorithmic[1] = executed[1] = 0.0;
  }
  algorithmic[3] = algorithmic[4] = 2.0 * b * Bc * D;
  executed[3] = executed[4] = 2.0 * b * Bc * D * (chunk_groups(p->nch_clip) + 1.0);
  if (p->weighted)  // fused weighted CE backward: the CLIP and the DINO product per chunk group, then G . Y
    executed[3] = executed[4] = 2.0 * b * Bc * (chunk_groups(p->nch_clip) * (D + Dd) + D);
  if (p->have_soft) {
    algorithmic[2] = executed[2] = 2.0 * b * Bs * (Dz + Dd + (p->have_text ? D : 0.0));
    if (p->fwd_sym) executed[2] *= 0.5 * (1.0 + 256.0 / std::max(256.0, Bs));  // upper block triangle + diagonal tiles
    algorithmic[5] = 2.0 * b * Bs * Dz;
    executed[5] = 2.0 * b * Bs * (chunk_groups(p->nch_stu) * (Dz + Dd) + Dz);
  }
  if (p->have_text) {
    algorithmic[6] = 2.0 * b * Bs * D;
    executed[6] = 2.0 * b * Bs * (chunk_groups(p->nch_txt) * (D + Dd) + D);
  }
  if (p->gmat) {
    // two-phase backward: slots 3..6 are the plain gradient GEMMs, slots 7 / 8 the logit-gradient kernels
    // (every similarity product recomputed once; the teacher product once for student and text)
    for (int k = 3; k < 7; ++k) executed[k] = algorithmic[k];
    if (n > 7) executed[7] = (p->clip_tr ? 1.0 : 2.0) * (2.0 * b * Bc * D);
    if (n > 8 && p->have_soft)  // world == 1: only the upper block triangle (plus the 256-wide diagonal blocks)
      executed[8] = ((p->clip_tr || p->sym_w) ? 0.5 * (1.0 + 256.0 / std::max(256.0, Bs)) : 1.0) * 2.0 * b * Bs *
                    (Dz + Dd + (p->have_text ? D : 0.0));
    (void)sw;
  }
  return 0;
}

extern "C" int dsoft_plan_launches_forward(const dsoft_plan_t* p) {
  if (!p) return 0;
  if (p->siglip) return 3;  // scalars, tile kernel, finalize
  if (p->distill) return 4;  // scalars, tile kernel x 2 directions, finalize
  return 1 /*pack*/ + 1 /*scalars*/ + 1 /*norms*/ + 2 /*clip x2*/ + (p->have_soft ? 1 : 0) + (p->fwd_sym ? 1 : 0) +
         1 /*finalize*/ + (p->weighted ? (p->wsym ? 2 : 1) * 7 + 1 : 0);
}
extern "C" int dsoft_plan_launches_backward(const dsoft_plan_t* p) {
  if (!p) return 0;
  if (p->siglip) return p->clip_tr ? 4 : 5;  // fp16 operands, [text rows' G,] two gradient GEMMs, finalize
  if (p->distill) return p->clip_tr ? 6 : 7;  // scalars + relayout, fp16 operands, G (x 2), two GEMMs, finalize
  if (p->gmat)
    return 3 /*lse stats, relayout, fp16 operands*/ + (p->weighted && !p->clip_tr ? 1 : 0) /*weighted relayout*/ +
           (p->clip_tr ? 1 : 2) /*clip G*/ + 2 /*clip GEMMs*/ +
           (p->have_soft ? 2 : 0) /*soft G, student GEMM*/ + (p->have_text ? 1 : 0) + 1 /*finalize*/;
  return 3 /*lse stats, relayout, fp16 operands*/ + (p->weighted && p->sh.world > 1 ? 1 : 0) /*weighted relayout*/ +
         2 * chunk_groups(p->nch_clip) /*clip, or weighted CE*/ + (p->have_soft ? chunk_groups(p->nch_stu) : 0) +
         (p->have_text ? chunk_groups(p->nch_txt) : 0) + 1 /*finalize*/;
}

// ------------------------------------------------------------------------------------------------
// TMA descriptors
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(sym);
  }
  return fn;
}

// bf16 matrix [rows][cols] with row pitch `pitch_elems`; box = 64 columns x 128 rows, 128B swizzle.
static int make_map(CUtensorMap* map, const void* base, int rows, int cols, size_t pitch_elems,
                    CUtensorMapDataType dt = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, int box_rows = BM, int box_cols = BK) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) return fail(DSOFT_ENODEV, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  cuuint64_t strides[1] = {static_cast<cuuint64_t>(pitch_elems) * 2};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(box_cols), static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, dt, 2, const_cast<void*>(base), dims, strides, box,
                   estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   box_cols * 2 == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return fail(DSOFT_ETMA, "cuTensorMapEncodeTiled failed (%d) base=%p rows=%d cols=%d pitch=%zu",
                static_cast<int>(r), base, rows, cols, pitch_elems);
  return 0;
}

// box_rows: 128 = one TMA box per operand tile; 64 = half tiles (CTA pairs stage half a column tile each)
static int make_maps(const dsoft_plan* p, const void* gathered, TileMaps* tm, int box_rows = BM) {
  const __nv_bfloat16* g = static_cast<const __nv_bfloat16*>(gathered);
  if (reinterpret_cast<uintptr_t>(g) % 16) return fail(DSOFT_EINVAL, "gathered buffer must be 16-byte aligned");
  const CUtensorMapDataType bf = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  int rc;
  if ((rc = make_map(&tm->m[0], g + p->offI, p->B, p->sh.D, p->row_elems, bf, box_rows))) return rc;
  if ((rc = make_map(&tm->m[1], g + p->offT, p->B, p->sh.D, p->row_elems, bf, box_rows))) return rc;
  if ((rc = make_map(&tm->m[2], g + p->offZ, p->B, p->Dz, p->row_elems, bf, box_rows))) return rc;
  if (p->have_soft || p->weighted || p->distill) {
    if ((rc = make_map(&tm->m[3], g + p->offD, p->B, p->sh.Dd, p->row_elems, bf, box_rows))) return rc;
  } else {
    tm->m[3] = tm->m[0];
  }
  tm->g[0] = tm->g[1] = tm->m[0];  // only the logit-gradient launches replace (and use) these
  return 0;
}

// ------------------------------------------------------------------------------------------------
// helper kernels (memory bound, tiny next to the tile kernels)
// ------------------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ float to_f32(T x);
template <>
__device__ __forceinline__ float to_f32<float>(float x) { return x; }
template <>
__device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 x) { return __bfloat162float(x); }
template <>
__device__ __forceinline__ float to_f32<__half>(__half x) { return __half2float(x); }

// All local matrices (image, text, student, dino; any float type, row stride ld) -> bf16 column slices of the
// packed rows, in ONE launch.
struct PackSrc {
  const void* src;
  int dtype;      // DSOFT_DT_*
  int64_t ld;     // elements
  int cols;
  int dst_off;    // column offset in the packed row
};
struct PackArgs {
  PackSrc m[4];
  int nmat, rows;
  int64_t dst_ld;
  int64_t pairs_end[4];  // prefix sums of rows * cols / 2
};

__device__ __forceinline__ float2 load_pair(const void* src, int dtype, int64_t idx) {
  if (dtype == DSOFT_DT_F32) {
    const float2 v = *reinterpret_cast<const float2*>(static_cast<const float*>(src) + idx);
    return v;
  } else if (dtype == DSOFT_DT_BF16) {
    return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(static_cast<const __nv_bfloat16*>(src) + idx));
  }
  return __half22float2(*reinterpret_cast<const __half2*>(static_cast<const __half*>(src) + idx));
}

// fast path: every source has 16-byte aligned rows -> 8 elements per thread and iteration (two 16-byte loads of
// fp32, or one of bf16 / fp16; one 16-byte store).  pairs_end counts pairs, so an octet index is a quarter of it.
__global__ void __launch_bounds__(256) pack_rows8_kernel(PackArgs a, __nv_bfloat16* __restrict__ dst) {
  const int64_t total = a.pairs_end[a.nmat - 1] / 4;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    int k = 0;
    while (i >= a.pairs_end[k] / 4) ++k;
    const int64_t j = i - (k ? a.pairs_end[k - 1] / 4 : 0);
    const PackSrc& m = a.m[k];
    const int oct_cols = m.cols / 8;
    const int r = static_cast<int>(j / oct_cols);
    const int c = static_cast<int>(j % oct_cols) * 8;
    const int64_t idx = r * m.ld + c;
    uint4 o;
    if (m.dtype == DSOFT_DT_F32) {
      const float4 x0 = __ldcs(reinterpret_cast<const float4*>(static_cast<const float*>(m.src) + idx));
      const float4 x1 = __ldcs(reinterpret_cast<const float4*>(static_cast<const float*>(m.src) + idx + 4));
      o = make_uint4(pack_bf16x2(x0.x, x0.y), pack_bf16x2(x0.z, x0.w), pack_bf16x2(x1.x, x1.y),
                     pack_bf16x2(x1.z, x1.w));
    } else if (m.dtype == DSOFT_DT_BF16) {
      o = __ldcs(reinterpret_cast<const uint4*>(static_cast<const __nv_bfloat16*>(m.src) + idx));
    } else {
      const uint4 raw = __ldcs(reinterpret_cast<const uint4*>(static_cast<const __half*>(m.src) + idx));
      const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
      uint32_t ow[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[q]));
        ow[q] = pack_bf16x2(f.x, f.y);
      }
      o = make_uint4(ow[0], ow[1], ow[2], ow[3]);
    }
    *reinterpret_cast<uint4*>(dst + r * a.dst_ld + m.dst_off + c) = o;
  }
}

__global__ void pack_rows_kernel(PackArgs a, __nv_bfloat16* __restrict__ dst) {
  const int64_t total = a.pairs_end[a.nmat - 1];
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    int k = 0;
    while (i >= a.pairs_end[k]) ++k;
    const int64_t j = i - (k ? a.pairs_end[k - 1] : 0);
    const PackSrc& m = a.m[k];
    const int half_cols = m.cols / 2;
    const int r = static_cast<int>(j / half_cols);
    const int c = static_cast<int>(j % half_cols) * 2;
    const float2 x = load_pair(m.src, m.dtype, r * m.ld + c);
    *reinterpret_cast<__nv_bfloat162*>(dst + r * a.dst_ld + m.dst_off + c) = __floats2bfloat162_rn(x.x, x.y);
  }
}

// one warp per row: out[r] = 1 / max(||row||, 1e-12)  (F.normalize eps, loss.py:345-359, 392); grid.y selects
// the matrix (text / student / dino); the per-matrix minimum feeds the power-of-two operand scale sigma
struct RinvArgs {
  const __nv_bfloat16* mat[3];
  int cols[3];
  float* out[3];
  float* rmin[3];
  int64_t ld;
  int rows, out_len;
  const __nv_bfloat16* dot_mat;  // optional (matrix 0 only): dot_out[r] = <mat[0] row r, dot_mat row r>, the CLIP
  float* dot_out;                // diagonal logit / scale = a lower bound of row r's and column r's log-sum-exp
};
constexpr int RINV_ROWS_PER_WARP = 4;
__global__ void __launch_bounds__(256) rinv_kernel(RinvArgs a) {
  __shared__ float wmin[8];
  const int k = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* out = a.out[k];
  const int ncol8 = a.cols[k] / 8;  // feature widths are multiples of 8: 16-byte loads
  float mn = __int_as_float(0x7f800000);
  for (int q = 0; q < RINV_ROWS_PER_WARP; ++q) {
    const int r = (blockIdx.x * 8 + warp) * RINV_ROWS_PER_WARP + q;
    if (r >= a.out_len) break;
    const bool want_dot = k == 0 && a.dot_out != nullptr;
    if (r >= a.rows) {
      if (lane == 0) {
        out[r] = 0.f;
        if (want_dot) a.dot_out[r] = 3.0e38f;  // padded columns never make a chunk look risky
      }
      continue;
    }
    const uint4* p = reinterpret_cast<const uint4*>(a.mat[k] + r * a.ld);
    float acc = 0.f, dot = 0.f;
    if (want_dot) {
      const uint4* p2 = reinterpret_cast<const uint4*>(a.dot_mat + r * a.ld);
      for (int c = lane; c < ncol8; c += 32) {
        const uint4 raw = __ldg(p + c), raw2 = __ldg(p2 + c);
        const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w}, w2[4] = {raw2.x, raw2.y, raw2.z, raw2.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[j]));
          const float2 g = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w2[j]));
          acc = fmaf(f.x, f.x, acc);
          acc = fmaf(f.y, f.y, acc);
          dot = fmaf(f.x, g.x, dot);
          dot = fmaf(f.y, g.y, dot);
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
      if (lane == 0) a.dot_out[r] = dot;
    } else {
      for (int c = lane; c < ncol8; c += 32) {
        const uint4 raw = __ldg(p + c);
        const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[j]));
          acc = fmaf(f.x, f.x, acc);
          acc = fmaf(f.y, f.y, acc);
        }
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    const float rv = 1.f / fmaxf(sqrtf(acc), 1e-12f);
    if (lane == 0) out[r] = rv;
    mn = fminf(mn, rv);
  }
  // one atomic per block (per row they serialise on a single address)
  if (lane == 0) wmin[warp] = mn;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < 8; ++w) mn = fminf(mn, wmin[w]);
    if (mn < __int_as_float(0x7f800000))
      atomicMin(reinterpret_cast<int*>(a.rmin[k]), __float_as_int(mn));  // positive floats order like ints
  }
}

// compute_student_tau (loss.py:166-175) + temperature reciprocals, all on device
__global__ void prep_scalars_kernel(const float* __restrict__ logit_scale, float teacher_temp,
                                    float text_temp, float* __restrict__ scal) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const float L2E = 1.4426950408889634f;
  const float s = *logit_scale;
  float mult = (s > 10.f) ? s : expf(s);
  mult = fminf(mult, 100.f);
  float tau_s = 1.f / mult;
  tau_s = fminf(fmaxf(tau_s, 0.008f), 0.02f);
  scal[SC_SCALE] = s;
  scal[SC_SCALE_L2] = s * L2E;
  scal[SC_ITS] = 1.f / tau_s;
  scal[SC_ITS_L2] = L2E / tau_s;
  scal[SC_ITT] = teacher_temp > 0.f ? 1.f / teacher_temp : 0.f;
  scal[SC_ITT_L2] = teacher_temp > 0.f ? L2E / teacher_temp : 0.f;
  scal[SC_ITX] = text_temp > 0.f ? 1.f / text_temp : 0.f;
  scal[SC_ITX_L2] = text_temp > 0.f ? L2E / text_temp : 0.f;
  scal[SC_RMIN_T] = scal[SC_RMIN_Z] = scal[SC_RMIN_D] = __int_as_float(0x7f800000);  // +inf
  scal[SC_TICKET_F] = scal[SC_TICKET_B] = 0.f;  // all-zero bits == integer 0
}

__device__ void block_reduce_rows(const float* __restrict__ in, int b, int nk, double* sums);
__device__ bool last_block_done(int* ticket);

struct FinFwdArgs {
  int b, np_c, np_s, have_soft, have_text;
  const float* pc_it;  // [2][np_c][b]
  const float* pc_ti;
  const float* ps;     // [7][np_s][b]
  const float* colsum; // symmetric forward: [6][Bcol] column-side sums (Zt, Aq, Ap, Ar, Zs, Ztt) by row, or null
  const float* lse_ti; // one-pass CLIP forward: text -> image log-sum-exp by row (= column of I . T^T), or null
  int Bcol;
  const float* diag;
  const float* scal;
  float* lse;      // [5][b]
  float* rowloss;  // [3][gridDim.x] per-block sums of the row losses
  int* ticket;     // zeroed by prep_scalars_kernel
  float lam_orig, lam_soft, text_lambda;
  float* losses;   // [5]: classic, soft_imgimg, soft_texttext, soft (= img + text_lambda * text), total
};

__device__ __forceinline__ float combine_lse2(const float* part, int np, int b, int i) {
  float m = M_FLOOR;
  for (int k = 0; k < np; ++k) m = fmaxf(m, part[k * b + i]);
  float s = 0.f;
  for (int k = 0; k < np; ++k) s += part[(np + k) * b + i] * exp2f(part[k * b + i] - m);
  return m + log2f(s);
}

// per-row combination of the column-split partial statistics -> LSEs (log2 domain) and row losses
__device__ __forceinline__ void finalize_fwd_rows(const FinFwdArgs& a, float (&rl)[3]) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  rl[0] = rl[1] = rl[2] = 0.f;
  if (i >= a.b) return;
  const float LN2 = 0.6931471805599453f;
  const float l_it = combine_lse2(a.pc_it, a.np_c, a.b, i);
  const float l_ti = a.lse_ti ? a.lse_ti[i] : combine_lse2(a.pc_ti, a.np_c, a.b, i);
  a.lse[0 * a.b + i] = l_it;
  a.lse[1 * a.b + i] = l_ti;
  // classic CE row term (loss.py:317-319): lse_it - L_ii + lse_ti - L_ii
  rl[0] = LN2 * (l_it + l_ti) - 2.f * a.scal[SC_SCALE] * a.diag[i];
  float l_t = 0.f, l_s = 0.f, l_x = 0.f, kl_s = 0.f, kl_x = 0.f;
  if (a.have_soft) {
    const int st = a.np_s * a.b;
    float m = M_FLOOR;
    for (int k = 0; k < a.np_s; ++k) m = fmaxf(m, a.ps[0 * st + k * a.b + i]);
    float zt = 0.f, aq = 0.f, ap = 0.f, ar = 0.f, zs = 0.f, zx = 0.f;
    for (int k = 0; k < a.np_s; ++k) {
      const int o = k * a.b + i;
      const float sc = exp2f(a.ps[0 * st + o] - m);
      zt += a.ps[1 * st + o] * sc;
      aq += a.ps[2 * st + o] * sc;
      ap += a.ps[3 * st + o] * sc;
      ar += a.ps[4 * st + o] * sc;
      zs += a.ps[5 * st + o];
      zx += a.ps[6 * st + o];
    }
    if (a.colsum) {  // every partial of the symmetric forward is relative to the same fixed maximum
      zt += a.colsum[0 * a.Bcol + i];
      aq += a.colsum[1 * a.Bcol + i];
      ap += a.colsum[2 * a.Bcol + i];
      ar += a.colsum[3 * a.Bcol + i];
      zs += a.colsum[4 * a.Bcol + i];
      zx += a.colsum[5 * a.Bcol + i];
      // the symmetric kernel accumulates sum w (q - M_t), sum w (p - M_s), sum w (r - M_x)
      aq += a.scal[SC_ITT_L2] * zt;
      ap += a.scal[SC_ITS_L2] * zt;
      ar += a.scal[SC_ITX_L2] * zt;
    }
    l_t = m + log2f(zt);
    l_s = a.scal[SC_ITS_L2] + log2f(zs);
    // KL(q || p) = E_q[q2 - p2] - lse_t + lse_s   (log2 units -> nats), loss.py:380-383
    kl_s = LN2 * ((aq - ap) / zt - l_t + l_s);
    if (a.have_text) {
      l_x = a.scal[SC_ITX_L2] + log2f(zx);
      kl_x = LN2 * ((aq - ar) / zt - l_t + l_x);
    }
  }
  a.lse[2 * a.b + i] = l_t;
  a.lse[3 * a.b + i] = l_s;
  a.lse[4 * a.b + i] = l_x;
  rl[1] = kl_s;
  rl[2] = kl_x;
}

// Symmetric forward: out[k][j] = sum over the warps w < 8 * (j / 256) of colpart[k][w][j] - the row blocks left of
// row j's own pair, four warps each - in a fixed order (deterministic).  grid (Bcol / 32, 6), block (32, 16).
// (DSOFT_SYM_W: columns from ncols_a on were only visited by the warps from w_lo on.)
__global__ void __launch_bounds__(512) soft_colreduce_kernel(const float* __restrict__ colpart, int cp_rows, int pitch,
                                                             int ncols, float* __restrict__ out, int ncols_a, int w_lo) {
  __shared__ float sh[16][33];
  const int j = blockIdx.x * 32 + threadIdx.x;
  const int k = blockIdx.y;
  const int wmax = min(cp_rows, 8 * (j >> 8));
  const int wmin = (j >= ncols_a) ? w_lo : 0;
  float acc = 0.f;
  if (j < ncols)
    for (int w = wmin + threadIdx.y; w < wmax; w += 16)
      acc += colpart[(static_cast<size_t>(k) * cp_rows + w) * pitch + j];
  sh[threadIdx.y][threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.y == 0) {
    float t = 0.f;
#pragma unroll
    for (int y = 0; y < 16; ++y) t += sh[y][threadIdx.x];
    out[static_cast<size_t>(k) * pitch + j] = t;
  }
}

// One-pass CLIP forward: out[j] = log2 sum_w colS[w][j] 2^(colM[w][j]) over all warp rows w (online maximum, fixed
// order -> deterministic).  grid (Bcol / 32), block (32, 16).
__global__ void __launch_bounds__(512) clip_colreduce_kernel(const float* __restrict__ colM,
                                                             const float* __restrict__ colS, int cp_rows, int pitch,
                                                             int ncols, float* __restrict__ out) {
  __shared__ float shm[16][33], shs[16][33];
  const int j = blockIdx.x * 32 + threadIdx.x;
  float m = M_FLOOR, s = 0.f;
  if (j < ncols) {
    for (int w = threadIdx.y; w < cp_rows; w += 16) {
      const size_t o = static_cast<size_t>(w) * pitch + j;
      const float mw = colM[o], sw = colS[o];
      const float mn = fmaxf(m, mw);
      s = s * exp2f(m - mn) + sw * exp2f(mw - mn);
      m = mn;
    }
  }
  shm[threadIdx.y][threadIdx.x] = m;
  shs[threadIdx.y][threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.y == 0) {
    float mm = M_FLOOR;
#pragma unroll
    for (int y = 0; y < 16; ++y) mm = fmaxf(mm, shm[y][threadIdx.x]);
    float t = 0.f;
#pragma unroll
    for (int y = 0; y < 16; ++y) t += shs[y][threadIdx.x] * exp2f(shm[y][threadIdx.x] - mm);
    out[j] = mm + log2f(t);
  }
}

__global__ void __launch_bounds__(128) finalize_fwd_kernel(FinFwdArgs a) {
  float rl[3];
  finalize_fwd_rows(a, rl);
  {  // this block's 128 row losses -> one partial per term (fixed order: deterministic)
    __shared__ float shp[3][4];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      float v = rl[k];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if ((threadIdx.x & 31) == 0) shp[k][threadIdx.x >> 5] = v;
    }
    __syncthreads();
    if (threadIdx.x < 3)
      a.rowloss[threadIdx.x * gridDim.x + blockIdx.x] =
          (shp[threadIdx.x][0] + shp[threadIdx.x][1]) + (shp[threadIdx.x][2] + shp[threadIdx.x][3]);
  }
  if (last_block_done(a.ticket)) {
    __shared__ double sums[3];
    block_reduce_rows(a.rowloss, gridDim.x, 3, sums);
    if (threadIdx.x == 0) {
      const double inv_b = 1.0 / a.b;
      const float classic = static_cast<float>(0.5 * inv_b * sums[0]);   // loss.py:317-319
      const float s_img = static_cast<float>(inv_b * sums[1]);           // loss.py:383 (batchmean)
      const float s_txt = static_cast<float>(inv_b * sums[2]);           // loss.py:396
      const float soft = s_img + a.text_lambda * s_txt;                  // loss.py:397
      a.losses[0] = classic;
      a.losses[1] = s_img;
      a.losses[2] = s_txt;
      a.losses[3] = soft;
      a.losses[4] = a.lam_orig * classic + a.lam_soft * soft;            // loss.py:473-477
      a.losses[5] = 0.f;                                                 // weighted CE: wce_final_kernel
    }
  }
}

// Deterministic reduction by ONE block (fixed thread -> index mapping, fp64): sums[k] = sum_i in[k][i].
// Called by the last block of a finalize kernel to finish (ticket pattern: no extra launch, no float atomics).
__device__ void block_reduce_rows(const float* __restrict__ in, int b, int nk, double* sums) {
  __shared__ double sh[32];
  for (int k = 0; k < nk; ++k) {
    double acc = 0.0;
    for (int i = threadIdx.x; i < b; i += blockDim.x) acc += static_cast<double>(in[k * b + i]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x < 32) {
      double v = (threadIdx.x < (blockDim.x >> 5)) ? sh[threadIdx.x] : 0.0;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (threadIdx.x == 0) sums[k] = v;
    }
    __syncthreads();
  }
}

// true for every thread of exactly one block: the last one to get here (after its global writes are visible)
__device__ bool last_block_done(int* ticket) {
  __shared__ int is_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const int t = atomicAdd(ticket, 1);
    is_last = (t == static_cast<int>(gridDim.x) - 1);
    if (is_last) *ticket = 0;  // ready for the next call (e.g. a second backward through the same forward)
  }
  __syncthreads();
  if (is_last) __threadfence();
  return is_last != 0;
}

// Extremes of the CLIP row log-sum-exps of all ranks (both directions), LSE_NB blocks -> partial (min, max) pairs;
// lse_relayout_kernel folds them into the reference exponent c of the factorised CLIP logit gradients
// 2^(x - c) (2^(c - lse_row) + 2^(c - lse_col)) and decides whether that form is safe (every 2^(c - lse) inside
// fp32: spread <= 200 log2 units; c >= -100 keeps 2^(0 - c) of padded entries finite).
constexpr int LSE_NB = 64;
__global__ void __launch_bounds__(256) lse_stats_kernel(const float* __restrict__ lse_all, int W, int b, int nr,
                                                        float* __restrict__ part) {
  __shared__ float smn[8], smx[8];
  float mn = __int_as_float(0x7f800000), mx = -__int_as_float(0x7f800000);
  const int n = W * 2 * b;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int r = i / (2 * b), k = i % (2 * b);
    const float v = lse_all[static_cast<size_t>(r) * nr * b + k];  // kinds 0 and 1 are contiguous
    mn = fminf(mn, v);
    mx = fmaxf(mx, v);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  if ((threadIdx.x & 31) == 0) { smn[threadIdx.x >> 5] = mn; smx[threadIdx.x >> 5] = mx; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < 8; ++w) { mn = fminf(mn, smn[w]); mx = fmaxf(mx, smx[w]); }
    part[blockIdx.x] = mn;
    part[LSE_NB + blockIdx.x] = mx;
  }
}

// [W][nr][b] (rank-major, as all-gathered; rows 0..4 used here) -> by global column, padded:
//   lsec   [5][Bcol]  the log-sum-exps themselves (zero padded; exact CLIP form and the fused backward)
//   colfac [5][Bcol]  column factors of the factorised logit gradients: 0 / 1 CLIP 2^(c - lse) for the image-rows
//                     launch (columns = text rows' lse_ti) and the text-rows launch (lse_it); 2 teacher
//                     2^(M_t - lt) (exact form: lt); 3 student 2^(M_s - ls); 4 text 2^(M_x - lx).  Zero (teacher
//                     exact form: +1e30, i.e. 2^(q - 1e30) = 0) for padded columns and wherever the column-side
//                     terms are dropped (gather_with_grad == False).
__global__ void __launch_bounds__(256) lse_relayout_kernel(const float* __restrict__ lse_all, int W, int b, int nr,
                                                           int Bcol,
                                                           float* __restrict__ scal, const float* __restrict__ part,
                                                           int fast_t, int drop_clip, int drop_soft,
                                                           float* __restrict__ out, float* __restrict__ colfac) {
  __shared__ float s_c;
  if (threadIdx.x < 32) {  // every block folds the LSE_NB partial extremes itself (64 + 64 floats)
    float mn = fminf(part[threadIdx.x], part[threadIdx.x + 32]);
    float mx = fmaxf(part[LSE_NB + threadIdx.x], part[LSE_NB + threadIdx.x + 32]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    if (threadIdx.x == 0) {
      const float c = 0.5f * (mn + mx);
      const bool ok = (mx - mn <= 200.f) && (c >= -100.f) && (c <= 1.0e30f);  // false for NaN / inf as well
      s_c = ok ? c : 0.f;
      if (blockIdx.x == 0) {
        scal[SC_C_CLIP] = ok ? c : 0.f;
        scal[SC_FAST_CLIP] = ok ? 1.f : 0.f;
      }
    }
  }
  __syncthreads();
  const float cclip = s_c;
  const int total = 5 * Bcol;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int k = i / Bcol, j = i % Bcol;
    const bool real = j < W * b;
    float v = 0.f;
    if (real) v = lse_all[(static_cast<size_t>(j / b) * nr + k) * b + (j % b)];
    out[i] = v;
    float f;
    if (k < 2) {
      // colfac[0] serves the launch whose columns are TEXT rows (their lse is kind 1), colfac[1] the other one
      const float lo = real ? lse_all[(static_cast<size_t>(j / b) * nr + (1 - k)) * b + (j % b)] : 0.f;
      f = (real && !drop_clip) ? exp2f(cclip - lo) : 0.f;
    } else if (k == 2) {
      if (fast_t) f = (real && !drop_soft) ? exp2f(scal[SC_ITT_L2] - v) : 0.f;
      else f = (real && !drop_soft) ? v : 1.0e30f;
    } else {
      f = (real && !drop_soft) ? exp2f(scal[k == 3 ? SC_ITS_L2 : SC_ITX_L2] - v) : 0.f;
    }
    colfac[i] = f;
  }
}

// fp16 copies of the gradient-GEMM operands, one warp per global row:
//   text | image (as used in the CLIP logits) | student_j * sigma_j | text_j * sigma_j
// sigma_j = 2^floor(log2(1/||row_j||)), PER ROW: a power-of-two scaling is exact, the scaled row has a norm in
// (1/2, 1] whatever the norm spread of the batch (an outlier row cannot push the others into fp16 subnormals),
// and bf16 -> fp16 is exact for |x| in [2^-14, 65504), so the operands reach the tensor core unrounded; the
// remaining factor mant(1/||row_j||) in [1, 2) is folded into the fp16 G tile instead.
__global__ void make_v16_kernel(const __nv_bfloat16* __restrict__ gathered, int row_elems, int B, int D,
                                int Dz, int offI, int offT, int offZ, int have_soft, int have_text,
                                const float* __restrict__ rinv_z, const float* __restrict__ rinv_t,
                                __half* __restrict__ v16, int v_row,
                                int v_offT, int v_offI, int v_offZn, int v_offTn) {
  const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (r >= B) return;
  const __nv_bfloat16* src = gathered + static_cast<size_t>(r) * row_elems;
  __half* dst = v16 + static_cast<size_t>(r) * v_row;
  const float st = have_text ? pow2_of(rinv_t[r]) : 0.f;
  const float sz = have_soft ? pow2_of(rinv_z[r]) : 0.f;
  for (int c = lane * 2; c < D; c += 64) {
    const float2 t = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(src + offT + c));
    const float2 im = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(src + offI + c));
    *reinterpret_cast<__half2*>(dst + v_offT + c) = __floats2half2_rn(t.x, t.y);
    *reinterpret_cast<__half2*>(dst + v_offI + c) = __floats2half2_rn(im.x, im.y);
    if (have_text) *reinterpret_cast<__half2*>(dst + v_offTn + c) = __floats2half2_rn(t.x * st, t.y * st);
  }
  if (have_soft) {
    for (int c = lane * 2; c < Dz; c += 64) {
      const float2 z = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(src + offZ + c));
      *reinterpret_cast<__half2*>(dst + v_offZn + c) = __floats2half2_rn(z.x * sz, z.y * sz);
    }
  }
}

struct FinBwdArgs {
  int b, D, Dz, row0, row_elems, offI, offT, offZ;
  int have_soft, have_text, have_proj, row_only;
  int sym_scaled;  // two-phase backward, world == 1: the soft G matrices carry mant(1/||y_i||) of their ROW as well
  // weighted CE: the CLIP logit-gradient matrices already carry g_c and g_w; the diagonal entry of both directions
  // is applied here in fp32
  int weighted, wsym;
  const float* wstat;  // [2 directions][4][Bcol] by global row: c, lse~, A, (std)
  int Bcol;
  float lam_w;
  int ns_c, ns_c2, ns_s, ns_x;  // split counts of acc1, acc2, acc3, acc4
  int nds;  // d(logit_scale) partials per row: nsplit x cluster size x 2 halves
  const __nv_bfloat16* gathered;
  const float* acc1;  // [ns_c][b][D]   sum_j G_clip . T_j   (image rows)
  const float* acc2;  // [ns_c2][b][D]  sum_j G_clip' . I_j  (text rows)
  const float* acc3;  // [ns_s][b][Dz]  sum_j G_stu . Z_j / ||Z_j||
  const float* acc4;  // [ns_x][b][D]   sum_j G_txt . T_j / ||T_j||
  const float* ds1;   // [2 ns_c][b]
  const float* ds2;
  const float* diag;
  const float* scal;
  const float* rinv_z;
  const float* rinv_t;
  const float* gout;  // [5] upstream grads of {classic, soft_img, soft_txt, soft, total}
  float lam_orig, lam_soft, text_lambda;
  int* ticket;
  float* d_scale;
  const float* lse_loc;  // [5][b] this rank's row LSEs (log2)
  float* d_image;
  float* d_text;
  float* d_student;
  float* dsrow;  // [gridDim.x] per-block sums of the d(logit_scale) row terms
};

__device__ __forceinline__ float block_sum_128(float v, float* sh) {  // finalize_bwd_kernel: 4 warps
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  return sh[0] + sh[1] + sh[2] + sh[3];
}

// One 128-thread block per local row: sum the column-split partial gradients, apply the fp32 one-hot
// part of the CE gradient, the temperature / batch factors and the chain rule through F.normalize.
// Every thread owns 4 consecutive features per pass (float4 traffic, sums stay in registers between the
// dot-product pass and the output pass); FB_MAXIT passes cover feature widths up to 512 * FB_MAXIT (template
// parameter: the per-thread arrays cost registers, and this kernel lives on occupancy).

__device__ __forceinline__ float4 sum_splits4(const float* __restrict__ part, int nsplit, int b, int width, int i,
                                               int f) {
  float4 u = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int s = 0; s < nsplit; ++s) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(part + (static_cast<size_t>(s) * b + i) * width + f));
    u.x += v.x; u.y += v.y; u.z += v.z; u.w += v.w;
  }
  return u;
}
__device__ __forceinline__ float4 load_bf16x4(const __nv_bfloat16* p) {
  const uint2 raw = *reinterpret_cast<const uint2*>(p);
  const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&raw.x));
  const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&raw.y));
  return make_float4(a.x, a.y, b.x, b.y);
}

// Diagonal entry of the CLIP logit-gradient matrix (applied in fp32: near convergence p_aa -> 1 and the entry is a
// small residual), the coefficient of the CLIP part and the diagonal's share of d(logit_scale).
//   classic:  dg = (p_it_aa - 1) + (p_ti_aa - 1); the matrix is unscaled, g_c s / (2b) is applied here; the row
//             partials of d(logit_scale) include the diagonal's probabilities, hence the - 2 dot_aa
//   weighted: the matrix already carries g_c gk and g_w gk and has no diagonal;
//             dg = g_c [(p_it_aa - 1) + (p_ti_aa - 1)] + g_w [(p~_it_aa - 1 + beta A_a p_it_aa c_a) + text direction]
//             (d CE~_a / d x_aa = p~_aa - 1 - beta A_a p_aa (r_aa - c_a) with r_aa = 0, loss.py:416-471), taken
//             times gk like the GEMM partials and the d(logit_scale) row partials; s / (2b gk) divides gk out
struct ClipDiag { float dg_img, dg_txt, coefc, ds_diag; };
__device__ __forceinline__ ClipDiag clip_diag(const FinBwdArgs& a, int i, float gc, float inv_b) {
  const float LN2 = 0.6931471805599453f;
  const float xd = a.scal[SC_SCALE_L2] * a.diag[i];
  const float dm_it = expm1f(LN2 * (xd - a.lse_loc[0 * a.b + i]));
  const float dm_ti = expm1f(LN2 * (xd - a.lse_loc[1 * a.b + i]));
  ClipDiag r;
  if (!a.weighted) {
    r.dg_img = a.row_only ? dm_it : dm_it + dm_ti;
    r.dg_txt = a.row_only ? dm_ti : dm_it + dm_ti;
    r.coefc = gc * a.scal[SC_SCALE] * 0.5f * inv_b;
    r.ds_diag = -2.f * a.diag[i];
  } else {
    const float gw = a.gout[5] + a.lam_w * a.gout[4];
    const float* wi = a.wstat;
    const float* wt = a.wstat + static_cast<size_t>(4) * a.Bcol;
    const int j = a.row0 + i;  // the statistics rows are indexed by global row
    const float g_img = expm1f(LN2 * (xd - wi[1 * a.Bcol + j])) +
                        a.scal[SC_WBETA + 0] * wi[2 * a.Bcol + j] * (dm_it + 1.f) * wi[0 * a.Bcol + j];
    const float g_txt = a.wsym ? expm1f(LN2 * (xd - wt[1 * a.Bcol + j])) +
                                     a.scal[SC_WBETA + 1] * wt[2 * a.Bcol + j] * (dm_ti + 1.f) * wt[0 * a.Bcol + j]
                               : dm_ti;
    const float gk = a.scal[SC_WCE_GK];
    const float dg = (gc * (dm_it + dm_ti) + gw * (g_img + g_txt)) * gk;
    r.dg_img = r.dg_txt = dg;
    if (a.row_only) {  // world > 1, gathered columns detached: each direction's own row term only
      r.dg_img = (gc * dm_it + gw * g_img) * gk;
      r.dg_txt = (gc * dm_ti + gw * g_txt) * gk;
    }
    r.coefc = a.scal[SC_SCALE] * 0.5f * inv_b * a.scal[SC_WCE_IGK];
    r.ds_diag = dg * a.diag[i];
  }
  return r;
}

template <int FB_MAXIT>
__global__ void __launch_bounds__(128) finalize_bwd_kernel(FinBwdArgs a) {
  __shared__ float sh[4];
  const int tid = threadIdx.x;
  float ds_block = 0.f;  // thread 0: this block's share of sum_i dsrow[i]
  // a few thousand blocks stride over the rows: one ticket atomic per BLOCK (per row they serialise on one
  // address and cost more than the gradient traffic)
  for (int i = blockIdx.x; i < a.b; i += gridDim.x) {
  const size_t gi = static_cast<size_t>(a.row0) + i;
  const __nv_bfloat16* rowp = a.gathered + gi * a.row_elems;
  const float inv_b = 1.f / static_cast<float>(a.b);
  // chain rule through soft = img + tl * txt and total = lam_orig * classic + lam_soft * soft
  const float g_soft = a.gout[3] + a.lam_soft * a.gout[4];
  const float gc = a.gout[0] + a.lam_orig * a.gout[4];
  const float gs = a.gout[1] + g_soft;
  const float gx = a.gout[2] + a.text_lambda * g_soft;
  const ClipDiag cd = clip_diag(a, i, gc, inv_b);
  const float coefc = cd.coefc, dg_img = cd.dg_img, dg_txt = cd.dg_txt;

  float4 di[FB_MAXIT], dt[FB_MAXIT];  // d_image / d_text of this thread's features (D <= 2048)
  float4 tfeat[FB_MAXIT];             // text features (reused by the text-text term)

  // ---- CLIP part (loss.py:317-319 backward)
#pragma unroll
  for (int it = 0; it < FB_MAXIT; ++it) {
    const int f = (it * 128 + tid) * 4;
    if (f < a.D) {
      const float4 u1 = sum_splits4(a.acc1, a.ns_c, a.b, a.D, i, f);
      const float4 u2 = sum_splits4(a.acc2, a.ns_c2, a.b, a.D, i, f);
      const float4 tf = load_bf16x4(rowp + a.offT + f);
      const float4 im = load_bf16x4(rowp + a.offI + f);
      tfeat[it] = tf;
      di[it] = make_float4(coefc * fmaf(dg_img, tf.x, u1.x), coefc * fmaf(dg_img, tf.y, u1.y),
                           coefc * fmaf(dg_img, tf.z, u1.z), coefc * fmaf(dg_img, tf.w, u1.w));
      dt[it] = make_float4(coefc * fmaf(dg_txt, im.x, u2.x), coefc * fmaf(dg_txt, im.y, u2.y),
                           coefc * fmaf(dg_txt, im.z, u2.z), coefc * fmaf(dg_txt, im.w, u2.w));
    }
  }
  if (tid == 0) {
    float d = 0.f;
    for (int s = 0; s < a.nds; ++s) d += a.ds1[s * a.b + i] + a.ds2[s * a.b + i];
    ds_block += d + cd.ds_diag;
  }

  // ---- student KL (loss.py:358-383 backward): d z~ = (g / (b tau_s)) * acc3 ; chain through normalize
  if (a.have_soft) {
    const float rz = a.rinv_z[gi];
    const float coefs = gs * a.scal[SC_ITS] * inv_b / (a.sym_scaled ? mant12(rz) : 1.f);
    float4 dz[FB_MAXIT], zt[FB_MAXIT];
    float dot = 0.f;
#pragma unroll
    for (int it = 0; it < FB_MAXIT; ++it) {
      const int f = (it * 128 + tid) * 4;
      if (f < a.Dz) {
        float4 u = sum_splits4(a.acc3, a.ns_s, a.b, a.Dz, i, f);
        float4 z = load_bf16x4(rowp + a.offZ + f);
        z.x *= rz; z.y *= rz; z.z *= rz; z.w *= rz;
        u.x *= coefs; u.y *= coefs; u.z *= coefs; u.w *= coefs;
        dot += z.x * u.x + z.y * u.y + z.z * u.z + z.w * u.w;
        dz[it] = u;
        zt[it] = z;
      }
    }
    dot = block_sum_128(dot, sh);
#pragma unroll
    for (int it = 0; it < FB_MAXIT; ++it) {
      const int f = (it * 128 + tid) * 4;
      if (f < a.Dz) {
        const float4 g4 = make_float4(rz * (dz[it].x - zt[it].x * dot), rz * (dz[it].y - zt[it].y * dot),
                                      rz * (dz[it].z - zt[it].z * dot), rz * (dz[it].w - zt[it].w * dot));
        if (a.have_proj) {
          *reinterpret_cast<float4*>(a.d_student + static_cast<size_t>(i) * a.Dz + f) = g4;
        } else {  // student == image features: same thread owns the same features (Dz == D)
          di[it].x += g4.x; di[it].y += g4.y; di[it].z += g4.z; di[it].w += g4.w;
        }
      }
    }
  }
  // ---- text-text KL (loss.py:387-397 backward)
  if (a.have_text) {
    const float rt = a.rinv_t[gi];
    const float coefx = gx * a.scal[SC_ITX] * inv_b / (a.sym_scaled ? mant12(rt) : 1.f);
    float4 dx[FB_MAXIT];
    float dot = 0.f;
#pragma unroll
    for (int it = 0; it < FB_MAXIT; ++it) {
      const int f = (it * 128 + tid) * 4;
      if (f < a.D) {
        float4 u = sum_splits4(a.acc4, a.ns_x, a.b, a.D, i, f);
        u.x *= coefx; u.y *= coefx; u.z *= coefx; u.w *= coefx;
        const float4 t = tfeat[it];
        dot += rt * (t.x * u.x + t.y * u.y + t.z * u.z + t.w * u.w);
        dx[it] = u;
      }
    }
    dot = block_sum_128(dot, sh);
#pragma unroll
    for (int it = 0; it < FB_MAXIT; ++it) {
      const int f = (it * 128 + tid) * 4;
      if (f < a.D) {
        const float4 t = tfeat[it];
        dt[it].x += rt * (dx[it].x - rt * t.x * dot);
        dt[it].y += rt * (dx[it].y - rt * t.y * dot);
        dt[it].z += rt * (dx[it].z - rt * t.z * dot);
        dt[it].w += rt * (dx[it].w - rt * t.w * dot);
      }
    }
  }
#pragma unroll
  for (int it = 0; it < FB_MAXIT; ++it) {
    const int f = (it * 128 + tid) * 4;
    if (f < a.D) {
      *reinterpret_cast<float4*>(a.d_image + static_cast<size_t>(i) * a.D + f) = di[it];
      *reinterpret_cast<float4*>(a.d_text + static_cast<size_t>(i) * a.D + f) = dt[it];
    }
  }
  __syncthreads();  // sh is reused by the next row
  }
  // ---- d logit_scale = g_classic / (2b) * sum_i dsrow[i], finished by the last block
  if (tid == 0) a.dsrow[blockIdx.x] = ds_block;
  if (last_block_done(a.ticket)) {
    __shared__ double sum1[1];
    block_reduce_rows(a.dsrow, gridDim.x, 1, sum1);
    // weighted: the row terms carry g_c, g_w and gk already
    const float gc = a.weighted ? a.scal[SC_WCE_IGK] : a.gout[0] + a.lam_orig * a.gout[4];
    if (threadIdx.x == 0) a.d_scale[0] = static_cast<float>(sum1[0] * static_cast<double>(gc) * 0.5 / a.b);
  }
}

// Same computation, ONE WARP PER ROW (feature widths up to 128 * NV): lane l owns the float4 groups l, l + 32, ...
// of every vector of its row, the two dot products of the normalise backward are warp shuffles, and nothing waits
// on a block barrier.  The block-per-row kernel above was latency bound (0.33 ms for ~0.6 GB at B = 32768: two
// __syncthreads-based reductions per row with 4 warps per row); it remains the path for wider features.
// NVD / NVZ: float4 groups per lane for the CLIP width D / the student width Dz; PROJ: the student gradient leaves
// through d_student (its registers die before the text part) instead of being added to d_image.
template <int NVD, int NVZ, bool PROJ>
__global__ void __launch_bounds__(256, 2) finalize_bwd_warp_kernel(FinBwdArgs a) {
  __shared__ float ds_sh[8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const float LN2 = 0.6931471805599453f;
  const float inv_b = 1.f / static_cast<float>(a.b);
  const float g_soft = a.gout[3] + a.lam_soft * a.gout[4];
  const float gc = a.gout[0] + a.lam_orig * a.gout[4];
  const float gs = a.gout[1] + g_soft;
  const float gx = a.gout[2] + a.text_lambda * g_soft;
  float ds_warp = 0.f;
  auto warp_sum = [](float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
  };
  for (int i = blockIdx.x * 8 + warp; i < a.b; i += gridDim.x * 8) {
    const size_t gi = static_cast<size_t>(a.row0) + i;
    const __nv_bfloat16* rowp = a.gathered + gi * a.row_elems;
    const ClipDiag cd = clip_diag(a, i, gc, inv_b);
    const float coefc = cd.coefc, dg_img = cd.dg_img, dg_txt = cd.dg_txt;
    float4 xs[NVZ];  // student term: d_student, or the share of d_image when the student IS the image feature
    float4 tf[NVD];  // text features
    float4 xt[NVD];  // text-text term's share of d_text
    // ---- student KL (loss.py:358-383 backward): (g / (b tau_s)) * acc3, chained through normalize
    if (a.have_soft) {
      const float rz = a.rinv_z[gi];
      const float coefs = gs * a.scal[SC_ITS] * inv_b / (a.sym_scaled ? mant12(rz) : 1.f);
      float4 zn[NVZ];
      float dot = 0.f;
#pragma unroll
      for (int it = 0; it < NVZ; ++it) {
        const int f = (it * 32 + lane) * 4;
        if (f < a.Dz) {
          float4 u = sum_splits4(a.acc3, a.ns_s, a.b, a.Dz, i, f);
          float4 z = load_bf16x4(rowp + a.offZ + f);
          z.x *= rz; z.y *= rz; z.z *= rz; z.w *= rz;
          u.x *= coefs; u.y *= coefs; u.z *= coefs; u.w *= coefs;
          dot += z.x * u.x + z.y * u.y + z.z * u.z + z.w * u.w;
          xs[it] = u;
          zn[it] = z;
        }
      }
      dot = warp_sum(dot);
#pragma unroll
      for (int it = 0; it < NVZ; ++it) {
        const int f = (it * 32 + lane) * 4;
        if (f < a.Dz) {
          const float4 g4 = make_float4(rz * (xs[it].x - zn[it].x * dot), rz * (xs[it].y - zn[it].y * dot),
                                        rz * (xs[it].z - zn[it].z * dot), rz * (xs[it].w - zn[it].w * dot));
          if constexpr (PROJ) *reinterpret_cast<float4*>(a.d_student + static_cast<size_t>(i) * a.Dz + f) = g4;
          else xs[it] = g4;
        }
      }
    }
#pragma unroll
    for (int it = 0; it < NVD; ++it) {
      const int f = (it * 32 + lane) * 4;
      if (f < a.D) tf[it] = load_bf16x4(rowp + a.offT + f);
    }
    // ---- text-text KL (loss.py:387-397 backward)
    if (a.have_text) {
      const float rt = a.rinv_t[gi];
      const float coefx = gx * a.scal[SC_ITX] * inv_b / (a.sym_scaled ? mant12(rt) : 1.f);
      float dot = 0.f;
#pragma unroll
      for (int it = 0; it < NVD; ++it) {
        const int f = (it * 32 + lane) * 4;
        if (f < a.D) {
          float4 u = sum_splits4(a.acc4, a.ns_x, a.b, a.D, i, f);
          u.x *= coefx; u.y *= coefx; u.z *= coefx; u.w *= coefx;
          const float4 t = tf[it];
          dot += rt * (t.x * u.x + t.y * u.y + t.z * u.z + t.w * u.w);
          xt[it] = u;
        }
      }
      dot = warp_sum(dot);
#pragma unroll
      for (int it = 0; it < NVD; ++it) {
        const int f = (it * 32 + lane) * 4;
        if (f < a.D) {
          const float4 t = tf[it];
          xt[it] = make_float4(rt * (xt[it].x - rt * t.x * dot), rt * (xt[it].y - rt * t.y * dot),
                               rt * (xt[it].z - rt * t.z * dot), rt * (xt[it].w - rt * t.w * dot));
        }
      }
    }
    // ---- CLIP part (loss.py:317-319 backward) + outputs
    const bool add_s = a.have_soft && !PROJ;  // student == image features: same lane owns the same features
#pragma unroll
    for (int it = 0; it < NVD; ++it) {
      const int f = (it * 32 + lane) * 4;
      if (f < a.D) {
        const float4 u1 = sum_splits4(a.acc1, a.ns_c, a.b, a.D, i, f);
        const float4 u2 = sum_splits4(a.acc2, a.ns_c2, a.b, a.D, i, f);
        const float4 t = tf[it];
        const float4 im = load_bf16x4(rowp + a.offI + f);
        float4 di = make_float4(coefc * fmaf(dg_img, t.x, u1.x), coefc * fmaf(dg_img, t.y, u1.y),
                                coefc * fmaf(dg_img, t.z, u1.z), coefc * fmaf(dg_img, t.w, u1.w));
        float4 dt = make_float4(coefc * fmaf(dg_txt, im.x, u2.x), coefc * fmaf(dg_txt, im.y, u2.y),
                                coefc * fmaf(dg_txt, im.z, u2.z), coefc * fmaf(dg_txt, im.w, u2.w));
        if constexpr (!PROJ) {
          if (add_s) { di.x += xs[it].x; di.y += xs[it].y; di.z += xs[it].z; di.w += xs[it].w; }
        }
        if (a.have_text) { dt.x += xt[it].x; dt.y += xt[it].y; dt.z += xt[it].z; dt.w += xt[it].w; }
        *reinterpret_cast<float4*>(a.d_image + static_cast<size_t>(i) * a.D + f) = di;
        *reinterpret_cast<float4*>(a.d_text + static_cast<size_t>(i) * a.D + f) = dt;
      }
    }
    float d = 0.f;
    for (int s = lane; s < a.nds; s += 32) d += a.ds1[s * a.b + i] + a.ds2[s * a.b + i];
    d = warp_sum(d);
    ds_warp += d + cd.ds_diag;
  }
  // ---- d logit_scale = g_classic / (2b) * sum_i dsrow[i], finished by the last block (fixed order: deterministic)
  if (lane == 0) ds_sh[warp] = ds_warp;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < 8; ++w) t += ds_sh[w];
    a.dsrow[blockIdx.x] = t;
  }
  if (last_block_done(a.ticket)) {
    __shared__ double sum1[1];
    block_reduce_rows(a.dsrow, gridDim.x, 1, sum1);
    if (threadIdx.x == 0)  // weighted: the row terms carry g_c, g_w and gk already
      a.d_scale[0] = static_cast<float>(sum1[0] * static_cast<double>(a.weighted ? a.scal[SC_WCE_IGK] : gc) * 0.5 / a.b);
  }
}

// ------------------------------------------------------------------------------------------------
// optional per-kernel timing (bench.py's roofline): CUDA events around each tile-kernel launch
// ------------------------------------------------------------------------------------------------
// PK_BWD_CLIP_I / _T: the fused backward's CLIP launches (of a weighted plan dsoft_bwd_kernel<MODE_WCE_X>, CLIP and
// DINO products), or with DSOFT_F_GMAT the CLIP gradient GEMMs
enum { PK_FWD_CLIP_IT = 0, PK_FWD_CLIP_TI, PK_FWD_SOFT, PK_BWD_CLIP_I, PK_BWD_CLIP_T, PK_BWD_STU, PK_BWD_TXT,
       PK_BWD_GCLIP, PK_BWD_GSOFT, PK_COUNT };
static const int PROF_MAX = 4096;
static struct {
  int on = 0;
  int n = 0;
  cudaEvent_t ev0[PROF_MAX], ev1[PROF_MAX];
  int kind[PROF_MAX];
  int created = 0;
} g_prof;

struct ProfScope {
  int idx = -1;
  cudaStream_t st;
  ProfScope(int kind, cudaStream_t s) : st(s) {
    if (!g_prof.on || g_prof.n >= PROF_MAX) return;
    if (g_prof.created <= g_prof.n) {
      cudaEventCreate(&g_prof.ev0[g_prof.n]);
      cudaEventCreate(&g_prof.ev1[g_prof.n]);
      g_prof.created = g_prof.n + 1;
    }
    idx = g_prof.n++;
    g_prof.kind[idx] = kind;
    cudaEventRecord(g_prof.ev0[idx], st);
  }
  ~ProfScope() {
    if (idx >= 0) cudaEventRecord(g_prof.ev1[idx], st);
  }
};

extern "C" int dsoft_profile_enable(int on) {
  g_prof.on = on;
  g_prof.n = 0;
  return 0;
}

// Synchronises the device, sums the recorded durations per kernel kind and resets the recorder.
extern "C" int dsoft_profile_read(double* ms_sum, int* counts, int n) {
  if (!ms_sum || !counts || n < PK_COUNT) return fail(DSOFT_EINVAL, "need %d slots", PK_COUNT);
  CUDA_TRY(cudaDeviceSynchronize());
  for (int k = 0; k < n; ++k) { ms_sum[k] = 0.0; counts[k] = 0; }
  for (int i = 0; i < g_prof.n; ++i) {
    float ms = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&ms, g_prof.ev0[i], g_prof.ev1[i]));
    ms_sum[g_prof.kind[i]] += ms;
    counts[g_prof.kind[i]] += 1;
  }
  g_prof.n = 0;
  return 0;
}

// ------------------------------------------------------------------------------------------------
// fork/join of independent tile kernels
//
// The tile kernels of one pass are mutually independent (they read the gathered table / statistics and write
// disjoint partial buffers), and every launch ends in a partially filled last wave. Launching them on forked
// side streams lets the next kernel's CTAs fill that tail; one CTA per SM (smem + 512 TMEM columns) means
// kernels never co-reside on an SM, so this is back-to-back execution without the idle tails. The side
// streams are joined back into the caller's stream before the entry point returns, so the caller sees plain
// stream-ordered semantics (and stream capture records a fork/join graph). Per-kernel timing
// (dsoft_profile_enable) forces serial launches so that each duration is an isolated measurement.
// ------------------------------------------------------------------------------------------------
static const int NSIDE = 3;
static int g_concurrency = -2;  // -2: read DSOFT_CONCURRENCY on first use; -1 auto, 0 off, 1 on

extern "C" int dsoft_set_concurrency(int on) {
  g_concurrency = on < 0 ? -1 : (on ? 1 : 0);
  return 0;
}

// auto: fork only when this rank's block of the similarity matrices is small (<= 2^28 elements).  Measured on
// B200: +7 % at B = 8192 and +3.7 % at b x B = 8192 x 32768 (tails of 1-3 wave kernels filled), but nothing
// at b x B >= 16384 x 32768, where the step is power capped and the extra activity only lowers the SM clock.
static bool concurrency_on(const dsoft_plan* p) {
  if (g_concurrency == -2) {
    const char* e = getenv("DSOFT_CONCURRENCY");
    g_concurrency = !e ? -1 : (e[0] == '0' ? 0 : (e[0] == '1' ? 1 : -1));
  }
  if (g_prof.on || g_concurrency == 0) return false;
  if (g_concurrency == 1) return true;
  return static_cast<double>(p->sh.b) * p->B <= 268435456.0;
}

extern "C" int dsoft_plan_concurrency(const dsoft_plan_t* p) {
  if (!p) return 0;
  if (g_prof.on) return 2;
  return concurrency_on(p) ? 1 : 0;
}

struct SideStreams {
  bool ready = false;
  cudaStream_t s[NSIDE];
  cudaEvent_t fork, join[NSIDE];
};

// one set per (host thread, device): events are re-recorded on every call
static int side_streams(SideStreams** out) {
  static thread_local SideStreams table[64];
  int dev = 0;
  CUDA_TRY(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64) return fail(DSOFT_EINVAL, "device ordinal %d out of range", dev);
  SideStreams& ss = table[dev];
  if (!ss.ready) {
    for (int i = 0; i < NSIDE; ++i) {
      CUDA_TRY(cudaStreamCreateWithFlags(&ss.s[i], cudaStreamNonBlocking));
      CUDA_TRY(cudaEventCreateWithFlags(&ss.join[i], cudaEventDisableTiming));
    }
    CUDA_TRY(cudaEventCreateWithFlags(&ss.fork, cudaEventDisableTiming));
    ss.ready = true;
  }
  *out = &ss;
  return 0;
}

struct Fork {
  cudaStream_t main_st = nullptr;
  SideStreams* ss = nullptr;
  bool forked[NSIDE] = {false, false, false};
  int begin(const dsoft_plan* p, cudaStream_t st) {
    main_st = st;
    if (!concurrency_on(p)) return 0;
    int rc = side_streams(&ss);
    if (rc) return rc;
    CUDA_TRY(cudaEventRecord(ss->fork, main_st));
    return 0;
  }
  // lane 0 is the caller's stream; lanes 1..NSIDE are side streams ordered after the fork point
  int lane(int i, cudaStream_t* out) {
    if (!ss || i <= 0) { *out = main_st; return 0; }
    const int k = (i - 1) % NSIDE;
    if (!forked[k]) {
      CUDA_TRY(cudaStreamWaitEvent(ss->s[k], ss->fork, 0));
      forked[k] = true;
    }
    *out = ss->s[k];
    return 0;
  }
  int join() {
    if (!ss) return 0;
    for (int k = 0; k < NSIDE; ++k) {
      if (!forked[k]) continue;
      CUDA_TRY(cudaEventRecord(ss->join[k], ss->s[k]));
      CUDA_TRY(cudaStreamWaitEvent(main_st, ss->join[k], 0));
      forked[k] = false;
    }
    return 0;
  }
};

// ------------------------------------------------------------------------------------------------
// launch helpers
// ------------------------------------------------------------------------------------------------
// Forward tile kernels run as CTA pairs (cluster of 2 consecutive row blocks, cta_group::2 MMAs).
template <typename K>
static int launch_fwd_pair(K kernel, int rbs, int nsplit, cudaStream_t st, const TileMaps& tm, const FwdParams& P,
                           int threads = NUM_THREADS) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((rbs + 1) / 2 * 2, nsplit, 1);
  cfg.blockDim = dim3(threads);
  cfg.dynamicSmemBytes = FWD_SMEM_BYTES;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  CUDA_TRY(cudaLaunchKernelEx(&cfg, kernel, tm, P));
  return 0;
}

// Backward tile kernel: the feature chunks of one (row block, column split) form a cluster along grid.x.
// More than X_MAXC chunks are split into several launches (each recomputes the S tiles once).
template <typename K>
static int launch_bwd(K kernel, int nch, int rbs, int nsplit, cudaStream_t st, const TileMaps& tm,
                      const CUtensorMap& vmap, BwdParams P) {
  const int csz = chunk_cluster(nch);
  for (int c0 = 0; c0 < nch; c0 += csz) {
    const int cg = std::min(csz, nch - c0);
    P.chunk0 = c0;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(cg, rbs, nsplit);
    cfg.blockDim = dim3(NUM_THREADS);
    cfg.dynamicSmemBytes = BWD_SMEM_BYTES;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = cg;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    CUDA_TRY(cudaLaunchKernelEx(&cfg, kernel, tm, vmap, P));
  }
  return 0;
}

// cudaFuncSetAttribute once per (kernel, device): K is only the function-pointer TYPE, so remember the
// pointer values that were configured
template <typename K>
static int set_smem(K kernel, int bytes) {
  static thread_local const void* done[16][2];
  static thread_local int ndone = 0;
  int dev = 0;
  CUDA_TRY(cudaGetDevice(&dev));
  const void* key = reinterpret_cast<const void*>(kernel);
  const void* devkey = reinterpret_cast<const void*>(static_cast<uintptr_t>(dev) + 1);
  for (int i = 0; i < ndone; ++i)
    if (done[i][0] == key && done[i][1] == devkey) return 0;
  CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  if (ndone < 16) {
    done[ndone][0] = key;
    done[ndone][1] = devkey;
    ++ndone;
  }
  return 0;
}

extern "C" int dsoft_pack(const dsoft_plan_t* p, const void* image, int image_dt, int64_t ld_image,
                          const void* text, int text_dt, int64_t ld_text, const void* student,
                          int student_dt, int64_t ld_student, const void* dino, int dino_dt,
                          int64_t ld_dino, void* gathered, void* stream) {
  if (!p || !image || !text || !gathered) return fail(DSOFT_EINVAL, "null argument");
  // student == NULL with Dp > 0: the caller fills the student columns itself (dsoft_head_forward);
  // dino == NULL with a soft term: the caller fills the DINO columns itself (dsoft_gather_rows)
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  __nv_bfloat16* base =
      static_cast<__nv_bfloat16*>(gathered) + static_cast<size_t>(p->sh.rank) * p->sh.b * p->row_elems;
  PackArgs a;
  memset(&a, 0, sizeof(a));
  a.rows = p->sh.b;
  a.dst_ld = p->row_elems;
  auto add = [&](const void* src, int dt, int64_t ld, int cols, int off) -> int {
    if (dt < DSOFT_DT_F32 || dt > DSOFT_DT_F16) return fail(DSOFT_EINVAL, "unknown dtype %d", dt);
    if (ld % 2 || reinterpret_cast<uintptr_t>(src) % 8)
      return fail(DSOFT_EINVAL, "pack sources need even row strides and 8-byte aligned base pointers");
    PackSrc& m = a.m[a.nmat];
    m.src = src; m.dtype = dt; m.ld = ld; m.cols = cols; m.dst_off = off;
    a.pairs_end[a.nmat] = (a.nmat ? a.pairs_end[a.nmat - 1] : 0) + static_cast<int64_t>(a.rows) * (cols / 2);
    ++a.nmat;
    return 0;
  };
  int rc;
  if ((rc = add(image, image_dt, ld_image, p->sh.D, p->offI))) return rc;
  if ((rc = add(text, text_dt, ld_text, p->sh.D, p->offT))) return rc;
  if ((p->have_proj || p->distill) && student && (rc = add(student, student_dt, ld_student, p->sh.Dp, p->offZ)))
    return rc;
  if ((p->have_soft || p->weighted || p->distill) && dino && (rc = add(dino, dino_dt, ld_dino, p->sh.Dd, p->offD))) return rc;
  bool vec8 = reinterpret_cast<uintptr_t>(base) % 16 == 0 && a.dst_ld % 8 == 0;
  for (int k = 0; k < a.nmat; ++k) {
    const PackSrc& m = a.m[k];
    const int64_t per16 = m.dtype == DSOFT_DT_F32 ? 4 : 8;  // elements per 16 bytes
    vec8 = vec8 && reinterpret_cast<uintptr_t>(m.src) % 16 == 0 && m.ld % per16 == 0 && m.cols % 8 == 0 &&
           m.dst_off % 8 == 0;
  }
  const int threads = 256;
  const int64_t total = vec8 ? a.pairs_end[a.nmat - 1] / 4 : a.pairs_end[a.nmat - 1];
  const int blocks = static_cast<int>(std::min<int64_t>((total + threads - 1) / threads, 148 * 16));
  if (vec8) pack_rows8_kernel<<<blocks, threads, 0, st>>>(a, base);
  else pack_rows_kernel<<<blocks, threads, 0, st>>>(a, base);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------
// device-resident DINO feature table: gather by index with the range check on the device
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 load_oct_as_bf16(const void* src, int dtype, int64_t idx) {
  if (dtype == DSOFT_DT_BF16) return __ldg(reinterpret_cast<const uint4*>(static_cast<const __nv_bfloat16*>(src) + idx));
  if (dtype == DSOFT_DT_F32) {
    const float4 x0 = __ldg(reinterpret_cast<const float4*>(static_cast<const float*>(src) + idx));
    const float4 x1 = __ldg(reinterpret_cast<const float4*>(static_cast<const float*>(src) + idx + 4));
    return make_uint4(pack_bf16x2(x0.x, x0.y), pack_bf16x2(x0.z, x0.w), pack_bf16x2(x1.x, x1.y), pack_bf16x2(x1.z, x1.w));
  }
  const uint4 raw = __ldg(reinterpret_cast<const uint4*>(static_cast<const __half*>(src) + idx));
  const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
  uint32_t o[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[q]));
    o[q] = pack_bf16x2(f.x, f.y);
  }
  return make_uint4(o[0], o[1], o[2], o[3]);
}

// one warp per output row; lanes move 8 elements (16 bytes of bf16) at a time
__global__ void __launch_bounds__(256) gather_rows_kernel(const void* __restrict__ table, int table_dt, int64_t ld_table,
                                                          int64_t n_rows, int cols, const int64_t* __restrict__ indices,
                                                          int n, void* __restrict__ out, int out_dt, int64_t ld_out,
                                                          long long* __restrict__ status) {
  const int lane = threadIdx.x & 31;
  for (int i = blockIdx.x * 8 + (threadIdx.x >> 5); i < n; i += gridDim.x * 8) {
    const long long idx = indices[i];
    const bool ok = idx >= 0 && idx < n_rows;
    if (lane == 0) {  // sticky range record (train.py:255-268 reads min / max / examples on the host every step)
      atomicMin(status + 1, idx);
      atomicMax(status + 2, idx);
      if (!ok) {
        atomicAdd(reinterpret_cast<unsigned long long*>(status), 1ull);
        status[3] = idx;
      }
    }
    for (int c = lane * 8; c < cols; c += 256) {
      uint4 v = make_uint4(0u, 0u, 0u, 0u);
      if (ok) v = load_oct_as_bf16(table, table_dt, idx * ld_table + c);
      if (out_dt == DSOFT_DT_BF16) {
        *reinterpret_cast<uint4*>(static_cast<__nv_bfloat16*>(out) + i * ld_out + c) = v;
      } else {  // fp32 output
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
        float* o = static_cast<float*>(out) + i * ld_out + c;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[q]));
          o[2 * q] = f.x;
          o[2 * q + 1] = f.y;
        }
      }
    }
  }
}

extern "C" size_t dsoft_plan_dino_col_offset(const dsoft_plan_t* p) { return p ? p->offD : 0; }

extern "C" int dsoft_gather_rows(const void* table, int table_dt, int64_t ld_table, int64_t n_rows, int32_t cols,
                                 const int64_t* indices, int32_t n, void* out, int out_dt, int64_t ld_out,
                                 long long* status, void* stream) {
  if (!table || !indices || !out || !status) return fail(DSOFT_EINVAL, "null argument");
  if (table_dt < DSOFT_DT_F32 || table_dt > DSOFT_DT_F16) return fail(DSOFT_EINVAL, "unknown table dtype %d", table_dt);
  if (out_dt != DSOFT_DT_BF16 && out_dt != DSOFT_DT_F32) return fail(DSOFT_EINVAL, "output must be bf16 or fp32");
  if (cols <= 0 || cols % 8 || n < 0 || n_rows <= 0) return fail(DSOFT_EINVAL, "bad shape (cols=%d n=%d)", cols, n);
  const int64_t in_align = table_dt == DSOFT_DT_F32 ? 4 : 8, out_align = out_dt == DSOFT_DT_F32 ? 4 : 8;
  if (ld_table % in_align || ld_out % out_align || reinterpret_cast<uintptr_t>(table) % 16 ||
      reinterpret_cast<uintptr_t>(out) % 16)
    return fail(DSOFT_EINVAL, "gather needs 16-byte aligned rows");
  if (n == 0) return 0;
  int sms = 0;
  int rc = query_num_sms(&sms);
  if (rc) return rc;
  gather_rows_kernel<<<std::min(ceil_div(n, 8), sms * 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      table, table_dt, ld_table, n_rows, cols, indices, n, out, out_dt, ld_out, status);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

static void fill_clip_fwd(const dsoft_plan* p, FwdParams& P, int amap, int bmap, float* scal, float* part,
                          float* diag) {
  memset(&P, 0, sizeof(P));
  P.nprod = 1;
  P.a_map[0] = amap;
  P.b_map[0] = bmap;
  P.kchunks[0] = ceil_div(p->sh.D, BK);
  P.resident = P.kchunks[0] <= 8;
  P.bn = 2 * BN;
  P.row0 = p->sh.rank * p->sh.b;
  P.b = p->sh.b;
  P.col0 = 0;
  P.ncols = p->B;
  P.ntiles = ceil_div(p->B, 2 * BN);
  P.tiles_per_split = p->f_clip.tps;
  P.npart = 2 * p->f_clip.nsplit;
  P.scal = scal;
  P.part = part;
  P.diag = diag;
}

// ------------------------------------------------------------------------------------------------
// denominator-modulated ("weighted") CE branch, loss.py:416-471 + diagnostics loss.py:479-595
// ------------------------------------------------------------------------------------------------
// Per direction (image rows x text columns; text rows x image columns when weight_text_symmetry):
//   STAT tile pass -> wce_rows<0> (c_a, row std) -> wce_median (beta) -> LSE tile pass -> wce_rows<1> (lse~, A_a,
//   row CE) -> DBG tile pass -> wce_rows<2> (diagnostic rows);  then wce_final assembles the loss and the dbg
//   scalars.  Nothing of size B x B is stored; beta stays on the device (the reference's `.item()` syncs are gone).
// World > 1: every pass runs over this rank's [b x B] row block (row0 = rank * b).  beta is the median over all B
// rows, so the row stds leave through the caller's all-gather between wce_rows<0> and wce_median (phases 5 / 6),
// and c, lse~ and A travel with the LSE all-gather (lse_local rows 5 ..) for the backward's column side.
enum { WS_C = 0, WS_LSET = 1, WS_A = 2, WS_STD = 3 };       // state rows per direction: [dir * 4 + k][Bcol]
enum { WR_CE_MOD = 0, WR_CE_BASE, WR_PC, WR_L1, WR_CORR, WR_SABS, WR_SSQ, WR_MAX, WR_POS, WR_DIAG, WR_N };
enum { DBG_N = 32 };

struct WceRowsArgs {
  int b, np, dir;
  int row0, ncols;     // global index of local row 0; columns per row (B)
  float* sig;          // row std of local row i -> sig[(row0 + i) * sig_stride]
  int sig_stride;
  float* ext;          // world > 1: lse_local rows of this direction [3][b] (c, lse~, A), else null
  const float* part;   // [k][np][b]
  const float* lse;    // [b] log2 LSE of the unmodified logits of this direction
  const float* diag;   // [b] raw diagonal dot products
  const float* scal;
  float* wstat;        // state rows of this direction [4][Bcol], by global row
  int Bcol;
  float* wrows;        // [WR_N][b] of this direction
  float cc;
};

template <int PHASE>
__global__ void __launch_bounds__(256) wce_rows_kernel(WceRowsArgs a) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.b) return;
  const float LN2 = 0.6931471805599453f;
  const int st = a.np * a.b;
  float* ws = a.wstat + a.row0;
  if constexpr (PHASE == 0) {
    float c = 0.f;
    double s1 = 0.0, s2 = 0.0;  // sums of x and x^2 in log2 units; fp64 for the E[x^2] - E[x]^2 cancellation
    for (int k = 0; k < a.np; ++k) {
      c += a.part[0 * st + k * a.b + i];
      s1 += static_cast<double>(a.part[1 * st + k * a.b + i]);
      s2 += static_cast<double>(a.part[2 * st + k * a.b + i]);
    }
    const double n = a.ncols;
    const double var = (s2 - s1 * s1 / n) / (n - 1.0);  // torch.std: unbiased (loss.py:440)
    ws[WS_C * a.Bcol + i] = c;
    a.sig[static_cast<size_t>(a.row0 + i) * a.sig_stride] =
        static_cast<float>(sqrt(var > 0.0 ? var : 0.0)) * LN2;  // natural-log units
    if (a.ext) a.ext[i] = c;
  } else if constexpr (PHASE == 1) {
    float m = M_FLOOR;
    for (int k = 0; k < a.np; ++k) m = fmaxf(m, a.part[0 * st + k * a.b + i]);
    float s = 0.f, si = 0.f;
    for (int k = 0; k < a.np; ++k) {
      const float sc = exp2f(a.part[0 * st + k * a.b + i] - m);
      s += a.part[1 * st + k * a.b + i] * sc;
      si += a.part[2 * st + k * a.b + i] * sc;
    }
    const float lset = m + log2f(s);
    ws[WS_LSET * a.Bcol + i] = lset;
    ws[WS_A * a.Bcol + i] = si / s;
    if (a.ext) {
      a.ext[1 * a.b + i] = lset;
      a.ext[2 * a.b + i] = si / s;
    }
    const float xd = a.scal[SC_SCALE] * a.diag[i];
    a.wrows[WR_CE_MOD * a.b + i] = LN2 * lset - xd;       // loss.py:447 / 463: CE row of the modified logits
    a.wrows[WR_CE_BASE * a.b + i] = LN2 * a.lse[i] - xd;  // loss.py:541-542
  } else {
    float acc[11];
    for (int q = 0; q < 11; ++q) {
      float v = 0.f;
      for (int k = 0; k < a.np; ++k)
        v = (q == 9) ? fmaxf(v, a.part[q * st + k * a.b + i]) : v + a.part[q * st + k * a.b + i];
      acc[q] = v;
    }
    const float n = static_cast<float>(a.ncols);
    // rowwise Pearson correlation of r^ and (p~ - p), loss.py:528-536
    const float cov = acc[6] - acc[2] * acc[4] / n;
    const float vr = fmaxf(acc[3] - acc[2] * acc[2] / n, 0.f), vd = fmaxf(acc[5] - acc[4] * acc[4] / n, 0.f);
    a.wrows[WR_PC * a.b + i] = fabsf(acc[0]);
    a.wrows[WR_L1 * a.b + i] = acc[1];
    a.wrows[WR_CORR * a.b + i] = cov / (sqrtf(vr) * sqrtf(vd) + 1e-9f);
    a.wrows[WR_SABS * a.b + i] = acc[7];
    a.wrows[WR_SSQ * a.b + i] = acc[8];
    a.wrows[WR_MAX * a.b + i] = acc[9];
    a.wrows[WR_POS * a.b + i] = acc[10];
    a.wrows[WR_DIAG * a.b + i] = fabsf(fminf(fmaxf(-ws[WS_C * a.Bcol + i], -a.cc), a.cc));  // |r^_ii|, r_ii = 0
  }
}

// beta = rho * max(median_row(std), 1e-6) / c_clip (loss.py:440-443) over the b values v[i * stride].  torch.median
// returns the LOWER of the two middle values: the element of rank (b - 1) / 2.  One block, four 8-bit radix-select
// passes over the bit patterns (non-negative floats order like unsigned integers).
__global__ void __launch_bounds__(1024) wce_median_kernel(const float* __restrict__ v, int b, int stride, float rho,
                                                          float cc, float* __restrict__ scal, int dir) {
  __shared__ unsigned hist[256];
  __shared__ unsigned s_prefix, s_rank;
  if (threadIdx.x == 0) { s_prefix = 0u; s_rank = static_cast<unsigned>((b - 1) / 2); }
  __syncthreads();
  for (int shift = 24; shift >= 0; shift -= 8) {
    if (threadIdx.x < 256) hist[threadIdx.x] = 0u;
    __syncthreads();
    const unsigned prefix = s_prefix;
    const unsigned mask = shift == 24 ? 0u : (0xffffffffu << (shift + 8));
    for (int i = threadIdx.x; i < b; i += blockDim.x) {
      const unsigned key = __float_as_uint(v[static_cast<size_t>(i) * stride]);
      if ((key & mask) == prefix) atomicAdd(&hist[(key >> shift) & 255u], 1u);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      unsigned rank = s_rank, bin = 0u;
      for (; bin < 256u; ++bin) {
        if (rank < hist[bin]) break;
        rank -= hist[bin];
      }
      s_prefix = prefix | (bin << shift);
      s_rank = rank;
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const float sigma = fmaxf(__uint_as_float(s_prefix), 1e-6f);
    const float beta = rho * sigma / cc;
    scal[SC_WBETA + dir] = beta;
    scal[SC_WBETA2 + dir] = beta * 1.4426950408889634f;
  }
}

struct WceFinalArgs {
  int b, sym;
  int ncols;           // columns per row (B): the diagnostics over all entries count b x ncols
  const float* wrows;  // [2][WR_N][b]
  const float* lse;    // [5][b] (only the text direction's base CE needs it when !sym)
  const float* diag;
  const float* scal;
  float rho, cc, lam_w;
  float* losses;       // [6]: total (4) gets + lam_w * weighted, weighted -> (5)
  float* dbg;          // [DBG_N] or null
};

// one block: deterministic fp64 reductions over the per-row results, then the scalars
__global__ void __launch_bounds__(1024) wce_final_kernel(WceFinalArgs a) {
  __shared__ double sh[32];
  __shared__ double res[2][WR_N];
  const float LN2 = 0.6931471805599453f;
  for (int d = 0; d < 2; ++d) {
    for (int k = 0; k < WR_N; ++k) {
      double acc = 0.0;
      const bool is_max = (k == WR_MAX || k == WR_DIAG);
      const bool have = d == 0 || a.sym || k == WR_CE_BASE;
      if (have) {
        for (int i = threadIdx.x; i < a.b; i += blockDim.x) {
          double v;
          if (d == 1 && !a.sym) v = LN2 * a.lse[1 * a.b + i] - a.scal[SC_SCALE] * a.diag[i];  // plain text-direction CE
          else v = a.wrows[(d * WR_N + k) * a.b + i];
          acc = is_max ? fmax(acc, v) : acc + v;
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const double w = __shfl_xor_sync(0xffffffffu, acc, o);
        acc = is_max ? fmax(acc, w) : acc + w;
      }
      if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = acc;
      __syncthreads();
      if (threadIdx.x == 0) {
        double t = sh[0];
        for (int w = 1; w < 32; ++w) t = is_max ? fmax(t, sh[w]) : t + sh[w];
        res[d][k] = t;
      }
      __syncthreads();
    }
  }
  if (threadIdx.x != 0) return;
  const double n = a.b, nn = n * a.ncols, off = nn - n;
  const double ce_img_mod = res[0][WR_CE_MOD] / n, ce_img_base = res[0][WR_CE_BASE] / n;
  const double ce_txt_base = res[1][WR_CE_BASE] / n;
  const double ce_txt_mod = a.sym ? res[1][WR_CE_MOD] / n : ce_txt_base;
  const float weighted = static_cast<float>(0.5 * (ce_img_mod + ce_txt_mod));  // loss.py:466
  a.losses[5] = weighted;
  a.losses[4] += a.lam_w * weighted;                                           // loss.py:473-477
  if (!a.dbg) return;
  float* g = a.dbg;
  for (int k = 0; k < DBG_N; ++k) g[k] = 0.f;
  for (int d = 0; d < (a.sym ? 2 : 1); ++d) {
    const double beta = a.scal[SC_WBETA + d];
    const double sabs = beta * res[d][WR_SABS], ssq = beta * beta * res[d][WR_SSQ];
    const double var = (ssq - sabs * sabs / nn) / (nn - 1.0);  // std of |Delta| over all b x B entries (diag = 0)
    g[0 + d] = static_cast<float>(res[d][WR_PC] / n);          // pc_err
    g[2 + d] = static_cast<float>(res[d][WR_DIAG]);            // diag_max
    g[4 + 3 * d] = static_cast<float>(beta * res[d][WR_MAX]);  // delta max / mean / std
    g[5 + 3 * d] = static_cast<float>(sabs / nn);
    g[6 + 3 * d] = static_cast<float>(sqrt(var > 0.0 ? var : 0.0));
    g[10 + d] = static_cast<float>(res[d][WR_L1] / n);         // l1_prob_shift
    g[12 + d] = static_cast<float>(res[d][WR_CORR] / n);       // corr_rhat_dprob
    g[18 + 2 * d] = static_cast<float>(res[d][WR_POS] / off);  // pos_frac, neg_frac
    g[19 + 2 * d] = 1.f - g[18 + 2 * d];
    g[22 + d] = static_cast<float>(beta);
  }
  g[14] = static_cast<float>(ce_img_base);
  g[15] = static_cast<float>(ce_txt_base);
  g[16] = static_cast<float>(ce_img_mod);
  g[17] = static_cast<float>(ce_txt_mod);
  g[24] = a.rho;
  g[25] = a.cc;
}

// Backward scalar of the weighted CE branch: gk = 2^(14 - e) with |G| < 2^e, so that the fp16 logit gradient of
// MODE_WCE_G / MODE_WCE_X holds G gk with |G gk| < 2^15 at any upstream gradient (a GradScaler's 2^16 and more) and
// keeps its precision at small ones.  From wce_pair: e1, e2, p~ <= 1, A in [0, 1] and |r - c| <= 2, so
// |G| <= 2 |g_c| + |g_w| (2 + 2 beta_img + 2 beta_txt), beta_txt only when the text direction is modulated.  e is
// clamped only so that 1/gk, folded into the finalize's s / (2b gk), stays a normal fp32 number (gk <= 2^64).
__global__ void wce_gscale_kernel(const float* __restrict__ gout, float lam_orig, float lam_w, int wsym,
                                  float* __restrict__ scal) {
  const float gc = gout[0] + lam_orig * gout[4], gw = gout[5] + lam_w * gout[4];
  const float bsum = scal[SC_WBETA + 0] + (wsym ? scal[SC_WBETA + 1] : 0.f);
  int e = 0;
  frexpf(2.f * fabsf(gc) + fabsf(gw) * (2.f + 2.f * bsum), &e);
  e = max(e, -50);
  scal[SC_WCE_GK] = ldexpf(1.f, 14 - e);
  scal[SC_WCE_IGK] = ldexpf(1.f, e - 14);
}

// world > 1, backward: c, lse~ and A of every rank's rows ([W][nr][b] rows 5 + 3 d + k, as all-gathered) -> the
// state rows [d][k][Bcol] by global row (zero padded), where the column side of the logit-gradient kernels reads them
__global__ void __launch_bounds__(256) wce_relayout_kernel(const float* __restrict__ lse_all, int W, int b, int nr,
                                                           int Bcol, int nd, float* __restrict__ wstat) {
  static_assert(WS_C == 0 && WS_LSET == 1 && WS_A == 2, "lse_local carries c, lse~, A in state-row order");
  const int total = 3 * nd * Bcol;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int dk = i / Bcol, j = i % Bcol, d = dk / 3, k = dk % 3;
    wstat[(static_cast<size_t>(d) * 4 + k) * Bcol + j] =
        j < W * b ? lse_all[(static_cast<size_t>(j / b) * nr + 5 + dk) * b + (j % b)] : 0.f;
  }
}

template <typename K>
static int launch_fwd_pair(K kernel, int rbs, int nsplit, cudaStream_t st, const TileMaps& tm, const FwdParams& P,
                           int threads);
template <typename K>
static int set_smem(K kernel, int bytes);

static void fill_wce(const dsoft_plan* p, FwdParams& P, int dir, float* S, float* part) {
  memset(&P, 0, sizeof(P));
  P.nprod = 2;
  P.bn = 2 * BN;
  P.a_map[0] = dir == 0 ? 0 : 1;  // CLIP logits: image rows x text columns / text rows x image columns
  P.b_map[0] = dir == 0 ? 1 : 0;
  P.a_map[1] = P.b_map[1] = 3;    // DINO cosine (symmetric: r^T = r, loss.py:453)
  P.kchunks[0] = ceil_div(p->sh.D, BK);
  P.kchunks[1] = ceil_div(p->sh.Dd, BK);
  P.row0 = p->sh.rank * p->sh.b;
  P.b = p->sh.b;
  P.col0 = 0;
  P.ncols = p->B;
  P.ntiles = ceil_div(p->B, 2 * BN);
  P.tiles_per_split = p->f_wce.tps;
  P.npart = 2 * p->f_wce.nsplit;
  P.scal = S + p->st_scal;
  P.part = part;
  P.ncolvec = 1;
  P.colvec[0] = S + p->st_rinv_d;
  P.wdir = dir;
  P.wcc = p->sh.c_clip;
}

// forward of the weighted branch; runs after finalize_fwd_kernel (needs the CLIP row LSEs and the diagonal).
// part_a: the row statistics up to the row stds; part_b: median onward.  World > 1 runs them as two calls with the
// caller's all-gather of the row stds in between.
static int weighted_forward(const dsoft_plan* p, const TileMaps& tm, float* S, float* X, float* lse_local,
                            float lam_w, float* losses, float* dbg, cudaStream_t st, bool part_a, bool part_b) {
  const int b = p->sh.b, rbs = ceil_div(b, BM), ns = p->f_wce.nsplit, row0 = p->sh.rank * b;
  const bool multi = p->sh.world > 1;
  int rc;
  if ((rc = set_smem(dsoft_fwd_kernel<MODE_WCE_STAT, 2>, FWD_SMEM_BYTES))) return rc;
  if ((rc = set_smem(dsoft_fwd_kernel<MODE_WCE_LSE, 2>, FWD_SMEM_BYTES))) return rc;
  if ((rc = set_smem(dsoft_fwd_kernel<MODE_WCE_DBG, 2>, FWD_SMEM_BYTES))) return rc;
  float* part = X + p->sc_wpart;
  const int rg = ceil_div(b, 256);
  for (int stage = 0; stage < 2; ++stage) {
    if (!(stage == 0 ? part_a : part_b)) continue;
    for (int d = 0; d < p->wnd; ++d) {
      float* ws = S + p->st_wstat + static_cast<size_t>(d) * 4 * p->Bcol;
      FwdParams P;
      fill_wce(p, P, d, S, part);
      P.wrow[0] = lse_local + d * b;
      P.wrow[1] = ws + WS_C * p->Bcol + row0;
      P.wrow[2] = ws + WS_LSET * p->Bcol + row0;
      WceRowsArgs ra;
      ra.b = b; ra.np = 2 * ns; ra.dir = d; ra.part = part; ra.lse = lse_local + d * b; ra.diag = S + p->st_diag;
      ra.scal = S + p->st_scal; ra.wstat = ws; ra.Bcol = p->Bcol; ra.wrows = X + p->sc_wrows + static_cast<size_t>(d) * WR_N * b;
      ra.cc = p->sh.c_clip;
      ra.row0 = row0;
      ra.ncols = p->B;
      ra.sig = multi ? S + p->st_wsig + d : ws + WS_STD * p->Bcol;
      ra.sig_stride = multi ? p->wnd : 1;
      ra.ext = multi ? lse_local + static_cast<size_t>(5 + 3 * d) * b : nullptr;
      if (stage == 0) {
        if ((rc = launch_fwd_pair(dsoft_fwd_kernel<MODE_WCE_STAT, 2>, rbs, ns, st, tm, P))) return rc;
        wce_rows_kernel<0><<<rg, 256, 0, st>>>(ra);
      } else {
        // over all B rows: ra.sig is the start of the (all-gathered) block, indexed by global row
        wce_median_kernel<<<1, 1024, 0, st>>>(ra.sig, p->B, ra.sig_stride, p->sh.rho, p->sh.c_clip, S + p->st_scal, d);
        if ((rc = launch_fwd_pair(dsoft_fwd_kernel<MODE_WCE_LSE, 2>, rbs, ns, st, tm, P))) return rc;
        wce_rows_kernel<1><<<rg, 256, 0, st>>>(ra);
        if (dbg) {
          if ((rc = launch_fwd_pair(dsoft_fwd_kernel<MODE_WCE_DBG, 2>, rbs, ns, st, tm, P))) return rc;
          wce_rows_kernel<2><<<rg, 256, 0, st>>>(ra);
        }
      }
      CUDA_TRY(cudaGetLastError());
    }
  }
  if (!part_b) return 0;
  WceFinalArgs fa;
  fa.b = b; fa.sym = p->wsym; fa.wrows = X + p->sc_wrows; fa.lse = lse_local; fa.diag = S + p->st_diag;
  fa.scal = S + p->st_scal; fa.rho = p->sh.rho; fa.cc = p->sh.c_clip; fa.lam_w = lam_w; fa.losses = losses; fa.dbg = dbg;
  fa.ncols = p->B;
  wce_final_kernel<<<1, 1024, 0, st>>>(fa);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------
// projection head, forward (loss.py:214-238, 322-347): Linear [-> ReLU -> Linear] on the tcgen05 tile kernel,
// bias / ReLU / bf16 rounding in the epilogue, the last layer written into the student columns of `gathered`
// ------------------------------------------------------------------------------------------------
static int launch_linear(const dsoft_plan* p, const __nv_bfloat16* A, int a_rows, int64_t lda, int row0, int rows,
                         int K, const __nv_bfloat16* Wt, int N, const float* bias, int relu, __nv_bfloat16* out,
                         int64_t ld_out, cudaStream_t st) {
  if (K % 8 || N % 8 || lda % 8 || ld_out % 8)
    return fail(DSOFT_EINVAL, "head dims and row strides must be multiples of 8 (K=%d N=%d)", K, N);
  if (reinterpret_cast<uintptr_t>(A) % 16 || reinterpret_cast<uintptr_t>(Wt) % 16 ||
      reinterpret_cast<uintptr_t>(out) % 16 || (bias && reinterpret_cast<uintptr_t>(bias) % 16))
    return fail(DSOFT_EINVAL, "head operands must be 16-byte aligned");
  TileMaps tm;
  int rc;
  const CUtensorMapDataType bf = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  if ((rc = make_map(&tm.m[0], A, a_rows, K, static_cast<size_t>(lda), bf, 64))) return rc;
  if ((rc = make_map(&tm.m[1], Wt, N, K, static_cast<size_t>(K), bf, 64))) return rc;
  tm.m[2] = tm.m[3] = tm.g[0] = tm.g[1] = tm.m[0];
  FwdParams P;
  memset(&P, 0, sizeof(P));
  P.nprod = 1;
  P.a_map[0] = 0;
  P.b_map[0] = 1;
  P.kchunks[0] = ceil_div(K, BK);
  P.resident = P.kchunks[0] <= 8;
  P.bn = 2 * BN;
  P.row0 = row0;
  P.b = rows;
  P.col0 = 0;
  P.ncols = N;
  P.ntiles = ceil_div(N, 2 * BN);
  // enough row pairs to fill the machine: one CTA pair walks all N tiles of its rows (the row operand is loaded
  // once and tile t's epilogue overlaps tile t+1's MMAs); few row pairs (small per-rank batches): one tile per CTA
  const int pairs = ceil_div(ceil_div(rows, BM), 2);
  P.tiles_per_split = (2 * pairs >= p->num_sms) ? P.ntiles : 1;
  const int nsplit = ceil_div(P.ntiles, P.tiles_per_split);
  P.npart = 2 * nsplit;
  P.lin_out = out;
  P.lin_ld = static_cast<int>(ld_out);
  P.lin_bias = bias;
  P.lin_relu = relu;
  if ((rc = set_smem(dsoft_fwd_kernel<MODE_LINEAR, 2>, FWD_SMEM_BYTES))) return rc;
  return launch_fwd_pair(dsoft_fwd_kernel<MODE_LINEAR, 2>, ceil_div(rows, BM), nsplit, st, tm, P);
}

extern "C" int dsoft_head_forward(const dsoft_plan_t* p, void* gathered, const void* w1, const float* b1,
                                  const void* w2, const float* b2, int32_t hidden_dim, void* hidden, void* stream) {
  if (!p || !gathered || !w1) return fail(DSOFT_EINVAL, "null argument");
  if (!p->have_proj) return fail(DSOFT_EINVAL, "the plan has no projected student (Dp == 0)");
  const bool mlp = hidden_dim > 0;
  if (mlp && (!w2 || !hidden)) return fail(DSOFT_EINVAL, "an MLP head needs w2 and the hidden buffer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  __nv_bfloat16* g = static_cast<__nv_bfloat16*>(gathered);
  const int b = p->sh.b, row0 = p->sh.rank * b;
  __nv_bfloat16* zout = g + static_cast<size_t>(row0) * p->row_elems + p->offZ;  // student columns, local rows
  int rc;
  if (!mlp)  // Linear(D -> Dp)
    return launch_linear(p, g + p->offI, p->B, p->row_elems, row0, b, p->sh.D, static_cast<const __nv_bfloat16*>(w1),
                         p->sh.Dp, b1, 0, zout, p->row_elems, st);
  // Linear(D -> H) + ReLU -> hidden (kept for the backward), Linear(H -> Dp) -> student columns
  __nv_bfloat16* h = static_cast<__nv_bfloat16*>(hidden);
  if ((rc = launch_linear(p, g + p->offI, p->B, p->row_elems, row0, b, p->sh.D,
                          static_cast<const __nv_bfloat16*>(w1), hidden_dim, b1, 1, h, hidden_dim, st)))
    return rc;
  return launch_linear(p, h, b, hidden_dim, 0, b, hidden_dim, static_cast<const __nv_bfloat16*>(w2), p->sh.Dp, b2, 0,
                       zout, p->row_elems, st);
}

// ------------------------------------------------------------------------------------------------
// CLIP-blind pair statistics (open_clip_train/helpers.py:221-285, _pair_stats) on the Gram-tile kernel
// ------------------------------------------------------------------------------------------------
extern "C" int dsoft_pair_stats(const void* clip_a, const void* clip_b, int32_t k_clip, const void* dino_a,
                                const void* dino_b, int32_t k_dino, int32_t n, const float* cmin, const float* dmax,
                                int32_t n_thr, unsigned long long* counts, float gap_floor, void* cand,
                                uint32_t cand_cap, uint32_t* cand_count, void* stream) {
  if (!clip_a || !clip_b || !dino_a || !dino_b || !cand_count) return fail(DSOFT_EINVAL, "null argument");
  if (n <= 1 || k_clip <= 0 || k_dino <= 0 || k_clip % 8 || k_dino % 8)
    return fail(DSOFT_EINVAL, "need n > 1 and feature widths that are positive multiples of 8 (n=%d, %d, %d)", n,
                k_clip, k_dino);
  if (n_thr < 0 || n_thr > 8 || (n_thr > 0 && (!cmin || !dmax)))
    return fail(DSOFT_EINVAL, "at most 8 threshold pairs (got %d)", n_thr);
  if (cand_cap > 0 && !cand) return fail(DSOFT_EINVAL, "cand_cap > 0 needs a candidate buffer");
  for (const void* q : {clip_a, clip_b, dino_a, dino_b})
    if (reinterpret_cast<uintptr_t>(q) % 16) return fail(DSOFT_EINVAL, "operands must be 16-byte aligned");
  int sms = 0, rc = query_num_sms(&sms);
  if (rc) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  TileMaps tm;
  const CUtensorMapDataType bf = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  if ((rc = make_map(&tm.m[0], clip_a, n, k_clip, static_cast<size_t>(k_clip), bf, 64))) return rc;
  if ((rc = make_map(&tm.m[1], clip_b, n, k_clip, static_cast<size_t>(k_clip), bf, 64))) return rc;
  if ((rc = make_map(&tm.m[2], dino_a, n, k_dino, static_cast<size_t>(k_dino), bf, 64))) return rc;
  if ((rc = make_map(&tm.m[3], dino_b, n, k_dino, static_cast<size_t>(k_dino), bf, 64))) return rc;
  tm.g[0] = tm.g[1] = tm.m[0];
  FwdParams P;
  memset(&P, 0, sizeof(P));
  P.nprod = 2;
  P.a_map[0] = 0; P.b_map[0] = 1; P.kchunks[0] = ceil_div(k_clip, BK);
  P.a_map[1] = 2; P.b_map[1] = 3; P.kchunks[1] = ceil_div(k_dino, BK);
  P.bn = 2 * BN;
  P.row0 = 0;
  P.b = n;
  P.col0 = 0;
  P.ncols = n;
  P.ntiles = ceil_div(n, 2 * BN);
  P.tri = 1;  // upper block triangle: pairs i < j
  P.tiles_per_split = std::max(4, ceil_div(P.ntiles, 10));
  const int nsplit = ceil_div(P.ntiles, P.tiles_per_split);
  P.npart = 2 * nsplit;
  P.ncolvec = 0;
  P.pr_nthr = counts ? n_thr : 0;
  for (int k = 0; k < n_thr; ++k) {
    P.pr_cmin[k] = cmin[k];
    P.pr_dmax[k] = dmax[k];
  }
  P.pr_counts = (counts && n_thr > 0) ? counts : nullptr;
  P.pr_gap_floor = cand_cap > 0 ? gap_floor : 3.0e38f;
  P.pr_cand = static_cast<float4*>(cand);
  P.pr_cand_cap = cand_cap;
  P.pr_cand_count = cand_count;
  if ((rc = set_smem(dsoft_fwd_kernel<MODE_PAIRS, 2>, FWD_SMEM_BYTES))) return rc;
  return launch_fwd_pair(dsoft_fwd_kernel<MODE_PAIRS, 2>, ceil_div(n, BM), nsplit, st, tm, P);
}

// ------------------------------------------------------------------------------------------------
// Retrieval ranks (open_clip get_clip_metrics, open_clip_train/train.py) on the Gram-tile kernel: MODE_RANKS counts,
// per image and per caption, the non-positive scores above the positive's.  The thresholds come from a small fp32
// pre-pass over the same bf16 operands; nothing of size n_img x n_txt exists.
// Scratch: thr [n_txt padded to 256] fp32 | t(j) [same] int32 | p [n_img padded to 64] fp32
// ------------------------------------------------------------------------------------------------
static size_t rk_cols(int n_txt) { return static_cast<size_t>(ceil_div(n_txt, 2 * BN)) * (2 * BN); }

extern "C" size_t dsoft_retrieval_scratch_bytes(int32_t n_img, int32_t n_txt) {
  if (n_img <= 0 || n_txt <= 0) return 0;
  return 4 * (2 * rk_cols(n_txt) + align_up(static_cast<size_t>(n_img), 64));
}

// thr = +inf and t(j) = -1 past n_txt (nothing counts there), p = -inf, ranks = 0
__global__ void rk_init_kernel(const int32_t* __restrict__ tmap_in, int n_img, int n_txt, int ncols_pad,
                               float* __restrict__ thr, int* __restrict__ tmap, float* __restrict__ p,
                               int* __restrict__ rank_img, int* __restrict__ rank_txt) {
  const int n = max(ncols_pad, n_img);
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
    if (k < ncols_pad) {
      thr[k] = __int_as_float(0x7f800000);
      tmap[k] = (k < n_txt && tmap_in) ? tmap_in[k] : -1;
      if (k < n_txt) rank_txt[k] = 0;
    }
    if (k < n_img) {
      p[k] = __int_as_float(static_cast<int>(0xff800000u));
      rank_img[k] = 0;
    }
  }
}

// float maximum through integer atomics (order-independent): non-negative floats order as signed ints, negative ones
// in reverse as unsigned ints; -0.0 takes the unsigned path so that it still replaces -inf
__device__ __forceinline__ void atomic_max_f32(float* a, float v) {
  if (!signbit(v)) atomicMax(reinterpret_cast<int*>(a), __float_as_int(v));
  else atomicMin(reinterpret_cast<unsigned int*>(a), __float_as_uint(v));
}

// one warp per caption j: thr_j = <img[t(j)], txt[j]> in fp32 from the bf16 operands, p_t(j) = max(p_t(j), thr_j).
// A map entry outside [0, n_img) leaves thr_j = +inf (the caption counts nothing) instead of reading out of bounds.
__global__ void rk_thr_kernel(const __nv_bfloat16* __restrict__ img, const __nv_bfloat16* __restrict__ txt, int k,
                              int n_img, int n_txt, const int* __restrict__ tmap, int mapped, float* __restrict__ thr,
                              float* __restrict__ p) {
  const int j = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (j >= n_txt) return;
  const int i = mapped ? tmap[j] : j;
  if (i < 0 || i >= n_img) return;
  const uint4* a = reinterpret_cast<const uint4*>(img + static_cast<size_t>(i) * k);
  const uint4* b = reinterpret_cast<const uint4*>(txt + static_cast<size_t>(j) * k);
  float acc = 0.f;
  for (int c = lane; c < k / 8; c += 32) {
    const uint4 x = __ldg(a + c), y = __ldg(b + c);
    const __nv_bfloat162* xa = reinterpret_cast<const __nv_bfloat162*>(&x);
    const __nv_bfloat162* ya = reinterpret_cast<const __nv_bfloat162*>(&y);
#pragma unroll
    for (int h = 0; h < 4; ++h) {
      const float2 xf = __bfloat1622float2(xa[h]), yf = __bfloat1622float2(ya[h]);
      acc = fmaf(xf.x, yf.x, acc);
      acc = fmaf(xf.y, yf.y, acc);
    }
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) {
    thr[j] = acc;
    if (mapped) atomic_max_f32(p + i, acc);
    else p[i] = acc;
  }
}

extern "C" int dsoft_retrieval_ranks(const void* img, const void* txt, int32_t k, int32_t n_img, int32_t n_txt,
                                     const int32_t* text_image, int32_t* rank_img, int32_t* rank_txt, void* scratch,
                                     void* stream) {
  if (!img || !txt || !rank_img || !rank_txt || !scratch) return fail(DSOFT_EINVAL, "null argument");
  if (n_img <= 0 || n_txt <= 0 || k <= 0 || k % 8)
    return fail(DSOFT_EINVAL, "need n_img, n_txt > 0 and a feature width that is a positive multiple of 8 "
                              "(n_img=%d n_txt=%d k=%d)", n_img, n_txt, k);
  if (!text_image && n_img != n_txt)
    return fail(DSOFT_EINVAL, "without a caption -> image map n_img must equal n_txt (%d, %d)", n_img, n_txt);
  for (const void* q : {img, txt, static_cast<const void*>(scratch)})
    if (reinterpret_cast<uintptr_t>(q) % 16) return fail(DSOFT_EINVAL, "operands and scratch must be 16-byte aligned");
  int sms = 0, rc = query_num_sms(&sms);
  if (rc) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int ncols_pad = static_cast<int>(rk_cols(n_txt));
  float* thr = static_cast<float*>(scratch);
  int* tmap = reinterpret_cast<int*>(thr + ncols_pad);
  float* pmax = reinterpret_cast<float*>(tmap + ncols_pad);
  const int mapped = text_image != nullptr;
  const int ninit = std::max(ncols_pad, static_cast<int>(n_img));
  rk_init_kernel<<<std::min(ceil_div(ninit, 256), 4 * sms), 256, 0, st>>>(text_image, n_img, n_txt, ncols_pad, thr,
                                                                          tmap, pmax, rank_img, rank_txt);
  CUDA_TRY(cudaGetLastError());
  const __nv_bfloat16* a = static_cast<const __nv_bfloat16*>(img);
  const __nv_bfloat16* b = static_cast<const __nv_bfloat16*>(txt);
  rk_thr_kernel<<<ceil_div(n_txt, 8), 256, 0, st>>>(a, b, k, n_img, n_txt, tmap, mapped, thr, pmax);
  CUDA_TRY(cudaGetLastError());

  TileMaps tm;
  const CUtensorMapDataType bf = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  if ((rc = make_map(&tm.m[0], img, n_img, k, static_cast<size_t>(k), bf, 64))) return rc;
  if ((rc = make_map(&tm.m[1], txt, n_txt, k, static_cast<size_t>(k), bf, 64))) return rc;
  tm.m[2] = tm.m[3] = tm.g[0] = tm.g[1] = tm.m[0];
  FwdParams P;
  memset(&P, 0, sizeof(P));
  P.nprod = 1;
  P.a_map[0] = 0;
  P.b_map[0] = 1;
  P.kchunks[0] = ceil_div(k, BK);
  P.bn = 2 * BN;
  P.row0 = 0;
  P.b = n_img;
  P.col0 = 0;
  P.ncols = n_txt;
  P.ntiles = ceil_div(n_txt, 2 * BN);
  const int rbs = ceil_div(n_img, BM);
  const SplitPlan sp = choose_split(rbs, 1, P.ntiles, sms);
  P.tiles_per_split = sp.tps;
  P.npart = 2 * sp.nsplit;
  P.ncolvec = mapped ? 2 : 1;
  P.colvec[0] = thr;
  P.colvec[1] = reinterpret_cast<const float*>(tmap);
  P.rk_p = pmax;
  P.rk_img = rank_img;
  P.rk_txt = rank_txt;
  P.rk_mapped = mapped;
  if ((rc = set_smem(dsoft_fwd_kernel<MODE_RANKS, 2>, FWD_SMEM_BYTES))) return rc;
  return launch_fwd_pair(dsoft_fwd_kernel<MODE_RANKS, 2>, rbs, sp.nsplit, st, tm, P);
}

// ------------------------------------------------------------------------------------------------
// kNN top-k (DINO's knn_classifier) on the Gram-tile kernel: MODE_TOPK keeps, per query, the KL best keys of each
// 128-column strip of each column split in registers (KL = 32 for k <= 32, else 64); knn_merge_kernel selects the
// top-k of those 2 nsplit sorted lists.  Nothing of size n_q x n_k exists.
// Scratch: key scale [n_k padded to 256] fp32 | partial scores [2 nsplit][n_q][KL] fp32 | their key indices int32
// ------------------------------------------------------------------------------------------------
static int knn_list(int k) { return k <= 32 ? 32 : 64; }
static bool knn_args_ok(int n_q, int n_k, int k) { return n_q > 0 && n_k > 0 && k >= 1 && k <= 64 && k <= n_k; }
static SplitPlan knn_split(int n_q, int n_k, int sms) {
  return choose_split(ceil_div(n_q, BM), 1, ceil_div(n_k, 2 * BN), sms);
}
static size_t knn_list_elems(int n_q, int k, const SplitPlan& sp) {
  return static_cast<size_t>(2 * sp.nsplit) * static_cast<size_t>(n_q) * knn_list(k);
}

extern "C" size_t dsoft_knn_scratch_bytes(int32_t n_q, int32_t n_k, int32_t k) {
  if (!knn_args_ok(n_q, n_k, k)) return 0;
  int sms = 0;
  if (query_num_sms(&sms)) return 0;
  return 4 * rk_cols(n_k) + 8 * knn_list_elems(n_q, k, knn_split(n_q, n_k, sms));
}

// the key scale padded to whole tiles (1 where none is given; columns past n_k never enter a list)
__global__ void knn_scale_kernel(const float* __restrict__ in, int n_k, int ncols_pad, float* __restrict__ out) {
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < ncols_pad; j += gridDim.x * blockDim.x)
    out[j] = (in && j < n_k) ? in[j] : 1.f;
}

// one warp per query: k steps of a merge of the 2 nsplit partial lists (each sorted by decreasing score, ties by
// increasing key index; a key lies in exactly one list).  Lane l holds the heads of lists l, l + 32, ..; per step the
// warp reduces the lanes' best heads to the winner and its lane advances that list.
template <int KL>
__global__ void __launch_bounds__(256) knn_merge_kernel(const float* __restrict__ pv, const int* __restrict__ pi,
                                                        int nlists, int n_q, int k, float* __restrict__ out_v,
                                                        int* __restrict__ out_i) {
  constexpr int R = 4;  // lists per lane: nlists = 2 nsplit <= 128
  const int q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (q >= n_q) return;
  const float neg_inf = __int_as_float(static_cast<int>(0xff800000u));
  auto better = [](float a, int ai, float b, int bi) { return a > b || (a == b && ai < bi); };
  int pos[R] = {0, 0, 0, 0};
  float hv[R];
  int hi[R];
  auto head = [&](int r) {
    const int l = lane + 32 * r;
    if (l < nlists && pos[r] < KL) {
      const size_t o = (static_cast<size_t>(l) * n_q + q) * KL + pos[r];
      hv[r] = pv[o];
      hi[r] = pi[o];
    } else {
      hv[r] = neg_inf;
      hi[r] = 0x7fffffff;
    }
  };
#pragma unroll
  for (int r = 0; r < R; ++r) head(r);
  for (int n = 0; n < k; ++n) {
    float bv = hv[0];
    int bi = hi[0], br = 0;
#pragma unroll
    for (int r = 1; r < R; ++r)
      if (better(hv[r], hi[r], bv, bi)) {
        bv = hv[r];
        bi = hi[r];
        br = r;
      }
    float wv = bv;
    int wi = bi;
#pragma unroll
    for (int o = 16; o; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, wv, o);
      const int oi = __shfl_xor_sync(0xffffffffu, wi, o);
      if (better(ov, oi, wv, wi)) {
        wv = ov;
        wi = oi;
      }
    }
    if (lane == 0) {
      out_v[static_cast<size_t>(q) * k + n] = wv;
      out_i[static_cast<size_t>(q) * k + n] = wi;
    }
    if (bi == wi) {  // key indices are unique, so exactly one lane holds the winner
#pragma unroll
      for (int r = 0; r < R; ++r)
        if (r == br) {
          ++pos[r];
          head(r);
        }
    }
  }
}

template <int MODE>
static int knn_launch(const TileMaps& tm, const FwdParams& P, int rbs, int nsplit, int n_q, int k, float* values,
                      int32_t* indices, cudaStream_t st) {
  int rc;
  if ((rc = set_smem(dsoft_fwd_kernel<MODE, 2>, FWD_SMEM_BYTES))) return rc;
  if ((rc = launch_fwd_pair(dsoft_fwd_kernel<MODE, 2>, rbs, nsplit, st, tm, P))) return rc;
  knn_merge_kernel<topk_list(MODE)><<<ceil_div(n_q, 8), 256, 0, st>>>(P.tk_val, P.tk_idx, 2 * nsplit, n_q, k, values,
                                                                      indices);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

extern "C" int dsoft_knn_topk(const void* q_dev, const void* k_dev, int32_t width, int32_t n_q, int32_t n_k,
                              int32_t k, const float* key_scale_dev, const float* query_scale_dev, float* values_dev,
                              int32_t* indices_dev, void* scratch_dev, void* stream) {
  if (!q_dev || !k_dev || !values_dev || !indices_dev || !scratch_dev) return fail(DSOFT_EINVAL, "null argument");
  if (n_q <= 0 || n_k <= 0 || width <= 0 || width % 8)
    return fail(DSOFT_EINVAL, "need n_q, n_k > 0 and a feature width that is a positive multiple of 8 "
                              "(n_q=%d n_k=%d width=%d)", n_q, n_k, width);
  if (!knn_args_ok(n_q, n_k, k)) return fail(DSOFT_EINVAL, "need 1 <= k <= 64 and k <= n_k (k=%d n_k=%d)", k, n_k);
  for (const void* p : {q_dev, k_dev, static_cast<const void*>(scratch_dev)})
    if (reinterpret_cast<uintptr_t>(p) % 16) return fail(DSOFT_EINVAL, "operands and scratch must be 16-byte aligned");
  int sms = 0, rc = query_num_sms(&sms);
  if (rc) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const SplitPlan sp = knn_split(n_q, n_k, sms);
  const int ncols_pad = static_cast<int>(rk_cols(n_k));
  float* kscale = static_cast<float*>(scratch_dev);
  float* pv = kscale + ncols_pad;
  int* pi = reinterpret_cast<int*>(pv + knn_list_elems(n_q, k, sp));
  knn_scale_kernel<<<std::min(ceil_div(ncols_pad, 256), 4 * sms), 256, 0, st>>>(key_scale_dev, n_k, ncols_pad,
                                                                                kscale);
  CUDA_TRY(cudaGetLastError());

  TileMaps tm;
  const CUtensorMapDataType bf = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  if ((rc = make_map(&tm.m[0], q_dev, n_q, width, static_cast<size_t>(width), bf, 64))) return rc;
  if ((rc = make_map(&tm.m[1], k_dev, n_k, width, static_cast<size_t>(width), bf, 64))) return rc;
  tm.m[2] = tm.m[3] = tm.g[0] = tm.g[1] = tm.m[0];
  FwdParams P;
  memset(&P, 0, sizeof(P));
  P.nprod = 1;
  P.a_map[0] = 0;
  P.b_map[0] = 1;
  P.kchunks[0] = ceil_div(width, BK);
  P.bn = 2 * BN;
  P.row0 = 0;
  P.b = n_q;
  P.col0 = 0;
  P.ncols = n_k;
  P.ntiles = ceil_div(n_k, 2 * BN);
  P.tiles_per_split = sp.tps;
  P.npart = 2 * sp.nsplit;
  P.ncolvec = 1;
  P.colvec[0] = kscale;
  P.tk_qscale = query_scale_dev;
  P.tk_val = pv;
  P.tk_idx = pi;
  const int rbs = ceil_div(n_q, BM);
  if (knn_list(k) == 32)
    return knn_launch<MODE_TOPK32>(tm, P, rbs, sp.nsplit, n_q, k, values_dev, indices_dev, st);
  return knn_launch<MODE_TOPK>(tm, P, rbs, sp.nsplit, n_q, k, values_dev, indices_dev, st);
}

// ------------------------------------------------------------------------------------------------
// Embedding geometry (Wang & Isola's uniformity, cosine histograms, alignment) on the Gram-tile kernel: MODE_GEOM sums
// the exponentials and counts the histogram of the pairs in scope.  Two sets take their positives from an fp32
// pre-pass (gm_pos_kernel) and the tile pass masks them, so every positive is counted once.  Nothing of size
// n_a x n_b exists.
// Scratch: column scale [ncols padded to 256] fp32 | t(j) [same] int32 | tile partials [CTAs] fp64 |
//          positives' partials [pos_blocks] fp64
// ------------------------------------------------------------------------------------------------
struct GeomPlan {
  int ncols, ncols_pad, tps, nsplit, ctas, pos_blocks;
};
static bool geom_args_ok(int n_a, int n_b, int bins) {
  return (n_b == 0 ? n_a >= 2 : (n_a >= 1 && n_b >= 1)) && bins >= 0 && bins <= GEOM_BINS_MAX;
}
static GeomPlan geom_plan(int n_a, int n_b, int sms) {
  GeomPlan g;
  const bool one = n_b == 0;
  g.ncols = one ? n_a : n_b;
  g.ncols_pad = static_cast<int>(rk_cols(g.ncols));
  const int rbs = ceil_div(n_a, BM), ntiles = ceil_div(g.ncols, 2 * BN);
  // one set: the upper block triangle in chunks from the row's end, as dsoft_pair_stats; two sets: the rectangle
  const int tps = one ? std::max(4, ceil_div(ntiles, 10)) : choose_split(rbs, 1, ntiles, sms).tps;
  g.tps = std::min(tps, 1 << 16);  // a CTA's 32-bit histogram counts: 8 warps x 32 rows x 128 columns per tile
  g.nsplit = ceil_div(ntiles, g.tps);
  g.ctas = (rbs + 1) / 2 * 2 * g.nsplit;
  g.pos_blocks = one ? 0 : std::min(ceil_div(n_b, 8), 1024);
  return g;
}

extern "C" size_t dsoft_geometry_scratch_bytes(int32_t n_a, int32_t n_b, int32_t bins) {
  if (!geom_args_ok(n_a, n_b, bins)) return 0;
  int sms = 0;
  if (query_num_sms(&sms)) return 0;
  const GeomPlan g = geom_plan(n_a, n_b, sms);
  return 8 * static_cast<size_t>(g.ncols_pad) + 8 * static_cast<size_t>(g.ctas + g.pos_blocks);
}

// t(j) padded to whole tiles with -1 (mapped two sets), and the histograms zeroed
__global__ void gm_init_kernel(const int32_t* __restrict__ tmap_in, int n, int ncols_pad, int* __restrict__ tmap,
                               unsigned long long* __restrict__ hist, int nhist) {
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < max(ncols_pad, nhist); j += gridDim.x * blockDim.x) {
    if (tmap_in && j < ncols_pad) tmap[j] = j < n ? tmap_in[j] : -1;
    if (j < nhist) hist[j] = 0ull;
  }
}

// Two sets, the positives: one warp per caption j over a fixed grid (so the partials always add in the same order).
// cos = <a_t(j), b_j> b_scale[j] a_scale[t(j)] in fp32 from the bf16 operands, as rk_thr_kernel; the positive
// histogram in shared memory, flushed once per block into the 64-bit counters; (2 - 2 cos)^(alpha / 2) in fp64 into
// the block's partial.  A map entry outside [0, n_a) counts nothing.
__global__ void __launch_bounds__(256) gm_pos_kernel(const __nv_bfloat16* __restrict__ a,
                                                     const __nv_bfloat16* __restrict__ b, int k, int n_a, int n_b,
                                                     const int32_t* __restrict__ tmap, const float* __restrict__ a_scale,
                                                     const float* __restrict__ b_scale, float alpha, float lo, float hi,
                                                     float bscale, int bins, unsigned long long* __restrict__ hist,
                                                     float* __restrict__ pos_cos, double* __restrict__ part) {
  __shared__ uint32_t h[GEOM_BINS_MAX + 2];
  __shared__ double ws[8];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nh = bins + 2;
  for (int q = threadIdx.x; q < nh; q += blockDim.x) h[q] = 0u;
  __syncthreads();
  double al = 0.0;
  for (int j = blockIdx.x * 8 + warp; j < n_b; j += gridDim.x * 8) {
    const int i = tmap ? tmap[j] : j;
    if (i < 0 || i >= n_a) continue;  // warp-uniform
    const uint4* x4 = reinterpret_cast<const uint4*>(a + static_cast<size_t>(i) * k);
    const uint4* y4 = reinterpret_cast<const uint4*>(b + static_cast<size_t>(j) * k);
    float acc = 0.f;
    for (int c = lane; c < k / 8; c += 32) {
      const uint4 x = __ldg(x4 + c), y = __ldg(y4 + c);
      const __nv_bfloat162* xa = reinterpret_cast<const __nv_bfloat162*>(&x);
      const __nv_bfloat162* ya = reinterpret_cast<const __nv_bfloat162*>(&y);
#pragma unroll
      for (int hh = 0; hh < 4; ++hh) {
        const float2 xf = __bfloat1622float2(xa[hh]), yf = __bfloat1622float2(ya[hh]);
        acc = fmaf(xf.x, yf.x, acc);
        acc = fmaf(xf.y, yf.y, acc);
      }
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) {
      const float cs = (acc * (b_scale ? b_scale[j] : 1.f)) * (a_scale ? a_scale[i] : 1.f);
      if (pos_cos) pos_cos[j] = cs;
      al += pow(fmax(2.0 - 2.0 * static_cast<double>(cs), 0.0), 0.5 * static_cast<double>(alpha));
      if (bins) atomicAdd(&h[geom_bin(cs, lo, hi, bscale, bins)], 1u);
    }
  }
  if (lane == 0) ws[warp] = al;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int w = 0; w < 8; ++w) s += ws[w];
    part[blockIdx.x] = s;
  }
  if (bins)
    for (int q = threadIdx.x; q < nh; q += blockDim.x)
      if (h[q]) atomicAdd(hist + q, static_cast<unsigned long long>(h[q]));
}

// one block: sums[0] = the tile partials, sums[1] = the positives' partials, each reduced in a fixed order
__global__ void __launch_bounds__(256) gm_finalize_kernel(const double* __restrict__ tile, int ntile,
                                                          const double* __restrict__ pos, int npos,
                                                          double* __restrict__ sums) {
  __shared__ double s[2][256];
  double x = 0.0, y = 0.0;
  for (int q = threadIdx.x; q < ntile; q += 256) x += tile[q];
  for (int q = threadIdx.x; q < npos; q += 256) y += pos[q];
  s[0][threadIdx.x] = x;
  s[1][threadIdx.x] = y;
  __syncthreads();
  for (int o = 128; o; o >>= 1) {
    if (threadIdx.x < o) {
      s[0][threadIdx.x] += s[0][threadIdx.x + o];
      s[1][threadIdx.x] += s[1][threadIdx.x + o];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    sums[0] = s[0][0];
    sums[1] = s[1][0];
  }
}

extern "C" int dsoft_geometry(const void* a_dev, const void* b_dev, int32_t width, int32_t n_a, int32_t n_b,
                              const float* a_scale_dev, const float* b_scale_dev, const int32_t* text_image_dev,
                              float t, float alpha, float lo, float hi, int32_t bins, double* sums_dev,
                              unsigned long long* hist_dev, float* pos_cos_dev, void* scratch_dev, void* stream) {
  if (!a_dev || !sums_dev || !scratch_dev || (bins > 0 && !hist_dev)) return fail(DSOFT_EINVAL, "null argument");
  const bool one = n_b == 0;
  if (width <= 0 || width % 8)
    return fail(DSOFT_EINVAL, "the feature width must be a positive multiple of 8 (width=%d)", width);
  if (!geom_args_ok(n_a, n_b, bins))
    return fail(DSOFT_EINVAL, "need n_a >= 2 for one set (n_b = 0) or n_a, n_b >= 1 for two, and 0 <= bins <= %d "
                              "(n_a=%d n_b=%d bins=%d)", GEOM_BINS_MAX, n_a, n_b, bins);
  if (!(t >= 0.f && t <= 20.f)) return fail(DSOFT_EINVAL, "t must lie in [0, 20] (t=%g)", t);
  if (bins > 0 && !(std::isfinite(lo) && std::isfinite(hi) && lo < hi))
    return fail(DSOFT_EINVAL, "the histogram range needs finite lo < hi (lo=%g hi=%g)", lo, hi);
  if (one && (text_image_dev || pos_cos_dev))
    return fail(DSOFT_EINVAL, "one set (n_b = 0) has no positives: text_image and pos_cos must be NULL");
  if (!one && !(alpha > 0.f && std::isfinite(alpha))) return fail(DSOFT_EINVAL, "alpha must be > 0 (alpha=%g)", alpha);
  if (!one && !b_dev) return fail(DSOFT_EINVAL, "two sets need b_dev");
  if (!one && !text_image_dev && n_a != n_b)
    return fail(DSOFT_EINVAL, "without a caption -> image map n_a must equal n_b (%d, %d)", n_a, n_b);
  const void* bcol = b_dev ? b_dev : a_dev;
  for (const void* q : {a_dev, bcol, static_cast<const void*>(scratch_dev)})
    if (reinterpret_cast<uintptr_t>(q) % 16) return fail(DSOFT_EINVAL, "operands and scratch must be 16-byte aligned");
  int sms = 0, rc = query_num_sms(&sms);
  if (rc) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const GeomPlan g = geom_plan(n_a, n_b, sms);
  float* cscale = static_cast<float*>(scratch_dev);
  int* tmap = reinterpret_cast<int*>(cscale + g.ncols_pad);
  double* tpart = reinterpret_cast<double*>(tmap + g.ncols_pad);
  double* ppart = tpart + g.ctas;
  const int nh = bins + 2, nhist = bins ? (one ? nh : 2 * nh) : 0;
  const float bscale = bins ? static_cast<float>(static_cast<double>(bins) / (static_cast<double>(hi) - lo)) : 0.f;
  const int grid = std::min(ceil_div(std::max(g.ncols_pad, nhist), 256), 4 * sms);
  knn_scale_kernel<<<grid, 256, 0, st>>>(one ? a_scale_dev : b_scale_dev, g.ncols, g.ncols_pad, cscale);
  CUDA_TRY(cudaGetLastError());
  gm_init_kernel<<<grid, 256, 0, st>>>(one ? nullptr : text_image_dev, g.ncols, g.ncols_pad, tmap, hist_dev, nhist);
  CUDA_TRY(cudaGetLastError());
  if (!one) {
    gm_pos_kernel<<<g.pos_blocks, 256, 0, st>>>(static_cast<const __nv_bfloat16*>(a_dev),
                                                static_cast<const __nv_bfloat16*>(b_dev), width, n_a, n_b,
                                                text_image_dev, a_scale_dev, b_scale_dev, alpha, lo, hi, bscale, bins,
                                                hist_dev, pos_cos_dev, ppart);
    CUDA_TRY(cudaGetLastError());
  }
  const bool tiles = bins > 0 || t > 0.f;  // two sets without a histogram: the pre-pass is the whole result
  if (tiles) {
    TileMaps tm;
    const CUtensorMapDataType bf = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
    if ((rc = make_map(&tm.m[0], a_dev, n_a, width, static_cast<size_t>(width), bf, 64))) return rc;
    if ((rc = make_map(&tm.m[1], bcol, g.ncols, width, static_cast<size_t>(width), bf, 64))) return rc;
    tm.m[2] = tm.m[3] = tm.g[0] = tm.g[1] = tm.m[0];
    FwdParams P;
    memset(&P, 0, sizeof(P));
    P.nprod = 1;
    P.a_map[0] = 0;
    P.b_map[0] = 1;
    P.kchunks[0] = ceil_div(width, BK);
    P.bn = 2 * BN;
    P.row0 = 0;
    P.b = n_a;
    P.col0 = 0;
    P.ncols = g.ncols;
    P.ntiles = ceil_div(g.ncols, 2 * BN);
    P.tiles_per_split = g.tps;
    P.npart = 2 * g.nsplit;
    P.tri = one ? 1 : 0;  // one set: upper block triangle, pairs i < j
    P.gm_mapped = (!one && text_image_dev) ? 1 : 0;
    P.ncolvec = P.gm_mapped ? 2 : 1;
    P.colvec[0] = cscale;
    P.colvec[1] = reinterpret_cast<const float*>(tmap);
    P.gm_rscale = a_scale_dev;
    P.gm_kappa = static_cast<float>(2.0 * t * 1.4426950408889634);
    P.gm_bins = bins;
    P.gm_lo = lo;
    P.gm_hi = hi;
    P.gm_bscale = bscale;
    P.gm_hist = (bins && !one) ? hist_dev + nh : hist_dev;
    P.gm_part = tpart;
    if ((rc = set_smem(dsoft_fwd_kernel<MODE_GEOM, 2>, FWD_SMEM_BYTES))) return rc;
    if ((rc = launch_fwd_pair(dsoft_fwd_kernel<MODE_GEOM, 2>, ceil_div(n_a, BM), g.nsplit, st, tm, P))) return rc;
  }
  gm_finalize_kernel<<<1, 256, 0, st>>>(tpart, tiles ? g.ctas : 0, ppart, g.pos_blocks, sums_dev);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

// phase 0: the whole forward; of a DSOFT_SYM_W plan: 4 = operand statistics, 1 = the soft part up to the column-sum
// exchange, 3 = the CLIP part (independent of 1 and of the exchange), 2 = finalize; of a weighted plan: 5 = up to the
// weighted row statistics (row stds), 6 = median onward
static int forward_impl(const dsoft_plan_t* p, const void* gathered, const float* logit_scale,
                        const float* lambdas, void* state, void* scratch, float* lse_local,
                        float* losses, float* dbg, void* stream, int phase);

extern "C" int dsoft_forward(const dsoft_plan_t* p, const void* gathered, const float* logit_scale,
                             const float* lambdas, void* state, void* scratch, float* lse_local,
                             float* losses, float* dbg, void* stream) {
  if (p && p->sym_w)
    return fail(DSOFT_EINVAL, "this plan shares the symmetric soft tiles across ranks (DSOFT_SYM_W): call "
                              "dsoft_forward_phase 4, 1, 3 (next to the column-sum exchange), 2");
  if (p && p->weighted && p->sh.world > 1)
    return fail(DSOFT_EINVAL, "the weighted CE branch at world > 1 needs the row stds of all ranks: call "
                              "dsoft_forward_phase 5, all-gather the row-std block, then phase 6");
  return forward_impl(p, gathered, logit_scale, lambdas, state, scratch, lse_local, losses, dbg, stream, 0);
}

extern "C" int dsoft_forward_phase(const dsoft_plan_t* p, const void* gathered, const float* logit_scale,
                                   const float* lambdas, void* state, void* scratch, float* lse_local,
                                   float* losses, float* dbg, void* stream, int phase) {
  if (!p) return fail(DSOFT_EINVAL, "null argument");
  // 1..4: the symmetric soft tiles' schedule; 5 / 6: around the row-std exchange of the weighted branch
  const bool wmulti = p->weighted && p->sh.world > 1;
  if (phase < 1 || phase > 6 || (phase >= 5 && !p->weighted) || (phase <= 4 && wmulti))
    return fail(DSOFT_EINVAL, wmulti ? "a weighted plan at world > 1 takes phases 5 and 6"
                                     : (p->weighted ? "phase must be 1..6" : "phase must be 4, 1, 3 or 2"));
  return forward_impl(p, gathered, logit_scale, lambdas, state, scratch, lse_local, losses, dbg, stream, phase);
}

static int forward_impl(const dsoft_plan_t* p, const void* gathered, const float* logit_scale,
                        const float* lambdas, void* state, void* scratch, float* lse_local,
                        float* losses, float* dbg, void* stream, int phase) {
  if (!p || !gathered || !logit_scale || !lambdas || !state || !scratch || !lse_local || !losses)
    return fail(DSOFT_EINVAL, "null argument");
  if (p->siglip) return fail(DSOFT_EINVAL, "a DSOFT_F_SIGLIP plan runs through dsoft_siglip_forward");
  if (p->distill) return fail(DSOFT_EINVAL, "a DSOFT_F_DISTILL plan runs through dsoft_distill_forward");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* S = static_cast<float*>(state);
  float* X = static_cast<float*>(scratch);
  const __nv_bfloat16* g = static_cast<const __nv_bfloat16*>(gathered);
  const int b = p->sh.b;
  const int rbs = ceil_div(b, BM);
  TileMaps tm;
  int rc = make_maps(p, gathered, &tm, 64);  // 64-row boxes: each CTA of a pair stages half a column tile
  if (rc) return rc;

  // phases of a DSOFT_SYM_W plan: 4 = operand statistics, 1 = soft tile kernel + column reduction, 3 = CLIP kernels
  // (the caller's column-sum exchange runs next to them), 2 = finalize; 0 = everything.  Weighted plans: 5 = all of
  // phase 0 up to the weighted row stds, 6 = the rest of the weighted branch (after the caller's row-std all-gather)
  const bool whole = phase == 0 || phase == 5;
  const bool do_pro = whole || phase == 4, do_soft = whole || phase == 1, do_clip = whole || phase == 3;
  if (phase != 2 && phase != 6) {
  if (do_pro) {
  prep_scalars_kernel<<<1, 32, 0, st>>>(logit_scale, p->have_soft ? p->sh.teacher_temp : 0.f,
                                        p->have_text ? p->sh.text_temp : 0.f, S + p->st_scal);
  CUDA_TRY(cudaGetLastError());

  {  // inverse norms of text / student / dino rows of all ranks: one launch, grid.y = matrix
    RinvArgs ra;
    memset(&ra, 0, sizeof(ra));
    ra.ld = p->row_elems;
    ra.rows = p->B;
    ra.out_len = p->Bcol;
    ra.mat[0] = g + p->offT; ra.cols[0] = p->sh.D;  ra.out[0] = S + p->st_rinv_t; ra.rmin[0] = S + p->st_scal + SC_RMIN_T;
    ra.mat[1] = g + p->offZ; ra.cols[1] = p->Dz;    ra.out[1] = S + p->st_rinv_z; ra.rmin[1] = S + p->st_scal + SC_RMIN_Z;
    ra.mat[2] = g + p->offD; ra.cols[2] = p->sh.Dd; ra.out[2] = S + p->st_rinv_d; ra.rmin[2] = S + p->st_scal + SC_RMIN_D;
    if (p->clip_sym) {  // diagonal dot products: lower bounds of the log-sum-exps for the one-pass CLIP forward
      ra.dot_mat = g + p->offI;
      ra.dot_out = S + p->st_dbound;
    }
    rinv_kernel<<<dim3(ceil_div(p->Bcol, 8 * RINV_ROWS_PER_WARP), (p->have_soft || p->weighted) ? 3 : 1), 256, 0,
                  st>>>(ra);
    CUDA_TRY(cudaGetLastError());
  }
  }  // do_pro: scalars + norms

  if ((rc = set_smem(dsoft_fwd_kernel<MODE_CLIP, 2>, FWD_SMEM_BYTES))) return rc;
  if ((rc = set_smem(dsoft_fwd_kernel<MODE_SOFT, 2>, FWD_SMEM_BYTES))) return rc;

  // the three tile kernels are independent: fork them (largest first), join before the finalize
  Fork fk;
  if ((rc = fk.begin(p, st))) return rc;
  cudaStream_t ks = st;
  int lane = 0;
  FwdParams P;
  if (p->have_soft && do_soft) {
    memset(&P, 0, sizeof(P));
    P.nprod = p->have_text ? 3 : 2;
    P.bn = 2 * BN;
    P.a_map[0] = P.b_map[0] = 3;  // teacher: dino . dino^T       (loss.py:373)
    P.a_map[1] = P.b_map[1] = 2;  // student: Zs . Zs^T           (loss.py:372)
    P.a_map[2] = P.b_map[2] = 1;  // text:    Tn . Tn^T           (loss.py:394)
    P.kchunks[0] = ceil_div(p->sh.Dd, BK);
    P.kchunks[1] = ceil_div(p->Dz, BK);
    P.kchunks[2] = ceil_div(p->sh.D, BK);
    P.row0 = p->sh.rank * b;
    P.b = b;
    P.col0 = p->s_col0;
    P.ncols = p->s_ncols;
    P.ntiles = p->ntiles_s;
    P.tiles_per_split = p->f_soft.tps;
    P.npart = 2 * p->f_soft.nsplit;
    P.scal = S + p->st_scal;
    P.rinv[0] = S + p->st_rinv_d;
    P.rinv[1] = S + p->st_rinv_z;
    P.rinv[2] = S + p->st_rinv_t;
    P.part = X + p->sc_ps;
    if ((rc = fk.lane(lane++, &ks))) return rc;
    if (p->fwd_sym) {
      // upper block triangle only, the other half through column reductions (dsoft_fwd_kernel<MODE_SOFT_SYM16>)
      if ((rc = set_smem(dsoft_fwd_kernel<MODE_SOFT_SYM16, 2>, FWD_SMEM_BYTES))) return rc;
      P.tri = 1;
      P.tiles_per_split = p->f_sym.tps;
      P.npart = 2 * p->f_sym.nsplit;
      P.colpart = X + p->sc_colpart;
      P.cp_rows = 4 * rbs;
      P.cp_pitch = p->Bcol;
      if (p->sym_w) {  // primed columns wrapping around the global batch, short rows (plan: sym_w)
        P.wrap = p->B;
        P.rb_half = p->sw_rb_half;
        P.ntiles_a = p->sw_ncols_a / (2 * BN);
      }
      ProfScope ps(PK_FWD_SOFT, ks);
      if ((rc = launch_fwd_pair(dsoft_fwd_kernel<MODE_SOFT_SYM16, 2>, rbs, p->f_sym.nsplit, ks, tm, P))) return rc;
      // column sums by PRIMED column: [0, b) are this rank's own rows, the rest belongs to the ranks behind it
      soft_colreduce_kernel<<<dim3(p->Bcol / 32, 6), dim3(32, 16), 0, ks>>>(
          X + p->sc_colpart, 4 * rbs, p->Bcol, p->s_ncols, X + p->sc_colsum, p->sym_w ? p->sw_ncols_a : p->s_ncols,
          4 * p->sw_rb_half);
    } else {
      ProfScope ps(PK_FWD_SOFT, ks);
      if ((rc = launch_fwd_pair(dsoft_fwd_kernel<MODE_SOFT, 2>, rbs, p->f_soft.nsplit, ks, tm, P))) return rc;
    }
    CUDA_TRY(cudaGetLastError());
  }
  // image -> text (loss.py:266/272) and text -> image (loss.py:267/273)
  if (do_clip) {
  fill_clip_fwd(p, P, 0, 1, S + p->st_scal, X + p->sc_pc_it, S + p->st_diag);
  if ((rc = fk.lane(lane++, &ks))) return rc;
  if (p->clip_sym) {
    // world == 1: text -> image is the transpose; one pass with per-warp column partials (MODE_CLIP_SYM)
    if ((rc = set_smem(dsoft_fwd_kernel<MODE_CLIP_SYM, 2>, FWD_SMEM_BYTES))) return rc;
    P.colM = X + p->sc_clipM;
    P.colS = X + p->sc_clipS;
    P.cp_rows = 4 * rbs;
    P.cp_pitch = p->Bcol;
    P.dbound = S + p->st_dbound;
    ProfScope ps(PK_FWD_CLIP_IT, ks);
    P.npart = 4 * p->f_clip.nsplit;  // sixteen epilogue warps: four 64-column strips per split
    if ((rc = launch_fwd_pair(dsoft_fwd_kernel<MODE_CLIP_SYM, 2>, rbs, p->f_clip.nsplit, ks, tm, P,
                              fwd_threads(MODE_CLIP_SYM))))
      return rc;
    clip_colreduce_kernel<<<p->Bcol / 32, dim3(32, 16), 0, ks>>>(X + p->sc_clipM, X + p->sc_clipS, 4 * rbs, p->Bcol,
                                                                  p->B, X + p->sc_lse_ti);
    CUDA_TRY(cudaGetLastError());
  } else {
    {
      ProfScope ps(PK_FWD_CLIP_IT, ks);
      if ((rc = launch_fwd_pair(dsoft_fwd_kernel<MODE_CLIP, 2>, rbs, p->f_clip.nsplit, ks, tm, P))) return rc;
    }
    CUDA_TRY(cudaGetLastError());
    // same diagonal as the image -> text launch (which may run concurrently): only that one stores it
    fill_clip_fwd(p, P, 1, 0, S + p->st_scal, X + p->sc_pc_ti, nullptr);
    if ((rc = fk.lane(lane++, &ks))) return rc;
    {
      ProfScope ps(PK_FWD_CLIP_TI, ks);
      if ((rc = launch_fwd_pair(dsoft_fwd_kernel<MODE_CLIP, 2>, rbs, p->f_clip.nsplit, ks, tm, P))) return rc;
    }
    CUDA_TRY(cudaGetLastError());
  }
  }  // do_clip
  if ((rc = fk.join())) return rc;
  }  // phase != 2 && phase != 6
  if (phase == 1 || phase == 3 || phase == 4) return 0;
  if (phase == 6) return weighted_forward(p, tm, S, X, lse_local, lambdas[3], losses, dbg, st, false, true);

  FinFwdArgs fa;
  fa.b = b;
  fa.np_c = (p->clip_sym ? 4 : 2) * p->f_clip.nsplit;
  fa.np_s = 2 * (p->fwd_sym ? p->f_sym.nsplit : p->f_soft.nsplit);
  fa.have_soft = p->have_soft;
  fa.have_text = p->have_text;
  fa.pc_it = X + p->sc_pc_it;
  fa.pc_ti = X + p->sc_pc_ti;
  fa.ps = X + p->sc_ps;
  fa.colsum = p->fwd_sym ? X + p->sc_colsum : nullptr;
  fa.lse_ti = p->clip_sym ? X + p->sc_lse_ti : nullptr;
  fa.Bcol = p->Bcol;
  fa.diag = S + p->st_diag;
  fa.scal = S + p->st_scal;
  fa.lse = lse_local;
  fa.rowloss = X + p->sc_rowloss;
  fa.ticket = reinterpret_cast<int*>(S + p->st_scal + SC_TICKET_F);
  fa.lam_orig = lambdas[0];
  fa.lam_soft = lambdas[1];
  fa.text_lambda = lambdas[2];
  fa.losses = losses;
  finalize_fwd_kernel<<<ceil_div(b, 128), 128, 0, st>>>(fa);
  CUDA_TRY(cudaGetLastError());
  if (p->weighted) return weighted_forward(p, tm, S, X, lse_local, lambdas[3], losses, dbg, st, true, phase != 5);
  return 0;
}


// Gradient GEMM launch: acc[split][b][dout] = G[b][pitch] . Y16[ycol0 + ..][voff .. voff + dout)
// transposed = true (world == 1 only): acc[split][col][dout] = G^T . Y16, K runs over G's rows
// tri (world == 1, symmetrically scaled soft G of which only the upper block triangle exists): blocks left of each
// row pair's diagonal block are read transposed from the same matrix
// DSOFT_SYM_W extras of a gradient GEMM launch (all zero otherwise; see GyParams)
struct GySym {
  int ywrap = 0, rb0 = 0, out_rows = 0, pair_half = 0, kend_a = 0, rb_a = 0, klo_b = 0;
};
static int launch_gy(const dsoft_plan* p, const __half* G, int pitch, const __half* v16, int voff, int dout,
                     int ycol0, const SplitPlan& sp, float* acc, cudaStream_t st, bool transposed = false,
                     bool tri = false, const GySym* sym = nullptr) {
  CUtensorMap gmap, gmap64, vmap;
  int rc;
  // blocked G: 64 columns x (row blocks * K tiles * 128) rows, one 16 KiB box per (row block, K tile)
  const int rbs = ceil_div(p->sh.b, BM);
  const int g_rows = rbs * (pitch / BK) * BM;
  if ((rc = make_map(&gmap, G, g_rows, BK, BK, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, BM))) return rc;
  if ((rc = make_map(&gmap64, G, g_rows, BK, BK, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 64))) return rc;
  if ((rc = make_map(&vmap, v16 + voff, p->B, dout, p->v_row, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 64))) return rc;
  GyParams P;
  memset(&P, 0, sizeof(P));
  P.b = p->sh.b;
  P.dout = dout;
  P.ksteps = transposed ? rbs * 2 : pitch / BK;
  P.steps_per_split = sp.tps;
  P.nsplit = sp.nsplit;
  P.ycol0 = ycol0;
  P.g_ktiles = pitch / BK;
  P.tri = tri ? 1 : 0;
  P.acc_part = acc;
  int pairs = ceil_div(rbs, 2);
  if (sym) {
    P.ywrap = sym->ywrap;
    P.rb0 = sym->rb0;
    P.pair_half = sym->pair_half;
    P.kend_a = sym->kend_a;
    P.rb_a = sym->rb_a;
    P.klo_b = sym->klo_b;
    if (sym->out_rows) {  // transposed products for other ranks' rows: output rows = primed columns from 128 rb0 on
      P.b = sym->out_rows;
      pairs = ceil_div(sym->out_rows, 2 * BM);
    }
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(2, ceil_div(dout, GY_N), pairs * sp.nsplit);
  cfg.blockDim = dim3(NUM_THREADS);
  cfg.dynamicSmemBytes = GY_SMEM_BYTES;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (transposed) CUDA_TRY(cudaLaunchKernelEx(&cfg, dsoft_gy_kernel<true>, gmap, gmap64, vmap, P));
  else CUDA_TRY(cudaLaunchKernelEx(&cfg, dsoft_gy_kernel<false>, gmap, gmap64, vmap, P));
  return 0;
}

// DSOFT_F_GMAT backward.  Phase 1: the forward main loop again, its epilogue writing fp16 logit-gradient
// tiles; phase 2: gradient GEMMs.  Three independent lanes on forked streams:
//   soft (G kernel -> student GEMM -> text GEMM) | CLIP image rows (G -> GEMM) | CLIP text rows (G -> GEMM)
// store map of a blocked fp16 G matrix: 64 columns x (row blocks * K tiles * 128) rows, box = 64 x 32, SW128
// box_cols = 64: one K tile x 32 rows (eight epilogue warps); 32: half a K tile (MODE_CLIP_G's sixteen warps)
static int make_gstore_map(const dsoft_plan* p, CUtensorMap* map, const __half* G, int pitch, int box_cols = BK) {
  const int rbs = ceil_div(p->sh.b, BM);
  return make_map(map, G, rbs * (pitch / BK) * BM, BK, BK, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 32, box_cols);
}

static int backward_two_phase(const dsoft_plan* p, const void* gathered, float* S, float* X, const float* lse_loc,
                              const float* lsec, const __half* v16, const float* gout, const float* lambdas,
                              cudaStream_t st, bool do_soft = true, bool do_clip = true) {
  const float* colfac = S + p->st_colfac;
  const int b = p->sh.b;
  const int rbs = ceil_div(b, BM);
  int rc;
  TileMaps tm;
  if ((rc = make_maps(p, gathered, &tm, 64))) return rc;
  if ((rc = set_smem(dsoft_gy_kernel<false>, GY_SMEM_BYTES))) return rc;
  if ((rc = set_smem(dsoft_gy_kernel<true>, GY_SMEM_BYTES))) return rc;
  if ((rc = set_smem(dsoft_fwd_kernel<MODE_CLIP_G, 2>, FWD_SMEM_BYTES))) return rc;
  if ((rc = set_smem(dsoft_fwd_kernel<MODE_SOFT_G, 2>, FWD_SMEM_BYTES))) return rc;
  __half* Gci = reinterpret_cast<__half*>(X + p->sc_Gci);
  __half* Gct = reinterpret_cast<__half*>(X + p->sc_Gct);
  __half* Gs = reinterpret_cast<__half*>(X + p->sc_Gs);
  __half* Gx = reinterpret_cast<__half*>(X + p->sc_Gx);
  Fork fk;
  if ((rc = fk.begin(p, st))) return rc;
  cudaStream_t ks = st;
  int lane = 0;
  FwdParams P;
  if (p->have_soft && do_soft) {
    if ((rc = fk.lane(lane++, &ks))) return rc;
    memset(&P, 0, sizeof(P));
    P.nprod = p->have_text ? 3 : 2;
    P.bn = 2 * BN;
    P.a_map[0] = P.b_map[0] = 3;
    P.a_map[1] = P.b_map[1] = 2;
    P.a_map[2] = P.b_map[2] = 1;
    P.kchunks[0] = ceil_div(p->sh.Dd, BK);
    P.kchunks[1] = ceil_div(p->Dz, BK);
    P.kchunks[2] = ceil_div(p->sh.D, BK);
    P.row0 = p->sh.rank * b;
    P.b = b;
    P.col0 = p->s_col0;
    P.ncols = p->s_ncols;
    P.ntiles = p->ntiles_s;
    P.tiles_per_split = p->f_soft.tps;
    P.npart = 2 * p->f_soft.nsplit;
    P.scal = S + p->st_scal;
    P.rinv[0] = S + p->st_rinv_d;
    P.rinv[1] = S + p->st_rinv_z;
    P.rinv[2] = S + p->st_rinv_t;
    for (int k = 0; k < 3; ++k) {
      P.lse_row[k] = lse_loc + (2 + k) * b;
      // column factors incl. the gather_with_grad == False case (zeros): lse_relayout_kernel.  Local soft scope
      // keeps the column-side terms: both sides of Zs Zs^T / Tn Tn^T are live local tensors (loss.py:358-397)
      P.colfac[k] = colfac + static_cast<size_t>(2 + k) * p->Bcol;
    }
    P.fast_t = p->fast_t;
    P.gout[0] = Gs;
    P.gout[1] = Gx;
    P.g_pitch = p->pitch_s;
    if ((rc = make_gstore_map(p, &tm.g[0], Gs, p->pitch_s))) return rc;
    if ((rc = make_gstore_map(p, &tm.g[1], p->have_text ? Gx : Gs, p->pitch_s))) return rc;
    // world == 1: the student / text / teacher matrices are symmetric, so G is: only the tiles from each row
    // pair's diagonal block onwards are computed (half the work), in column chunks small enough to balance the
    // triangular load; the gradient GEMMs read the other half through the transposed blocks
    // world > 1 with DSOFT_SYM_W: the same in primed column coordinates for the tiles this rank owns
    const bool tri = p->clip_tr || p->sym_w;
    int nsplit = p->f_soft.nsplit;
    if (tri) {
      P.tri = 1;
      P.tiles_per_split = std::max(4, ceil_div(p->ntiles_s, 10));
      nsplit = ceil_div(p->ntiles_s, P.tiles_per_split);
    }
    GySym loc, rem;  // local rows' products / transposed products for the rows of the ranks behind this one
    SplitPlan one;
    if (p->sym_w) {
      P.wrap = p->B;
      P.rb_half = p->sw_rb_half;
      P.ntiles_a = p->sw_ncols_a / (2 * BN);
      loc.ywrap = p->B;
      loc.pair_half = p->sw_rb_half / 2;
      loc.kend_a = p->sw_ncols_a / BK;
      rem.rb0 = b / BM;
      rem.out_rows = p->s_ncols - b;
      if (p->sw_rb_half) {  // the contested block's columns only exist in the rows from b/2 on
        rem.rb_a = p->sw_ncols_a / BM;
        rem.klo_b = (b / 2) / BK;
      }
      one.nsplit = 1;
      one.tps = rbs * 2;
    }
    {
      ProfScope ps(PK_BWD_GSOFT, ks);
      if ((rc = launch_fwd_pair(dsoft_fwd_kernel<MODE_SOFT_G, 2>, rbs, nsplit, ks, tm, P))) return rc;
    }
    {
      ProfScope ps(PK_BWD_STU, ks);
      if ((rc = launch_gy(p, Gs, p->pitch_s, v16, p->v_offZn, p->Dz, p->s_col0, p->g_stu, X + p->sc_acc3, ks, false,
                          tri, p->sym_w ? &loc : nullptr)))
        return rc;
      if (p->sym_w && (rc = launch_gy(p, Gs, p->pitch_s, v16, p->v_offZn, p->Dz, p->sh.rank * b, one,
                                      X + p->sc_accR3, ks, true, false, &rem)))
        return rc;
    }
    if (p->have_text) {
      ProfScope ps(PK_BWD_TXT, ks);
      if ((rc = launch_gy(p, Gx, p->pitch_s, v16, p->v_offTn, p->sh.D, p->s_col0, p->g_txt, X + p->sc_acc4, ks, false,
                          tri, p->sym_w ? &loc : nullptr)))
        return rc;
      if (p->sym_w && (rc = launch_gy(p, Gx, p->pitch_s, v16, p->v_offTn, p->sh.D, p->sh.rank * b, one,
                                      X + p->sc_accR4, ks, true, false, &rem)))
        return rc;
    }
  }
  if (!do_clip) return fk.join();
  if (p->weighted) {
    // world == 1: ONE logit-gradient matrix carries  g_c * classic CE + g_w * weighted CE  of both directions
    // (loss.py:416-471 backward); the two gradient GEMMs below are the classic ones.  World > 1: one matrix per
    // direction, like the CLIP launches below: the row side is this rank's rows of direction d, the column side the
    // other direction's rows of all ranks (statistics relayouted from lse_all by wce_relayout_kernel)
    if ((rc = set_smem(dsoft_fwd_kernel<MODE_WCE_G, 2>, FWD_SMEM_BYTES))) return rc;
    const size_t r0 = static_cast<size_t>(p->sh.rank) * b;
    for (int d = 0; d < (p->clip_tr ? 1 : 2); ++d) {
      if ((rc = fk.lane(lane++, &ks))) return rc;
      fill_wce(p, P, d, S, nullptr);
      const float* wr = S + p->st_wstat + static_cast<size_t>(d) * 4 * p->Bcol;      // row-side direction
      const float* wc = S + p->st_wstat + static_cast<size_t>(1 - d) * 4 * p->Bcol;  // column-side direction
      P.wrow[0] = lse_loc + d * b;
      P.wrow[1] = wr + WS_C * p->Bcol + r0;
      P.wrow[2] = wr + WS_LSET * p->Bcol + r0;
      P.wrow[3] = wr + WS_A * p->Bcol + r0;
      P.ncolvec = 5;
      P.colvec[1] = lsec + static_cast<size_t>(1 - d) * p->Bcol;  // lse of the other direction, by column
      P.colvec[2] = wc + WS_LSET * p->Bcol;                       // (only read when that direction is modulated)
      P.colvec[3] = wc + WS_C * p->Bcol;
      P.colvec[4] = wc + WS_A * p->Bcol;
      P.wsym = d == 0 ? p->wsym : 1;
      P.wrow_plain = d == 1 && !p->wsym;
      P.wsplit = !p->clip_tr;
      P.row_only = p->row_only;
      P.wgout = gout;
      P.wlam[0] = lambdas[0];
      P.wlam[1] = lambdas[3];
      P.gout[0] = d == 0 ? Gci : Gct;
      P.g_pitch = p->pitch_c;
      P.npart = 2 * p->f_wce.nsplit;
      P.ds_part = X + (d == 0 ? p->sc_ds1 : p->sc_ds2);
      if ((rc = make_gstore_map(p, &tm.g[0], P.gout[0], p->pitch_c))) return rc;
      tm.g[1] = tm.g[0];
      {
        ProfScope ps(PK_BWD_GCLIP, ks);
        if ((rc = launch_fwd_pair(dsoft_fwd_kernel<MODE_WCE_G, 2>, rbs, p->f_wce.nsplit, ks, tm, P))) return rc;
      }
      {
        ProfScope ps(d == 0 ? PK_BWD_CLIP_I : PK_BWD_CLIP_T, ks);
        if ((rc = launch_gy(p, P.gout[0], p->pitch_c, v16, d == 0 ? p->v_offT : p->v_offI, p->sh.D, 0, p->g_clip,
                            X + (d == 0 ? p->sc_acc1 : p->sc_acc2), ks)))
          return rc;
      }
    }
  }
  for (int d = 0; d < (p->weighted ? 0 : (p->clip_tr ? 1 : 2)); ++d) {  // d = 0: image rows (dI = G . T), d = 1: text rows
    if ((rc = fk.lane(lane++, &ks))) return rc;
    fill_clip_fwd(p, P, d == 0 ? 0 : 1, d == 0 ? 1 : 0, S + p->st_scal, nullptr, nullptr);
    P.lse_row[0] = lse_loc + d * b;
    P.lse_col[0] = lsec + static_cast<size_t>(1 - d) * p->Bcol;
    P.colfac[0] = colfac + static_cast<size_t>(d) * p->Bcol;
    P.gout[0] = d == 0 ? Gci : Gct;
    P.g_pitch = p->pitch_c;
    if ((rc = make_gstore_map(p, &tm.g[0], P.gout[0], p->pitch_c))) return rc;
    tm.g[1] = tm.g[0];
    P.row_only = p->row_only;
    P.ds_part = X + (d == 0 ? p->sc_ds1 : p->sc_ds2);
    P.ds_both = p->clip_tr;
    {
      ProfScope ps(PK_BWD_GCLIP, ks);
      if ((rc = launch_fwd_pair(dsoft_fwd_kernel<MODE_CLIP_G, 2>, rbs, p->f_clip.nsplit, ks, tm, P))) return rc;
    }
    {
      ProfScope ps(d == 0 ? PK_BWD_CLIP_I : PK_BWD_CLIP_T, ks);
      if ((rc = launch_gy(p, P.gout[0], p->pitch_c, v16, d == 0 ? p->v_offT : p->v_offI, p->sh.D, 0, p->g_clip,
                          X + (d == 0 ? p->sc_acc1 : p->sc_acc2), ks)))
        return rc;
    }
  }
  if (p->clip_tr) {
    // world == 1: G_text[j][i] = p_ti[j,i] + p_it[i,j] = G_image[i][j]: dT = G_image^T . I, no second G matrix;
    // the text rows' d(logit_scale) partials were folded into the image rows' (ds_both)
    CUDA_TRY(cudaMemsetAsync(X + p->sc_ds2, 0,
                             sizeof(float) * 2 * std::max(p->f_clip.nsplit, p->weighted ? p->f_wce.nsplit : 0) * b, ks));
    ProfScope ps(PK_BWD_CLIP_T, ks);
    if ((rc = launch_gy(p, Gci, p->pitch_c, v16, p->v_offI, p->sh.D, 0, p->g_clip_t, X + p->sc_acc2, ks, true)))
      return rc;
  }
  return fk.join();
}

// phase 0: the whole backward; of a DSOFT_SYM_W plan: 4 = statistics relayout + fp16 operands, 1 = the soft part up to
// the exchange of the transposed products (logit-gradient kernel + gradient GEMMs), 3 = the CLIP part (independent of
// 1 and of the exchange), 2 = the finalize kernel
static int backward_impl(const dsoft_plan_t* p, const void* gathered, const void* state, void* scratch,
                         const float* lse_all, const float* gout, const float* lambdas, float* d_image,
                         float* d_text, float* d_student, float* d_scale, void* stream, int phase);

extern "C" int dsoft_backward(const dsoft_plan_t* p, const void* gathered, const void* state, void* scratch,
                              const float* lse_all, const float* gout, const float* lambdas, float* d_image,
                              float* d_text, float* d_student, float* d_scale, void* stream) {
  if (p && p->sym_w)
    return fail(DSOFT_EINVAL, "this plan shares the symmetric soft tiles across ranks (DSOFT_SYM_W): call "
                              "dsoft_backward_phase 4, 1, 3 (next to the exchange of the transposed products), 2");
  return backward_impl(p, gathered, state, scratch, lse_all, gout, lambdas, d_image, d_text, d_student, d_scale,
                       stream, 0);
}

extern "C" int dsoft_backward_phase(const dsoft_plan_t* p, const void* gathered, const void* state, void* scratch,
                                    const float* lse_all, const float* gout, const float* lambdas, float* d_image,
                                    float* d_text, float* d_student, float* d_scale, void* stream, int phase) {
  if (phase < 1 || phase > 4) return fail(DSOFT_EINVAL, "phase must be 4, 1, 3 or 2");
  return backward_impl(p, gathered, state, scratch, lse_all, gout, lambdas, d_image, d_text, d_student, d_scale,
                       stream, phase);
}

// Layout of the two exchanges of a DSOFT_SYM_W plan, in floats / rows (out[12]):
//  [0] 1 if the plan uses them            [1] b                          [2] Bcol (pitch of the column sums)
//  [3] offset of the column sums [6][Bcol] in the FORWARD scratch (primed columns; [0, b) = this rank's rows)
//  [4] primed columns this rank computes (s_ncols): the blocks 1 .. belong to ranks rank+1, rank+2, ...
//  [5] offset of the student products for other ranks' rows [s_ncols - b][Dz] in the BACKWARD scratch, [6] Dz
//  [7] the same for the text term [s_ncols - b][D], [8] D (0: no text term)
//  [9] offset of this rank's own student partial sums (split 0: [b][Dz]), [10] of the text ones ([b][D])
//  [11] number of K splits of those partial sums (received products are added to split 0)
// Rows of the per-row statistics lse_local / lse_all carry (5, more for a weighted plan at world > 1)
extern "C" int dsoft_plan_lse_rows(const dsoft_plan_t* p) { return p ? p->lse_rows : 0; }

// Row-std block of a weighted plan at world > 1 (out[3], in floats): [0] offset in `state`, [1] floats per rank
// (rank r's block starts at [0] + r * [1]), [2] directions per row.  All zero for every other plan.
extern "C" int dsoft_plan_wsigma_info(const dsoft_plan_t* p, long long* out, int n) {
  if (!p || !out || n < 3) return fail(DSOFT_EINVAL, "need 3 slots");
  for (int k = 0; k < n; ++k) out[k] = 0;
  if (p->weighted && p->sh.world > 1) {
    out[0] = static_cast<long long>(p->st_wsig);
    out[1] = static_cast<long long>(p->wnd) * p->sh.b;
    out[2] = p->wnd;
  }
  return 0;
}

extern "C" int dsoft_plan_symw_info(const dsoft_plan_t* p, long long* out, int n) {
  if (!p || !out || n < 12) return fail(DSOFT_EINVAL, "need 12 slots");
  for (int k = 0; k < n; ++k) out[k] = 0;
  out[0] = p->sym_w;
  out[1] = p->sh.b;
  out[2] = p->Bcol;
  out[3] = static_cast<long long>(p->sc_colsum);
  out[4] = p->s_ncols;
  out[5] = static_cast<long long>(p->sc_accR3);
  out[6] = p->Dz;
  out[7] = static_cast<long long>(p->sc_accR4);
  out[8] = p->have_text ? p->sh.D : 0;
  out[9] = static_cast<long long>(p->sc_acc3);
  out[10] = static_cast<long long>(p->sc_acc4);
  out[11] = p->gmat ? p->g_stu.nsplit : 1;
  return 0;
}

static int backward_impl(const dsoft_plan_t* p, const void* gathered, const void* state, void* scratch,
                         const float* lse_all, const float* gout, const float* lambdas, float* d_image,
                         float* d_text, float* d_student, float* d_scale, void* stream, int phase) {
  if (!p || !gathered || !state || !scratch || !lse_all || !gout || !lambdas || !d_image || !d_text || !d_scale)
    return fail(DSOFT_EINVAL, "null argument");
  if (p->siglip) return fail(DSOFT_EINVAL, "a DSOFT_F_SIGLIP plan runs through dsoft_siglip_backward");
  if (p->distill) return fail(DSOFT_EINVAL, "a DSOFT_F_DISTILL plan runs through dsoft_distill_backward");
  if (p->have_proj && !d_student) return fail(DSOFT_EINVAL, "d_student is null but the plan has Dp > 0");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // state is logically const for the caller; the relayouted LSE columns live in it
  float* S = const_cast<float*>(static_cast<const float*>(state));
  float* X = static_cast<float*>(scratch);
  const int b = p->sh.b;
  const int rbs = ceil_div(b, BM);
  TileMaps tm;
  int rc = make_maps(p, gathered, &tm);
  if (rc) return rc;

  float* lsec = S + p->st_lsecols;
  const float* lse_loc = lse_all + static_cast<size_t>(p->sh.rank) * p->lse_rows * b;
  // phases of a DSOFT_SYM_W plan: 1 = statistics relayout + fp16 operands + soft lane (G kernel, GEMMs incl. the
  // transposed products), 3 = CLIP lanes (the caller's exchange of the transposed products runs next to them),
  // 2 = finalize; 0 = everything
  if (phase != 2) {
  __half* v16 = reinterpret_cast<__half*>(X + p->sc_v16);
  if (phase == 0 || phase == 4) {
  lse_stats_kernel<<<LSE_NB, 256, 0, st>>>(lse_all, p->sh.world, b, p->lse_rows, S + p->st_lsestat);
  CUDA_TRY(cudaGetLastError());
  lse_relayout_kernel<<<ceil_div(5 * p->Bcol, 1024), 256, 0, st>>>(
      lse_all, p->sh.world, b, p->lse_rows, p->Bcol, S + p->st_scal, S + p->st_lsestat, p->fast_t, p->row_only,
      p->row_only && !p->soft_local, lsec, S + p->st_colfac);
  CUDA_TRY(cudaGetLastError());
  if (p->weighted && p->sh.world > 1) {
    wce_relayout_kernel<<<ceil_div(3 * p->wnd * p->Bcol, 1024), 256, 0, st>>>(lse_all, p->sh.world, b, p->lse_rows,
                                                                             p->Bcol, p->wnd, S + p->st_wstat);
    CUDA_TRY(cudaGetLastError());
  }
  if (p->weighted) {
    wce_gscale_kernel<<<1, 1, 0, st>>>(gout, lambdas[0], lambdas[3], p->wsym, S + p->st_scal);
    CUDA_TRY(cudaGetLastError());
  }
  make_v16_kernel<<<ceil_div(p->B, 8), 256, 0, st>>>(
      static_cast<const __nv_bfloat16*>(gathered), p->row_elems, p->B, p->sh.D, p->Dz, p->offI, p->offT,
      p->offZ, p->have_soft, p->have_text, S + p->st_rinv_z, S + p->st_rinv_t, v16, p->v_row, p->v_offT, p->v_offI,
      p->v_offZn, p->v_offTn);
  CUDA_TRY(cudaGetLastError());
  }  // prologue
  CUtensorMap vmap;
  auto vmap_for = [&](int voff, int cols) {
    return make_map(&vmap, v16 + voff, p->B, cols, p->v_row, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 64);
  };

  if (p->gmat) {
    if ((rc = backward_two_phase(p, gathered, S, X, lse_loc, lsec, v16, gout, lambdas, st, phase == 0 || phase == 1,
                                 phase == 0 || phase == 3)))
      return rc;
  } else {
  if ((rc = set_smem(dsoft_bwd_kernel<MODE_CLIP>, BWD_SMEM_BYTES))) return rc;
  if ((rc = set_smem(dsoft_bwd_kernel<MODE_SOFT>, BWD_SMEM_BYTES))) return rc;
  if (p->weighted && (rc = set_smem(dsoft_bwd_kernel<MODE_WCE_X>, BWD_SMEM_BYTES))) return rc;

  BwdParams P;
  auto base = [&](const SplitPlan& sp, int col0, int ncols, int ntiles) {
    memset(&P, 0, sizeof(P));
    P.row0 = p->sh.rank * b;
    P.b = b;
    P.col0 = col0;
    P.ncols = ncols;
    P.ntiles = ntiles;
    P.tiles_per_split = sp.tps;
    P.nsplit = sp.nsplit;
    P.row_only = p->row_only;
    P.scal = S + p->st_scal;
  };
  // the four tile kernels are independent: fork them (largest first), join before the finalize
  Fork fk;
  if ((rc = fk.begin(p, st))) return rc;
  cudaStream_t ks = st;
  int lane = 0;
  if (p->have_soft) {
    base(p->b_stu, p->s_col0, p->s_ncols, p->ntiles_s128);
    P.nprod = 2;
    P.a_map[0] = P.b_map[0] = 3;
    P.kchunks[0] = ceil_div(p->sh.Dd, BK);
    P.a_map[1] = P.b_map[1] = 2;
    P.kchunks[1] = ceil_div(p->Dz, BK);
    P.dout = p->Dz;
    P.row_only = p->row_only && !p->soft_local;  // local scope: live tensors on both sides (loss.py:358-397)
    if ((rc = vmap_for(p->v_offZn, p->Dz))) return rc;
    P.tau_idx = SC_ITS_L2;
    P.lse_t_row = lse_loc + 2 * b;
    P.lse_t_col = lsec + 2 * p->Bcol;
    P.lse_y_row = lse_loc + 3 * b;
    P.lse_y_col = lsec + 3 * p->Bcol;
    P.rinv_d = S + p->st_rinv_d;
    P.rinv_y = S + p->st_rinv_z;
    P.acc_part = X + p->sc_acc3;
    if ((rc = fk.lane(lane++, &ks))) return rc;
    {
      ProfScope ps(PK_BWD_STU, ks);
      if ((rc = launch_bwd(dsoft_bwd_kernel<MODE_SOFT>, p->nch_stu, rbs, p->b_stu.nsplit, ks, tm, vmap, P))) return rc;
    }
    CUDA_TRY(cudaGetLastError());
    if (p->have_text) {
      base(p->b_txt, p->s_col0, p->s_ncols, p->ntiles_s128);
      P.nprod = 2;
      P.a_map[0] = P.b_map[0] = 3;
      P.kchunks[0] = ceil_div(p->sh.Dd, BK);
      P.a_map[1] = P.b_map[1] = 1;
      P.kchunks[1] = ceil_div(p->sh.D, BK);
      P.dout = p->sh.D;
      P.row_only = p->row_only && !p->soft_local;
      if ((rc = vmap_for(p->v_offTn, p->sh.D))) return rc;
      P.tau_idx = SC_ITX_L2;
      P.lse_t_row = lse_loc + 2 * b;
      P.lse_t_col = lsec + 2 * p->Bcol;
      P.lse_y_row = lse_loc + 4 * b;
      P.lse_y_col = lsec + 4 * p->Bcol;
      P.rinv_d = S + p->st_rinv_d;
      P.rinv_y = S + p->st_rinv_t;
      P.acc_part = X + p->sc_acc4;
      if ((rc = fk.lane(lane++, &ks))) return rc;
      {
        ProfScope ps(PK_BWD_TXT, ks);
        if ((rc = launch_bwd(dsoft_bwd_kernel<MODE_SOFT>, p->nch_txt, rbs, p->b_txt.nsplit, ks, tm, vmap, P)))
          return rc;
      }
      CUDA_TRY(cudaGetLastError());
    }
  }

  // weighted CE branch: the CLIP launches below run MODE_WCE_X instead, whose G carries g_c * classic CE + g_w *
  // weighted CE of the pair's two directions (MODE_WCE_G's entry), from a CLIP and a DINO tile per column tile.  Row
  // side = this rank's rows of direction d, column side = the other direction's per-row statistics by global column
  // (world 1: st_wstat by global row is that view; world > 1: wce_relayout_kernel above).  There is no transposed
  // GEMM here, so each launch takes its own direction's d(logit_scale) row term (wsplit) at every world size.
  auto set_wce = [&](int d) {
    const size_t r0 = static_cast<size_t>(p->sh.rank) * b;
    const float* wr = S + p->st_wstat + static_cast<size_t>(d) * 4 * p->Bcol;      // row-side direction
    const float* wc = S + p->st_wstat + static_cast<size_t>(1 - d) * 4 * p->Bcol;  // column-side direction
    P.nprod = 2;
    P.a_map[1] = P.b_map[1] = 3;  // DINO cosine
    P.kchunks[1] = ceil_div(p->sh.Dd, BK);
    P.rinv_d = S + p->st_rinv_d;
    P.wrow[0] = lse_loc + d * b;
    P.wrow[1] = wr + WS_C * p->Bcol + r0;
    P.wrow[2] = wr + WS_LSET * p->Bcol + r0;
    P.wrow[3] = wr + WS_A * p->Bcol + r0;
    P.wcol[0] = lsec + static_cast<size_t>(1 - d) * p->Bcol;  // lse of the other direction, by column
    P.wcol[1] = wc + WS_LSET * p->Bcol;                       // (only read when that direction is modulated)
    P.wcol[2] = wc + WS_C * p->Bcol;
    P.wcol[3] = wc + WS_A * p->Bcol;
    P.wdir = d;
    P.wsym = d == 0 ? p->wsym : 1;
    P.wrow_plain = d == 1 && !p->wsym;
    P.wsplit = 1;
    P.wcc = p->sh.c_clip;
    P.wlam[0] = lambdas[0];
    P.wlam[1] = lambdas[3];
    P.wgout = gout;
  };
  auto clip_kernel = p->weighted ? dsoft_bwd_kernel<MODE_WCE_X> : dsoft_bwd_kernel<MODE_CLIP>;
  // ---- CLIP, image rows: d image = s/(2b) sum_j (p_it[a,j] + p_ti[j,a]) T_j - ...
  base(p->b_clip, 0, p->B, p->ntiles_g);
  P.nprod = 1;
  P.a_map[0] = 0;
  P.b_map[0] = 1;
  P.kchunks[0] = ceil_div(p->sh.D, BK);
  P.dout = p->sh.D;
  P.want_ds = 1;
  if ((rc = vmap_for(p->v_offT, p->sh.D))) return rc;
  P.lse_row = lse_loc + 0 * b;
  P.lse_col = lsec + 1 * p->Bcol;
  P.acc_part = X + p->sc_acc1;
  P.ds_part = X + p->sc_ds1;
  if (p->weighted) set_wce(0);
  if ((rc = fk.lane(lane++, &ks))) return rc;
  {
    ProfScope ps(PK_BWD_CLIP_I, ks);
    if ((rc = launch_bwd(clip_kernel, p->nch_clip, rbs, p->b_clip.nsplit, ks, tm, vmap, P))) return rc;
  }
  CUDA_TRY(cudaGetLastError());
  // ---- CLIP, text rows
  P.a_map[0] = 1;
  P.b_map[0] = 0;
  if ((rc = vmap_for(p->v_offI, p->sh.D))) return rc;
  P.lse_row = lse_loc + 1 * b;
  P.lse_col = lsec + 0 * p->Bcol;
  P.acc_part = X + p->sc_acc2;
  P.ds_part = X + p->sc_ds2;
  if (p->weighted) set_wce(1);
  if ((rc = fk.lane(lane++, &ks))) return rc;
  {
    ProfScope ps(PK_BWD_CLIP_T, ks);
    if ((rc = launch_bwd(clip_kernel, p->nch_clip, rbs, p->b_clip.nsplit, ks, tm, vmap, P))) return rc;
  }
  CUDA_TRY(cudaGetLastError());

  if ((rc = fk.join())) return rc;
  }  // !p->gmat
  }  // phase != 2
  if (phase != 0 && phase != 2) return 0;

  FinBwdArgs fa;
  memset(&fa, 0, sizeof(fa));
  fa.b = b;
  fa.D = p->sh.D;
  fa.Dz = p->Dz;
  fa.row0 = p->sh.rank * b;
  fa.row_elems = p->row_elems;
  fa.offI = p->offI;
  fa.offT = p->offT;
  fa.offZ = p->offZ;
  fa.have_soft = p->have_soft;
  fa.have_text = p->have_text;
  fa.have_proj = p->have_proj;
  fa.row_only = p->row_only;
  fa.sym_scaled = p->gmat && (p->clip_tr || p->sym_w);
  fa.weighted = p->weighted;
  fa.wsym = p->wsym;
  fa.wstat = S + p->st_wstat;
  fa.Bcol = p->Bcol;
  fa.lam_w = lambdas[3];
  fa.ns_c = p->gmat ? p->g_clip.nsplit : p->b_clip.nsplit;
  fa.ns_c2 = (p->gmat && p->clip_tr) ? p->g_clip_t.nsplit : fa.ns_c;
  fa.nds = p->gmat ? 2 * (p->weighted ? p->f_wce.nsplit : p->f_clip.nsplit)
                   : 2 * p->b_clip.nsplit * chunk_cluster(p->nch_clip);
  fa.ns_s = p->gmat ? p->g_stu.nsplit : p->b_stu.nsplit;
  fa.ns_x = p->gmat ? p->g_txt.nsplit : p->b_txt.nsplit;
  fa.gathered = static_cast<const __nv_bfloat16*>(gathered);
  fa.acc1 = X + p->sc_acc1;
  fa.acc2 = X + p->sc_acc2;
  fa.acc3 = X + p->sc_acc3;
  fa.acc4 = X + p->sc_acc4;
  fa.ds1 = X + p->sc_ds1;
  fa.ds2 = X + p->sc_ds2;
  fa.diag = S + p->st_diag;
  fa.scal = S + p->st_scal;
  fa.rinv_z = S + p->st_rinv_z;
  fa.rinv_t = S + p->st_rinv_t;
  fa.gout = gout;
  fa.lse_loc = lse_loc;
  fa.d_image = d_image;
  fa.d_text = d_text;
  fa.d_student = d_student;
  fa.dsrow = X + p->sc_dsrow;
  fa.lam_orig = lambdas[0];
  fa.lam_soft = lambdas[1];
  fa.text_lambda = lambdas[2];
  fa.ticket = reinterpret_cast<int*>(S + p->st_scal + SC_TICKET_B);
  fa.d_scale = d_scale;
  {
    const int width = std::max(p->sh.D, p->Dz);
    if (width <= 1024) {  // one warp per row, 8 rows per block; lanes own ceil(width / 128) float4 groups
      const dim3 grid(std::min(ceil_div(b, 8), p->num_sms * 16));
      const int nd = p->sh.D <= 512 ? 4 : (p->sh.D <= 768 ? 6 : 8);
      const int nz = p->Dz <= 512 ? 4 : (p->Dz <= 768 ? 6 : 8);
#define DSOFT_FIN(ND, NZ)                                                                         \
  if (nd == ND && nz == NZ) {                                                                     \
    if (p->have_proj) finalize_bwd_warp_kernel<ND, NZ, true><<<grid, 256, 0, st>>>(fa);           \
    else finalize_bwd_warp_kernel<ND, NZ, false><<<grid, 256, 0, st>>>(fa);                       \
  }
      DSOFT_FIN(4, 4) DSOFT_FIN(4, 6) DSOFT_FIN(4, 8) DSOFT_FIN(6, 4) DSOFT_FIN(6, 6) DSOFT_FIN(6, 8)
      DSOFT_FIN(8, 4) DSOFT_FIN(8, 6) DSOFT_FIN(8, 8)
#undef DSOFT_FIN
    } else {
      finalize_bwd_kernel<4><<<dim3(std::min(b, p->num_sms * 16)), 128, 0, st>>>(fa);
    }
  }
  CUDA_TRY(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------
// SigLIP sigmoid loss (open_clip SigLipLoss) on the Gram-tile kernels: dsoft_fwd_kernel<MODE_SIGLIP> computes every
// pair's loss term and logit gradient from the pair's own logit, so the forward writes the fp16 G tile as it goes and
// the backward is the two gradient GEMMs.  Rank r owns image rows [r b, (r+1) b) against all B captions; at world > 1
// the text rows' G (T_local . I_all^T, same pairs transposed) is computed by a second launch in the backward, so the
// forward-to-backward interval holds one [b x B] G, and a forward without gradient needs none.
// ------------------------------------------------------------------------------------------------
__global__ void siglip_prep_kernel(const float* __restrict__ logit_scale, const float* __restrict__ logit_bias,
                                   float* __restrict__ scal) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  scal[SC_SCALE] = *logit_scale;
  scal[SC_SIG_BIAS] = logit_bias ? *logit_bias : 0.f;
  scal[SC_SIG_GX] = scal[SC_SIG_G] = 0.f;
  scal[SC_TICKET_S] = 0.f;  // all-zero bits == integer 0
}

struct SgFinFwdArgs {
  int b, npart;
  const float* part;  // [3][npart][b]: loss, G x, G
  float* blk;         // [3][gridDim.x]
  float* scal;
  float* loss;
  int* ticket;
};

// loss = sum / b; the sums of G x and G stay in the state for the backward.  Rows -> per-block fp32 sums in a fixed
// order, then the last block adds the blocks in fp64 (deterministic, as finalize_fwd_kernel).
__global__ void __launch_bounds__(128) siglip_finalize_fwd_kernel(SgFinFwdArgs a) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  float r[3] = {0.f, 0.f, 0.f};
  if (i < a.b)
    for (int k = 0; k < 3; ++k)
      for (int s = 0; s < a.npart; ++s) r[k] += a.part[(static_cast<size_t>(k) * a.npart + s) * a.b + i];
  __shared__ float shp[3][4];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    float v = r[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) shp[k][threadIdx.x >> 5] = v;
  }
  __syncthreads();
  if (threadIdx.x < 3)
    a.blk[threadIdx.x * gridDim.x + blockIdx.x] =
        (shp[threadIdx.x][0] + shp[threadIdx.x][1]) + (shp[threadIdx.x][2] + shp[threadIdx.x][3]);
  if (last_block_done(a.ticket)) {
    __shared__ double sums[3];
    block_reduce_rows(a.blk, gridDim.x, 3, sums);
    if (threadIdx.x == 0) {
      a.loss[0] = static_cast<float>(sums[0] / a.b);
      a.scal[SC_SIG_GX] = static_cast<float>(sums[1]);
      a.scal[SC_SIG_G] = static_cast<float>(sums[2]);
    }
  }
}

struct SgFinBwdArgs {
  int b, D, ns1, ns2;
  const float* acc1;  // [ns1][b][D]  sum_j (G 2^k)_ij T_j   (image rows)
  const float* acc2;  // [ns2][b][D]  sum_i (G 2^k)_ij I_i   (text rows)
  const float* scal;
  const float* gout;
  float* d_image;
  float* d_text;
  float* d_scale;
  float* d_bias;
};

// d image / d text = gout s / (b 2^k) x the summed split partials; d s = gout / b sum G x, d beta = gout / b sum G
__global__ void __launch_bounds__(256) siglip_finalize_bwd_kernel(SgFinBwdArgs a) {
  const float g = a.gout[0] / static_cast<float>(a.b);
  const float coef = g * a.scal[SC_SCALE] * (1.f / static_cast<float>(1 << SIG_GK));
  const int q = a.D / 4;
  const size_t n = static_cast<size_t>(a.b) * q;
  for (size_t idx = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; idx < n;
       idx += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int i = static_cast<int>(idx / q);
    const int f = static_cast<int>(idx % q) * 4;
    float4 u = sum_splits4(a.acc1, a.ns1, a.b, a.D, i, f);
    *reinterpret_cast<float4*>(a.d_image + static_cast<size_t>(i) * a.D + f) =
        make_float4(u.x * coef, u.y * coef, u.z * coef, u.w * coef);
    u = sum_splits4(a.acc2, a.ns2, a.b, a.D, i, f);
    *reinterpret_cast<float4*>(a.d_text + static_cast<size_t>(i) * a.D + f) =
        make_float4(u.x * coef, u.y * coef, u.z * coef, u.w * coef);
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    a.d_scale[0] = g * a.scal[SC_SIG_GX];
    if (a.d_bias) a.d_bias[0] = g * a.scal[SC_SIG_G];
  }
}

extern "C" size_t dsoft_siglip_g_bytes(const dsoft_plan_t* p) {
  if (!p || !p->siglip) return 0;
  return static_cast<size_t>(ceil_div(p->sh.b, BM)) * BM * p->pitch_c * 2;
}

extern "C" int dsoft_siglip_forward(const dsoft_plan_t* p, const void* gathered, const float* logit_scale,
                                    const float* logit_bias, void* state, void* scratch, void* g, float* loss,
                                    void* stream) {
  if (!p || !gathered || !logit_scale || !state || !scratch || !loss) return fail(DSOFT_EINVAL, "null argument");
  if (!p->siglip) return fail(DSOFT_EINVAL, "dsoft_siglip_forward needs a DSOFT_F_SIGLIP plan");
  if (reinterpret_cast<uintptr_t>(g) % 16) return fail(DSOFT_EINVAL, "g must be 16-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* S = static_cast<float*>(state);
  float* X = static_cast<float*>(scratch);
  const int b = p->sh.b;
  TileMaps tm;
  int rc = make_maps(p, gathered, &tm, 64);
  if (rc) return rc;
  siglip_prep_kernel<<<1, 32, 0, st>>>(logit_scale, logit_bias, S + p->st_scal);
  CUDA_TRY(cudaGetLastError());
  FwdParams P;
  fill_clip_fwd(p, P, 0, 1, S + p->st_scal, X + p->sg_part, nullptr);
  P.gout[0] = static_cast<__half*>(g);
  P.g_pitch = p->pitch_c;
  if (g && (rc = make_gstore_map(p, &tm.g[0], static_cast<const __half*>(g), p->pitch_c))) return rc;
  tm.g[1] = tm.g[0];
  if ((rc = set_smem(dsoft_fwd_kernel<MODE_SIGLIP, 2>, FWD_SMEM_BYTES))) return rc;
  {
    ProfScope ps(PK_FWD_CLIP_IT, st);
    if ((rc = launch_fwd_pair(dsoft_fwd_kernel<MODE_SIGLIP, 2>, ceil_div(b, BM), p->f_clip.nsplit, st, tm, P)))
      return rc;
  }
  SgFinFwdArgs fa;
  fa.b = b;
  fa.npart = P.npart;
  fa.part = X + p->sg_part;
  fa.blk = X + p->sg_blk;
  fa.scal = S + p->st_scal;
  fa.loss = loss;
  fa.ticket = reinterpret_cast<int*>(S + p->st_scal + SC_TICKET_S);
  siglip_finalize_fwd_kernel<<<ceil_div(b, 128), 128, 0, st>>>(fa);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

extern "C" int dsoft_siglip_backward(const dsoft_plan_t* p, const void* gathered, const void* state, void* scratch,
                                     const void* g, const float* gout, float* d_image, float* d_text, float* d_scale,
                                     float* d_bias, void* stream) {
  if (!p || !gathered || !state || !scratch || !g || !gout || !d_image || !d_text || !d_scale)
    return fail(DSOFT_EINVAL, "null argument");
  if (!p->siglip) return fail(DSOFT_EINVAL, "dsoft_siglip_backward needs a DSOFT_F_SIGLIP plan");
  if (reinterpret_cast<uintptr_t>(g) % 16 || reinterpret_cast<uintptr_t>(d_image) % 16 ||
      reinterpret_cast<uintptr_t>(d_text) % 16)
    return fail(DSOFT_EINVAL, "g, d_image and d_text must be 16-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* S = const_cast<float*>(static_cast<const float*>(state));
  float* X = static_cast<float*>(scratch);
  const int b = p->sh.b;
  const __half* G = static_cast<const __half*>(g);
  __half* v16 = reinterpret_cast<__half*>(X + p->sc_v16);
  TileMaps tm;
  int rc = make_maps(p, gathered, &tm, 64);
  if (rc) return rc;
  make_v16_kernel<<<ceil_div(p->B, 8), 256, 0, st>>>(
      static_cast<const __nv_bfloat16*>(gathered), p->row_elems, p->B, p->sh.D, p->Dz, p->offI, p->offT, p->offZ, 0, 0,
      nullptr, nullptr, v16, p->v_row, p->v_offT, p->v_offI, 0, 0);
  CUDA_TRY(cudaGetLastError());
  if ((rc = set_smem(dsoft_gy_kernel<false>, GY_SMEM_BYTES))) return rc;
  if ((rc = set_smem(dsoft_gy_kernel<true>, GY_SMEM_BYTES))) return rc;
  const __half* Gt = G;  // world == 1: the text rows' G is the transpose of the image rows' one
  if (!p->clip_tr) {
    __half* Gw = reinterpret_cast<__half*>(X + p->sg_Gt);
    FwdParams P;
    fill_clip_fwd(p, P, 1, 0, S + p->st_scal, nullptr, nullptr);
    P.gout[0] = Gw;
    P.g_pitch = p->pitch_c;
    if ((rc = make_gstore_map(p, &tm.g[0], Gw, p->pitch_c))) return rc;
    tm.g[1] = tm.g[0];
    if ((rc = set_smem(dsoft_fwd_kernel<MODE_SIGLIP, 2>, FWD_SMEM_BYTES))) return rc;
    ProfScope ps(PK_BWD_GCLIP, st);
    if ((rc = launch_fwd_pair(dsoft_fwd_kernel<MODE_SIGLIP, 2>, ceil_div(b, BM), p->f_clip.nsplit, st, tm, P)))
      return rc;
    Gt = Gw;
  }
  {
    ProfScope ps(PK_BWD_CLIP_I, st);
    if ((rc = launch_gy(p, G, p->pitch_c, v16, p->v_offT, p->sh.D, 0, p->g_clip, X + p->sc_acc1, st))) return rc;
  }
  {
    ProfScope ps(PK_BWD_CLIP_T, st);
    if ((rc = launch_gy(p, Gt, p->pitch_c, v16, p->v_offI, p->sh.D, 0, p->clip_tr ? p->g_clip_t : p->g_clip,
                        X + p->sc_acc2, st, p->clip_tr)))
      return rc;
  }
  SgFinBwdArgs fa;
  fa.b = b;
  fa.D = p->sh.D;
  fa.ns1 = p->g_clip.nsplit;
  fa.ns2 = p->clip_tr ? p->g_clip_t.nsplit : p->g_clip.nsplit;
  fa.acc1 = X + p->sc_acc1;
  fa.acc2 = X + p->sc_acc2;
  fa.scal = S + p->st_scal;
  fa.gout = gout;
  fa.d_image = d_image;
  fa.d_text = d_text;
  fa.d_scale = d_scale;
  fa.d_bias = d_bias;
  const size_t work = static_cast<size_t>(b) * (p->sh.D / 4);
  siglip_finalize_bwd_kernel<<<static_cast<int>(std::min<size_t>((work + 255) / 256, p->num_sms * 8)), 256, 0, st>>>(fa);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------
// DistillClipLoss (open_clip) on the Gram-tile kernels.  x = s I T^T (student), t = s_t I_t T_t^T (teacher); p / q
// their soft-maxes over rows (image -> text) or columns (text -> image):
//   contrastive = 1/2 [CE_row(x, diag) + CE_col(x, diag)],  distill = 1/2 [CE_row(x, q_row) + CE_col(x, q_col)]
//   dL/dx_ij = 1/(2b) [(g_c + g_d)(p_r + p_c) - g_d (q_r + q_c) - 2 g_c delta_ij]
// Forward: dsoft_fwd_kernel<MODE_DIST_FWD> once per direction (its rows against all B columns), then a finalize that
// merges the split partials into the per-row log-sum-exps (the [4][b] statistics the backward's column side needs)
// and reduces the losses and the d(logit_scale) sums in fp64.  Backward: dsoft_fwd_kernel<MODE_DIST_G> writes the
// fp16 G of one direction's rows (world 1: one matrix serves both directions, dT = G^T I), the gradient GEMMs, and a
// finalize that applies the diagonal entries in fp32 and the s / (2b) factors.
// ------------------------------------------------------------------------------------------------
__global__ void dist_prep_kernel(const float* __restrict__ logit_scale, const float* __restrict__ dist_scale,
                                 float* __restrict__ scal) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const float L2E = 1.4426950408889634f;
  const float s = *logit_scale;
  scal[SC_SCALE] = s;
  scal[SC_SCALE_L2] = s * L2E;
  scal[SC_DST_TSCALE_L2] = *dist_scale * L2E;
  scal[SC_DST_SPD] = scal[SC_DST_SPQ] = 0.f;
  scal[SC_TICKET_DST] = 0.f;  // all-zero bits == integer 0
}

static void fill_dist(const dsoft_plan* p, FwdParams& P, int dir, float* S) {
  memset(&P, 0, sizeof(P));
  P.nprod = 2;
  P.bn = 2 * BN;
  P.a_map[0] = dir == 0 ? 0 : 1;  // student: image rows x text columns / text rows x image columns
  P.b_map[0] = dir == 0 ? 1 : 0;
  P.a_map[1] = dir == 0 ? 2 : 3;  // teacher: the same pairs of the teacher blocks
  P.b_map[1] = dir == 0 ? 3 : 2;
  P.kchunks[0] = ceil_div(p->sh.D, BK);
  P.kchunks[1] = ceil_div(p->sh.Dd, BK);
  P.row0 = p->sh.rank * p->sh.b;
  P.b = p->sh.b;
  P.col0 = 0;
  P.ncols = p->B;
  P.ntiles = ceil_div(p->B, 2 * BN);
  P.tiles_per_split = p->f_wce.tps;
  P.npart = 2 * p->f_wce.nsplit;
  P.scal = S + p->st_scal;
  P.wdir = dir;
}

struct DlFinFwdArgs {
  int b, npart;
  const float* part;  // [2][6][npart][b]: student m, sum, sum (x-m); teacher m_t, sum, sum (x-m) weighted by teacher
  const float* diag;  // [2][2][b] raw diagonal dot products (direction, student / teacher)
  float* stats;       // [4][b] out: student / teacher lse (log2) of the image rows, then of the text rows
  float* blk;         // [4][gridDim.x]
  float* scal;
  float* losses;      // [2]: contrastive, distill
  int* ticket;
};

// One thread per (direction, local row): merge the split partials, write the row's two log-sum-exps, and sum
//   contrastive: lse - x_ii,  distill: lse - sum q x,  sum p x - x_ii,  sum p x - sum q x   (natural units)
// per block in a fixed order; the last block adds the blocks in fp64 (deterministic, as finalize_fwd_kernel).
__global__ void __launch_bounds__(128) dist_finalize_fwd_kernel(DlFinFwdArgs a) {
  const float LN2 = 0.6931471805599453f;
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  float v[4] = {0.f, 0.f, 0.f, 0.f};
  if (r < 2 * a.b) {
    const int dir = r >= a.b, i = r - dir * a.b;
    const size_t st = static_cast<size_t>(a.npart) * a.b;
    const float* pp = a.part + dir * 6 * st + i;
    float M = M_FLOOR, Mt = M_FLOOR;
    for (int s = 0; s < a.npart; ++s) {
      M = fmaxf(M, pp[0 * st + s * a.b]);
      Mt = fmaxf(Mt, pp[3 * st + s * a.b]);
    }
    float S = 0.f, Ps = 0.f, St = 0.f, Q = 0.f;
    for (int s = 0; s < a.npart; ++s) {
      const size_t o = static_cast<size_t>(s) * a.b;
      const float dm = pp[0 * st + o] - M;
      const float f = exp2f(dm), ft = exp2f(pp[3 * st + o] - Mt);
      S = fmaf(pp[1 * st + o], f, S);
      Ps = fmaf(f, fmaf(dm, pp[1 * st + o], pp[2 * st + o]), Ps);
      St = fmaf(pp[4 * st + o], ft, St);
      Q = fmaf(ft, fmaf(dm, pp[4 * st + o], pp[5 * st + o]), Q);
    }
    const float l2s = log2f(S);
    a.stats[(2 * dir + 0) * a.b + i] = M + l2s;
    a.stats[(2 * dir + 1) * a.b + i] = Mt + log2f(St);
    const float d2 = a.diag[(2 * dir) * a.b + i] * a.scal[SC_SCALE_L2];  // as the tile kernel scales it
    const float px = Ps / S, qx = Q / St;  // sum p (x - M), sum q (x - M), log2 units
    v[0] = LN2 * ((M - d2) + l2s);
    v[1] = LN2 * (l2s - qx);
    v[2] = LN2 * (px + (M - d2));
    v[3] = LN2 * (px - qx);
  }
  __shared__ float shp[4][4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    float x = v[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    if ((threadIdx.x & 31) == 0) shp[k][threadIdx.x >> 5] = x;
  }
  __syncthreads();
  if (threadIdx.x < 4)
    a.blk[threadIdx.x * gridDim.x + blockIdx.x] =
        (shp[threadIdx.x][0] + shp[threadIdx.x][1]) + (shp[threadIdx.x][2] + shp[threadIdx.x][3]);
  if (last_block_done(a.ticket)) {
    __shared__ double sums[4];
    block_reduce_rows(a.blk, gridDim.x, 4, sums);
    if (threadIdx.x == 0) {
      a.losses[0] = static_cast<float>(sums[0] * 0.5 / a.b);
      a.losses[1] = static_cast<float>(sums[1] * 0.5 / a.b);
      a.scal[SC_DST_SPD] = static_cast<float>(sums[2]);
      a.scal[SC_DST_SPQ] = static_cast<float>(sums[3]);
    }
  }
}

// Backward scalars: gk = 2^(14 - max(0, e)) with |g_c| + |g_d| < 2^e, so that |G gk| < 2^15 (|G| <= 2 (|g_c| + |g_d|))
// and probabilities down to 2^-28 stay normal fp16 numbers; and the column side's statistics by global column,
// [4][Bcol] from the all-gathered [W][4][b] (zero past B).
__global__ void __launch_bounds__(256) dist_relayout_kernel(const float* __restrict__ stats_all, int W, int b, int Bcol,
                                                            const float* __restrict__ gout, float* __restrict__ scal,
                                                            float* __restrict__ col) {
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    const float gc = gout[0], gd = gout[1];
    int e = 0;
    frexpf(fabsf(gc) + fabsf(gd), &e);
    const float gk = ldexpf(1.f, 14 - max(e, 0));
    scal[SC_DST_GK] = gk;
    scal[SC_DST_GC] = gc * gk;
    scal[SC_DST_GD] = gd * gk;
  }
  if (!col) return;
  const int B = W * b;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < 4 * Bcol; idx += gridDim.x * blockDim.x) {
    const int k = idx / Bcol, g = idx - k * Bcol;
    float v = 0.f;
    if (g < B) {
      const int w = g / b;
      v = stats_all[(static_cast<size_t>(w) * 4 + k) * b + (g - w * b)];
    }
    col[idx] = v;
  }
}

struct DlFinBwdArgs {
  int b, D, row0, row_elems, offI, offT, ns1, ns2, row_only;
  const __nv_bfloat16* gathered;
  const float* acc1;   // [ns1][b][D]  sum_j (G gk)_ij T_j   (image rows)
  const float* acc2;   // [ns2][b][D]  sum_i (G gk)_ij I_i   (text rows)
  const float* stats;  // [4][b] this rank's row statistics (log2 lse: image student / teacher, text student / teacher)
  const float* diag;   // [2][2][b] raw diagonal dot products
  const float* scal;
  const float* gout;   // [2] g_c, g_d
  float* d_image;
  float* d_text;
  float* d_scale;
};

// one term of the diagonal entry, in fp32: g_c (p - 1) + g_d (p - q) with p = 2^(x - lse), q = 2^(t - lse_t)
__device__ __forceinline__ float dist_diag_term(float gc, float gd, float x2, float t2, float lse, float lset) {
  const float LN2 = 0.6931471805599453f;
  const float pm1 = expm1f(LN2 * (x2 - lse)), qm1 = expm1f(LN2 * (t2 - lset));
  return fmaf(gc, pm1, gd * (pm1 - qm1));
}

// One warp per local row: d image = s / (2b) (sum of the split partials / gk + dg_I T_i), d text likewise with I_i;
// dg = the pair (i, i)'s entry of dL/dx (2b), row side plus (unless row_only) column side.  d s from the forward's
// sums: (g_c sum (p x - x_ii) + g_d sum (p x - q x)) / (2 b s).
__global__ void __launch_bounds__(256) dist_finalize_bwd_kernel(DlFinBwdArgs a) {
  const float gc = a.gout[0], gd = a.gout[1];
  const float s = a.scal[SC_SCALE], s2 = a.scal[SC_SCALE_L2], st2 = a.scal[SC_DST_TSCALE_L2];
  const float coef = s * 0.5f / static_cast<float>(a.b);
  const float igk = 1.f / a.scal[SC_DST_GK];
  const int lane = threadIdx.x & 31;
  for (int i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); i < a.b; i += gridDim.x * (blockDim.x >> 5)) {
    const float* S = a.stats;
    const float xI = a.diag[0 * a.b + i] * s2, tI = a.diag[1 * a.b + i] * st2;  // image row i, column i
    const float xT = a.diag[2 * a.b + i] * s2, tT = a.diag[3 * a.b + i] * st2;  // text row i, column i
    float dgI = dist_diag_term(gc, gd, xI, tI, S[0 * a.b + i], S[1 * a.b + i]);
    float dgT = dist_diag_term(gc, gd, xT, tT, S[2 * a.b + i], S[3 * a.b + i]);
    if (!a.row_only) {
      dgI += dist_diag_term(gc, gd, xI, tI, S[2 * a.b + i], S[3 * a.b + i]);
      dgT += dist_diag_term(gc, gd, xT, tT, S[0 * a.b + i], S[1 * a.b + i]);
    }
    const __nv_bfloat16* row = a.gathered + static_cast<size_t>(a.row0 + i) * a.row_elems;
    for (int f = lane * 4; f < a.D; f += 128) {
      const float4 ti = load_bf16x4(row + a.offT + f), ii = load_bf16x4(row + a.offI + f);
      float4 u = sum_splits4(a.acc1, a.ns1, a.b, a.D, i, f);
      *reinterpret_cast<float4*>(a.d_image + static_cast<size_t>(i) * a.D + f) =
          make_float4(coef * fmaf(u.x, igk, dgI * ti.x), coef * fmaf(u.y, igk, dgI * ti.y),
                      coef * fmaf(u.z, igk, dgI * ti.z), coef * fmaf(u.w, igk, dgI * ti.w));
      u = sum_splits4(a.acc2, a.ns2, a.b, a.D, i, f);
      *reinterpret_cast<float4*>(a.d_text + static_cast<size_t>(i) * a.D + f) =
          make_float4(coef * fmaf(u.x, igk, dgT * ii.x), coef * fmaf(u.y, igk, dgT * ii.y),
                      coef * fmaf(u.z, igk, dgT * ii.z), coef * fmaf(u.w, igk, dgT * ii.w));
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0)
    a.d_scale[0] = (gc * a.scal[SC_DST_SPD] + gd * a.scal[SC_DST_SPQ]) * 0.5f / (static_cast<float>(a.b) * s);
}

extern "C" size_t dsoft_distill_g_bytes(const dsoft_plan_t* p) {
  if (!p || !p->distill) return 0;
  return static_cast<size_t>(ceil_div(p->sh.b, BM)) * BM * p->pitch_c * 2;
}

extern "C" int dsoft_distill_forward(const dsoft_plan_t* p, const void* gathered, const float* logit_scale,
                                     const float* dist_logit_scale, void* state, void* scratch, float* stats,
                                     float* losses, void* stream) {
  if (!p || !gathered || !logit_scale || !dist_logit_scale || !state || !scratch || !stats || !losses)
    return fail(DSOFT_EINVAL, "null argument");
  if (!p->distill) return fail(DSOFT_EINVAL, "dsoft_distill_forward needs a DSOFT_F_DISTILL plan");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* S = static_cast<float*>(state);
  float* X = static_cast<float*>(scratch);
  const int b = p->sh.b, rbs = ceil_div(b, BM);
  const size_t dpart = static_cast<size_t>(6) * 2 * p->f_wce.nsplit * b;
  TileMaps tm;
  int rc = make_maps(p, gathered, &tm, 64);
  if (rc) return rc;
  dist_prep_kernel<<<1, 32, 0, st>>>(logit_scale, dist_logit_scale, S + p->st_scal);
  CUDA_TRY(cudaGetLastError());
  if ((rc = set_smem(dsoft_fwd_kernel<MODE_DIST_FWD, 2>, FWD_SMEM_BYTES))) return rc;
  for (int d = 0; d < 2; ++d) {
    FwdParams P;
    fill_dist(p, P, d, S);
    P.part = X + p->dl_part + d * dpart;
    P.diag = S + p->st_ddiag + static_cast<size_t>(d) * 2 * b;
    ProfScope ps(d == 0 ? PK_FWD_CLIP_IT : PK_FWD_CLIP_TI, st);
    if ((rc = launch_fwd_pair(dsoft_fwd_kernel<MODE_DIST_FWD, 2>, rbs, p->f_wce.nsplit, st, tm, P))) return rc;
  }
  DlFinFwdArgs fa;
  fa.b = b;
  fa.npart = 2 * p->f_wce.nsplit;
  fa.part = X + p->dl_part;
  fa.diag = S + p->st_ddiag;
  fa.stats = stats;
  fa.blk = X + p->dl_blk;
  fa.scal = S + p->st_scal;
  fa.losses = losses;
  fa.ticket = reinterpret_cast<int*>(S + p->st_scal + SC_TICKET_DST);
  dist_finalize_fwd_kernel<<<ceil_div(2 * b, 128), 128, 0, st>>>(fa);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

extern "C" int dsoft_distill_backward(const dsoft_plan_t* p, const void* gathered, const void* state, void* scratch,
                                      const float* stats_all, void* g, const float* gout, float* d_image,
                                      float* d_text, float* d_scale, void* stream) {
  if (!p || !gathered || !state || !scratch || !stats_all || !g || !gout || !d_image || !d_text || !d_scale)
    return fail(DSOFT_EINVAL, "null argument");
  if (!p->distill) return fail(DSOFT_EINVAL, "dsoft_distill_backward needs a DSOFT_F_DISTILL plan");
  if (reinterpret_cast<uintptr_t>(g) % 16 || reinterpret_cast<uintptr_t>(d_image) % 16 ||
      reinterpret_cast<uintptr_t>(d_text) % 16)
    return fail(DSOFT_EINVAL, "g, d_image and d_text must be 16-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* S = const_cast<float*>(static_cast<const float*>(state));  // the backward's scalars live in the scalar block
  float* X = static_cast<float*>(scratch);
  const int b = p->sh.b, rbs = ceil_div(b, BM);
  // row_only: the caller passes this rank's [4][b] only, and the column side is not read
  const float* stats_loc = p->row_only ? stats_all : stats_all + static_cast<size_t>(p->sh.rank) * 4 * b;
  float* col = p->row_only ? nullptr : X + p->dl_col;
  __half* G = static_cast<__half*>(g);
  __half* v16 = reinterpret_cast<__half*>(X + p->sc_v16);
  TileMaps tm;
  int rc = make_maps(p, gathered, &tm, 64);
  if (rc) return rc;
  dist_relayout_kernel<<<col ? std::min(ceil_div(4 * p->Bcol, 256), p->num_sms * 4) : 1, 256, 0, st>>>(
      stats_all, p->sh.world, b, p->Bcol, gout, S + p->st_scal, col);
  CUDA_TRY(cudaGetLastError());
  make_v16_kernel<<<ceil_div(p->B, 8), 256, 0, st>>>(
      static_cast<const __nv_bfloat16*>(gathered), p->row_elems, p->B, p->sh.D, p->Dz, p->offI, p->offT, p->offZ, 0, 0,
      nullptr, nullptr, v16, p->v_row, p->v_offT, p->v_offI, 0, 0);
  CUDA_TRY(cudaGetLastError());
  if ((rc = set_smem(dsoft_gy_kernel<false>, GY_SMEM_BYTES))) return rc;
  if ((rc = set_smem(dsoft_gy_kernel<true>, GY_SMEM_BYTES))) return rc;
  if ((rc = set_smem(dsoft_fwd_kernel<MODE_DIST_G, 2>, FWD_SMEM_BYTES))) return rc;
  if ((rc = make_gstore_map(p, &tm.g[0], G, p->pitch_c))) return rc;
  tm.g[1] = tm.g[0];
  // d = 0: image rows (dI = G . T; world 1 also dT = G^T . I), d = 1 (world > 1): text rows into the same buffer
  for (int d = 0; d < (p->clip_tr ? 1 : 2); ++d) {
    FwdParams P;
    fill_dist(p, P, d, S);
    P.wrow[0] = stats_loc + static_cast<size_t>(2 * d) * b;
    P.wrow[1] = stats_loc + static_cast<size_t>(2 * d + 1) * b;
    P.ncolvec = col ? 2 : 0;
    if (col) {
      P.colvec[0] = col + static_cast<size_t>(2 * (1 - d)) * p->Bcol;
      P.colvec[1] = col + static_cast<size_t>(2 * (1 - d) + 1) * p->Bcol;
    }
    P.row_only = p->row_only;
    P.gout[0] = G;
    P.g_pitch = p->pitch_c;
    {
      ProfScope ps(PK_BWD_GCLIP, st);
      if ((rc = launch_fwd_pair(dsoft_fwd_kernel<MODE_DIST_G, 2>, rbs, p->f_wce.nsplit, st, tm, P))) return rc;
    }
    if (d == 0) {
      ProfScope ps(PK_BWD_CLIP_I, st);
      if ((rc = launch_gy(p, G, p->pitch_c, v16, p->v_offT, p->sh.D, 0, p->g_clip, X + p->sc_acc1, st))) return rc;
    }
    if (p->clip_tr || d == 1) {
      ProfScope ps(PK_BWD_CLIP_T, st);
      if ((rc = launch_gy(p, G, p->pitch_c, v16, p->v_offI, p->sh.D, 0, p->clip_tr ? p->g_clip_t : p->g_clip,
                          X + p->sc_acc2, st, p->clip_tr)))
        return rc;
    }
  }
  DlFinBwdArgs fa;
  fa.b = b;
  fa.D = p->sh.D;
  fa.row0 = p->sh.rank * b;
  fa.row_elems = p->row_elems;
  fa.offI = p->offI;
  fa.offT = p->offT;
  fa.ns1 = p->g_clip.nsplit;
  fa.ns2 = p->clip_tr ? p->g_clip_t.nsplit : p->g_clip.nsplit;
  fa.row_only = p->row_only;
  fa.gathered = static_cast<const __nv_bfloat16*>(gathered);
  fa.acc1 = X + p->sc_acc1;
  fa.acc2 = X + p->sc_acc2;
  fa.stats = stats_loc;
  fa.diag = S + p->st_ddiag;
  fa.scal = S + p->st_scal;
  fa.gout = gout;
  fa.d_image = d_image;
  fa.d_text = d_text;
  fa.d_scale = d_scale;
  dist_finalize_bwd_kernel<<<std::min(ceil_div(b, 8), p->num_sms * 8), 256, 0, st>>>(fa);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------
// bring-up self tests (exercise exactly the TMA / tcgen05 / TMEM plumbing of the loss kernels)
// ------------------------------------------------------------------------------------------------
extern "C" int dsoft_selftest_gemm(const void* a, const void* bmat, float* c, int M, int N, int K,
                                   void* stream) {
  if (!a || !bmat || !c || M <= 0 || N <= 0 || K <= 0 || K % 8)
    return fail(DSOFT_EINVAL, "bad selftest arguments");
  int sms = 0;
  int rc = query_num_sms(&sms);
  if (rc) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  TileMaps tm;
  if ((rc = make_map(&tm.m[0], a, M, K, K, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 64))) return rc;
  if ((rc = make_map(&tm.m[1], bmat, N, K, K, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 64))) return rc;
  tm.m[2] = tm.m[0];
  tm.m[3] = tm.m[1];
  if ((rc = set_smem(dsoft_fwd_kernel<MODE_RAW, 2>, FWD_SMEM_BYTES))) return rc;
  FwdParams P;
  memset(&P, 0, sizeof(P));
  P.nprod = 1;
  P.a_map[0] = 0;
  P.b_map[0] = 1;
  P.kchunks[0] = ceil_div(K, BK);
  // exercise all four operand-staging modes of the forward kernel (resident / streamed row operand,
  // 128- / 256-column tiles) across the test shapes
  P.bn = (K % 128 == 0) ? 2 * BN : BN;
  P.resident = (P.kchunks[0] <= 8 && (M / BM) % 2 == 0) ? 1 : 0;
  P.row0 = 0;
  P.b = M;
  P.col0 = 0;
  P.ncols = N;
  P.ntiles = ceil_div(N, P.bn);
  const int nsplit = std::min(P.ntiles, 3);
  P.tiles_per_split = ceil_div(P.ntiles, nsplit);
  P.npart = 0;
  P.part = c;
  if ((rc = launch_fwd_pair(dsoft_fwd_kernel<MODE_RAW, 2>, ceil_div(M, BM), ceil_div(P.ntiles, P.tiles_per_split), st,
                            tm, P)))
    return rc;
  return 0;
}

// out[M][F] (fp32) = fp16(A . B^T) . V   with A [M][K], B [N][K] bf16 and V [N][F] fp16: the backward data
// path (tile -> fp16 G in swizzled smem -> second tcgen05 GEMM with an MN-major operand) without any soft-max.
extern "C" int dsoft_selftest_chain(const void* a, const void* bmat, const void* vmat, float* out, int M,
                                    int N, int K, int F, void* stream) {
  if (!a || !bmat || !vmat || !out || M <= 0 || N <= 0 || K <= 0 || K % 8 || F <= 0 || F % 8)
    return fail(DSOFT_EINVAL, "bad selftest arguments");
  int sms = 0;
  int rc = query_num_sms(&sms);
  if (rc) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  TileMaps tm;
  if ((rc = make_map(&tm.m[0], a, M, K, K))) return rc;
  if ((rc = make_map(&tm.m[1], bmat, N, K, K))) return rc;
  tm.m[2] = tm.m[0];
  tm.m[3] = tm.m[0];
  CUtensorMap vmap;
  if ((rc = make_map(&vmap, vmat, N, F, F, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 64))) return rc;
  if ((rc = set_smem(dsoft_bwd_kernel<MODE_RAW>, BWD_SMEM_BYTES))) return rc;
  BwdParams P;
  memset(&P, 0, sizeof(P));
  P.nprod = 1;
  P.a_map[0] = 0;
  P.b_map[0] = 1;
  P.kchunks[0] = ceil_div(K, BK);
  P.dout = F;
  P.row0 = 0;
  P.b = M;
  P.col0 = 0;
  P.ncols = N;
  P.ntiles = ceil_div(N, BN);
  P.tiles_per_split = P.ntiles;  // single split: `out` is the only partial
  P.nsplit = 1;
  P.acc_part = out;
  if ((rc = launch_bwd(dsoft_bwd_kernel<MODE_RAW>, ceil_div(F, CHUNK_F), ceil_div(M, BM), 1, st, tm, vmap, P)))
    return rc;
  return 0;
}
