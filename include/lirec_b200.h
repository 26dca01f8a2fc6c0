/*
 * lirec_b200.h — C ABI of liblirec_b200.so (sm_100a only).
 *
 * This is the drop-in boundary for the LIReC hot path: the forward/backward of
 * reference mlp/model.py as driven by mlp/train.py and mlp/test.py.  The
 * reference has no native code and no FFI; every entry point below replaces a
 * group of ATen call sites of the reference, cited per function as
 * `<file>:<lines>` relative to the reference tree.  The Python side
 * (lirec_b200/_ext.py) binds these with ctypes; INTEGRATION.md shows the stub.
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / ATen types;
 *   - every pointer is a DEVICE pointer unless the name ends in `_host`;
 *   - the caller owns every buffer; the library never allocates device memory
 *     and keeps no pointer after a call returns;
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*), the
 *     library never synchronises;
 *   - return value 0 = OK, negative = error; lirec_last_error() gives the text
 *     (thread-local).  There is no CPU fallback: on a device that is not
 *     sm_100 every compute entry point fails with LIREC_ERR_ARCH.
 */
#ifndef LIREC_B200_H_
#define LIREC_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LIREC_ABI_VERSION 3

enum lirec_status {
  LIREC_OK = 0,
  LIREC_ERR_ARG = -1,     /* bad shape / alignment / null pointer            */
  LIREC_ERR_ARCH = -2,    /* device is not sm_100                            */
  LIREC_ERR_CUDA = -3,    /* a CUDA runtime / driver call failed             */
  LIREC_ERR_LIMIT = -4    /* too many problems / passes / tensor maps        */
};

/* ---- library ---------------------------------------------------------- */
int lirec_abi_version(void);
const char* lirec_last_error(void);
/* 0 if `device` can run the kernels (compute capability 10.x), else LIREC_ERR_ARCH */
int lirec_device_check(int device);

/* ---- dropout stream ----------------------------------------------------
 * Counter-based mask shared by every kernel that applies or re-derives a
 * dropout mask (reference: nn.Dropout at mlp/model.py:52,62,88,353).  keep(r,c)
 * is a pure function of (seed, stream_id, row r, column c); the oracle mirrors
 * it (oracle/dropout.py) so train-mode parity can be checked with masks on.  */
typedef struct lirec_dropout {
  float p;             /* drop probability; 0 disables                       */
  uint32_t seed;       /* per-step seed                                      */
  uint32_t stream_id;  /* which dropout site                                 */
  int32_t col_off;     /* added to the column before hashing                 */
} lirec_dropout;

/* keep(row, col) evaluated on the HOST with the kernels' code (test aid, no GPU needed). */
int lirec_dropout_keep_host(uint32_t seed, uint32_t stream_id, uint32_t row, uint32_t col, float p);

/* ---- grouped tcgen05 GEMM ---------------------------------------------
 * D[m,n] = epilogue( alpha * sum_pass sum_k A_pass[m,k] * B_pass[n,k] )
 * bf16 operands, fp32 accumulation in TMEM.  Replaces nn.Linear forward
 * (cuBLAS sgemm, mlp/model.py:281-294,307-322,333,336,352) and the autograd
 * mm/addmm pairs of its backward (mlp/train.py:62).
 *
 * An operand is a 2-D bf16 view (ptr, rows, cols, ld).  K-major use: rows
 * index M (or N), cols index K.  MN-major use (mn_major=1): rows index K, cols
 * index M (or N) — this is how dgrad reads W[out,in] and wgrad reads dY / X
 * without a transposed copy.  A pass is one K-segment; several passes
 * accumulate into the same tile (hi/lo split operands, concatenated inputs). */
#define LIREC_GEMM_MAX_PASSES 4
#define LIREC_GEMM_MAX_PROBLEMS 32
#define LIREC_GEMM_MAX_MAPS 64

typedef struct lirec_operand {
  const void* ptr;  /* bf16, 16-byte aligned                                 */
  int64_t rows, cols;
  int64_t ld;       /* elements between rows; ld*2 must be a multiple of 16  */
} lirec_operand;

typedef struct lirec_gemm_pass {
  lirec_operand a, b;
  int32_t a_mn_off, a_k_off;  /* element offsets inside the view             */
  int32_t b_mn_off, b_k_off;
  int32_t k_len;              /* reduction length of this pass (elements)    */
} lirec_gemm_pass;

enum lirec_act { LIREC_ACT_NONE = 0, LIREC_ACT_RELU = 1, LIREC_ACT_TANH = 2 };
enum lirec_post {
  LIREC_POST_NONE = 0,
  LIREC_POST_DROPOUT = 1, /* v *= keep(m,n) / (1-p)                          */
  LIREC_POST_DRELU = 2,   /* v *= post_scale * [aux_hi(m,n) > 0]             */
  LIREC_POST_DTANH = 3,   /* v *= keep(m,n)/(1-p) * (1 - ((aux_hi+aux_lo)*(1-p))^2) */
  LIREC_POST_SIGN_MASK = 4 /* v unchanged; SIDE OUTPUT: bit (n & 31) of ((uint32_t*)aux)[m*aux_ld + (n >> 5)] =
                            * [v > 0] — the ReLU gate of a forward layer as 1 bit per element, so the backward
                            * scatter (lirec_rows_expand_bwd) need not re-read the fp32 activations.  Needs
                            * N % 32 == 0, aux_ld >= N / 32 (in 32-bit words), no split-K.                  */
};
enum lirec_out {
  LIREC_OUT_F32 = 0,
  LIREC_OUT_SPLIT_BF16 = 1,   /* hi at out[m*ld_m + col_off + n], lo at + lo_off                     */
  LIREC_OUT_SPLIT_BF16_T = 2  /* transposed: hi at out[(col_off + n)*ld_m + m], lo at row + lo_off   */
};

typedef struct lirec_epilogue {
  float alpha;
  const float* bias;        /* [N] or NULL                                   */
  const int32_t* row_flag;  /* [M] or NULL: bias only where row_flag[m] != 0 */
  int32_t act;              /* lirec_act                                     */
  int32_t post;             /* lirec_post                                    */
  float post_scale;
  lirec_dropout drop;
  const void* aux;          /* bf16 split tensor for DRELU / DTANH           */
  int64_t aux_ld;
  int32_t aux_col_off, aux_lo_off;
  int32_t out_kind;         /* lirec_out                                     */
  void* out;
  int64_t out_ld_m, out_ld_n; /* F32: &out[m*ld_m + n*ld_n]; SPLIT / SPLIT_T: ld_m only (row pitch) */
  int32_t out_col_off;      /* SPLIT: hi at col_off+n, lo at col_off+lo_off+n */
  int32_t out_lo_off;
  int32_t accumulate;       /* F32 only: out += v                            */
} lirec_epilogue;

typedef struct lirec_gemm_problem {
  int32_t M, N;
  int32_t a_mn_major, b_mn_major;
  int32_t num_passes;
  lirec_gemm_pass pass[LIREC_GEMM_MAX_PASSES];
  lirec_epilogue epi;
  /* split-K: when split_k > 1 the reduction range of every pass is cut into split_k slices of whole
   * 64-element k-blocks; slice s runs as its own tiles and writes its partial result to
   * out + s * split_stride (elements).  The caller sums the slices (fixed order = deterministic).
   * Needs an F32 output without activation, post op or accumulate; a bias is added in slice 0 only. */
  int32_t split_k;
  int64_t split_stride;
} lirec_gemm_problem;

/* One persistent launch over all tiles of all problems (host array).  Kernel choice per launch: the
 * CTA-pair kernel (256-row tiles, tcgen05 cta_group::2) unless the launch is too small to fill 60 % of
 * the clusters and fits one wave of 128x128 tiles (single-CTA kernel). */
int lirec_gemm_grouped(const lirec_gemm_problem* problems_host, int num_problems,
                       void* stream);
/* Per-launch timing of the GEMM kernel (CUDA events on the launching stream), for bench.py's
 * roofline line: begin() starts recording, end() synchronises on the recorded events and returns
 * the number of launches, filling duration (ms), executed MMA flops, tile and problem counts. */
int lirec_profile_begin(void);
/* Pause (0) / resume (1) the recording between begin() and end() without dropping what was recorded: an event pair
 * around every launch costs host time and breaks the programmatic-dependent-launch chain (13 % of a 64-clip step),
 * so bench.py records the launches of every 8th step of its timed region only.                                 */
int lirec_profile_sample(int32_t on);
int lirec_profile_end(float* ms_host, double* flops_host, int32_t* tiles_host, int32_t* problems_host,
                      int max_records);
/* Number of kernels the last lirec_* call on this thread launched. */
int lirec_last_launch_count(void);

/* ---- segmented reductions over ragged sequences -------------------------
 * Temporal pooling of variable-length frame / token / track sequences
 * (reference: np.max(axis=0) at mixed_utils/mixed_features.py:54,61,105; empty
 * segment -> zeros, text_utils/text_features.py:171-178, mixed_features.py:89-93).
 * x: [total_rows, dim] fp32, seg_off: [nseg+1] int32 prefix sums.
 * mode: 0 = max, 1 = mean.  out_bf16 / out_f32 may each be NULL.
 * row_idx: NULL for contiguous segments (segment s reduces rows [seg_off[s], seg_off[s+1])), else the
 * reduction runs over GATHERED rows: segment s reduces x[row_idx[r]] for r in [seg_off[s], seg_off[s+1]).
 * The dialog tokens of a clip are the union of the token ranges of every subtitle line that overlaps the
 * clip's time span (reference text_utils/text_features.py:151-168), not one contiguous range.          */
int lirec_seg_reduce_f32(const float* x, const int32_t* row_idx, const int32_t* seg_off,
                         int32_t nseg, int32_t dim, int32_t mode, float* out_f32,
                         int64_t out_f32_ld, void* out_bf16, int64_t out_bf16_ld, void* stream);

/* Softmax-weighted member of the same family, forward and backward — PARITY UNPINNED BY CONSTRUCTION: the
 * reference has no softmax / attention pooling (np.max at mixed_features.py:54, 61, 105; masked mean at
 * mlp/model.py:301-304); BASELINE.json's north_star asks for it and SURVEY.md §0.1 frames it as the third
 * member of {max, mean, softmax-weighted} over the same offset tables.
 *     out[s, c] = sum_{r in seg s} w[r, c] x[r, c],   w[., c] = softmax_r(beta * score[r, c])
 * score_mode 0: score = x (scores NULL; beta -> inf is the max, beta = 0 the mean); 1: per-element tensor
 * `scores` [total, dim]; 2: one score per row `scores` [total] (attention pooling).  An empty segment gives zeros.
 * lse: log-normaliser the backward needs, [nseg, lse_ld] (modes 0 / 1) or [nseg] (mode 2); may be NULL in fwd.
 * bwd writes d_x [total, dim] for every row of every segment and, if not NULL, d_scores ([total, dim] in mode 1,
 * [total] in mode 2; in mode 0 the score path is folded into d_x).  total_rows > 0: the rows of d_x / d_scores
 * outside [seg_off[0], seg_off[nseg]) — rows no segment owns — are zero-filled by the same launch, so the caller
 * need not clear the buffers first (a memset of d_x costs half the kernel's own time); 0: they are left untouched. */
int lirec_seg_softmax_pool_fwd(const float* x, const float* scores, int32_t score_mode,
                               const int32_t* seg_off, int32_t nseg, int32_t dim, float beta,
                               float* out, int64_t out_ld, float* lse, int64_t lse_ld, void* stream);
int lirec_seg_softmax_pool_bwd(const float* x, const float* scores, int32_t score_mode,
                               const int32_t* seg_off, int32_t nseg, int32_t dim, float beta,
                               const float* out, int64_t out_ld, const float* lse, int64_t lse_ld,
                               const float* d_out, int64_t d_out_ld, float* d_x, float* d_scores,
                               int64_t total_rows, void* stream);

/* ---- ragged row kernels of the modality encoder --------------------------
 * Layer-1 outputs are computed once per UNIQUE bank row (clip text, clip
 * visual, person track).  These kernels expand them to encoder rows by the
 * (clip, track1, track2) row tables, apply the layer-1 dropout + ReLU
 * (reference relu(dropout(.)) at mlp/model.py:282,287,293-294) and, for the
 * context branch, the masked mean over each candidate's context rows
 * (mlp/model.py:301-304,309,315,323-324), which commutes with the second
 * Linear.  Output is a hi/lo bf16 split [n_out, 4*2*J] laid out
 * [txt hi|lo, vis hi|lo, tr1 hi|lo, tr2 hi|lo].
 *
 * r1_* : relu(L1) of the unique rows, fp32 [*, J]; r1_tr1/r1_tr2 index the
 *        same track bank rows through different weights.
 * rows : [n_rows,3] int32 (clip, track1, track2).
 * seg_off : NULL -> one output row per table row (ints branch); else
 *        [n_out+1] prefix sums and output row c is the mean over its segment.
 * guard_zero: 1 -> empty segment gives 0 (MaxTracks, model.py:303); 0 -> 0/0 = NaN
 *        (MidFusionMultiClip, model.py:175).                                  */
int lirec_rows_expand_fwd(const float* r1_txt, const float* r1_vis, const float* r1_tr1,
                          const float* r1_tr2, int32_t J, const int32_t* rows,
                          const int32_t* seg_off, int32_t n_out, int32_t guard_zero,
                          lirec_dropout drop, void* out_split, int64_t out_ld,
                          int32_t* row_flag_out, void* stream);

/* Backward of lirec_rows_expand_fwd onto the unique rows of ONE bank slot.
 * d_in : fp32 [n_out, ld] gradient w.r.t. the (pre-split) expanded rows of
 *        this slot (column offset already applied by the caller).
 * inv_off/inv_idx : CSR from unique row u to the table rows that reference it.
 * owner : NULL (ints) or [n_rows] candidate index of each context row;
 * seg_off: NULL or [n_out+1] (context) to derive 1/n.
 * slot : 0 txt, 1 vis, 2 tr1, 3 tr2 (selects the dropout columns).
 * sign : ReLU gate [r1 > 0] of the unique rows as bits, in the LIREC_POST_SIGN_MASK layout: bit (j & 31)
 *        of sign[u*sign_ld + (j >> 5)]; 8-byte aligned, sign_ld even and >= J/32 words.  J % 64 == 0.
 * Writes dZ1 = [r1 > 0] * sum(...) TRANSPOSED as a hi/lo split [2*J, out_pitch] (hi rows [0,J),
 * lo rows [J,2J); out_pitch >= n_unique, a multiple of 8; 16-byte aligned) — the K-major operand
 * of the first-layer wgrad GEMM.                                                  */
int lirec_rows_expand_bwd(const float* d_in, int64_t d_ld, const uint32_t* sign, int64_t sign_ld,
                          int32_t J, int32_t slot, const int32_t* inv_off, const int32_t* inv_idx,
                          int32_t n_unique, const int32_t* owner, const int32_t* seg_off,
                          lirec_dropout drop, void* out_split, int64_t out_pitch, void* stream);

/* Spatial / person-box mean of I3D feature maps fused with the temporal max:
 *   out[s, c] = max over the elements e of segment s of mean(maps[frame_e, c, y0:y1, x0:x1]).
 * maps: fp32 [T, C, H, W]; elem: int32 [n_elem, 5] = (frame, y0, y1, x0, x1), computed on the host with
 * the reference's float64 box arithmetic (lirec_b200/visual_utils/visual_features.py);
 * seg_off: [nseg+1] prefix sums over elements.  frame < 0: an all-zero row that takes part in the max
 * (reference visual_features.py:130-131); empty box: NaN; empty segment: zeros.
 * scratch: NULL, or fp32 [n_elem, C] (16-byte aligned, C % 4 == 0): the means of all elements are then
 * computed in one fully parallel pass and reduced by the segmented-max kernel (2-3x the bandwidth of
 * the single-pass form on long tracks).
 * Replaces np.mean over H x W / over the person box (visual_utils/visual_features.py:67-69, 133-134)
 * followed by np.max over frames / track elements (mixed_utils/mixed_features.py:54, 104-105).  */
int lirec_roi_max_pool_f32(const float* maps, int32_t T, int32_t C, int32_t H, int32_t W,
                           const int32_t* elem, int32_t n_elem, const int32_t* seg_off, int32_t nseg,
                           float* scratch, float* out_f32, int64_t out_f32_ld, void* out_bf16,
                           int64_t out_bf16_ld, void* stream);

/* Row gather out[i, :] = bank[idx[i], :] over bf16 rows (dim, bank_ld, out_ld in elements,
 * multiples of 8; idx outside [0, n_bank) gives a zero row).  Replaces the host-side
 * np.hstack / np.tile assembly of cached vectors into batch rows (reference
 * mixed_utils/mixed_features.py:115-125, classification_dataloader.py:329-334, 393-416):
 * the split's pooled feature banks stay resident in HBM and a batch ships only indices.  */
int lirec_gather_rows(const void* bank, int64_t bank_ld, int32_t n_bank, const int32_t* idx,
                      int32_t n, int32_t dim, void* out, int64_t out_ld, void* stream);

/* fp32 [rows, cols] -> TRANSPOSED hi/lo bf16 split [2*pad, pitch]: hi at out_split[c*pitch + r],
 * lo at out_split[(pad + c)*pitch + r]; rows c in [cols, pad) are zero (pad >= cols, pitch >= rows). */
int lirec_split_f32(const float* x, int64_t ld, int32_t rows, int32_t cols, void* out_split,
                    int64_t pitch, int32_t pad, void* stream);
/* fp32 -> bf16 (round to nearest even), n elements. */
int lirec_cast_bf16(const float* x, void* out, int64_t n, void* stream);

/* ---- losses: fused forward + gradient over ragged candidate tables -------
 * All losses are sigmoid + max-margin hinges (reference mlp/model.py:381-575).
 * Each writes per-clip loss terms (already divided by the batch size) and
 * d(loss)/d(logits); the scalar loss is the sum of loss_per_clip.            */
typedef struct lirec_track_loss_cfg {
  float margin;        /* opt.tr_margin                                      */
  float lymbda;        /* weight of the interaction term                     */
  int32_t n_classes;   /* C                                                  */
  int32_t n_rels;      /* R (the None class has index R); 0 -> no rel term   */
  int32_t tr_correct;  /* supervised assignment (t* = 0)                     */
  int32_t max_neg;     /* opt.tr_max_neg && opt.tr_sum_max_flag              */
  int32_t max_slots;   /* T: reference slot count, only used by max_neg      */
  int32_t cat_distr;   /* opt.tr_cat_distr: sample t* from the softmax scores
                          (model.py:468-471, 538-543) instead of the arg-max   */
  uint32_t seed;       /* counter-hash seed of that draw (per step)           */
} lirec_track_loss_cfg;

/* MarginLoss (model.py:444-494) when n_rels == 0, MarginTrackRelsLoss
 * (model.py:497-575) otherwise.  ints: [Ni, C] fp32, rels: [Ni, R] fp32,
 * cand_off: [B+1], labels: [B], rels_label: [Ni], gt_tracks: [B,2],
 * multilab: [B, C] uint8 (1 = class may be used as a negative).
 * Outputs: loss_per_clip [B], assign [B] (t*), d_ints [Ni,C], d_rels [Ni,R]. */
int lirec_loss_track_fwd_bwd(const float* ints, const float* rels, const int32_t* cand_off,
                             int32_t B, const int32_t* labels, const int32_t* rels_label,
                             const int32_t* gt_tracks, const uint8_t* multilab,
                             lirec_track_loss_cfg cfg, float* loss_per_clip, int32_t* assign,
                             float* d_ints, float* d_rels, void* stream);

/* Softmax cross-entropy rows, forward + gradient: either term of MultiTaskCrossEntropyLoss
 * (model.py:357-378, F.cross_entropy with optional class weights).  rows with label < 0 are
 * skipped; scale = 1 / (sum of class weights of the selected rows) gives the mean reduction.  */
int lirec_loss_ce_fwd_bwd(const float* logits, int64_t ld, int32_t rows, int32_t C,
                          const int32_t* labels, const float* class_weights, float scale,
                          float* loss_per_row, float* d_logits, int64_t d_ld, void* stream);

/* MaxMarginCrossEntropyLoss (model.py:422-441) and the two terms of
 * MultiTaskMaxMargin (model.py:381-419): a row-wise hinge
 *   loss_row = sum_c relu(m - s[y] + s[c]) over c != y with weight[c] != 0.
 * rows with label < 0 are skipped; scale multiplies loss and gradient.       */
int lirec_loss_rowmargin_fwd_bwd(const float* logits, int64_t ld, int32_t rows, int32_t C,
                                 const int32_t* labels, const uint8_t* weights, float margin,
                                 float scale, float* loss_per_row, float* d_logits,
                                 int64_t d_ld, void* stream);

/* Multi-label sigmoid binary cross-entropy, forward + gradient (the reference has no BCE: parity is
 * unpinned by construction; the tests' reference is torch's binary_cross_entropy_with_logits in fp64).
 * Per element with target t and weight w:
 *   l = w * (t * softplus(-x) + (1 - t) * softplus(x)),  dl/dx = w * (sigma(x) - t),
 * softplus(x) = max(x,0) + log1p(exp(-|x|)), finite for any finite logit.  Masks are [rows or B, C]
 * uint8; NULL means none.  Every element of the gradient rows a call owns is written.
 *
 * Row form: t_c = 1 for c == label or pos_mask[i,c] != 0; w_c = 0 for a non-target with
 * neg_mask[i,c] == 0 (neg_mask NULL: every non-target is a negative).
 *   loss_per_row[i] = scale * sum_c w_c * l_c;  rows with label < 0 get 0 and a zero gradient row. */
int lirec_loss_bce_fwd_bwd(const float* logits, int64_t ld, int32_t rows, int32_t C, const int32_t* labels,
                           const uint8_t* neg_mask, const uint8_t* pos_mask, float scale,
                           float* loss_per_row, float* d_logits, int64_t d_ld, void* stream);

/* Track form over the same inputs as lirec_loss_track_fwd_bwd, plus pos_mask [B, C] (NULL: none).
 * t* is chosen exactly as there (arg-max, tr_correct, cat_distr) and written to assign[b].  The
 * interaction positives are (t*, y) and (t*, c) for pos_mask[b,c] != 0; the negatives are the margin
 * loss's sum-form negatives minus those positives; every other (slot, class) has weight 0.  The
 * relationship positive is (t*, r0) when live, its negatives the margin loss's relationship negatives.
 *   loss_per_clip[b] = lymbda / B * sum_ints l + 1 / B * sum_rels l
 * cfg.margin is ignored; cfg.max_neg != 0 is LIREC_ERR_ARG (max-negative is a hinge idea).          */
int lirec_loss_bce_track_fwd_bwd(const float* ints, const float* rels, const int32_t* cand_off, int32_t B,
                                 const int32_t* labels, const int32_t* rels_label, const int32_t* gt_tracks,
                                 const uint8_t* multilab, const uint8_t* pos_mask, lirec_track_loss_cfg cfg,
                                 float* loss_per_clip, int32_t* assign, float* d_ints, float* d_rels, void* stream);

/* Prediction arg-maxes of the evaluation loop (reference utils/evaluation.py:114-175, 179-271:
 * track assignment for the GT class (+ relationship), joint (t,c[,r]) arg-max, class / relationship
 * arg-max at the two GT slots), computed on the ragged logits so only 8 integers per clip go back to
 * the host.  out: int32 [B, 8] = {pr_track, joint_t, joint_c, joint_r, cls_gt0, cls_gt1, rel_gt0,
 * rel_gt1}; lowest index wins ties, like np.argmax.  n_rels == 0 -> interaction-only form.        */
int lirec_predict_tracks(const float* ints, const float* rels, const int32_t* cand_off, int32_t B,
                         const int32_t* labels, const int32_t* rels_label, const int32_t* gt_tracks,
                         int32_t n_classes, int32_t n_rels, int32_t* out, void* stream);

/* ---- the model hot path: one call per direction ---------------------------
 * Native launch sequence for the forward and backward of Modalities
 * (mlp/model.py:19-92), MidFusionMultiClip (:95-211), MidFusionMultiClipMaxTracks
 * (:214-339) and GatingUnit (:342-354) over a PACKED ragged batch: layer 1 once per
 * unique bank row, ragged expansion / masked mean, layer 2 + tanh + dropout, gate,
 * heads.  The host sequence is C++ so a step is ~12 launches, not ~150 ATen calls. */
typedef struct lirec_linear {
  const void* w_bf16;  /* [out_f, in_f] bf16 shadow of the fp32 nn.Linear weight      */
  const float* bias;   /* [out_f] fp32                                                */
  float* grad_w;       /* [out_f, in_f] fp32, written (not accumulated) by backward   */
  float* grad_b;       /* [out_f] fp32                                                */
  int32_t out_f, in_f;
} lirec_linear;

/* the 8 Linears of one modality encoder (model.py:222-246): first layers txt_*, vis_*,
 * tracks1_*, tracks2_*; second layers txt2_*, vis2_*, tracks12_*, tracks22_*          */
typedef struct lirec_encoder {
  lirec_linear l1[4];
  lirec_linear l2[4];
} lirec_encoder;

typedef struct lirec_model_params {
  lirec_encoder enc_ints, enc_ctx;
  lirec_linear gate;      /* gates_ints.fc_out: [gate_dim, 2*3J]                      */
  lirec_linear out_ints;  /* [n_classes, gate_dim or 3J]                              */
  lirec_linear out_ctx;   /* [n_rels, 3J]                                             */
} lirec_model_params;

typedef struct lirec_model_cfg {
  int32_t text_dim, visual_dim, track_dim;  /* 768, 2048, 2048                        */
  int32_t joint_dim;                         /* J = 512                                */
  int32_t gate_dim;                          /* joint_dim * mid_m_ints = 3072          */
  int32_t n_classes, n_rels;
  int32_t ctx, gates;                        /* opt.ctx, opt.gates (opt.ints: no_ints) */
  int32_t guard_zero;                        /* 1: MaxTracks divider guard (model.py:303) */
  float dropout_p;                           /* opt.dropout                            */
  int32_t slot_mask;                         /* bit s: modality slot present (0 txt, 1 vis, 2 tracks1,
                                                3 tracks2); 0 = all.  Modalities with opt.modality 't' / 'v'
                                                or without tracks (model.py:27-46, 78-86) drop slots; the
                                                concatenated feature shrinks accordingly               */
  int32_t no_ints;                           /* 1: opt.ints == 0 (model.py:102, 140, 151, 208, 220, 256, 278, 335) — no
                                                interaction branch and no interaction head: the model is the context
                                                branch + relationship head (needs ctx = 1, gates = 0; out_ints /
                                                d_ints / enc_ints / out_ints parameters are ignored and may be NULL) */
} lirec_model_cfg;

/* Packed ragged batch (device pointers).  Every encoder row — candidate row or context
 * row — is a triple (clip, track1, track2) of bank row indices; a missing track points
 * at an all-zero bank row.  Bank rows [0, n_*_ints) are the ones the ints branch uses. */
typedef struct lirec_batch {
  const void* clip_bank;   /* bf16 [n_clip, text_dim + visual_dim]                    */
  int64_t clip_ld;
  int32_t n_clip, n_clip_ints;
  const void* track_bank;  /* bf16 [n_track, track_dim]                               */
  int64_t track_ld;
  int32_t n_track, n_track_ints;
  int32_t n_cand;          /* Ni: candidate rows in the batch                         */
  int32_t n_ctx_rows;      /* Nx: valid context rows in the batch                     */
  const int32_t* cand_rows;  /* [Ni, 3]                                               */
  const int32_t* ctx_rows;   /* [Nx, 3]                                               */
  const int32_t* ctx_off;    /* [Ni + 1] prefix sums                                  */
  const int32_t* ctx_owner;  /* [Nx] candidate of each context row                    */
  /* CSR inverses (unique bank row -> referencing table rows), slot 0 clip (txt+vis),
   * 1 track1, 2 track2; only needed by backward                                      */
  const int32_t* inv_cand_off[3];
  const int32_t* inv_cand_idx[3];
  const int32_t* inv_ctx_off[3];
  const int32_t* inv_ctx_idx[3];
  uint32_t seed;           /* dropout seed of this step                               */
  int32_t training;        /* 0: no dropout                                           */
} lirec_batch;

size_t lirec_model_workspace_bytes(const lirec_model_cfg* cfg, const lirec_batch* batch_host);
/* out_ints: fp32 [Ni, n_classes]; out_rels: fp32 [Ni, n_rels] (NULL when ctx == 0).
 * The workspace keeps the activations backward needs.                               */
int lirec_model_forward(const lirec_model_cfg* cfg, const lirec_model_params* params,
                        const lirec_batch* batch, void* workspace, size_t workspace_bytes,
                        float* out_ints, float* out_rels, void* stream);
/* d_ints / d_rels: fp32 gradients w.r.t. the logits.  Writes every grad_w / grad_b.
 * heads_event (a cudaEvent_t; may be NULL): recorded on `stream` as soon as the gradients of the gate and of the
 * two heads are final in the flat gradient buffer: a data-parallel caller starts the exchange + Adam of that range
 * (53 % of the weights) on another stream while the encoder stages of backward still run (lirec_b200/dp.py).
 * Autograd runs backward as one opaque call (mlp/train.py:62). */
int lirec_model_backward(const lirec_model_cfg* cfg, const lirec_model_params* params,
                         const lirec_batch* batch, void* workspace, size_t workspace_bytes,
                         const float* d_ints, const float* d_rels, void* stream, void* heads_event);

/* White-box test aid: byte offsets of the named workspace buffers (see csrc/model.cu). */
int lirec_model_workspace_layout(const lirec_model_cfg* cfg, const lirec_batch* batch_host,
                                 int64_t* offsets, int max_entries);

/* ---- host-side batch assembly (no GPU work) ---------------------------------
 * Replaces the np.tile / hstack / vstack assembly of cached 6912-d rows in the reference's DataLoader
 * workers (mixed_utils/classification_dataloader.py:329-334, 393-416, 474-497, mixed_features.py:115-125)
 * and the default collate (mlp/train.py:33-37): a record carries only (clip, track1, track2) index triples
 * into the DATASET banks; this call turns the concatenated triples of a batch into every integer table of
 * a lirec_batch, in one int32 arena that crosses PCIe in one copy.  All pointers are HOST pointers.
 *   cand_host [Ni,3] / cand_counts_host [B]: candidate triples per clip (reference slot order);
 *   ctx_host [Nx,3] / ctx_counts_host [Ni]: context triples per candidate (both NULL: no context branch);
 *   zero_clip: the dataset's all-zero clip row; track row 0 is the all-zero track.  References to either
 *   are redirected to one private zero row per clip.
 * Batch bank rows: rows the candidates use (ascending dataset row, private zero rows first), then the rows
 * only context uses.  layout_host [24][2] = (offset, length) in arena_host of cand_off, cand_rows, ctx_off,
 * ctx_rows, ctx_owner, labels, rels_label, gt_tracks, inv_cand_off0, inv_cand_idx0, .._off1, .._idx1, .._off2,
 * .._idx2, inv_ctx_off0 .. inv_ctx_idx2, cand_clip, cand_slot, clip_src, track_src (length -1 = absent;
 * labels / rels_label / gt_tracks are reserved for the caller to fill; clip_src / track_src = dataset-bank
 * row behind every batch bank row).  sizes_host [4] = n_clip, n_clip_ints, n_track, n_track_ints.          */
#define LIREC_COLLATE_NUM_TABLES 24
int64_t lirec_collate_arena_bound(int64_t B, int64_t n_cand, int64_t n_ctx, int32_t has_ctx);
int lirec_collate_tables(const int32_t* cand_host, const int32_t* cand_counts_host, int32_t B,
                         const int32_t* ctx_host, const int32_t* ctx_counts_host, int32_t zero_clip,
                         int32_t n_clip_rows, int32_t n_track_rows, int32_t max_slots,
                         int32_t* arena_host, int64_t arena_cap, int64_t* layout_host, int32_t* sizes_host);

/* Ragged gather in front of lirec_collate_tables for datasets that keep every record's triples back to back in
 * dataset-level tables (lirec_b200/mixed_utils/cached_clips.py): ds_cand_off [n_items + 1] / ds_cand [*, 3] = CSR of
 * the candidate triples by item; ds_ctx_off [n_cand_total + 1] / ds_ctx_cnt [n_cand_total] / ds_ctx [*, 3] = CSR of
 * the context triples by candidate (all three NULL: no context branch); idx [B] = the items of the batch.  Writes the
 * batch's candidate triples, per-clip candidate counts, the dataset position of every candidate (cand_pos_out, may be
 * NULL), context triples and per-candidate context counts — the inputs of lirec_collate_tables — and their row counts.
 * Replaces the per-item `__getitem__` + list concatenation of the reference's loader (classification_dataloader.py
 * :291-616 + default collate) for index-only records.  HOST pointers only.                                         */
int lirec_collate_gather(const int64_t* ds_cand_off, const int32_t* ds_cand, const int64_t* ds_ctx_off,
                         const int32_t* ds_ctx_cnt, const int32_t* ds_ctx, const int64_t* idx, int32_t B,
                         int32_t* cand_out, int32_t* counts_out, int64_t* cand_pos_out, int64_t max_cand,
                         int32_t* ctx_out, int32_t* ctx_counts_out, int64_t max_ctx, int64_t* n_cand_out,
                         int64_t* n_ctx_out);

/* ---- optimizer -----------------------------------------------------------
 * torch.optim.Adam with coupled L2 (reference mlp/model.py:599-601) over one
 * flat buffer; also refreshes the bf16 shadow of the weights.
 * coresident != 0 launches the same pass in CTAs small enough to share an SM with a resident CTA of the
 * persistent GEMM kernels (which leave ~18 % of the register file), for a range whose gradients are final while
 * backward is still running on another stream.  Identical results.                                              */
int lirec_adam_flat(float* param, const float* grad, float* exp_avg, float* exp_avg_sq,
                    void* param_bf16, int64_t n, float lr, float beta1, float beta2, float eps,
                    float weight_decay, int32_t step, float grad_scale, int32_t coresident, void* stream);

/* LAMB (You et al., "Large Batch Optimization for Deep Learning", ICLR 2020) over the same flat buffers, for
 * large-batch training.  Tensor l is floats [tensor_begin[l], tensor_begin[l] + tensor_len[l]) of the buffers
 * (DEVICE arrays [n_tensors]; the tensors are disjoint and lie inside [0, n)).  Per element, step t:
 *   g = grad_scale * grad;  m = b1*m + (1-b1)*g;  v = b2*v + (1-b2)*g*g
 *   u = (m / bc1) / (sqrt(v) / sqrt(bc2) + eps) + weight_decay * w            (decoupled weight decay)
 *   r_l = ||w_l|| / ||u_l|| if both norms > 0, else 1                          (norms over the old w)
 *   w = w - lr * r_l * u;  param_bf16 = rn_bf16(w)  (param_bf16 may be NULL)
 * with bc1 = 1 - b1^t, bc2 = 1 - b2^t in double.  No ratio clamp, no exclusions; NaN and Inf propagate.
 * The betas come as their complements one_minus_beta1 = 1 - b1, one_minus_beta2 = 1 - b2 (each in (0, 1]): fp32
 * holds 1 - b to full precision where 1 - fp32(0.999) is 1.3e-5 off 0.001; b = 1 - (1 - b) is formed in double.
 * Two launches: moments + per-chunk partial norms, then trust ratios + update.  Each tensor is cut into chunks of
 * LIREC_LAMB_CHUNK floats; the norms are summed in a fixed order (fp64 across chunks, no atomics), so results are
 * bitwise reproducible.  `partials` is caller-owned device scratch of n_partials chunk entries of two doubles,
 * n_partials >= LIREC_LAMB_PARTIALS(n, n_tensors).  trust_out (optional, DEVICE [n_tensors]) receives every r_l.
 * A tensor of length <= 0 is empty: nothing is read or written for it and its r_l is 1.  Floats outside every
 * tensor (the padding between segments) are neither read into a norm nor written.                           */
#define LIREC_LAMB_CHUNK 8192
#define LIREC_LAMB_PARTIALS(n, n_tensors) ((n) / LIREC_LAMB_CHUNK + (n_tensors))
int lirec_lamb_flat(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, void* param_bf16,
                    const int64_t* tensor_begin, const int64_t* tensor_len, int32_t n_tensors, int64_t n,
                    double* partials, int64_t n_partials, float lr, float one_minus_beta1,
                    float one_minus_beta2, float eps, float weight_decay, int32_t step, float grad_scale,
                    float* trust_out, void* stream);

/* Global-norm gradient clipping over the flat gradient buffer, in place: torch.nn.utils.clip_grad_norm_(params,
 * max_norm) with norm_type 2, applied to the gradient an optimizer is about to consume.  Same tensor table as
 * lirec_lamb_flat (DEVICE arrays tensor_begin / tensor_len [n_tensors], disjoint, inside [0, n)):
 *   norm = || grad_scale * grad ||_2 over every tensor          (grad_scale: the data-parallel 1/world average)
 *   coef = min(max_norm / (norm + 1e-6), 1) in fp32             (a NaN norm gives a NaN coef, an Inf norm 0)
 *   grad = grad * coef                                          (grad_scale is NOT applied: the optimizer does)
 * When coef is exactly 1 the buffer is not written.  Three launches: per-chunk sums of squares (fp32 within a
 * thread, fp64 across the CTA), one CTA that sums them in a fixed order in fp64 (each tensor's chunks in order, then
 * the tensors in table order), and the scale; no host sync, no float atomics, bitwise reproducible.  `partials` is
 * the same caller-owned scratch as lirec_lamb_flat's (n_partials entries of two doubles, n_partials >=
 * LIREC_LAMB_PARTIALS(n, n_tensors)).  norm_out (DEVICE float, required) receives the pre-clip norm;
 * tensor_norms_out (optional, DEVICE [n_tensors]) the pre-clip norm of every tensor.  max_norm must be finite and
 * > 0.  Floats outside every tensor are neither read nor written.                                                 */
int lirec_grad_clip_flat(float* grad, const int64_t* tensor_begin, const int64_t* tensor_len, int32_t n_tensors,
                         int64_t n, double* partials, int64_t n_partials, float max_norm, float grad_scale,
                         float* norm_out, float* tensor_norms_out, void* stream);

/* Exponential moving average of the flat weights, for evaluation and checkpoints (the update of
 * torch.optim.swa_utils.AveragedModel with get_ema_multi_avg_fn(decay), i.e. torch._foreach_lerp_):
 *   ema[i] = lerp(ema[i], param[i], a),  a = one_minus_decay = 1 - decay, elementwise in fp32, i in [0, n):
 *     a < 0.5:  ema + a * (param - ema)          otherwise:  param - (param - ema) * (1 - a)
 * each rounded as one FMA, as torch.lerp's kernel computes it.  NaN and Inf propagate like torch.lerp.  param is read
 * and never written.  Pass the complement, formed in double: fp32 holds 1 - decay to full precision where
 * 1 - fp32(0.9999) loses digits.  One launch, no host sync.  one_minus_decay must be finite and in (0, 1).  */
int lirec_ema_update_flat(float* ema, const float* param, int64_t n, float one_minus_decay, void* stream);

/* Exchange param[i] and ema[i] for i in [0, n) (evaluate the average, then swap back), and when param_bf16 is not
 * NULL write param_bf16[i] = rn_bf16(new param[i]) with lirec_cast_bf16's rounding, so the shadow equals
 * lirec_cast_bf16(param) bit for bit afterwards.  Two swaps restore all three buffers when the shadow was
 * lirec_cast_bf16(param) to begin with.  One launch.                                                          */
int lirec_ema_swap_flat(float* param, float* ema, void* param_bf16, int64_t n, void* stream);
/* Both EMA entry points refuse a NULL param / ema, n < 0 and a buffer that is not 16-byte aligned; n == 0 enqueues
 * nothing.                                                                                                     */

/* ---- data parallel: in-switch gradient exchange, bucket by bucket --------
 * Replaces ncclAllReduce(flat gradient) of a data-parallel step (the reference is single-process, SURVEY.md
 * §2.3; the optimizer stays torch.optim.Adam's arithmetic, mlp/model.py:599-601, through lirec_adam_flat on the
 * same range afterwards).  `grad_multicast` is the NVSwitch multicast address of the flat fp32 gradient buffer,
 * which lives in SYMMETRIC memory on every rank (lirec_b200/dp.py obtains both from
 * torch.distributed._symmetric_memory).  The call enqueues on `stream`: a cross-GPU barrier, this rank's 1/world
 * shard of floats [offset, offset + n) reduced inside the switch (multimem.ld_reduce.add) and broadcast
 * (multimem.st), and a second barrier — afterwards every rank holds the SUM over ranks in that range.
 * flag_ptrs_dev: device array [world] of every rank's peer-mapped, zero-initialised flag buffer of
 * lirec_dp_flag_words(world) uint32; `channel` (0..3) selects the flag slots, so chains for different buckets may
 * be in flight on different streams at the same time (all ranks must use the same channel for the same bucket).
 * coresident != 0 (all three passes): CTAs small enough to share an SM with a resident CTA of the persistent GEMM
 * kernels, for a bucket exchanged on a side stream while backward still runs (see lirec_adam_flat).          */
int lirec_dp_flag_words(int32_t world);
/* Exchange + optimizer + parameter broadcast in ONE pass (ZeRO-1 style), the default data-parallel step: every
 * rank owns the Adam moments of its 1/world shard.  For its shard it sums the gradients inside the switch
 * (multimem.ld_reduce.add on grad_multicast), applies torch.optim.Adam's update (mlp/model.py:599-601, same
 * arithmetic as lirec_adam_flat) to the local parameters `param` with grad * grad_scale, stores the moments
 * locally and multicast-stores the new fp32 parameters and their bf16 shadow into EVERY rank's buffers
 * (param_multicast / param_bf16_multicast: the multicast addresses of the symmetric parameter buffers).
 * exp_avg / exp_avg_sq are full-size arrays of which only this rank's shard [n/4*rank/world, n/4*(rank+1)/world)
 * (in 16-byte units) is read and written.  Barriers before and after as in lirec_dp_exchange.               */
int lirec_dp_reduce_adam_bcast(const void* grad_multicast, const float* param, void* param_multicast,
                               void* param_bf16_multicast, float* exp_avg, float* exp_avg_sq, int64_t n,
                               float lr, float beta1, float beta2, float eps, float weight_decay,
                               int32_t step, float grad_scale, int32_t rank, int32_t world,
                               const void* flag_ptrs_dev, int32_t channel, int32_t coresident, void* stream);
int lirec_dp_exchange(void* grad_multicast, int64_t offset, int64_t n, int32_t rank, int32_t world,
                      const void* flag_ptrs_dev, int32_t channel, int32_t coresident, void* stream);

/* The same pass over plain peer pointers instead of the multicast object (P2P loads of every rank's gradient
 * shard, P2P stores of the new parameters into every rank): the better transport at 2 ranks, where an in-switch
 * reduction drags the requester's own copy through the switch as well.  peer_bases_dev: device array [world] of
 * every rank's peer-mapped symmetric allocation; *_off: byte offsets of the gradient, fp32 parameter and bf16
 * shadow buffers inside it.  world must be 2, 4 or 8.                                                        */
int lirec_dp_reduce_adam_bcast_peer(const void* peer_bases_dev, int64_t grad_off, int64_t param_off,
                                    int64_t bf16_off, float* exp_avg, float* exp_avg_sq, int64_t n,
                                    float lr, float beta1, float beta2, float eps, float weight_decay,
                                    int32_t step, float grad_scale, int32_t rank, int32_t world,
                                    const void* flag_ptrs_dev, int32_t channel, int32_t coresident, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LIREC_B200_H_ */
