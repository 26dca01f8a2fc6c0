// model.cu — native launch sequence of the model hot path over a packed ragged batch.
//
// Reference: Modalities.forward (mlp/model.py:54-92), MidFusionMultiClip.forward
// (:147-211), MidFusionMultiClipMaxTracks.forward (:265-339), GatingUnit.forward
// (:349-354) and the autograd backward of all of them (mlp/train.py:62).
//
// Restructuring relative to the reference (same function, different schedule):
//   1. every 6912-d input row is (clip text|visual, track1, track2) of cached vectors
//      (classification_dataloader.py:329-334, mixed_features.py:115-125), so the first
//      Linear of each modality runs ONCE PER UNIQUE BANK ROW, not once per
//      (candidate, context) row;
//   2. relu(dropout(.)) is applied while expanding the unique rows to encoder rows by
//      the (clip, track1, track2) row tables;
//   3. the context branch's masked mean (model.py:301-324) commutes with its second
//      Linear, so it is taken over the expanded rows BEFORE layer 2, which then runs on
//      one row per candidate;
//   4. activations that feed another GEMM are kept as hi/lo bf16 pairs, so the bf16
//      tensor-core products carry ~16 mantissa bits (the 1e-3 parity bar of the spec
//      cannot be met with single-bf16 activations, SURVEY.md §7.3);
//   5. bias gradients are GEMMs against a ones (or row-flag) column, so every parameter
//      gradient of a stage comes out of one grouped launch, deterministically.
#include <vector>

#include "gemm.cuh"
#include "rows.cuh"

namespace lirec {
namespace model {

typedef __nv_bfloat16 bf16;

// dropout sites (stream ids of the counter hash)
enum { DS_L1_INTS = 1, DS_L1_CTX = 2, DS_CAT_INTS = 3, DS_CAT_CTX = 4, DS_GATE = 5 };

static inline int64_t round_up(int64_t v, int64_t a) { return (v + a - 1) / a * a; }

struct Dims {
  int J, F, Gd, C, R, CP, RP;
  int Ni, Nx, nc, nci, nt, nti;
  int cs[4], outw[4], inw[4];
  bool act[4];        // modality slot present (Modalities with opt.modality 't'/'v' or without tracks)
  int ones_rows;
  int NiP, ncP[2], ntP[2], onesP;   // row pitches of the transposed gradient buffers (multiples of 64)
  bool ctx, gates;
  bool ints;           // interaction (candidate) branch present: opt.ints (reference model.py:102, 140, 151, 208)
  int br0;             // first branch of the loops over {0: ints, 1: ctx}
};

static Dims make_dims(const lirec_model_cfg& c, const lirec_batch& b) {
  Dims d;
  d.J = c.joint_dim;
  d.Gd = c.gate_dim;
  d.C = c.n_classes;
  d.R = c.n_rels;
  d.CP = (int)round_up(d.C, 64);
  d.RP = (int)round_up(std::max(d.R, 1), 64);
  d.Ni = b.n_cand;
  d.Nx = b.n_ctx_rows;
  d.nc = b.n_clip;
  d.nci = b.n_clip_ints;
  d.nt = b.n_track;
  d.nti = b.n_track_ints;
  d.outw[0] = d.J; d.outw[1] = d.J; d.outw[2] = d.J / 2; d.outw[3] = d.J / 2;
  const int mask = (c.slot_mask & 15) ? (c.slot_mask & 15) : 15;
  d.F = 0;
  for (int s = 0; s < 4; ++s) {     // concat order txt | vis | tracks1 | tracks2 (model.py:80-86, 296)
    d.act[s] = (mask >> s) & 1;
    d.cs[s] = d.F;
    if (d.act[s]) d.F += d.outw[s];
  }
  d.inw[0] = c.text_dim; d.inw[1] = c.visual_dim; d.inw[2] = c.track_dim; d.inw[3] = c.track_dim;
  d.ctx = c.ctx != 0;
  d.gates = c.gates != 0;
  d.ints = c.no_ints == 0;
  d.br0 = d.ints ? 0 : 1;
  d.ones_rows = std::max(std::max(d.Ni, d.nc), d.nt);
  d.NiP = (int)round_up(d.Ni, 64);
  d.ncP[0] = (int)round_up(d.nci, 64); d.ncP[1] = (int)round_up(d.nc, 64);
  d.ntP[0] = (int)round_up(d.nti, 64); d.ntP[1] = (int)round_up(d.nt, 64);
  d.onesP = (int)round_up(d.ones_rows, 64);
  return d;
}

struct Workspace {
  float* r1[2][4];    // relu(L1) of the unique rows, per branch and slot
  bf16* a2[2];        // expanded / pooled layer-2 inputs  [Ni, 8J]
  int32_t* flag_c;    // [Ni] context segment non-empty
  bf16* flagT;        // [1, NiP] the same flag as the K-major operand of the bias-gradient GEMMs
  bf16* onesT;        // [1, onesP] ones
  bf16* f2[2];        // dropout(tanh(concat)) hi|lo       [Ni, 6J]
  bf16* g2;           // gate output hi|lo                  [Ni, 2Gd]
  // Backward temporaries.  Every activation gradient is kept TRANSPOSED ([feature, row], hi rows then
  // lo rows, row pitch NiP / nuP): it is the K-major B operand of the weight-gradient GEMM that reduces
  // over the batch rows and the MN-major A operand of the next data-gradient GEMM — the two operand
  // forms the CTA-pair tcgen05 kernel runs at full rate (an MN-major B operand does not).
  bf16* dliT;         // [2CP, NiP]
  bf16* dlrT;         // [2RP, NiP]
  bf16* dpregT;       // [2Gd, NiP]
  bf16* dz2T[2];      // [6J, NiP]
  float* da2[2];      // [Ni, 4J]
  bf16* dz1T[2][4];   // [2J, nuP]
  // [in, out] copies of the weights the data-gradient GEMMs multiply by (K-major B operands)
  bf16* out_intsT;    // [Gd or 3J, CP]
  bf16* out_ctxT;     // [3J, RP]
  bf16* gateT;        // [6J, Gd]
  bf16* l2T[2][4];    // [J, outw]
  uint32_t* sgn[2][4];  // [n_unique, J / 32] ReLU gate of layer 1, one bit per element (LIREC_POST_SIGN_MASK)
  int32_t* ref_out[3];  // per-reference tables of the context inverse CSRs (rows::ref_tables), [Nx] each
  float* ref_w[3];
  float* pool;        // split-K partial gradients
  size_t pool_floats;
  size_t bytes;
};

// ---- split-K of long, few-tile reductions -----------------------------------------------------
// A weight / bias gradient reduces over all rows of the batch (thousands of k-blocks) but has only a
// handful of output tiles, so on its own it would occupy a few SMs for the whole stage.  Such a
// problem is cut into S row ranges that write partial results into a pool; one small kernel sums
// the partials into the flat gradient buffer at the end of backward, in a fixed order
// (deterministic, no atomics).
static int split_factor(int out_f, int in_f, int passes, int rows) {
  // tiles of the (M = in_f, N = out_f) pair-kernel problem: 256 x (256 | 128)
  const int bn = out_f > 128 ? 256 : 128;
  const int tiles = ((in_f + 255) / 256) * ((out_f + bn - 1) / bn);
  const int kb = passes * ((rows + 63) / 64);
  if (tiles >= 64 || kb < 128) return 1;
  return std::max(1, std::min(std::min(8, kb / 64), (74 + tiles - 1) / tiles));
}
// K-slices of the interaction head's forward GEMM ([Ni, C <= 128] output: one pair tile per 256 rows)
static int head_split(int Ni, int width) {
  const int tiles = (Ni + 255) / 256;
  const int kb = (width + 63) / 64;
  return std::max(1, std::min(std::min(8, kb / 8), 74 / std::max(1, tiles)));
}
static size_t split_pool_floats(const Dims& d) {
  size_t n = 0;
  auto add = [&](int out_f, int in_f, int passes, int rows) {
    const int S = split_factor(out_f, in_f, passes, rows);
    if (S > 1) n += (size_t)S * out_f * in_f;
  };
  const int hw = d.gates ? d.Gd : d.F;
  if (d.ints) { add(d.C, hw, 3, d.Ni); add(d.C, 1, 2, d.Ni); }
  if (d.ctx) { add(d.R, d.F, 3, d.Ni); add(d.R, 1, 2, d.Ni); }
  if (d.gates) { add(d.Gd, d.F, 3, d.Ni); add(d.Gd, d.F, 3, d.Ni); add(d.Gd, 1, 2, d.Ni); }
  for (int br = d.br0; br < (d.ctx ? 2 : 1); ++br) {
    const int ncl = br ? d.nc : d.nci, ntr = br ? d.nt : d.nti;
    for (int s = 0; s < 4; ++s) {
      if (!d.act[s]) continue;
      add(d.outw[s], d.J, 3, d.Ni); add(d.outw[s], 1, 2, d.Ni);
      const int nu = (s < 2) ? ncl : ntr;
      add(d.J, d.inw[s], 2, nu); add(d.J, 1, 2, nu);
    }
  }
  // forward reuses the pool for the split interaction head (backward starts after forward has drained it)
  const int hs = d.ints ? head_split(d.Ni, hw) : 1;
  if (hs > 1) n = std::max(n, (size_t)hs * d.Ni * d.C);
  return n;
}

static Workspace carve(const Dims& d, void* base) {
  Workspace w;
  size_t off = 0;
  auto take = [&](size_t bytes) -> void* {
    void* p = base ? static_cast<char*>(base) + off : nullptr;
    off += (size_t)round_up((int64_t)std::max<size_t>(bytes, 16), 256);
    return p;
  };
  const int nbr = d.ctx ? 2 : 1;
  for (int br = 0; br < 2; ++br)
    for (int s = 0; s < 4; ++s) {
      w.r1[br][s] = nullptr;
      w.dz1T[br][s] = nullptr;
      w.l2T[br][s] = nullptr;
    }
  w.a2[0] = w.f2[0] = w.dz2T[0] = nullptr;
  w.a2[1] = w.f2[1] = w.dz2T[1] = nullptr;
  w.da2[0] = w.da2[1] = nullptr;
  for (int br = d.br0; br < nbr; ++br) {
    const int ncl = br ? d.nc : d.nci, ntr = br ? d.nt : d.nti;
    for (int s = 0; s < 4; ++s) {
      if (!d.act[s]) continue;
      const int nu = (s < 2) ? ncl : ntr;
      const int nuP = (s < 2) ? d.ncP[br] : d.ntP[br];
      w.r1[br][s] = static_cast<float*>(take((size_t)nu * d.J * 4));
      w.dz1T[br][s] = static_cast<bf16*>(take((size_t)2 * d.J * nuP * 2));
      w.l2T[br][s] = static_cast<bf16*>(take((size_t)d.J * d.outw[s] * 2));
    }
    w.a2[br] = static_cast<bf16*>(take((size_t)d.Ni * 8 * d.J * 2));
    w.f2[br] = static_cast<bf16*>(take((size_t)d.Ni * 2 * d.F * 2));
    w.dz2T[br] = static_cast<bf16*>(take((size_t)2 * d.F * d.NiP * 2));
    w.da2[br] = static_cast<float*>(take((size_t)d.Ni * 4 * d.J * 4));
  }
  w.flag_c = static_cast<int32_t*>(take((size_t)d.Ni * 4));
  w.flagT = static_cast<bf16*>(take((size_t)d.NiP * 2));
  w.onesT = static_cast<bf16*>(take((size_t)d.onesP * 2));
  w.g2 = static_cast<bf16*>(take((size_t)d.Ni * 2 * d.Gd * 2));
  w.dpregT = static_cast<bf16*>(take((size_t)2 * d.Gd * d.NiP * 2));
  w.dliT = static_cast<bf16*>(take((size_t)2 * d.CP * d.NiP * 2));
  w.dlrT = static_cast<bf16*>(take((size_t)2 * d.RP * d.NiP * 2));
  w.out_intsT = static_cast<bf16*>(take((size_t)(d.gates ? d.Gd : d.F) * d.CP * 2));
  w.out_ctxT = static_cast<bf16*>(take((size_t)d.F * d.RP * 2));
  w.gateT = static_cast<bf16*>(take((size_t)2 * d.F * d.Gd * 2));
  w.pool_floats = split_pool_floats(d);
  w.pool = static_cast<float*>(take(w.pool_floats * 4));
  for (int br = 0; br < 2; ++br)
    for (int s = 0; s < 4; ++s) {
      w.sgn[br][s] = nullptr;
      if (br >= d.br0 && br < nbr && d.act[s]) {
        const int nu = (s < 2) ? (br ? d.nc : d.nci) : (br ? d.nt : d.nti);
        w.sgn[br][s] = static_cast<uint32_t*>(take((size_t)nu * (d.J / 32) * 4));
      }
    }
  for (int y = 0; y < 3; ++y) {            // appended last: lirec_model_workspace_layout keeps its indices
    w.ref_out[y] = d.ctx ? static_cast<int32_t*>(take((size_t)d.Nx * 4)) : nullptr;
    w.ref_w[y] = d.ctx ? static_cast<float*>(take((size_t)d.Nx * 4)) : nullptr;
  }
  w.bytes = off;
  return w;
}

__global__ void fill_bf16_kernel(bf16* p, int64_t n, float v) {
  pdl_wait();
  pdl_trigger();
  const bf16 b = __float2bfloat16_rn(v);
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    p[i] = b;
}

struct ReduceJob {
  float* dst;
  const float* src;
  int32_t M, N, S;
  int64_t dst_ld;
};
constexpr int MAX_REDUCE_JOBS = 96;
struct ReduceJobs {
  ReduceJob job[MAX_REDUCE_JOBS];
  int32_t n;
};
// One thread sums one group of four consecutive elements over the S partial slices (S independent
// 128-bit loads in flight), so the big first-layer jobs stream at HBM rate; blockIdx.y selects the job
// and CTAs beyond a job's size exit at once.
__global__ void __launch_bounds__(256) reduce_partials_kernel(const ReduceJobs jobs) {
  pdl_wait();
  pdl_trigger();
  const ReduceJob& j = jobs.job[blockIdx.y];
  const int64_t total = (int64_t)j.M * j.N;
  const bool vec = (j.N % 4 == 0) && (j.dst_ld % 4 == 0) && (total % 4 == 0) &&
                   ((reinterpret_cast<uintptr_t>(j.src) | reinterpret_cast<uintptr_t>(j.dst)) & 15) == 0;
  if (vec) {
    const int64_t i = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) * 4;
    if (i >= total) return;
    float4 acc = *reinterpret_cast<const float4*>(j.src + i);
    for (int s = 1; s < j.S; ++s) {
      const float4 v = *reinterpret_cast<const float4*>(j.src + (int64_t)s * total + i);
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    const int m = (int)(i / j.N), n = (int)(i - (int64_t)m * j.N);
    *reinterpret_cast<float4*>(j.dst + (int64_t)m * j.dst_ld + n) = acc;
  } else {
    const bool contiguous = j.dst_ld == j.N;     // no (m, n) decomposition: 64-bit divisions dominate otherwise
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
      float acc = 0.f;
      for (int s = 0; s < j.S; ++s) acc += j.src[(int64_t)s * total + i];
      if (contiguous) {
        j.dst[i] = acc;
      } else {
        const int m = (int)(i / j.N), n = (int)(i - (int64_t)m * j.N);
        j.dst[(int64_t)m * j.dst_ld + n] = acc;
      }
    }
  }
}

struct SplitCtx {
  float* pool;
  size_t pool_floats, used;
  ReduceJobs jobs;
};

// ---- small builders --------------------------------------------------------
static lirec_operand op(const void* p, int64_t rows, int64_t cols, int64_t ld) {
  lirec_operand o;
  o.ptr = p; o.rows = rows; o.cols = cols; o.ld = ld;
  return o;
}
static lirec_gemm_pass mk_pass(lirec_operand a, int a_mn, int a_k, lirec_operand b, int b_mn, int b_k, int k_len) {
  lirec_gemm_pass s;
  s.a = a; s.b = b;
  s.a_mn_off = a_mn; s.a_k_off = a_k; s.b_mn_off = b_mn; s.b_k_off = b_k;
  s.k_len = k_len;
  return s;
}
static lirec_gemm_problem mk_problem(int M, int N, bool a_mn, bool b_mn) {
  lirec_gemm_problem g;
  memset(&g, 0, sizeof(g));
  g.M = M; g.N = N;
  g.a_mn_major = a_mn; g.b_mn_major = b_mn;
  g.epi.alpha = 1.0f;
  g.epi.post_scale = 1.0f;
  g.epi.out_ld_n = 1;
  return g;
}
static void add_pass(lirec_gemm_problem& g, const lirec_gemm_pass& s) { g.pass[g.num_passes++] = s; }
static void out_f32(lirec_gemm_problem& g, float* out, int64_t ld_m, int64_t ld_n = 1) {
  g.epi.out_kind = LIREC_OUT_F32;
  g.epi.out = out; g.epi.out_ld_m = ld_m; g.epi.out_ld_n = ld_n;
}
static void out_split(lirec_gemm_problem& g, bf16* out, int64_t ld, int col_off, int lo_off) {
  g.epi.out_kind = LIREC_OUT_SPLIT_BF16;
  g.epi.out = out; g.epi.out_ld_m = ld; g.epi.out_col_off = col_off; g.epi.out_lo_off = lo_off;
}
static lirec_dropout mk_drop(float p, uint32_t seed, uint32_t stream_id, int col_off) {
  lirec_dropout d;
  d.p = p; d.seed = seed; d.stream_id = stream_id; d.col_off = col_off;
  return d;
}

static int validate(const lirec_model_cfg* cfg, const lirec_model_params* P, const lirec_batch* B,
                    const void* ws, size_t ws_bytes) {
  LIREC_REQUIRE(cfg && P && B && ws, "model: null argument");
  LIREC_REQUIRE(cfg->joint_dim > 0 && cfg->joint_dim % 128 == 0, "model: joint_dim=%d must be a multiple of 128",
                cfg->joint_dim);
  LIREC_REQUIRE(cfg->text_dim % 8 == 0 && cfg->visual_dim % 8 == 0 && cfg->track_dim % 8 == 0,
                "model: feature dims must be multiples of 8");
  LIREC_REQUIRE(!cfg->gates || cfg->ctx, "model: gates need the context branch");
  LIREC_REQUIRE(!cfg->no_ints || (cfg->ctx && !cfg->gates),
                "model: without the interaction branch (opt.ints = 0) the model is the context branch and its "
                "relationship head alone: ctx = 1, gates = 0 (the reference's GatingUnit needs both, model.py:349-352)");
  LIREC_REQUIRE(!cfg->ctx || (cfg->slot_mask & 15) == 0 || (cfg->slot_mask & 15) == 15,
                "model: the context models always use all four modality slots (slot_mask=%d)", cfg->slot_mask);
  LIREC_REQUIRE(!cfg->gates || cfg->gate_dim % 8 == 0, "model: gate_dim=%d", cfg->gate_dim);
  LIREC_REQUIRE((cfg->no_ints || cfg->n_classes > 0) && (!cfg->ctx || cfg->n_rels > 0), "model: n_classes=%d n_rels=%d",
                cfg->n_classes, cfg->n_rels);
  LIREC_REQUIRE(B->n_cand > 0, "model: empty batch");
  LIREC_REQUIRE(B->n_clip_ints > 0 && B->n_track_ints > 0 && B->n_clip >= B->n_clip_ints &&
                    B->n_track >= B->n_track_ints,
                "model: bank sizes clip %d/%d track %d/%d", B->n_clip_ints, B->n_clip, B->n_track_ints,
                B->n_track);
  LIREC_REQUIRE(B->clip_bank && B->track_bank && B->cand_rows, "model: null batch table");
  LIREC_REQUIRE(!cfg->ctx || (B->ctx_off && (B->n_ctx_rows == 0 || (B->ctx_rows && B->ctx_owner))),
                "model: context tables missing");
  LIREC_REQUIRE(cfg->dropout_p >= 0.f && cfg->dropout_p < 1.f, "model: dropout_p=%f", cfg->dropout_p);
  const Dims d = make_dims(*cfg, *B);
  const Workspace w = carve(d, nullptr);
  LIREC_REQUIRE(ws_bytes >= w.bytes, "model: workspace %zu < required %zu bytes", ws_bytes, w.bytes);
  LIREC_REQUIRE((reinterpret_cast<uintptr_t>(ws) & 255) == 0, "model: workspace must be 256-byte aligned");
  return LIREC_OK;
}

// Below this many candidate rows backward multiplies by the weights in place instead of transposing them.
static bool dgrad_in_place(int Ni) {
  const char* e = getenv("LIREC_DGRAD_INPLACE_ROWS");   // read per call: the tests switch it
  return Ni < (e ? atoi(e) : 1536);
}

// ---- [in, out] copies of the weights the data gradients multiply by (K-major B operands) ----------------
static int weight_transposes(const Dims& d, const lirec_model_params& P, const Workspace& w, cudaStream_t stream) {
  const int nbr = d.ctx ? 2 : 1;
  const int hw = d.gates ? d.Gd : d.F;
  rows::TransposeJobs tj;
  tj.n = 0;
  auto add = [&](const void* src, int out_f, int in_f, bf16* dst, int out_p) {
    rows::TransposeJob& j = tj.job[tj.n++];
    j.src = static_cast<const bf16*>(src); j.src_ld = in_f; j.R = out_f; j.C = in_f;
    j.dst = dst; j.dst_ld = out_p; j.Rp = out_p;
  };
  if (d.ints) add(P.out_ints.w_bf16, d.C, hw, w.out_intsT, d.CP);
  if (d.ctx) add(P.out_ctx.w_bf16, d.R, d.F, w.out_ctxT, d.RP);
  if (d.gates) add(P.gate.w_bf16, d.Gd, 2 * d.F, w.gateT, d.Gd);
  for (int br = d.br0; br < nbr; ++br)
    for (int s = 0; s < 4; ++s)
      if (d.act[s])
        add((br ? P.enc_ctx : P.enc_ints).l2[s].w_bf16, d.outw[s], d.J, w.l2T[br][s], d.outw[s]);
  return rows::transpose_bf16(tj, stream);
}

// The copies only depend on the weights, which are final when forward starts: a TRAINING forward launches them on
// a side stream of the library's own, next to the forward GEMMs, and leaves a note for the backward call on the
// same workspace, which then just waits for them (29 us off the critical path of a 1024-clip step).  A backward
// without that note (eval-mode autograd, another workspace) transposes inline.
static int context_ref_tables(const Dims& d, const lirec_batch& B, const Workspace& w, cudaStream_t stream) {
  rows::RefTableJobs rj;
  for (int y = 0; y < 3; ++y) {
    rj.inv_idx[y] = B.inv_ctx_idx[y];
    rj.ref_out[y] = w.ref_out[y];
    rj.ref_w[y] = w.ref_w[y];
  }
  rj.owner = B.ctx_owner;
  rj.seg_off = B.ctx_off;
  rj.n = d.Nx;
  return rows::ref_tables(rj, stream);
}
static bool has_ref_inputs(const Dims& d, const lirec_batch& B) {
  return d.ctx && d.Nx > 0 && B.ctx_owner && B.ctx_off && B.inv_ctx_idx[0] && B.inv_ctx_idx[1] && B.inv_ctx_idx[2];
}

struct SideTranspose {
  cudaStream_t stream = nullptr;
  cudaEvent_t in = nullptr, out = nullptr;
  const void* ws = nullptr;      // workspace whose W^T copies are in flight / done
  bool refs = false;             // ... and whose per-reference tables were built next to them
  int device = -1;
};
static thread_local SideTranspose g_side;

static bool side_ready() {
  int dev = -1;
  if (cudaGetDevice(&dev) != cudaSuccess) return false;
  if (g_side.stream && g_side.device == dev) return true;
  if (g_side.stream) return false;   // created for another device: keep it simple, inline on this one
  if (cudaStreamCreateWithFlags(&g_side.stream, cudaStreamNonBlocking) != cudaSuccess) return false;
  if (cudaEventCreateWithFlags(&g_side.in, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&g_side.out, cudaEventDisableTiming) != cudaSuccess) {
    g_side.stream = nullptr;
    return false;
  }
  g_side.device = dev;
  return true;
}

// ---------------------------------------------------------------------------
int forward(const lirec_model_cfg& cfg, const lirec_model_params& P, const lirec_batch& B, void* ws,
            float* out_ints, float* out_rels, cudaStream_t stream) {
  const Dims d = make_dims(cfg, B);
  const Workspace w = carve(d, ws);
  const float p = (B.training && cfg.dropout_p > 0.f) ? cfg.dropout_p : 0.f;
  const float keep_scale = 1.0f / (1.0f - p);
  const int nbr = d.ctx ? 2 : 1;
  const int J = d.J, F = d.F;
  int rc;

  g_side.ws = nullptr;
  if (B.training && !dgrad_in_place(d.Ni) && side_ready()) {
    LIREC_CUDA_OK(cudaEventRecord(g_side.in, stream));                 // weights (last Adam) are final here
    LIREC_CUDA_OK(cudaStreamWaitEvent(g_side.stream, g_side.in, 0));
    if ((rc = weight_transposes(d, P, w, g_side.stream)) != LIREC_OK) return rc;
    g_side.refs = has_ref_inputs(d, B);       // index tables only: nothing of this step's forward is needed
    if (g_side.refs && (rc = context_ref_tables(d, B, w, g_side.stream)) != LIREC_OK) return rc;
    LIREC_CUDA_OK(cudaEventRecord(g_side.out, g_side.stream));
    g_side.ws = ws;
  }

  {  // ones column for the bias-gradient GEMMs
    const int64_t n = d.onesP;
    LIREC_CUDA_OK(launch_pdl(fill_bf16_kernel, dim3((unsigned)std::min<int64_t>((n + 255) / 256, 1184)), dim3(256), 0, stream, w.onesT, n, 1.0f));
    note_launch();
  }

  // ---- layer 1 on the unique bank rows: relu(x W1^T + b1) -------------------
  std::vector<lirec_gemm_problem> pr;
  for (int br = d.br0; br < nbr; ++br) {
    const lirec_encoder& enc = br ? P.enc_ctx : P.enc_ints;
    const int ncl = br ? d.nc : d.nci, ntr = br ? d.nt : d.nti;
    for (int s = 0; s < 4; ++s) {
      if (!d.act[s]) continue;
      const int nu = (s < 2) ? ncl : ntr;
      lirec_operand a;
      if (s == 0) a = op(B.clip_bank, nu, d.inw[0], B.clip_ld);
      else if (s == 1) a = op(static_cast<const bf16*>(B.clip_bank) + d.inw[0], nu, d.inw[1], B.clip_ld);
      else a = op(B.track_bank, nu, d.inw[s], B.track_ld);
      lirec_gemm_problem g = mk_problem(nu, J, false, false);
      add_pass(g, mk_pass(a, 0, 0, op(enc.l1[s].w_bf16, J, d.inw[s], d.inw[s]), 0, 0, d.inw[s]));
      g.epi.bias = enc.l1[s].bias;
      g.epi.act = LIREC_ACT_RELU;
      out_f32(g, w.r1[br][s], J);
      g.epi.post = LIREC_POST_SIGN_MASK;     // the gate of relu, 1 bit per element, for backward's scatter-reduce
      g.epi.aux = w.sgn[br][s];
      g.epi.aux_ld = J / 32;
      pr.push_back(g);
    }
  }
  if ((rc = gemm::run_grouped(pr.data(), (int)pr.size(), stream)) != LIREC_OK) return rc;

  // ---- expansion to encoder rows (+ masked mean for the context branch) ------
  {
    rows::ExpandFwdJobs jobs;
    memset(&jobs, 0, sizeof(jobs));
    jobs.n = nbr - d.br0;
    for (int br = d.br0; br < nbr; ++br) {
      rows::ExpandFwdJob& j = jobs.job[br - d.br0];
      for (int s = 0; s < 4; ++s) j.r1[s] = w.r1[br][s];
      j.J = J;
      j.rows = br ? B.ctx_rows : B.cand_rows;
      j.seg_off = br ? B.ctx_off : nullptr;
      j.n_out = d.Ni;
      j.guard_zero = cfg.guard_zero;
      j.drop = mk_drop(p, B.seed, br ? DS_L1_CTX : DS_L1_INTS, 0);
      j.out = w.a2[br];
      j.out_ld = 8 * J;
      j.row_flag_out = br ? w.flag_c : nullptr;
      j.flag_bf16_out = br ? w.flagT : nullptr;
    }
    if ((rc = rows::expand_fwd(jobs, stream)) != LIREC_OK) return rc;
  }

  // ---- layer 2 + tanh + dropout into the concat slices -------------------------
  pr.clear();
  for (int br = d.br0; br < nbr; ++br) {
    const lirec_encoder& enc = br ? P.enc_ctx : P.enc_ints;
    for (int s = 0; s < 4; ++s) {
      if (!d.act[s]) continue;
      lirec_gemm_problem g = mk_problem(d.Ni, d.outw[s], false, false);
      const lirec_operand a = op(w.a2[br] + s * 2 * J, d.Ni, 2 * J, 8 * J);
      const lirec_operand b = op(enc.l2[s].w_bf16, d.outw[s], J, J);
      add_pass(g, mk_pass(a, 0, 0, b, 0, 0, J));
      add_pass(g, mk_pass(a, 0, J, b, 0, 0, J));
      g.epi.alpha = keep_scale;  // the 1/(1-p) of the layer-1 dropout
      g.epi.bias = enc.l2[s].bias;
      g.epi.row_flag = br ? w.flag_c : nullptr;
      g.epi.act = LIREC_ACT_TANH;
      g.epi.post = LIREC_POST_DROPOUT;
      g.epi.drop = mk_drop(p, B.seed, br ? DS_CAT_CTX : DS_CAT_INTS, d.cs[s]);
      out_split(g, w.f2[br], 2 * F, d.cs[s], F);
      pr.push_back(g);
    }
  }
  if ((rc = gemm::run_grouped(pr.data(), (int)pr.size(), stream)) != LIREC_OK) return rc;

  // ---- gate (+ relationship head, which only needs the context feature) ----------
  pr.clear();
  if (d.gates) {
    lirec_gemm_problem g = mk_problem(d.Ni, d.Gd, false, false);
    const lirec_operand fc = op(w.f2[1], d.Ni, 2 * F, 2 * F), fi = op(w.f2[0], d.Ni, 2 * F, 2 * F);
    const lirec_operand wg = op(P.gate.w_bf16, d.Gd, 2 * F, 2 * F);
    add_pass(g, mk_pass(fc, 0, 0, wg, 0, 0, F));  // cat order (rels, inters): model.py:352
    add_pass(g, mk_pass(fc, 0, F, wg, 0, 0, F));
    add_pass(g, mk_pass(fi, 0, 0, wg, 0, F, F));
    add_pass(g, mk_pass(fi, 0, F, wg, 0, F, F));
    g.epi.bias = P.gate.bias;
    g.epi.act = LIREC_ACT_RELU;
    g.epi.post = LIREC_POST_DROPOUT;
    g.epi.drop = mk_drop(p, B.seed, DS_GATE, 0);
    out_split(g, w.g2, 2 * d.Gd, 0, d.Gd);
    pr.push_back(g);
  }
  if (d.ctx) {
    LIREC_REQUIRE(out_rels != nullptr, "model: out_rels is null");
    lirec_gemm_problem g = mk_problem(d.Ni, d.R, false, false);
    const lirec_operand fc = op(w.f2[1], d.Ni, 2 * F, 2 * F);
    const lirec_operand wo = op(P.out_ctx.w_bf16, d.R, F, F);
    add_pass(g, mk_pass(fc, 0, 0, wo, 0, 0, F));
    add_pass(g, mk_pass(fc, 0, F, wo, 0, 0, F));
    g.epi.bias = P.out_ctx.bias;
    out_f32(g, out_rels, d.R);
    pr.push_back(g);
  }
  if (!pr.empty() && (rc = gemm::run_grouped(pr.data(), (int)pr.size(), stream)) != LIREC_OK) return rc;

  // ---- interaction head -----------------------------------------------------------
  pr.clear();
  if (d.ints) {
    LIREC_REQUIRE(out_ints != nullptr, "model: out_ints is null");
    const int width = d.gates ? d.Gd : F;
    const bf16* x = d.gates ? w.g2 : w.f2[0];
    lirec_gemm_problem g = mk_problem(d.Ni, d.C, false, false);
    const lirec_operand a = op(x, d.Ni, 2 * width, 2 * width);
    const lirec_operand wo = op(P.out_ints.w_bf16, d.C, width, width);
    add_pass(g, mk_pass(a, 0, 0, wo, 0, 0, width));
    add_pass(g, mk_pass(a, 0, width, wo, 0, 0, width));
    g.epi.bias = P.out_ints.bias;
    out_f32(g, out_ints, d.C);
    // One column of 256-row tiles (C <= 128) leaves most clusters idle and every busy SM pulling its
    // 2 x width K-range at per-SM bandwidth: split K so the launch covers the machine, and add the
    // partial [Ni, C] outputs up afterwards (bias rides in slice 0).
    const int S = head_split(d.Ni, width);
    ReduceJobs jobs;
    jobs.n = 0;
    if (S > 1 && (size_t)S * d.Ni * d.C <= w.pool_floats) {
      ReduceJob& j = jobs.job[jobs.n++];
      j.dst = out_ints; j.dst_ld = d.C; j.src = w.pool; j.M = d.Ni; j.N = d.C;
      j.S = gemm::split_k_slices((width + 63) / 64, S);
      g.split_k = S;
      g.split_stride = (int64_t)d.Ni * d.C;
      g.epi.out = w.pool;
    }
    pr.push_back(g);
    if ((rc = gemm::run_grouped(pr.data(), (int)pr.size(), stream)) != LIREC_OK) return rc;
    if (jobs.n > 0) {
      const int64_t total = (int64_t)d.Ni * d.C;
      dim3 grid((unsigned)((total + 1023) / 1024), jobs.n);
      LIREC_CUDA_OK(launch_pdl(reduce_partials_kernel, grid, dim3(256), 0, stream, jobs));
      note_launch();
    }
  }
  return LIREC_OK;
}

// ---------------------------------------------------------------------------
// Backward GEMM builders.  TGrad = a transposed hi/lo gradient tensor: rows [hi, hi + n) hold the hi
// parts of n features, rows [lo, lo + n) the lo parts, every row is `rows` batch rows long.
struct TGrad {
  const bf16* ptr;
  int buf_rows;      // rows of the whole buffer (for the tensor map)
  int64_t pitch;
  int hi, lo;
};

// Weight gradient dW[out_f, in_f] = alpha * dY^T X, run as D'[in_f, out_f] = X^T dY:
//   A = X  [rows, x_cols] natural, read MN-major (x_lo < 0: exact bf16, no lo part)
//   B = dY^T (TGrad) K-major
// and stored transposed into dW (lanes run along in_f, so the fp32 stores stay coalesced).
static lirec_gemm_problem wgrad_t(int out_f, int in_f, const TGrad& dy, const bf16* x, int64_t x_cols, int64_t x_ld,
                                  int x_hi, int x_lo, int rows, float alpha, float* grad, int64_t grad_ld) {
  lirec_gemm_problem g = mk_problem(in_f, out_f, true, false);
  const lirec_operand a = op(x, rows, x_cols, x_ld);
  const lirec_operand b = op(dy.ptr, dy.buf_rows, rows, dy.pitch);
  add_pass(g, mk_pass(a, x_hi, 0, b, dy.hi, 0, rows));
  if (x_lo >= 0) add_pass(g, mk_pass(a, x_lo, 0, b, dy.hi, 0, rows));
  add_pass(g, mk_pass(a, x_hi, 0, b, dy.lo, 0, rows));
  g.epi.alpha = alpha;
  out_f32(g, grad, 1, grad_ld);
  return g;
}
// bias gradient db[out_f] = dY^T v with v = ones or the 0/1 row flags, both [1, rows] K-major
static lirec_gemm_problem bgrad_t(int out_f, const TGrad& dy, const bf16* v, int rows, float* grad) {
  lirec_gemm_problem g = mk_problem(out_f, 1, false, false);
  const lirec_operand a = op(dy.ptr, dy.buf_rows, rows, dy.pitch);
  const lirec_operand b = op(v, 1, rows, round_up(rows, 64));
  add_pass(g, mk_pass(a, dy.hi, 0, b, 0, 0, rows));
  add_pass(g, mk_pass(a, dy.lo, 0, b, 0, 0, rows));
  out_f32(g, grad, 1);
  return g;
}
// data-gradient passes dX[rows, in_f] += dY W: A = dY^T (TGrad) read MN-major, B = W^T [in_f.., out_p] K-major
static void add_dgrad_passes(lirec_gemm_problem& g, const TGrad& dy, int rows, const bf16* wT, int wT_rows,
                             int out_p, int w_row_off, int k_len) {
  const lirec_operand a = op(dy.ptr, dy.buf_rows, rows, dy.pitch);
  const lirec_operand b = op(wT, wT_rows, out_p, out_p);
  add_pass(g, mk_pass(a, 0, dy.hi, b, w_row_off, 0, k_len));
  add_pass(g, mk_pass(a, 0, dy.lo, b, w_row_off, 0, k_len));
}
// The same passes against the weight IN PLACE: B = W [out_f, in_total] read MN-major (columns
// [in_off, in_off + N) of W are the problem's N).  Slower per tile than the K-major W^T copy, but it needs
// no per-step transposes (28 us for the 11 M second-layer / gate / head weights): what small batches
// want.  Rows of dY^T beyond out_f are zero (split_f32_t pads) and rows of W beyond out_f are TMA zero fill.
static void add_dgrad_passes_inplace(lirec_gemm_problem& g, const TGrad& dy, int rows, const void* w_bf16, int out_f,
                                     int in_total, int in_off) {
  const lirec_operand a = op(dy.ptr, dy.buf_rows, rows, dy.pitch);
  const lirec_operand b = op(w_bf16, out_f, in_total, in_total);
  g.b_mn_major = 1;
  add_pass(g, mk_pass(a, 0, dy.hi, b, in_off, 0, out_f));
  add_pass(g, mk_pass(a, 0, dy.lo, b, in_off, 0, out_f));
}
static void out_split_t(lirec_gemm_problem& g, bf16* out, int64_t pitch, int row_off, int lo_off) {
  g.epi.out_kind = LIREC_OUT_SPLIT_BF16_T;
  g.epi.out = out; g.epi.out_ld_m = pitch; g.epi.out_col_off = row_off; g.epi.out_lo_off = lo_off;
}

// Push a reduction-over-rows problem producing a [out_f, in_f] parameter gradient, split-K if that helps.
// The problem stores element (o, i) at out[o * ld + i] through (out_ld_m, out_ld_n); the pool slices use
// the same indexing with ld = in_f.
static void push_reduction(std::vector<lirec_gemm_problem>& pr, lirec_gemm_problem g, int out_f, int in_f, int rows,
                           bool transposed, SplitCtx& sc) {
  const int S = split_factor(out_f, in_f, g.num_passes, rows);
  const size_t need = (size_t)S * out_f * in_f;
  if (S > 1 && sc.used + need <= sc.pool_floats && sc.jobs.n < MAX_REDUCE_JOBS) {
    ReduceJob& j = sc.jobs.job[sc.jobs.n++];
    j.dst = static_cast<float*>(g.epi.out);
    j.dst_ld = transposed ? g.epi.out_ld_n : g.epi.out_ld_m;
    j.src = sc.pool + sc.used;
    j.M = out_f; j.N = in_f;
    j.S = gemm::split_k_slices((rows + 63) / 64, S);     // the slice count the GEMM will actually use
    g.split_k = S;
    g.split_stride = (int64_t)out_f * in_f;
    g.epi.out = sc.pool + sc.used;
    if (transposed) { g.epi.out_ld_m = 1; g.epi.out_ld_n = in_f; }
    else { g.epi.out_ld_m = in_f; g.epi.out_ld_n = 1; }
    sc.used += need;
  }
  pr.push_back(g);
}

// Sum the split-K partials collected so far into the flat gradient buffer (fixed order) and start a new list.
static int flush_partials(SplitCtx& sc, cudaStream_t stream) {
  if (sc.jobs.n > 0) {
    int64_t biggest = 0;
    for (int i = 0; i < sc.jobs.n; ++i) biggest = std::max<int64_t>(biggest, (int64_t)sc.jobs.job[i].M * sc.jobs.job[i].N);
    dim3 grid((unsigned)((biggest + 1023) / 1024), sc.jobs.n);
    LIREC_CUDA_OK(launch_pdl(reduce_partials_kernel, grid, dim3(256), 0, stream, sc.jobs));
    note_launch();
    sc.jobs.n = 0;
  }
  return LIREC_OK;
}

// heads_event (optional): recorded on `stream` as soon as the gradients of the gate and of the two heads are
// FINAL in the flat gradient buffer (after stage G and its split-K sums; after stage H for the models without
// a gate) — the data-parallel exchange and the Adam pass of those parameters (53 % of all weights) can then
// run on another stream while the encoder stages of backward are still going (lirec_b200/dp.py).
int backward(const lirec_model_cfg& cfg, const lirec_model_params& P, const lirec_batch& B, void* ws,
             const float* d_ints, const float* d_rels, cudaStream_t stream, cudaEvent_t heads_event) {
  const Dims d = make_dims(cfg, B);
  const Workspace w = carve(d, ws);
  const float p = (B.training && cfg.dropout_p > 0.f) ? cfg.dropout_p : 0.f;
  const float keep_scale = 1.0f / (1.0f - p);
  const int nbr = d.ctx ? 2 : 1;
  const int J = d.J, F = d.F, Ni = d.Ni, Gd = d.Gd, CP = d.CP, RP = d.RP, NiP = d.NiP;
  int rc;
  LIREC_REQUIRE((!d.ints || d_ints != nullptr) && (!d.ctx || d_rels != nullptr), "model backward: null logit gradient");
  for (int s = 0; s < 3; ++s) {
    LIREC_REQUIRE(!d.ints || (B.inv_cand_off[s] && B.inv_cand_idx[s]), "model backward: inverse candidate tables missing");
    LIREC_REQUIRE(!d.ctx || (B.inv_ctx_off[s] && (d.Nx == 0 || B.inv_ctx_idx[s])),
                  "model backward: inverse context tables missing");
  }
  const int hw = d.gates ? Gd : F;                 // width of the interaction head's input
  const bf16* hx = d.gates ? w.g2 : w.f2[0];

  // ---- [in, out] copies of the weights the data gradients multiply by ---------------------------
  const bool inplace = dgrad_in_place(Ni);
  bool refs_ready = false;
  if (!inplace) {
    if (g_side.ws == ws && g_side.stream) {               // launched next to this workspace's forward
      LIREC_CUDA_OK(cudaStreamWaitEvent(stream, g_side.out, 0));
      g_side.ws = nullptr;
      refs_ready = g_side.refs;
    } else if ((rc = weight_transposes(d, P, w, stream)) != LIREC_OK) {
      return rc;
    }
  }
  // per-reference tables: used when forward built them on the side stream (a few us off expand_bwd_t); building
  // them inline would cost what they save
  const bool use_refs = refs_ready && has_ref_inputs(d, B);

  SplitCtx sc;
  sc.pool = w.pool; sc.pool_floats = w.pool_floats; sc.used = 0; sc.jobs.n = 0;
  if (d.ints && (rc = rows::split_f32_t(d_ints, d.C, Ni, d.C, w.dliT, NiP, CP, stream)) != LIREC_OK) return rc;
  if (d.ctx && (rc = rows::split_f32_t(d_rels, d.R, Ni, d.R, w.dlrT, NiP, RP, stream)) != LIREC_OK) return rc;
  const TGrad dli{w.dliT, 2 * CP, NiP, 0, CP};
  const TGrad dlr{w.dlrT, 2 * RP, NiP, 0, RP};
  const TGrad dpg{w.dpregT, 2 * Gd, NiP, 0, Gd};

  // ---- stage H: head wgrad/bgrad + dgrad through the head --------------------
  // The head parameter gradients have no consumer inside backward: with a gate they ride in stage G's launch,
  // where their long memory-bound reductions (the [101, 3072] gradient streams the whole gate output) fill the
  // schedule next to the gate's compute-bound tiles instead of stretching this short launch.
  std::vector<lirec_gemm_problem> pr, head_red;
  std::vector<lirec_gemm_problem>& hr = d.gates ? head_red : pr;
  if (d.ints) {
    push_reduction(hr, wgrad_t(d.C, hw, dli, hx, 2 * hw, 2 * hw, 0, hw, Ni, 1.f, P.out_ints.grad_w, hw), d.C, hw, Ni,
                   true, sc);
    push_reduction(hr, bgrad_t(d.C, dli, w.onesT, Ni, P.out_ints.grad_b), d.C, 1, Ni, false, sc);
  }
  if (d.ctx) {
    push_reduction(hr, wgrad_t(d.R, F, dlr, w.f2[1], 2 * F, 2 * F, 0, F, Ni, 1.f, P.out_ctx.grad_w, F), d.R, F, Ni,
                   true, sc);
    push_reduction(hr, bgrad_t(d.R, dlr, w.onesT, Ni, P.out_ctx.grad_b), d.R, 1, Ni, false, sc);
  }
  if (d.ints) {
    lirec_gemm_problem g = mk_problem(Ni, hw, true, false);
    if (inplace) add_dgrad_passes_inplace(g, dli, Ni, P.out_ints.w_bf16, d.C, hw, 0);
    else add_dgrad_passes(g, dli, Ni, w.out_intsT, hw, CP, 0, CP);
    if (d.gates) {
      g.epi.post = LIREC_POST_DRELU;  // through dropout(relu(.)) of the gate: model.py:353
      g.epi.post_scale = keep_scale;
      g.epi.aux = w.g2; g.epi.aux_ld = 2 * Gd; g.epi.aux_col_off = 0; g.epi.aux_lo_off = Gd;
      out_split_t(g, w.dpregT, NiP, 0, Gd);
    } else {
      g.epi.post = LIREC_POST_DTANH;  // through dropout(tanh(.)): model.py:297
      g.epi.drop = mk_drop(p, B.seed, DS_CAT_INTS, 0);
      g.epi.aux = w.f2[0]; g.epi.aux_ld = 2 * F; g.epi.aux_col_off = 0; g.epi.aux_lo_off = F;
      out_split_t(g, w.dz2T[0], NiP, 0, F);
    }
    pr.push_back(g);
  }
  if (d.ctx && !d.gates) {
    lirec_gemm_problem g = mk_problem(Ni, F, true, false);
    if (inplace) add_dgrad_passes_inplace(g, dlr, Ni, P.out_ctx.w_bf16, d.R, F, 0);
    else add_dgrad_passes(g, dlr, Ni, w.out_ctxT, F, RP, 0, RP);
    g.epi.post = LIREC_POST_DTANH;
    g.epi.drop = mk_drop(p, B.seed, DS_CAT_CTX, 0);
    g.epi.aux = w.f2[1]; g.epi.aux_ld = 2 * F; g.epi.aux_col_off = 0; g.epi.aux_lo_off = F;
    out_split_t(g, w.dz2T[1], NiP, 0, F);
    pr.push_back(g);
  }
  if ((rc = gemm::run_grouped(pr.data(), (int)pr.size(), stream)) != LIREC_OK) return rc;
  if (heads_event && !d.gates) {
    if ((rc = flush_partials(sc, stream)) != LIREC_OK) return rc;
    LIREC_CUDA_OK(cudaEventRecord(heads_event, stream));
  }

  // ---- stage G: gate wgrad/bgrad + dgrad to the two concat features --------------
  if (d.gates) {
    pr = head_red;
    for (int h = 0; h < 2; ++h)  // columns [0,F) multiply the context feature, [F,2F) the ints feature
      push_reduction(pr, wgrad_t(Gd, F, dpg, w.f2[h ? 0 : 1], 2 * F, 2 * F, 0, F, Ni, 1.f, P.gate.grad_w + h * F,
                                 2 * F), Gd, F, Ni, true, sc);
    push_reduction(pr, bgrad_t(Gd, dpg, w.onesT, Ni, P.gate.grad_b), Gd, 1, Ni, false, sc);
    for (int h = 0; h < 2; ++h) {
      const int br = h ? 0 : 1;
      lirec_gemm_problem g = mk_problem(Ni, F, true, false);
      if (inplace) add_dgrad_passes_inplace(g, dpg, Ni, P.gate.w_bf16, Gd, 2 * F, h * F);
      else add_dgrad_passes(g, dpg, Ni, w.gateT, 2 * F, Gd, h * F, Gd);
      if (br == 1) {  // the context feature also feeds the relationship head
        if (inplace) add_dgrad_passes_inplace(g, dlr, Ni, P.out_ctx.w_bf16, d.R, F, 0);
        else add_dgrad_passes(g, dlr, Ni, w.out_ctxT, F, RP, 0, RP);
      }
      g.epi.post = LIREC_POST_DTANH;
      g.epi.drop = mk_drop(p, B.seed, br ? DS_CAT_CTX : DS_CAT_INTS, 0);
      g.epi.aux = w.f2[br]; g.epi.aux_ld = 2 * F; g.epi.aux_col_off = 0; g.epi.aux_lo_off = F;
      out_split_t(g, w.dz2T[br], NiP, 0, F);
      pr.push_back(g);
    }
    if ((rc = gemm::run_grouped(pr.data(), (int)pr.size(), stream)) != LIREC_OK) return rc;
    if (heads_event) {
      if ((rc = flush_partials(sc, stream)) != LIREC_OK) return rc;
      LIREC_CUDA_OK(cudaEventRecord(heads_event, stream));
    }
  }

  // ---- stage L2: second-layer wgrad/bgrad + dgrad to the expanded rows ------------
  // Same deferral: the second-layer parameter gradients run in the first-layer launch (which only waits for the
  // scatter-reduce of this stage's DATA gradients), leaving this launch the eight short data-gradient GEMMs.
  pr.clear();
  std::vector<lirec_gemm_problem> l2_red;
  for (int br = d.br0; br < nbr; ++br) {
    const lirec_encoder& enc = br ? P.enc_ctx : P.enc_ints;
    for (int s = 0; s < 4; ++s) {
      if (!d.act[s]) continue;
      const TGrad dz{w.dz2T[br], 2 * F, NiP, d.cs[s], F + d.cs[s]};
      push_reduction(l2_red, wgrad_t(d.outw[s], J, dz, w.a2[br], 8 * J, 8 * J, s * 2 * J, s * 2 * J + J, Ni,
                                     keep_scale, enc.l2[s].grad_w, J), d.outw[s], J, Ni, true, sc);
      push_reduction(l2_red, bgrad_t(d.outw[s], dz, br ? w.flagT : w.onesT, Ni, enc.l2[s].grad_b), d.outw[s], 1,
                     Ni, false, sc);
      lirec_gemm_problem g = mk_problem(Ni, J, true, false);
      if (inplace) add_dgrad_passes_inplace(g, dz, Ni, enc.l2[s].w_bf16, d.outw[s], J, 0);
      else add_dgrad_passes(g, dz, Ni, w.l2T[br][s], J, d.outw[s], 0, d.outw[s]);
      g.epi.alpha = keep_scale;
      out_f32(g, w.da2[br] + s * J, 4 * J);
      pr.push_back(g);
    }
  }
  if ((rc = gemm::run_grouped(pr.data(), (int)pr.size(), stream)) != LIREC_OK) return rc;

  // ---- scatter-reduce onto the unique bank rows (through relu(dropout(.))) ---------
  {
    rows::ExpandBwdJobs jobs;
    memset(&jobs, 0, sizeof(jobs));
    int n = 0;
    for (int br = d.br0; br < nbr; ++br) {
      const int ncl = br ? d.nc : d.nci, ntr = br ? d.nt : d.nti;
      for (int s = 0; s < 4; ++s) {
        if (!d.act[s]) continue;
        rows::ExpandBwdJob& j = jobs.job[n++];
        const int inv = (s < 2) ? 0 : (s - 1);
        j.d_in = w.da2[br] + s * J;
        j.d_ld = 4 * J;
        j.sign = w.sgn[br][s];
        j.sign_ld = J / 32;
        j.J = J;
        j.slot = s;
        j.inv_off = br ? B.inv_ctx_off[inv] : B.inv_cand_off[inv];
        j.inv_idx = br ? B.inv_ctx_idx[inv] : B.inv_cand_idx[inv];
        j.n_unique = (s < 2) ? ncl : ntr;
        j.owner = br ? B.ctx_owner : nullptr;
        j.seg_off = br ? B.ctx_off : nullptr;
        j.ref_out = (br && use_refs) ? w.ref_out[inv] : nullptr;
        j.ref_w = (br && use_refs) ? w.ref_w[inv] : nullptr;
        j.drop = mk_drop(p, B.seed, br ? DS_L1_CTX : DS_L1_INTS, 0);
        j.out = w.dz1T[br][s];
        j.out_pitch = (s < 2) ? d.ncP[br] : d.ntP[br];
      }
    }
    jobs.n = n;
    if ((rc = rows::expand_bwd(jobs, stream)) != LIREC_OK) return rc;
  }

  // ---- stage L1: first-layer wgrad/bgrad on the unique rows (inputs carry no grad) ----
  pr = l2_red;
  for (int br = d.br0; br < nbr; ++br) {
    const lirec_encoder& enc = br ? P.enc_ctx : P.enc_ints;
    const int ncl = br ? d.nc : d.nci, ntr = br ? d.nt : d.nti;
    for (int s = 0; s < 4; ++s) {
      if (!d.act[s]) continue;
      const int nu = (s < 2) ? ncl : ntr;
      const int nuP = (s < 2) ? d.ncP[br] : d.ntP[br];
      const bf16* x;
      int64_t x_ld;
      if (s == 0) { x = static_cast<const bf16*>(B.clip_bank); x_ld = B.clip_ld; }
      else if (s == 1) { x = static_cast<const bf16*>(B.clip_bank) + d.inw[0]; x_ld = B.clip_ld; }
      else { x = static_cast<const bf16*>(B.track_bank); x_ld = B.track_ld; }
      const TGrad dz{w.dz1T[br][s], 2 * J, nuP, 0, J};
      push_reduction(pr, wgrad_t(J, d.inw[s], dz, x, d.inw[s], x_ld, 0, -1, nu, 1.f, enc.l1[s].grad_w, d.inw[s]), J,
                     d.inw[s], nu, true, sc);
      push_reduction(pr, bgrad_t(J, dz, w.onesT, nu, enc.l1[s].grad_b), J, 1, nu, false, sc);
    }
  }
  if ((rc = gemm::run_grouped(pr.data(), (int)pr.size(), stream)) != LIREC_OK) return rc;

  // ---- sum the split-K partials into the flat gradient buffer (fixed order) -----------------------
  return flush_partials(sc, stream);
}

}  // namespace model
}  // namespace lirec

using namespace lirec;

extern "C" size_t lirec_model_workspace_bytes(const lirec_model_cfg* cfg, const lirec_batch* batch_host) {
  if (!cfg || !batch_host) return 0;
  const model::Dims d = model::make_dims(*cfg, *batch_host);
  return model::carve(d, nullptr).bytes;
}

// Debug / white-box test aid: byte offsets of the workspace buffers, in the order
// r1[2][4], dz1T[2][4], a2[2], f2[2], dz2T[2], da2[2], flag_c, flagT, onesT, g2, dpregT, dliT, dlrT
// (-1 for buffers the configuration does not use).  Returns the number of entries written.
extern "C" int lirec_model_workspace_layout(const lirec_model_cfg* cfg, const lirec_batch* batch_host,
                                            int64_t* offsets, int max_entries) {
  if (!cfg || !batch_host || !offsets || max_entries < 31) return -1;
  const model::Dims d = model::make_dims(*cfg, *batch_host);
  char* base = reinterpret_cast<char*>(static_cast<uintptr_t>(4096));
  const model::Workspace w = model::carve(d, base);
  int n = 0;
  auto put = [&](const void* p) { offsets[n++] = p ? (reinterpret_cast<const char*>(p) - base) : -1; };
  for (int br = 0; br < 2; ++br) for (int s = 0; s < 4; ++s) put(w.r1[br][s]);
  for (int br = 0; br < 2; ++br) for (int s = 0; s < 4; ++s) put(w.dz1T[br][s]);
  for (int br = 0; br < 2; ++br) put(w.a2[br]);
  for (int br = 0; br < 2; ++br) put(w.f2[br]);
  for (int br = 0; br < 2; ++br) put(w.dz2T[br]);
  for (int br = 0; br < 2; ++br) put(w.da2[br]);
  put(w.flag_c); put(w.flagT); put(w.onesT); put(w.g2); put(w.dpregT); put(w.dliT); put(w.dlrT);
  return n;
}

extern "C" int lirec_model_forward(const lirec_model_cfg* cfg, const lirec_model_params* params,
                                   const lirec_batch* batch, void* workspace, size_t workspace_bytes,
                                   float* out_ints, float* out_rels, void* stream) {
  LIREC_ENTER();
  int rc = model::validate(cfg, params, batch, workspace, workspace_bytes);
  if (rc != LIREC_OK) return rc;
  return model::forward(*cfg, *params, *batch, workspace, out_ints, out_rels, static_cast<cudaStream_t>(stream));
}

extern "C" int lirec_model_backward(const lirec_model_cfg* cfg, const lirec_model_params* params,
                                    const lirec_batch* batch, void* workspace, size_t workspace_bytes,
                                    const float* d_ints, const float* d_rels, void* stream, void* heads_event) {
  LIREC_ENTER();
  int rc = model::validate(cfg, params, batch, workspace, workspace_bytes);
  if (rc != LIREC_OK) return rc;
  return model::backward(*cfg, *params, *batch, workspace, d_ints, d_rels, static_cast<cudaStream_t>(stream),
                         static_cast<cudaEvent_t>(heads_event));
}
