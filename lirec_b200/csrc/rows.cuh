// rows.cuh — job tables and host launchers of the ragged-row kernels (rows.cu).
#pragma once
#include <algorithm>

#include "common.cuh"

namespace lirec {
namespace rows {

constexpr int MAX_JOBS = 8;

// One expansion: unique layer-1 rows (4 bank slots) -> n_out split rows.
struct ExpandFwdJob {
  const float* r1[4];       // relu(L1) of the unique rows: txt, vis, tr1, tr2; each [*, J]
  int32_t J;
  const int32_t* rows;      // [n_rows, 3] (clip, track1, track2)
  const int32_t* seg_off;   // NULL (one row per output) or [n_out + 1]
  int32_t n_out;
  int32_t guard_zero;
  lirec_dropout drop;
  __nv_bfloat16* out;       // [n_out, out_ld], slot s at columns [s*2J, (s+1)*2J) as hi|lo
  int64_t out_ld;
  int32_t* row_flag_out;    // [n_out] or NULL: 1 where the segment is non-empty
  __nv_bfloat16* flag_bf16_out;  // [n_out] or NULL: the same flag as a bf16 row ([1, n_out] K-major GEMM operand)
};
struct ExpandFwdJobs {
  ExpandFwdJob job[MAX_JOBS];
  int32_t n;
};

// One scatter-reduce: gradient of the expanded rows -> unique rows of one slot.
struct ExpandBwdJob {
  const float* d_in;        // [n_out, d_ld] fp32 (column offset of the slot already applied)
  int64_t d_ld;
  const uint32_t* sign;     // ReLU gate: bit (j & 31) of sign[u * sign_ld + (j >> 5)] = [r1[u, j] > 0], as the
  int64_t sign_ld;          // layer-1 GEMM epilogue writes it (LIREC_POST_SIGN_MASK)
  int32_t J, slot;          // J % 64 == 0
  const int32_t* inv_off;   // [n_unique + 1]
  const int32_t* inv_idx;   // table rows referencing each unique row
  int32_t n_unique;
  const int32_t* owner;     // NULL (ints) or [n_rows] candidate of each context row
  const int32_t* seg_off;   // NULL or [n_out + 1]
  const int32_t* ref_out;   // optional, parallel to inv_idx (ref_tables): owner[inv_idx[q]] ...
  const float* ref_w;       // ... and 1 / its segment length, so the kernel skips two dependent lookups
  lirec_dropout drop;
  __nv_bfloat16* out;       // transposed [2J, out_pitch]: hi rows [0, J), lo rows [J, 2J)
  int64_t out_pitch;        // row pitch (elements), >= n_unique
};
struct ExpandBwdJobs {
  ExpandBwdJob job[MAX_JOBS];
  int32_t n;
};

// Per-REFERENCE tables of the context branch's inverse CSRs: ref_out[q] = owner[inv_idx[q]] (the candidate row whose
// gradient reference q reads) and ref_w[q] = 1 / (its number of context rows).
struct RefTableJobs {
  const int32_t* inv_idx[3];
  int32_t* ref_out[3];
  float* ref_w[3];
  const int32_t* owner;
  const int32_t* seg_off;
  int32_t n;                // references per table (= context rows)
};
int ref_tables(const RefTableJobs& jobs, cudaStream_t stream);

// dst[c, r] = src[r, c] (bf16), zero for R <= r < Rp
struct TransposeJob {
  const __nv_bfloat16* src;
  int64_t src_ld;
  int32_t R, C;
  __nv_bfloat16* dst;
  int64_t dst_ld;
  int32_t Rp;
};
constexpr int MAX_TRANSPOSE_JOBS = 16;
struct TransposeJobs {
  TransposeJob job[MAX_TRANSPOSE_JOBS];
  int32_t n;
};

int seg_reduce(const float* x, const int32_t* seg_off, int nseg, int dim, int mode, float* out_f32,
               int64_t out_f32_ld, void* out_bf16, int64_t out_bf16_ld, cudaStream_t stream, const int32_t* row_idx = nullptr);
int expand_fwd(const ExpandFwdJobs& jobs, cudaStream_t stream);
int expand_bwd(const ExpandBwdJobs& jobs, cudaStream_t stream);
int cast_bf16(const float* x, void* out, int64_t n, cudaStream_t stream);
int roi_max_pool(const float* maps, int T, int C, int H, int W, const int32_t* elem, int n_elem,
                 const int32_t* seg_off, int nseg, float* scratch, float* out_f32, int64_t out_f32_ld, void* out_bf16,
                 int64_t out_bf16_ld, cudaStream_t stream);
int gather_rows(const void* bank, int64_t bank_ld, int n_bank, const int32_t* idx, int n, int dim, void* out,
                int64_t out_ld, cudaStream_t stream);
int split_f32_t(const float* x, int64_t ld, int rows, int cols, void* out, int64_t pitch, int pad,
                cudaStream_t stream);
int transpose_bf16(const TransposeJobs& jobs, cudaStream_t stream);

}  // namespace rows
}  // namespace lirec
