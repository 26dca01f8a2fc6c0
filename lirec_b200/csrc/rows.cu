// rows.cu — HBM-bound ragged-row kernels: segmented pooling, row expansion by offset
// tables (forward + backward), hi/lo split and bf16 casts.
//
// All kernels map one CTA to one output row (or one unique bank row) and one thread
// to a 128-bit column group, so every global access is a coalesced 16-byte load or
// store; the reductions run sequentially over the (short) segment in registers, which
// keeps them deterministic.
#include "rows.cuh"

namespace lirec {
namespace rows {

__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// ---------------------------------------------------------------------------
// Segmented max / mean over ragged [total, dim] fp32 rows.
// Reference: np.max(..., axis=0) in mixed_utils/mixed_features.py:54,61,105; an empty
// segment yields zeros (text_features.py:171-178, mixed_features.py:89-93).
// NaN propagates like np.max.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
seg_reduce_kernel(const float* __restrict__ x, const int32_t* __restrict__ seg_off,
                  const int32_t* __restrict__ row_idx, int dim,
                  int mode, float* __restrict__ out_f32, int64_t out_f32_ld,
                  __nv_bfloat16* __restrict__ out_bf16, int64_t out_bf16_ld) {
  const int seg = blockIdx.x;
  const int col = (blockIdx.y * blockDim.x + threadIdx.x) * 4;
  if (col >= dim) return;
  const int beg = seg_off[seg], end = seg_off[seg + 1];
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  if (end > beg && row_idx) {
    // gathered segment (the token ranges of a clip's dialog lines, text_features.py:151-168): same
    // reduction over rows x[row_idx[r]]
    for (int r = beg; r < end; ++r) {
      const float4 a = ld4(x + static_cast<int64_t>(row_idx[r]) * dim + col);
      if (mode == 0) {
        if (r == beg) acc = a;
        else {
          if (a.x > acc.x || a.x != a.x) acc.x = a.x;
          if (a.y > acc.y || a.y != a.y) acc.y = a.y;
          if (a.z > acc.z || a.z != a.z) acc.z = a.z;
          if (a.w > acc.w || a.w != a.w) acc.w = a.w;
        }
      } else {
        acc.x += a.x; acc.y += a.y; acc.z += a.z; acc.w += a.w;
      }
    }
    if (mode == 1) {
      const float inv = 1.0f / static_cast<float>(end - beg);
      acc.x *= inv; acc.y *= inv; acc.z *= inv; acc.w *= inv;
    }
  } else if (end > beg) {
    const float* p = x + static_cast<int64_t>(beg) * dim + col;
    if (mode == 0) {
      acc = ld4(p);
      int r = beg + 1;
      p += dim;
      // 4 independent 128-bit loads in flight per thread
      for (; r + 3 < end; r += 4, p += 4 * static_cast<int64_t>(dim)) {
        const float4 a = ld4(p), b = ld4(p + dim), c = ld4(p + 2 * static_cast<int64_t>(dim)),
                     d = ld4(p + 3 * static_cast<int64_t>(dim));
#define LIREC_MAXN(m, v) m = ((v) > (m) || (v) != (v)) ? (v) : (m)
        LIREC_MAXN(acc.x, a.x); LIREC_MAXN(acc.y, a.y); LIREC_MAXN(acc.z, a.z); LIREC_MAXN(acc.w, a.w);
        LIREC_MAXN(acc.x, b.x); LIREC_MAXN(acc.y, b.y); LIREC_MAXN(acc.z, b.z); LIREC_MAXN(acc.w, b.w);
        LIREC_MAXN(acc.x, c.x); LIREC_MAXN(acc.y, c.y); LIREC_MAXN(acc.z, c.z); LIREC_MAXN(acc.w, c.w);
        LIREC_MAXN(acc.x, d.x); LIREC_MAXN(acc.y, d.y); LIREC_MAXN(acc.z, d.z); LIREC_MAXN(acc.w, d.w);
      }
      for (; r < end; ++r, p += dim) {
        const float4 a = ld4(p);
        LIREC_MAXN(acc.x, a.x); LIREC_MAXN(acc.y, a.y); LIREC_MAXN(acc.z, a.z); LIREC_MAXN(acc.w, a.w);
      }
#undef LIREC_MAXN
    } else {
      for (int r = beg; r < end; ++r, p += dim) {
        const float4 a = ld4(p);
        acc.x += a.x; acc.y += a.y; acc.z += a.z; acc.w += a.w;
      }
      const float inv = 1.0f / static_cast<float>(end - beg);
      acc.x *= inv; acc.y *= inv; acc.z *= inv; acc.w *= inv;
    }
  }
  if (out_f32) *reinterpret_cast<float4*>(out_f32 + static_cast<int64_t>(seg) * out_f32_ld + col) = acc;
  if (out_bf16) {
    __nv_bfloat162 lo = __floats2bfloat162_rn(acc.x, acc.y);
    __nv_bfloat162 hi = __floats2bfloat162_rn(acc.z, acc.w);
    uint2 w;
    w.x = *reinterpret_cast<uint32_t*>(&lo);
    w.y = *reinterpret_cast<uint32_t*>(&hi);
    *reinterpret_cast<uint2*>(out_bf16 + static_cast<int64_t>(seg) * out_bf16_ld + col) = w;
  }
}

// ---------------------------------------------------------------------------
// Forward expansion: unique layer-1 rows -> encoder rows (ints) or per-candidate
// masked means over context rows (ctx), with the layer-1 dropout mask.
// ---------------------------------------------------------------------------
__device__ __forceinline__ void store_split4(__nv_bfloat16* hi_ptr, __nv_bfloat16* lo_ptr, float4 v) {
  __nv_bfloat16 h[4], l[4];
  split_bf16(v.x, h[0], l[0]);
  split_bf16(v.y, h[1], l[1]);
  split_bf16(v.z, h[2], l[2]);
  split_bf16(v.w, h[3], l[3]);
  uint2 wh, wl;
  wh.x = __bfloat16_as_ushort(h[0]) | (static_cast<uint32_t>(__bfloat16_as_ushort(h[1])) << 16);
  wh.y = __bfloat16_as_ushort(h[2]) | (static_cast<uint32_t>(__bfloat16_as_ushort(h[3])) << 16);
  wl.x = __bfloat16_as_ushort(l[0]) | (static_cast<uint32_t>(__bfloat16_as_ushort(l[1])) << 16);
  wl.y = __bfloat16_as_ushort(l[2]) | (static_cast<uint32_t>(__bfloat16_as_ushort(l[3])) << 16);
  *reinterpret_cast<uint2*>(hi_ptr) = wh;
  *reinterpret_cast<uint2*>(lo_ptr) = wl;
}

constexpr int EF_IDX = 96;     // row triples of a segment staged in shared memory (longer segments read the rest in place)
__global__ void __launch_bounds__(128)
expand_fwd_kernel(const ExpandFwdJobs jobs) {
  pdl_wait();
  pdl_trigger();
  const ExpandFwdJob& jb = jobs.job[blockIdx.y];
  const int o = blockIdx.x;
  if (o >= jb.n_out) return;
  const int J = jb.J;
  const float* __restrict__ src[4] = {jb.r1[0], jb.r1[1], jb.r1[2], jb.r1[3]};
  int beg = o, end = o + 1;
  if (jb.seg_off) { beg = jb.seg_off[o]; end = jb.seg_off[o + 1]; }
  const int n = end - beg;
  // The segment's (clip, track1, track2) triples are fetched ONCE, coalesced, into shared memory: the row
  // gathers of consecutive context rows then depend on no global load and several of them are in flight
  // at a time (the kernel was bound by the idx -> row load chain: 70 % long-scoreboard stalls in ncu).
  __shared__ int32_t s_idx[3 * EF_IDX];
  for (int k = threadIdx.x; k < 3 * min(n, EF_IDX); k += blockDim.x) s_idx[k] = jb.rows[3 * static_cast<int64_t>(beg) + k];
  __syncthreads();
  const uint32_t thr = drop_threshold(jb.drop.p);
  for (int j = threadIdx.x * 4; j < J; j += blockDim.x * 4) {
    float4 acc[4];
#pragma unroll
    for (int s = 0; s < 4; ++s) acc[s] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 2
    for (int x = beg; x < end; ++x) {
      int3 idx;
      if (x - beg < EF_IDX) idx = make_int3(s_idx[3 * (x - beg)], s_idx[3 * (x - beg) + 1], s_idx[3 * (x - beg) + 2]);
      else idx = *reinterpret_cast<const int3*>(jb.rows + 3 * static_cast<int64_t>(x));
      const int u[4] = {idx.x, idx.x, idx.y, idx.z};
      float4 v[4];
#pragma unroll
      for (int s = 0; s < 4; ++s)
        v[s] = src[s] ? ld4(src[s] + static_cast<int64_t>(u[s]) * J + j) : make_float4(0.f, 0.f, 0.f, 0.f);
      if (jb.drop.p > 0.f) {
        const uint32_t rkey = drop_row_key(jb.drop.seed, jb.drop.stream_id, static_cast<uint32_t>(x));
#pragma unroll
        for (int s = 0; s < 4; ++s) {
          const uint32_t c = static_cast<uint32_t>(jb.drop.col_off + s * J + j);   // multiple of 4
          const uint32_t w0 = drop_word(rkey, c >> 1), w1 = drop_word(rkey, (c >> 1) + 1);
          if ((w0 & 0xFFFFu) < thr) v[s].x = 0.f;
          if ((w0 >> 16) < thr) v[s].y = 0.f;
          if ((w1 & 0xFFFFu) < thr) v[s].z = 0.f;
          if ((w1 >> 16) < thr) v[s].w = 0.f;
        }
      }
#pragma unroll
      for (int s = 0; s < 4; ++s) {
        acc[s].x += v[s].x; acc[s].y += v[s].y; acc[s].z += v[s].z; acc[s].w += v[s].w;
      }
    }
    if (jb.seg_off) {
      // masked mean over the segment; empty segment: 0 (guard) or 0/0 = NaN (reference
      // MidFusionMultiClip has no guard, mlp/model.py:175 vs :303)
      const float inv = (n > 0) ? 1.0f / static_cast<float>(n)
                                : (jb.guard_zero ? 0.f : __int_as_float(0x7fc00000));
#pragma unroll
      for (int s = 0; s < 4; ++s) {
        if (n > 0 || jb.guard_zero) {
          acc[s].x *= inv; acc[s].y *= inv; acc[s].z *= inv; acc[s].w *= inv;
        } else {
          acc[s] = make_float4(inv, inv, inv, inv);
        }
      }
    }
    __nv_bfloat16* orow = jb.out + static_cast<int64_t>(o) * jb.out_ld;
#pragma unroll
    for (int s = 0; s < 4; ++s)
      if (src[s]) store_split4(orow + s * 2 * J + j, orow + s * 2 * J + J + j, acc[s]);
  }
  if (jb.row_flag_out && threadIdx.x == 0) jb.row_flag_out[o] = (n > 0) ? 1 : 0;
  if (jb.flag_bf16_out && threadIdx.x == 0) jb.flag_bf16_out[o] = __float2bfloat16_rn(n > 0 ? 1.f : 0.f);
}

// Per-reference (owner, 1 / segment length) of the context branch's three inverse CSRs, see rows.cuh.
__global__ void __launch_bounds__(256)
ref_tables_kernel(const RefTableJobs jobs) {
  pdl_wait();
  pdl_trigger();
  const int y = blockIdx.y;
  const int32_t* idx = y == 0 ? jobs.inv_idx[0] : y == 1 ? jobs.inv_idx[1] : jobs.inv_idx[2];
  int32_t* out = y == 0 ? jobs.ref_out[0] : y == 1 ? jobs.ref_out[1] : jobs.ref_out[2];
  float* wgt = y == 0 ? jobs.ref_w[0] : y == 1 ? jobs.ref_w[1] : jobs.ref_w[2];
  for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < jobs.n; q += gridDim.x * blockDim.x) {
    const int o = jobs.owner[idx[q]];
    out[q] = o;
    wgt[q] = 1.0f / static_cast<float>(jobs.seg_off[o + 1] - jobs.seg_off[o]);
  }
}

// ---------------------------------------------------------------------------
// Backward of the expansion onto the unique rows of one bank slot:
//   dZ1[u] = [r1[u] > 0] * sum_{i in inv(u)} keep(i) * w_i * d_in[o_i]
// with the ReLU gate [r1 > 0] read from the 1-bit mask of the layer-1 GEMM (LIREC_POST_SIGN_MASK), written
// TRANSPOSED: out[(j) * pitch + u] (hi rows [0, J), lo rows [J, 2J)), the K-major B operand of the
// first-layer weight-gradient GEMM.  One CTA owns 64 consecutive unique rows
// and walks the J columns in chunks of 64: thread t reduces 16 columns of row t/4, the chunk is
// transposed through shared memory, and every output row segment is 64 rows x 2 B = one 128-byte line.
// ---------------------------------------------------------------------------
constexpr int EBT_ROWS = 64;
constexpr int EBT_COLS = 64;
constexpr int EBT_REFS = 1536;
constexpr int EBT_ZSPLIT = 4;
__global__ void __launch_bounds__(256, 4)
expand_bwd_t_kernel(const ExpandBwdJobs jobs) {
  pdl_wait();
  pdl_trigger();
  const ExpandBwdJob& jb = jobs.job[blockIdx.y];
  const int u0 = blockIdx.x * EBT_ROWS;
  if (u0 >= jb.n_unique) return;
  __shared__ __align__(16) __nv_bfloat16 tile[2][EBT_COLS][EBT_ROWS + 8];   // [hi|lo][col][row], padded
  __shared__ int32_t ref_row[EBT_REFS];     // table row i (dropout key)
  __shared__ int32_t ref_out[EBT_REFS];     // expanded row o whose gradient is read
  __shared__ float ref_w[EBT_REFS];         // 1 / segment length (1 for the ints branch)
  const int J = jb.J;
  const int lr = threadIdx.x >> 2;            // local unique row
  // this thread's 16 columns of a 64-column chunk: float4 number (t & 3) of each 16-column group, so the
  // four lanes of a row read 64 contiguous bytes per load instruction (two full sectors)
  const int q4 = (threadIdx.x & 3) * 4;
  const int u = u0 + lr;
  const bool live = u < jb.n_unique;
  // The references of 64 consecutive unique rows are one contiguous span of the CSR: resolve
  // idx -> owner -> 1/len ONCE per CTA, one reference per thread (three dependent loads, all in flight
  // together), instead of once per thread per column chunk.
  // With the per-reference tables of ref_tables() the chain is inv_off -> (idx, out, w) -> gradient rows: two
  // dependent memory round trips less per CTA (a CTA lives for ~6 us, of which this chain was more than half).
  __shared__ int32_t row_off[EBT_ROWS + 1];
  if (threadIdx.x <= EBT_ROWS) row_off[threadIdx.x] = jb.inv_off[min(u0 + static_cast<int>(threadIdx.x), jb.n_unique)];
  const int q0 = jb.inv_off[u0], q1 = jb.inv_off[min(u0 + EBT_ROWS, jb.n_unique)];
  for (int q = q0 + threadIdx.x; q < min(q1, q0 + EBT_REFS); q += blockDim.x) {
    const int i = jb.inv_idx[q];
    int o = i;
    float w = 1.0f;
    if (jb.ref_out) {
      o = jb.ref_out[q];
      w = jb.ref_w[q];
    } else if (jb.owner) {
      o = jb.owner[i];
      w = 1.0f / static_cast<float>(jb.seg_off[o + 1] - jb.seg_off[o]);
    }
    ref_row[q - q0] = i; ref_out[q - q0] = o; ref_w[q - q0] = w;
  }
  __syncthreads();
  int beg = 0, end = 0;
  if (live) { beg = row_off[lr]; end = row_off[lr + 1]; }
  const uint32_t thr = drop_threshold(jb.drop.p);
  // blockIdx.z takes a slice of the column chunks: more, shorter CTAs fill the last wave of the ragged
  // job list (the ints-branch jobs have 10x fewer unique rows than the context-branch ones)
  const int c_per = ((J / EBT_COLS + gridDim.z - 1) / gridDim.z) * EBT_COLS;
  const int c_beg = blockIdx.z * c_per, c_end = min(J, c_beg + c_per);
  for (int c0 = c_beg; c0 < c_end; c0 += EBT_COLS) {
    float acc[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) acc[k] = 0.f;
    const int j = c0 + q4;
    uint2 gate = make_uint2(0u, 0u);       // issued ahead of the reference loop (c0 % 64 == 0: 8-byte aligned)
    if (live) gate = *reinterpret_cast<const uint2*>(jb.sign + static_cast<int64_t>(u) * jb.sign_ld + (c0 >> 5));
    // Latency hiding without registers: the gradient pieces of the NEXT chunk are pulled into L2 now; a row's
    // 64 columns are two 128-byte lines, taken by the first two lanes of its quad.
    if (live && (threadIdx.x & 3) < 2 && c0 + EBT_COLS < c_end) {
      const int half = 32 * (threadIdx.x & 3);
      for (int q = beg; q < min(end, beg + 4); ++q)
        if (q - q0 < EBT_REFS)
          prefetch_l2(jb.d_in + static_cast<int64_t>(ref_out[q - q0]) * jb.d_ld + c0 + EBT_COLS + half);
    }
    for (int q = beg; q < end; ++q) {
      int i, o;
      float w;
      if (q - q0 < EBT_REFS) {
        i = ref_row[q - q0]; o = ref_out[q - q0]; w = ref_w[q - q0];
      } else {
        i = jb.inv_idx[q]; o = i; w = 1.0f;
        if (jb.ref_out) {
          o = jb.ref_out[q];
          w = jb.ref_w[q];
        } else if (jb.owner) {
          o = jb.owner[i];
          w = 1.0f / static_cast<float>(jb.seg_off[o + 1] - jb.seg_off[o]);
        }
      }
      const float* gp = jb.d_in + static_cast<int64_t>(o) * jb.d_ld + j;
      float4 g[4] = {ld4(gp), ld4(gp + 16), ld4(gp + 32), ld4(gp + 48)};
      if (jb.drop.p > 0.f) {
        const uint32_t rkey = drop_row_key(jb.drop.seed, jb.drop.stream_id, static_cast<uint32_t>(i));
        const uint32_t cp = static_cast<uint32_t>(jb.drop.col_off + jb.slot * J + j) >> 1;   // j % 4 == 0
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const uint32_t w0 = drop_word(rkey, cp + 8 * k), w1 = drop_word(rkey, cp + 8 * k + 1);
          if ((w0 & 0xFFFFu) < thr) g[k].x = 0.f;
          if ((w0 >> 16) < thr) g[k].y = 0.f;
          if ((w1 & 0xFFFFu) < thr) g[k].z = 0.f;
          if ((w1 >> 16) < thr) g[k].w = 0.f;
        }
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        acc[4 * k] += w * g[k].x; acc[4 * k + 1] += w * g[k].y;
        acc[4 * k + 2] += w * g[k].z; acc[4 * k + 3] += w * g[k].w;
      }
    }
    if (live) {
      // ReLU gate from the 1-bit-per-element mask of the forward GEMM (8 bytes per row and chunk instead of 256)
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const uint32_t bits = ((k < 2) ? gate.x : gate.y) >> (16 * (k & 1) + q4);
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (!((bits >> e) & 1u)) acc[4 * k + e] = 0.f;
      }
    }
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      __nv_bfloat16 h, l;
      split_bf16(acc[k], h, l);
      const int col = 16 * (k >> 2) + q4 + (k & 3);      // acc[4 * kk + e] is column 16 * kk + q4 + e
      tile[0][col][lr] = h;
      tile[1][col][lr] = l;
    }
    __syncthreads();
    // write-out: thread t -> column t/4, 16 rows (32 bytes) of hi and of lo
    {
      const int col = threadIdx.x >> 2, r0 = (threadIdx.x & 3) * 16;
      const int nrow = min(EBT_ROWS, jb.n_unique - u0);
#pragma unroll
      for (int part = 0; part < 2; ++part) {
        __nv_bfloat16* dst = jb.out + (static_cast<int64_t>(part) * J + c0 + col) * jb.out_pitch + u0 + r0;
        const __nv_bfloat16* src = &tile[part][col][r0];
        if (r0 + 16 <= nrow) {
          reinterpret_cast<uint4*>(dst)[0] = reinterpret_cast<const uint4*>(src)[0];
          reinterpret_cast<uint4*>(dst)[1] = reinterpret_cast<const uint4*>(src)[1];
        } else {
          for (int k = 0; r0 + k < nrow; ++k) dst[k] = src[k];
        }
      }
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------
// fp32 [rows, cols] -> TRANSPOSED hi/lo bf16 split: out[c * pitch + r] (hi, c < pad) and
// out[(pad + c) * pitch + r] (lo); rows c in [cols, pad) are zero.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
split_t_kernel(const float* __restrict__ x, int64_t ld, int rows, int cols, __nv_bfloat16* __restrict__ out,
               int64_t pitch, int pad) {
  pdl_wait();
  pdl_trigger();
  const int c = blockIdx.y;
  for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += gridDim.x * blockDim.x) {
    const float v = (c < cols) ? x[static_cast<int64_t>(r) * ld + c] : 0.f;
    __nv_bfloat16 h, l;
    split_bf16(v, h, l);
    out[static_cast<int64_t>(c) * pitch + r] = h;
    out[static_cast<int64_t>(pad + c) * pitch + r] = l;
  }
}

// ---------------------------------------------------------------------------
// Batched bf16 transposes with zero padding: dst[c, r] = src[r, c] for r < R, 0 for R <= r < Rp.
// Gives backward the [in, out] (K-major) copy of every weight its data-gradient GEMMs multiply by.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
transpose_bf16_kernel(const TransposeJobs jobs) {
  pdl_wait();
  pdl_trigger();
  const TransposeJob& jb = jobs.job[blockIdx.y];
  const int tiles_c = (jb.C + 63) / 64, tiles_r = (jb.Rp + 63) / 64;
  __shared__ __nv_bfloat16 tile[64][64 + 2];
  const bool vec = (jb.C % 2 == 0) && (jb.src_ld % 2 == 0) && (jb.Rp % 2 == 0) && (jb.dst_ld % 2 == 0) &&
                   (reinterpret_cast<uintptr_t>(jb.src) % 4 == 0) && (reinterpret_cast<uintptr_t>(jb.dst) % 4 == 0);
  const __nv_bfloat16 zero = __float2bfloat16_rn(0.f);
  for (int t = blockIdx.x; t < tiles_c * tiles_r; t += gridDim.x) {
    const int r0 = (t / tiles_c) * 64, c0 = (t % tiles_c) * 64;
    if (vec) {
      // load: 32 column pairs x 64 rows, one 4-byte load per element pair (128 B per row per warp)
      for (int k = threadIdx.x; k < 64 * 32; k += blockDim.x) {
        const int r = r0 + k / 32, c = c0 + 2 * (k % 32);
        __nv_bfloat162 v = __halves2bfloat162(zero, zero);
        if (r < jb.R && c < jb.C) v = *reinterpret_cast<const __nv_bfloat162*>(jb.src + static_cast<int64_t>(r) * jb.src_ld + c);
        tile[k / 32][2 * (k % 32)] = v.x;
        tile[k / 32][2 * (k % 32) + 1] = v.y;
      }
      __syncthreads();
      for (int k = threadIdx.x; k < 64 * 32; k += blockDim.x) {
        const int c = c0 + k / 32, r = r0 + 2 * (k % 32);
        if (c < jb.C && r < jb.Rp)
          *reinterpret_cast<__nv_bfloat162*>(jb.dst + static_cast<int64_t>(c) * jb.dst_ld + r) =
              __halves2bfloat162(tile[2 * (k % 32)][k / 32], tile[2 * (k % 32) + 1][k / 32]);
      }
    } else {
      for (int k = threadIdx.x; k < 64 * 64; k += blockDim.x) {
        const int r = r0 + k / 64, c = c0 + k % 64;
        tile[k / 64][k % 64] = (r < jb.R && c < jb.C) ? jb.src[static_cast<int64_t>(r) * jb.src_ld + c] : zero;
      }
      __syncthreads();
      for (int k = threadIdx.x; k < 64 * 64; k += blockDim.x) {
        const int c = c0 + k / 64, r = r0 + k % 64;
        if (c < jb.C && r < jb.Rp) jb.dst[static_cast<int64_t>(c) * jb.dst_ld + r] = tile[k % 64][k / 64];
      }
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------
// fp32 -> bf16 cast
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
cast_bf16_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ out, int64_t n) {
  const int64_t n4 = n / 4;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n4; i += stride) {
    const float4 v = reinterpret_cast<const float4*>(x)[i];
    __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
    uint2 w;
    w.x = *reinterpret_cast<uint32_t*>(&a);
    w.y = *reinterpret_cast<uint32_t*>(&b);
    reinterpret_cast<uint2*>(out)[i] = w;
  }
  for (int64_t i = n4 * 4 + blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n; i += stride)
    out[i] = __float2bfloat16_rn(x[i]);
}

// ---------------------------------------------------------------------------
// Spatial / ROI mean of I3D feature maps fused with the temporal max over a segment of elements:
//   out[s, c] = max_{e in seg s} mean_{y0<=y<y1, x0<=x<x1} maps[frame_e, c, y, x]
// Reference: clip visual = np.max over frames of the H x W mean (visual_features.py:67-69,
// mixed_features.py:54); person track = np.max over track elements of the mean over the person box
// derived from the face box (visual_features.py:105-135, mixed_features.py:104-105).  The reference
// quirks are kept: an element with frame < 0 (frame index == T, :130-131) is an all-zero row that
// still takes part in the max; an empty box averages nothing and gives NaN, which np.max propagates;
// an empty segment gives zeros (mixed_features.py:89-93).
// One warp owns one (segment, channel): lanes stride over the flattened box of one H x W plane (a
// contiguous <= 2 KB region), a shuffle tree sums the lanes, and the running max lives in lane 0.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
roi_max_pool_kernel(const float* __restrict__ maps, int C, int HW, int W, const int32_t* __restrict__ elem,
                    const int32_t* __restrict__ seg_off, float* __restrict__ out_f32, int64_t out_f32_ld,
                    __nv_bfloat16* __restrict__ out_bf16, int64_t out_bf16_ld) {
  const int seg = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int c = blockIdx.y * (blockDim.x >> 5) + warp;
  if (c >= C) return;
  const int beg = seg_off[seg], end = seg_off[seg + 1];
  float best = 0.f;
  bool first = true;
  for (int e = beg; e < end; ++e) {
    const int32_t* el = elem + 5 * static_cast<int64_t>(e);
    const int frame = el[0], y0 = el[1], y1 = el[2], x0 = el[3], x1 = el[4];
    float v = 0.f;
    if (frame >= 0) {
      const int w = x1 - x0, h = y1 - y0;
      const int n = (w > 0 && h > 0) ? w * h : 0;
      const float* plane = maps + (static_cast<int64_t>(frame) * C + c) * HW;
      float acc = 0.f;
      if (w == W) {                                   // full-width box: one contiguous run
        const float* p = plane + y0 * W;
        for (int i = lane; i < n; i += 32) acc += p[i];
      } else {
        for (int i = lane; i < n; i += 32) {
          const int yy = i / w, xx = i - yy * w;
          acc += plane[(y0 + yy) * W + x0 + xx];
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
      v = (n > 0) ? acc / static_cast<float>(n) : __int_as_float(0x7fc00000);
    }
    if (first || v > best || v != v) best = (best != best) ? best : v;   // NaN sticks, like np.max
    first = false;
  }
  if (lane == 0) {
    if (out_f32) out_f32[static_cast<int64_t>(seg) * out_f32_ld + c] = best;
    if (out_bf16) out_bf16[static_cast<int64_t>(seg) * out_bf16_ld + c] = __float2bfloat16_rn(best);
  }
}

// Two-stage form of the same pooling, used when the caller provides a scratch buffer: stage 1 writes the
// box mean of EVERY (element, channel) — one warp per element and four channels, so thousands of warps
// keep independent plane reads in flight instead of walking a segment's elements one after another —
// and stage 2 is the segmented max kernel above (which runs at the HBM roofline).  The scratch costs
// n_elem * C * 4 B of extra traffic, ~1 % of the map bytes read.
__global__ void __launch_bounds__(256)
roi_mean_kernel(const float* __restrict__ maps, int C, int HW, int W, const int32_t* __restrict__ elem,
                float* __restrict__ out, int64_t out_ld) {
  const int e = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int c0 = (blockIdx.y * (blockDim.x >> 5) + warp) * 4;
  if (c0 >= C) return;
  const int32_t* el = elem + 5 * static_cast<int64_t>(e);
  const int frame = el[0], y0 = el[1], y1 = el[2], x0 = el[3], x1 = el[4];
  const int w = x1 - x0, h = y1 - y0;
  const int n = (w > 0 && h > 0) ? w * h : 0;
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  if (frame >= 0 && n > 0) {
    const float* plane = maps + (static_cast<int64_t>(frame) * C + c0) * HW;
    if (w == W && n == HW && c0 + 3 < C && (reinterpret_cast<uintptr_t>(plane) & 15) == 0) {
      // whole frames (the clip-level pooling, visual_features.py:67-69): the four planes of this warp are ONE
      // contiguous, 16-byte aligned run of 4 * HW floats, read as 128-bit pieces.  Piece i holds elements
      // [4i, 4i + 4) and plane k elements [k HW, (k + 1) HW): all pieces in [ceil(k HW / 4), floor((k + 1) HW / 4))
      // belong to plane k alone and cost one load + four adds; the (at most three) pieces that straddle a plane
      // boundary are read element-wise by twelve lanes.  The first version classified every element by comparing
      // its index with the boundaries — ~50 instructions per 16 bytes, issue-bound at 31-38 % of the HBM peak.
      const float4* p4 = reinterpret_cast<const float4*>(plane);
      int lo[4], hi[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) { lo[k] = (k * HW + 3) >> 2; hi[k] = ((k + 1) * HW) >> 2; }
      // one piece of each of the four planes per iteration: eight independent 16-byte loads in flight per lane
#pragma unroll 2
      for (int i = lane; i < (HW >> 2) + 1; i += 32) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          if (lo[k] + i < hi[k]) {
            const float4 v = __ldg(p4 + lo[k] + i);
            acc[k] += (v.x + v.y) + (v.z + v.w);
          }
        }
      }
      if (lane < 12) {
        const int k = 1 + (lane >> 2), b = k * HW;
        if (b & 3) {
          const int e = (b & ~3) + (lane & 3);
          const float v = __ldg(plane + e);
          const int ch = (e >= b) ? k : k - 1;
#pragma unroll
          for (int t = 0; t < 4; ++t) acc[t] += (ch == t) ? v : 0.f;
        }
      }
    } else if (w == W) {
      const float* p = plane + y0 * W;
#pragma unroll 4
      for (int i = lane; i < n; i += 32) {
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if (c0 + k < C) acc[k] += p[static_cast<int64_t>(k) * HW + i];
      }
    } else {
      for (int i = lane; i < n; i += 32) {
        const int yy = i / w, xx = i - yy * w;
        const int o = (y0 + yy) * W + x0 + xx;
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if (c0 + k < C) acc[k] += plane[static_cast<int64_t>(k) * HW + o];
      }
    }
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], o);
  }
  if (lane == 0) {
    float* orow = out + static_cast<int64_t>(e) * out_ld + c0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (c0 + k >= C) break;
      float v = 0.f;                                            // frame < 0: the zero row the reference keeps
      if (frame >= 0) v = (n > 0) ? acc[k] / static_cast<float>(n) : __int_as_float(0x7fc00000);
      orow[k] = v;
    }
  }
}

// ---------------------------------------------------------------------------
// Row gather: out[i, :] = bank[idx[i], :] (bf16 rows, 16-byte column groups).  Builds the per-batch
// feature banks from dataset banks that stay resident in HBM.  One warp per row (warp-strided over the rows):
// the row index is read once, the lanes walk the row's 16-byte groups four at a time (four 128-bit loads in
// flight per lane, then four stores), no division anywhere.  The loader launches it on its copy stream while the
// step's persistent GEMM CTAs hold the SMs: 256 threads x <= 40 registers fit beside one of them, so the gather
// overlaps the (tensor-bound) GEMMs instead of waiting for a gap between launches — hence the depth per lane.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
gather_rows_kernel(const uint4* __restrict__ bank, int64_t bank_ld16, int n_bank, const int32_t* __restrict__ idx,
                   int n, int cols16, uint4* __restrict__ out, int64_t out_ld16) {
  const int lane = threadIdx.x & 31;
  const int warps = (gridDim.x * blockDim.x) >> 5;
  for (int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < n; r += warps) {
    const int src = idx[r];
    const bool ok = src >= 0 && src < n_bank;                    // out of range -> zero row
    const uint4* in = bank + static_cast<int64_t>(ok ? src : 0) * bank_ld16;
    uint4* o = out + static_cast<int64_t>(r) * out_ld16;
    int c = lane;
    for (; c + 96 < cols16; c += 128) {
      uint4 v[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) v[k] = ok ? in[c + 32 * k] : make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
      for (int k = 0; k < 4; ++k) o[c + 32 * k] = v[k];
    }
    for (; c < cols16; c += 32) o[c] = ok ? in[c] : make_uint4(0u, 0u, 0u, 0u);
  }
}

// ---------------------------------------------------------------------------
// host launchers
// ---------------------------------------------------------------------------
int roi_max_pool(const float* maps, int T, int C, int H, int W, const int32_t* elem, int n_elem,
                 const int32_t* seg_off, int nseg, float* scratch, float* out_f32, int64_t out_f32_ld, void* out_bf16,
                 int64_t out_bf16_ld, cudaStream_t stream) {
  LIREC_REQUIRE(maps && elem && seg_off, "roi_max_pool: null argument");
  LIREC_REQUIRE(T > 0 && C > 0 && H > 0 && W > 0, "roi_max_pool: maps [%d, %d, %d, %d]", T, C, H, W);
  LIREC_REQUIRE(out_f32 || out_bf16, "roi_max_pool: no output");
  if (nseg <= 0) return LIREC_OK;
  if (scratch && n_elem > 0 && C % 4 == 0 && (reinterpret_cast<uintptr_t>(scratch) & 15) == 0) {
    dim3 g1(n_elem, (C + 31) / 32);
    roi_mean_kernel<<<g1, 256, 0, stream>>>(maps, C, H * W, W, elem, scratch, C);
    LIREC_CUDA_OK(cudaGetLastError());
    note_launch();
    return seg_reduce(scratch, seg_off, nseg, C, 0, out_f32, out_f32_ld, out_bf16, out_bf16_ld, stream);
  }
  dim3 grid(nseg, (C + 7) / 8);
  roi_max_pool_kernel<<<grid, 256, 0, stream>>>(maps, C, H * W, W, elem, seg_off, out_f32, out_f32_ld,
                                                reinterpret_cast<__nv_bfloat16*>(out_bf16), out_bf16_ld);
  LIREC_CUDA_OK(cudaGetLastError());
  note_launch();
  return LIREC_OK;
}

int gather_rows(const void* bank, int64_t bank_ld, int n_bank, const int32_t* idx, int n, int dim, void* out,
                int64_t out_ld, cudaStream_t stream) {
  LIREC_REQUIRE(dim > 0 && dim % 8 == 0 && bank_ld % 8 == 0 && out_ld % 8 == 0,
                "gather_rows: dim=%d and the row pitches must be multiples of 8 bf16 elements", dim);
  LIREC_REQUIRE((reinterpret_cast<uintptr_t>(bank) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0,
                "gather_rows: bank / out not 16-byte aligned");
  LIREC_REQUIRE(bank && idx && out && n_bank > 0, "gather_rows: null argument");
  if (n <= 0) return LIREC_OK;
  const int cols16 = dim / 8;
  const int grid = std::min((n + 7) / 8, 148 * 16);              // eight rows (warps) per CTA
  gather_rows_kernel<<<grid, 256, 0, stream>>>(static_cast<const uint4*>(bank), bank_ld / 8, n_bank, idx, n, cols16,
                                               static_cast<uint4*>(out), out_ld / 8);
  LIREC_CUDA_OK(cudaGetLastError());
  note_launch();
  return LIREC_OK;
}

int seg_reduce(const float* x, const int32_t* seg_off, int nseg, int dim, int mode, float* out_f32,
               int64_t out_f32_ld, void* out_bf16, int64_t out_bf16_ld, cudaStream_t stream, const int32_t* row_idx) {
  LIREC_REQUIRE(dim > 0 && dim % 4 == 0, "seg_reduce: dim=%d must be a positive multiple of 4", dim);
  LIREC_REQUIRE(mode == 0 || mode == 1, "seg_reduce: mode=%d", mode);
  LIREC_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15) == 0, "seg_reduce: x not 16-byte aligned");
  LIREC_REQUIRE(out_f32 || out_bf16, "seg_reduce: no output");
  LIREC_REQUIRE(!out_f32 || ((reinterpret_cast<uintptr_t>(out_f32) & 15) == 0 && out_f32_ld % 4 == 0),
                "seg_reduce: fp32 output not 16-byte aligned");
  LIREC_REQUIRE(!out_bf16 || ((reinterpret_cast<uintptr_t>(out_bf16) & 7) == 0 && out_bf16_ld % 4 == 0),
                "seg_reduce: bf16 output not 8-byte aligned");
  if (nseg <= 0) return LIREC_OK;
  dim3 grid(nseg, (dim / 4 + 127) / 128);
  seg_reduce_kernel<<<grid, 128, 0, stream>>>(x, seg_off, row_idx, dim, mode, out_f32, out_f32_ld,
                                              reinterpret_cast<__nv_bfloat16*>(out_bf16), out_bf16_ld);
  LIREC_CUDA_OK(cudaGetLastError());
  note_launch();
  return LIREC_OK;
}

int expand_fwd(const ExpandFwdJobs& jobs, cudaStream_t stream) {
  int max_out = 0;
  for (int i = 0; i < jobs.n; ++i) {
    const ExpandFwdJob& j = jobs.job[i];
    LIREC_REQUIRE(j.J > 0 && j.J % 4 == 0, "expand_fwd: J=%d", j.J);
    LIREC_REQUIRE(j.out_ld % 4 == 0 && (reinterpret_cast<uintptr_t>(j.out) & 7) == 0,
                  "expand_fwd: output not 8-byte aligned");
    max_out = std::max(max_out, j.n_out);
  }
  if (max_out == 0 || jobs.n == 0) return LIREC_OK;
  dim3 grid(max_out, jobs.n);
  LIREC_CUDA_OK(launch_pdl(expand_fwd_kernel, grid, dim3(128), 0, stream, jobs));
  note_launch();
  return LIREC_OK;
}

int ref_tables(const RefTableJobs& jobs, cudaStream_t stream) {
  if (jobs.n <= 0) return LIREC_OK;
  LIREC_REQUIRE(jobs.owner && jobs.seg_off, "ref_tables: null argument");
  for (int y = 0; y < 3; ++y)
    LIREC_REQUIRE(jobs.inv_idx[y] && jobs.ref_out[y] && jobs.ref_w[y], "ref_tables: null table %d", y);
  dim3 grid(std::min((jobs.n + 255) / 256, 148 * 4), 3);
  LIREC_CUDA_OK(launch_pdl(ref_tables_kernel, grid, dim3(256), 0, stream, jobs));
  note_launch();
  return LIREC_OK;
}

int expand_bwd(const ExpandBwdJobs& jobs, cudaStream_t stream) {
  int max_u = 0, max_j = 0;
  for (int i = 0; i < jobs.n; ++i) {
    const ExpandBwdJob& j = jobs.job[i];
    LIREC_REQUIRE(j.J > 0 && j.J % EBT_COLS == 0 && j.d_ld % 4 == 0,
                  "expand_bwd: J=%d must be a positive multiple of 64, d_ld=%lld a multiple of 4", j.J,
                  (long long)j.d_ld);
    LIREC_REQUIRE(j.out_pitch % 8 == 0 && j.out_pitch >= j.n_unique && (reinterpret_cast<uintptr_t>(j.out) & 15) == 0,
                  "expand_bwd: output needs 16-byte alignment and a pitch >= n_unique that is a multiple of 8");
    LIREC_REQUIRE(j.sign && (reinterpret_cast<uintptr_t>(j.sign) & 7) == 0 && j.sign_ld % 2 == 0 &&
                      j.sign_ld >= j.J / 32,
                  "expand_bwd: sign mask must be non-NULL, 8-byte aligned, with an even pitch >= J / 32 words");
    max_u = std::max(max_u, j.n_unique);
    max_j = std::max(max_j, j.J);
  }
  if (max_u == 0 || jobs.n == 0) return LIREC_OK;
  // column split over grid.z: 4 at bench sizes; 8 (one 64-column chunk per CTA) when the whole launch is
  // under ~2 k CTAs — measured on B200: 64-clip batches 41 -> 27 us, 1024-clip batches 141 -> 149 us
  const int row_ctas = (max_u + EBT_ROWS - 1) / EBT_ROWS;
  const int zsplit = (static_cast<long>(row_ctas) * jobs.n * EBT_ZSPLIT <= 2048) ? 2 * EBT_ZSPLIT : EBT_ZSPLIT;
  dim3 grid(row_ctas, jobs.n, std::max(1, std::min(zsplit, max_j / EBT_COLS)));
  LIREC_CUDA_OK(launch_pdl(expand_bwd_t_kernel, grid, dim3(256), 0, stream, jobs));
  LIREC_CUDA_OK(cudaGetLastError());
  note_launch();
  return LIREC_OK;
}

int split_f32_t(const float* x, int64_t ld, int rows, int cols, void* out, int64_t pitch, int pad,
                cudaStream_t stream) {
  LIREC_REQUIRE(pad >= cols && pitch >= rows, "split_f32_t: pad=%d cols=%d pitch=%lld rows=%d", pad, cols,
                (long long)pitch, rows);
  if (rows <= 0) return LIREC_OK;
  dim3 grid(std::min((rows + 255) / 256, 64), pad);
  LIREC_CUDA_OK(launch_pdl(split_t_kernel, grid, dim3(256), 0, stream, x, ld, rows, cols, reinterpret_cast<__nv_bfloat16*>(out), pitch, pad));
  note_launch();
  return LIREC_OK;
}

int transpose_bf16(const TransposeJobs& jobs, cudaStream_t stream) {
  if (jobs.n == 0) return LIREC_OK;
  int max_tiles = 0;
  for (int i = 0; i < jobs.n; ++i) {
    const TransposeJob& j = jobs.job[i];
    LIREC_REQUIRE(j.src && j.dst && j.R > 0 && j.C > 0 && j.Rp >= j.R && j.dst_ld >= j.Rp,
                  "transpose_bf16: bad job %d", i);
    max_tiles = std::max(max_tiles, ((j.C + 63) / 64) * ((j.Rp + 63) / 64));
  }
  dim3 grid(std::min(max_tiles, 148 * 4), jobs.n);
  LIREC_CUDA_OK(launch_pdl(transpose_bf16_kernel, grid, dim3(256), 0, stream, jobs));
  note_launch();
  return LIREC_OK;
}

int cast_bf16(const float* x, void* out, int64_t n, cudaStream_t stream) {
  if (n <= 0) return LIREC_OK;
  LIREC_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 7) == 0,
                "cast_bf16: pointers not aligned");
  const int grid = static_cast<int>(std::min<int64_t>((n / 4 + 255) / 256 + 1, 148 * 8));
  cast_bf16_kernel<<<grid, 256, 0, stream>>>(x, reinterpret_cast<__nv_bfloat16*>(out), n);
  LIREC_CUDA_OK(cudaGetLastError());
  note_launch();
  return LIREC_OK;
}

}  // namespace rows
}  // namespace lirec

// ---------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------
using namespace lirec;

extern "C" int lirec_seg_reduce_f32(const float* x, const int32_t* row_idx, const int32_t* seg_off, int32_t nseg,
                                    int32_t dim, int32_t mode, float* out_f32, int64_t out_f32_ld, void* out_bf16,
                                    int64_t out_bf16_ld, void* stream) {
  LIREC_ENTER();
  return rows::seg_reduce(x, seg_off, nseg, dim, mode, out_f32, out_f32_ld, out_bf16, out_bf16_ld,
                          static_cast<cudaStream_t>(stream), row_idx);
}

extern "C" int lirec_rows_expand_fwd(const float* r1_txt, const float* r1_vis, const float* r1_tr1,
                                     const float* r1_tr2, int32_t J, const int32_t* rows_tbl,
                                     const int32_t* seg_off, int32_t n_out, int32_t guard_zero,
                                     lirec_dropout drop, void* out_split, int64_t out_ld,
                                     int32_t* row_flag_out, void* stream) {
  LIREC_ENTER();
  rows::ExpandFwdJobs jobs;
  jobs.n = 1;
  rows::ExpandFwdJob& j = jobs.job[0];
  j.r1[0] = r1_txt; j.r1[1] = r1_vis; j.r1[2] = r1_tr1; j.r1[3] = r1_tr2;
  j.J = J;
  j.rows = rows_tbl;
  j.seg_off = seg_off;
  j.n_out = n_out;
  j.guard_zero = guard_zero;
  j.drop = drop;
  j.out = reinterpret_cast<__nv_bfloat16*>(out_split);
  j.out_ld = out_ld;
  j.row_flag_out = row_flag_out;
  j.flag_bf16_out = nullptr;
  return rows::expand_fwd(jobs, static_cast<cudaStream_t>(stream));
}

extern "C" int lirec_rows_expand_bwd(const float* d_in, int64_t d_ld, const uint32_t* sign, int64_t sign_ld,
                                     int32_t J, int32_t slot, const int32_t* inv_off, const int32_t* inv_idx,
                                     int32_t n_unique, const int32_t* owner, const int32_t* seg_off,
                                     lirec_dropout drop, void* out_split, int64_t out_pitch, void* stream) {
  LIREC_ENTER();
  LIREC_REQUIRE((owner == nullptr) == (seg_off == nullptr), "expand_bwd: owner and seg_off go together");
  rows::ExpandBwdJobs jobs;
  jobs.n = 1;
  rows::ExpandBwdJob& j = jobs.job[0];
  j.d_in = d_in; j.d_ld = d_ld; j.J = J; j.slot = slot;
  j.sign = sign; j.sign_ld = sign_ld;
  j.inv_off = inv_off; j.inv_idx = inv_idx; j.n_unique = n_unique;
  j.owner = owner; j.seg_off = seg_off; j.drop = drop;
  j.ref_out = nullptr; j.ref_w = nullptr;
  j.out = reinterpret_cast<__nv_bfloat16*>(out_split);
  j.out_pitch = out_pitch;
  return rows::expand_bwd(jobs, static_cast<cudaStream_t>(stream));
}

extern "C" int lirec_roi_max_pool_f32(const float* maps, int32_t T, int32_t C, int32_t H, int32_t W,
                                      const int32_t* elem, int32_t n_elem, const int32_t* seg_off, int32_t nseg,
                                      float* scratch, float* out_f32, int64_t out_f32_ld, void* out_bf16,
                                      int64_t out_bf16_ld, void* stream) {
  LIREC_ENTER();
  return rows::roi_max_pool(maps, T, C, H, W, elem, n_elem, seg_off, nseg, scratch, out_f32, out_f32_ld, out_bf16,
                            out_bf16_ld, static_cast<cudaStream_t>(stream));
}

extern "C" int lirec_gather_rows(const void* bank, int64_t bank_ld, int32_t n_bank, const int32_t* idx, int32_t n,
                                 int32_t dim, void* out, int64_t out_ld, void* stream) {
  LIREC_ENTER();
  return rows::gather_rows(bank, bank_ld, n_bank, idx, n, dim, out, out_ld, static_cast<cudaStream_t>(stream));
}

extern "C" int lirec_split_f32(const float* x, int64_t ld, int32_t rows_n, int32_t cols, void* out_split,
                               int64_t pitch, int32_t pad, void* stream) {
  LIREC_ENTER();
  return rows::split_f32_t(x, ld, rows_n, cols, out_split, pitch, pad, static_cast<cudaStream_t>(stream));
}

extern "C" int lirec_cast_bf16(const float* x, void* out, int64_t n, void* stream) {
  LIREC_ENTER();
  return rows::cast_bf16(x, out, n, static_cast<cudaStream_t>(stream));
}
