// softpool.cu — softmax-weighted segmented reduction over ragged sequences, forward and backward.
//
// PARITY UNPINNED BY CONSTRUCTION.  The reference has no attention and no softmax pooling: its temporal
// pooling is np.max over axis 0 (mixed_utils/mixed_features.py:54, 61, 105) and its pooling over context clips
// a masked mean (mlp/model.py:301-304).  BASELINE.json's north_star names "masked temporal attention pooling as a
// segmented softmax-weighted reduction"; SURVEY.md §0.1 resolves that as ONE reduction family over the same
// offset tables, {max, mean, softmax-weighted}, of which only max and mean have a reference oracle
// (lirec_seg_reduce_f32).  This is the third member:
//
//     y[s, c] = sum_{r in seg s} w[r, c] * x[r, c],      w[., c] = softmax_r( beta * score[r, c] )
//
// with score = x itself (per element; `scores == NULL`), a per-element score tensor [total, dim], or ONE score
// per row [total] (attention pooling: score_ld == 0).  It is pinned against a float64 numpy statement and
// against its two limits, which ARE the reference's poolings: beta = 0 (or all-zero scores) is the masked mean,
// beta -> inf with score = x is the max (tests/test_pooling_gpu.py).  An empty segment yields zeros, like the
// other two modes.
//
// Layout: one CTA of 128 threads per (segment, column group), one thread per four columns, the segment's rows
// walked in batches of four (their loads issued together) with an online softmax in the base-2 domain (running
// max, running normaliser, running weighted sum; one rescale per batch, no branch), so every global access is a
// coalesced 16-byte load and the result is deterministic.  The CTA splits its rows over four row lanes of 128
// columns each and merges the lanes' states in a fixed order.  HBM-bound: forward reads x
// (+ scores) once; backward reads x, scores, dy and the forward's log-normaliser once and writes dx (+ dscores) once.
#include "rows.cuh"

namespace lirec {
namespace softpool {

__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ float ex2(float v) {
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v));
  return r;
}
__device__ __forceinline__ float lg2(float v) {
  float r;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v));
  return r;
}

constexpr float LOG2E = 1.4426950408889634f;
constexpr float LN2 = 0.6931471805599453f;
constexpr float M_EMPTY = -3.0e38f;      // running maximum of a column that has seen no row yet (finite: no inf - inf)
constexpr int RB = 4;                    // rows per batch: their loads are issued together
// Row lanes per CTA.  Measured on a B200 (profiles/r02_stress_sweep.txt): four row lanes of 128 columns tie with one
// lane of 512 columns on many short segments (2048 segments of ~32 rows, dim 2048: 79 vs 81 % of the HBM peak) and
// win everywhere else (dim 768: 74 vs 68 %, 512 segments of ~512 rows: 93 vs 80 %).
constexpr int LANES = 4;
constexpr int TPR = 128 / LANES;         // threads per row lane, four columns each

// Online softmax-weighted sum of one column, base-2 domain: t = beta * log2(e) * score.  A batch of RB rows is
// folded with ONE rescale of the running sums (RB + 1 ex2 per RB elements, no branch): with one row per update and
// a branch on "new maximum" the forward was issue-bound (two divergent paths, two MUFU per element; 35-53 % of
// the HBM peak where the max / mean members of the family, with the same access pattern, reach 80-100 %).
struct Online {
  float m, z, acc;
  __device__ __forceinline__ void init() { m = M_EMPTY; z = 0.f; acc = 0.f; }
  __device__ __forceinline__ void add4(float t0, float t1, float t2, float t3, float x0, float x1, float x2, float x3) {
    const float mn = fmaxf(fmaxf(fmaxf(t0, t1), fmaxf(t2, t3)), m);
    const float k = ex2(m - mn);
    const float e0 = ex2(t0 - mn), e1 = ex2(t1 - mn), e2 = ex2(t2 - mn), e3 = ex2(t3 - mn);
    z = fmaf(z, k, (e0 + e1) + (e2 + e3));
    acc = fmaf(acc, k, fmaf(e0, x0, fmaf(e1, x1, fmaf(e2, x2, e3 * x3))));
    m = mn;
  }
  __device__ __forceinline__ void add1(float t, float x) {
    const float mn = fmaxf(t, m);
    const float k = ex2(m - mn), e = ex2(t - mn);
    z = fmaf(z, k, e);
    acc = fmaf(acc, k, e * x);
    m = mn;
  }
  __device__ __forceinline__ void merge(float m2, float z2, float a2) {      // fixed order: deterministic
    const float mn = fmaxf(m, m2);
    const float k1 = ex2(m - mn), k2 = ex2(m2 - mn);
    z = z * k1 + z2 * k2;
    acc = acc * k1 + a2 * k2;
    m = mn;
  }
};

// One CTA of 128 threads per (segment, column group).  LANES row lanes share the CTA: lane l walks rows
// beg + l, beg + l + LANES, ... over TPR * 4 columns and the lanes' partial states are merged through
// shared memory in lane order.
// MODE: 0 = score is x, 1 = per-element tensor [total, dim], 2 = one score per row [total].
template <int MODE>
__global__ void __launch_bounds__(128)
fwd_kernel(const float* __restrict__ x, const float* __restrict__ scores, const int32_t* __restrict__ seg_off, int dim,
           float beta, float* __restrict__ out, int64_t out_ld, float* __restrict__ lse, int64_t lse_ld) {
  const int seg = blockIdx.x;
  const int ct = threadIdx.x % TPR, lane = threadIdx.x / TPR;
  const int col = (blockIdx.y * TPR + ct) * 4;
  const bool live = col < dim;
  const int beg = seg_off[seg];
  const int end = live ? seg_off[seg + 1] : beg;
  const float c = beta * LOG2E;
  Online o[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) o[k].init();
  const float* xp = x + col;
  const float* sp = scores + (MODE == 1 ? col : 0);
  int r = beg + lane;
  for (; r + (RB - 1) * LANES < end; r += RB * LANES) {
    float4 a[RB], s[RB];
#pragma unroll
    for (int k = 0; k < RB; ++k) a[k] = ld4(xp + static_cast<int64_t>(r + k * LANES) * dim);
#pragma unroll
    for (int k = 0; k < RB; ++k) {
      if (MODE == 0) s[k] = a[k];
      else if (MODE == 1) s[k] = ld4(sp + static_cast<int64_t>(r + k * LANES) * dim);
      else s[k].x = sp[r + k * LANES];
    }
    if (MODE == 2) {
      // one weight per row: the exponentials are shared by the thread's four columns (column 0 carries m and z)
      const float t0 = c * s[0].x, t1 = c * s[1].x, t2 = c * s[2].x, t3 = c * s[3].x;
      const float mn = fmaxf(fmaxf(fmaxf(t0, t1), fmaxf(t2, t3)), o[0].m);
      const float k = ex2(o[0].m - mn);
      const float e0 = ex2(t0 - mn), e1 = ex2(t1 - mn), e2 = ex2(t2 - mn), e3 = ex2(t3 - mn);
      o[0].z = fmaf(o[0].z, k, (e0 + e1) + (e2 + e3));
      o[0].m = mn;
      o[0].acc = fmaf(o[0].acc, k, fmaf(e0, a[0].x, fmaf(e1, a[1].x, fmaf(e2, a[2].x, e3 * a[3].x))));
      o[1].acc = fmaf(o[1].acc, k, fmaf(e0, a[0].y, fmaf(e1, a[1].y, fmaf(e2, a[2].y, e3 * a[3].y))));
      o[2].acc = fmaf(o[2].acc, k, fmaf(e0, a[0].z, fmaf(e1, a[1].z, fmaf(e2, a[2].z, e3 * a[3].z))));
      o[3].acc = fmaf(o[3].acc, k, fmaf(e0, a[0].w, fmaf(e1, a[1].w, fmaf(e2, a[2].w, e3 * a[3].w))));
    } else {
      o[0].add4(c * s[0].x, c * s[1].x, c * s[2].x, c * s[3].x, a[0].x, a[1].x, a[2].x, a[3].x);
      o[1].add4(c * s[0].y, c * s[1].y, c * s[2].y, c * s[3].y, a[0].y, a[1].y, a[2].y, a[3].y);
      o[2].add4(c * s[0].z, c * s[1].z, c * s[2].z, c * s[3].z, a[0].z, a[1].z, a[2].z, a[3].z);
      o[3].add4(c * s[0].w, c * s[1].w, c * s[2].w, c * s[3].w, a[0].w, a[1].w, a[2].w, a[3].w);
    }
  }
  for (; r < end; r += LANES) {
    const float4 a = ld4(xp + static_cast<int64_t>(r) * dim);
    if (MODE == 2) {
      const float t = c * sp[r];
      const float mn = fmaxf(t, o[0].m);
      const float k = ex2(o[0].m - mn), e = ex2(t - mn);
      o[0].z = fmaf(o[0].z, k, e);
      o[0].m = mn;
      o[0].acc = fmaf(o[0].acc, k, e * a.x); o[1].acc = fmaf(o[1].acc, k, e * a.y);
      o[2].acc = fmaf(o[2].acc, k, e * a.z); o[3].acc = fmaf(o[3].acc, k, e * a.w);
    } else {
      const float4 s = MODE == 0 ? a : ld4(sp + static_cast<int64_t>(r) * dim);
      o[0].add1(c * s.x, a.x); o[1].add1(c * s.y, a.y); o[2].add1(c * s.z, a.z); o[3].add1(c * s.w, a.w);
    }
  }
  if (MODE == 2) {
#pragma unroll
    for (int k = 1; k < 4; ++k) { o[k].m = o[0].m; o[k].z = o[0].z; }
  }
  __shared__ float part[LANES - 1][12][TPR];
  if (lane > 0) {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      part[lane - 1][3 * k][ct] = o[k].m; part[lane - 1][3 * k + 1][ct] = o[k].z; part[lane - 1][3 * k + 2][ct] = o[k].acc;
    }
  }
  __syncthreads();
  if (lane > 0) return;
#pragma unroll
  for (int l = 0; l < LANES - 1; ++l)
#pragma unroll
    for (int k = 0; k < 4; ++k) o[k].merge(part[l][3 * k][ct], part[l][3 * k + 1][ct], part[l][3 * k + 2][ct]);
  if (!live) return;
  float4 y = make_float4(0.f, 0.f, 0.f, 0.f), l = make_float4(0.f, 0.f, 0.f, 0.f);
  if (end > beg) {
    y = make_float4(o[0].acc / o[0].z, o[1].acc / o[1].z, o[2].acc / o[2].z, o[3].acc / o[3].z);
    l = make_float4((o[0].m + lg2(o[0].z)) * LN2, (o[1].m + lg2(o[1].z)) * LN2, (o[2].m + lg2(o[2].z)) * LN2,
                    (o[3].m + lg2(o[3].z)) * LN2);           // natural-log normaliser of beta * score
  }
  st4(out + static_cast<int64_t>(seg) * out_ld + col, y);
  if (lse) {
    if (MODE == 2) {
      if (col == 0) lse[seg] = l.x;                      // one normaliser per segment
    } else {
      st4(lse + static_cast<int64_t>(seg) * lse_ld + col, l);
    }
  }
}

// Backward, per-element scores (score_mode 0 / 1), same CTA shape as the forward (no merge: rows are independent):
//   w = exp(beta * s - lse);  dx = w * dy (+ ds when score is x);  ds = beta * w * (x - y) * dy
template <int MODE>
__global__ void __launch_bounds__(128)
bwd_elem_kernel(const float* __restrict__ x, const float* __restrict__ scores, const int32_t* __restrict__ seg_off,
                int dim, float beta, const float* __restrict__ y, int64_t y_ld, const float* __restrict__ lse,
                int64_t lse_ld, const float* __restrict__ dy, int64_t dy_ld, float* __restrict__ dx,
                float* __restrict__ dscores, int64_t total_rows) {
  const int seg = blockIdx.x;
  const int ct = threadIdx.x % TPR, lane = threadIdx.x / TPR;
  const int col = (blockIdx.y * TPR + ct) * 4;
  if (col >= dim) return;
  const int beg = seg_off[seg], end = seg_off[seg + 1];
  if (total_rows > 0 && (seg == 0 || seg == gridDim.x - 1)) {
    // rows no segment owns (before the first / after the last offset) have zero gradient
    const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int side = 0; side < 2; ++side) {
      if ((side == 0 && seg != 0) || (side == 1 && seg != gridDim.x - 1)) continue;
      const int64_t a = side ? end : 0, b = side ? total_rows : beg;
      for (int64_t r = a + lane; r < b; r += LANES) {
        st4(dx + r * dim + col, zero);
        if (MODE == 1 && dscores) st4(dscores + r * dim + col, zero);
      }
    }
  }
  if (end <= beg) return;
  const float c = beta * LOG2E;
  const float4 yy = ld4(y + static_cast<int64_t>(seg) * y_ld + col);
  float4 ll = ld4(lse + static_cast<int64_t>(seg) * lse_ld + col);
  ll.x *= LOG2E; ll.y *= LOG2E; ll.z *= LOG2E; ll.w *= LOG2E;
  const float4 g = ld4(dy + static_cast<int64_t>(seg) * dy_ld + col);
  auto one = [&](int64_t at, const float4& a, const float4& s) {
    const float4 w = make_float4(ex2(fmaf(c, s.x, -ll.x)), ex2(fmaf(c, s.y, -ll.y)), ex2(fmaf(c, s.z, -ll.z)),
                                 ex2(fmaf(c, s.w, -ll.w)));
    float4 gx = make_float4(w.x * g.x, w.y * g.y, w.z * g.z, w.w * g.w);
    const float4 gs = make_float4(beta * gx.x * (a.x - yy.x), beta * gx.y * (a.y - yy.y), beta * gx.z * (a.z - yy.z),
                                  beta * gx.w * (a.w - yy.w));
    if (MODE == 0) { gx.x += gs.x; gx.y += gs.y; gx.z += gs.z; gx.w += gs.w; }
    else if (dscores) st4(dscores + at, gs);
    st4(dx + at, gx);
  };
  int r = beg + lane;
  for (; r + (RB - 1) * LANES < end; r += RB * LANES) {
    float4 a[RB], s[RB];
#pragma unroll
    for (int k = 0; k < RB; ++k) a[k] = ld4(x + static_cast<int64_t>(r + k * LANES) * dim + col);
#pragma unroll
    for (int k = 0; k < RB; ++k) s[k] = MODE == 0 ? a[k] : ld4(scores + static_cast<int64_t>(r + k * LANES) * dim + col);
#pragma unroll
    for (int k = 0; k < RB; ++k) one(static_cast<int64_t>(r + k * LANES) * dim + col, a[k], s[k]);
  }
  for (; r < end; r += LANES) {
    const int64_t at = static_cast<int64_t>(r) * dim + col;
    const float4 a = ld4(x + at);
    const float4 s = MODE == 0 ? a : ld4(scores + at);
    one(at, a, s);
  }
}

// Backward, one score per row (score_mode 2).  CTAs of 8 warps per (segment, row chunk); a warp owns two rows at a
// time (rows beg + j, beg + j + stride) and walks their columns 256 at a time, so the segment's y / dy pieces are
// loaded once per pair of rows and eight 16-byte loads of x are in flight per lane; a row's dot product is a
// warp-shuffle reduction with no block barrier and a fixed order:
//   w_r = exp(beta * s_r - lse);  dx[r, :] = w_r * dy;  ds_r = beta * w_r * sum_c (x[r, c] - y[c]) * dy[c]
__global__ void __launch_bounds__(256)
bwd_row_kernel(const float* __restrict__ x, const float* __restrict__ scores, const int32_t* __restrict__ seg_off,
               int dim, float beta, const float* __restrict__ y, int64_t y_ld, const float* __restrict__ lse,
               const float* __restrict__ dy, int64_t dy_ld, float* __restrict__ dx, float* __restrict__ dscores,
               int64_t total_rows) {
  const int seg = blockIdx.x;
  const int beg = seg_off[seg], end = seg_off[seg + 1];
  const int warp = threadIdx.x >> 5, ln = threadIdx.x & 31;
  const int stride = 8 * gridDim.y, first = blockIdx.y * 8 + warp;
  if (total_rows > 0 && (seg == 0 || seg == gridDim.x - 1)) {
    // rows no segment owns (before the first / after the last offset) have zero gradient
    const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int side = 0; side < 2; ++side) {
      if ((side == 0 && seg != 0) || (side == 1 && seg != gridDim.x - 1)) continue;
      const int64_t a = side ? end : 0, b = side ? total_rows : beg;
      for (int64_t r = a + first; r < b; r += stride) {
        for (int cc = ln * 4; cc < dim; cc += 128) st4(dx + r * dim + cc, zero);
        if (dscores && ln == 0) dscores[r] = 0.f;
      }
    }
  }
  if (end <= beg) return;
  const float l2 = lse[seg] * LOG2E, c = beta * LOG2E;
  const float* yrow = y + static_cast<int64_t>(seg) * y_ld;
  const float* grow = dy + static_cast<int64_t>(seg) * dy_ld;
  for (int r = beg + first; r < end; r += 2 * stride) {
    const bool two = r + stride < end;
    const int r1 = two ? r + stride : r;                    // a lone last row is computed twice, stored once
    const float w0 = ex2(fmaf(c, scores[r], -l2)), w1 = ex2(fmaf(c, scores[r1], -l2));
    const float* x0 = x + static_cast<int64_t>(r) * dim;
    const float* x1 = x + static_cast<int64_t>(r1) * dim;
    float* d0 = dx + static_cast<int64_t>(r) * dim;
    float* d1 = dx + static_cast<int64_t>(r1) * dim;
    float dot0 = 0.f, dot1 = 0.f;
    int cc = ln * 4;
    for (; cc + 3 * 128 < dim; cc += 4 * 128) {
      float4 a0[4], a1[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) { a0[k] = ld4(x0 + cc + 128 * k); a1[k] = ld4(x1 + cc + 128 * k); }
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float4 yy = ld4(yrow + cc + 128 * k), g = ld4(grow + cc + 128 * k);
        st4(d0 + cc + 128 * k, make_float4(w0 * g.x, w0 * g.y, w0 * g.z, w0 * g.w));
        if (two) st4(d1 + cc + 128 * k, make_float4(w1 * g.x, w1 * g.y, w1 * g.z, w1 * g.w));
        dot0 += (a0[k].x - yy.x) * g.x + (a0[k].y - yy.y) * g.y + (a0[k].z - yy.z) * g.z + (a0[k].w - yy.w) * g.w;
        dot1 += (a1[k].x - yy.x) * g.x + (a1[k].y - yy.y) * g.y + (a1[k].z - yy.z) * g.z + (a1[k].w - yy.w) * g.w;
      }
    }
    for (; cc < dim; cc += 128) {
      const float4 a0 = ld4(x0 + cc), a1 = ld4(x1 + cc), yy = ld4(yrow + cc), g = ld4(grow + cc);
      st4(d0 + cc, make_float4(w0 * g.x, w0 * g.y, w0 * g.z, w0 * g.w));
      if (two) st4(d1 + cc, make_float4(w1 * g.x, w1 * g.y, w1 * g.z, w1 * g.w));
      dot0 += (a0.x - yy.x) * g.x + (a0.y - yy.y) * g.y + (a0.z - yy.z) * g.z + (a0.w - yy.w) * g.w;
      dot1 += (a1.x - yy.x) * g.x + (a1.y - yy.y) * g.y + (a1.z - yy.z) * g.z + (a1.w - yy.w) * g.w;
    }
    if (dscores) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        dot0 += __shfl_xor_sync(0xffffffffu, dot0, o);
        dot1 += __shfl_xor_sync(0xffffffffu, dot1, o);
      }
      if (ln == 0) {
        dscores[r] = beta * w0 * dot0;
        if (two) dscores[r1] = beta * w1 * dot1;
      }
    }
  }
}

// row chunks per segment of the per-row-score backward: enough CTAs for ~8 per SM
static int row_chunks(int nseg) {
  static int sms = 0;
  if (!sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (sms <= 0) sms = 148;
  }
  return std::max(1, std::min(8, (sms * 8 + nseg - 1) / nseg));
}

static int check(const float* x, const int32_t* seg_off, int dim, int score_mode, const float* scores) {
  LIREC_REQUIRE(x && seg_off, "seg_softmax_pool: null argument");
  LIREC_REQUIRE(dim > 0 && dim % 4 == 0, "seg_softmax_pool: dim=%d must be a positive multiple of 4", dim);
  LIREC_REQUIRE(score_mode >= 0 && score_mode <= 2, "seg_softmax_pool: score_mode=%d", score_mode);
  LIREC_REQUIRE((score_mode == 0) == (scores == nullptr), "seg_softmax_pool: scores must be NULL exactly for score_mode 0");
  LIREC_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15) == 0 &&
                    (score_mode != 1 || (reinterpret_cast<uintptr_t>(scores) & 15) == 0),
                "seg_softmax_pool: x / scores not 16-byte aligned");
  return LIREC_OK;
}

}  // namespace softpool
}  // namespace lirec

using namespace lirec;

extern "C" int lirec_seg_softmax_pool_fwd(const float* x, const float* scores, int32_t score_mode,
                                          const int32_t* seg_off, int32_t nseg, int32_t dim, float beta,
                                          float* out, int64_t out_ld, float* lse, int64_t lse_ld, void* stream) {
  LIREC_ENTER();
  int rc = softpool::check(x, seg_off, dim, score_mode, scores);
  if (rc != LIREC_OK) return rc;
  LIREC_REQUIRE(out && (reinterpret_cast<uintptr_t>(out) & 15) == 0 && out_ld % 4 == 0,
                "seg_softmax_pool_fwd: output not 16-byte aligned");
  LIREC_REQUIRE(!lse || score_mode == 2 || ((reinterpret_cast<uintptr_t>(lse) & 15) == 0 && lse_ld % 4 == 0),
                "seg_softmax_pool_fwd: lse not 16-byte aligned");
  if (nseg <= 0) return LIREC_OK;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  auto kernel = score_mode == 0   ? softpool::fwd_kernel<0>
                : score_mode == 1 ? softpool::fwd_kernel<1>
                                  : softpool::fwd_kernel<2>;
  kernel<<<dim3(nseg, (dim / 4 + softpool::TPR - 1) / softpool::TPR), 128, 0, s>>>(x, scores, seg_off, dim, beta, out,
                                                                                  out_ld, lse, lse_ld);
  LIREC_CUDA_OK(cudaGetLastError());
  note_launch();
  return LIREC_OK;
}

extern "C" int lirec_seg_softmax_pool_bwd(const float* x, const float* scores, int32_t score_mode,
                                          const int32_t* seg_off, int32_t nseg, int32_t dim, float beta,
                                          const float* out, int64_t out_ld, const float* lse, int64_t lse_ld,
                                          const float* d_out, int64_t d_out_ld, float* d_x, float* d_scores,
                                          int64_t total_rows, void* stream) {
  LIREC_ENTER();
  int rc = softpool::check(x, seg_off, dim, score_mode, scores);
  if (rc != LIREC_OK) return rc;
  LIREC_REQUIRE(out && lse && d_out && d_x, "seg_softmax_pool_bwd: null argument");
  LIREC_REQUIRE(((reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(d_out) | reinterpret_cast<uintptr_t>(d_x)) & 15) == 0 &&
                    out_ld % 4 == 0 && d_out_ld % 4 == 0,
                "seg_softmax_pool_bwd: buffers not 16-byte aligned");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (nseg <= 0) {                                    // no segment owns any row: every gradient is zero
    if (total_rows > 0) {
      LIREC_CUDA_OK(cudaMemsetAsync(d_x, 0, static_cast<size_t>(total_rows) * dim * 4, s));
      if (d_scores) LIREC_CUDA_OK(cudaMemsetAsync(d_scores, 0, static_cast<size_t>(total_rows) * (score_mode == 2 ? 1 : dim) * 4, s));
    }
    return LIREC_OK;
  }
  if (score_mode == 2) {
    softpool::bwd_row_kernel<<<dim3(nseg, softpool::row_chunks(nseg)), 256, 0, s>>>(x, scores, seg_off, dim, beta, out, out_ld, lse, d_out, d_out_ld, d_x,
                                                  d_scores, total_rows);
  } else {
    LIREC_REQUIRE((reinterpret_cast<uintptr_t>(lse) & 15) == 0 && lse_ld % 4 == 0 &&
                      (!d_scores || (reinterpret_cast<uintptr_t>(d_scores) & 15) == 0),
                  "seg_softmax_pool_bwd: lse / d_scores not 16-byte aligned");
    auto kernel = score_mode == 0 ? softpool::bwd_elem_kernel<0> : softpool::bwd_elem_kernel<1>;
    kernel<<<dim3(nseg, (dim / 4 + softpool::TPR - 1) / softpool::TPR), 128, 0, s>>>(
        x, scores, seg_off, dim, beta, out, out_ld, lse, lse_ld, d_out, d_out_ld, d_x, d_scores, total_rows);
  }
  LIREC_CUDA_OK(cudaGetLastError());
  note_launch();
  return LIREC_OK;
}
