// loss.cu — fused forward + gradient kernels of the reference's max-margin losses, over
// ragged candidate tables, and the flat Adam step.
//
// The reference builds every loss from ~25-40 tiny ATen kernels plus host-side
// np.ones masks (mlp/model.py:381-575).  Here one CTA handles one clip: it masks,
// applies the sigmoid, scores every candidate (track-pair) slot, takes the arg-max
// assignment (lowest index on ties, like torch.argmax), sums the hinge terms and
// writes d(loss)/d(logits) in the same pass.  Empty slots are never materialised: the
// reference sets them to -inf (sigma = 0, zero gradient), which is what skipping does.
#include <algorithm>
#include <cmath>

#include "common.cuh"

namespace lirec {
namespace loss {

__device__ __forceinline__ float sigmoidf(float x) { return 1.0f / (1.0f + expf(-x)); }

// softplus(x) = max(x, 0) + log1p(exp(-|x|)) stays finite and exact for logits far outside [-88, 88].
__device__ __forceinline__ float softplusf(float x) { return fmaxf(x, 0.f) + log1pf(expf(-fabsf(x))); }

__device__ __forceinline__ float block_sum(float v, float* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  float t = 0.f;
  for (int w = 0; w < (blockDim.x >> 5); ++w) t += red[w];  // fixed order: deterministic
  return t;
}

__device__ __forceinline__ float block_max(float v, float* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  float t = red[0];
  for (int w = 1; w < (blockDim.x >> 5); ++w) t = fmaxf(t, red[w]);
  return t;
}

constexpr int MAX_SLOTS = 128;

// The weakly supervised track assignment t* of clip b over its n candidate slots, shared by the margin and
// the BCE track losses: slot 0 under tr_correct, a counter-hash draw from the softmax scores under
// cat_distr, otherwise the arg-max of sigma(ints[t,y]) (+ sigma(rels[t,r0])) with the lowest index winning
// ties.  Called by every thread of the CTA; returns t* to all of them and writes assign[b].
__device__ __forceinline__ int track_assign(const float* __restrict__ xi, const float* __restrict__ xr,
                                            const int32_t* __restrict__ rels_lab, int n, int C, int R, int y, int r0,
                                            int b, const lirec_track_loss_cfg& cfg, int32_t* __restrict__ assign) {
  __shared__ float s_score[MAX_SLOTS];
  __shared__ int s_tstar;
  const bool has_rels = R > 0;
  // ---- per-slot assignment score: sigma(ints[t,y]) (+ sigma(rels[t,r0])) ----
  for (int t = threadIdx.x; t < n; t += blockDim.x) {
    float sc = sigmoidf(xi[static_cast<int64_t>(t) * C + y]);
    if (has_rels) {
      const bool rel_on = rels_lab[t] != R;  // None-labelled slots are all -inf
      const float pr = (rel_on && r0 < R) ? sigmoidf(xr[static_cast<int64_t>(t) * R + r0]) : 0.f;
      sc = sc + pr;
    }
    s_score[t] = sc;
  }
  // ---- tr_cat_distr: the assignment is SAMPLED from (softmax_t(ints[t,y]) + softmax_t(rels[t,r0])) / 2
  // (model.py:468-471, 538-543; a relationship column that is -inf everywhere gives NaN -> 0 there).
  // The uniform draw comes from the counter hash of (seed, clip), mirrored by oracle/dropout.py.
  if (cfg.cat_distr && !cfg.tr_correct) {
    __shared__ float s_p[MAX_SLOTS];
    if (threadIdx.x == 0) {
      float mx = -INFINITY, mxr = -INFINITY;
      for (int t = 0; t < n; ++t) {
        mx = fmaxf(mx, xi[static_cast<int64_t>(t) * C + y]);
        if (has_rels && r0 < R && rels_lab[t] != R) mxr = fmaxf(mxr, xr[static_cast<int64_t>(t) * R + r0]);
      }
      float zi = 0.f, zr = 0.f;
      for (int t = 0; t < n; ++t) {
        zi += expf(xi[static_cast<int64_t>(t) * C + y] - mx);
        if (has_rels && r0 < R && rels_lab[t] != R) zr += expf(xr[static_cast<int64_t>(t) * R + r0] - mxr);
      }
      float total = 0.f;
      for (int t = 0; t < n; ++t) {
        float pt = expf(xi[static_cast<int64_t>(t) * C + y] - mx) / zi;
        if (has_rels) {
          float pr = 0.f;
          if (r0 < R && rels_lab[t] != R && zr > 0.f) pr = expf(xr[static_cast<int64_t>(t) * R + r0] - mxr) / zr;
          pt = 0.5f * (pt + pr);
        }
        s_p[t] = pt;
        total += pt;
      }
      const uint32_t h = fmix32(cfg.seed ^ fmix32(static_cast<uint32_t>(b) + 0x51ED270Bu));
      const float u = static_cast<float>(h >> 8) * (1.0f / 16777216.0f) * total;
      float acc = 0.f;
      int pick = n - 1;
      for (int t = 0; t < n; ++t) {
        acc += s_p[t];
        if (u < acc) { pick = t; break; }
      }
      s_tstar = pick;
      assign[b] = pick;
    }
  }
  __syncthreads();
  if (threadIdx.x == 0 && !(cfg.cat_distr && !cfg.tr_correct)) {
    int best = 0;
    if (!cfg.tr_correct) {
      float bv = s_score[0];
      for (int t = 1; t < n; ++t)
        if (s_score[t] > bv) { bv = s_score[t]; best = t; }
      // empty slots score exactly 0 and sit after the valid prefix, so they can only win a
      // tie against a valid slot scoring 0, which the lowest-index rule gives to the valid one
    }
    s_tstar = best;
    assign[b] = best;
  }
  __syncthreads();
  return s_tstar;
}

// The negatives of the track losses, shared by the margin loss's sum and max forms and by the BCE.
// Interaction (t, c): a class that multilab keeps for the clip, other than the label; under tr_correct the
// label is a positive only on the ground-truth slots, and a negative on every other slot.
__device__ __forceinline__ bool int_negative(const uint8_t* __restrict__ ml, int t, int c, int y, int gt0, int gt1,
                                             bool tr_correct) {
  return ml[c] != 0 && (tr_correct ? !(c == y && (t == gt0 || t == gt1)) : c != y);
}

// Relationship (t, r) of a slot labelled lab: none when lab is None (R); otherwise every class other than lab
// under tr_correct, and other than the ground-truth pairs' classes r0 and r1 without it.
__device__ __forceinline__ bool rel_negative(int lab, int r, int R, int r0, int r1, bool tr_correct) {
  return lab != R && (tr_correct ? r != lab : (r != r0 && r != r1));
}

// One CTA per clip; t* is track_assign's.  Both forms sum over the same negatives (int_negative, rel_negative).
//   hinge (kBce = false): MarginLoss (mlp/model.py:444-494) / MarginTrackRelsLoss (mlp/model.py:497-575): one hinge
//     m - sigma(x[t*, y]) + sigma(x[neg]) per negative, or under max_neg one per slot on its hardest negative.
//   BCE (kBce = true): the positives are (t*, y) and (t*, c) for pos_mask[b, c] != 0, the negatives minus those
//     positives are the zeros, and every other (slot, class) has weight 0.  The relationship positive is
//     (t*, r0) when live.
//   loss_per_clip = lymbda / B * sum_ints l + 1 / B * sum_rels l
template <bool kBce>
__device__ __forceinline__ void track_loss_body(const float* __restrict__ ints, const float* __restrict__ rels,
                                                const int32_t* __restrict__ cand_off, int B,
                                                const int32_t* __restrict__ labels,
                                                const int32_t* __restrict__ rels_label,
                                                const int32_t* __restrict__ gt_tracks,
                                                const uint8_t* __restrict__ multilab,
                                                const uint8_t* __restrict__ pos_mask, const lirec_track_loss_cfg& cfg,
                                                float* __restrict__ loss_per_clip, int32_t* __restrict__ assign,
                                                float* __restrict__ d_ints, float* __restrict__ d_rels) {
  pdl_wait();
  pdl_trigger();
  __shared__ float s_red[8];
  const int b = blockIdx.x;
  const int beg = cand_off[b], n = cand_off[b + 1] - beg;
  const int C = cfg.n_classes, R = cfg.n_rels;
  const bool has_rels = R > 0;
  const int y = labels[b];
  const int gt0 = gt_tracks[2 * b], gt1 = gt_tracks[2 * b + 1];
  // relationship class of the ground-truth pair(s); slots past the valid prefix carry the
  // reference's pad label 0 (classification_dataloader.py:430)
  int r0 = 0, r1 = 0;
  if (has_rels) {
    r0 = (gt0 < n) ? rels_label[beg + gt0] : 0;
    r1 = (gt1 < n) ? rels_label[beg + gt1] : 0;
  }
  const float* xi = ints + static_cast<int64_t>(beg) * C;
  const float* xr = has_rels ? rels + static_cast<int64_t>(beg) * R : nullptr;
  float* gi = d_ints + static_cast<int64_t>(beg) * C;
  float* gr = has_rels ? d_rels + static_cast<int64_t>(beg) * R : nullptr;
  const float invB = 1.0f / static_cast<float>(B);
  const int ts = track_assign(xi, xr, has_rels ? rels_label + beg : nullptr, n, C, R, y, r0, b, cfg, assign);
  const bool pos_r_live = has_rels && (rels_label[beg + ts] != R) && (r0 < R);
  float pos = 0.f, pos_r = 0.f;  // the hinge's positive scores
  if constexpr (!kBce) {
    pos = sigmoidf(xi[static_cast<int64_t>(ts) * C + y]);
    pos_r = pos_r_live ? sigmoidf(xr[static_cast<int64_t>(ts) * R + r0]) : 0.f;
  }
  const float mi = cfg.margin - pos, mr = cfg.margin - pos_r;
  const float wi = cfg.lymbda * invB, wr = invB;

  float loss_i = 0.f, cnt_i = 0.f, loss_r = 0.f, cnt_r = 0.f;
  if (kBce || !cfg.max_neg) {
    // ---- sum over every (slot, class) negative, and the BCE's positives ----
    for (int e = threadIdx.x; e < n * C; e += blockDim.x) {
      const int t = e / C, c = e - t * C;
      float g = 0.f;
      if constexpr (kBce) {
        const bool pos = (t == ts) && (c == y || (pos_mask != nullptr && pos_mask[static_cast<int64_t>(b) * C + c] != 0));
        const bool neg = int_negative(multilab + static_cast<int64_t>(b) * C, t, c, y, gt0, gt1, cfg.tr_correct);
        if (pos) {
          const float v = xi[e];
          loss_i += softplusf(-v);
          g = wi * (sigmoidf(v) - 1.f);
        } else if (neg) {
          const float v = xi[e];
          loss_i += softplusf(v);
          g = wi * sigmoidf(v);
        }
      } else if (int_negative(multilab + static_cast<int64_t>(b) * C, t, c, y, gt0, gt1, cfg.tr_correct)) {
        const float s = sigmoidf(xi[e]);
        const float h = mi + s;
        if (h > 0.f) { loss_i += h; cnt_i += 1.f; g = wi * s * (1.f - s); }
      }
      gi[e] = g;
    }
    if (has_rels) {
      for (int e = threadIdx.x; e < n * R; e += blockDim.x) {
        const int t = e / R, r = e - t * R;
        float g = 0.f;
        if constexpr (kBce) {
          const bool pos = pos_r_live && t == ts && r == r0;
          const bool neg = rel_negative(rels_label[beg + t], r, R, r0, r1, cfg.tr_correct);
          if (pos) {
            const float v = xr[e];
            loss_r += softplusf(-v);
            g = wr * (sigmoidf(v) - 1.f);
          } else if (neg) {
            const float v = xr[e];
            loss_r += softplusf(v);
            g = wr * sigmoidf(v);
          }
        } else if (rel_negative(rels_label[beg + t], r, R, r0, r1, cfg.tr_correct)) {
          const float s = sigmoidf(xr[e]);
          const float h = mr + s;
          if (h > 0.f) { loss_r += h; cnt_r += 1.f; g = wr * s * (1.f - s); }
        }
        gr[e] = g;
      }
    }
  } else if constexpr (!kBce) {
    // ---- max-negative variant: one hinge per slot on its hardest negative; the
    // reference also adds relu(m - pos) for every EMPTY slot (model.py:485-486,558-562)
    for (int e = threadIdx.x; e < n * C; e += blockDim.x) gi[e] = 0.f;
    if (has_rels)
      for (int e = threadIdx.x; e < n * R; e += blockDim.x) gr[e] = 0.f;
    __syncthreads();
    for (int t = threadIdx.x; t < cfg.max_slots; t += blockDim.x) {
      float best = 0.f;
      int bc = -1;
      if (t < n) {
        for (int c = 0; c < C; ++c) {
          if (!int_negative(multilab + static_cast<int64_t>(b) * C, t, c, y, gt0, gt1, cfg.tr_correct)) continue;
          const float s = sigmoidf(xi[static_cast<int64_t>(t) * C + c]);
          if (s > best) { best = s; bc = c; }
        }
      }
      const float h = mi + best;
      if (h > 0.f) {
        loss_i += h; cnt_i += 1.f;
        if (bc >= 0) gi[static_cast<int64_t>(t) * C + bc] = wi * best * (1.f - best);
      }
      if (has_rels) {
        float bestr = 0.f;
        int br = -1;
        if (t < n) {
          const int lab = rels_label[beg + t];
          for (int r = 0; r < R; ++r) {
            if (!rel_negative(lab, r, R, r0, r1, cfg.tr_correct)) continue;
            const float s = sigmoidf(xr[static_cast<int64_t>(t) * R + r]);
            if (s > bestr) { bestr = s; br = r; }
          }
        }
        const float hr = mr + bestr;
        if (hr > 0.f) {
          loss_r += hr; cnt_r += 1.f;
          if (br >= 0) gr[static_cast<int64_t>(t) * R + br] = wr * bestr * (1.f - bestr);
        }
      }
    }
  }
  loss_i = block_sum(loss_i, s_red);
  if constexpr (!kBce) cnt_i = block_sum(cnt_i, s_red);
  if (has_rels) {
    loss_r = block_sum(loss_r, s_red);
    if constexpr (!kBce) cnt_r = block_sum(cnt_r, s_red);
  }
  if constexpr (!kBce) __syncthreads();
  if (threadIdx.x == 0) {
    if constexpr (!kBce) {
      // the positive receives minus the number of active hinges
      gi[static_cast<int64_t>(ts) * C + y] += -cnt_i * wi * pos * (1.f - pos);
      if (has_rels && pos_r_live) gr[static_cast<int64_t>(ts) * R + r0] += -cnt_r * wr * pos_r * (1.f - pos_r);
    }
    loss_per_clip[b] = cfg.lymbda * loss_i * invB + loss_r * invB;
  }
}

__global__ void __launch_bounds__(128)
track_loss_kernel(const float* __restrict__ ints, const float* __restrict__ rels,
                  const int32_t* __restrict__ cand_off, int B, const int32_t* __restrict__ labels,
                  const int32_t* __restrict__ rels_label, const int32_t* __restrict__ gt_tracks,
                  const uint8_t* __restrict__ multilab, lirec_track_loss_cfg cfg,
                  float* __restrict__ loss_per_clip, int32_t* __restrict__ assign,
                  float* __restrict__ d_ints, float* __restrict__ d_rels) {
  track_loss_body<false>(ints, rels, cand_off, B, labels, rels_label, gt_tracks, multilab, nullptr, cfg,
                         loss_per_clip, assign, d_ints, d_rels);
}

__global__ void __launch_bounds__(128)
bce_track_kernel(const float* __restrict__ ints, const float* __restrict__ rels,
                 const int32_t* __restrict__ cand_off, int B, const int32_t* __restrict__ labels,
                 const int32_t* __restrict__ rels_label, const int32_t* __restrict__ gt_tracks,
                 const uint8_t* __restrict__ multilab, const uint8_t* __restrict__ pos_mask, lirec_track_loss_cfg cfg,
                 float* __restrict__ loss_per_clip, int32_t* __restrict__ assign, float* __restrict__ d_ints,
                 float* __restrict__ d_rels) {
  track_loss_body<true>(ints, rels, cand_off, B, labels, rels_label, gt_tracks, multilab, pos_mask, cfg,
                        loss_per_clip, assign, d_ints, d_rels);
}

// Row-wise hinge: MaxMarginCrossEntropyLoss (model.py:422-441) and both terms of
// MultiTaskMaxMargin (model.py:381-419).
__global__ void __launch_bounds__(128)
rowmargin_kernel(const float* __restrict__ logits, int64_t ld, int rows, int C,
                 const int32_t* __restrict__ labels, const uint8_t* __restrict__ weights, float margin,
                 float scale, float* __restrict__ loss_per_row, float* __restrict__ d_logits, int64_t d_ld) {
  pdl_wait();
  pdl_trigger();
  __shared__ float s_red[8];
  const int b = blockIdx.x;
  const int y = labels[b];
  float* g = d_logits + static_cast<int64_t>(b) * d_ld;
  if (y < 0) {  // row not selected (relationship label None)
    for (int c = threadIdx.x; c < C; c += blockDim.x) g[c] = 0.f;
    if (threadIdx.x == 0) loss_per_row[b] = 0.f;
    return;
  }
  const float* x = logits + static_cast<int64_t>(b) * ld;
  const float pos = sigmoidf(x[y]);
  float l = 0.f, cnt = 0.f;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const bool neg = (c != y) && (weights == nullptr || weights[static_cast<int64_t>(b) * C + c] != 0);
    float gv = 0.f;
    if (neg) {
      const float s = sigmoidf(x[c]);
      const float h = margin - pos + s;
      if (h > 0.f) { l += h; cnt += 1.f; gv = scale * s * (1.f - s); }
    }
    if (c != y) g[c] = gv;
  }
  l = block_sum(l, s_red);
  cnt = block_sum(cnt, s_red);
  if (threadIdx.x == 0) {
    g[y] = -cnt * scale * pos * (1.f - pos);
    loss_per_row[b] = l * scale;
  }
}


// Row-wise softmax cross-entropy, forward + gradient: both terms of MultiTaskCrossEntropyLoss
// (model.py:357-378; F.cross_entropy with optional class weights, mean reduction).  The caller passes
// scale = 1 / sum_i w[y_i] over the selected rows; rows with label < 0 are skipped.
//   loss_row = scale * w[y] * (logsumexp(x) - x[y]);  d/dx_c = scale * w[y] * (softmax_c - [c == y])
__global__ void __launch_bounds__(128)
ce_kernel(const float* __restrict__ logits, int64_t ld, int C, const int32_t* __restrict__ labels,
          const float* __restrict__ class_w, float scale, float* __restrict__ loss_per_row,
          float* __restrict__ d_logits, int64_t d_ld) {
  __shared__ float s_red[8];
  const int b = blockIdx.x;
  const int y = labels[b];
  float* g = d_logits + static_cast<int64_t>(b) * d_ld;
  if (y < 0) {
    for (int c = threadIdx.x; c < C; c += blockDim.x) g[c] = 0.f;
    if (threadIdx.x == 0) loss_per_row[b] = 0.f;
    return;
  }
  const float* x = logits + static_cast<int64_t>(b) * ld;
  float mx = -INFINITY;
  for (int c = threadIdx.x; c < C; c += blockDim.x) mx = fmaxf(mx, x[c]);
  mx = block_max(mx, s_red);
  float z = 0.f;
  for (int c = threadIdx.x; c < C; c += blockDim.x) z += expf(x[c] - mx);
  z = block_sum(z, s_red);
  const float w = (class_w ? class_w[y] : 1.0f) * scale;
  for (int c = threadIdx.x; c < C; c += blockDim.x) g[c] = w * (expf(x[c] - mx) / z - (c == y ? 1.f : 0.f));
  if (threadIdx.x == 0) loss_per_row[b] = w * (logf(z) + mx - x[y]);
}

// ---- sigmoid binary cross-entropy (multi-label) --------------------------------------------------------
// Per element with target t and weight w:  l = w * (t ? softplus(-x) : softplus(x)),  dl/dx = w * (sigma(x) - t).
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

constexpr int BCE_ROWS_PER_CTA = 4;  // one warp per row: rows are short (C = 101 or R = 15)

// Row form: target 1 on the label and on pos_mask, weight 0 on the non-targets that neg_mask excludes.
//   loss_row = scale * sum_c w_c * BCE(x_c, t_c);  d/dx_c = scale * w_c * (sigma(x_c) - t_c)
// Rows with label < 0 get loss 0 and a zero gradient row.
__global__ void __launch_bounds__(32 * BCE_ROWS_PER_CTA)
bce_rows_kernel(const float* __restrict__ logits, int64_t ld, int rows, int C, const int32_t* __restrict__ labels,
                const uint8_t* __restrict__ neg_mask, const uint8_t* __restrict__ pos_mask, float scale,
                float* __restrict__ loss_per_row, float* __restrict__ d_logits, int64_t d_ld) {
  pdl_wait();
  pdl_trigger();
  const int lane = threadIdx.x & 31;
  const int b = blockIdx.x * BCE_ROWS_PER_CTA + (threadIdx.x >> 5);
  if (b >= rows) return;
  const int y = labels[b];
  float* g = d_logits + static_cast<int64_t>(b) * d_ld;
  if (y < 0) {
    for (int c = lane; c < C; c += 32) g[c] = 0.f;
    if (lane == 0) loss_per_row[b] = 0.f;
    return;
  }
  const float* x = logits + static_cast<int64_t>(b) * ld;
  const uint8_t* nm = neg_mask ? neg_mask + static_cast<int64_t>(b) * C : nullptr;
  const uint8_t* pm = pos_mask ? pos_mask + static_cast<int64_t>(b) * C : nullptr;
  float l = 0.f;
  for (int c = lane; c < C; c += 32) {
    const float v = x[c];
    const bool pos = (c == y) || (pm != nullptr && pm[c] != 0);
    float gv = 0.f;
    if (pos) {
      l += softplusf(-v);
      gv = scale * (sigmoidf(v) - 1.f);
    } else if (nm == nullptr || nm[c] != 0) {
      l += softplusf(v);
      gv = scale * sigmoidf(v);
    }
    g[c] = gv;
  }
  l = warp_sum(l);
  if (lane == 0) loss_per_row[b] = scale * l;
}

// Prediction arg-maxes of the evaluation loop (reference utils/evaluation.py:114-175, 179-271), one CTA
// per clip over its valid candidate slots; empty slots are -inf there, i.e. never win.
//   out[b] = { pr_track, joint_t, joint_c, joint_r, cls_at_gt0, cls_at_gt1, rel_at_gt0, rel_at_gt1 }
//   pr_track : argmax_t sigma(ints[t,y]) (+ sigma(rels (+) 0)[t, r_gt])           (:137, :221-222)
//   joint    : first arg-max of sigma(ints)[t,c] (+ sigma(rels (+) 0)[t,r]) over the flattened
//              (t,c[,r]) index, the sum taken in double like numpy's float32 + float64  (:144-147, :229-235)
//   cls/rel at gt_i : argmax over classes / relationship classes of the raw logits of slot gt_tracks[b,i]
//              (-1 when that slot is empty)                                              (:152, :241-243)
// Ties resolve to the lowest flattened index, like np.argmax.
__global__ void __launch_bounds__(128)
predict_kernel(const float* __restrict__ ints, const float* __restrict__ rels,
               const int32_t* __restrict__ cand_off, const int32_t* __restrict__ labels,
               const int32_t* __restrict__ rels_label, const int32_t* __restrict__ gt_tracks, int C, int R,
               int32_t* __restrict__ out) {
  __shared__ double s_val[128];
  __shared__ long long s_idx[128];
  const int b = blockIdx.x, tid = threadIdx.x;
  const int beg = cand_off[b], n = cand_off[b + 1] - beg;
  const bool has_rels = R > 0;
  const int R1 = has_rels ? R + 1 : 1;
  const int y = labels[b];
  const int gt0 = gt_tracks[2 * b], gt1 = gt_tracks[2 * b + 1];
  const float* xi = ints + static_cast<int64_t>(beg) * C;
  const float* xr = has_rels ? rels + static_cast<int64_t>(beg) * R : nullptr;
  // relationship label of the ground-truth slot: evaluation.py:208 takes gt_rels[:, 0]
  const int rg = has_rels ? rels_label[beg] : 0;

  auto reduce_first_max = [&](double v, long long i) -> long long {
    s_val[tid] = v; s_idx[tid] = i;
    __syncthreads();
    for (int o = 64; o > 0; o >>= 1) {
      if (tid < o) {
        const double v2 = s_val[tid + o]; const long long i2 = s_idx[tid + o];
        if (v2 > s_val[tid] || (v2 == s_val[tid] && i2 < s_idx[tid])) { s_val[tid] = v2; s_idx[tid] = i2; }
      }
      __syncthreads();
    }
    const long long r = s_idx[0];
    __syncthreads();
    return r;
  };
  const double NEG = -1e300;
  // ---- track assignment for the ground-truth class (and relationship) ----
  {
    double v = NEG; long long idx = 0x7fffffffffffLL;
    for (int t = tid; t < n; t += blockDim.x) {
      double sc = static_cast<double>(sigmoidf(xi[static_cast<int64_t>(t) * C + y]));
      if (has_rels) sc += (rg < R) ? static_cast<double>(sigmoidf(xr[static_cast<int64_t>(t) * R + rg])) : 0.0;
      if (sc > v) { v = sc; idx = t; }
    }
    const long long r = reduce_first_max(v, idx);
    if (tid == 0) out[8 * b + 0] = static_cast<int32_t>(r);
  }
  // ---- joint (t, c[, r]) arg-max ----
  {
    double v = NEG; long long idx = 0x7fffffffffffLL;
    const long long total = static_cast<long long>(n) * C * R1;
    for (long long e = tid; e < total; e += blockDim.x) {
      const int t = static_cast<int>(e / (C * R1));
      const int rem = static_cast<int>(e - static_cast<long long>(t) * C * R1);
      const int c = rem / R1, r = rem - c * R1;
      double sc = static_cast<double>(sigmoidf(xi[static_cast<int64_t>(t) * C + c]));
      if (has_rels) sc += (r < R) ? static_cast<double>(sigmoidf(xr[static_cast<int64_t>(t) * R + r])) : 0.0;
      if (sc > v) { v = sc; idx = e; }
    }
    const long long r = reduce_first_max(v, idx);
    if (tid == 0) {
      const int t = static_cast<int>(r / (C * R1));
      const int rem = static_cast<int>(r - static_cast<long long>(t) * C * R1);
      out[8 * b + 1] = t; out[8 * b + 2] = rem / R1; out[8 * b + 3] = has_rels ? rem % R1 : -1;
    }
  }
  // ---- class / relationship arg-max at the ground-truth slots ----
  for (int i = 0; i < 2; ++i) {
    const int g = i ? gt1 : gt0;
    double v = NEG; long long idx = 0x7fffffffffffLL;
    if (g < n)
      for (int c = tid; c < C; c += blockDim.x) {
        const double sc = xi[static_cast<int64_t>(g) * C + c];
        if (sc > v) { v = sc; idx = c; }
      }
    long long r = reduce_first_max(v, idx);
    if (tid == 0) out[8 * b + 4 + i] = (g < n) ? static_cast<int32_t>(r) : -1;
    v = NEG; idx = 0x7fffffffffffLL;
    if (has_rels && g < n)
      for (int c = tid; c < R; c += blockDim.x) {
        const double sc = xr[static_cast<int64_t>(g) * R + c];
        if (sc > v) { v = sc; idx = c; }
      }
    r = reduce_first_max(v, idx);
    if (tid == 0) out[8 * b + 6 + i] = (has_rels && g < n) ? static_cast<int32_t>(r) : -1;
  }
}

// torch.optim.Adam (coupled L2) over the flat parameter buffer + bf16 shadow refresh.
__global__ void __launch_bounds__(256)
adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
            float* __restrict__ v, __nv_bfloat16* __restrict__ pb, int64_t n, float lr, float beta1,
            float beta2, float eps, float wd, float bc1, float bc2_sqrt, float grad_scale) {
  pdl_wait();
  pdl_trigger();
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  const int64_t tid = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  const float step = lr / bc1;
  // 128-bit path over the 16-byte aligned bulk (the flat buffers are: segments are 256-byte aligned), same
  // per-element arithmetic as the scalar tail below
  const bool vec = ((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(m) |
                     reinterpret_cast<uintptr_t>(v)) & 15) == 0 && (reinterpret_cast<uintptr_t>(pb) & 7) == 0;
  const int64_t n4 = vec ? n / 4 : 0;
  for (int64_t i = tid; i < n4; i += stride) {
    float4 pv = reinterpret_cast<const float4*>(p)[i];
    const float4 gr = reinterpret_cast<const float4*>(g)[i];
    float4 mv = reinterpret_cast<const float4*>(m)[i];
    float4 vv = reinterpret_cast<const float4*>(v)[i];
    float* pp = &pv.x; const float* gg = &gr.x; float* mm = &mv.x; float* vp = &vv.x;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float gv = gg[k] * grad_scale + wd * pp[k];
      mm[k] = beta1 * mm[k] + (1.f - beta1) * gv;
      vp[k] = beta2 * vp[k] + (1.f - beta2) * gv * gv;
      pp[k] -= step * mm[k] / (sqrtf(vp[k]) / bc2_sqrt + eps);
    }
    reinterpret_cast<float4*>(m)[i] = mv;
    reinterpret_cast<float4*>(v)[i] = vv;
    reinterpret_cast<float4*>(p)[i] = pv;
    if (pb) {
      const __nv_bfloat162 lo = __floats2bfloat162_rn(pv.x, pv.y), hi = __floats2bfloat162_rn(pv.z, pv.w);
      uint2 w;
      w.x = *reinterpret_cast<const uint32_t*>(&lo);
      w.y = *reinterpret_cast<const uint32_t*>(&hi);
      reinterpret_cast<uint2*>(pb)[i] = w;
    }
  }
  for (int64_t i = 4 * n4 + tid; i < n; i += stride) {
    float pv = p[i];
    const float gv = g[i] * grad_scale + wd * pv;
    const float mv = beta1 * m[i] + (1.f - beta1) * gv;
    const float vv = beta2 * v[i] + (1.f - beta2) * gv * gv;
    m[i] = mv;
    v[i] = vv;
    pv -= step * mv / (sqrtf(vv) / bc2_sqrt + eps);
    p[i] = pv;
    if (pb) pb[i] = __float2bfloat16_rn(pv);
  }
}

// ---- Chunked passes over a tensor table of the flat buffer (LAMB, gradient clipping)
// Every tensor l of the table (floats [begin[l], begin[l] + len[l])) is cut into chunks of LIREC_LAMB_CHUNK floats
// that never cross its end; chunks are numbered tensor by tensor in table order, and one CTA of CHUNK_THREADS owns
// one chunk.  Floats outside every tensor (the padding between segments) are never touched.  Sums run in a fixed
// order that depends only on the chunk size and the CTA size, never on the grid: per thread over its elements, a
// shuffle butterfly, the warps in order; across chunks in fp64.  No float atomics.
constexpr int CHUNK_THREADS = 256;

__device__ __forceinline__ int64_t flat_chunks(int64_t len) {
  return len > 0 ? (len + LIREC_LAMB_CHUNK - 1) / LIREC_LAMB_CHUNK : 1;  // an empty tensor keeps one (empty) chunk
}

struct FlatChunk {
  int l;              // tensor, -1 past the last chunk
  int64_t k;          // chunk within the tensor
  int64_t base, cnt;  // the tensor's first chunk and its chunk count
};

// The tensor that owns chunk c: a block-wide scan of the chunk counts, 256 table entries at a time.  All threads.
__device__ FlatChunk flat_locate(const int64_t* __restrict__ len, int n_tensors, int64_t c) {
  __shared__ long long s_warp[CHUNK_THREADS / 32];
  __shared__ FlatChunk s_hit;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_hit.l = -1;
  long long carry = 0;
  for (int t0 = 0; t0 < n_tensors; t0 += CHUNK_THREADS) {
    const int l = t0 + static_cast<int>(threadIdx.x);
    const long long cnt = l < n_tensors ? flat_chunks(len[l]) : 0;
    long long x = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const long long y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) s_warp[warp] = x;
    __syncthreads();
    long long before = carry, total = 0;
#pragma unroll
    for (int w = 0; w < CHUNK_THREADS / 32; ++w) {
      if (w < warp) before += s_warp[w];
      total += s_warp[w];
    }
    const long long excl = before + x - cnt;
    if (l < n_tensors && c >= excl && c < excl + cnt) s_hit = FlatChunk{l, c - excl, excl, cnt};
    carry += total;
    __syncthreads();
    if (s_hit.l >= 0 || c < carry) break;
  }
  return s_hit;
}

__device__ __forceinline__ double2 flat_block_sum2(double a, double b) {
  __shared__ double2 s_red[CHUNK_THREADS / 32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    a += __shfl_xor_sync(0xffffffffu, a, o);
    b += __shfl_xor_sync(0xffffffffu, b, o);
  }
  if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = make_double2(a, b);
  __syncthreads();
  double2 t = make_double2(0.0, 0.0);
#pragma unroll
  for (int w = 0; w < CHUNK_THREADS / 32; ++w) {
    t.x += s_red[w].x;
    t.y += s_red[w].y;
  }
  return t;
}

// [off, off + n) of the flat buffers: the chunk this CTA owns.
__device__ __forceinline__ int flat_chunk_span(const int64_t* __restrict__ begin, const int64_t* __restrict__ len,
                                               const FlatChunk& ch, int64_t* off) {
  const int64_t l = len[ch.l];
  *off = begin[ch.l] + ch.k * LIREC_LAMB_CHUNK;
  return l > 0 ? static_cast<int>(min(static_cast<int64_t>(LIREC_LAMB_CHUNK), l - ch.k * LIREC_LAMB_CHUNK)) : 0;
}

// ---- LAMB (You et al., ICLR 2020) over the flat buffer: Adam moments, decoupled weight decay, per-tensor trust ratio
// One CTA per chunk in both passes:
//   lamb_moments_kernel: m, v <- Adam moments of g = grad_scale * grad; u = lamb_u(m, v, w);
//                        partials[chunk] = (sum w^2, sum u^2) over the chunk
//   lamb_apply_kernel  : r_l = ||w_l|| / ||u_l|| from tensor l's partials (1 unless both are > 0);
//                        w <- w - lr * r_l * u, bf16 shadow <- rn_bf16(w)
// Pass 2 recomputes u from the stored moments and the old w with the same helper, so the norm is the norm of the u
// that is applied.  Across chunks, thread t sums a contiguous run of the tensor's partials in chunk order, then the
// block sum.

// u of one element.  Explicit round-to-nearest intrinsics: the compiler may not contract or reorder them, so both
// passes compute the same bits.
__device__ __forceinline__ float lamb_u(float m, float v, float w, float inv_bc1, float inv_bc2_sqrt, float eps,
                                        float wd) {
  const float den = __fadd_rn(__fmul_rn(__fsqrt_rn(v), inv_bc2_sqrt), eps);
  return __fadd_rn(__fdiv_rn(__fmul_rn(m, inv_bc1), den), __fmul_rn(wd, w));
}

__global__ void __launch_bounds__(CHUNK_THREADS)
lamb_moments_kernel(const float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                    float* __restrict__ v, const int64_t* __restrict__ begin, const int64_t* __restrict__ len,
                    int n_tensors, double2* __restrict__ partials, float beta1, float beta2, float c1, float c2,
                    float eps, float wd, float inv_bc1, float inv_bc2_sqrt, float grad_scale) {
  pdl_wait();
  pdl_trigger();
  const FlatChunk ch = flat_locate(len, n_tensors, blockIdx.x);
  if (ch.l < 0) return;
  int64_t off;
  const int n = flat_chunk_span(begin, len, ch, &off);
  const float* pc = p + off; const float* gc = g + off; float* mc = m + off; float* vc = v + off;
  const bool vec = ((reinterpret_cast<uintptr_t>(pc) | reinterpret_cast<uintptr_t>(gc) |
                     reinterpret_cast<uintptr_t>(mc) | reinterpret_cast<uintptr_t>(vc)) & 15) == 0;
  const int n4 = vec ? n / 4 : 0;
  float sw = 0.f, su = 0.f;
  for (int i = threadIdx.x; i < n4; i += CHUNK_THREADS) {
    const float4 pv = reinterpret_cast<const float4*>(pc)[i];
    const float4 gr = reinterpret_cast<const float4*>(gc)[i];
    float4 mv = reinterpret_cast<const float4*>(mc)[i];
    float4 vv = reinterpret_cast<const float4*>(vc)[i];
    const float* pp = &pv.x; const float* gg = &gr.x; float* mm = &mv.x; float* vp = &vv.x;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float gv = gg[k] * grad_scale;
      mm[k] = beta1 * mm[k] + c1 * gv;
      vp[k] = beta2 * vp[k] + c2 * gv * gv;
      const float u = lamb_u(mm[k], vp[k], pp[k], inv_bc1, inv_bc2_sqrt, eps, wd);
      sw += pp[k] * pp[k];
      su += u * u;
    }
    reinterpret_cast<float4*>(mc)[i] = mv;
    reinterpret_cast<float4*>(vc)[i] = vv;
  }
  for (int i = 4 * n4 + threadIdx.x; i < n; i += CHUNK_THREADS) {
    const float pv = pc[i];
    const float gv = gc[i] * grad_scale;
    const float mv = beta1 * mc[i] + c1 * gv;
    const float vv = beta2 * vc[i] + c2 * gv * gv;
    mc[i] = mv;
    vc[i] = vv;
    const float u = lamb_u(mv, vv, pv, inv_bc1, inv_bc2_sqrt, eps, wd);
    sw += pv * pv;
    su += u * u;
  }
  const double2 s = flat_block_sum2(sw, su);
  if (threadIdx.x == 0) partials[blockIdx.x] = s;
}

__global__ void __launch_bounds__(CHUNK_THREADS)
lamb_apply_kernel(float* __restrict__ p, const float* __restrict__ m, const float* __restrict__ v,
                  __nv_bfloat16* __restrict__ pb, const int64_t* __restrict__ begin, const int64_t* __restrict__ len,
                  int n_tensors, const double2* __restrict__ partials, float* __restrict__ trust_out, float lr,
                  float eps, float wd, float inv_bc1, float inv_bc2_sqrt) {
  pdl_wait();
  pdl_trigger();
  const FlatChunk ch = flat_locate(len, n_tensors, blockIdx.x);
  if (ch.l < 0) return;
  // trust ratio of the tensor: thread t sums a contiguous run of its chunks' partials in chunk order
  const int64_t run = (ch.cnt + CHUNK_THREADS - 1) / CHUNK_THREADS;
  const int64_t j0 = min(ch.cnt, run * threadIdx.x), j1 = min(ch.cnt, j0 + run);
  double sw = 0.0, su = 0.0;
  for (int64_t j = j0; j < j1; ++j) {
    const double2 q = partials[ch.base + j];
    sw += q.x;
    su += q.y;
  }
  const double2 s = flat_block_sum2(sw, su);
  const double r = (s.x > 0.0 && s.y > 0.0) ? sqrt(s.x) / sqrt(s.y) : 1.0;
  if (trust_out && ch.k == 0 && threadIdx.x == 0) trust_out[ch.l] = static_cast<float>(r);
  const float step = static_cast<float>(static_cast<double>(lr) * r);

  int64_t off;
  const int n = flat_chunk_span(begin, len, ch, &off);
  float* pc = p + off; const float* mc = m + off; const float* vc = v + off;
  __nv_bfloat16* bc = pb ? pb + off : nullptr;
  const bool vec = ((reinterpret_cast<uintptr_t>(pc) | reinterpret_cast<uintptr_t>(mc) |
                     reinterpret_cast<uintptr_t>(vc)) & 15) == 0 && (reinterpret_cast<uintptr_t>(bc) & 7) == 0;
  const int n4 = vec ? n / 4 : 0;
  for (int i = threadIdx.x; i < n4; i += CHUNK_THREADS) {
    float4 pv = reinterpret_cast<const float4*>(pc)[i];
    const float4 mv = reinterpret_cast<const float4*>(mc)[i];
    const float4 vv = reinterpret_cast<const float4*>(vc)[i];
    float* pp = &pv.x; const float* mm = &mv.x; const float* vp = &vv.x;
#pragma unroll
    for (int k = 0; k < 4; ++k)
      pp[k] = __fsub_rn(pp[k], __fmul_rn(step, lamb_u(mm[k], vp[k], pp[k], inv_bc1, inv_bc2_sqrt, eps, wd)));
    reinterpret_cast<float4*>(pc)[i] = pv;
    if (bc) {
      const __nv_bfloat162 lo = __floats2bfloat162_rn(pv.x, pv.y), hi = __floats2bfloat162_rn(pv.z, pv.w);
      uint2 w;
      w.x = *reinterpret_cast<const uint32_t*>(&lo);
      w.y = *reinterpret_cast<const uint32_t*>(&hi);
      reinterpret_cast<uint2*>(bc)[i] = w;
    }
  }
  for (int i = 4 * n4 + threadIdx.x; i < n; i += CHUNK_THREADS) {
    const float pv = __fsub_rn(pc[i], __fmul_rn(step, lamb_u(mc[i], vc[i], pc[i], inv_bc1, inv_bc2_sqrt, eps, wd)));
    pc[i] = pv;
    if (bc) bc[i] = __float2bfloat16_rn(pv);
  }
}

// ---- Global-norm gradient clipping over the flat gradient buffer (torch.nn.utils.clip_grad_norm_, norm_type 2)
//   clip_norm_kernel : one CTA per chunk; partials[chunk] = sum (grad_scale * g)^2 over the chunk
//   clip_coef_kernel : one CTA; each tensor's partials summed in chunk order (fp64), then the tensors in table order
//                      (fp64); norm = sqrt(total), coef = min(max_norm / (norm + 1e-6), 1) in fp32
//   clip_scale_kernel: one CTA per chunk; g <- g * coef, and nothing at all when coef is exactly 1
__global__ void __launch_bounds__(CHUNK_THREADS)
clip_norm_kernel(const float* __restrict__ g, const int64_t* __restrict__ begin, const int64_t* __restrict__ len,
                 int n_tensors, double* __restrict__ partials, float grad_scale) {
  pdl_wait();
  pdl_trigger();
  const FlatChunk ch = flat_locate(len, n_tensors, blockIdx.x);
  if (ch.l < 0) return;
  int64_t off;
  const int n = flat_chunk_span(begin, len, ch, &off);
  const float* gc = g + off;
  const int n4 = (reinterpret_cast<uintptr_t>(gc) & 15) == 0 ? n / 4 : 0;
  float s = 0.f;
  for (int i = threadIdx.x; i < n4; i += CHUNK_THREADS) {
    const float4 gr = reinterpret_cast<const float4*>(gc)[i];
    const float* gg = &gr.x;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float x = __fmul_rn(gg[k], grad_scale);
      s = __fmaf_rn(x, x, s);
    }
  }
  for (int i = 4 * n4 + threadIdx.x; i < n; i += CHUNK_THREADS) {
    const float x = __fmul_rn(gc[i], grad_scale);
    s = __fmaf_rn(x, x, s);
  }
  const double2 t = flat_block_sum2(s, 0.0);
  if (threadIdx.x == 0) partials[blockIdx.x] = t.x;
}

// Warp w takes tensor t0 + w of each group of CHUNK_THREADS / 32 tensors: lane k sums a contiguous run of the
// tensor's partials in chunk order, then a shuffle butterfly; thread 0 adds the group's tensors in table order.
__global__ void __launch_bounds__(CHUNK_THREADS)
clip_coef_kernel(const int64_t* __restrict__ len, int n_tensors, const double* __restrict__ partials, float max_norm,
                 float* __restrict__ norm_out, float* __restrict__ tensor_norms_out, float* __restrict__ coef_out) {
  constexpr int WARPS = CHUNK_THREADS / 32;
  __shared__ double s_tensor[WARPS];
  pdl_wait();
  pdl_trigger();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double total = 0.0;
  int64_t group_base = 0;  // first chunk of tensor t0
  for (int t0 = 0; t0 < n_tensors; t0 += WARPS) {
    const int l = t0 + warp, t1 = min(t0 + WARPS, n_tensors);
    int64_t base = group_base, cnt = 0, group = 0;
    for (int j = t0; j < t1; ++j) {
      const int64_t c = flat_chunks(len[j]);
      if (j < l) base += c;
      if (j == l) cnt = c;
      group += c;
    }
    double s = 0.0;
    if (l < n_tensors) {
      const int64_t run = (cnt + 31) / 32;
      const int64_t j0 = min(cnt, run * lane), j1 = min(cnt, j0 + run);
      for (int64_t j = j0; j < j1; ++j) s += partials[base + j];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if (lane == 0 && tensor_norms_out) tensor_norms_out[l] = static_cast<float>(sqrt(s));
    }
    if (lane == 0) s_tensor[warp] = s;
    __syncthreads();
    if (threadIdx.x == 0)
      for (int w = 0; w < t1 - t0; ++w) total += s_tensor[w];
    __syncthreads();
    group_base += group;
  }
  if (threadIdx.x == 0) {
    const float norm = static_cast<float>(sqrt(total));
    const float coef = __fdiv_rn(max_norm, __fadd_rn(norm, 1e-6f));
    *norm_out = norm;
    *coef_out = coef > 1.f ? 1.f : coef;  // torch.clamp(max=1) keeps a NaN, where fminf(NaN, 1) would give 1
  }
}

__global__ void __launch_bounds__(CHUNK_THREADS)
clip_scale_kernel(float* __restrict__ g, const int64_t* __restrict__ begin, const int64_t* __restrict__ len,
                  int n_tensors, const float* __restrict__ coef) {
  pdl_wait();
  pdl_trigger();
  const float c = *coef;
  if (c == 1.f) return;  // not clipped: the buffer stays as it is, bitwise what g * 1 gives
  const FlatChunk ch = flat_locate(len, n_tensors, blockIdx.x);
  if (ch.l < 0) return;
  int64_t off;
  const int n = flat_chunk_span(begin, len, ch, &off);
  float* gc = g + off;
  const int n4 = (reinterpret_cast<uintptr_t>(gc) & 15) == 0 ? n / 4 : 0;
  for (int i = threadIdx.x; i < n4; i += CHUNK_THREADS) {
    float4 gr = reinterpret_cast<const float4*>(gc)[i];
    gr.x = __fmul_rn(gr.x, c);
    gr.y = __fmul_rn(gr.y, c);
    gr.z = __fmul_rn(gr.z, c);
    gr.w = __fmul_rn(gr.w, c);
    reinterpret_cast<float4*>(gc)[i] = gr;
  }
  for (int i = 4 * n4 + threadIdx.x; i < n; i += CHUNK_THREADS) gc[i] = __fmul_rn(gc[i], c);
}

}  // namespace loss
}  // namespace lirec

using namespace lirec;

// The arguments both track-loss entry points take; `what` names the loss in the error.
static int check_track_loss_args(const char* what, const float* ints, const float* rels, const int32_t* cand_off,
                                 const int32_t* labels, const int32_t* rels_label, const int32_t* gt_tracks,
                                 const uint8_t* multilab, const lirec_track_loss_cfg& cfg, const float* loss_per_clip,
                                 const int32_t* assign, const float* d_ints, const float* d_rels) {
  LIREC_REQUIRE(ints && cand_off && labels && gt_tracks && multilab && loss_per_clip && assign && d_ints,
                "%s: null pointer", what);
  LIREC_REQUIRE(cfg.n_classes > 0 && cfg.n_rels >= 0, "%s: n_classes=%d n_rels=%d", what, cfg.n_classes,
                cfg.n_rels);
  LIREC_REQUIRE(cfg.n_rels == 0 || (rels && rels_label && d_rels), "%s: rel tensors missing", what);
  LIREC_REQUIRE(cfg.max_slots > 0 && cfg.max_slots <= loss::MAX_SLOTS, "%s: max_slots=%d (limit %d)", what,
                cfg.max_slots, loss::MAX_SLOTS);
  return LIREC_OK;
}

extern "C" int lirec_loss_track_fwd_bwd(const float* ints, const float* rels, const int32_t* cand_off,
                                        int32_t B, const int32_t* labels, const int32_t* rels_label,
                                        const int32_t* gt_tracks, const uint8_t* multilab,
                                        lirec_track_loss_cfg cfg, float* loss_per_clip, int32_t* assign,
                                        float* d_ints, float* d_rels, void* stream) {
  LIREC_ENTER();
  const int rc = check_track_loss_args("track loss", ints, rels, cand_off, labels, rels_label, gt_tracks, multilab,
                                       cfg, loss_per_clip, assign, d_ints, d_rels);
  if (rc != LIREC_OK) return rc;
  if (B <= 0) return LIREC_OK;
  LIREC_CUDA_OK(launch_pdl(loss::track_loss_kernel, dim3(B), dim3(128), 0, static_cast<cudaStream_t>(stream), ints, rels,
                           cand_off, B, labels, rels_label, gt_tracks, multilab, cfg, loss_per_clip, assign, d_ints,
                           d_rels));
  note_launch();
  return LIREC_OK;
}

extern "C" int lirec_loss_rowmargin_fwd_bwd(const float* logits, int64_t ld, int32_t rows, int32_t C,
                                            const int32_t* labels, const uint8_t* weights, float margin,
                                            float scale, float* loss_per_row, float* d_logits, int64_t d_ld,
                                            void* stream) {
  LIREC_ENTER();
  LIREC_REQUIRE(logits && labels && loss_per_row && d_logits && C > 0, "rowmargin loss: bad arguments");
  if (rows <= 0) return LIREC_OK;
  LIREC_CUDA_OK(launch_pdl(loss::rowmargin_kernel, dim3(rows), dim3(128), 0, static_cast<cudaStream_t>(stream), logits,
                           ld, rows, C, labels, weights, margin, scale, loss_per_row, d_logits, d_ld));
  note_launch();
  return LIREC_OK;
}

extern "C" int lirec_loss_ce_fwd_bwd(const float* logits, int64_t ld, int32_t rows, int32_t C, const int32_t* labels,
                                     const float* class_weights, float scale, float* loss_per_row,
                                     float* d_logits, int64_t d_ld, void* stream) {
  LIREC_ENTER();
  LIREC_REQUIRE(logits && labels && loss_per_row && d_logits && C > 0, "ce loss: bad arguments");
  if (rows <= 0) return LIREC_OK;
  loss::ce_kernel<<<rows, 128, 0, static_cast<cudaStream_t>(stream)>>>(logits, ld, C, labels, class_weights, scale,
                                                                      loss_per_row, d_logits, d_ld);
  LIREC_CUDA_OK(cudaGetLastError());
  note_launch();
  return LIREC_OK;
}

extern "C" int lirec_loss_bce_fwd_bwd(const float* logits, int64_t ld, int32_t rows, int32_t C, const int32_t* labels,
                                      const uint8_t* neg_mask, const uint8_t* pos_mask, float scale,
                                      float* loss_per_row, float* d_logits, int64_t d_ld, void* stream) {
  LIREC_ENTER();
  LIREC_REQUIRE(logits && labels && loss_per_row && d_logits && C > 0, "bce loss: bad arguments");
  if (rows <= 0) return LIREC_OK;
  const int grid = (rows + loss::BCE_ROWS_PER_CTA - 1) / loss::BCE_ROWS_PER_CTA;
  LIREC_CUDA_OK(launch_pdl(loss::bce_rows_kernel, dim3(grid), dim3(32 * loss::BCE_ROWS_PER_CTA), 0,
                           static_cast<cudaStream_t>(stream), logits, ld, rows, C, labels, neg_mask, pos_mask, scale,
                           loss_per_row, d_logits, d_ld));
  note_launch();
  return LIREC_OK;
}

extern "C" int lirec_loss_bce_track_fwd_bwd(const float* ints, const float* rels, const int32_t* cand_off, int32_t B,
                                            const int32_t* labels, const int32_t* rels_label, const int32_t* gt_tracks,
                                            const uint8_t* multilab, const uint8_t* pos_mask, lirec_track_loss_cfg cfg,
                                            float* loss_per_clip, int32_t* assign, float* d_ints, float* d_rels,
                                            void* stream) {
  LIREC_ENTER();
  const int rc = check_track_loss_args("bce track loss", ints, rels, cand_off, labels, rels_label, gt_tracks,
                                       multilab, cfg, loss_per_clip, assign, d_ints, d_rels);
  if (rc != LIREC_OK) return rc;
  LIREC_REQUIRE(!cfg.max_neg, "bce track loss: max_neg is a hinge variant, the BCE has no max-negative form");
  if (B <= 0) return LIREC_OK;
  LIREC_CUDA_OK(launch_pdl(loss::bce_track_kernel, dim3(B), dim3(128), 0, static_cast<cudaStream_t>(stream), ints, rels,
                           cand_off, B, labels, rels_label, gt_tracks, multilab, pos_mask, cfg, loss_per_clip, assign,
                           d_ints, d_rels));
  note_launch();
  return LIREC_OK;
}

extern "C" int lirec_predict_tracks(const float* ints, const float* rels, const int32_t* cand_off, int32_t B,
                                    const int32_t* labels, const int32_t* rels_label, const int32_t* gt_tracks,
                                    int32_t n_classes, int32_t n_rels, int32_t* out, void* stream) {
  LIREC_ENTER();
  LIREC_REQUIRE(ints && cand_off && labels && gt_tracks && out && n_classes > 0, "predict: bad arguments");
  LIREC_REQUIRE(n_rels == 0 || (rels && rels_label), "predict: relationship tensors missing");
  if (B <= 0) return LIREC_OK;
  loss::predict_kernel<<<B, 128, 0, static_cast<cudaStream_t>(stream)>>>(ints, rels, cand_off, labels, rels_label,
                                                                        gt_tracks, n_classes, n_rels, out);
  LIREC_CUDA_OK(cudaGetLastError());
  note_launch();
  return LIREC_OK;
}

extern "C" int lirec_adam_flat(float* param, const float* grad, float* exp_avg, float* exp_avg_sq,
                               void* param_bf16, int64_t n, float lr, float beta1, float beta2, float eps,
                               float weight_decay, int32_t step, float grad_scale, int32_t coresident,
                               void* stream) {
  LIREC_ENTER();
  LIREC_REQUIRE(param && grad && exp_avg && exp_avg_sq && n >= 0 && step >= 1, "adam: bad arguments");
  if (n == 0) return LIREC_OK;
  // bias corrections in double like torch's Python-side arithmetic
  const float bc1 = static_cast<float>(1.0 - pow(static_cast<double>(beta1), static_cast<double>(step)));
  const float bc2 = static_cast<float>(1.0 - pow(static_cast<double>(beta2), static_cast<double>(step)));
  // coresident: CTAs that fit next to a resident GEMM CTA (common.cuh), so a pass launched on a side stream really
  // runs during backward instead of after it; same kernel, same arithmetic, same element -> thread order
  static const int co_threads = coresident_threads(reinterpret_cast<const void*>(loss::adam_kernel), 256);
  const int threads = coresident ? co_threads : 256;
  const int grid = static_cast<int>(std::min<int64_t>((n / 4 + threads - 1) / threads + 1, 148 * 16));
  LIREC_CUDA_OK(launch_pdl(loss::adam_kernel, dim3(grid), dim3(threads), 0, static_cast<cudaStream_t>(stream), param, grad,
                           exp_avg, exp_avg_sq, reinterpret_cast<__nv_bfloat16*>(param_bf16), n, lr, beta1, beta2, eps,
                           weight_decay, bc1, sqrtf(bc2), grad_scale));
  note_launch();
  return LIREC_OK;
}

extern "C" int lirec_lamb_flat(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, void* param_bf16,
                               const int64_t* tensor_begin, const int64_t* tensor_len, int32_t n_tensors, int64_t n,
                               double* partials, int64_t n_partials, float lr, float one_minus_beta1,
                               float one_minus_beta2, float eps, float weight_decay, int32_t step, float grad_scale,
                               float* trust_out, void* stream) {
  LIREC_ENTER();
  LIREC_REQUIRE(param && grad && exp_avg && exp_avg_sq && tensor_begin && tensor_len && partials,
                "lamb: null pointer");
  LIREC_REQUIRE(step >= 1, "lamb: step=%d (the first step is 1)", step);
  LIREC_REQUIRE(n_tensors >= 1 && n >= 1, "lamb: n_tensors=%d n=%lld", n_tensors, static_cast<long long>(n));
  const int64_t chunks = LIREC_LAMB_PARTIALS(n, n_tensors);
  LIREC_REQUIRE(n_partials >= chunks, "lamb: partials hold %lld chunks, %lld needed", static_cast<long long>(n_partials),
                static_cast<long long>(chunks));
  LIREC_REQUIRE(chunks <= 0x7fffffff, "lamb: %lld chunks", static_cast<long long>(chunks));
  LIREC_REQUIRE(one_minus_beta1 > 0.f && one_minus_beta1 <= 1.f && one_minus_beta2 > 0.f && one_minus_beta2 <= 1.f,
                "lamb: 1 - beta1 = %g, 1 - beta2 = %g (each in (0, 1])", one_minus_beta1, one_minus_beta2);
  // beta = 1 - (1 - beta) in double: the complement carries the digits that an fp32 beta near 1 drops
  // (fp32 1 - fp32(0.999) is 1.3e-5 off 0.001), and beta formed from it is exact to fp32 rounding
  const double b1 = 1.0 - static_cast<double>(one_minus_beta1), b2 = 1.0 - static_cast<double>(one_minus_beta2);
  // bias corrections in double like lirec_adam_flat
  const double bc1 = 1.0 - pow(b1, static_cast<double>(step));
  const double bc2 = 1.0 - pow(b2, static_cast<double>(step));
  const float inv_bc1 = static_cast<float>(1.0 / bc1), inv_bc2_sqrt = static_cast<float>(1.0 / sqrt(bc2));
  const cudaStream_t s = static_cast<cudaStream_t>(stream);
  double2* part = reinterpret_cast<double2*>(partials);
  // one CTA per chunk; the bound leaves at most n_tensors CTAs without a chunk, and they return at once
  const dim3 grid(static_cast<unsigned>(chunks));
  LIREC_CUDA_OK(launch_pdl(loss::lamb_moments_kernel, grid, dim3(loss::CHUNK_THREADS), 0, s, param, grad, exp_avg,
                           exp_avg_sq, tensor_begin, tensor_len, n_tensors, part, static_cast<float>(b1),
                           static_cast<float>(b2), one_minus_beta1, one_minus_beta2, eps, weight_decay, inv_bc1,
                           inv_bc2_sqrt, grad_scale));
  LIREC_CUDA_OK(launch_pdl(loss::lamb_apply_kernel, grid, dim3(loss::CHUNK_THREADS), 0, s, param, exp_avg, exp_avg_sq,
                           reinterpret_cast<__nv_bfloat16*>(param_bf16), tensor_begin, tensor_len, n_tensors,
                           static_cast<const double2*>(part), trust_out, lr, eps, weight_decay, inv_bc1,
                           inv_bc2_sqrt));
  note_launch(2);
  return LIREC_OK;
}

extern "C" int lirec_grad_clip_flat(float* grad, const int64_t* tensor_begin, const int64_t* tensor_len,
                                    int32_t n_tensors, int64_t n, double* partials, int64_t n_partials,
                                    float max_norm, float grad_scale, float* norm_out, float* tensor_norms_out,
                                    void* stream) {
  LIREC_ENTER();
  LIREC_REQUIRE(grad && tensor_begin && tensor_len && partials && norm_out, "grad clip: null pointer");
  LIREC_REQUIRE(n_tensors >= 1 && n >= 1, "grad clip: n_tensors=%d n=%lld", n_tensors, static_cast<long long>(n));
  const int64_t chunks = LIREC_LAMB_PARTIALS(n, n_tensors);
  LIREC_REQUIRE(n_partials >= chunks, "grad clip: partials hold %lld chunks, %lld needed",
                static_cast<long long>(n_partials), static_cast<long long>(chunks));
  LIREC_REQUIRE(chunks <= 0x7fffffff, "grad clip: %lld chunks", static_cast<long long>(chunks));
  LIREC_REQUIRE(std::isfinite(max_norm) && max_norm > 0.f, "grad clip: max_norm=%g (finite and > 0)", max_norm);
  const cudaStream_t s = static_cast<cudaStream_t>(stream);
  // the chunk sums take the first `chunks` doubles of the partials; the clip coefficient travels from the norm pass
  // to the scale pass in the double after them (the entries hold two doubles each, so it exists)
  float* coef = reinterpret_cast<float*>(partials + chunks);
  const dim3 grid(static_cast<unsigned>(chunks));
  LIREC_CUDA_OK(launch_pdl(loss::clip_norm_kernel, grid, dim3(loss::CHUNK_THREADS), 0, s,
                           static_cast<const float*>(grad), tensor_begin, tensor_len, n_tensors, partials,
                           grad_scale));
  LIREC_CUDA_OK(launch_pdl(loss::clip_coef_kernel, dim3(1), dim3(loss::CHUNK_THREADS), 0, s, tensor_len, n_tensors,
                           static_cast<const double*>(partials), max_norm, norm_out, tensor_norms_out, coef));
  LIREC_CUDA_OK(launch_pdl(loss::clip_scale_kernel, grid, dim3(loss::CHUNK_THREADS), 0, s, grad, tensor_begin,
                           tensor_len, n_tensors, static_cast<const float*>(coef)));
  note_launch(3);
  return LIREC_OK;
}
