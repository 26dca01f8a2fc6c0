// gemm_tcgen05.cu — grouped, persistent, warp-specialised bf16 GEMM for sm_100a.
//
//   D[m,n] = epilogue( alpha * sum_pass sum_k A_pass[m,k] * B_pass[n,k] )
//
// Replaces the nn.Linear forward calls of the reference (cuBLAS sgemm at
// mlp/model.py:281-294, 307-322, 333, 336, 352) and the mm/addmm pairs autograd
// runs for them in backward (mlp/train.py:62).  Design (B200-first, not a port):
//   * operands arrive by TMA (cp.async.bulk.tensor.2d, 128B swizzle) into a
//     multi-stage shared-memory ring guarded by mbarriers;
//   * one elected thread issues tcgen05.mma (kind::f16, bf16 x bf16 -> fp32) with
//     the accumulator in TMEM, double-buffered so the epilogue of tile i overlaps
//     the main loop of tile i+1;
//   * both operands may be K-major or MN-major, so dgrad reads W[out,in] and wgrad
//     reads dY / X in place — no transposed copies in HBM;
//   * a problem is a list of passes (K-segments) accumulated in the same tile:
//     hi/lo split operands (fp32-grade products from bf16 MMAs) and concatenated
//     inputs (GatingUnit's cat, model.py:352) are just extra passes;
//   * one launch covers the tiles of up to 32 problems (the 8 modality Linears of
//     a layer, or all wgrad/dgrad/bias-grad problems of a backward stage);
//   * the epilogue fuses bias, ReLU/tanh, dropout (counter hash), the ReLU / tanh
//     derivative masks of backward, the hi/lo split of the output, and strided or
//     transposed fp32 stores straight into the flat gradient buffer.
#include <cuda.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "gemm.cuh"

namespace lirec {
namespace gemm {

constexpr int BM = 128;       // tile rows  (UMMA M, cta_group::1)
constexpr int BK = 64;        // bf16 elements per k-block = one 128B swizzle span
constexpr int BN128 = 128;    // tile columns of the single-CTA kernel
constexpr int UMMA_K = 16;
// LIREC_GEMM_TRACE=1 (variant build, tools/gemm_trace.py): every role stamps clock64() per tile into a device
// buffer — producer first / last issue, MMA accumulator-free / first-operands / commit, epilogue wake / done.
#ifndef LIREC_GEMM_TRACE
#define LIREC_GEMM_TRACE 0
#endif
#if LIREC_GEMM_TRACE
#define LIREC_TRACE(field)                                                                        \
  do {                                                                                            \
    if (P.trace && trace_k < 64) P.trace[(static_cast<size_t>(unit) * 64 + trace_k) * 8 + (field)] = clock64(); \
  } while (0)
#else
#define LIREC_TRACE(field) do { } while (0)
#endif
constexpr int NUM_EPI_WARPS = 8;
constexpr int NUM_THREADS = 64 + 32 * NUM_EPI_WARPS;
// Warp roles.  The SM's issue arbiter favours the highest warp id of a sub-partition, so the two
// single-thread roles whose latency paces the whole CTA (TMA producer, MMA issuer) take the TOP ids
// and the eight math-heavy epilogue warps the low ones.
constexpr int PRODUCER_WARP = NUM_EPI_WARPS;
constexpr int MMA_WARP = NUM_EPI_WARPS + 1;
constexpr int MAX_PASSES = LIREC_GEMM_MAX_PASSES;
constexpr int MAX_PROBLEMS = LIREC_GEMM_MAX_PROBLEMS;
constexpr int MAX_MAPS = LIREC_GEMM_MAX_MAPS;

// One operand tile fetched per stage: tensor map, MN offset and first K offset (elements).
struct DevLoad {
  int32_t mn_off, k_off;
  int16_t map, pad;
};
// A GROUP of passes that walk the same k range and share operand tiles.  One pipeline stage holds up to two A
// tiles and two B tiles of one k-block and feeds up to four MMAs over them:
//     forward with a hi/lo split input   (x_hi, W) (x_lo, W)                  2 A, 1 B, 2 MMAs
//     weight gradient                    (x_hi, dy_hi) (x_lo, dy_hi) (x_hi, dy_lo)   2 A, 2 B, 3 MMAs
//     first-layer weight gradient        (x, dy_hi) (x, dy_lo)                1 A, 2 B, 2 MMAs
//     data gradient                      (dy_hi, W^T) (dy_lo, W^T)            2 A, 1 B, 2 MMAs
//     single pass                        two consecutive k-blocks per stage   2 A, 2 B, 2 MMAs
// so a shared tile crosses L2 -> shared memory ONCE instead of once per pass: 24 / 21 KB of operand bytes per
// 256x256x64 MMA block instead of 32 KB.  The pair kernel at 32 KB per block asks L2 for ~64 B/clk/SM at the
// full tensor rate, which B200's L2 does not deliver (round-1 ncu: tensor pipe 63-78 % active on the long-K
// launches, 19-28 % on the short-K ones).
struct DevGroup {
  DevLoad a[2], b[2];
  int32_t k_iters;             // stages this group takes per tile (before split-K)
  int32_t k_step;              // K elements advanced per stage (64, or 128 for the two-k-block form)
  int8_t na, nb, nmma, pad;
  int8_t mma_a[4], mma_b[4];   // operand slots of each MMA
};
constexpr int MAX_GROUPS = 3;

struct DevEpi {
  float alpha;
  const float* bias;
  const int32_t* row_flag;
  int32_t act, post;
  float post_scale;
  float drop_p;
  uint32_t drop_seed, drop_stream;
  int32_t drop_col_off;
  const __nv_bfloat16* aux;
  int64_t aux_ld;
  int32_t aux_col_off, aux_lo_off;
  int32_t out_kind;
  void* out;
  int64_t out_ld_m, out_ld_n;
  int32_t out_col_off, out_lo_off;
  int32_t accumulate;
  int32_t vec_ok;      // 16-byte vector stores are legal for this problem
  int32_t aux_vec_ok;  // 16-byte vector loads of aux are legal
  int32_t bias_vec_ok;
};

struct DevProblem {
  int32_t M, N;
  int32_t bn;                  // tile width of this problem (pair kernel: 128 or 256 per CTA pair)
  int32_t tiles_n, tiles_mn;   // tiles per row of tiles / per split slice
  int32_t split_chunk;         // group iterations per split-K slice (0x3fffffff: no split)
  int64_t split_stride;        // elements between the partial outputs of consecutive slices
  int32_t num_groups;
  int32_t a_mn_major, b_mn_major;
  DevGroup group[MAX_GROUPS];
  DevEpi epi;
};

constexpr int EPI_STAGE_BYTES = 4096;   // per epilogue warp: a 32 x 32 chunk as bf16 hi + lo (pair kernel)
constexpr int MAX_ORDERED_TILES = 5120;
constexpr uint16_t NO_TILE = 0xFFFF;

struct alignas(64) GemmParams {
  CUtensorMap maps[MAX_MAPS];
  DevProblem probs[MAX_PROBLEMS];
  int32_t tile_start[MAX_PROBLEMS + 1];
  int32_t num_problems;
  int32_t total_tiles;
  // Host-computed schedule: slot i of the persistent loop (i = blockIdx.x + j * gridDim.x) runs tile
  // tile_order[i] (NO_TILE = idle).  Longest-processing-time-first over a per-tile cost model, so a
  // launch mixing 400-k-block wgrad tiles with 4-k-block dgrad tiles still finishes together.
  int32_t num_slots;
  int32_t use_order;
#if LIREC_GEMM_TRACE
  unsigned long long* trace;    // [units][TRACE_TILES][8] SM-clock stamps per tile (variant build only)
#endif
  uint16_t tile_order[MAX_ORDERED_TILES];
};
static_assert(sizeof(GemmParams) < 32000, "kernel parameter space");

// ---------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// try_wait with a suspend-time hint: the warp sleeps in hardware instead of re-polling (epilogue warps
// wait for a whole mainloop; their polling must not steal issue slots from the TMA / MMA threads)
__device__ __forceinline__ bool mbar_try_wait_hint(uint32_t bar, uint32_t parity, uint32_t ns) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(bar), "r"(parity), "r"(ns)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait_sleepy(uint32_t bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait_hint(bar, parity, 100000u)) {
    if (clock64() - t0 > 4000000000LL) __trap();
  }
}
// Bounded wait: a protocol bug traps (kernel error) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000LL) __trap();  // ~2 s at 1.9 GHz
  }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar,
                                            int32_t c0, int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar)
               : "memory");
}
__device__ __forceinline__ void tc_mma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                            uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// 32 lanes x 32 columns of fp32 accumulator -> 32 registers per thread
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
      "tcgen05.wait::ld.sync.aligned;"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]),
        "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]),
        "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}

// ---- CTA-pair (cta_group::2) variants ---------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
// shared::cluster address of the same smem offset in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_rank(uint32_t local, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local), "r"(rank));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n"
               "barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// Relaxed: the arrive only has to be ordered after this warp's TMEM reads, which the preceding
// tcgen05.fence::before_thread_sync does; a release here would also wait for the epilogue's global stores.
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr)
               : "memory");
}
// TMA load issued by either CTA of a pair: data lands in the issuing CTA's smem, the byte count is
// signalled on an mbarrier that may live in the peer (leader) CTA.
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* map,
                                                 uint32_t bar_cluster, int32_t c0, int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar_cluster), "r"(c0), "r"(c1)
      : "memory");
}
// commit of the leader's outstanding MMAs, arriving on the barrier at this smem offset in BOTH CTAs
__device__ __forceinline__ void tc_commit_pair(uint32_t bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
      ::"r"(bar), "h"(static_cast<uint16_t>(3))
      : "memory");
}
__device__ __forceinline__ void tc_mma_bf16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                                 uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// Shared-memory matrix descriptor (tcgen05), 128B swizzle, version 1.
//   K-major : rows of 64 bf16 (128 B); 8-row groups 1024 B apart (SBO); LBO unused.
//   MN-major: k-rows of 64 MN elements (128 B); 8-k-row groups 1024 B apart (SBO);
//             consecutive 64-wide MN chunks `lbo_bytes` apart (LBO).
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes,
                                                   uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= static_cast<uint64_t>(1) << 46;  // descriptor version (sm_100)
  d |= static_cast<uint64_t>(2) << 61;  // SWIZZLE_128B
  return d;
}

// ---------------------------------------------------------------------------
// Epilogue for one 32-column chunk held by one thread (one output row, as tcgen05.ld 32x32b delivers
// it).  Per element the budget is a few instructions: a 128x128 tile is 16 K elements for eight warps,
// so anything heavier than ~20 instructions per element makes short-K tiles epilogue-bound.  Hence
// the exp-based tanh, one dropout hash word per column pair, and 128-bit loads of the auxiliary tensor.
// ---------------------------------------------------------------------------
__device__ __forceinline__ float tanh_fast(float x) {
  // tanh(x) = 1 - 2 / (e^{2x} + 1): four instructions (mul, ex2, add+rcp, fma), no clamp needed —
  // e^{2x} = inf gives 1 - 0 and e^{2x} = 0 gives 1 - 2.  abs err ~1e-7, like (t - 1) / (t + 1).
  const float t = __expf(2.0f * x);
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(t + 1.0f));   // 1 ulp; rcp(inf) = 0
  return fmaf(-2.0f, r, 1.0f);
}
// hi/lo split of two values at once: hi2 / lo2 = packed bf16 pairs (a in the low half).  Two packed
// converts instead of four scalar ones, and the hi parts come back as floats by shift / mask.
__device__ __forceinline__ void split_bf16x2(float a, float b, uint32_t& hi2, uint32_t& lo2) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  hi2 = *reinterpret_cast<const uint32_t*>(&h);
  const float ha = __uint_as_float(hi2 << 16), hb = __uint_as_float(hi2 & 0xFFFF0000u);
  const __nv_bfloat162 l = __floats2bfloat162_rn(a - ha, b - hb);
  lo2 = *reinterpret_cast<const uint32_t*>(&l);
}

// vec: 16-byte loads of a full chunk; otherwise element loads of the first nvalid columns (the rest read as 0 —
// columns past N may lie past the end of the tensor)
__device__ __forceinline__ void load_bf16x32(const __nv_bfloat16* p, bool vec, int nvalid, float (&out)[32]) {
  if (vec) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const uint4 w = __ldg(reinterpret_cast<const uint4*>(p) + q);
      const uint32_t u[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        out[8 * q + 2 * k] = __uint_as_float(u[k] << 16);
        out[8 * q + 2 * k + 1] = __uint_as_float(u[k] & 0xFFFF0000u);
      }
    }
  } else {
#pragma unroll
    for (int j = 0; j < 32; ++j) out[j] = j < nvalid ? __bfloat162float(p[j]) : 0.f;
  }
}

// The auxiliary tensor of a backward epilogue (gate output for DRELU, concat feature hi + lo for DTANH) of ONE
// 32-column chunk, as raw bf16 pairs.  It is loaded AHEAD of use — for a tile's first chunk before the warp
// waits for the accumulator, for every further chunk right after the previous chunk's math — because a chunk
// that starts its global loads only after tcgen05.ld returned spends most of its time waiting for them (ncu,
// head data-gradient launch: 38 % of all samples on the first use of these loads).
struct AuxRegs {
  uint4 hi[4], lo[4];
  bool ready;
};
__device__ __forceinline__ void aux_prefetch(const DevEpi& e, int M, int N, int m_true, int n0, AuxRegs& a) {
  a.ready = false;
  if ((e.post != LIREC_POST_DRELU && e.post != LIREC_POST_DTANH) || !e.aux_vec_ok || n0 + 32 > N) return;
  const int m = min(m_true, M - 1);
  const uint4* ap = reinterpret_cast<const uint4*>(e.aux + static_cast<int64_t>(m) * e.aux_ld + e.aux_col_off + n0);
#pragma unroll
  for (int q = 0; q < 4; ++q) a.hi[q] = __ldg(ap + q);
  if (e.post == LIREC_POST_DTANH) {
    const uint4* lp = reinterpret_cast<const uint4*>(e.aux + static_cast<int64_t>(m) * e.aux_ld + e.aux_col_off + n0 +
                                                     e.aux_lo_off);
#pragma unroll
    for (int q = 0; q < 4; ++q) a.lo[q] = __ldg(lp + q);
  }
  a.ready = true;
}
__device__ __forceinline__ void unpack_bf16x32(const uint4 (&w4)[4], float (&out)[32]) {
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const uint32_t u[4] = {w4[q].x, w4[q].y, w4[q].z, w4[q].w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      out[8 * q + 2 * k] = __uint_as_float(u[k] << 16);
      out[8 * q + 2 * k + 1] = __uint_as_float(u[k] & 0xFFFF0000u);
    }
  }
}

// `stage`: this warp's 4 KB shared-memory staging area (or nullptr): the transposed split output goes
// through it so that the warp stores 16-byte pieces of eight consecutive rows instead of 2-byte elements.
// `aux`: the chunk's preloaded auxiliary registers (aux.ready == false: loaded here); `after_math()` runs once
// the chunk's values no longer depend on them (the caller issues the next chunk's prefetch there).
template <typename AfterMath>
__device__ __forceinline__ void epilogue_chunk(const DevEpi& e, int M, int N, int m_true, int n0,
                                               const uint32_t (&acc)[32], int64_t slice_off,
                                               bool first_slice, uint8_t* stage, int lane, const AuxRegs& aux,
                                               AfterMath&& after_math) {
  if (n0 >= N) return;                                     // warp-uniform
  const bool staged_t = (e.out_kind == LIREC_OUT_SPLIT_BF16_T) && stage != nullptr;
  // natural-layout outputs of a FULL chunk also leave through the staging area: the accumulator arrives one
  // ROW per thread (tcgen05.ld 32x32b), so direct stores put 16 bytes of 32 different rows into every store
  // instruction — 32 wavefronts and 32 half-written sectors each (in-kernel trace: the epilogue of the
  // second-layer data-gradient tiles, alpha * acc -> fp32, took 7.9 us against 5.3 us of MMA).  Staged, a store
  // instruction carries whole 128-byte lines of 4 rows (fp32) / 64-byte halves of 8 rows (bf16 hi, lo).
  const bool staged_n = stage != nullptr && (N - n0 >= 32) && e.vec_ok &&
                        ((e.out_kind == LIREC_OUT_F32 && e.out_ld_n == 1 && !e.accumulate) ||
                         e.out_kind == LIREC_OUT_SPLIT_BF16);
  if (m_true >= M && !staged_t && !staged_n) return;
  // a staged store is a warp-cooperative step: rows beyond M tag along on the last valid row's
  // inputs (their values are never stored)
  const int m = min(m_true, M - 1);
  const int nvalid = min(32, N - n0);
  const bool full = nvalid == 32;
  // split-K: the partial sums are added up afterwards, so the bias goes into slice 0 only
  const bool bias_on = first_slice && e.bias != nullptr && (e.row_flag == nullptr || e.row_flag[m] != 0);
  float v[32];
#pragma unroll
  for (int j = 0; j < 32; ++j) v[j] = e.alpha * __uint_as_float(acc[j]);
  if (bias_on) {
    if (full && e.bias_vec_ok) {
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const float4 b4 = __ldg(reinterpret_cast<const float4*>(e.bias + n0) + q);
        v[4 * q] += b4.x; v[4 * q + 1] += b4.y; v[4 * q + 2] += b4.z; v[4 * q + 3] += b4.w;
      }
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (j < nvalid) v[j] += __ldg(e.bias + n0 + j);
    }
  }
  if (e.act == LIREC_ACT_RELU) {
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
  } else if (e.act == LIREC_ACT_TANH) {
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = tanh_fast(v[j]);
  }
  const bool drop_on = e.drop_p > 0.f;
  const float keep_scale = drop_on ? 1.0f / (1.0f - e.drop_p) : 1.0f;
  if (e.post == LIREC_POST_DROPOUT) {
    if (drop_on) {
      const uint32_t rkey = drop_row_key(e.drop_seed, e.drop_stream, static_cast<uint32_t>(m));
      const uint32_t thr = drop_threshold(e.drop_p);
      const uint32_t pair0 = static_cast<uint32_t>(n0 + e.drop_col_off) >> 1;   // n0 + col_off is even
#pragma unroll
      for (int j = 0; j < 32; j += 2) {
        const uint32_t w = drop_word(rkey, pair0 + (j >> 1));
        v[j] = ((w & 0xFFFFu) >= thr) ? v[j] * keep_scale : 0.f;
        v[j + 1] = ((w >> 16) >= thr) ? v[j + 1] * keep_scale : 0.f;
      }
    }
  } else if (e.post == LIREC_POST_DRELU) {
    float g[32];
    if (aux.ready) unpack_bf16x32(aux.hi, g);
    else load_bf16x32(e.aux + static_cast<int64_t>(m) * e.aux_ld + e.aux_col_off + n0, full && e.aux_vec_ok, nvalid, g);
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = (g[j] > 0.f) ? v[j] * e.post_scale : 0.f;
  } else if (e.post == LIREC_POST_DTANH) {
    float hi[32], lo[32];
    const __nv_bfloat16* ap = e.aux + static_cast<int64_t>(m) * e.aux_ld + e.aux_col_off + n0;
    if (aux.ready) {
      unpack_bf16x32(aux.hi, hi);
      unpack_bf16x32(aux.lo, lo);
    } else {
      load_bf16x32(ap, full && e.aux_vec_ok, nvalid, hi);
      load_bf16x32(ap + e.aux_lo_off, full && e.aux_vec_ok, nvalid, lo);
    }
    const float unscale = 1.0f - e.drop_p;   // undo the 1/(1-p) of the forward dropout
    uint32_t rkey = 0, thr = 0, pair0 = 0;
    if (drop_on) {
      rkey = drop_row_key(e.drop_seed, e.drop_stream, static_cast<uint32_t>(m));
      thr = drop_threshold(e.drop_p);
      pair0 = static_cast<uint32_t>(n0 + e.drop_col_off) >> 1;
    }
#pragma unroll
    for (int j = 0; j < 32; j += 2) {
      bool k0 = true, k1 = true;
      if (drop_on) {
        const uint32_t w = drop_word(rkey, pair0 + (j >> 1));
        k0 = (w & 0xFFFFu) >= thr;
        k1 = (w >> 16) >= thr;
      }
      const float t0 = (hi[j] + lo[j]) * unscale, t1 = (hi[j + 1] + lo[j + 1]) * unscale;
      v[j] = k0 ? v[j] * keep_scale * (1.0f - t0 * t0) : 0.f;
      v[j + 1] = k1 ? v[j + 1] * keep_scale * (1.0f - t1 * t1) : 0.f;
    }
  }
  if (e.post == LIREC_POST_SIGN_MASK && m_true < M && full) {
    // this thread holds 32 consecutive columns of row m: its ReLU gate is one 32-bit word
    uint32_t mk = 0;
#pragma unroll
    for (int j = 0; j < 32; ++j) mk |= (v[j] > 0.f ? 1u : 0u) << j;
    reinterpret_cast<uint32_t*>(const_cast<__nv_bfloat16*>(e.aux))[static_cast<int64_t>(m_true) * e.aux_ld + (n0 >> 5)] = mk;
  }
  after_math();
  if (staged_n && e.out_kind == LIREC_OUT_F32) {
    // [32 rows][8 x 16 B], piece q of row r at slot q ^ (r & 7): conflict-free both ways
    float4* s4 = reinterpret_cast<float4*>(stage);
#pragma unroll
    for (int q = 0; q < 8; ++q)
      s4[lane * 8 + (q ^ (lane & 7))] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
    __syncwarp();
    const int mbase = m_true - lane;
    float* ob = reinterpret_cast<float*>(e.out) + slice_off + n0;
#pragma unroll
    for (int it = 0; it < 8; ++it) {
      const int row = it * 4 + (lane >> 3), pc = lane & 7;
      const float4 w = s4[row * 8 + (pc ^ (row & 7))];
      if (mbase + row < M)
        *reinterpret_cast<float4*>(ob + static_cast<int64_t>(mbase + row) * e.out_ld_m + pc * 4) = w;
    }
    __syncwarp();
  } else if (staged_n) {
    // bf16 hi | lo: two [32 rows][4 x 16 B] planes, piece j of row r at slot j ^ ((r >> 1) & 3)
    uint4* sh = reinterpret_cast<uint4*>(stage);
    uint4* sl = sh + 128;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      uint32_t h[4], l[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) split_bf16x2(v[8 * j + 2 * q], v[8 * j + 2 * q + 1], h[q], l[q]);
      const int slot = lane * 4 + (j ^ ((lane >> 1) & 3));
      sh[slot] = make_uint4(h[0], h[1], h[2], h[3]);
      sl[slot] = make_uint4(l[0], l[1], l[2], l[3]);
    }
    __syncwarp();
    const int mbase = m_true - lane;
    __nv_bfloat16* ob = reinterpret_cast<__nv_bfloat16*>(e.out) + e.out_col_off + n0;
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      const int row = it * 8 + (lane >> 2), pc = lane & 3;
      const int slot = row * 4 + (pc ^ ((row >> 1) & 3));
      if (mbase + row < M) {
        __nv_bfloat16* o = ob + static_cast<int64_t>(mbase + row) * e.out_ld_m + pc * 8;
        *reinterpret_cast<uint4*>(o) = sh[slot];
        *reinterpret_cast<uint4*>(o + e.out_lo_off) = sl[slot];
      }
    }
    __syncwarp();
  } else if (e.out_kind == LIREC_OUT_F32) {
    float* o = reinterpret_cast<float*>(e.out) + slice_off + static_cast<int64_t>(m) * e.out_ld_m +
               static_cast<int64_t>(n0) * e.out_ld_n;
    if (e.out_ld_n == 1 && e.vec_ok && full) {
      float4* o4 = reinterpret_cast<float4*>(o);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float4 w = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
        if (e.accumulate) {
          const float4 old = o4[j];
          w.x += old.x; w.y += old.y; w.z += old.z; w.w += old.w;
        }
        o4[j] = w;
      }
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        if (j < nvalid) {
          float* p = o + static_cast<int64_t>(j) * e.out_ld_n;
          *p = e.accumulate ? (*p + v[j]) : v[j];
        }
      }
    }
  } else if (staged_t) {
    // transposed hi/lo split through shared memory: element (m, n) -> out[(col_off + n) * ld + m].
    // The warp holds 32 consecutive m (lanes) x 32 n (registers).  It writes the chunk as [n][m] into
    // its staging area, then every lane moves 16 bytes = eight consecutive m of one n: a store
    // instruction covers 8 columns x 64 contiguous bytes (direct 2-byte stores: one column x 64 B).
    __nv_bfloat16* sh = reinterpret_cast<__nv_bfloat16*>(stage);
    __nv_bfloat16* sl = sh + 32 * 32;
    unsigned short* shu = reinterpret_cast<unsigned short*>(sh);
    unsigned short* slu = reinterpret_cast<unsigned short*>(sl);
#pragma unroll
    for (int j = 0; j < 32; j += 2) {
      uint32_t h2, l2;
      split_bf16x2(v[j], v[j + 1], h2, l2);
      shu[j * 32 + lane] = static_cast<unsigned short>(h2);
      shu[(j + 1) * 32 + lane] = static_cast<unsigned short>(h2 >> 16);
      slu[j * 32 + lane] = static_cast<unsigned short>(l2);
      slu[(j + 1) * 32 + lane] = static_cast<unsigned short>(l2 >> 16);
    }
    __syncwarp();
    const int part = lane & 3;
    const int mrow = (m_true - lane) + part * 8;            // first of this lane's eight rows
    const bool rows_ok = mrow + 8 <= M;
    const int64_t lo_off = static_cast<int64_t>(e.out_lo_off) * e.out_ld_m;
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      const int col = it * 8 + (lane >> 2);
      if (col < nvalid && mrow < M) {
        __nv_bfloat16* g = reinterpret_cast<__nv_bfloat16*>(e.out) +
                           static_cast<int64_t>(e.out_col_off + n0 + col) * e.out_ld_m + mrow;
        const __nv_bfloat16* ph = sh + col * 32 + part * 8;
        const __nv_bfloat16* pl = sl + col * 32 + part * 8;
        if (e.vec_ok && rows_ok) {
          *reinterpret_cast<uint4*>(g) = *reinterpret_cast<const uint4*>(ph);
          *reinterpret_cast<uint4*>(g + lo_off) = *reinterpret_cast<const uint4*>(pl);
        } else {
          for (int q = 0; q < 8; ++q) {
            if (mrow + q < M) {
              g[q] = ph[q];
              g[q + lo_off] = pl[q];
            }
          }
        }
      }
    }
    __syncwarp();                                           // the next chunk reuses the staging area
  } else if (e.out_kind == LIREC_OUT_SPLIT_BF16_T) {
    // transposed hi/lo split: element (m, n) -> out[(col_off + n) * ld + m].  The 32 lanes of a warp
    // hold 32 consecutive m, so every store instruction writes 64 contiguous bytes.
    __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(e.out) +
                       static_cast<int64_t>(e.out_col_off + n0) * e.out_ld_m + m;
    const int64_t lo_off = static_cast<int64_t>(e.out_lo_off) * e.out_ld_m;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      if (j < nvalid) {
        __nv_bfloat16 h, l;
        split_bf16(v[j], h, l);
        o[static_cast<int64_t>(j) * e.out_ld_m] = h;
        o[static_cast<int64_t>(j) * e.out_ld_m + lo_off] = l;
      }
    }
  } else {  // hi/lo bf16 split
    __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(e.out) +
                       static_cast<int64_t>(m) * e.out_ld_m + e.out_col_off + n0;
    if (e.vec_ok && full) {
      uint4* ohi = reinterpret_cast<uint4*>(o);
      uint4* olo = reinterpret_cast<uint4*>(o + e.out_lo_off);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        uint32_t h[4], l[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) split_bf16x2(v[8 * j + 2 * q], v[8 * j + 2 * q + 1], h[q], l[q]);
        ohi[j] = make_uint4(h[0], h[1], h[2], h[3]);
        olo[j] = make_uint4(l[0], l[1], l[2], l[3]);
      }
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        if (j < nvalid) {
          __nv_bfloat16 h, l;
          split_bf16(v[j], h, l);
          o[j] = h;
          o[j + e.out_lo_off] = l;
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------
// The kernel body, shared by the two launch forms:
//   PAIR = false  one CTA per 128 x 128 tile (cta_group::1) — launches too small to fill the clusters;
//   PAIR = true   the two SMs of a TPC run ONE 256 x bn tile (cta_group::2, bn = 128 or 256 per problem).
//                 Each CTA stages its own 128 rows of A and bn/2 rows of B, so a k-block costs each SM half
//                 the shared-memory fill and operand reads of two independent 128x128 tiles:
//                   * both CTAs' producers issue their TMA loads; every load signals the LEADER's full barrier;
//                   * the leader's MMA thread issues tcgen05.mma.cta_group::2 and commits (multicast) to the
//                     stage-empty and accumulator-full barriers of both CTAs;
//                   * each CTA's eight epilogue warps drain their own 128 accumulator lanes and arrive on the
//                     leader's accumulator-empty barrier.
// A pipeline stage = four 16 KB slots (A0, A1, B0, B1) holding the operand tiles of one DevGroup step.
// ---------------------------------------------------------------------------
constexpr uint32_t SLOT_BYTES = BM * BK * 2;            // 16 KB: 128 rows x 64 bf16
constexpr uint32_t GSTAGE_BYTES = 4 * SLOT_BYTES;       // 64 KB
constexpr int GSTAGES = 3;

template <bool PAIR>
__device__ __forceinline__ void gemm_body(const GemmParams& P, uint8_t* smem_raw) {
  constexpr int STAGES = GSTAGES;
  constexpr uint32_t ACC_COLS = PAIR ? 256 : 128;  // accumulator buffer stride in TMEM columns
  constexpr uint32_t TMEM_COLS = 2 * ACC_COLS;
  constexpr int TILE_M = PAIR ? 2 * BM : BM;

  // 1024-byte alignment is required by the 128B swizzle atoms
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * GSTAGE_BYTES);
  uint64_t* full_bar = bars;                       // PAIR: used in the leader only
  uint64_t* empty_bar = bars + STAGES;             // per CTA
  uint64_t* tfull_bar = bars + 2 * STAGES;         // per CTA
  uint64_t* tempty_bar = bars + 2 * STAGES + 2;    // PAIR: used in the leader only
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = PAIR ? cluster_ctarank() : 0u;
  const int unit = PAIR ? (blockIdx.x >> 1) : blockIdx.x;          // persistent worker id
  const int num_units = PAIR ? (gridDim.x >> 1) : gridDim.x;

  if (warp == PRODUCER_WARP && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(smem_u32(&full_bar[s]), 1);
      mbar_init(smem_u32(&empty_bar[s]), 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(smem_u32(&tfull_bar[s]), 1);
      mbar_init(smem_u32(&tempty_bar[s]), (PAIR ? 2 : 1) * NUM_EPI_WARPS);  // one arrive per epilogue warp
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == MMA_WARP) {
    if constexpr (PAIR) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                   "r"(TMEM_COLS)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                   "r"(TMEM_COLS)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before();
  __syncthreads();
  if constexpr (PAIR) cluster_sync_all();   // the peer's barriers are initialised before anything signals them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // everything above touched only shared / tensor memory and the kernel parameters: it may run while the
  // previous kernel of the stream is still finishing (programmatic dependent launch)
  pdl_wait();
  pdl_trigger();

  if (warp == PRODUCER_WARP) {
    // ===================== TMA producer (PAIR: both CTAs) =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      int trace_k = -1;
      for (int slot = unit; slot < P.num_slots; slot += num_units) {
        const int t = P.use_order ? static_cast<int>(P.tile_order[slot]) : slot;
        if (t == NO_TILE) continue;
        ++trace_k;
        if (rank == 0) LIREC_TRACE(0);
        int p = 0;
        while (t >= P.tile_start[p + 1]) ++p;
        const DevProblem& pr = P.probs[p];
        const int local = t - P.tile_start[p];
        const int slice = local / pr.tiles_mn, rem = local - slice * pr.tiles_mn;
        const int brows = PAIR ? (pr.bn >> 1) : BN128;                  // B rows this CTA stages
        const int m0 = (rem / pr.tiles_n) * TILE_M + static_cast<int>(rank) * BM;
        const int n0 = (rem % pr.tiles_n) * (PAIR ? pr.bn : BN128) + static_cast<int>(rank) * brows;
        const uint32_t b_bytes = static_cast<uint32_t>(brows) * (BK * 2);
        for (int g = 0; g < pr.num_groups; ++g) {
          const DevGroup& G = pr.group[g];
          const int it_end = min(G.k_iters, (slice + 1) * pr.split_chunk);
          const uint32_t cta_bytes = static_cast<uint32_t>(G.na) * SLOT_BYTES + static_cast<uint32_t>(G.nb) * b_bytes;
          for (int it = slice * pr.split_chunk; it < it_end; ++it) {
            mbar_wait(smem_u32(&empty_bar[stage]), phase ^ 1);
            const uint32_t fb_local = smem_u32(&full_bar[stage]);
            uint32_t fb = fb_local;
            if constexpr (PAIR) {
              if (rank == 0) mbar_expect_tx(fb_local, 2 * cta_bytes);   // both CTAs' bytes land here
              fb = mapa_rank(fb_local, 0);
            } else {
              mbar_expect_tx(fb_local, cta_bytes);
            }
            const uint32_t s0 = smem_u32(smem + stage * GSTAGE_BYTES);
            const int kadv = it * G.k_step;
            for (int j = 0; j < G.na; ++j) {
              const DevLoad& L = G.a[j];
              const CUtensorMap* map = &P.maps[L.map];
              const uint32_t dst = s0 + j * SLOT_BYTES;
              if (!pr.a_mn_major) {
                if constexpr (PAIR) tma_load_2d_pair(dst, map, fb, L.k_off + kadv, L.mn_off + m0);
                else tma_load_2d(dst, map, fb, L.k_off + kadv, L.mn_off + m0);
              } else {
#pragma unroll
                for (int h = 0; h < BM / 64; ++h) {
                  if constexpr (PAIR) tma_load_2d_pair(dst + h * (BK * 128), map, fb, L.mn_off + m0 + h * 64, L.k_off + kadv);
                  else tma_load_2d(dst + h * (BK * 128), map, fb, L.mn_off + m0 + h * 64, L.k_off + kadv);
                }
              }
            }
            for (int j = 0; j < G.nb; ++j) {
              const DevLoad& L = G.b[j];
              const CUtensorMap* map = &P.maps[L.map];
              const uint32_t dst = s0 + (2 + j) * SLOT_BYTES;
              if (!pr.b_mn_major) {
                if constexpr (PAIR) tma_load_2d_pair(dst, map, fb, L.k_off + kadv, L.mn_off + n0);
                else tma_load_2d(dst, map, fb, L.k_off + kadv, L.mn_off + n0);
              } else {
                for (int h = 0; h < brows / 64; ++h) {
                  if constexpr (PAIR) tma_load_2d_pair(dst + h * (BK * 128), map, fb, L.mn_off + n0 + h * 64, L.k_off + kadv);
                  else tma_load_2d(dst + h * (BK * 128), map, fb, L.mn_off + n0 + h * 64, L.k_off + kadv);
                }
              }
            }
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
        }
        if (rank == 0) LIREC_TRACE(1);
      }
    }
  } else if (warp == MMA_WARP) {
    // ===================== MMA issuer (PAIR: leader CTA only) =====================
    if (lane == 0 && rank == 0) {
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      int trace_k = -1;
      for (int slot = unit; slot < P.num_slots; slot += num_units) {
        const int t = P.use_order ? static_cast<int>(P.tile_order[slot]) : slot;
        if (t == NO_TILE) continue;
        ++trace_k;
        int p = 0;
        while (t >= P.tile_start[p + 1]) ++p;
        const DevProblem& pr = P.probs[p];
        // instruction descriptor: D=f32, A=B=bf16, majorness, N>>3, M>>4 (PAIR: M = 256 over the pair)
        const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) |
                               (static_cast<uint32_t>(pr.a_mn_major) << 15) |
                               (static_cast<uint32_t>(pr.b_mn_major) << 16) |
                               (static_cast<uint32_t>((PAIR ? pr.bn : BN128) >> 3) << 17) |
                               (static_cast<uint32_t>(TILE_M >> 4) << 24);
        LIREC_TRACE(2);
        mbar_wait(smem_u32(&tempty_bar[acc]), acc_phase ^ 1);
        tc_fence_after();
        LIREC_TRACE(3);
        const uint32_t tmem_d = tmem_base + static_cast<uint32_t>(acc) * ACC_COLS;
        uint32_t accumulate = 0;
        const int slice = (t - P.tile_start[p]) / pr.tiles_mn;
        for (int g = 0; g < pr.num_groups; ++g) {
          const DevGroup& G = pr.group[g];
          const int it_end = min(G.k_iters, (slice + 1) * pr.split_chunk);
          for (int it = slice * pr.split_chunk; it < it_end; ++it) {
            mbar_wait(smem_u32(&full_bar[stage]), phase);
            tc_fence_after();
            if (g == 0 && it == slice * pr.split_chunk) LIREC_TRACE(4);
            const uint32_t s0 = smem_u32(smem + stage * GSTAGE_BYTES);
            for (int j = 0; j < G.nmma; ++j) {
              const uint32_t sa = s0 + static_cast<uint32_t>(G.mma_a[j]) * SLOT_BYTES;
              const uint32_t sb = s0 + static_cast<uint32_t>(2 + G.mma_b[j]) * SLOT_BYTES;
#pragma unroll
              for (int k = 0; k < BK / UMMA_K; ++k) {
                const uint64_t adesc = pr.a_mn_major
                                           ? make_smem_desc(sa + k * (UMMA_K * 128), BK * 128, 1024)
                                           : make_smem_desc(sa + k * (UMMA_K * 2), 16, 1024);
                const uint64_t bdesc = pr.b_mn_major
                                           ? make_smem_desc(sb + k * (UMMA_K * 128), BK * 128, 1024)
                                           : make_smem_desc(sb + k * (UMMA_K * 2), 16, 1024);
                if constexpr (PAIR) tc_mma_bf16_pair(tmem_d, adesc, bdesc, idesc, accumulate);
                else tc_mma_bf16(tmem_d, adesc, bdesc, idesc, accumulate);
                accumulate = 1;
              }
            }
            // frees the stage (PAIR: in both CTAs) when its MMAs retire
            if constexpr (PAIR) tc_commit_pair(smem_u32(&empty_bar[stage]));
            else tc_commit(smem_u32(&empty_bar[stage]));
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
        }
        // accumulator complete -> epilogue(s)
        if constexpr (PAIR) tc_commit_pair(smem_u32(&tfull_bar[acc]));
        else tc_commit(smem_u32(&tfull_bar[acc]));
        LIREC_TRACE(5);
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else {
    // ===================== epilogue warps (0..7) =====================
    // two warps per TMEM lane quarter; they split the 32-column chunks of the tile between them
    const int quarter = warp & 3;            // TMEM lane quarter this warp may read
    const int half = warp >> 2;              // 0 or 1
    uint8_t* epi_stage = smem + STAGES * GSTAGE_BYTES + 256 + warp * EPI_STAGE_BYTES;
    int acc = 0;
    uint32_t acc_phase = 0;
    int trace_k = -1;
    for (int slot = unit; slot < P.num_slots; slot += num_units) {
      const int t = P.use_order ? static_cast<int>(P.tile_order[slot]) : slot;
      if (t == NO_TILE) continue;
      ++trace_k;
      int p = 0;
      while (t >= P.tile_start[p + 1]) ++p;
      const DevProblem& pr = P.probs[p];
      const int local = t - P.tile_start[p];
      const int slice = local / pr.tiles_mn, rem = local - slice * pr.tiles_mn;
      const int tile_n = PAIR ? pr.bn : BN128;
      const int m0 = (rem / pr.tiles_n) * TILE_M + static_cast<int>(rank) * BM;
      const int n0 = (rem % pr.tiles_n) * tile_n;
      const int chunks = tile_n >> 5;
      // the epilogue descriptor out of parameter space once per tile (indexed constant loads per use cost a
      // long-scoreboard stall each), and the first chunk's auxiliary loads in flight BEFORE the accumulator wait
      const DevEpi e = pr.epi;
      const int M = pr.M, N = pr.N;
      const int m_row = m0 + quarter * 32 + lane;
      const int64_t slice_off = static_cast<int64_t>(slice) * pr.split_stride;
      AuxRegs aux;
      aux_prefetch(e, M, N, m_row, n0 + half * 32, aux);
      mbar_wait_sleepy(smem_u32(&tfull_bar[acc]), acc_phase);
      tc_fence_after();
      if (warp == 0 && lane == 0 && rank == 0) LIREC_TRACE(6);
#pragma unroll 1
      for (int c = half; c < chunks; c += NUM_EPI_WARPS / 4) {
        uint32_t r[32];
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) +
                               static_cast<uint32_t>(acc) * ACC_COLS + static_cast<uint32_t>(c * 32);
        tmem_ld_32x32(taddr, r);
        const int cn = c + NUM_EPI_WARPS / 4;
        epilogue_chunk(e, M, N, m_row, n0 + c * 32, r, slice_off, slice == 0, epi_stage, lane, aux, [&]() {
          if (cn < chunks) aux_prefetch(e, M, N, m_row, n0 + cn * 32, aux);
          else aux.ready = false;
        });
      }
      tc_fence_before();
      __syncwarp();
      if (warp == 0 && lane == 0 && rank == 0) LIREC_TRACE(7);
      if (lane == 0) {
        if constexpr (PAIR) mbar_arrive_cluster(mapa_rank(smem_u32(&tempty_bar[acc]), 0));
        else mbar_arrive(smem_u32(&tempty_bar[acc]));
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
  }

  // PAIR: neither CTA may leave (or free TMEM) while the pair still reads its smem / signals its barriers
  tc_fence_before();
  __syncthreads();
  if constexpr (PAIR) cluster_sync_all();
  if (warp == MMA_WARP) {
    tc_fence_after();
    if constexpr (PAIR)
      asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
    else
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

__global__ void __launch_bounds__(NUM_THREADS, 1)
lirec_gemm_tcgen05_kernel(const __grid_constant__ GemmParams P) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  gemm_body<false>(P, smem_raw);
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1)
lirec_gemm_tcgen05_pair_kernel(const __grid_constant__ GemmParams P) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  gemm_body<true>(P, smem_raw);
}

// ---------------------------------------------------------------------------
// Host side: tensor maps, problem table, launch
// ---------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
      q != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(p);
  return fn;
}

struct MapKey {
  const void* ptr;
  int64_t rows, cols, ld;
  int box_rows;
  bool operator==(const MapKey& o) const {
    return ptr == o.ptr && rows == o.rows && cols == o.cols && ld == o.ld && box_rows == o.box_rows;
  }
};

static int encode_map(CUtensorMap* out, const MapKey& k) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return fail(LIREC_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  if ((reinterpret_cast<uintptr_t>(k.ptr) & 15) != 0 || ((k.ld * 2) & 15) != 0)
    return fail(LIREC_ERR_ARG, "GEMM operand %p (ld=%lld) is not 16-byte aligned", k.ptr,
                (long long)k.ld);
  if (k.rows <= 0 || k.cols <= 0)
    return fail(LIREC_ERR_ARG, "GEMM operand with empty extent (%lld x %lld)", (long long)k.rows,
                (long long)k.cols);
  cuuint64_t gdim[2] = {static_cast<cuuint64_t>(k.cols), static_cast<cuuint64_t>(k.rows)};
  cuuint64_t gstr[1] = {static_cast<cuuint64_t>(k.ld) * 2};
  cuuint32_t box[2] = {64, static_cast<cuuint32_t>(k.box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(k.ptr), gdim, gstr,
                  box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return fail(LIREC_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) rows=%lld cols=%lld ld=%lld",
                (int)r, (long long)k.rows, (long long)k.cols, (long long)k.ld);
  return LIREC_OK;
}

// ---- optional per-launch timing (CUDA events on the launching stream), used by bench.py ----
struct ProfRec {
  cudaEvent_t e0, e1;
  double flops;   // executed MMA flops: sum over problems of 2*M*N*K (all passes)
  int tiles, problems;
};
static bool g_prof_on = false;
static std::vector<ProfRec> g_prof;      // records of the current capture
static std::vector<ProfRec> g_prof_pool;  // events are reused across captures
static double g_pending_flops = 0.0;
static int g_pending_problems = 0;

// Longest-processing-time-first assignment of tiles to the `grid` persistent CTAs.
// cost(tile) = k-blocks of its problem + a constant for the epilogue (in k-block units).
static void schedule_tiles(GemmParams& P, int grid) {
  P.use_order = 0;
  P.num_slots = P.total_tiles;
  if (P.total_tiles > MAX_ORDERED_TILES || P.total_tiles >= NO_TILE || grid <= 0) return;
  struct T { int cost; int tile; };
  std::vector<T> tiles;
  tiles.reserve(P.total_tiles);
  bool uniform = true;
  int first_cost = -1;
  for (int p = 0; p < P.num_problems; ++p) {
    int kb = 0;                                     // MMA k-blocks per tile (of one split slice)
    for (int g = 0; g < P.probs[p].num_groups; ++g)
      kb += std::min(P.probs[p].group[g].k_iters, P.probs[p].split_chunk) * P.probs[p].group[g].nmma;
    const DevEpi& e = P.probs[p].epi;
    const int epi = (e.act == LIREC_ACT_TANH || e.post != LIREC_POST_NONE) ? 10 : (e.out_kind == LIREC_OUT_F32 ? 4 : 6);
    const int cost = kb + epi * P.probs[p].bn / 128;
    if (first_cost < 0) first_cost = cost;
    uniform = uniform && (cost == first_cost);
    for (int t = P.tile_start[p]; t < P.tile_start[p + 1]; ++t) tiles.push_back(T{cost, t});
  }
  if (uniform) return;  // identity order is already balanced
  std::stable_sort(tiles.begin(), tiles.end(), [](const T& a, const T& b) { return a.cost > b.cost; });
  std::vector<long long> load(grid, 0);
  std::vector<std::vector<uint16_t>> lists(grid);
  // min-heap over (load, cta); ties go to the lowest cta id so neighbouring tiles run side by side
  std::vector<std::pair<long long, int>> heap;
  heap.reserve(grid);
  for (int c = 0; c < grid; ++c) heap.push_back({0, c});
  auto cmp = [](const std::pair<long long, int>& a, const std::pair<long long, int>& b) { return a > b; };
  std::make_heap(heap.begin(), heap.end(), cmp);
  for (const T& t : tiles) {
    std::pop_heap(heap.begin(), heap.end(), cmp);
    auto& top = heap.back();
    lists[top.second].push_back(static_cast<uint16_t>(t.tile));
    top.first += t.cost;
    std::push_heap(heap.begin(), heap.end(), cmp);
  }
  size_t depth = 0;
  for (auto& l : lists) depth = std::max(depth, l.size());
  if (depth * grid > MAX_ORDERED_TILES) return;
  for (size_t j = 0; j < depth; ++j)
    for (int c = 0; c < grid; ++c) P.tile_order[j * grid + c] = j < lists[c].size() ? lists[c][j] : NO_TILE;
  P.num_slots = static_cast<int>(depth) * grid;
  P.use_order = 1;
}

static int record_begin(ProfRec& rec, const GemmParams& P, cudaStream_t stream) {
  if (!g_prof_on) return LIREC_OK;
  if (!g_prof_pool.empty()) { rec = g_prof_pool.back(); g_prof_pool.pop_back(); }
  else {
    LIREC_CUDA_OK(cudaEventCreate(&rec.e0));
    LIREC_CUDA_OK(cudaEventCreate(&rec.e1));
  }
  rec.flops = g_pending_flops; rec.tiles = P.total_tiles; rec.problems = g_pending_problems;
  LIREC_CUDA_OK(cudaEventRecord(rec.e0, stream));
  return LIREC_OK;
}
static int record_end(ProfRec& rec, cudaStream_t stream) {
  if (!g_prof_on) return LIREC_OK;
  LIREC_CUDA_OK(cudaEventRecord(rec.e1, stream));
  g_prof.push_back(rec);
  return LIREC_OK;
}

}  // namespace gemm
// see common.cuh: what one resident GEMM CTA leaves of an SM's 64 K registers (the larger of the two kernels)
int gemm_free_registers() {
  static int v = -1;
  if (v < 0) {
    int regs = 0;
    for (const void* k : {reinterpret_cast<const void*>(gemm::lirec_gemm_tcgen05_kernel),
                          reinterpret_cast<const void*>(gemm::lirec_gemm_tcgen05_pair_kernel)}) {
      cudaFuncAttributes a;
      if (cudaFuncGetAttributes(&a, k) == cudaSuccess) regs = a.numRegs > regs ? a.numRegs : regs;
      else cudaGetLastError();
    }
    if (regs == 0) regs = 168;
    v = 65536 - (gemm::NUM_THREADS / 32) * ((regs + 7) / 8 * 8) * 32;
  }
  return v;
}
namespace gemm {

constexpr size_t GEMM_SMEM = GSTAGES * GSTAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/ +
                             NUM_EPI_WARPS * EPI_STAGE_BYTES /*epilogue staging*/;
static_assert(GEMM_SMEM <= 232448, "shared memory budget");

#if LIREC_GEMM_TRACE
// Variant build only: one device buffer of clock stamps per launch, copied back synchronously and appended to the
// file named by LIREC_GEMM_TRACE_FILE as "launch <n> units <u> tiles <t>" followed by u * 64 * 8 numbers.
static unsigned long long* g_trace_dev = nullptr;
static int g_trace_launch = 0;
static void trace_prepare(GemmParams& P, int units) {
  P.trace = nullptr;
  if (!getenv("LIREC_GEMM_TRACE_FILE")) return;
  if (!g_trace_dev) cudaMalloc(&g_trace_dev, sizeof(unsigned long long) * 148 * 64 * 8);
  cudaMemset(g_trace_dev, 0, sizeof(unsigned long long) * 148 * 64 * 8);
  P.trace = g_trace_dev;
  (void)units;
}
static void trace_dump(const GemmParams& P, int units, cudaStream_t stream) {
  if (!P.trace) return;
  cudaStreamSynchronize(stream);
  std::vector<unsigned long long> h(static_cast<size_t>(units) * 64 * 8);
  cudaMemcpy(h.data(), g_trace_dev, h.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost);
  FILE* f = fopen(getenv("LIREC_GEMM_TRACE_FILE"), "a");
  if (!f) return;
  fprintf(f, "launch %d units %d tiles %d problems %d\n", g_trace_launch++, units, P.total_tiles, P.num_problems);
  for (size_t i = 0; i < h.size(); ++i) fprintf(f, "%llu%c", h[i], (i % 8 == 7) ? '\n' : ' ');
  fclose(f);
}
#else
static void trace_prepare(GemmParams&, int) {}
static void trace_dump(const GemmParams&, int, cudaStream_t) {}
#endif

static int launch_single(const GemmParams& P, cudaStream_t stream) {
  static bool configured = false;
  static int num_sms = 0;
  if (!configured) {
    LIREC_CUDA_OK(cudaFuncSetAttribute(lirec_gemm_tcgen05_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)GEMM_SMEM));
    int dev = 0;
    LIREC_CUDA_OK(cudaGetDevice(&dev));
    LIREC_CUDA_OK(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev));
    configured = true;
  }
  const int grid = std::min(P.total_tiles, num_sms);
  schedule_tiles(const_cast<GemmParams&>(P), grid);
  trace_prepare(const_cast<GemmParams&>(P), grid);
  ProfRec rec{};
  int rc = record_begin(rec, P, stream);
  if (rc != LIREC_OK) return rc;
  LIREC_CUDA_OK(launch_pdl(lirec_gemm_tcgen05_kernel, dim3(grid), dim3(NUM_THREADS), GEMM_SMEM, stream, P));
  trace_dump(P, grid, stream);
  if ((rc = record_end(rec, stream)) != LIREC_OK) return rc;
  note_launch();
  return LIREC_OK;
}

// CTA-pair launch: one cluster of two CTAs per TPC, persistent over the pair tiles.
static int launch_pair(const GemmParams& P, cudaStream_t stream) {
  static bool configured = false;
  static int max_clusters = 0;
  if (!configured) {
    LIREC_CUDA_OK(cudaFuncSetAttribute(lirec_gemm_tcgen05_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)GEMM_SMEM));
    int dev = 0, num_sms = 0;
    LIREC_CUDA_OK(cudaGetDevice(&dev));
    LIREC_CUDA_OK(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev));
    max_clusters = num_sms / 2;
    // the hardware may not be able to co-schedule a pair on every TPC (e.g. a GPC with an odd SM count)
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(num_sms / 2 * 2);
    cfg.blockDim = dim3(NUM_THREADS);
    cfg.dynamicSmemBytes = GEMM_SMEM;
    int active = 0;
    if (cudaOccupancyMaxActiveClusters(&active, lirec_gemm_tcgen05_pair_kernel, &cfg) == cudaSuccess && active > 0)
      max_clusters = std::min(max_clusters, active);
    else
      (void)cudaGetLastError();
    configured = true;
  }
  const int clusters = std::min(P.total_tiles, max_clusters);
  schedule_tiles(const_cast<GemmParams&>(P), clusters);
  trace_prepare(const_cast<GemmParams&>(P), clusters);
  ProfRec rec{};
  int rc = record_begin(rec, P, stream);
  if (rc != LIREC_OK) return rc;
  LIREC_CUDA_OK(launch_pdl(lirec_gemm_tcgen05_pair_kernel, dim3(2 * clusters), dim3(NUM_THREADS), GEMM_SMEM, stream, P));
  trace_dump(P, clusters, stream);
  if ((rc = record_end(rec, stream)) != LIREC_OK) return rc;
  note_launch();
  return LIREC_OK;
}

// Which kernel runs a launch: the CTA-pair kernel (256-row tiles over two SMs) or the single-CTA 128x128
// kernel.  The pair kernel is the fast one per tile, but at small row counts (the reference's 64-clip
// batches: ~530 candidate rows = 3 pair tiles per column of tiles) its tiles cover under 60 % of the 74
// clusters while the same launch cut into 128x128 tiles still fits one wave of the 148 SMs: then the
// single-CTA kernel finishes sooner.
static bool choose_pair_kernel(const lirec_gemm_problem* probs, int nprobs) {
  long pair_tiles = 0, single_tiles = 0;
  for (int i = 0; i < nprobs; ++i) {
    const lirec_gemm_problem& g = probs[i];
    if (g.M <= 0 || g.N <= 0) continue;
    int max_kb = 0;
    for (int ps = 0; ps < g.num_passes; ++ps) max_kb = std::max(max_kb, (g.pass[ps].k_len + BK - 1) / BK);
    const int split = std::max(1, std::min(g.split_k, max_kb));
    const int bn = g.N > 128 ? 256 : 128;
    pair_tiles += (long)((g.M + 2 * BM - 1) / (2 * BM)) * ((g.N + bn - 1) / bn) * split;
    single_tiles += (long)((g.M + BM - 1) / BM) * ((g.N + 127) / 128) * split;
  }
  return !(pair_tiles * 10 <= 74 * 6 && single_tiles <= 148);
}

int run_grouped(const lirec_gemm_problem* probs, int nprobs, cudaStream_t stream) {
  LIREC_REQUIRE(nprobs >= 0 && nprobs <= MAX_PROBLEMS, "too many GEMM problems (%d > %d)", nprobs,
                MAX_PROBLEMS);
  const bool pair = choose_pair_kernel(probs, nprobs);
  const int tile_m = pair ? 2 * BM : BM;
  static thread_local GemmParams P;  // 16 KB: keep it off the stack
  std::vector<MapKey> keys;
  keys.reserve(MAX_MAPS);
  // A pass reads exactly [k_off, k_off + k_len) of its operands, but TMA fetches whole 64-element k-blocks: when
  // k_len is not a multiple of 64 the pass's map ends its K extent (cols K-major, rows MN-major) at k_off + k_len,
  // so the rest of the last k-block is zero fill instead of the operand's next columns / rows.
  auto map_index = [&](const lirec_operand& op, bool mn_major, int tile_mn, int k_off, int k_len) -> int {
    MapKey k{op.ptr, op.rows, op.cols, op.ld, mn_major ? BK : tile_mn};
    if (k_len % BK != 0) {
      int64_t& k_extent = mn_major ? k.rows : k.cols;
      k_extent = std::min<int64_t>(k_extent, static_cast<int64_t>(k_off) + k_len);
    }
    for (size_t i = 0; i < keys.size(); ++i)
      if (keys[i] == k) return (int)i;
    if ((int)keys.size() >= MAX_MAPS) return -1;
    keys.push_back(k);
    return (int)keys.size() - 1;
  };

  // largest problems first so the static round-robin tile schedule balances
  std::vector<int> order;
  std::vector<double> cost(nprobs, 0.0);
  for (int i = 0; i < nprobs; ++i) {
    if (probs[i].M <= 0 || probs[i].N <= 0) continue;
    int64_t k = 0;
    for (int ps = 0; ps < probs[i].num_passes; ++ps) k += probs[i].pass[ps].k_len;
    cost[i] = (double)k;
    order.push_back(i);
  }
  std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return cost[a] > cost[b]; });

  int np = 0, tiles = 0;
  for (int idx : order) {
    const lirec_gemm_problem& g = probs[idx];
    LIREC_REQUIRE(g.num_passes >= 1 && g.num_passes <= MAX_PASSES, "problem %d: num_passes=%d", idx,
                  g.num_passes);
    DevProblem& d = P.probs[np];
    d.M = g.M;
    d.N = g.N;
    // pair kernel: 256 x 256 tiles, 256 x 128 for narrow outputs (heads, bias gradients)
    d.bn = pair ? (g.N > 128 ? 256 : 128) : 128;
    const int b_box = pair ? d.bn / 2 : d.bn;       // B rows one CTA stages per k-block
    const int tiles_m = (g.M + tile_m - 1) / tile_m;
    d.tiles_n = (g.N + d.bn - 1) / d.bn;
    d.tiles_mn = tiles_m * d.tiles_n;
    int max_kb = 0;
    for (int ps = 0; ps < g.num_passes; ++ps) max_kb = std::max(max_kb, (g.pass[ps].k_len + BK - 1) / BK);
    const int split = split_k_slices(max_kb, g.split_k);
    LIREC_REQUIRE(split == 1 || g.epi.out_kind == LIREC_OUT_F32, "problem %d: split-K needs an fp32 output", idx);
    LIREC_REQUIRE(split == 1 || (g.epi.act == LIREC_ACT_NONE && g.epi.post == LIREC_POST_NONE && !g.epi.accumulate),
                  "problem %d: split-K partial sums cannot carry an activation, post op or accumulate", idx);
    LIREC_REQUIRE(g.epi.out_kind == LIREC_OUT_F32 || g.epi.out_kind == LIREC_OUT_SPLIT_BF16 ||
                      g.epi.out_kind == LIREC_OUT_SPLIT_BF16_T,
                  "problem %d: out_kind=%d", idx, g.epi.out_kind);
    LIREC_REQUIRE(!g.epi.accumulate || g.epi.out_kind == LIREC_OUT_F32, "problem %d: accumulate needs an fp32 output",
                  idx);
    d.split_chunk = (split > 1) ? (max_kb + split - 1) / split : 0x3fffffff;
    d.split_stride = g.split_stride;
    d.a_mn_major = g.a_mn_major ? 1 : 0;
    d.b_mn_major = g.b_mn_major ? 1 : 0;
    // ---- passes -> groups: consecutive passes over the same k range that share operand tiles run out of ONE
    // pipeline stage (see DevGroup).  Order of accumulation inside a tile changes, the sum does not.
    struct Spec { int map, mn_off, k_off; };
    auto same = [](const Spec& x, const Spec& y) { return x.map == y.map && x.mn_off == y.mn_off && x.k_off == y.k_off; };
    d.num_groups = 0;
    int cur_kb = -1;
    std::vector<Spec> ga, gb;
    auto flush = [&]() { ga.clear(); gb.clear(); cur_kb = -1; };
    for (int ps = 0; ps < g.num_passes; ++ps) {
      const lirec_gemm_pass& s = g.pass[ps];
      LIREC_REQUIRE(s.k_len > 0, "problem %d pass %d: k_len=%d", idx, ps, s.k_len);
      // a TMA box starts 16-byte aligned along the view's columns (k_off K-major, mn_off MN-major); an unaligned
      // start never completes its load and the pipeline would wait forever
      LIREC_REQUIRE((d.a_mn_major ? s.a_mn_off : s.a_k_off) % 8 == 0 && (d.b_mn_major ? s.b_mn_off : s.b_k_off) % 8 == 0,
                    "problem %d pass %d: offsets along an operand's columns must be multiples of 8 elements", idx, ps);
      const int ia = map_index(s.a, d.a_mn_major, BM, s.a_k_off, s.k_len);
      const int ib = map_index(s.b, d.b_mn_major, b_box, s.b_k_off, s.k_len);
      if (ia < 0 || ib < 0) return fail(LIREC_ERR_LIMIT, "more than %d tensor maps in one launch", MAX_MAPS);
      const Spec sa{ia, s.a_mn_off, s.a_k_off}, sb{ib, s.b_mn_off, s.b_k_off};
      const int kb = (s.k_len + BK - 1) / BK;
      int ja = -1, jb = -1;
      bool fits = d.num_groups > 0 && kb == cur_kb && d.group[d.num_groups - 1].nmma < 4;
      if (fits) {
        for (size_t q = 0; q < ga.size(); ++q) if (same(ga[q], sa)) ja = (int)q;
        for (size_t q = 0; q < gb.size(); ++q) if (same(gb[q], sb)) jb = (int)q;
        if ((ja < 0 && ga.size() >= 2) || (jb < 0 && gb.size() >= 2)) fits = false;
      }
      if (!fits) {
        LIREC_REQUIRE(d.num_groups < MAX_GROUPS, "problem %d: its passes need more than %d operand groups", idx, MAX_GROUPS);
        flush();
        DevGroup& G = d.group[d.num_groups++];
        memset(&G, 0, sizeof(G));
        G.k_iters = kb;
        G.k_step = BK;
        cur_kb = kb;
        ja = jb = -1;
      }
      DevGroup& G = d.group[d.num_groups - 1];
      if (ja < 0) { ja = (int)ga.size(); ga.push_back(sa); G.a[ja] = DevLoad{sa.mn_off, sa.k_off, (int16_t)sa.map, 0}; G.na = (int8_t)ga.size(); }
      if (jb < 0) { jb = (int)gb.size(); gb.push_back(sb); G.b[jb] = DevLoad{sb.mn_off, sb.k_off, (int16_t)sb.map, 0}; G.nb = (int8_t)gb.size(); }
      G.mma_a[G.nmma] = (int8_t)ja;
      G.mma_b[G.nmma] = (int8_t)jb;
      ++G.nmma;
    }
    // a lone pass (nothing to share): two consecutive k-blocks per stage, so three stages still keep six
    // k-blocks in flight; an odd k-block count leaves a one-block tail group
    if (split == 1) {
      const int ng = d.num_groups;
      for (int q = 0; q < ng; ++q) {
        DevGroup& G = d.group[q];
        if (G.nmma != 1 || G.k_iters < 2 || d.num_groups >= MAX_GROUPS + (G.k_iters % 2 == 0 ? 1 : 0)) continue;
        const int kb = G.k_iters;
        if (kb % 2) {                                    // tail group: the last k-block alone
          DevGroup& T = d.group[d.num_groups++];
          T = G;
          T.a[0].k_off += (kb - 1) * BK;
          T.b[0].k_off += (kb - 1) * BK;
          T.k_iters = 1;
        }
        G.a[1] = G.a[0]; G.a[1].k_off += BK;
        G.b[1] = G.b[0]; G.b[1].k_off += BK;
        G.na = G.nb = 2;
        G.nmma = 2;
        G.mma_a[1] = 1; G.mma_b[1] = 1;
        G.k_iters = kb / 2;
        G.k_step = 2 * BK;
      }
    }
    const lirec_epilogue& e = g.epi;
    LIREC_REQUIRE(e.out != nullptr, "problem %d: null output", idx);
    DevEpi& de = d.epi;
    de.alpha = e.alpha;
    de.bias = e.bias;
    de.row_flag = e.row_flag;
    de.act = e.act;
    de.post = e.post;
    de.post_scale = e.post_scale;
    de.drop_p = e.drop.p;
    de.drop_seed = e.drop.seed;
    de.drop_stream = e.drop.stream_id;
    de.drop_col_off = e.drop.col_off;
    de.aux = reinterpret_cast<const __nv_bfloat16*>(e.aux);
    de.aux_ld = e.aux_ld;
    de.aux_col_off = e.aux_col_off;
    de.aux_lo_off = e.aux_lo_off;
    de.out_kind = e.out_kind;
    de.out = e.out;
    de.out_ld_m = e.out_ld_m;
    de.out_ld_n = e.out_ld_n;
    de.out_col_off = e.out_col_off;
    de.out_lo_off = e.out_lo_off;
    de.accumulate = e.accumulate;
    if ((e.post == LIREC_POST_DRELU || e.post == LIREC_POST_DTANH || e.post == LIREC_POST_SIGN_MASK) && e.aux == nullptr)
      return fail(LIREC_ERR_ARG, "problem %d: post op needs aux", idx);
    if (e.post == LIREC_POST_SIGN_MASK &&
        (g.N % 32 != 0 || e.aux_ld < g.N / 32 || (reinterpret_cast<uintptr_t>(e.aux) & 3) != 0))
      return fail(LIREC_ERR_ARG, "problem %d: sign mask needs N %% 32 == 0 and aux_ld >= N / 32 words", idx);
    const uintptr_t ob = reinterpret_cast<uintptr_t>(e.out);
    if (e.out_kind == LIREC_OUT_F32)   // every split-K slice starts 16-byte aligned too
      de.vec_ok = (e.out_ld_n == 1 && (ob & 15) == 0 && (e.out_ld_m % 4) == 0 && (split == 1 || g.split_stride % 4 == 0))
                      ? 1 : 0;
    else if (e.out_kind == LIREC_OUT_SPLIT_BF16_T)   // 16-byte pieces of eight consecutive m (staged store)
      de.vec_ok = ((ob & 15) == 0 && (e.out_ld_m % 8) == 0) ? 1 : 0;
    else
      de.vec_ok = ((ob & 15) == 0 && (e.out_ld_m % 8) == 0 && (e.out_col_off % 8) == 0 &&
                   (e.out_lo_off % 8) == 0)
                      ? 1
                      : 0;
    de.aux_vec_ok = (e.aux != nullptr && (reinterpret_cast<uintptr_t>(e.aux) & 15) == 0 && (e.aux_ld % 8) == 0 &&
                     (e.aux_col_off % 8) == 0 && (e.aux_lo_off % 8) == 0) ? 1 : 0;
    de.bias_vec_ok = (e.bias != nullptr && (reinterpret_cast<uintptr_t>(e.bias) & 15) == 0) ? 1 : 0;
    LIREC_REQUIRE((e.drop.col_off & 1) == 0, "problem %d: dropout col_off must be even", idx);
    P.tile_start[np] = tiles;
    tiles += d.tiles_mn * split;
    ++np;
  }
  P.tile_start[np] = tiles;
  for (int i = np + 1; i <= MAX_PROBLEMS; ++i) P.tile_start[i] = 0x7fffffff;
  P.num_problems = np;
  P.total_tiles = tiles;
  if (tiles == 0) return LIREC_OK;
  if (g_prof_on) {
    g_pending_flops = 0.0;
    g_pending_problems = np;
    for (int idx : order) {
      double k = 0;
      for (int ps = 0; ps < probs[idx].num_passes; ++ps) k += probs[idx].pass[ps].k_len;
      g_pending_flops += 2.0 * probs[idx].M * probs[idx].N * k;
    }
  }
  for (size_t i = 0; i < keys.size(); ++i) {
    int rc = encode_map(&P.maps[i], keys[i]);
    if (rc != LIREC_OK) return rc;
  }
  return pair ? launch_pair(P, stream) : launch_single(P, stream);
}

}  // namespace gemm
}  // namespace lirec

extern "C" int lirec_profile_begin(void) {
  using namespace lirec::gemm;
  for (auto& r : g_prof) g_prof_pool.push_back(r);
  g_prof.clear();
  g_prof_on = true;
  return LIREC_OK;
}

extern "C" int lirec_profile_sample(int32_t on) {
  lirec::gemm::g_prof_on = on != 0;
  return LIREC_OK;
}

extern "C" int lirec_profile_end(float* ms, double* flops, int32_t* tiles, int32_t* problems, int max_records) {
  using namespace lirec::gemm;
  g_prof_on = false;
  int n = 0;
  for (auto& r : g_prof) {
    if (n >= max_records) break;
    if (cudaEventSynchronize(r.e1) != cudaSuccess) return lirec::fail(LIREC_ERR_CUDA, "profile: event sync failed");
    float t = 0.f;
    if (cudaEventElapsedTime(&t, r.e0, r.e1) != cudaSuccess) return lirec::fail(LIREC_ERR_CUDA, "profile: elapsed failed");
    if (ms) ms[n] = t;
    if (flops) flops[n] = r.flops;
    if (tiles) tiles[n] = r.tiles;
    if (problems) problems[n] = r.problems;
    ++n;
  }
  return n;
}

extern "C" int lirec_gemm_grouped(const lirec_gemm_problem* problems_host, int num_problems,
                                  void* stream) {
  LIREC_ENTER();
  LIREC_REQUIRE(problems_host != nullptr || num_problems == 0, "null problem table");
  return lirec::gemm::run_grouped(problems_host, num_problems, static_cast<cudaStream_t>(stream));
}
