// dp.cu — data-parallel gradient exchange over NVSwitch multicast, bucket by bucket.
//
// The reference is single-process (SURVEY.md §2.3); data-parallel training over clips adds exactly one
// exchange per step: the sum of the flat fp32 gradient buffer over ranks, followed by Adam
// (reference optimizer: torch.optim.Adam, mlp/model.py:599-601).  The stock way is ncclAllReduce and
// then the Adam kernel, both after the last backward launch.  Here the flat gradient buffer is cut into
// buckets (lirec_b200/dp.py: gate + heads, 53 % of the bytes and final ~0.6 ms before backward ends, and the
// encoders) and each bucket runs, on whatever stream the caller chooses, the chain
//
//   barrier   cross-GPU: every rank's backward has written this bucket (flags in peer memory,
//             release/acquire at system scope; one CTA);
//   reduce    each rank reduces ITS 1/world shard of the bucket inside the switch
//             (multimem.ld_reduce.add.v4.f32 on the multicast address pulls the shard from all ranks and
//             sums it in the NVSwitch) and broadcasts the sum to every rank with one multimem.st — the
//             bucket is reduced in place, 1/world of it leaves each GPU once and arrives once, both link
//             directions busy at the same time;
//   barrier   all shards have landed everywhere and nobody reads peer memory any more (so the next
//             backward may overwrite the gradients);
//
// followed by lirec_adam_flat over the bucket.  The first bucket's chain is launched on a side stream as
// soon as backward has recorded its "head gradients final" event (lirec_model_backward), so its exchange
// and its Adam pass overlap the second-layer / first-layer backward stages.
//
// Round 1 did all of this in ONE kernel whose CTAs spun on each other (grid-wide flags): that needs every
// CTA co-resident, which a plain launch does not guarantee (ADVICE r1).  The chain above is separate
// launches ordered by the stream: the only spin left is the single-CTA cross-GPU barrier, which waits for
// PEERS and never for another CTA of its own grid.
//
// The gradient buffer must be symmetric memory mapped into a multicast object on every rank
// (lirec_b200/dp.py allocates it with torch.distributed._symmetric_memory; torch only provides the
// allocation and the rendezvous, no arithmetic).  Every spin is bounded: a dead peer traps (kernel error)
// instead of hanging the GPU forever.
#include <algorithm>
#include <cmath>

#include "common.cuh"

namespace lirec {
namespace dp {

constexpr int THREADS = 256;
constexpr int MAX_CHANNELS = 4;                 // independent chains in flight (one per bucket)
constexpr uint32_t SPIN_LIMIT = 1u << 28;       // minutes of NVLink round trips

__device__ __forceinline__ uint32_t cas_release_sys(uint32_t* p, uint32_t cmp, uint32_t val) {
  uint32_t old;
  asm volatile("atom.global.release.sys.cas.b32 %0, [%1], %2, %3;" : "=r"(old) : "l"(p), "r"(cmp), "r"(val) : "memory");
  return old;
}
__device__ __forceinline__ uint32_t cas_acquire_sys(uint32_t* p, uint32_t cmp, uint32_t val) {
  uint32_t old;
  asm volatile("atom.global.acquire.sys.cas.b32 %0, [%1], %2, %3;" : "=r"(old) : "l"(p), "r"(cmp), "r"(val) : "memory");
  return old;
}
__device__ __forceinline__ float4 multimem_ld_reduce_add(const float* mc) {
  float4 v;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(mc) : "memory");
  return v;
}
__device__ __forceinline__ void multimem_st(float* mc, float4 v) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};"
               ::"l"(mc), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// flag[slot * world + src] in the flag buffer of rank dst: "src has reached `slot`".  A put flips the
// peer's slot 0 -> 1 (spinning while the previous use is still unconsumed), a wait flips the local slot
// 1 -> 0, so the slots reset themselves and the barrier is reusable without an epoch.
__global__ void __launch_bounds__(32) barrier_kernel(uint32_t* const* flags, int rank, int world, int slot) {
  const int t = threadIdx.x;
  __threadfence_system();        // everything earlier kernels of this stream wrote is visible before the signal
  if (t < world) {
    uint32_t spins = 0;
    uint32_t* remote = flags[t] + slot * world + rank;
    while (cas_release_sys(remote, 0u, 1u) != 0u) {
      if (++spins > SPIN_LIMIT) __trap();
      __nanosleep(64);
    }
    uint32_t* local = flags[rank] + slot * world + t;
    spins = 0;
    while (cas_acquire_sys(local, 1u, 0u) != 1u) {
      if (++spins > SPIN_LIMIT) __trap();
      __nanosleep(64);
    }
  }
  __threadfence_system();
}

// This rank's shard [beg4, end4) (in float4 units) of a bucket: reduced in the switch, broadcast to all.
// Four independent 16-byte reductions in flight per thread: an in-switch reduction is a ~3 us round trip, so
// the links are only covered by many outstanding requests.
__global__ void __launch_bounds__(THREADS) reduce_bcast_kernel(float* __restrict__ g_mc, int64_t beg4, int64_t end4) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  int64_t i = beg4 + blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  for (; i + 3 * stride < end4; i += 4 * stride) {
    const float4 a = multimem_ld_reduce_add(g_mc + 4 * i);
    const float4 b = multimem_ld_reduce_add(g_mc + 4 * (i + stride));
    const float4 c = multimem_ld_reduce_add(g_mc + 4 * (i + 2 * stride));
    const float4 d = multimem_ld_reduce_add(g_mc + 4 * (i + 3 * stride));
    multimem_st(g_mc + 4 * i, a);
    multimem_st(g_mc + 4 * (i + stride), b);
    multimem_st(g_mc + 4 * (i + 2 * stride), c);
    multimem_st(g_mc + 4 * (i + 3 * stride), d);
  }
  for (; i < end4; i += stride) multimem_st(g_mc + 4 * i, multimem_ld_reduce_add(g_mc + 4 * i));
  __threadfence_system();        // this thread's broadcasts are performed before the kernel retires
}

// ---- exchange + Adam + parameter broadcast in one pass (ZeRO-1 style) -----------------------------------
// Each rank owns the Adam moments of ITS 1/world shard only.  For every 16-byte piece of the shard:
//   g   = multimem.ld_reduce.add over all ranks' gradient buffers           (sum inside the switch)
//   p,m,v -> Adam (same arithmetic as loss.cu:adam_kernel), m and v stored locally
//   p'  -> multimem.st into EVERY rank's fp32 parameter buffer, bf16(p') -> every rank's bf16 shadow
// so the summed gradients never travel back: the broadcast carries 6 bytes per parameter (fp32 + bf16) instead of
// 4 bytes of gradient followed by a 30-byte-per-parameter Adam pass over the WHOLE replica on every rank
// (553 MB of HBM traffic per rank and step, 83 us).  Replicas stay bit-identical by construction: every rank,
// the owner included, receives the owner's p' through the same multicast store.
struct ShardAdamArgs {
  const float* g_mc;        // multicast address of the gradient buffer
  const float* p;           // local fp32 parameters
  float* p_mc;              // multicast address of the fp32 parameters
  __nv_bfloat16* pb_mc;     // multicast address of the bf16 shadow
  float* m;
  float* v;
  int64_t beg4, end4;
  float lr, beta1, beta2, eps, wd, bc1, bc2_sqrt, grad_scale;
};

__device__ __forceinline__ void multimem_st_b64(void* mc, uint32_t a, uint32_t b) {
  asm volatile("multimem.st.relaxed.sys.global.v2.f32 [%0], {%1, %2};"
               ::"l"(mc), "f"(__uint_as_float(a)), "f"(__uint_as_float(b)) : "memory");
}

__device__ __forceinline__ void shard_adam_piece(const ShardAdamArgs& a, int64_t i, float4 g) {
  float4 pv = reinterpret_cast<const float4*>(a.p)[i];
  float4 mv = reinterpret_cast<const float4*>(a.m)[i];
  float4 vv = reinterpret_cast<const float4*>(a.v)[i];
  float* pp = &pv.x; const float* gg = &g.x; float* mm = &mv.x; float* vp = &vv.x;
  const float step = a.lr / a.bc1;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const float gv = gg[k] * a.grad_scale + a.wd * pp[k];
    mm[k] = a.beta1 * mm[k] + (1.f - a.beta1) * gv;
    vp[k] = a.beta2 * vp[k] + (1.f - a.beta2) * gv * gv;
    pp[k] -= step * mm[k] / (sqrtf(vp[k]) / a.bc2_sqrt + a.eps);
  }
  reinterpret_cast<float4*>(a.m)[i] = mv;
  reinterpret_cast<float4*>(a.v)[i] = vv;
  multimem_st(a.p_mc + 4 * i, pv);
  const __nv_bfloat162 lo = __floats2bfloat162_rn(pv.x, pv.y), hi = __floats2bfloat162_rn(pv.z, pv.w);
  multimem_st_b64(a.pb_mc + 4 * i, *reinterpret_cast<const uint32_t*>(&lo), *reinterpret_cast<const uint32_t*>(&hi));
}

__global__ void __launch_bounds__(THREADS) reduce_adam_bcast_kernel(const ShardAdamArgs a) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  int64_t i = a.beg4 + blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  for (; i + stride < a.end4; i += 2 * stride) {           // two in-switch reductions in flight per thread
    const float4 g0 = multimem_ld_reduce_add(a.g_mc + 4 * i);
    const float4 g1 = multimem_ld_reduce_add(a.g_mc + 4 * (i + stride));
    shard_adam_piece(a, i, g0);
    shard_adam_piece(a, i + stride, g1);
  }
  for (; i < a.end4; i += stride) shard_adam_piece(a, i, multimem_ld_reduce_add(a.g_mc + 4 * i));
  __threadfence_system();
}

// The same pass over plain peer pointers (P2P loads / stores through NVLink, no multicast): at 2 ranks an
// in-switch reduction also pulls the requester's OWN copy through the switch and a multicast store sends the
// owner its own data back, 147 MB per direction and step against 92 MB for direct peer accesses (measured at
// 2 ranks: 0.30 ms against ncclAllReduce + Adam's 0.26 ms); from 4 ranks on the switch wins (it reads every
// rank's gradients once and replicates one copy of the parameters).  Summation order is fixed (rank 0, 1, ...).
struct PeerShardArgs {
  const char* const* bases;  // device array [world]: every rank's symmetric allocation (peer-mapped)
  int64_t grad_off, param_off, bf16_off;   // byte offsets inside the allocation
  float* m;
  float* v;
  int64_t beg4, end4;
  int32_t rank, world;
  float lr, beta1, beta2, eps, wd, bc1, bc2_sqrt, grad_scale;
};

template <int WORLD>
__global__ void __launch_bounds__(THREADS) reduce_adam_bcast_peer_kernel(const PeerShardArgs a) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  const float step = a.lr / a.bc1;
  const char* base[WORLD];
#pragma unroll
  for (int r = 0; r < WORLD; ++r) base[r] = a.bases[r];
  const float4* p_loc = reinterpret_cast<const float4*>(a.bases[a.rank] + a.param_off);   // (no dynamic index into base[])
  for (int64_t i = a.beg4 + blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < a.end4; i += stride) {
    float4 g[WORLD];
#pragma unroll
    for (int r = 0; r < WORLD; ++r) g[r] = __ldcv(reinterpret_cast<const float4*>(base[r] + a.grad_off) + i);
    float4 pv = p_loc[i];
    float4 mv = reinterpret_cast<const float4*>(a.m)[i];
    float4 vv = reinterpret_cast<const float4*>(a.v)[i];
    float4 gs = g[0];
#pragma unroll
    for (int r = 1; r < WORLD; ++r) { gs.x += g[r].x; gs.y += g[r].y; gs.z += g[r].z; gs.w += g[r].w; }
    float* pp = &pv.x; const float* gg = &gs.x; float* mm = &mv.x; float* vp = &vv.x;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float gv = gg[k] * a.grad_scale + a.wd * pp[k];
      mm[k] = a.beta1 * mm[k] + (1.f - a.beta1) * gv;
      vp[k] = a.beta2 * vp[k] + (1.f - a.beta2) * gv * gv;
      pp[k] -= step * mm[k] / (sqrtf(vp[k]) / a.bc2_sqrt + a.eps);
    }
    reinterpret_cast<float4*>(a.m)[i] = mv;
    reinterpret_cast<float4*>(a.v)[i] = vv;
    const __nv_bfloat162 lo = __floats2bfloat162_rn(pv.x, pv.y), hi = __floats2bfloat162_rn(pv.z, pv.w);
    uint2 w;
    w.x = *reinterpret_cast<const uint32_t*>(&lo);
    w.y = *reinterpret_cast<const uint32_t*>(&hi);
#pragma unroll
    for (int r = 0; r < WORLD; ++r) {
      reinterpret_cast<float4*>(const_cast<char*>(base[r]) + a.param_off)[i] = pv;
      reinterpret_cast<uint2*>(const_cast<char*>(base[r]) + a.bf16_off)[i] = w;
    }
  }
  __threadfence_system();
}

}  // namespace dp
}  // namespace lirec

using namespace lirec;

extern "C" int lirec_dp_flag_words(int32_t world) { return 2 * dp::MAX_CHANNELS * std::max(world, 1); }

// CTA size of a pass: 256 threads alone on the machine, or the largest CTA that fits beside a resident GEMM CTA
// (common.cuh) when the pass is meant to run during backward
template <typename K>
static int pass_threads(K kernel, int32_t coresident) {
  return coresident ? coresident_threads(reinterpret_cast<const void*>(kernel), dp::THREADS) : dp::THREADS;
}

extern "C" int lirec_dp_exchange(void* grad_multicast, int64_t offset, int64_t n, int32_t rank, int32_t world,
                                 const void* flag_ptrs_dev, int32_t channel, int32_t coresident, void* stream) {
  LIREC_ENTER();
  LIREC_REQUIRE(grad_multicast && flag_ptrs_dev, "dp_exchange: null argument");
  LIREC_REQUIRE(n > 0 && n % 4 == 0 && offset >= 0 && offset % 4 == 0,
                "dp_exchange: offset=%lld n=%lld must be multiples of 4 floats", (long long)offset, (long long)n);
  LIREC_REQUIRE(world >= 2 && world <= 32 && rank >= 0 && rank < world, "dp_exchange: rank %d of %d", rank, world);
  LIREC_REQUIRE(channel >= 0 && channel < dp::MAX_CHANNELS, "dp_exchange: channel %d", channel);
  LIREC_REQUIRE((reinterpret_cast<uintptr_t>(grad_multicast) & 15) == 0, "dp_exchange: buffer must be 16-byte aligned");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  uint32_t* const* flags = static_cast<uint32_t* const*>(flag_ptrs_dev);
  float* mc = static_cast<float*>(grad_multicast) + offset;
  const int64_t n4 = n / 4;
  const int64_t beg = n4 * rank / world, end = n4 * (rank + 1) / world;
  dp::barrier_kernel<<<1, 32, 0, s>>>(flags, rank, world, 2 * channel);
  LIREC_CUDA_OK(cudaGetLastError());
  note_launch();
  if (end > beg) {
    const int threads = pass_threads(dp::reduce_bcast_kernel, coresident);
    const int64_t per_cta = static_cast<int64_t>(threads) * 4;
    const int grid = static_cast<int>(std::min<int64_t>((end - beg + per_cta - 1) / per_cta, 148 * 4));
    dp::reduce_bcast_kernel<<<grid, threads, 0, s>>>(mc, beg, end);
    LIREC_CUDA_OK(cudaGetLastError());
    note_launch();
  }
  dp::barrier_kernel<<<1, 32, 0, s>>>(flags, rank, world, 2 * channel + 1);
  LIREC_CUDA_OK(cudaGetLastError());
  note_launch();
  return LIREC_OK;
}

extern "C" int lirec_dp_reduce_adam_bcast(const void* grad_multicast, const float* param, void* param_multicast,
                                          void* param_bf16_multicast, float* exp_avg, float* exp_avg_sq, int64_t n,
                                          float lr, float beta1, float beta2, float eps, float weight_decay,
                                          int32_t step, float grad_scale, int32_t rank, int32_t world,
                                          const void* flag_ptrs_dev, int32_t channel, int32_t coresident,
                                          void* stream) {
  LIREC_ENTER();
  LIREC_REQUIRE(grad_multicast && param && param_multicast && param_bf16_multicast && exp_avg && exp_avg_sq &&
                    flag_ptrs_dev, "dp_reduce_adam_bcast: null argument");
  LIREC_REQUIRE(n > 0 && n % 4 == 0, "dp_reduce_adam_bcast: n=%lld must be a positive multiple of 4", (long long)n);
  LIREC_REQUIRE(world >= 2 && world <= 32 && rank >= 0 && rank < world, "dp_reduce_adam_bcast: rank %d of %d", rank, world);
  LIREC_REQUIRE(channel >= 0 && channel < dp::MAX_CHANNELS && step >= 1, "dp_reduce_adam_bcast: channel %d step %d", channel, step);
  LIREC_REQUIRE(((reinterpret_cast<uintptr_t>(grad_multicast) | reinterpret_cast<uintptr_t>(param) |
                  reinterpret_cast<uintptr_t>(param_multicast) | reinterpret_cast<uintptr_t>(exp_avg) |
                  reinterpret_cast<uintptr_t>(exp_avg_sq)) & 15) == 0 &&
                    (reinterpret_cast<uintptr_t>(param_bf16_multicast) & 7) == 0,
                "dp_reduce_adam_bcast: buffers must be 16-byte aligned");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  uint32_t* const* flags = static_cast<uint32_t* const*>(flag_ptrs_dev);
  dp::ShardAdamArgs a;
  a.g_mc = static_cast<const float*>(grad_multicast);
  a.p = param;
  a.p_mc = static_cast<float*>(param_multicast);
  a.pb_mc = static_cast<__nv_bfloat16*>(param_bf16_multicast);
  a.m = exp_avg; a.v = exp_avg_sq;
  const int64_t n4 = n / 4;
  a.beg4 = n4 * rank / world;
  a.end4 = n4 * (rank + 1) / world;
  a.lr = lr; a.beta1 = beta1; a.beta2 = beta2; a.eps = eps; a.wd = weight_decay;
  a.bc1 = static_cast<float>(1.0 - pow(static_cast<double>(beta1), static_cast<double>(step)));
  a.bc2_sqrt = sqrtf(static_cast<float>(1.0 - pow(static_cast<double>(beta2), static_cast<double>(step))));
  a.grad_scale = grad_scale;
  dp::barrier_kernel<<<1, 32, 0, s>>>(flags, rank, world, 2 * channel);     // every rank's gradients are complete
  LIREC_CUDA_OK(cudaGetLastError());
  note_launch();
  if (a.end4 > a.beg4) {
    const int threads = pass_threads(dp::reduce_adam_bcast_kernel, coresident);
    const int64_t per_cta = static_cast<int64_t>(threads) * 2;
    const int grid = static_cast<int>(std::min<int64_t>((a.end4 - a.beg4 + per_cta - 1) / per_cta, 148 * 8));
    dp::reduce_adam_bcast_kernel<<<grid, threads, 0, s>>>(a);
    LIREC_CUDA_OK(cudaGetLastError());
    note_launch();
  }
  dp::barrier_kernel<<<1, 32, 0, s>>>(flags, rank, world, 2 * channel + 1);  // all shards landed everywhere
  LIREC_CUDA_OK(cudaGetLastError());
  note_launch();
  return LIREC_OK;
}

extern "C" int lirec_dp_reduce_adam_bcast_peer(const void* peer_bases_dev, int64_t grad_off, int64_t param_off,
                                               int64_t bf16_off, float* exp_avg, float* exp_avg_sq, int64_t n,
                                               float lr, float beta1, float beta2, float eps, float weight_decay,
                                               int32_t step, float grad_scale, int32_t rank, int32_t world,
                                               const void* flag_ptrs_dev, int32_t channel, int32_t coresident,
                                               void* stream) {
  LIREC_ENTER();
  LIREC_REQUIRE(peer_bases_dev && exp_avg && exp_avg_sq && flag_ptrs_dev, "dp_reduce_adam_bcast_peer: null argument");
  LIREC_REQUIRE(n > 0 && n % 4 == 0, "dp_reduce_adam_bcast_peer: n=%lld must be a positive multiple of 4", (long long)n);
  LIREC_REQUIRE((world == 2 || world == 4 || world == 8) && rank >= 0 && rank < world,
                "dp_reduce_adam_bcast_peer: rank %d of %d (2, 4 or 8 ranks)", rank, world);
  LIREC_REQUIRE(channel >= 0 && channel < dp::MAX_CHANNELS && step >= 1, "dp_reduce_adam_bcast_peer: channel %d step %d",
                channel, step);
  LIREC_REQUIRE(grad_off % 16 == 0 && param_off % 16 == 0 && bf16_off % 16 == 0 &&
                    ((reinterpret_cast<uintptr_t>(exp_avg) | reinterpret_cast<uintptr_t>(exp_avg_sq)) & 15) == 0,
                "dp_reduce_adam_bcast_peer: offsets / buffers must be 16-byte aligned");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  uint32_t* const* flags = static_cast<uint32_t* const*>(flag_ptrs_dev);
  dp::PeerShardArgs a;
  a.bases = static_cast<const char* const*>(peer_bases_dev);
  a.grad_off = grad_off; a.param_off = param_off; a.bf16_off = bf16_off;
  a.m = exp_avg; a.v = exp_avg_sq;
  const int64_t n4 = n / 4;
  a.beg4 = n4 * rank / world;
  a.end4 = n4 * (rank + 1) / world;
  a.rank = rank; a.world = world;
  a.lr = lr; a.beta1 = beta1; a.beta2 = beta2; a.eps = eps; a.wd = weight_decay;
  a.bc1 = static_cast<float>(1.0 - pow(static_cast<double>(beta1), static_cast<double>(step)));
  a.bc2_sqrt = sqrtf(static_cast<float>(1.0 - pow(static_cast<double>(beta2), static_cast<double>(step))));
  a.grad_scale = grad_scale;
  dp::barrier_kernel<<<1, 32, 0, s>>>(flags, rank, world, 2 * channel);
  LIREC_CUDA_OK(cudaGetLastError());
  note_launch();
  if (a.end4 > a.beg4) {
    const int threads = world == 2   ? pass_threads(dp::reduce_adam_bcast_peer_kernel<2>, coresident)
                        : world == 4 ? pass_threads(dp::reduce_adam_bcast_peer_kernel<4>, coresident)
                                     : pass_threads(dp::reduce_adam_bcast_peer_kernel<8>, coresident);
    const int grid = static_cast<int>(std::min<int64_t>((a.end4 - a.beg4 + threads - 1) / threads, 148 * 8));
    if (world == 2) dp::reduce_adam_bcast_peer_kernel<2><<<grid, threads, 0, s>>>(a);
    else if (world == 4) dp::reduce_adam_bcast_peer_kernel<4><<<grid, threads, 0, s>>>(a);
    else dp::reduce_adam_bcast_peer_kernel<8><<<grid, threads, 0, s>>>(a);
    LIREC_CUDA_OK(cudaGetLastError());
    note_launch();
  }
  dp::barrier_kernel<<<1, 32, 0, s>>>(flags, rank, world, 2 * channel + 1);
  LIREC_CUDA_OK(cudaGetLastError());
  note_launch();
  return LIREC_OK;
}
