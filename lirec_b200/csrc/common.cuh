// common.cuh — shared host/device helpers of liblirec_b200 (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <cstdarg>
#include <cstdio>

#include "../../include/lirec_b200.h"

namespace lirec {

// ---- error plumbing (thread-local text behind lirec_last_error) ------------
char* err_buf();
int fail(int code, const char* fmt, ...);
void note_launch(int n = 1);
void reset_launch_count();
int check_arch();  // LIREC_OK when the current device is sm_100

#define LIREC_CUDA_OK(expr)                                                          \
  do {                                                                               \
    cudaError_t e__ = (expr);                                                        \
    if (e__ != cudaSuccess)                                                          \
      return ::lirec::fail(LIREC_ERR_CUDA, "%s failed: %s (%s:%d)", #expr,           \
                           cudaGetErrorString(e__), __FILE__, __LINE__);             \
  } while (0)

#define LIREC_REQUIRE(cond, ...)                                  \
  do {                                                            \
    if (!(cond)) return ::lirec::fail(LIREC_ERR_ARG, __VA_ARGS__); \
  } while (0)

#define LIREC_ENTER()                      \
  ::lirec::reset_launch_count();           \
  do {                                     \
    int a__ = ::lirec::check_arch();       \
    if (a__ != LIREC_OK) return a__;       \
  } while (0)

// ---- programmatic dependent launch (PDL) -------------------------------------------------------------
// A train step is ~20 dependent launches on one stream; between two of them the stream idles for the launch
// latency of the next grid and for its prologue (TMEM allocation, barrier init, descriptor fetch) — ~3 us each,
// 10 % of a 64-clip step.  Kernels launched through launch_pdl() may be scheduled BEFORE their predecessor has
// finished; each calls pdl_wait() ahead of its first global access (it returns once every prerequisite grid has
// completed and flushed its memory) and pdl_trigger() right after, so its own successor can be set up early too.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                              Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ---- launch shapes that fit NEXT TO a resident GEMM CTA ------------------------------------------------
// The persistent GEMM kernels hold one CTA per SM for a whole launch: 320 threads x 168 registers (82 % of the
// register file) and all but ~1.7 KB of shared memory.  A memory-bound pass meant to run CONCURRENTLY with
// backward (the overlapped part of Adam, the gradient exchange of the gate + head bucket) is only co-scheduled
// if one of its CTAs fits into what is left — 11.7 k registers, no shared memory: a 256-thread CTA of a
// 47-register kernel does not (12.3 k), so the first "overlapped" versions simply ran after the GEMM had left
// the SM.  coresident_threads(kernel) = the largest CTA (multiple of 32, <= cap) of `kernel` that still fits.
int gemm_free_registers();                           // gemm_tcgen05.cu: 64 K minus one GEMM CTA's allocation
int coresident_threads(const void* kernel, int cap);

// ---- dropout hash (mirrored bit-for-bit by oracle/dropout.py) ---------------
__host__ __device__ __forceinline__ uint32_t fmix32(uint32_t h) {
  h ^= h >> 16;
  h *= 0x85EBCA6Bu;
  h ^= h >> 13;
  h *= 0xC2B2AE35u;
  h ^= h >> 16;
  return h;
}
// row-dependent half of the hash, hoisted out of per-column loops
__host__ __device__ __forceinline__ uint32_t drop_row_key(uint32_t seed, uint32_t stream_id,
                                                           uint32_t row) {
  return fmix32(seed ^ (stream_id * 0x9E3779B1u) ^ fmix32(row + 0x7F4A7C15u));
}
// One 32-bit hash word covers two adjacent columns (16 bits each).
__host__ __device__ __forceinline__ uint32_t drop_word(uint32_t row_key, uint32_t col_pair) {
  return fmix32(row_key ^ (col_pair * 0x9E3779B1u + 0x632BE5ABu));
}
// keep threshold on the 16-bit lane: drop iff lane < p * 65536
__host__ __device__ __forceinline__ uint32_t drop_threshold(float p) {
  return static_cast<uint32_t>(p * 65536.0f + 0.5f);
}
__host__ __device__ __forceinline__ bool drop_keep_word(uint32_t word, uint32_t col, uint32_t thr) {
  return ((word >> ((col & 1u) * 16u)) & 0xFFFFu) >= thr;
}
// true if element (row, col) is kept
__host__ __device__ __forceinline__ bool drop_keep(uint32_t row_key, uint32_t col, float p) {
  return drop_keep_word(drop_word(row_key, col >> 1), col, drop_threshold(p));
}

// ---- hi/lo bf16 split: x ~= hi + lo with |err| <= 2^-17 |x| -----------------
__device__ __forceinline__ void split_bf16(float x, __nv_bfloat16& hi, __nv_bfloat16& lo) {
  hi = __float2bfloat16_rn(x);
  lo = __float2bfloat16_rn(x - __bfloat162float(hi));
}

}  // namespace lirec
