// gemm.cuh — host entry of the grouped tcgen05 GEMM (gemm_tcgen05.cu).
#pragma once
#include "common.cuh"

namespace lirec {
namespace gemm {
// Split-K slices a problem writes (include/lirec_b200.h): the k-blocks of its longest pass, `kb`, are cut into
// slices of ceil(kb / min(split_k, kb)) k-blocks each, so fewer than split_k slices may come out (kb = 9,
// split_k = 4: three slices of three).  The caller sums exactly this many partial outputs.
inline int split_k_slices(int kb, int split_k) {
  const int split = split_k < kb ? split_k : kb;
  if (split <= 1) return 1;
  const int chunk = (kb + split - 1) / split;
  return (kb + chunk - 1) / chunk;
}
// Encodes the tensor maps, builds the tile table and launches ONE persistent kernel.
int run_grouped(const lirec_gemm_problem* probs, int nprobs, cudaStream_t stream);
}  // namespace gemm
}  // namespace lirec
