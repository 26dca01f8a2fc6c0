// abi.cu — error plumbing and device checks behind the C ABI (include/lirec_b200.h).
#include <cstdlib>
#include <cstring>

#include "common.cuh"

namespace lirec {

static thread_local char g_err[512] = "";
static thread_local int g_launches = 0;

char* err_buf() { return g_err; }

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

void note_launch(int n) { g_launches += n; }
void reset_launch_count() { g_launches = 0; }

// Largest CTA of `kernel` (a multiple of 32 threads, <= cap) whose registers fit beside one resident GEMM CTA.
// Registers are allocated per warp, the per-thread count rounded up to a multiple of 8.
int coresident_threads(const void* kernel, int cap) {
  cudaFuncAttributes a;
  if (cudaFuncGetAttributes(&a, kernel) != cudaSuccess) {
    cudaGetLastError();
    return 64;
  }
  const int per_warp = ((a.numRegs + 7) / 8 * 8) * 32;
  const int warps = gemm_free_registers() / (per_warp > 0 ? per_warp : 1);
  const int t = 32 * (warps < 1 ? 1 : warps);
  return t < cap ? t : cap;
}

// No CPU fallback and no other architecture: anything but sm_100 is an error.
int check_arch() {
  static thread_local int cached_dev = -1;
  static thread_local int cached_rc = LIREC_ERR_ARCH;
  int dev = -1;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess)
    return fail(LIREC_ERR_ARCH, "no CUDA device available (%s); liblirec_b200 has no CPU fallback",
                cudaGetErrorString(e));
  if (dev == cached_dev) {
    if (cached_rc != LIREC_OK) fail(cached_rc, "device %d is not sm_100 (B200 required)", dev);
    return cached_rc;
  }
  int major = 0, minor = 0;
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess ||
      cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev) != cudaSuccess)
    return fail(LIREC_ERR_CUDA, "cannot query compute capability of device %d", dev);
  cached_dev = dev;
  cached_rc = (major == 10) ? LIREC_OK : LIREC_ERR_ARCH;
  if (cached_rc != LIREC_OK)
    return fail(LIREC_ERR_ARCH, "device %d is sm_%d%d; liblirec_b200 is built for sm_100a only", dev,
                major, minor);
  return LIREC_OK;
}

}  // namespace lirec

extern "C" int lirec_abi_version(void) { return LIREC_ABI_VERSION; }
extern "C" const char* lirec_last_error(void) { return lirec::err_buf(); }
extern "C" int lirec_last_launch_count(void) { return lirec::g_launches; }
// Host evaluation of the dropout hash (same code the kernels run), so the numpy mirror in
// oracle/dropout.py can be checked bit-for-bit without a GPU.
extern "C" int lirec_dropout_keep_host(uint32_t seed, uint32_t stream_id, uint32_t row, uint32_t col, float p) {
  return lirec::drop_keep(lirec::drop_row_key(seed, stream_id, row), col, p) ? 1 : 0;
}

extern "C" int lirec_device_check(int device) {
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0)
    return lirec::fail(LIREC_ERR_ARCH, "no CUDA device available; liblirec_b200 has no CPU fallback");
  if (device < 0 || device >= count) return lirec::fail(LIREC_ERR_ARG, "device %d out of range", device);
  int major = 0;
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device) != cudaSuccess)
    return lirec::fail(LIREC_ERR_CUDA, "cannot query device %d", device);
  if (major != 10) return lirec::fail(LIREC_ERR_ARCH, "device %d is not sm_100", device);
  return LIREC_OK;
}
