// libtfcb200: error plumbing, allocation helpers, ABI bookkeeping.
#include <mutex>

#include "common.cuh"

namespace tfcb {

std::atomic<int64_t> g_launches{0};

std::string& last_error() {
  static thread_local std::string msg;
  return msg;
}

int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  last_error() = buf;
  return code;
}

namespace {
std::once_flag g_pool_once;

void tune_pool() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return;
  cudaMemPool_t pool;
  if (cudaDeviceGetDefaultMemPool(&pool, dev) != cudaSuccess) return;
  // keep freed blocks: handle creation / finalize run once per batch and must not hit cudaMalloc
  unsigned long long keep = ~0ull;
  cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
  (void)cudaGetLastError();
}
}  // namespace

int dev_alloc(void** p, size_t bytes, cudaStream_t s) {
  std::call_once(g_pool_once, tune_pool);
  *p = nullptr;
  if (bytes == 0) bytes = 1;
  cudaError_t e = cudaMallocAsync(p, bytes, s);
  if (e != cudaSuccess) {
    (void)cudaGetLastError();
    *p = nullptr;
    return fail(e == cudaErrorMemoryAllocation ? TFCB_OUT_OF_MEMORY : TFCB_CUDA_ERROR,
                "cudaMallocAsync(%zu bytes) failed: %s", bytes, cudaGetErrorString(e));
  }
  return TFCB_OK;
}

void dev_free(void* p, cudaStream_t s) {
  if (p) {
    if (cudaFreeAsync(p, s) != cudaSuccess) (void)cudaGetLastError();
  }
}

int device_sm_count() {
  int dev = 0, n = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
  return n > 0 ? n : 148;
}

}  // namespace tfcb

extern "C" {

int tfcb_abi_version(void) { return TFCB_ABI_VERSION; }

const char* tfcb_last_error(void) { return tfcb::last_error().c_str(); }

int64_t tfcb_launch_count(void) { return tfcb::g_launches.load(); }

}  // extern "C"
