// Shared host/device helpers for libtfcb200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <string>

#include "tfcb200.h"

namespace tfcb {

// ---- error plumbing -------------------------------------------------------------------------
std::string& last_error();  // thread local, defined in api.cu
int fail(int code, const char* fmt, ...);
extern std::atomic<int64_t> g_launches;

#define TFCB_CUDA_TRY(expr)                                                                      \
  do {                                                                                           \
    cudaError_t e__ = (expr);                                                                    \
    if (e__ != cudaSuccess) {                                                                    \
      (void)cudaGetLastError();                                                                  \
      return ::tfcb::fail(e__ == cudaErrorMemoryAllocation ? TFCB_OUT_OF_MEMORY : TFCB_CUDA_ERROR, \
                          "CUDA error '%s' at %s:%d", cudaGetErrorString(e__), __FILE__, __LINE__); \
    }                                                                                            \
  } while (0)

#define TFCB_TRY(expr)             \
  do {                             \
    int rc__ = (expr);             \
    if (rc__ != TFCB_OK) return rc__; \
  } while (0)

#define TFCB_LAUNCHED() (::tfcb::g_launches.fetch_add(1, std::memory_order_relaxed))

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

// Stream-ordered allocation helpers (the default mempool keeps freed blocks, so per-call handle
// creation does not hit cudaMalloc after the first use).
int dev_alloc(void** p, size_t bytes, cudaStream_t s);
void dev_free(void* p, cudaStream_t s);

// Multiprocessors of the current device, asked on every call (the process may switch devices); 148 if the query fails.
int device_sm_count();

// Per-CTA dgamma / dbeta partial sums the GDN backward workspace holds (tfcb_gdn_backward_workspace_bytes): every
// backward kernel that writes partials runs at most this many CTAs.
constexpr int kGdnPartSlots = 148;

// ---- range-coder arithmetic shared by the encoder and the decoder -----------------------------
// floor(((span + 1) * c) / 2^p) truncated to 32 bits, for span < 2^32, c <= 2^16, 1 <= p <= 16.
// One IMAD.WIDE.U32 (with the `+ c` folded into the 64-bit addend) and one funnel shift.
// Reference: `(size * u) >> precision` in range_coder.cc:69-70 with the rewrite suggested at :66-68.
__device__ __forceinline__ uint32_t scale_cum(uint32_t span, uint32_t c, uint32_t p) {
  const unsigned long long t = (unsigned long long)span * c + c;
  return (uint32_t)(t >> p);
}

// Device-side first-error record: {code, stream, position, offending value, limit}.
enum DevErr : int { kErrNone = 0, kErrIndex = 1, kErrValue = 2, kErrCapacity = 3, kErrCdf = 4 };
struct DevError {
  int code;
  int aux;
  long long stream;
  long long pos;
  long long value;
  long long limit;
};

__device__ __forceinline__ void report(DevError* e, int code, long long stream, long long pos,
                                       long long value, long long limit, int aux = 0) {
  if (atomicCAS(&e->code, 0, code) == 0) {
    e->stream = stream;
    e->pos = pos;
    e->value = value;
    e->limit = limit;
    e->aux = aux;
    __threadfence();
  }
}

}  // namespace tfcb
