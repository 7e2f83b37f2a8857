// common.h -- error plumbing shared by the C-ABI translation units.
#pragma once
#include <cstdarg>
#include <cstddef>
#include <cstdio>
#include <cstring>
#include <cuda_runtime.h>

#include "../../include/walker_b200.h"

namespace wb {

// last error message of the calling thread (wb_last_error)
char* last_error_buffer();
int32_t fail(int32_t code, const char* fmt, ...);
// true when a usable sm_100 device is current; otherwise records the error
int32_t require_device();

// Pinned (page-locked) host memory is addressable from the device under unified addressing: the device-side alias of `p`, or
// null when `p` is ordinary pageable memory
inline void* device_alias_of_pinned(const void* p, size_t bytes) {
  cudaPointerAttributes a{}, b{};
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess || a.type != cudaMemoryTypeHost || !a.devicePointer) {
    cudaGetLastError();
    return nullptr;
  }
  // the last byte must be page-locked too and alias at the same distance (one contiguous mapping, or pages pinned by wb_host_pin)
  const char* last = static_cast<const char*>(p) + bytes - 1;
  if (cudaPointerGetAttributes(&b, last) != cudaSuccess || b.type != cudaMemoryTypeHost ||
      static_cast<char*>(b.devicePointer) - static_cast<char*>(a.devicePointer) != (ptrdiff_t)(bytes - 1)) {
    cudaGetLastError();
    return nullptr;
  }
  return a.devicePointer;
}

#define WB_CUDA(expr)                                                                             \
  do {                                                                                            \
    cudaError_t _e = (expr);                                                                      \
    if (_e != cudaSuccess) return wb::fail(WB_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(_e)); \
  } while (0)

#define WB_REQUIRE(cond, msg)                             \
  do {                                                    \
    if (!(cond)) return wb::fail(WB_ERR_INVALID, "%s", msg); \
  } while (0)

inline size_t align16(size_t b) { return (b + 15) / 16 * 16; }

// The table of one call (items, Adam corrections, copy pairs ...): filled in pinned host memory and uploaded to its device copy
// with one copy.  The pinned copy is reused by the next call, so that call first waits until this upload has read it.
struct PinnedTable {
  char* host = nullptr;
  char* dev = nullptr;
  size_t bytes = 0;
  cudaEvent_t copied = nullptr;  // the previous upload has left the pinned copy

  PinnedTable() = default;
  PinnedTable(const PinnedTable&) = delete;
  PinnedTable& operator=(const PinnedTable&) = delete;
  ~PinnedTable() {
    if (host) cudaFreeHost(host);
    cudaFree(dev);
    if (copied) cudaEventDestroy(copied);
  }
  // host / dev at least `want` bytes long, once the previous upload has left the pinned copy
  int32_t reserve(size_t want) {
    if (!copied) WB_CUDA(cudaEventCreateWithFlags(&copied, cudaEventDisableTiming));
    WB_CUDA(cudaEventSynchronize(copied));
    if (want > bytes) {
      if (host) cudaFreeHost(host);
      cudaFree(dev);
      host = nullptr;
      dev = nullptr;
      bytes = 0;
      WB_CUDA(cudaHostAlloc(&host, want, cudaHostAllocDefault));
      WB_CUDA(cudaMalloc(&dev, want));
      bytes = want;
    }
    return WB_OK;
  }
  // the first `used` bytes of the pinned copy -> dev, enqueued on `stream`
  int32_t upload(size_t used, cudaStream_t stream) {
    WB_CUDA(cudaMemcpyAsync(dev, host, used, cudaMemcpyHostToDevice, stream));
    WB_CUDA(cudaEventRecord(copied, stream));
    return WB_OK;
  }
};

}  // namespace wb
