// Shared host-side plumbing for libferreus_b200: error propagation, device buffers, launch counter.
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <cstdint>
#include <cstdio>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/ferreus_b200.h"

namespace fb {

struct Error : std::runtime_error {
  int code;
  uint64_t index;
  Error(int c, const std::string &msg, uint64_t idx = 0) : std::runtime_error(msg), code(c), index(idx) {}
};

void set_last_error(const std::string &msg);
extern std::atomic<uint64_t> g_launches;

// body of a C entry point: exceptions become error codes and the fb_last_error() message
template <class F>
int guarded(F &&f, uint64_t *bad = nullptr) {
  try {
    f();
    return FB_OK;
  } catch (const Error &e) {
    set_last_error(e.what());
    if (bad && e.code == FB_ERR_POINT_OUTSIDE_TREE) *bad = e.index;
    return e.code;
  } catch (const std::exception &e) {
    set_last_error(e.what());
    return FB_ERR_CUDA;
  }
}

#define FB_CUDA(expr)                                                                              \
  do {                                                                                             \
    cudaError_t _e = (expr);                                                                       \
    if (_e != cudaSuccess)                                                                         \
      throw fb::Error(FB_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e) + " at " +   \
                                       __FILE__ + ":" + std::to_string(__LINE__));                 \
  } while (0)

#define FB_REQUIRE(cond, msg)                                        \
  do {                                                               \
    if (!(cond)) throw fb::Error(FB_ERR_INVALID_ARGUMENT, (msg));    \
  } while (0)

// counts every kernel this library launches (bench.py reports it as gpu_launches)
#define FB_LAUNCH(kernel, grid, block, smem, stream, ...)                 \
  do {                                                                    \
    kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__);           \
    fb::g_launches.fetch_add(1, std::memory_order_relaxed);               \
    FB_CUDA(cudaGetLastError());                                          \
  } while (0)

// Device memory comes from a per-process cache (fmm.cu): a released block is kept and handed out again to the next
// request of a similar size, so repeated fits / tree builds do not pay cudaMalloc / cudaFree (tens of ms each for the
// multi-GB factor pools, and the source of 0.9-1.9 s swings of the 1M-point fit).  dev_free synchronises the device
// first, exactly like the cudaFree it replaces; fb_trim_memory() returns the cache to the driver.
void *dev_alloc(size_t bytes);
void dev_free(void *p);
size_t dev_cache_trim();

template <class T>
struct DBuf {  // device buffer, grows on demand, never shrinks
  T *p = nullptr;
  size_t cap = 0;
  DBuf() = default;
  DBuf(const DBuf &) = delete;
  DBuf &operator=(const DBuf &) = delete;
  ~DBuf() {
    if (p) dev_free(p);
  }
  void reserve(size_t n) {
    if (n <= cap) return;
    if (p) dev_free(p);
    p = nullptr;
    cap = 0;
    p = static_cast<T *>(dev_alloc((n ? n : 1) * sizeof(T)));
    cap = n ? n : 1;
  }
  void upload(const std::vector<T> &h, cudaStream_t s) {
    reserve(h.size());
    if (!h.empty()) FB_CUDA(cudaMemcpyAsync(p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice, s));
  }
  void zero(size_t n, cudaStream_t s) {
    reserve(n);
    if (n) FB_CUDA(cudaMemsetAsync(p, 0, n * sizeof(T), s));
  }
};

template <class T>
struct PinnedBuf {  // pinned host staging buffer
  T *p = nullptr;
  size_t cap = 0;
  ~PinnedBuf() {
    if (p) cudaFreeHost(p);
  }
  void reserve(size_t n) {
    if (n <= cap) return;
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
    FB_CUDA(cudaMallocHost((void **)&p, (n ? n : 1) * sizeof(T)));
    cap = n ? n : 1;
  }
};

}  // namespace fb
