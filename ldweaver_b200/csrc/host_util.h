// Host-side plumbing shared by the C-ABI entry points: error capture (no exceptions or aborts cross the
// ABI), CUDA checks, device buffers, TMA tensor-map encoding through the driver entry point (so the
// library needs no -lcuda at link time).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <exception>
#include <new>

#include <string>
#include <thread>
#include <vector>

#include "../../include/ldw.h"

namespace ldw {

std::string& last_error_ref();
int set_error(int code, const char* fmt, ...);

#define LDW_CUDA(call)                                                                                     \
  do {                                                                                                     \
    cudaError_t e__ = (call);                                                                              \
    if (e__ != cudaSuccess)                                                                                \
      return ldw::set_error(LDW_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
  } while (0)

// No exception crosses the C ABI (include/ldw.h): a host entry point runs its body through this.
template <class F>
inline int guarded(const char* who, F body) {
  try {
    return body();
  } catch (const std::bad_alloc&) {
    return set_error(LDW_ERR_NOMEM, "%s: out of host memory", who);
  } catch (const std::exception& e) {
    return set_error(LDW_ERR_INTERNAL, "%s: %s", who, e.what());
  } catch (...) {
    return set_error(LDW_ERR_INTERNAL, "%s: unknown failure", who);
  }
}

#define LDW_TRY(call)        \
  do {                       \
    int rc__ = (call);       \
    if (rc__ != 0) return rc__; \
  } while (0)

// Runs fn(i) for i in [0, n) on up to `max_threads` host threads (static interleaved split).  fn must not throw.
template <class F>
inline void parallel_for(int64_t n, int max_threads, F fn) {
  int nt = (int)std::min<int64_t>(std::min<int64_t>(n, max_threads), std::max(1u, std::thread::hardware_concurrency()));
  if (nt <= 1) {
    for (int64_t i = 0; i < n; i++) fn(i);
    return;
  }
  std::vector<std::thread> th;
  for (int t = 0; t < nt; t++)
    th.emplace_back([=]() {
      for (int64_t i = t; i < n; i += nt) fn(i);
    });
  for (auto& x : th) x.join();
}

// Device memory comes from a per-device cache of freed blocks: cudaMalloc / cudaFree of the gigabyte-sized operand
// and link arrays cost tens of milliseconds and cudaFree synchronises the device, which would otherwise dominate a
// plan-create / scan / plan-destroy cycle.  Blocks are only handed back after the owning stream has been
// synchronised (all DevBuf owners release after their last use completed).  dev_cache_trim() returns the cached
// blocks of the current device to the driver (called by ldw_destroy and on allocation failure).
cudaError_t dev_alloc(void** p, size_t bytes, size_t* granted);
void dev_free(void* p, size_t granted);
void dev_cache_trim();

// Simple owning device buffer.
struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
  DevBuf() {}
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { release(); }
  void release() {
    if (p) dev_free(p, bytes);
    p = nullptr;
    bytes = 0;
  }
  int alloc(size_t n) {
    release();
    if (n == 0) n = 16;
    size_t granted = 0;
    cudaError_t e = dev_alloc(&p, n, &granted);
    if (e != cudaSuccess) {
      p = nullptr;
      return set_error(LDW_ERR_NOMEM, "cudaMalloc(%zu) failed: %s", n, cudaGetErrorString(e));
    }
    bytes = granted;
    return 0;
  }
  int ensure(size_t n) { return (n <= bytes && p) ? 0 : alloc(n); }
  template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

struct PinnedBuf {
  void* p = nullptr;
  size_t bytes = 0;
  PinnedBuf() {}
  PinnedBuf(const PinnedBuf&) = delete;
  PinnedBuf& operator=(const PinnedBuf&) = delete;
  ~PinnedBuf() { release(); }
  void release() {
    if (p) cudaFreeHost(p);
    p = nullptr;
    bytes = 0;
  }
  int ensure(size_t n) {
    if (n <= bytes && p) return 0;
    release();
    if (n == 0) n = 16;
    cudaError_t e = cudaMallocHost(&p, n);
    if (e != cudaSuccess) {
      p = nullptr;
      return set_error(LDW_ERR_NOMEM, "cudaMallocHost(%zu) failed: %s", n, cudaGetErrorString(e));
    }
    bytes = n;
    return 0;
  }
  template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

// Owning CUDA event.  Destroying it while recorded work is pending is allowed: the driver releases it on completion.
struct Event {
  cudaEvent_t e = nullptr;
  Event() {}
  Event(const Event&) = delete;
  Event& operator=(const Event&) = delete;
  Event(Event&& o) noexcept : e(o.e) { o.e = nullptr; }
  Event& operator=(Event&& o) noexcept {
    if (this != &o) {
      release();
      e = o.e;
      o.e = nullptr;
    }
    return *this;
  }
  ~Event() { release(); }
  void release() {
    if (e) cudaEventDestroy(e);
    e = nullptr;
  }
  int create(unsigned flags = cudaEventDefault) {
    release();
    LDW_CUDA(cudaEventCreateWithFlags(&e, flags));
    return 0;
  }
  operator cudaEvent_t() const { return e; }
};

// 2-D uint8 tensor [rows][kbytes] (kbytes contiguous), box = 128 bytes x box_rows, 128B swizzle.
int make_tmap_u8_sw128(CUtensorMap* out, const void* gptr, uint64_t rows, uint64_t kbytes, uint32_t box_rows);

inline int64_t round_up(int64_t x, int64_t m) { return (x + m - 1) / m * m; }

}  // namespace ldw
