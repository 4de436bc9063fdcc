// host_util.h -- error plumbing and device-memory arena shared by the host side of libavc_b200.
#pragma once
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdio>
#include <string>
#include <utility>
#include <vector>

#include "../../include/avc_b200.h"

namespace avc {

struct Fail {
  int code;
  std::string msg;
};

[[noreturn]] inline void fail(int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  throw Fail{code, buf};
}

#define CK(expr)                                                                              \
  do {                                                                                        \
    cudaError_t e_ = (expr);                                                                  \
    if (e_ != cudaSuccess) fail(AVC_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)

// the library works on the handle's device and leaves the caller's current device as it found it
struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {          // dev < 0: nothing to do
    if (dev < 0) return;
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (prev != dev) cudaSetDevice(dev); else prev = -1;
  }
  DeviceGuard(const DeviceGuard&) = delete;
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

// ---- device memory owned by the handle / a plan ---------------------------------------------
// Slabs released by a finished attack are kept by the handle's pool and handed to the next one:
// cudaFree / cudaMalloc of the 32 MiB slabs cost up to hundreds of ms per attack call otherwise.
struct SlabPool {
  std::vector<std::pair<void*, size_t>> free_slabs;
  size_t held = 0;
  static constexpr size_t kMaxHeld = 6ull << 30;   // beyond this, released slabs go back to the driver
  void* take(size_t sz) {
    for (size_t i = 0; i < free_slabs.size(); ++i)
      if (free_slabs[i].second == sz) {
        void* p = free_slabs[i].first;
        free_slabs.erase(free_slabs.begin() + i);
        held -= sz;
        return p;
      }
    return nullptr;
  }
  void give(void* p, size_t sz) {
    if (held + sz > kMaxHeld) { cudaFree(p); return; }
    free_slabs.emplace_back(p, sz);
    held += sz;
  }
  ~SlabPool() {
    for (auto& s : free_slabs) cudaFree(s.first);
  }
};

struct Arena {
  // bump allocator over zero-initialised slabs: one cudaMalloc per 32 MiB instead of one per tensor
  static constexpr size_t kSlab = 32u << 20;
  std::vector<std::pair<void*, size_t>> slabs;
  SlabPool* pool = nullptr;
  char* cur = nullptr;
  size_t left = 0;
  size_t bytes = 0;
  // Stream the zero fills and uploads are ordered on.  With `ordered` set they are issued asynchronously on the
  // CALLER's stream, so kernels launched there afterwards see them even when that stream is non-blocking (a
  // torch.cuda.Stream): the legacy default stream the plain cudaMemset / cudaMemcpy run on does not order against it.
  cudaStream_t stream = nullptr;
  bool ordered = false;
  Arena() = default;
  explicit Arena(SlabPool* p) : pool(p) {}
  Arena(SlabPool* p, cudaStream_t st) : pool(p), stream(st), ordered(true) {}
  Arena(const Arena&) = delete;
  Arena& operator=(const Arena&) = delete;
  // A finished arena can be rewound and bump-allocated again: a caller that repeats the SAME allocation sequence (one
  // training step after another on the same shapes) gets the same addresses back without a new zero fill of every slab --
  // at 2-3 GB of step buffers the fills were a tenth of a PredictiveModel step.  Buffers then hold the previous step's
  // bytes instead of zeros: only for callers whose kernels write everything they read.  A sequence that diverges from the
  // recorded one simply continues on fresh (zeroed) slabs.
  size_t replay = 0;
  bool replaying = false;
  void rewind() { cur = nullptr; left = 0; replay = 0; replaying = true; }
  float* f(size_t n) {
    const size_t b = (n * sizeof(float) + 255) / 256 * 256;
    if (b > left) {
      const size_t sz = b > kSlab ? (b + kSlab - 1) / kSlab * kSlab : kSlab;
      void* p = nullptr;
      if (replaying && replay < slabs.size() && slabs[replay].second == sz) {
        p = slabs[replay++].first;
      } else {
        if (replaying && replay < slabs.size()) {      // diverged: the rest of the recording is of no use
          for (size_t i = replay; i < slabs.size(); ++i) { if (pool) pool->give(slabs[i].first, slabs[i].second); else cudaFree(slabs[i].first); bytes -= slabs[i].second; }
          slabs.resize(replay);
        }
        p = pool ? pool->take(sz) : nullptr;
        if (!p) CK(cudaMalloc(&p, sz));
        if (ordered) CK(cudaMemsetAsync(p, 0, sz, stream)); else CK(cudaMemset(p, 0, sz));
        slabs.emplace_back(p, sz);
        bytes += sz;
        replay = slabs.size();
      }
      if (b > kSlab) return static_cast<float*>(p);   // dedicated slab, keep the current one
      cur = static_cast<char*>(p);
      left = sz;
    }
    float* r = reinterpret_cast<float*>(cur);
    cur += b;
    left -= b;
    return r;
  }
  template <class T>
  T* raw(size_t n) {
    return reinterpret_cast<T*>(f((n * sizeof(T) + 3) / 4));
  }
  float* upload(const std::vector<float>& v) {
    float* p = f(v.size());
    // pageable source: the async form stages the bytes before it returns, the device copy is ordered on `stream`
    if (ordered) CK(cudaMemcpyAsync(p, v.data(), v.size() * sizeof(float), cudaMemcpyHostToDevice, stream));
    else CK(cudaMemcpy(p, v.data(), v.size() * sizeof(float), cudaMemcpyHostToDevice));
    return p;
  }
  int* upload(const std::vector<int>& v) {
    int* p = raw<int>(v.size());
    if (ordered) CK(cudaMemcpyAsync(p, v.data(), v.size() * sizeof(int), cudaMemcpyHostToDevice, stream));
    else CK(cudaMemcpy(p, v.data(), v.size() * sizeof(int), cudaMemcpyHostToDevice));
    return p;
  }
  ~Arena() {
    for (auto& s : slabs) {
      if (pool) pool->give(s.first, s.second); else cudaFree(s.first);
    }
  }
};

}  // namespace avc
