// tnb200 — shared helpers for the CUDA translation unit (sm_100a only).
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <mutex>
#include <cmath>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/tnb200.h"

namespace tnb {

inline std::string& last_error_ref() {
  static thread_local std::string s;
  return s;
}
inline int fail(int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  last_error_ref() = buf;
  return code;
}
inline std::atomic<uint64_t>& launch_counter() {
  static std::atomic<uint64_t> c{0};
  return c;
}
#define TNB_COUNT_LAUNCH() (::tnb::launch_counter().fetch_add(1, std::memory_order_relaxed))

#define TNB_CUDA(expr)                                                                              \
  do {                                                                                              \
    cudaError_t e__ = (expr);                                                                       \
    if (e__ != cudaSuccess)                                                                         \
      return ::tnb::fail(TNB_ERR_CUDA, "%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(e__)); \
  } while (0)
#define TNB_LAUNCH_CHECK()                                                                          \
  do {                                                                                              \
    TNB_COUNT_LAUNCH();                                                                             \
    cudaError_t e__ = cudaGetLastError();                                                           \
    if (e__ != cudaSuccess)                                                                         \
      return ::tnb::fail(TNB_ERR_CUDA, "%s:%d: kernel launch -> %s", __FILE__, __LINE__, cudaGetErrorString(e__)); \
  } while (0)
#define TNB_TRY(expr)            \
  do {                           \
    int rc__ = (expr);           \
    if (rc__ != TNB_OK) return rc__; \
  } while (0)

template <typename T>
inline T ceil_div(T a, T b) {
  return (a + b - 1) / b;
}
inline size_t align_up(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }

// Bump allocator over a caller-provided workspace.
struct Arena {
  char* base;
  size_t cap;
  size_t off = 0;
  bool ok = true;
  Arena(void* p, size_t n) : base(static_cast<char*>(p)), cap(n) {}
  template <typename T>
  T* take(size_t count) {
    size_t bytes = align_up(count * sizeof(T));
    if (off + bytes > cap) {
      ok = false;
      off += bytes;
      return nullptr;
    }
    T* p = reinterpret_cast<T*>(base + off);
    off += bytes;
    return p;
  }
};
// Sizing twin of Arena: same calls, only counts.
struct ArenaSizer {
  size_t off = 0;
  bool ok = true;
  template <typename T>
  T* take(size_t count) {
    off += align_up(count * sizeof(T));
    return nullptr;
  }
};

struct DeviceInfo {
  int sm_count = 0;
  int cc_major = 0, cc_minor = 0;
  bool valid = false;
};
inline const DeviceInfo& device_info() {
  static thread_local DeviceInfo info;
  static thread_local int cached_dev = -1;
  int dev = -1;
  if (cudaGetDevice(&dev) != cudaSuccess) {
    info.valid = false;
    return info;
  }
  if (dev != cached_dev) {
    cudaDeviceProp p;
    if (cudaGetDeviceProperties(&p, dev) == cudaSuccess) {
      info.sm_count = p.multiProcessorCount;
      info.cc_major = p.major;
      info.cc_minor = p.minor;
      info.valid = true;
      cached_dev = dev;
    } else {
      info.valid = false;
    }
  }
  return info;
}

// Per-device caches: cudaFuncSetAttribute, events and occupancy answers belong to ONE device, so everything that
// remembers "already done" is indexed by the current device ordinal (a process may drive several GPUs, and several
// host threads may share one).
constexpr int TNB_MAX_DEVICES = 64;
inline int current_device_index() {
  int d = 0;
  if (cudaGetDevice(&d) != cudaSuccess || d < 0) d = 0;
  return d % TNB_MAX_DEVICES;
}
struct PerDeviceFlag {
  std::atomic<int> v[TNB_MAX_DEVICES];  // zero-initialised as a static
};
// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) once per (call site, device); racing threads at worst set it twice.
template <typename K>
inline cudaError_t ensure_dyn_smem(PerDeviceFlag& f, K kernel, int bytes) {
  const int d = current_device_index();
  if (f.v[d].load(std::memory_order_acquire)) return cudaSuccess;
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess) f.v[d].store(1, std::memory_order_release);
  return e;
}

// SMs left free by the persistent / one-CTA-per-SM kernels (tensor-core Gram, projection).  With several
// decompositions in flight on different streams the latency-bound one-CTA kernels of one tensor (Jacobi, Cholesky,
// rank rule) then run beside the bandwidth-bound kernels of another instead of queueing behind them.
inline std::atomic<int>& reserved_sms_ref() {
  static std::atomic<int> r{0};
  return r;
}
inline int usable_sms() {
  const int sms = device_info().valid ? device_info().sm_count : 148;
  int r = reserved_sms_ref().load(std::memory_order_relaxed);
  if (r < 0) r = 0;
  if (r > sms - 8) r = sms - 8;
  return sms - r;
}

// TNB_FLAG_CONCURRENT: the bandwidth-bound whole-GPU kernels (tensor-core Gram, projection) of the decompositions in
// flight are chained across their streams, one at a time, each sized to usable_sms(): the reserved SMs then stay free
// for the latency-bound eigen chains of the OTHER decompositions (one-CTA Jacobi / Cholesky kernels, small
// products), which would otherwise queue behind — or steal an SM from and double the time of — a one-wave kernel.
class BigKernelGate {
 public:
  BigKernelGate(cudaStream_t st, bool enabled) : st_(st), on_(enabled), dev_(enabled ? current_device_index() : 0) {
    if (!on_) return;
    mu().lock();
    cudaEvent_t& e = ev();
    if (!e && cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) {
      e = nullptr;
      cudaGetLastError();
      return;  // no chaining possible: the kernels still run, only unordered against the other streams
    }
    if (cudaStreamWaitEvent(st_, e, 0) != cudaSuccess) cudaGetLastError();
  }
  ~BigKernelGate() {
    if (!on_) return;
    if (ev() && cudaEventRecord(ev(), st_) != cudaSuccess) cudaGetLastError();
    mu().unlock();
  }
  BigKernelGate(const BigKernelGate&) = delete;
  BigKernelGate& operator=(const BigKernelGate&) = delete;

 private:
  // one gate (mutex + event) per device: big kernels of different GPUs never wait on each other
  std::mutex& mu() { static std::mutex m[TNB_MAX_DEVICES]; return m[dev_]; }
  cudaEvent_t& ev() { static cudaEvent_t e[TNB_MAX_DEVICES] = {}; return e[dev_]; }
  cudaStream_t st_;
  bool on_;
  int dev_;
};

// Device-side early exit of kernels that were enqueued speculatively (sync-free solver chains, chfsi_dev.cuh):
// words[0] = done, words[1] = error, words[2] = stage at which `done` was raised.  A kernel of stage s does nothing
// when an error was raised or when the chain converged at an earlier stage.
__device__ __forceinline__ bool tnb_skip(const int* words, int stage) {
  if (!words) return false;
  const int done = __ldcg(words), err = __ldcg(words + 1), at = __ldcg(words + 2);
  return err != 0 || (done != 0 && stage > at);
}

// Pinned host scratch for reading small results back (ranks, Ritz values).
inline void* pinned_scratch(size_t bytes) {
  static thread_local void* p = nullptr;
  static thread_local size_t cap = 0;
  if (bytes > cap) {
    if (p) cudaFreeHost(p);
    size_t n = bytes < 65536 ? 65536 : bytes;
    if (cudaHostAlloc(&p, n, cudaHostAllocDefault) != cudaSuccess) {
      p = nullptr;
      cap = 0;
      return nullptr;
    }
    cap = n;
  }
  return p;
}

}  // namespace tnb
