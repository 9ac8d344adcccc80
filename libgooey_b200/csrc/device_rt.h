// device_rt.h — small CUDA runtime helpers shared by the host-side classes:
// error latch, device buffers, once-per-device kernel attributes.
#pragma once
#include <cstdio>
#include <cstdlib>
#include <cuda_runtime.h>
#include <cstdint>
#include <cstring>
#include <mutex>
#include <set>
#include <string>
#include <tuple>
#include <vector>
#include <stdexcept>

namespace gh {

std::string& last_error();
inline void set_error(const std::string& s) { last_error() = s; }

struct CudaError : std::runtime_error { using std::runtime_error::runtime_error; };

#define GH_CUDA(call)                                                                            \
  do {                                                                                           \
    cudaError_t _e = (call);                                                                     \
    if (_e != cudaSuccess) {                                                                     \
      char _b[512];                                                                              \
      snprintf(_b, sizeof _b, "CUDA error %s at %s:%d: %s", cudaGetErrorName(_e), __FILE__, __LINE__, cudaGetErrorString(_e)); \
      throw gh::CudaError(_b);                                                                   \
    }                                                                                            \
  } while (0)

template <class T> struct DevBuf {
  T* p = nullptr;
  size_t n = 0;
  DevBuf() {}
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { if (p) cudaFree(p); }
  // Growth frees and re-allocates, and cudaFree waits for the whole device: a per-piece table that outgrows its buffer by a few
  // entries in the middle of a render drains the pipeline (measured: ~0.5 s at the bar boundary of an 8192-engine bounce).
  // Small buffers therefore grow with 50 % headroom; large ones (voice / output blocks) are sized exactly.
  void alloc(size_t count) {
    if (count <= n && p) return;
    static const bool trace = getenv("GOOEY_B200_TRACE") != nullptr;
    if (trace && p) fprintf(stderr, "[gooey trace] device buffer regrown: %zu -> %zu bytes (cudaFree drains the device)\n", n * sizeof(T), count * sizeof(T));
    if (p) { cudaFree(p); p = nullptr; }
    if (count * sizeof(T) <= ((size_t)64 << 20)) count += count / 2 + 64;
    n = count;
    if (count) GH_CUDA(cudaMalloc(&p, count * sizeof(T)));
  }
  void upload(const T* src, size_t count, cudaStream_t s) {
    alloc(count);
    if (count) GH_CUDA(cudaMemcpyAsync(p, src, count * sizeof(T), cudaMemcpyHostToDevice, s));
  }
  void zero(cudaStream_t s) { if (p && n) GH_CUDA(cudaMemsetAsync(p, 0, n * sizeof(T), s)); }
};

// cudaFuncSetAttribute(kernel, attr, value) on the current device, once per (device, kernel, attribute).  Thread safe: the
// groups of a batch that spans several devices are rendered by one host thread each.
inline void func_attr_once(const void* kernel, cudaFuncAttribute attr, int value) {
  static std::mutex mu;
  static std::set<std::tuple<int, const void*, int>> done;
  int dev = 0;
  GH_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lk(mu);
  if (done.insert({dev, kernel, (int)attr}).second) GH_CUDA(cudaFuncSetAttribute(kernel, attr, value));
}

inline int pad32(int n) { return (n + 31) & ~31; }

}  // namespace gh
