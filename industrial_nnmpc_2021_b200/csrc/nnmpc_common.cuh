// Shared helpers for libnnmpc: error reporting, launch accounting, device buffers.
#pragma once
#include <cuda_runtime.h>
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <new>
#include "../../include/nnmpc.h"

namespace nnmpc {

extern thread_local char g_last_error[512];
extern std::atomic<long long> g_launches;
extern std::atomic<long long> g_iterations;

inline int set_error(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_last_error, sizeof(g_last_error), fmt, ap);
  va_end(ap);
  return code;
}

#define NNMPC_CUDA(call)                                                                       \
  do {                                                                                         \
    cudaError_t e__ = (call);                                                                  \
    if (e__ != cudaSuccess)                                                                    \
      return nnmpc::set_error(NNMPC_ERR_CUDA, "%s:%d: %s -> %s", __FILE__, __LINE__, #call,    \
                              cudaGetErrorString(e__));                                        \
  } while (0)

#define NNMPC_TRY(call)          \
  do {                           \
    int r__ = (call);            \
    if (r__ < 0) return r__;     \
  } while (0)

inline void count_launch(int k = 1) { g_launches.fetch_add(k, std::memory_order_relaxed); }

// Grid of the one-CTA-per-listed-row kernels: the list length lives on the device and is usually far below the slot
// count, so the grid is capped at one resident wave (148 SMs x 8 CTAs of 256 threads) and the CTAs stride over the list.
inline unsigned row_grid(long long max_rows) {
  const long long cap = 148 * 8;
  return (unsigned)(max_rows < 1 ? 1 : (max_rows < cap ? max_rows : cap));
}

// Keras relu that keeps a NaN, as the reference's np.where(x < 0, 0, x) does.  Bit-identical to x > 0 ? x : 0 for
// every other input, including -0.0 -> +0.0: the row maxima below are atomicMax on float bit patterns, where -0.0f
// (0x80000000) would outrank every positive float.
__device__ __forceinline__ double relu_keep_nan(double x) { return (x > 0.0 || x != x) ? x : 0.0; }

// running maximum of non-negative floats that ends as the positive NaN 0x7fffffff once it meets a NaN: that bit
// pattern outranks every other float in an atomicMax on the bits, so the row maximum of a NaN row stays NaN
__device__ __forceinline__ float row_max_keep_nan(float m, float h) {
  return (m != m || h != h) ? __int_as_float(0x7fffffff) : fmaxf(m, h);
}

// clip in the reference's order (np.where(u > ub, ub, u), then np.where(u < lb, lb, u)): a NaN stays NaN
__device__ __forceinline__ double clip_keep_nan(double v, double lb, double ub) {
  v = v > ub ? ub : v;
  return v < lb ? lb : v;
}

// RAII-less grow-only device buffer (handles free explicitly in destroy)
template <class T>
struct DevBuf {
  T* p = nullptr;
  size_t cap = 0;  // elements
  int ensure(size_t n) {
    if (n <= cap) return 0;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    cudaError_t e = cudaMalloc((void**)&p, n * sizeof(T));
    if (e != cudaSuccess) {
      cudaGetLastError();
      return set_error(NNMPC_ERR_NOMEM, "cudaMalloc(%zu bytes) failed: %s", n * sizeof(T), cudaGetErrorString(e));
    }
    cap = n;
    return 0;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
};

inline int upload(double** dst, const double* host, size_t n) {
  NNMPC_CUDA(cudaMalloc((void**)dst, n * sizeof(double)));
  NNMPC_CUDA(cudaMemcpy(*dst, host, n * sizeof(double), cudaMemcpyHostToDevice));
  return 0;
}

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) cudaSetDevice(dev);
    else prev = -1;
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

}  // namespace nnmpc
