// Shared helpers for the honk2_b200 native library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cstdint>
#include <cstdio>
#include <cstdarg>
#include <mutex>
#include <string>
#include <vector>
#include "../../include/honk2_b200.h"

namespace kws {

void set_error(const char* fmt, ...);
extern thread_local int64_t g_launches;  // kernels launched on this thread since last reset

#define KWS_CUDA(expr)                                                                      \
  do {                                                                                      \
    cudaError_t _e = (expr);                                                                \
    if (_e != cudaSuccess) {                                                                \
      ::kws::set_error("%s failed at %s:%d: %s", #expr, __FILE__, __LINE__,                 \
                       cudaGetErrorString(_e));                                             \
      return KWS_ERR_CUDA;                                                                  \
    }                                                                                       \
  } while (0)

#define KWS_CHECK_LAUNCH()                                                                  \
  do {                                                                                      \
    ++::kws::g_launches;                                                                    \
    KWS_CUDA(cudaGetLastError());                                                           \
  } while (0)

#define KWS_REQUIRE(cond, ...)                                                              \
  do {                                                                                      \
    if (!(cond)) {                                                                          \
      ::kws::set_error(__VA_ARGS__);                                                        \
      return KWS_ERR_INVALID;                                                               \
    }                                                                                       \
  } while (0)

#define KWS_TRY(expr)                                                                       \
  do {                                                                                      \
    int _s = (expr);                                                                        \
    if (_s != KWS_OK) return _s;                                                            \
  } while (0)

template <typename T>
__host__ __device__ constexpr T ceil_div(T a, T b) { return (a + b - 1) / b; }
template <typename T>
__host__ __device__ constexpr T round_up(T a, T b) { return ceil_div(a, b) * b; }

constexpr int kNumSMs = 148;  // B200

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

// A kernel's dynamic shared memory limit belongs to the kernel, not to the object that launches it.  Objects that plan
// their own shared memory when they are created (front-ends, CNN plans, live CNN states) only ever raise it: lowering it
// for a smaller object would make every larger one that already exists fail its launches with "invalid argument".
template <typename K>
cudaError_t raise_dynamic_smem(K* kernel, size_t bytes) {
  static std::mutex mu;
  std::lock_guard<std::mutex> lock(mu);
  cudaFuncAttributes a;
  cudaError_t e = cudaFuncGetAttributes(&a, reinterpret_cast<const void*>(kernel));
  if (e != cudaSuccess || (size_t)a.maxDynamicSharedSizeBytes >= bytes) return e;
  return cudaFuncSetAttribute(reinterpret_cast<const void*>(kernel), cudaFuncAttributeMaxDynamicSharedMemorySize,
                              (int)bytes);
}

// ResNet geometry shared by the fp32 and tensor-core paths: the dilation of C -> C layer i (1-based, resnet.py:21-23),
// the AvgPool window after conv_0 (pool 0, 0 = absent, resnet.py:40-44), and the map it leaves of a T x F input.
inline int resnet_dilation(const kws_resnet_config& c, int i) { return c.use_dilation ? 1 << ((i - 1) / 3) : 1; }
struct PoolWindow { int h, w; };
inline PoolWindow resnet_pool(const kws_resnet_config& c) { return {c.pool_h > 0 ? c.pool_h : 1, c.pool_w > 0 ? c.pool_w : 1}; }
inline void resnet_map(const kws_resnet_config& c, int T, int F, int* H, int* W) {
  const PoolWindow pool = resnet_pool(c);
  *H = T / pool.h;
  *W = F / pool.w;
}

// bump allocator over a caller-provided workspace
struct Arena {
  char* base;
  size_t cap, off;
  Arena(void* p, size_t n) : base(static_cast<char*>(p)), cap(n), off(0) {}
  template <typename T>
  T* take(size_t count) {
    size_t bytes = round_up<size_t>(count * sizeof(T), 256);
    T* p = reinterpret_cast<T*>(base + off);
    off += bytes;
    return p;
  }
  bool ok() const { return off <= cap; }
};


// Optional per-launch timing (bench roofline): an event is recorded before every layer launch;
// launch i lasts from event i to event i+1.  Categories: 0 = C->C convolution, 1 = everything else.
struct LaunchProfiler {
  bool enabled = false;
  std::vector<cudaEvent_t> pool;
  std::vector<int> cats;
  size_t used = 0;
  double ms[2] = {0, 0};
  int64_t n[2] = {0, 0};
  void tick(int cat, cudaStream_t st) {
    if (!enabled) return;
    if (used == pool.size()) {
      cudaEvent_t e;
      if (cudaEventCreate(&e) != cudaSuccess) { enabled = false; return; }
      pool.push_back(e);
    }
    cudaEventRecord(pool[used++], st);
    cats.push_back(cat);
  }
  void finish(cudaStream_t st) {
    if (!enabled || used == 0) return;
    tick(-1, st);
    cudaEventSynchronize(pool[used - 1]);
    for (size_t i = 0; i + 1 < used; ++i) {
      float t = 0.f;
      cudaEventElapsedTime(&t, pool[i], pool[i + 1]);
      ms[cats[i]] += t;
      n[cats[i]] += 1;
    }
    used = 0;
    cats.clear();
  }
  void reset() { ms[0] = ms[1] = 0; n[0] = n[1] = 0; }
  ~LaunchProfiler() { for (auto e : pool) cudaEventDestroy(e); }
};

}  // namespace kws
