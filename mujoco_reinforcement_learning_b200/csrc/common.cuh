// Shared helpers for libb200ppo (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include <utility>

#include "b200ppo.h"

#define B2_EXPORT __attribute__((visibility("default")))

namespace b200ppo {

void set_error(const char* fmt, ...);
void count_launch();

#define B2_CHECK_ARG(cond, ...)           \
  do {                                    \
    if (!(cond)) {                        \
      ::b200ppo::set_error(__VA_ARGS__);  \
      return B200PPO_EINVAL;              \
    }                                     \
  } while (0)

#define B2_CUDA(expr)                                                                              \
  do {                                                                                             \
    cudaError_t _e = (expr);                                                                       \
    if (_e != cudaSuccess) {                                                                       \
      ::b200ppo::set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      return B200PPO_ECUDA;                                                                        \
    }                                                                                              \
  } while (0)

// every kernel launch of the library is followed by this: counts it, then checks the launch
#define B2_LAUNCH_CHECK()                \
  do {                                   \
    ::b200ppo::count_launch();           \
    B2_CUDA(cudaGetLastError());         \
  } while (0)

#define B2_TRY(expr)            \
  do {                          \
    int _r = (expr);            \
    if (_r != B200PPO_OK) return _r; \
  } while (0)

// Owns one cudaMalloc'd array and its capacity in elements; frees it when destroyed.  Never give one static storage
// duration: its destructor would run after the CUDA runtime has shut down.
template <typename T>
class DevBuf {
 public:
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  DevBuf(DevBuf&& o) noexcept : p_(o.p_), cap_(o.cap_) { o.p_ = nullptr; o.cap_ = 0; }
  DevBuf& operator=(DevBuf&& o) noexcept {
    std::swap(p_, o.p_);
    std::swap(cap_, o.cap_);
    return *this;
  }
  ~DevBuf() { reset(); }

  // Frees what it holds (without synchronising), then allocates max(elems, 1) elements, zeroed on request.
  int alloc(int64_t elems, bool zero = false) {
    reset();
    if (elems <= 0) elems = 1;
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&p_), size_t(elems) * sizeof(T));
    if (e != cudaSuccess) {
      p_ = nullptr;
      set_error("cudaMalloc(%lld bytes) failed: %s", (long long)(elems * sizeof(T)), cudaGetErrorString(e));
      return e == cudaErrorMemoryAllocation ? B200PPO_ENOMEM : B200PPO_ECUDA;
    }
    cap_ = elems;
    if (zero) B2_CUDA(cudaMemset(p_, 0, size_t(elems) * sizeof(T)));
    return B200PPO_OK;
  }
  // Room for `elems` elements.  Growing waits for the device (queued work may still use the old array) and drops the
  // contents; after a failure the buffer is empty, so the next call tries again.
  int grow(int64_t elems) {
    if (elems <= cap_) return B200PPO_OK;
    B2_CUDA(cudaDeviceSynchronize());
    return alloc(elems);
  }
  void reset() {
    if (p_ != nullptr) cudaFree(p_);
    p_ = nullptr;
    cap_ = 0;
  }
  T* get() const { return p_; }
  operator T*() const { return p_; }
  int64_t cap() const { return cap_; }

 private:
  T* p_ = nullptr;
  int64_t cap_ = 0;
};

inline int num_sms() {
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
      sms = 148;
  }
  return sms;
}

// ---- programmatic dependent launch (PDL) ---------------------------------------------------------------------------------
// The minibatch loop is a chain of short kernels (7 launches of 15-50 us at the bench shape, far less at small
// minibatches), so launch latency and each kernel's set-up (barrier init, TMEM allocation, loading stationary weights)
// are a visible share of the step.  Kernels of that chain are launched with the programmatic-serialization attribute:
// a CTA of kernel n+1 may start as soon as every CTA of kernel n has passed pdl_wait_then_release(), i.e. while kernel
// n is still draining, does its set-up, and blocks in griddepcontrol.wait until kernel n has completed and flushed.
// Rules that keep this correct: (1) every kernel launched this way calls the wait before touching anything the
// previous kernel wrote, and releases its dependents only AFTER its own wait — so when a CTA of kernel n+1 runs, kernel
// n-1 and everything before it is complete; (2) before the wait a kernel may only READ data written two or more kernels
// back (the stationary weights, except in the kernel right after the optimizer) and writes nothing global.
inline bool pdl_enabled() {
  static const bool on = []() {
    const char* e = getenv("B200PPO_PDL");
    return !(e != nullptr && e[0] == '0');
  }();
  return on;
}

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

// No-ops when the kernel was launched without the attribute.
__device__ __forceinline__ void pdl_wait_then_release() {
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Streaming 128-bit accesses: data touched once, keep it out of L1.
__device__ __forceinline__ float4 ldg_stream4(const float* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ void stg_stream4(float* p, float4 v) {
  asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}


// Final combine of per-CTA partials [n_cta][width] by the last CTA: thread (part, c) sums a contiguous slice of
// CTAs with independent (pipelined) L2 loads, then the slices are added in slice order — a fixed order, so the
// result is deterministic, without the serial chain of L2 round trips a single thread per column would pay.
template <int THREADS>
__device__ __forceinline__ float combine_partials(const float* partials, unsigned n_cta, int width, int c_out, float* s_scratch) {
  // s_scratch: THREADS floats.  Returns the total of column c_out to threads with threadIdx.x == c_out (< width).
  constexpr int COLS = 64;                 // columns handled per slice row (width <= 64)
  constexpr int PARTS = THREADS / COLS;    // slices
  const int tid = threadIdx.x, c = tid % COLS, part = tid / COLS;
  float s = 0.f;
  if (c < width && part < PARTS) {
    const unsigned per = (n_cta + PARTS - 1) / PARTS;
    const unsigned k0 = part * per, k1 = min(n_cta, k0 + per);
    // 16 independent L2 loads in flight per thread: the owner block sits on the optimizer kernel's critical path
    unsigned k = k0;
    for (; k + 16 <= k1; k += 16) {
      float v[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) v[j] = __ldcg(partials + size_t(k + j) * width + c);
#pragma unroll
      for (int j = 0; j < 16; ++j) s += v[j];
    }
    for (; k < k1; ++k) s += __ldcg(partials + size_t(k) * width + c);
  }
  s_scratch[tid] = s;
  __syncthreads();
  float total = 0.f;
  if (tid < width) {
    for (int p = 0; p < PARTS; ++p) total += s_scratch[p * COLS + tid];
  }
  (void)c_out;
  return total;
}

}  // namespace b200ppo
