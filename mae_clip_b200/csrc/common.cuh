// Shared host/device helpers for the mae_clip_b200 kernels (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <nvtx3/nvToolsExt.h>
#include <stdint.h>
#include <stdio.h>
#include <atomic>
#include <string>

#include "../../include/mae_clip_b200.h"

namespace mc {

// ---- error plumbing (thread-local message, integer status across the ABI) ----
void set_error(const char* fmt, ...);
int arch_check();  // MC_OK when the current device is compute capability 10.x

#define MC_REQUIRE(cond, code, ...)      \
  do {                                   \
    if (!(cond)) {                       \
      ::mc::set_error(__VA_ARGS__);      \
      return (code);                     \
    }                                    \
  } while (0)

#define MC_CUDA(call)                                                              \
  do {                                                                             \
    cudaError_t e_ = (call);                                                       \
    if (e_ != cudaSuccess) {                                                       \
      ::mc::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_),      \
                      __FILE__, __LINE__);                                         \
      return MC_ERR_CUDA;                                                          \
    }                                                                              \
  } while (0)

// every kernel launch of the library goes through this: error check + launch counter
// (mc_kernel_launch_count(): bench.py reports how many of OUR kernels ran in the timed region)
void count_launch();
#define MC_LAUNCH_CHECK()          \
  do {                             \
    ::mc::count_launch();          \
    MC_CUDA(cudaGetLastError());   \
  } while (0)

// Every compute entry point of the C ABI opens with this: the sm_100 check, and an NVTX range named after the entry
// point for the duration of the call (tracing row of SURVEY section 5: `nsys` shows the phases of a step by name,
// `ncu --nvtx --nvtx-include "mc_clip_bwd/"` profiles the kernels of one phase; header-only NVTX v3, a no-op load of a
// function pointer when no tool is attached).
struct NvtxScope {
  explicit NvtxScope(const char* name) { nvtxRangePushA(name); }
  ~NvtxScope() { nvtxRangePop(); }
  NvtxScope(const NvtxScope&) = delete;
  NvtxScope& operator=(const NvtxScope&) = delete;
};
#define MC_ARCH_GUARD()                        \
  ::mc::NvtxScope mc_nvtx_scope_(__func__);    \
  do {                                         \
    int a_ = ::mc::arch_check();               \
    if (a_ != MC_OK) return a_;                \
  } while (0)

inline bool aligned(const void* p, size_t a) { return (reinterpret_cast<uintptr_t>(p) % a) == 0; }
inline size_t round_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
inline int num_sms() {
  static std::atomic<int> cached[64];  // per device; 0 = not queried yet
  int dev = 0;
  cudaGetDevice(&dev);
  std::atomic<int>& slot = cached[dev & 63];
  int n = slot.load(std::memory_order_relaxed);
  if (n == 0) {
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
    slot.store(n, std::memory_order_relaxed);
  }
  return n;
}

// Opt a kernel in to more than 48 KB of dynamic shared memory, once per device (the attribute is
// per context).  `done` is a per-kernel bit mask of devices already configured; a racing second
// call just sets the same attribute again.
template <typename F>
inline cudaError_t ensure_dynamic_smem(F* kernel, int bytes, std::atomic<unsigned long long>& done) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  const unsigned long long bit = 1ull << (dev & 63);
  if (done.load(std::memory_order_acquire) & bit) return cudaSuccess;
  e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess) done.fetch_or(bit, std::memory_order_release);
  return e;
}

// ---- device helpers ----
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;

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
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// order-preserving unsigned integer of a float (larger float -> larger integer), so that atomicMax on it is a float
// max.  No number (only one NaN pattern) maps to 0, which therefore serves as "never set"; ord_to_float(0) = +inf.
__device__ __forceinline__ unsigned int float_to_ord(float f) {
  const unsigned int u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord_to_float(unsigned int k) {
  if (k == 0u) return INFINITY;
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k);
}

// online log-sum-exp accumulator (natural-log domain)
struct Lse {
  float m, s;
  __device__ __forceinline__ void init() { m = -INFINITY; s = 0.f; }
  __device__ __forceinline__ void add(float v) {
    if (v > m) {
      s = s * __expf(m - v) + 1.f;  // exp(-inf)=0 covers the first element
      m = v;
    } else {
      s += __expf(v - m);
    }
  }
  __device__ __forceinline__ void merge(float m2, float s2) {
    float mn = fmaxf(m, m2);
    if (mn == -INFINITY) return;
    s = s * __expf(m - mn) + s2 * __expf(m2 - mn);
    m = mn;
  }
  __device__ __forceinline__ float value() const { return m + __logf(s); }
};

__device__ __forceinline__ void warp_merge_lse(Lse& a) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    float m2 = __shfl_xor_sync(0xffffffffu, a.m, o);
    float s2 = __shfl_xor_sync(0xffffffffu, a.s, o);
    a.merge(m2, s2);
  }
}

// streaming 16-byte loads/stores that do not pollute L1
__device__ __forceinline__ float4 ld_stream(const float4* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ void st_stream(float4* p, float4 v) {
  asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y),
               "f"(v.z), "f"(v.w));
}
__device__ __forceinline__ uint4 ld_stream(const uint4* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ void st_stream(uint4* p, uint4 v) {
  asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y),
               "r"(v.z), "r"(v.w));
}

// ---- generic strided fp32 GEMM (SIMT FMA tiles; bring-up / cross-check engine) ----
// C[i,j] = alpha * sum_k A(i,k) B(k,j) (+ bias[j]) (+ C[i,j] when accumulate); optional second
// output gelu_out[i,j] = gelu(C[i,j]).  A(i,k) = A[i*sai + k*sak], B(k,j) = B[k*sbk + j*sbj].
struct SgemmArgs {
  const float* A;
  int64_t sai, sak;
  const float* B;
  int64_t sbk, sbj;
  float* C;
  int64_t ldc;
  int M, N, K;
  float alpha;
  const float* bias;   // length N or null
  float* gelu_out;     // same layout as C or null
  int accumulate;      // 1: C += result
};
int sgemm(const SgemmArgs& a, cudaStream_t stream);

__device__ __forceinline__ float gelu_erf(float x) {
  return 0.5f * x * (1.f + erff(x * 0.70710678118654752440f));
}
__device__ __forceinline__ float gelu_erf_grad(float x) {
  const float kInvSqrt2Pi = 0.3989422804014327f;
  float cdf = 0.5f * (1.f + erff(x * 0.70710678118654752440f));
  return cdf + x * kInvSqrt2Pi * __expf(-0.5f * x * x);
}

}  // namespace mc
