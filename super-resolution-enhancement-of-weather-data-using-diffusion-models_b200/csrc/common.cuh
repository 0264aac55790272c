// common.cuh -- shared helpers for libwsr (error reporting, dtype access, launch checks).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include "../../include/wsr.h"

namespace wsr {

void set_error(const char* fmt, ...);

#define WSR_REQUIRE(cond, code, ...)                \
  do {                                              \
    if (!(cond)) {                                  \
      ::wsr::set_error(__VA_ARGS__);                \
      return (code);                                \
    }                                               \
  } while (0)

#define WSR_CUDA_OK(expr)                                                                       \
  do {                                                                                          \
    cudaError_t e__ = (expr);                                                                   \
    if (e__ != cudaSuccess) {                                                                   \
      ::wsr::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
      return WSR_E_CUDA;                                                                        \
    }                                                                                           \
  } while (0)

#define WSR_LAUNCH_OK() WSR_CUDA_OK(cudaGetLastError())


// ---- programmatic dependent launch ------------------------------------------------------------------------------------
// A step is ~190 dependent launches; with plain stream order every kernel starts only after its predecessor has fully
// drained AND its own launch latency + prologue (barrier init, tensor-map prefetch, TMEM allocation, GroupNorm scale table)
// has elapsed.  Kernels launched through launch_pdl() may be scheduled while the predecessor is still running: they do their
// input-independent prologue, then block in pdl_wait() until the predecessor grid has completed and its memory is visible.
// EVERY global-memory access that may depend on (or be overwritten under) earlier work must come after pdl_wait().
// Measured on B200 (bench.py, CUDA-graph replay of the step, A/B on one box): 17.39 ms with the attribute vs 17.17 ms without -- the
// graph already keeps launch gaps short and the device runs under its power cap -- so the attribute is OFF unless
// wsr_set_pdl(1) (pdl_wait() is then a no-op).
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// process-wide switch (common.cu), off by default; wsr_set_pdl() sets it (the sampling loop switches it on
// while it captures the step graph of a SMALL batch, where launch gaps are a visible share of the step: 3.39 -> 3.31 ms at 8 images)
extern int g_pdl_mode;
static inline bool pdl_enabled() { return g_pdl_mode != 0; }

template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

static inline bool valid_dtype(int dt) { return dt == WSR_F32 || dt == WSR_BF16; }
static inline int dtype_size(int dt) { return dt == WSR_BF16 ? 2 : 4; }

template <typename T> __device__ __forceinline__ float ldf(const T* p);
template <> __device__ __forceinline__ float ldf<float>(const float* p) { return *p; }
template <> __device__ __forceinline__ float ldf<__nv_bfloat16>(const __nv_bfloat16* p) { return __bfloat162float(*p); }

template <typename T> __device__ __forceinline__ void stf(T* p, float v);
template <> __device__ __forceinline__ void stf<float>(float* p, float v) { *p = v; }
template <> __device__ __forceinline__ void stf<__nv_bfloat16>(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }

// runtime-dtype scalar access (used in epilogues where the dtype is a kernel argument)
__device__ __forceinline__ float ld_dt(const void* p, int64_t i, int dt) {
  return dt == WSR_BF16 ? __bfloat162float(((const __nv_bfloat16*)p)[i]) : ((const float*)p)[i];
}
__device__ __forceinline__ void st_dt(void* p, int64_t i, int dt, float v) {
  if (dt == WSR_BF16) ((__nv_bfloat16*)p)[i] = __float2bfloat16_rn(v);
  else ((float*)p)[i] = v;
}

// 16-byte vector access to VEC consecutive channels, widened to fp32 registers
template <typename T, int VEC> struct VecLoad;
template <> struct VecLoad<float, 4> {
  typedef float4 Raw;
  static __device__ __forceinline__ Raw ldraw(const float* p) { return *(const float4*)p; }
  static __device__ __forceinline__ void widen(const Raw& q, float (&v)[4]) { v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w; }
  static __device__ __forceinline__ void ld(const float* p, float (&v)[4]) { float4 q = *(const float4*)p; v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w; }
  static __device__ __forceinline__ void st(float* p, const float (&v)[4]) { *(float4*)p = make_float4(v[0], v[1], v[2], v[3]); }
};
template <> struct VecLoad<float, 1> {
  typedef float Raw;
  static __device__ __forceinline__ Raw ldraw(const float* p) { return *p; }
  static __device__ __forceinline__ void widen(const Raw& q, float (&v)[1]) { v[0] = q; }
  static __device__ __forceinline__ void ld(const float* p, float (&v)[1]) { v[0] = *p; }
  static __device__ __forceinline__ void st(float* p, const float (&v)[1]) { *p = v[0]; }
};
template <> struct VecLoad<__nv_bfloat16, 8> {
  typedef uint4 Raw;
  static __device__ __forceinline__ Raw ldraw(const __nv_bfloat16* p) { return *(const uint4*)p; }
  static __device__ __forceinline__ void widen(const Raw& q, float (&v)[8]) {
    const __nv_bfloat162* h = (const __nv_bfloat162*)&q;
#pragma unroll
    for (int i = 0; i < 4; ++i) { float2 f = __bfloat1622float2(h[i]); v[2 * i] = f.x; v[2 * i + 1] = f.y; }
  }
  static __device__ __forceinline__ void ld(const __nv_bfloat16* p, float (&v)[8]) {
    uint4 q = *(const uint4*)p;
    const __nv_bfloat162* h = (const __nv_bfloat162*)&q;
#pragma unroll
    for (int i = 0; i < 4; ++i) { float2 f = __bfloat1622float2(h[i]); v[2 * i] = f.x; v[2 * i + 1] = f.y; }
  }
  static __device__ __forceinline__ void st(__nv_bfloat16* p, const float (&v)[8]) {
    uint4 q;
    __nv_bfloat162* h = (__nv_bfloat162*)&q;
#pragma unroll
    for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
    *(uint4*)p = q;
  }
};
template <> struct VecLoad<__nv_bfloat16, 1> {
  typedef __nv_bfloat16 Raw;
  static __device__ __forceinline__ Raw ldraw(const __nv_bfloat16* p) { return *p; }
  static __device__ __forceinline__ void widen(const Raw& q, float (&v)[1]) { v[0] = __bfloat162float(q); }
  static __device__ __forceinline__ void ld(const __nv_bfloat16* p, float (&v)[1]) { v[0] = __bfloat162float(*p); }
  static __device__ __forceinline__ void st(__nv_bfloat16* p, const float (&v)[1]) { *p = __float2bfloat16_rn(v[0]); }
};

__device__ __forceinline__ float apply_act(float v, int act) {
  switch (act) {
    case WSR_ACT_LRELU02: return v > 0.f ? v : 0.2f * v;
    case WSR_ACT_RELU: return v > 0.f ? v : 0.f;
    case WSR_ACT_SWISH: return v / (1.f + __expf(-v));
    case WSR_ACT_MISH: {
      float sp = v > 20.f ? v : log1pf(__expf(v));
      return v * tanhf(sp);
    }
    default: return v;
  }
}

// x * sigmoid(x) with ONE SFU op: sigmoid(x) = 0.5 * tanh(0.5 x) + 0.5 (tanh.approx.f32, rel. error ~2^-11: below the
// bf16 rounding of the stored result).  Used on bf16 outputs only; fp32 check mode keeps the exact form.
__device__ __forceinline__ float swish_fast(float v) {
  float h = 0.5f * v, t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
  return fmaf(h, t, h);
}

// Dispatch a templated launcher on a runtime dtype.
#define WSR_DISPATCH_DTYPE(dt, T, ...)                 \
  do {                                                 \
    if ((dt) == WSR_BF16) { using T = __nv_bfloat16; __VA_ARGS__; } \
    else { using T = float; __VA_ARGS__; }             \
  } while (0)

}  // namespace wsr
