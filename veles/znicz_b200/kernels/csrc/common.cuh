// Shared device helpers for the sm_100a kernels of znicz_b200.
// No torch headers here: .cu files compile in seconds; ext.cpp does the binding.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>

#include <string.h>
#include <stdlib.h>

namespace zn {

// ---- programmatic dependent launch -------------------------------------------------------------
// Every kernel of the step is launched with the programmatic-stream-serialization attribute
// (also inside captured CUDA graphs, where it becomes a programmatic edge): kernel N+1's CTAs are
// scheduled as soon as all CTAs of kernel N have started, run their prologue (index math, smem
// carve-up, barrier init, TMEM allocation) and block in pdl_wait() until kernel N has completed
// and flushed. The ~25 launches of a training step otherwise pay one full drain + launch latency
// each. ZNICZ_PDL=0 switches the attribute off (plain stream order).
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

inline bool pdl_enabled() {
  static int on = -1;
  if (on < 0) { const char* e = getenv("ZNICZ_PDL"); on = (e && atoi(e) == 0) ? 0 : 1; }
  return on != 0;
}

template <typename... KArgs, typename... Args>
inline cudaError_t launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem,
                            cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ---- activation codes (must match ops/nn_units.py and ops/activation.py) ----
enum Act : int {
  ACT_LINEAR = 0, ACT_TANH = 1, ACT_RELU = 2 /*softplus*/, ACT_STRICT_RELU = 3,
  ACT_SIGMOID = 4, ACT_MUL = 5, ACT_LOG = 6, ACT_TANHLOG = 7, ACT_SINCOS = 8
};

// ---- dtype load/store in fp32 math ----
template <typename T> __device__ __forceinline__ float ldf(const T* p);
template <> __device__ __forceinline__ float ldf<float>(const float* p) { return *p; }
template <> __device__ __forceinline__ float ldf<__nv_bfloat16>(const __nv_bfloat16* p) {
  return __bfloat162float(*p);
}
template <typename T> __device__ __forceinline__ void stf(T* p, float v);
template <> __device__ __forceinline__ void stf<float>(float* p, float v) { *p = v; }
template <> __device__ __forceinline__ void stf<__nv_bfloat16>(__nv_bfloat16* p, float v) {
  *p = __float2bfloat16_rn(v);
}

// 8-element vector access (16 B for bf16, 32 B for fp32)
template <typename T> struct Vec8 { float v[8]; };
template <typename T> __device__ __forceinline__ void ld8(const T* p, float (&v)[8]);
template <> __device__ __forceinline__ void ld8<float>(const float* p, float (&v)[8]) {
  float4 a = *reinterpret_cast<const float4*>(p);
  float4 b = *reinterpret_cast<const float4*>(p + 4);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
template <> __device__ __forceinline__ void ld8<__nv_bfloat16>(const __nv_bfloat16* p, float (&v)[8]) {
  uint4 raw = *reinterpret_cast<const uint4*>(p);
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&raw);
#pragma unroll
  for (int i = 0; i < 4; ++i) { float2 f = __bfloat1622float2(h[i]); v[2 * i] = f.x; v[2 * i + 1] = f.y; }
}
template <typename T> __device__ __forceinline__ void st8(T* p, const float (&v)[8]);
template <> __device__ __forceinline__ void st8<float>(float* p, const float (&v)[8]) {
  *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  *reinterpret_cast<float4*>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
}
template <> __device__ __forceinline__ void st8<__nv_bfloat16>(__nv_bfloat16* p, const float (&v)[8]) {
  uint4 raw;
  __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&raw);
#pragma unroll
  for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
  *reinterpret_cast<uint4*>(p) = raw;
}

// ---- activations (forward in terms of s; derivative in terms of x and/or y) ----
__device__ __forceinline__ float act_fwd(int act, float s, float factor = 1.f, int idx = 0) {
  switch (act) {
    case ACT_TANH: return 1.7159f * tanhf(0.6666f * s);
    case ACT_RELU: return s > 15.f ? s : log1pf(__expf(s));
    case ACT_STRICT_RELU: return fmaxf(s, 0.f);
    case ACT_SIGMOID: return 1.f / (1.f + __expf(-s));
    case ACT_MUL: return s * factor;
    case ACT_LOG: return logf(s + sqrtf(s * s + 1.f));
    case ACT_TANHLOG: {
      float a = fabsf(s);
      if (a > 3.f) return copysignf(logf(a * 305.459953195f) * 0.242528761112f, s);
      return 1.7159f * tanhf(0.6666f * s);
    }
    case ACT_SINCOS: return (idx & 1) ? sinf(s) : cosf(s);
    default: return s;
  }
}
// The five layer activations that can sit in a GEMM/conv epilogue. Small code on purpose: the
// generic act_fwd() drags sinf/cosf/logf slow paths into every unrolled epilogue element and
// made the tcgen05 kernels ~45k SASS instructions (instruction-fetch bound).
__device__ __forceinline__ float act_fwd5(int act, float s) {          // accurate (fp32 paths)
  if (act == ACT_LINEAR) return s;
  if (act == ACT_STRICT_RELU) return fmaxf(s, 0.f);
  if (act == ACT_TANH) return 1.7159f * tanhf(0.6666f * s);
  if (act == ACT_SIGMOID) return 1.f / (1.f + __expf(-s));
  return s > 15.f ? s : log1pf(__expf(s));                             // ACT_RELU = softplus
}
__device__ __forceinline__ float tanh_approx(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float act_fwd5_fast(int act, float s) {     // bf16-output epilogues
  if (act == ACT_LINEAR) return s;
  if (act == ACT_STRICT_RELU) return fmaxf(s, 0.f);
  if (act == ACT_TANH) return 1.7159f * tanh_approx(0.6666f * s);
  if (act == ACT_SIGMOID) return __fdividef(1.f, 1.f + __expf(-s));
  return s > 15.f ? s : __logf(1.f + __expf(s));
}

// derivative factor f'(.) given pre-activation x (may be unused) and output y
__device__ __forceinline__ float act_deriv(int act, float x, float y, float factor = 1.f, int idx = 0) {
  switch (act) {
    case ACT_TANH: return y * y * (-0.388484177f) + 1.14381894f;
    case ACT_RELU: return 1.f - __expf(-y);
    case ACT_STRICT_RELU: return y > 0.f ? 1.f : 0.f;
    case ACT_SIGMOID: return y * (1.f - y);
    case ACT_MUL: return factor;
    case ACT_LOG: return rsqrtf(x * x + 1.f);
    case ACT_TANHLOG: {
      float a = fabsf(x);
      if (a > 3.f) return 0.242528761112f / a;
      return y * y * (-0.388484177f) + 1.14381894f;
    }
    case ACT_SINCOS: return (idx & 1) ? cosf(x) : -sinf(x);
    default: return 1.f;
  }
}

// ---- counter-based hash (must match ops/pooling.py::hash_u32) ----
__host__ __device__ __forceinline__ uint32_t hash_u32(uint32_t seed, uint32_t counter, uint64_t idx) {
  uint64_t k = idx * 0x9E3779B1ull + (uint64_t)seed + (uint64_t)counter * 0x85EBCA77ull;
  uint32_t x = (uint32_t)(k & 0xFFFFFFFFull);
  x ^= x >> 16; x *= 0x85EBCA6Bu; x ^= x >> 13; x *= 0xC2B2AE35u; x ^= x >> 16;
  return x;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

}  // namespace zn

#define ZN_CHECK_LAUNCH() do { } while (0)
