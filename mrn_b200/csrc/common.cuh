// Shared device/host helpers for the mrn_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>
#include <math.h>

#define MRNB_OK 0
#define MRNB_ERR_ARG (-1)
#define MRNB_ERR_WORKSPACE (-2)
#define MRNB_ERR_LAUNCH (-3)
#define MRNB_ERR_UNSUPPORTED (-4)

#define MRNB_MAX_EXPERTS 8

void mrnb_set_error(const char* fmt, ...);
extern "C" void mrnb_count_launch(int n);   // launch counter (bench.py's gpu_launches)

#define MRNB_CHECK_ARG(cond, ...)                        \
  do {                                                   \
    if (!(cond)) {                                       \
      mrnb_set_error(__VA_ARGS__);                       \
      return MRNB_ERR_ARG;                               \
    }                                                    \
  } while (0)

#define MRNB_CHECK_LAUNCH(name)                                               \
  do {                                                                        \
    cudaError_t e__ = cudaGetLastError();                                     \
    mrnb_count_launch(1);                                                     \
    if (e__ != cudaSuccess) {                                                 \
      mrnb_set_error("%s: launch failed: %s", name, cudaGetErrorString(e__)); \
      return MRNB_ERR_LAUNCH;                                                 \
    }                                                                         \
  } while (0)

#define MRNB_TRY(expr)            \
  do {                            \
    int rc__ = (expr);            \
    if (rc__ != MRNB_OK) return rc__; \
  } while (0)

// Optional per-kernel-family timing with CUDA events on the launching stream (bench.py roofline); off by default.
enum { MRNB_PROF_TCGEMM = 0, MRNB_PROF_SGEMM, MRNB_PROF_ATTN, MRNB_PROF_LN, MRNB_PROF_CONV, MRNB_PROF_COMBINE,
       MRNB_PROF_CTC, MRNB_PROF_ROUTER_EW, MRNB_PROF_OPTIM, MRNB_PROF_MISC, MRNB_PROF_MLP, MRNB_PROF_TCGEMM2,
       MRNB_PROF_MIXER, MRNB_PROF_COUNT };
void mrnb_prof_begin(int family, cudaStream_t st, double flops, double bytes);
void mrnb_prof_end(int family, cudaStream_t st);
struct MrnbProfScope {
  int family; cudaStream_t st;
  MrnbProfScope(int f, cudaStream_t s, double flops = 0.0, double bytes = 0.0) : family(f), st(s) { mrnb_prof_begin(f, s, flops, bytes); }
  ~MrnbProfScope() { mrnb_prof_end(family, st); }
};

static inline int cdiv(long a, long b) { return (int)((a + b - 1) / b); }

// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float gelu_erf(float x) {
  // nn.GELU() exact form: 0.5 x (1 + erf(x / sqrt(2)))
  return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f));
}
// erf-form GELU for values that are rounded to bf16 afterwards (tensor-core mode): x * Phi(x) with
// Phi(x) = 0.5 (1 + tanh(q(x))), q an odd minimax polynomial fitted to atanh(erf(x / sqrt 2)) on [0, 7]
// (max |error| of x*Phi(x) 2.5e-5, i.e. 20x tighter than the usual tanh-GELU and far below bf16 rounding),
// evaluated with the hardware tanh (MUFU.TANH): 9 instructions instead of erff's ~35.  fp32 mode keeps erff.
__device__ __forceinline__ float gelu_fast(float x) {
  const float x2 = fminf(x * x, 49.0f);            // beyond |x| = 7 the polynomial is frozen: tanh saturates with the right sign
  float p = fmaf(x2, -3.51516867e-4f, 3.70056465e-2f);
  p = fmaf(x2, p, 0.797507884f);
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(x * p));
  const float h = 0.5f * x;
  return fmaf(h, t, h);
}
// Same minimax form on two values at once in f16x2 (HFMA2 + MUFU.TANH.F16x2): ~4 instructions per element.
// Used where the result feeds a tensor-core operand directly (fused MLP: P is an f16 A-operand, 11-bit mantissa).
__device__ __forceinline__ __half2 gelu_fast_h2(__half2 x) {
  const __half2 x2 = __hmin2(__hmul2(x, x), __float2half2_rn(49.0f));
  __half2 p = __hfma2(x2, __float2half2_rn(-3.51516867e-4f), __float2half2_rn(3.70056465e-2f));
  p = __hfma2(x2, p, __float2half2_rn(0.797507884f));
  const __half2 q = __hmul2(x, p);
  uint32_t qi = *reinterpret_cast<const uint32_t*>(&q), ti;
  asm("tanh.approx.f16x2 %0, %1;" : "=r"(ti) : "r"(qi));
  const __half2 t = *reinterpret_cast<const __half2*>(&ti);
  const __half2 h = __hmul2(x, __float2half2_rn(0.5f));
  return __hfma2(h, t, h);
}
// d/dx [x Phi(x)] = Phi(x) + x phi(x) with the same minimax Phi as gelu_fast and phi through ex2.approx: for gradients
// that are rounded to bf16 GEMM operands (tensor-core mode); |error| < 1e-4.
__device__ __forceinline__ float gelu_fast_grad(float x) {
  const float xx = x * x;
  const float x2 = fminf(xx, 49.0f);
  float p = fmaf(x2, -3.51516867e-4f, 3.70056465e-2f);
  p = fmaf(x2, p, 0.797507884f);
  float t, e;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(x * p));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(xx * -0.72134752044448170368f));     // exp(-x^2 / 2)
  return fmaf(0.5f, t, 0.5f) + x * 0.39894228040143267794f * e;
}
__device__ __forceinline__ float gelu_erf_grad(float x) {
  const float cdf = 0.5f * (1.0f + erff(x * 0.70710678118654752440f));
  const float pdf = 0.39894228040143267794f * expf(-0.5f * x * x);
  return cdf + x * pdf;
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
// Sum 16 per-lane values across the warp with recursive halving: 16 shuffles instead of 16 x 5.  Returns, in every
// lane, the warp total of value index (lane >> 1) & 15.
__device__ __forceinline__ float warp_reduce16(float (&v)[16], int lane) {
  const bool b4 = lane & 16, b3 = lane & 8, b2 = lane & 4, b1 = lane & 2;
  float w8[8], w4[4], w2[2];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const float send = b4 ? v[i] : v[i + 8], keep = b4 ? v[i + 8] : v[i];
    w8[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float send = b3 ? w8[i] : w8[i + 4], keep = b3 ? w8[i + 4] : w8[i];
    w4[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
  }
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const float send = b2 ? w4[i] : w4[i + 2], keep = b2 ? w4[i + 2] : w4[i];
    w2[i] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
  }
  const float send = b1 ? w2[0] : w2[1], keep = b1 ? w2[1] : w2[0];
  float r = keep + __shfl_xor_sync(0xffffffffu, send, 2);
  r += __shfl_xor_sync(0xffffffffu, r, 1);
  return r;
}

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// log(exp(a)+exp(b)) with -inf handling
__device__ __forceinline__ float log_add(float a, float b) {
  const float m = fmaxf(a, b);            // fmaxf drops a NaN operand ...
  if (m == -INFINITY) return a + b;       // ... so (-inf, -inf) -> -inf but (NaN, -inf) -> NaN: a NaN never turns into "impossible"
  return m + log1pf(expf(-fabsf(a - b)));
}
