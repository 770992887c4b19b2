// Helpers shared by the expert recognisers (svtr.cu, crnn.cu) and, through train_util.cuh, their training paths: grouped
// Linear dispatch (CUDA-core fp32 engine or tcgen05 bf16 engine), workspace carving, the NHWC im2col, BatchNorm
// finalisation and the fp32 -> AT cast.  Everything here has internal linkage.
#pragma once
#include "common.cuh"
#include "gemm_f32.h"
#include "gemm_tc.h"

namespace {

// ------------------------------------------------------------------------------------------------
// linear<AT>: grouped Linear over experts: out[g, m, :] = epi(A[g, m, :] . W[g]^T + b[g])
// ------------------------------------------------------------------------------------------------
struct LinearArgs {
  const void* A; long lda; long a_gstride;       // AT
  const float* W32; const void* W16; long w_gstride;   // [groups, N, K]
  const float* bias; long bias_gstride;
  void* out; long ldo; long o_gstride; int out_is_f32;   // out dtype: fp32 or AT
  const float* res; const float* rowscale; int rows_per_scale; long rowscale_gstride;
  int M, N, K, groups, gelu;
  int relu;
  // tensor-core mode only: fused LayerNorm of the output rows -> ln_out (AT) [groups][M][N]
  void* ln_out; const float* ln_gamma; const float* ln_beta; float ln_eps;
};

template <typename AT>
int linear(const LinearArgs& a, cudaStream_t st);

template <>
int linear<float>(const LinearArgs& a, cudaStream_t st) {
  MrnbGemm g = mrnb_gemm_nt((const float*)a.A, a.lda, a.W32, a.K, (float*)a.out, a.ldo, a.M, a.N, a.K);
  g.batch = a.groups; g.sAb = a.a_gstride; g.sBb = a.w_gstride; g.sCb = a.o_gstride;
  g.bias_n = a.bias; g.bias_bstride = a.bias_gstride;
  g.res = a.res; g.rowscale = a.rowscale; g.rows_per_scale = a.rows_per_scale > 0 ? a.rows_per_scale : 1;
  g.rowscale_bstride = a.rowscale_gstride;
  g.act = a.gelu ? 1 : (a.relu ? 2 : 0);
  return mrnb_sgemm(g, st);
}

template <>
int linear<__nv_bfloat16>(const LinearArgs& a, cudaStream_t st) {
  MrnbTcGemm g{};
  g.A = a.A; g.lda = a.lda; g.a_gstride = a.a_gstride;
  g.W = a.W16; g.ldw = a.K; g.w_gstride = a.w_gstride;
  g.bias = a.bias; g.bias_gstride = a.bias_gstride;
  g.out = a.out; g.ldo = a.ldo; g.o_gstride = a.o_gstride; g.out_f32 = a.out_is_f32;
  g.res = a.res; g.rowscale = a.rowscale; g.rows_per_scale = a.rows_per_scale > 0 ? a.rows_per_scale : 1;
  g.rowscale_gstride = a.rowscale_gstride;
  g.M = a.M; g.N = a.N; g.K = a.K; g.groups = a.groups; g.gelu = a.gelu; g.relu = a.relu;
  g.ln_out = a.ln_out; g.ln_gstride = (long)a.M * a.N; g.ln_gamma = a.ln_gamma; g.ln_beta = a.ln_beta; g.ln_eps = a.ln_eps;
  return mrnb_tc_gemm(g, st);
}

inline size_t align_up(size_t v, size_t a = 256) { return (v + a - 1) / a * a; }

struct Workspace {
  char* base; size_t off, cap;
  template <typename T> T* take(size_t n) {
    T* p = reinterpret_cast<T*>(base + off);
    off = align_up(off + n * sizeof(T));
    return p;
  }
};

// im2col of a KH x KW convolution with zero padding `pad` and stride (sh, sw) over NHWC x[B,H,W,C]:
// col[(b,oh,ow), (kh,kw,c)] with ih = oh*sh - pad + kh, iw = ow*sw - pad + kw, zero outside the image.  Four channels
// per thread (C % 4 == 0).  Output columns ow >= the true output width (a padded frame axis) are filled by the same rule.
template <typename OT>
__global__ void im2col_nhwc_kernel(const float* __restrict__ x, OT* __restrict__ col, int H, int W, int C, int KH, int KW,
                                   int pad, int sh, int sw, int Ho, int Wo, long total4) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total4) return;
  const int c4 = C / 4;
  const int c = (int)(i % c4) * 4;
  long r = i / c4;
  const int tap = (int)(r % (KH * KW)); r /= (KH * KW);
  const int ow = (int)(r % Wo); r /= Wo;
  const int oh = (int)(r % Ho);
  const long b = r / Ho;
  const int ih = oh * sh - pad + tap / KW, iw = ow * sw - pad + tap % KW;
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  if (ih >= 0 && ih < H && iw >= 0 && iw < W) v = *reinterpret_cast<const float4*>(x + ((b * H + ih) * W + iw) * C + c);
  if constexpr (sizeof(OT) == 4) {
    *reinterpret_cast<float4*>(col + i * 4) = v;
  } else {                                        // four bf16 values = one 8-byte store
    __nv_bfloat162 h0 = __floats2bfloat162_rn(v.x, v.y), h1 = __floats2bfloat162_rn(v.z, v.w);
    *reinterpret_cast<uint2*>(col + i * 4) = make_uint2(*reinterpret_cast<uint32_t*>(&h0), *reinterpret_cast<uint32_t*>(&h1));
  }
}

// BN finalize: scale/shift per (expert, channel) from batch statistics (train) or running statistics (eval);
// in train mode also the running-stat update with momentum 0.1 and the unbiased variance (nn.BatchNorm2d).
// use_batch_stats / update_running are per-expert bit masks (bit e = expert e).  mean_rstd, when not null, receives
// (mean, 1/sqrt(var + eps)) per (expert, channel) for the BatchNorm backward.
__global__ void bn_finalize_kernel(const double* __restrict__ stats, const float* __restrict__ gamma,
                                   const float* __restrict__ beta, float* __restrict__ run_mean,
                                   float* __restrict__ run_var, float* __restrict__ scale_shift /*[I,C,2]*/,
                                   float* __restrict__ mean_rstd /*[I,C,2] or null*/, int I, int C, double count,
                                   int use_batch_stats, int update_running, float eps) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= I * C) return;
  float mean, var;
  const int e = idx / C;
  if ((use_batch_stats >> e) & 1) {
    const double m = stats[idx * 2] / count;
    double v = stats[idx * 2 + 1] / count - m * m;
    if (v < 0) v = 0;
    mean = (float)m; var = (float)v;
    if ((update_running >> e) & 1) {
      run_mean[idx] = 0.9f * run_mean[idx] + 0.1f * mean;
      run_var[idx] = 0.9f * run_var[idx] + 0.1f * (float)(v * count / (count - 1.0));
    }
  } else {
    mean = run_mean[idx]; var = run_var[idx];
  }
  const float rstd = rsqrtf(var + eps);
  const float sc = gamma[idx] * rstd;
  scale_shift[idx * 2] = sc;
  scale_shift[idx * 2 + 1] = beta[idx] - mean * sc;
  if (mean_rstd) { mean_rstd[idx * 2] = mean; mean_rstd[idx * 2 + 1] = rstd; }
}

template <typename AT>
__global__ void cast_kernel(const float* __restrict__ x, AT* __restrict__ y, long n) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) y[i] = from_f32<AT>(x[i]);
}


}  // namespace
