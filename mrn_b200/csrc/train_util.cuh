// Building blocks shared by the expert-training translation units (svtr_train.cu, crnn_train.cu): column sums (bias
// gradients, BatchNorm statistics), the forward / backward GEMM dispatch (CUDA-core fp32 engine or tcgen05 bf16 engines),
// small casts, the convolution lowering (bf16 im2col, col2im, conv0 weight padding) and the BatchNorm-backward apply
// pass.  Everything has internal linkage.
#pragma once
#include "common.cuh"
#include "gemm_f32.h"
#include "gemm_tc.h"
#include "gemm_tc2.h"
#include "expert_util.cuh"

namespace {

// ------------------------------------------------------------------------------------------------
// Column sums over rows (bias gradients; BatchNorm statistics with SQ).  block (32, 8), grid (cdiv(C,32), chunks).
// out must be zeroed; partial sums are combined with atomics.
// ------------------------------------------------------------------------------------------------
template <typename T, bool SQ>
__global__ void __launch_bounds__(256)
colsum_kernel(const T* __restrict__ x, long ld, long rows, int C, float* __restrict__ out, double* __restrict__ out2) {
  __shared__ double sh[8][32][SQ ? 2 : 1];
  const int c = blockIdx.x * 32 + threadIdx.x, ty = threadIdx.y;
  const long per = (rows + gridDim.y - 1) / gridDim.y;
  const long r0 = (long)blockIdx.y * per, r1 = (r0 + per < rows) ? r0 + per : rows;
  double s1 = 0.0, s2 = 0.0;
  float f1 = 0.f;
  if (c < C) {
    for (long r = r0 + ty; r < r1; r += 8) {
      const float v = to_f32<T>(x[r * ld + c]);
      if (SQ) { s1 += v; s2 += (double)v * v; } else f1 += v;
    }
  }
  if (!SQ) s1 = f1;
  sh[ty][threadIdx.x][0] = s1;
  if (SQ) sh[ty][threadIdx.x][SQ ? 1 : 0] = s2;
  __syncthreads();
  if (ty == 0 && c < C) {
    double a = 0.0, b = 0.0;
#pragma unroll
    for (int k = 0; k < 8; ++k) { a += sh[k][threadIdx.x][0]; if (SQ) b += sh[k][threadIdx.x][SQ ? 1 : 0]; }
    if (SQ) { atomicAdd(out2 + c * 2, a); atomicAdd(out2 + c * 2 + 1, b); }
    else atomicAdd(out + c, (float)a);
  }
}

// Vector variant for C % 64 == 0 with aligned rows: a thread owns four adjacent columns (one 16- or 8-byte load per row),
// a block owns 64 columns x 16 rows in flight.  grid (C / 64, chunks), block 256.
template <typename T>
__global__ void __launch_bounds__(256)
colsum_vec4_kernel(const T* __restrict__ x, long ld, long rows, float* __restrict__ out) {
  __shared__ float sh[16][64];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int c = blockIdx.x * 64 + tx * 4;
  const long per = (rows + gridDim.y - 1) / gridDim.y;
  const long r0 = (long)blockIdx.y * per, r1 = (r0 + per < rows) ? r0 + per : rows;
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  for (long r = r0 + ty; r < r1; r += 16) {
    if constexpr (sizeof(T) == 4) {
      const float4 v = *reinterpret_cast<const float4*>(x + r * ld + c);
      a0 += v.x; a1 += v.y; a2 += v.z; a3 += v.w;
    } else {
      const uint2 v = *reinterpret_cast<const uint2*>(x + r * ld + c);
      const __nv_bfloat162 p = *reinterpret_cast<const __nv_bfloat162*>(&v.x), q = *reinterpret_cast<const __nv_bfloat162*>(&v.y);
      a0 += __bfloat162float(p.x); a1 += __bfloat162float(p.y); a2 += __bfloat162float(q.x); a3 += __bfloat162float(q.y);
    }
  }
  sh[ty][tx * 4] = a0; sh[ty][tx * 4 + 1] = a1; sh[ty][tx * 4 + 2] = a2; sh[ty][tx * 4 + 3] = a3;
  __syncthreads();
  if (threadIdx.x < 64) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 16; ++k) t += sh[k][threadIdx.x];
    atomicAdd(out + blockIdx.x * 64 + threadIdx.x, t);
  }
}

template <typename T>
int launch_colsum(const T* x, long ld, long rows, int C, float* out, cudaStream_t st) {
  int chunks = (int)(rows / 256); if (chunks < 1) chunks = 1; if (chunks > 64) chunks = 64;
  if (C % 64 == 0 && ld % 4 == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0) {
    int ch = (int)(rows / 512); if (ch < 1) ch = 1;
    const int want = (148 * 4 + C / 64 - 1) / (C / 64);            // ~4 blocks per SM over all column groups
    if (ch > want) ch = want;
    colsum_vec4_kernel<T><<<dim3(C / 64, ch), 256, 0, st>>>(x, ld, rows, out);
    MRNB_CHECK_LAUNCH("colsum_vec4_kernel");
    return MRNB_OK;
  }
  colsum_kernel<T, false><<<dim3(cdiv(C, 32), chunks), dim3(32, 8), 0, st>>>(x, ld, rows, C, out, nullptr);
  MRNB_CHECK_LAUNCH("colsum_kernel");
  return MRNB_OK;
}
int launch_colstats(const float* x, long rows, int C, double* stats, cudaStream_t st) {
  int chunks = (int)(rows / 256); if (chunks < 1) chunks = 1; if (chunks > 148) chunks = 148;
  colsum_kernel<float, true><<<dim3(cdiv(C, 32), chunks), dim3(32, 8), 0, st>>>(x, C, rows, C, nullptr, stats);
  MRNB_CHECK_LAUNCH("colsum_kernel");
  return MRNB_OK;
}

// ------------------------------------------------------------------------------------------------
// GEMM dispatch.  Forward Linear: linear<AT>() (CUDA cores fp32 / persistent tcgen05 bf16).  Backward:
//   dX[M,K] = dY[M,N] . W[N,K];   dW[N,K] (+)= dY[M,N]^T . X[M,K]  (split over the M rows, atomics into a zeroed dW).
// fp32: gemm_f32.cu.  bf16: the general tcgen05 engine (gemm_tc2.cu) reading every tensor where it lies -- dY K-major
// and W MN-major for dX; dY and X both MN-major for dW -- so no transposed copy is ever made.  A contraction length
// that is not a multiple of 64 (the ragged charset C) is rounded up: TMA zero-fills both operands beyond their extent.
// ------------------------------------------------------------------------------------------------
typedef __nv_bfloat16 bf16;

template <typename AT>
int lin(const AT* A, long lda, const float* W32, const void* W16, const float* bias, void* out, long ldo, bool out_f32,
        int M, int N, int K, const float* res, const float* rowscale, int rows_per_scale, cudaStream_t st) {
  LinearArgs a{};
  a.A = A; a.lda = lda; a.a_gstride = (long)M * lda;
  a.W32 = W32; a.W16 = W16; a.w_gstride = (long)N * K;
  a.bias = bias; a.bias_gstride = N;
  a.out = out; a.ldo = ldo; a.o_gstride = (long)M * ldo; a.out_is_f32 = out_f32 ? 1 : 0;
  a.res = res; a.rowscale = rowscale; a.rows_per_scale = rows_per_scale;
  a.M = M; a.N = N; a.K = K; a.groups = 1;
  if (sizeof(AT) == 2) MRNB_CHECK_ARG(W16, "svtr_train: bf16 mode needs the 16-bit weight shadow (pack->h / fc_w16)");
  return linear<AT>(a, st);
}

// res (optional, dX's addressing): added to the product in the epilogue, before any 16-bit copy is written
int gemm_dx_f32(const float* dY, long ldy, const float* W, float* dX, long ldx, int M, int N, int K, cudaStream_t st,
                const float* res = nullptr) {
  MrnbGemm g{};
  g.res = res;
  g.A = dY; g.am = mrnb_axis(ldy); g.ak = mrnb_axis(1); g.a_kfast = 1;
  g.B = W; g.bk = mrnb_axis(K); g.bn = mrnb_axis(1); g.b_kfast = 0;
  g.C = dX; g.cm = mrnb_axis(ldx); g.cn = mrnb_axis(1);
  g.M = M; g.N = K; g.K = N; g.batch = 1; g.splitk = 1; g.alpha = 1.f; g.rows_per_scale = 1;
  return mrnb_sgemm(g, st);
}
int gemm_dw_f32(const float* dY, long ldy, const float* X, long ldx, float* dW, int rows, int N, int K, cudaStream_t st) {
  MrnbGemm g{};
  g.A = dY; g.am = mrnb_axis(1); g.ak = mrnb_axis(ldy); g.a_kfast = 0;
  g.B = X; g.bk = mrnb_axis(ldx); g.bn = mrnb_axis(1); g.b_kfast = 0;
  g.C = dW; g.cm = mrnb_axis(K); g.cn = mrnb_axis(1);
  g.M = N; g.N = K; g.K = rows; g.batch = 1; g.alpha = 1.f; g.rows_per_scale = 1;
  const int tile = (N >= 96 && K >= 96) ? 128 : 64;
  const long tiles = (long)cdiv(N, tile) * cdiv(K, tile);
  long sk = (148L * 4 + tiles - 1) / tiles;
  const long maxsk = rows / 128 > 0 ? rows / 128 : 1;
  if (sk > maxsk) sk = maxsk;
  if (sk < 1) sk = 1;
  g.splitk = (int)sk;
  return mrnb_sgemm(g, st);
}
int gemm_dx_tc(const bf16* dY, long ldy, const void* W16, float* dX, bf16* dX16, long ldx, int M, int N, int K, cudaStream_t st,
               const float* res = nullptr) {
  MrnbTcGemm2 g{};
  g.res = res;
  g.a = mrnb_operand_k2d(dY, M, N, ldy, 128, 1);
  g.b = mrnb_operand_mn2d(W16, K, N, K, 1);
  g.out32 = dX; g.out16 = dX16; g.cm = mrnb_axis(ldx); g.cn = mrnb_axis(1);
  g.M = M; g.N = K; g.K = (N + 63) / 64 * 64; g.groups = 1; g.splitk = 1; g.alpha = 1.f;
  return mrnb_tc_gemm2(g, st);
}
int gemm_dw_tc(const bf16* dY, long ldy, const bf16* X, long ldx, float* dW, int rows, int N, int K, cudaStream_t st) {
  // a contraction length (rows) that is not a multiple of 64 is rounded up: both MN-major operands are zero-filled by TMA
  MrnbTcGemm2 g{};
  g.a = mrnb_operand_mn2d(dY, N, rows, ldy, 1);
  g.b = mrnb_operand_mn2d(X, K, rows, ldx, 1);
  g.out32 = dW; g.cm = mrnb_axis(K); g.cn = mrnb_axis(1);
  g.M = N; g.N = K; g.K = (rows + 63) / 64 * 64; g.groups = 1; g.alpha = 1.f;
  const long tiles = (long)cdiv(N, 128) * cdiv(K, K >= 128 ? 128 : 64);
  long sk = (148L * 3 + tiles - 1) / tiles;
  const long maxsk = rows / 256 > 0 ? rows / 256 : 1;
  if (sk > maxsk) sk = maxsk;
  if (sk < 1) sk = 1;
  g.splitk = (int)sk;
  return mrnb_tc_gemm2(g, st);
}
// one gradient tensor in both flavours: fp32 (elementwise math, bias sums) and, in bf16 mode, its 16-bit GEMM operand
struct Grad { const float* f; const bf16* h; long ld; };

template <typename AT>
int gemm_dx(const Grad& dY, const float* W32, const void* W16, float* dX, bf16* dX16, long ldx, int M, int N, int K, cudaStream_t st,
            const float* res = nullptr) {
  if constexpr (sizeof(AT) == 4) return gemm_dx_f32(dY.f, dY.ld, W32, dX, ldx, M, N, K, st, res);
  else return gemm_dx_tc(dY.h, dY.ld, W16, dX, dX16, ldx, M, N, K, st, res);
}

// a training pack's feature [rows, 256] (AT) -> the caller's fp32 buffer: a copy in fp32 mode, the widened bf16 value
// (the operand the classifier head reads) in bf16 mode
template <typename AT>
__global__ void widen_kernel(const AT* __restrict__ x, float* __restrict__ y, long n) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) y[i] = to_f32<AT>(x[i]);
}
template <typename AT>
int gemm_dw(const Grad& dY, const AT* X, long ldx, float* dW, int rows, int N, int K, cudaStream_t st) {
  if constexpr (sizeof(AT) == 4) return gemm_dw_f32(dY.f, dY.ld, X, ldx, dW, rows, N, K, st);
  else return gemm_dw_tc(dY.h, dY.ld, X, ldx, dW, rows, N, K, st);
}

// fp32 [rows, C] (ld; vector loads when it is a multiple of 4) -> bf16 [rows, ld16] (a multiple of 8), columns C..ld16 zero; eight columns per thread
__global__ void cast_pad_rows_kernel(const float* __restrict__ x, long ld, int C, bf16* __restrict__ y, long ld16, long total) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;          // one group of 8 output columns
  const long per_row = ld16 / 8;
  if (i >= total / 8) return;
  const long r = i / per_row;
  const int c = (int)(i % per_row) * 8;
  float v[8];
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int cc = c + 4 * h;
    float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
    if ((ld & 3) == 0 && cc + 4 <= ld) {
      t = *reinterpret_cast<const float4*>(x + r * ld + cc);
    } else {                                               // unaligned rows: scalar loads
      const float* s = x + r * ld + cc;
      if (cc < C) t.x = s[0];
      if (cc + 1 < C) t.y = s[1];
      if (cc + 2 < C) t.z = s[2];
      if (cc + 3 < C) t.w = s[3];
    }
    v[4 * h] = cc < C ? t.x : 0.f; v[4 * h + 1] = cc + 1 < C ? t.y : 0.f;
    v[4 * h + 2] = cc + 2 < C ? t.z : 0.f; v[4 * h + 3] = cc + 3 < C ? t.w : 0.f;
  }
  uint32_t pk[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    __nv_bfloat162 hh = __floats2bfloat162_rn(v[2 * u], v[2 * u + 1]);
    pk[u] = *reinterpret_cast<uint32_t*>(&hh);
  }
  *reinterpret_cast<uint4*>(y + r * ld16 + c) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
}

// ------------------------------------------------------------------------------------------------
// Convolution lowering.  The forward GEMM reads im2col_nhwc_kernel's layout col[(b,oh,ow), (kh,kw,c)] (expert_util.cuh);
// col2im is its transpose.
// ------------------------------------------------------------------------------------------------
// bf16 im2col, eight channels per thread (two 16-byte loads, one 16-byte store); the channel count and the window are
// template parameters so that only the (row -> b, oh, ow) split divides by runtime values.
template <int C, int KH, int KW>
__global__ void __launch_bounds__(256)
im2col_nhwc_bf16_kernel(const float* __restrict__ x, bf16* __restrict__ col, int H, int W, int pad, int sh, int sw, int Ho,
                        int Wo, long pairs) {
  constexpr int G = C / 8, KK = KH * KW;
  const long pair = (long)blockIdx.x * (256 / G) + threadIdx.x / G;      // (output pixel, tap)
  if (pair >= pairs) return;
  const int c = (threadIdx.x % G) * 8;
  const int tap = (int)(pair % KK);
  long r = pair / KK;
  const int ow = (int)(r % Wo); r /= Wo;
  const int oh = (int)(r % Ho);
  const long b = r / Ho;
  const int ih = oh * sh - pad + tap / KW, iw = ow * sw - pad + tap % KW;
  uint4 o = make_uint4(0u, 0u, 0u, 0u);
  if (ih >= 0 && ih < H && iw >= 0 && iw < W) {
    const float4* src = reinterpret_cast<const float4*>(x + ((b * H + ih) * W + iw) * C + c);
    const float4 v0 = src[0], v1 = src[1];
    __nv_bfloat162 h0 = __floats2bfloat162_rn(v0.x, v0.y), h1 = __floats2bfloat162_rn(v0.z, v0.w);
    __nv_bfloat162 h2 = __floats2bfloat162_rn(v1.x, v1.y), h3 = __floats2bfloat162_rn(v1.z, v1.w);
    o = make_uint4(*reinterpret_cast<uint32_t*>(&h0), *reinterpret_cast<uint32_t*>(&h1), *reinterpret_cast<uint32_t*>(&h2),
                   *reinterpret_cast<uint32_t*>(&h3));
  }
  *reinterpret_cast<uint4*>(col + pair * C + c) = o;
}

// im2col of `rows` output pixels into the AT GEMM operand.  bf16 mode uses the eight-channel kernel for the channel counts
// and windows of the SVTR and CRNN convolutions; everything else takes the four-channel kernel.
template <typename AT>
int launch_im2col(const float* x, AT* col, int H, int W, int C, int KH, int KW, int pad, int sh, int sw, int Ho, int Wo,
                  long rows, cudaStream_t st) {
  if constexpr (sizeof(AT) == 2) {
    const long pairs = rows * KH * KW;
#define IM2COL_CASE(C_, KH_, KW_)                                                                                                 \
    if (C == C_ && KH == KH_ && KW == KW_) {                                                                                      \
      im2col_nhwc_bf16_kernel<C_, KH_, KW_><<<cdiv(pairs, 256 / (C_ / 8)), 256, 0, st>>>(x, col, H, W, pad, sh, sw, Ho, Wo, pairs); \
      MRNB_CHECK_LAUNCH("im2col_nhwc_bf16_kernel");                                                                               \
      return MRNB_OK;                                                                                                             \
    }
    IM2COL_CASE(32, 3, 3) IM2COL_CASE(64, 3, 3) IM2COL_CASE(128, 3, 3) IM2COL_CASE(256, 3, 3) IM2COL_CASE(512, 3, 3)
    IM2COL_CASE(512, 2, 2)
#undef IM2COL_CASE
  }
  const long c4 = rows * KH * KW * C / 4;
  im2col_nhwc_kernel<AT><<<cdiv(c4, 256), 256, 0, st>>>(x, col, H, W, C, KH, KW, pad, sh, sw, Ho, Wo, c4);
  MRNB_CHECK_LAUNCH("im2col_nhwc_kernel");
  return MRNB_OK;
}

// transpose of the im2col: dx[b,ih,iw,c] = sum of dcol over the (oh, ow, kh, kw) that read this pixel, taps in ascending
// (kh, kw) order.  Four channels per thread.
template <int KH, int KW>
__global__ void col2im_nhwc_kernel(const float* __restrict__ dcol, float* __restrict__ dx, int H, int W, int C, int pad,
                                   int sh, int sw, int Ho, int Wo, long total4) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total4) return;
  const int c4 = C / 4;
  const int c = (int)(i % c4) * 4;
  long r = i / c4;
  const int iw = (int)(r % W); r /= W;
  const int ih = (int)(r % H);
  const long b = r / H;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int kh = 0; kh < KH; ++kh) {
    const int th = ih + pad - kh;
    if (th < 0 || th % sh != 0) continue;
    const int oh = th / sh;
    if (oh >= Ho) continue;
#pragma unroll
    for (int kw = 0; kw < KW; ++kw) {
      const int tw = iw + pad - kw;
      if (tw < 0 || tw % sw != 0) continue;
      const int ow = tw / sw;
      if (ow >= Wo) continue;
      const float4 v = *reinterpret_cast<const float4*>(dcol + (((b * Ho + oh) * Wo + ow) * (KH * KW) + kh * KW + kw) * C + c);
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
  }
  *reinterpret_cast<float4*>(dx + i * 4) = acc;
}

// conv0 on the tensor cores: its weight [cout, 36] fp32 -> [cout, 64] bf16, the 36 taps zero padded to one 64-wide
// k-block; and back, the gradient [cout, 64] fp32 -> its first 36 columns
__global__ void pad_w0_kernel(const float* __restrict__ w, bf16* __restrict__ wp, int cout) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= cout * 64) return;
  const int o = i >> 6, k = i & 63;
  wp[i] = __float2bfloat16_rn(k < 36 ? w[o * 36 + k] : 0.f);
}
__global__ void unpad_dw0_kernel(const float* __restrict__ dwp, float* __restrict__ dw, int cout) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= cout * 36) return;
  dw[i] = dwp[(i / 36) * 64 + i % 36];
}

// ------------------------------------------------------------------------------------------------
// conv0 input gradient: the gradient with respect to the image of the first convolution of an expert (4 input
// channels, 3 x 3, pad 1, stride S, on the 32 x 256 image; Ho = 32 / S, Wo = 256 / S):
//   dimage[b,c,ih,iw] = sum over the taps (kh, kw) and output channels o that read pixel (ih, iw) of d[b,oh,ow,o] w[o,c,kh,kw]
// d: the gradient at conv0's output, NHWC [B,Ho,Wo,COUT] fp32.  dimage: NCHW [B,4,32,256] fp32, every element written.
// A gather, one thread per image pixel computing its four channels: taps in ascending (kh, kw) order, output channels in
// ascending order within a tap -- no atomics, so the result is bitwise repeatable.  The weight sits in shared memory as
// one float4 (its four input channels) per (tap, o).  W_HWC: the weight is [COUT,3,3,4] (the CRNN training pack), else
// nn.Conv2d's [COUT,4,3,3] (the SVTR pack).  Block = one image row (256 threads), grid (32, B).
// ------------------------------------------------------------------------------------------------
template <int COUT, int S, bool W_HWC>
__global__ void __launch_bounds__(256)
conv0_dimage_kernel(const float* __restrict__ d, const float* __restrict__ w, float* __restrict__ dimage) {
  constexpr int H = 32, W = 256, Ho = H / S, Wo = W / S;
  __shared__ float4 wsh[9 * COUT];                        // [tap][o]
  for (int i = threadIdx.x; i < 9 * COUT; i += blockDim.x) {
    const int o = i % COUT, tap = i / COUT;
    float v[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) v[c] = W_HWC ? w[(o * 9 + tap) * 4 + c] : w[(o * 4 + c) * 9 + tap];
    wsh[i] = make_float4(v[0], v[1], v[2], v[3]);
  }
  __syncthreads();
  const int iw = threadIdx.x, ih = blockIdx.x;
  const long b = blockIdx.y;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int kh = 0; kh < 3; ++kh) {
    const int th = ih + 1 - kh;
    if (th < 0 || th % S != 0 || th / S >= Ho) continue;
    const int oh = th / S;
#pragma unroll
    for (int kw = 0; kw < 3; ++kw) {
      const int tw = iw + 1 - kw;
      if (tw < 0 || tw % S != 0 || tw / S >= Wo) continue;
      const float4* src = reinterpret_cast<const float4*>(d + ((b * Ho + oh) * Wo + tw / S) * COUT);
      const float4* wt = wsh + (kh * 3 + kw) * COUT;
#pragma unroll 4
      for (int o4 = 0; o4 < COUT / 4; ++o4) {
        const float4 g = __ldg(src + o4);
        const float gv[4] = {g.x, g.y, g.z, g.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float4 wv = wt[o4 * 4 + j];
          acc.x = fmaf(gv[j], wv.x, acc.x); acc.y = fmaf(gv[j], wv.y, acc.y);
          acc.z = fmaf(gv[j], wv.z, acc.z); acc.w = fmaf(gv[j], wv.w, acc.w);
        }
      }
    }
  }
  float* out = dimage + (b * 4 * H + ih) * W + iw;
  out[0] = acc.x; out[(long)H * W] = acc.y; out[2L * H * W] = acc.z; out[3L * H * W] = acc.w;
}

// SVTR patch embedding conv0 (4 -> 32, stride 2): d [B,16,128,32], w [32,4,3,3]
int launch_svtr_conv0_dimage(const float* d, const float* w, float* dimage, int B, cudaStream_t st) {
  conv0_dimage_kernel<32, 2, false><<<dim3(32, B), 256, 0, st>>>(d, w, dimage);
  MRNB_CHECK_LAUNCH("conv0_dimage_kernel");
  return MRNB_OK;
}
// CRNN VGG conv0 (4 -> 64, stride 1): d [B,32,256,64], w [64,3,3,4]
int launch_crnn_conv0_dimage(const float* d, const float* w, float* dimage, int B, cudaStream_t st) {
  conv0_dimage_kernel<64, 1, true><<<dim3(32, B), 256, 0, st>>>(d, w, dimage);
  MRNB_CHECK_LAUNCH("conv0_dimage_kernel");
  return MRNB_OK;
}

// ------------------------------------------------------------------------------------------------
// BatchNorm backward, apply pass (after a reduce pass that left S1 = sum dz, S2 = sum dz * xhat per channel in sums):
// draw = gamma*rstd * (dz - S1/n - xhat * S2/n)   (batch statistics)   or   gamma*rstd * dz   (running statistics),
// written over d (+ optional 16-bit copy);  dgamma = S2, dbeta = S1 (both NULL: no parameter gradient, the input-only
// backward)
// ------------------------------------------------------------------------------------------------
__global__ void bn_bwd_apply_kernel(const float* __restrict__ raw, float* __restrict__ d, const float* __restrict__ ss,
                                    const float* __restrict__ mr, const double* __restrict__ sums, double count,
                                    int use_batch, float* __restrict__ dgamma, float* __restrict__ dbeta, int C, long total,
                                    bf16* __restrict__ d16) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (dgamma && i < C) { dgamma[i] = (float)sums[i * 2 + 1]; dbeta[i] = (float)sums[i * 2]; }
  if (i >= total) return;
  const int c = (int)(i % C);
  float dz = d[i];
  if (use_batch) {
    const float xh = (raw[i] - mr[c * 2]) * mr[c * 2 + 1];
    dz = dz - (float)(sums[c * 2] / count) - xh * (float)(sums[c * 2 + 1] / count);
  }
  const float v = ss[c * 2] * dz;
  d[i] = v;
  if (d16) d16[i] = __float2bfloat16_rn(v);
}
}  // namespace
