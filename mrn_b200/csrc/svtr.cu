// SVTR expert recogniser forward, grouped over the N per-task experts (one launch covers every expert).
//
// Reference (paths relative to /root/reference):
//   modules/svtr.py:500-528   SVTR.forward_features        modules/svtr.py:200-204  Block.forward (pre-norm)
//   modules/svtr.py:133-152   Attention.forward (Local mask :116-128)   modules/svtr.py:61-67  Mlp
//   modules/svtr.py:246-254   PatchEmbed (conv-BN-GELU x2)  modules/svtr.py:285-312  SubSample (conv s(2,1) + LN)
//   modules/model.py:82-101   Model_Extractor.forward (permute / avg-pool over H=1 / Linear 512->256)
//   modules/model.py:133-148  Model.forward (CTC head fc)
//
// Layout: activations are token-major [expert][sample][token][channel]; the residual stream is fp32, GEMM operands
// are AT (float in the fp32 parity mode, bf16 in the tensor-core mode).  Every dense contraction goes through
// linear<AT>() -> gemm_f32.cu (CUDA cores) or gemm_tc.cu (tcgen05/TMEM/TMA).
#include "common.cuh"
#include "gemm_f32.h"
#include "gemm_tc.h"
#include "mlp_tc.h"
#include "mixer_tc.h"
#include <stdlib.h>
#include "svtr.h"
#include "expert_util.cuh"

int mrnb_attention_tc(const void* qkv, void* out, int groups, int N, int d, int heads, int H, int W, int local, cudaStream_t st);

namespace {

// ------------------------------------------------------------------------------------------------
// LayerNorm over the channel axis: one warp per row.  gamma/beta are [groups, D]; group = row / rows_per_group.
// ------------------------------------------------------------------------------------------------
// Optional second LayerNorm (y2, bf16): y2 = LN_2(LN_1(x)) in the same pass -- the SubSample norm followed by the next
// stage's first norm1 (modules/svtr.py:311 then :201).
template <typename OT, int D, int RPW = 4>
__global__ void __launch_bounds__(256)
layernorm_kernel(const float* x, long x_gs, OT* y, long y_gs, const float* __restrict__ gamma,
                 const float* __restrict__ beta, long rows, long rows_per_group, float eps,
                 __nv_bfloat16* __restrict__ y2 = nullptr, long y2_gs = 0, const float* __restrict__ gamma2 = nullptr,
                 const float* __restrict__ beta2 = nullptr, float eps2 = 0.f) {
  constexpr int VPT = D / 32;
  // RPW rows per warp: all loads are issued before the first reduction
  const long row0 = ((long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * RPW;
  const int lane = threadIdx.x & 31;
  float v[RPW][VPT];
#pragma unroll
  for (int r = 0; r < RPW; ++r) {
    const long row = row0 + r;
    if (row < rows) {
      const float* xr = x + (row / rows_per_group) * x_gs + (row % rows_per_group) * D;
      if constexpr (VPT >= 4) {
#pragma unroll
        for (int c = 0; c < VPT / 4; ++c) {
          const float4 t = *reinterpret_cast<const float4*>(xr + c * 128 + lane * 4);
          v[r][c * 4] = t.x; v[r][c * 4 + 1] = t.y; v[r][c * 4 + 2] = t.z; v[r][c * 4 + 3] = t.w;
        }
      } else {
        const float2 t = *reinterpret_cast<const float2*>(xr + lane * 2);
        v[r][0] = t.x; v[r][1] = t.y;
      }
    } else {
#pragma unroll
      for (int j = 0; j < VPT; ++j) v[r][j] = 0.f;
    }
  }
#pragma unroll
  for (int r = 0; r < RPW; ++r) {
    const long row = row0 + r;
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < VPT; ++j) s += v[r][j];
    const float mean = warp_sum(s) * (1.0f / D);
    float q = 0.f;
#pragma unroll
    for (int j = 0; j < VPT; ++j) { const float d = v[r][j] - mean; q = fmaf(d, d, q); }
    const float rstd = rsqrtf(warp_sum(q) * (1.0f / D) + eps);
    if (row >= rows) continue;
    const long grp = row / rows_per_group;
    const float* g = gamma + grp * D;
    const float* bt = beta + grp * D;
    OT* yr = y + grp * y_gs + (row % rows_per_group) * D;
    if constexpr (VPT >= 4) {
#pragma unroll
      for (int c = 0; c < VPT / 4; ++c) {
        const int idx = c * 128 + lane * 4;
        const float4 g4 = *reinterpret_cast<const float4*>(g + idx), b4 = *reinterpret_cast<const float4*>(bt + idx);
        const float o0 = (v[r][c * 4] - mean) * rstd * g4.x + b4.x, o1 = (v[r][c * 4 + 1] - mean) * rstd * g4.y + b4.y;
        const float o2 = (v[r][c * 4 + 2] - mean) * rstd * g4.z + b4.z, o3 = (v[r][c * 4 + 3] - mean) * rstd * g4.w + b4.w;
        v[r][c * 4] = o0; v[r][c * 4 + 1] = o1; v[r][c * 4 + 2] = o2; v[r][c * 4 + 3] = o3;      // kept for the second norm
        if constexpr (sizeof(OT) == 4) {
          *reinterpret_cast<float4*>(yr + idx) = make_float4(o0, o1, o2, o3);
        } else {
          __nv_bfloat162 h0 = __floats2bfloat162_rn(o0, o1), h1 = __floats2bfloat162_rn(o2, o3);
          *reinterpret_cast<uint2*>(yr + idx) = make_uint2(*reinterpret_cast<uint32_t*>(&h0), *reinterpret_cast<uint32_t*>(&h1));
        }
      }
    } else {
      const int idx = lane * 2;
      const float o0 = (v[r][0] - mean) * rstd * g[idx] + bt[idx], o1 = (v[r][1] - mean) * rstd * g[idx + 1] + bt[idx + 1];
      if constexpr (sizeof(OT) == 4) {
        *reinterpret_cast<float2*>(yr + idx) = make_float2(o0, o1);
      } else {
        __nv_bfloat162 h0 = __floats2bfloat162_rn(o0, o1);
        *reinterpret_cast<uint32_t*>(yr + idx) = *reinterpret_cast<uint32_t*>(&h0);
      }
    }
    if constexpr (VPT >= 4) {
      if (y2) {                                   // warp-uniform
        float s2 = 0.f;
#pragma unroll
        for (int j = 0; j < VPT; ++j) s2 += v[r][j];
        const float mean2 = warp_sum(s2) * (1.0f / D);
        float q2 = 0.f;
#pragma unroll
        for (int j = 0; j < VPT; ++j) { const float d = v[r][j] - mean2; q2 = fmaf(d, d, q2); }
        const float rstd2 = rsqrtf(warp_sum(q2) * (1.0f / D) + eps2);
        __nv_bfloat16* y2r = y2 + grp * y2_gs + (row % rows_per_group) * D;
#pragma unroll
        for (int c = 0; c < VPT / 4; ++c) {
          const int idx = c * 128 + lane * 4;
          const float4 g4 = *reinterpret_cast<const float4*>(gamma2 + grp * D + idx), b4 = *reinterpret_cast<const float4*>(beta2 + grp * D + idx);
          __nv_bfloat162 h0 = __floats2bfloat162_rn((v[r][c * 4] - mean2) * rstd2 * g4.x + b4.x, (v[r][c * 4 + 1] - mean2) * rstd2 * g4.y + b4.y);
          __nv_bfloat162 h1 = __floats2bfloat162_rn((v[r][c * 4 + 2] - mean2) * rstd2 * g4.z + b4.z, (v[r][c * 4 + 3] - mean2) * rstd2 * g4.w + b4.w);
          *reinterpret_cast<uint2*>(y2r + idx) = make_uint2(*reinterpret_cast<uint32_t*>(&h0), *reinterpret_cast<uint32_t*>(&h1));
        }
      }
    }
  }
}

template <typename OT>
int launch_layernorm(const float* x, long x_gs, OT* y, long y_gs, const float* gamma, const float* beta, long rows,
                     long rows_per_group, int D, float eps, cudaStream_t st) {
  const int grid = cdiv(rows, 8 * 4);
  MrnbProfScope prof(MRNB_PROF_LN, st, 0.0, (double)rows * D * (4 + sizeof(OT)));
  // 128 / 256 wide: two rows per warp (measured 5 % faster than four in the step: 4.72 vs 4.49 TB/s; eight: 3.93)
  switch (D) {
    case 64: layernorm_kernel<OT, 64><<<grid, 256, 0, st>>>(x, x_gs, y, y_gs, gamma, beta, rows, rows_per_group, eps); break;
    case 128: layernorm_kernel<OT, 128, 2><<<cdiv(rows, 8 * 2), 256, 0, st>>>(x, x_gs, y, y_gs, gamma, beta, rows, rows_per_group, eps); break;
    case 256: layernorm_kernel<OT, 256, 2><<<cdiv(rows, 8 * 2), 256, 0, st>>>(x, x_gs, y, y_gs, gamma, beta, rows, rows_per_group, eps); break;
    case 512: layernorm_kernel<OT, 512><<<grid, 256, 0, st>>>(x, x_gs, y, y_gs, gamma, beta, rows, rows_per_group, eps); break;
    default: mrnb_set_error("layernorm: unsupported D=%d", D); return MRNB_ERR_UNSUPPORTED;
  }
  MRNB_CHECK_LAUNCH("layernorm_kernel");
  return MRNB_OK;
}

// y = LN_1(x) in place-compatible fp32, y2 = LN_2(y) in bf16 (D = 128 / 256)
int launch_layernorm2(const float* x, long x_gs, float* y, long y_gs, const float* gamma, const float* beta, float eps,
                      __nv_bfloat16* y2, long y2_gs, const float* gamma2, const float* beta2, float eps2, long rows,
                      long rows_per_group, int D, cudaStream_t st) {
  const int grid = cdiv(rows, 8 * 2);
  MrnbProfScope prof(MRNB_PROF_LN, st, 0.0, (double)rows * D * (4 + 4 + 2));
  if (D == 128) layernorm_kernel<float, 128, 2><<<grid, 256, 0, st>>>(x, x_gs, y, y_gs, gamma, beta, rows, rows_per_group, eps, y2, y2_gs, gamma2, beta2, eps2);
  else if (D == 256) layernorm_kernel<float, 256, 2><<<grid, 256, 0, st>>>(x, x_gs, y, y_gs, gamma, beta, rows, rows_per_group, eps, y2, y2_gs, gamma2, beta2, eps2);
  else { mrnb_set_error("layernorm2: unsupported D=%d", D); return MRNB_ERR_UNSUPPORTED; }
  MRNB_CHECK_LAUNCH("layernorm_kernel");
  return MRNB_OK;
}

// ------------------------------------------------------------------------------------------------
// Patch embedding.  conv0: 4->32, 3x3 s2 p1 on the NCHW image (shared by all experts) -> raw NHWC [I,B,16,128,32]
// plus per-channel sum / sum-of-squares for train-mode BatchNorm.
// ------------------------------------------------------------------------------------------------
template <typename OT>
__global__ void __launch_bounds__(128)
conv0_kernel(const float* __restrict__ img, const float* __restrict__ w /*[I,32,4,3,3]*/,
             const float* __restrict__ bias /*[I,32]*/, OT* __restrict__ out, double* __restrict__ stats /*[I,32,2]*/,
             int B) {
  // grid: (16 output rows, B, I); block: 128 threads = 128 output columns
  const int oh = blockIdx.x, b = blockIdx.y, e = blockIdx.z, ow = threadIdx.x;
  __shared__ __align__(16) float sw[32 * 36];
  __shared__ float sb[32];
  __shared__ float red[4][32][2];
  for (int k = threadIdx.x; k < 32 * 36; k += 128) sw[k] = w[(long)e * 32 * 36 + k];
  if (threadIdx.x < 32) sb[threadIdx.x] = bias[e * 32 + threadIdx.x];
  __syncthreads();
  float in[36];
#pragma unroll
  for (int c = 0; c < 4; ++c)
#pragma unroll
    for (int kh = 0; kh < 3; ++kh)
#pragma unroll
      for (int kw = 0; kw < 3; ++kw) {
        const int ih = oh * 2 - 1 + kh, iw = ow * 2 - 1 + kw;
        in[c * 9 + kh * 3 + kw] = (ih >= 0 && ih < 32 && iw >= 0 && iw < 256)
                                      ? __ldg(img + (((long)b * 4 + c) * 32 + ih) * 256 + iw) : 0.f;
      }
  OT* o = out + ((((long)e * B + b) * 16 + oh) * 128 + ow) * 32;
  const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
  // 36 taps x 32 channels per thread; the weights come from shared memory as broadcast 16-byte loads (9 per channel)
  float r[32];
#pragma unroll
  for (int oc = 0; oc < 32; ++oc) {
    const float4* w4 = reinterpret_cast<const float4*>(sw + oc * 36);
    float a = sb[oc];
#pragma unroll
    for (int k4 = 0; k4 < 9; ++k4) {
      const float4 wv = w4[k4];
      a = fmaf(in[k4 * 4], wv.x, a); a = fmaf(in[k4 * 4 + 1], wv.y, a);
      a = fmaf(in[k4 * 4 + 2], wv.z, a); a = fmaf(in[k4 * 4 + 3], wv.w, a);
    }
    r[oc] = a;
  }
#pragma unroll
  for (int oc0 = 0; oc0 < 32; oc0 += 8) {
    if constexpr (sizeof(OT) == 4) {
      *reinterpret_cast<float4*>(o + oc0) = make_float4(r[oc0], r[oc0 + 1], r[oc0 + 2], r[oc0 + 3]);
      *reinterpret_cast<float4*>(o + oc0 + 4) = make_float4(r[oc0 + 4], r[oc0 + 5], r[oc0 + 6], r[oc0 + 7]);
    } else {
      uint32_t pk[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        __nv_bfloat162 h = __floats2bfloat162_rn(r[oc0 + 2 * u], r[oc0 + 2 * u + 1]);
        pk[u] = *reinterpret_cast<uint32_t*>(&h);
      }
      *reinterpret_cast<uint4*>(o + oc0) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
    }
    if (stats) {
      float v[16];
#pragma unroll
      for (int u = 0; u < 8; ++u) { v[u] = r[oc0 + u]; v[8 + u] = r[oc0 + u] * r[oc0 + u]; }
      const float tot = warp_reduce16(v, lane);
      if ((lane & 1) == 0) {
        const int idx = (lane >> 1) & 15;
        red[wp][oc0 + (idx & 7)][idx >> 3] = tot;
      }
    }
  }
  if (stats) {
    __syncthreads();
    if (threadIdx.x < 64) {
      const int c = threadIdx.x >> 1, k = threadIdx.x & 1;
      const double t = (double)red[0][c][k] + (double)red[1][c][k] + (double)red[2][c][k] + (double)red[3][c][k];
      atomicAdd(stats + ((long)e * 32 + c) * 2 + k, t);
    }
  }
}

// The same convolution with TWO vertically adjacent output rows per thread: every broadcast 16-byte weight load feeds
// eight FMAs instead of four (the one-row kernel is co-limited by the SM's shared-memory load path: 288 LDS.128 next to
// 1152 FFMA per thread), and the five input rows the two windows cover are loaded once (60 instead of 72 taps).
// grid: (8 row pairs, B, I); block: 128 threads = 128 output columns.
template <typename OT>
__global__ void __launch_bounds__(128)
conv0_rows2_kernel(const float* __restrict__ img, const float* __restrict__ w /*[I,32,4,3,3]*/,
                   const float* __restrict__ bias /*[I,32]*/, OT* __restrict__ out, double* __restrict__ stats /*[I,32,2]*/,
                   int B) {
  const int oh0 = blockIdx.x * 2, b = blockIdx.y, e = blockIdx.z, ow = threadIdx.x;
  __shared__ __align__(16) float sw[32 * 36];
  __shared__ float sb[32];
  __shared__ float red[4][32][2];
  for (int k = threadIdx.x; k < 32 * 36; k += 128) sw[k] = w[(long)e * 32 * 36 + k];
  if (threadIdx.x < 32) sb[threadIdx.x] = bias[e * 32 + threadIdx.x];
  __syncthreads();
  float in[4][5][3];                           // input rows 2 * oh0 - 1 .. 2 * oh0 + 3
#pragma unroll
  for (int c = 0; c < 4; ++c)
#pragma unroll
    for (int rr = 0; rr < 5; ++rr)
#pragma unroll
      for (int kw = 0; kw < 3; ++kw) {
        const int ih = oh0 * 2 - 1 + rr, iw = ow * 2 - 1 + kw;
        in[c][rr][kw] = (ih >= 0 && ih < 32 && iw >= 0 && iw < 256) ? __ldg(img + (((long)b * 4 + c) * 32 + ih) * 256 + iw) : 0.f;
      }
  const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
  float r0[32], r1[32];
#pragma unroll
  for (int oc = 0; oc < 32; ++oc) {
    const float4* w4 = reinterpret_cast<const float4*>(sw + oc * 36);
    float a0 = sb[oc], a1 = a0;
#pragma unroll
    for (int k4 = 0; k4 < 9; ++k4) {
      const float4 wv = w4[k4];
      const float wq[4] = {wv.x, wv.y, wv.z, wv.w};
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int k = k4 * 4 + u, c = k / 9, kh = (k % 9) / 3, kw = k % 3;
        a0 = fmaf(in[c][kh][kw], wq[u], a0);
        a1 = fmaf(in[c][kh + 2][kw], wq[u], a1);
      }
    }
    r0[oc] = a0; r1[oc] = a1;
  }
#pragma unroll
  for (int p = 0; p < 2; ++p) {
    OT* o = out + ((((long)e * B + b) * 16 + oh0 + p) * 128 + ow) * 32;
#pragma unroll
    for (int oc0 = 0; oc0 < 32; oc0 += 8) {
      if constexpr (sizeof(OT) == 4) {
        *reinterpret_cast<float4*>(o + oc0) = p ? make_float4(r1[oc0], r1[oc0 + 1], r1[oc0 + 2], r1[oc0 + 3]) : make_float4(r0[oc0], r0[oc0 + 1], r0[oc0 + 2], r0[oc0 + 3]);
        *reinterpret_cast<float4*>(o + oc0 + 4) = p ? make_float4(r1[oc0 + 4], r1[oc0 + 5], r1[oc0 + 6], r1[oc0 + 7]) : make_float4(r0[oc0 + 4], r0[oc0 + 5], r0[oc0 + 6], r0[oc0 + 7]);
      } else {
        uint32_t pk[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          __nv_bfloat162 h = p ? __floats2bfloat162_rn(r1[oc0 + 2 * u], r1[oc0 + 2 * u + 1]) : __floats2bfloat162_rn(r0[oc0 + 2 * u], r0[oc0 + 2 * u + 1]);
          pk[u] = *reinterpret_cast<uint32_t*>(&h);
        }
        *reinterpret_cast<uint4*>(o + oc0) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
      }
    }
  }
  if (stats) {
#pragma unroll
    for (int oc0 = 0; oc0 < 32; oc0 += 8) {
      float v[16];
#pragma unroll
      for (int u = 0; u < 8; ++u) { v[u] = r0[oc0 + u] + r1[oc0 + u]; v[8 + u] = fmaf(r0[oc0 + u], r0[oc0 + u], r1[oc0 + u] * r1[oc0 + u]); }
      const float tot = warp_reduce16(v, lane);
      if ((lane & 1) == 0) {
        const int idx = (lane >> 1) & 15;
        red[wp][oc0 + (idx & 7)][idx >> 3] = tot;
      }
    }
    __syncthreads();
    if (threadIdx.x < 64) {
      const int c = threadIdx.x >> 1, k = threadIdx.x & 1;
      const double t = (double)red[0][c][k] + (double)red[1][c][k] + (double)red[2][c][k] + (double)red[3][c][k];
      atomicAdd(stats + ((long)e * 32 + c) * 2 + k, t);
    }
  }
}

// conv1: 32->64, 3x3 s2 p1 over GELU(BN(conv0)) (applied on load) -> raw NHWC [I,B,8,64,64] + BN statistics.
// grid (8 output rows, B, I); block 256 = 64 output columns x 4 groups of 16 output channels.
__global__ void __launch_bounds__(256)
conv1_kernel(const float* __restrict__ in /*[I,B,16,128,32]*/, const float* __restrict__ ss0 /*[I,32,2]*/,
             const float* __restrict__ w /*[I,64,3,3,32]*/, const float* __restrict__ bias /*[I,64]*/,
             float* __restrict__ out, double* __restrict__ stats /*[I,64,2]*/, int B) {
  extern __shared__ float sm[];
  float* s_in = sm;                       // [3][130][33]  (column index iw+1, zero border)
  float* s_w = sm + 12872;               // [288][64] (16B aligned)     k-major so a warp reads 16 consecutive oc (broadcast x4)
  const int oh = blockIdx.x, b = blockIdx.y, e = blockIdx.z, tid = threadIdx.x;
  for (int k = tid; k < 64 * 288; k += 256) {
    const int oc = k / 288, kk = k % 288;
    s_w[kk * 64 + oc] = w[(long)e * 64 * 288 + k];
  }
  for (int k = tid; k < 3 * 130 * 32; k += 256) {
    const int c = k % 32, col = (k / 32) % 130, r = k / (32 * 130);
    const int ih = oh * 2 - 1 + r, iw = col - 1;
    float v = 0.f;
    if (ih >= 0 && ih < 16 && iw >= 0 && iw < 128) {
      const float raw = in[((((long)e * B + b) * 16 + ih) * 128 + iw) * 32 + c];
      v = gelu_erf(fmaf(raw, ss0[(e * 32 + c) * 2], ss0[(e * 32 + c) * 2 + 1]));
    }
    s_in[(r * 130 + col) * 33 + c] = v;
  }
  __syncthreads();
  const int ow = tid & 63, og = tid >> 6;   // og: which 16 output channels
  float acc[16];
#pragma unroll
  for (int u = 0; u < 16; ++u) acc[u] = bias[e * 64 + og * 16 + u];
  for (int kh = 0; kh < 3; ++kh)
    for (int kw = 0; kw < 3; ++kw) {
      const float* ip = s_in + (kh * 130 + ow * 2 + kw) * 33;
      const float* wp_ = s_w + ((kh * 3 + kw) * 32) * 64 + og * 16;
#pragma unroll 8
      for (int c = 0; c < 32; ++c) {
        const float x = ip[c];
        const float4* w4 = reinterpret_cast<const float4*>(wp_ + c * 64);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float4 ww = w4[u];
          acc[u * 4] = fmaf(x, ww.x, acc[u * 4]); acc[u * 4 + 1] = fmaf(x, ww.y, acc[u * 4 + 1]);
          acc[u * 4 + 2] = fmaf(x, ww.z, acc[u * 4 + 2]); acc[u * 4 + 3] = fmaf(x, ww.w, acc[u * 4 + 3]);
        }
      }
    }
  float* o = out + ((((long)e * B + b) * 8 + oh) * 64 + ow) * 64 + og * 16;
#pragma unroll
  for (int u = 0; u < 4; ++u)
    *reinterpret_cast<float4*>(o + u * 4) = make_float4(acc[u * 4], acc[u * 4 + 1], acc[u * 4 + 2], acc[u * 4 + 3]);
  if (stats) {
    __shared__ float red[8][16][2];
    const int lane = tid & 31, wp = tid >> 5;      // warps 2*og, 2*og+1 share a channel group
#pragma unroll
    for (int u = 0; u < 16; ++u) {
      const float s1 = warp_sum(acc[u]), s2 = warp_sum(acc[u] * acc[u]);
      if (lane == 0) { red[wp][u][0] = s1; red[wp][u][1] = s2; }
    }
    __syncthreads();
    if (tid < 128) {
      const int c = tid >> 1, k = tid & 1, g = c >> 4, u = c & 15;
      atomicAdd(stats + ((long)e * 64 + c) * 2 + k, (double)red[2 * g][u][k] + (double)red[2 * g + 1][u][k]);
    }
  }
}

// bf16 mode: GELU(BN(conv0 raw)) -> bf16 NHWC activation with one zero pixel on each side of every row
// [img][16][130][32], the layout the implicit-GEMM conv1 gathers with TMA (two pixels = one 128-byte k-slot).
__global__ void bn_gelu_pad_kernel(const __nv_bfloat16* __restrict__ raw /*[I*B,16,128,32]*/, const float* __restrict__ ss0,
                                   __nv_bfloat16* __restrict__ act /*[I*B,16,130,32]*/, int B, long total8) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total8) return;
  const int c = (int)(i & 3) * 8;
  const int col = (int)((i >> 2) % 130);
  const long rowi = (i >> 2) / 130;            // img * 16 + h
  const int e = (int)(rowi / (16L * B));
  uint4 o = make_uint4(0u, 0u, 0u, 0u);
  if (col >= 1 && col <= 128) {
    const uint4 v = *reinterpret_cast<const uint4*>(raw + (rowi * 128 + (col - 1)) * 32 + c);
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&v);
    const float* ss = ss0 + (e * 32 + c) * 2;
    uint32_t pk[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      // minimax-tanh GELU (|error| 2.5e-5, below the bf16 rounding of the result): with erff the kernel was ALU bound
      const float a = gelu_fast(fmaf(__bfloat162float(h[u].x), ss[4 * u], ss[4 * u + 1]));
      const float b2 = gelu_fast(fmaf(__bfloat162float(h[u].y), ss[4 * u + 2], ss[4 * u + 3]));
      __nv_bfloat162 r = __floats2bfloat162_rn(a, b2);
      pk[u] = *reinterpret_cast<uint32_t*>(&r);
    }
    o = make_uint4(pk[0], pk[1], pk[2], pk[3]);
  }
  *reinterpret_cast<uint4*>(act + i * 8) = o;
}

// per-channel sum / sum of squares of a [I][rows][64] fp32 tensor (BatchNorm statistics of conv1), fp64 accumulation
__global__ void __launch_bounds__(256)
bn_stats_rows_kernel(const float* __restrict__ x, long rows, double* __restrict__ stats /*[I,64,2]*/) {
  __shared__ double sh[4][64][2];
  const int e = blockIdx.y, c = threadIdx.x & 63, rg = threadIdx.x >> 6;
  const long per = (rows + gridDim.x - 1) / gridDim.x;
  const long r0 = (long)blockIdx.x * per, r1 = r0 + per < rows ? r0 + per : rows;
  double s1 = 0.0, s2 = 0.0;
  const float* xp = x + (long)e * rows * 64 + c;
  for (long r = r0 + rg; r < r1; r += 4) { const float v = xp[r * 64]; s1 += v; s2 += (double)v * v; }
  sh[rg][c][0] = s1; sh[rg][c][1] = s2;
  __syncthreads();
  if (threadIdx.x < 128) {
    const int cc = threadIdx.x >> 1, k = threadIdx.x & 1;
    atomicAdd(stats + ((long)e * 64 + cc) * 2 + k, sh[0][cc][k] + sh[1][cc][k] + sh[2][cc][k] + sh[3][cc][k]);
  }
}

// tokens: x[e,b,n,c] = GELU(BN(conv1 raw)) + pos_embed[e,n,c]      (svtr.py:246-254,511)
// FAST (tensor-core mode): minimax-tanh GELU (|error| 2.5e-5) -- with erff the kernel is ALU bound (3.6 TB/s)
template <bool FAST>
__global__ void embed_kernel(const float* __restrict__ raw, const float* __restrict__ ss1 /*[I,64,2]*/,
                             const float* __restrict__ pos /*[I,512,64]*/, float* __restrict__ x, long per_expert,
                             __nv_bfloat16* __restrict__ ln_out /* optional: LN1 of blocks1.0, [I][rows][64] */,
                             const float* __restrict__ ln_gamma /*[I,64]*/, const float* __restrict__ ln_beta, float ln_eps) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;     // float4 index; a token row = 16 consecutive threads
  const int e = blockIdx.y;
  if (i * 4 >= per_expert) return;                                // per_expert % 1024 == 0: whole warps leave together
  const long off = (long)e * per_expert + i * 4;
  const int c = (int)((i * 4) % 64);
  const long n = ((i * 4) / 64) % 512;
  const float4 r = *reinterpret_cast<const float4*>(raw + off);
  const float4 p = *reinterpret_cast<const float4*>(pos + ((long)e * 512 + n) * 64 + c);
  const float* ss = ss1 + (e * 64 + c) * 2;
  float4 o;
  const float a0 = fmaf(r.x, ss[0], ss[1]), a1 = fmaf(r.y, ss[2], ss[3]), a2 = fmaf(r.z, ss[4], ss[5]), a3 = fmaf(r.w, ss[6], ss[7]);
  o.x = (FAST ? gelu_fast(a0) : gelu_erf(a0)) + p.x;
  o.y = (FAST ? gelu_fast(a1) : gelu_erf(a1)) + p.y;
  o.z = (FAST ? gelu_fast(a2) : gelu_erf(a2)) + p.z;
  o.w = (FAST ? gelu_fast(a3) : gelu_erf(a3)) + p.w;
  *reinterpret_cast<float4*>(x + off) = o;
  if (ln_out) {
    float s = (o.x + o.y) + (o.z + o.w);
#pragma unroll
    for (int k = 8; k > 0; k >>= 1) s += __shfl_xor_sync(0xffffffffu, s, k);
    const float mean = s * (1.0f / 64);
    const float d0 = o.x - mean, d1 = o.y - mean, d2 = o.z - mean, d3 = o.w - mean;
    float q = fmaf(d0, d0, fmaf(d1, d1, fmaf(d2, d2, d3 * d3)));
#pragma unroll
    for (int k = 8; k > 0; k >>= 1) q += __shfl_xor_sync(0xffffffffu, q, k);
    const float rstd = rsqrtf(q * (1.0f / 64) + ln_eps);
    const float4 g4 = *reinterpret_cast<const float4*>(ln_gamma + e * 64 + c), b4 = *reinterpret_cast<const float4*>(ln_beta + e * 64 + c);
    __nv_bfloat162 h0 = __floats2bfloat162_rn(d0 * rstd * g4.x + b4.x, d1 * rstd * g4.y + b4.y);
    __nv_bfloat162 h1 = __floats2bfloat162_rn(d2 * rstd * g4.z + b4.z, d3 * rstd * g4.w + b4.w);
    *reinterpret_cast<uint2*>(ln_out + off) = make_uint2(*reinterpret_cast<uint32_t*>(&h0), *reinterpret_cast<uint32_t*>(&h1));
  }
}

// ------------------------------------------------------------------------------------------------
// Attention.  One CTA per (expert*sample, head); one thread per query; K/V of the head staged in shared memory
// (row stride 36 floats: conflict-free LDS.128 both for broadcast (Global) and lane-distinct (Local) rows).
// Local mixer: |dh| <= 3, |dw| <= 5 window as index bounds (svtr.py:116-128), no dense mask.
// ------------------------------------------------------------------------------------------------
constexpr int KV_LD = 36;

template <typename AT, bool LOCAL>
__global__ void __launch_bounds__(512)
attention_kernel(const AT* __restrict__ qkv, AT* __restrict__ out, int N, int d, int heads, int H, int W) {
  extern __shared__ float sm[];
  float* sK = sm;
  float* sV = sm + (size_t)N * KV_LD;
  const int g = blockIdx.x, h = blockIdx.y, tid = threadIdx.x;
  const AT* base = qkv + (long)g * N * 3 * d;
  for (int k = tid; k < N * 32; k += blockDim.x) {
    const int n = k >> 5, j = k & 31;
    sK[n * KV_LD + j] = to_f32<AT>(base[(long)n * 3 * d + d + h * 32 + j]);
    sV[n * KV_LD + j] = to_f32<AT>(base[(long)n * 3 * d + 2 * d + h * 32 + j]);
  }
  __syncthreads();
  const int n = tid;
  if (n >= N) return;
  float q[32], acc[32];
  const float scale = 0.17677669529663688110f;    // 32^-0.5 (head_dim = 32 for every stage)
#pragma unroll
  for (int j = 0; j < 32; ++j) { q[j] = to_f32<AT>(base[(long)n * 3 * d + h * 32 + j]) * scale; acc[j] = 0.f; }
  float m = -INFINITY, l = 0.f;

  auto step = [&](int key, bool valid) {
    const float4* kr = reinterpret_cast<const float4*>(sK + key * KV_LD);
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 kk = kr[j];
      s = fmaf(q[4 * j], kk.x, s); s = fmaf(q[4 * j + 1], kk.y, s);
      s = fmaf(q[4 * j + 2], kk.z, s); s = fmaf(q[4 * j + 3], kk.w, s);
    }
    if (!valid) return;
    float p;
    if (s > m) {
      const float corr = expf(m - s);
      l *= corr;
#pragma unroll
      for (int j = 0; j < 32; ++j) acc[j] *= corr;
      m = s;
      p = 1.f;
    } else {
      p = expf(s - m);
    }
    l += p;
    const float4* vr = reinterpret_cast<const float4*>(sV + key * KV_LD);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 vv = vr[j];
      acc[4 * j] = fmaf(p, vv.x, acc[4 * j]); acc[4 * j + 1] = fmaf(p, vv.y, acc[4 * j + 1]);
      acc[4 * j + 2] = fmaf(p, vv.z, acc[4 * j + 2]); acc[4 * j + 3] = fmaf(p, vv.w, acc[4 * j + 3]);
    }
  };

  if constexpr (LOCAL) {
    const int qh = n / W, qw = n % W;
    for (int dh = -3; dh <= 3; ++dh) {
      const int kh = qh + dh;
      if (kh < 0 || kh >= H) continue;
      for (int dw = -5; dw <= 5; ++dw) {
        const int kw = qw + dw;
        const bool valid = kw >= 0 && kw < W;
        step(kh * W + (valid ? kw : qw), valid);
      }
    }
  } else {
    for (int key = 0; key < N; ++key) step(key, true);
  }
  const float inv = 1.0f / l;
  AT* o = out + ((long)g * N + n) * d + h * 32;
#pragma unroll
  for (int j = 0; j < 32; ++j) o[j] = from_f32<AT>(acc[j] * inv);
}

// ------------------------------------------------------------------------------------------------
// im2col for the SubSample conv (3x3, stride (2,1), pad 1) over token-major x[g, H, W, C]:
//   col[(g, oh, w), (kh, kw, c)] ; the conv weight is packed as [Cout, kh, kw, Cin] to match.
// ------------------------------------------------------------------------------------------------
template <typename AT>
__global__ void im2col_kernel(const float* __restrict__ x, long x_gs, int bc, AT* __restrict__ col, int H, int W, int C,
                              long total4) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;    // one float4 of channels
  if (i >= total4) return;
  const int c4 = C / 4;
  const int c = (int)(i % c4) * 4;
  long r = i / c4;
  const int tap = (int)(r % 9); r /= 9;
  const int w = (int)(r % W); r /= W;
  const int oh = (int)(r % (H / 2));
  const long g = r / (H / 2);
  const int ih = oh * 2 - 1 + tap / 3, iw = w - 1 + tap % 3;
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  if (ih >= 0 && ih < H && iw >= 0 && iw < W)
    v = *reinterpret_cast<const float4*>(x + (g / bc) * x_gs + (((g % bc) * H + ih) * W + iw) * C + c);
  AT* o = col + i * 4;
  o[0] = from_f32<AT>(v.x); o[1] = from_f32<AT>(v.y); o[2] = from_f32<AT>(v.z); o[3] = from_f32<AT>(v.w);
}

// bf16 copy of a grouped fp32 tensor: y[g][i] = x[g * x_gs + i], 4 elements per thread
__global__ void cast_groups_kernel(const float* __restrict__ x, long x_gs, __nv_bfloat16* __restrict__ y, long per_group4,
                                   long total4) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total4) return;
  const long g = i / per_group4, r = i % per_group4;
  const float4 v = *reinterpret_cast<const float4*>(x + g * x_gs + r * 4);
  __nv_bfloat162 h0 = __floats2bfloat162_rn(v.x, v.y), h1 = __floats2bfloat162_rn(v.z, v.w);
  *reinterpret_cast<uint2*>(y + i * 4) = make_uint2(*reinterpret_cast<uint32_t*>(&h0), *reinterpret_cast<uint32_t*>(&h1));
}

// features [I, Bc, T, D] (expert-major, fp32) -> router layout [Bc, I, T, D] fp32   (torch.stack(...,1), model.py:400)
// and, in the same pass, the bf16 copy (expert-major) that feeds the classifier heads
__global__ void feature_scatter_kernel(const float* __restrict__ src, float* __restrict__ dst, __nv_bfloat16* __restrict__ src16,
                                       int I, int Bc, long TD) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  const long total = (long)I * Bc * TD / 4;
  if (i >= total) return;
  const long e4 = i * 4;
  const long td = e4 % TD;
  const long b = (e4 / TD) % Bc;
  const long e = e4 / (TD * Bc);
  const float4 v = *reinterpret_cast<const float4*>(src + e4);
  if (dst) *reinterpret_cast<float4*>(dst + (b * I + e) * TD + td) = v;
  if (src16) {
    __nv_bfloat162 h0 = __floats2bfloat162_rn(v.x, v.y), h1 = __floats2bfloat162_rn(v.z, v.w);
    *reinterpret_cast<uint2*>(src16 + e4) = make_uint2(*reinterpret_cast<uint32_t*>(&h0), *reinterpret_cast<uint32_t*>(&h1));
  }
}

// First branch of a Block in tensor-core mode: the fused mixer kernel (mixer_tc.cu) or the unfused qkv GEMM / attention /
// proj GEMM sequence.  MRNB_MIXER = 0: never fused, 1 (default): fused for the 64- and 128-wide stages, 2: always fused,
// 3: fused for the 64-wide stage only.  Per launch at 1536 units (tools/mixer_bench.py, persistent attention kernel):
// d = 64 fused 0.467 ms vs unfused 0.565; d = 128 fused 0.465 vs unfused 0.41 in isolation -- but inside the step the
// unfused d = 128 blocks (qkv 117 + attention 229 + proj/LN 117 us) come out at the same 0.46 ms with twice the DRAM
// traffic (step 12.05 vs 11.99 ms), so they stay fused; d = 256 fused 0.448 vs unfused 0.341: unfused.
bool use_fused_mixer(int d) {
  static int v = -1;
  if (v < 0) { const char* e = getenv("MRNB_MIXER"); v = e ? atoi(e) : 1; }
  return v == 2 || (v == 1 && d <= 128) || (v == 3 && d <= 64);
}

template <typename AT>
size_t svtr_workspace_bytes_t(int I, int B, int Bc) {
  size_t s = 0;
  s += align_up((size_t)I * B * 16 * 128 * 32 * 4);        // conv0 raw (fp32; bf16 mode: bf16 raw + padded bf16 activation)
  if (sizeof(AT) == 2) s += align_up((size_t)I * B * 16 * 130 * 32 * 2);
  s += align_up((size_t)I * B * 8 * 64 * 64 * 4);          // conv1 raw
  s += align_up((size_t)I * 96 * 2 * 8);                    // stats
  s += align_up((size_t)I * 96 * 2 * 4);                    // scale/shift
  s += align_up((size_t)I * B * 32768 * 4);                 // x (all samples)
  const size_t u = (size_t)I * Bc * 32768;
  s += align_up(u * 4);                                     // xb (subsample output / ping-pong)
  s += align_up(u * sizeof(AT));                            // ln out
  s += align_up(u * 3 * sizeof(AT));                        // qkv
  s += align_up(u * sizeof(AT));                            // attention out
  s += align_up(u * 9 / 2 * sizeof(AT));                    // mlp hidden (4u) / im2col (4.5u)
  s += align_up((size_t)I * Bc * 64 * 256 * 4);             // features expert-major fp32
  s += align_up((size_t)I * Bc * 64 * 256 * sizeof(AT));    // features AT (classifier operand)
  return s + 4096;
}

template <typename AT>
struct SvtrWs {
  float* conv0; __nv_bfloat16* act0p; float* conv1; double* stats; float* ss; float* xall; float* xb;
  AT* lnout; AT* qkv; AT* att; AT* big; float* feat32; AT* featat;
};
template <typename AT>
SvtrWs<AT> carve_svtr(void* ws, size_t ws_bytes, int I, int B, int Bc) {
  Workspace W{(char*)ws, 0, ws_bytes};
  SvtrWs<AT> w{};
  w.conv0 = W.take<float>((size_t)I * B * 16 * 128 * 32);
  w.act0p = nullptr;
  if (sizeof(AT) == 2) w.act0p = W.take<__nv_bfloat16>((size_t)I * B * 16 * 130 * 32);
  w.conv1 = W.take<float>((size_t)I * B * 8 * 64 * 64);
  w.stats = W.take<double>((size_t)I * 96 * 2);
  w.ss = W.take<float>((size_t)I * 96 * 2);
  w.xall = W.take<float>((size_t)I * B * 32768);
  const size_t u = (size_t)I * Bc * 32768;
  w.xb = W.take<float>(u);
  w.lnout = W.take<AT>(u);
  w.qkv = W.take<AT>(u * 3);
  w.att = W.take<AT>(u);
  w.big = W.take<AT>(u * 9 / 2);
  w.feat32 = W.take<float>((size_t)I * Bc * 64 * 256);
  w.featat = W.take<AT>((size_t)I * Bc * 64 * 256);
  return w;
}

// Classifier heads fc_i = Linear(256, C_i) of every expert (modules/model.py:164,181) on the expert-major features
// [I][bc * 64][256].  Tensor-core mode: ONE grouped launch over the ragged (expert, m tile, n tile) list when the bf16
// weights are stacked in one allocation (ops.SvtrPack); route != NULL computes only the (expert, sample) pairs the hard
// route selects (modules/model.py:383-393: the other experts' logits are never read).  logits[e] == NULL skips expert e.
template <typename AT>
int svtr_heads(const MrnbSvtrPack& P, const void* fa, int bc, int b0, float* const* logits, const long* ld_logits,
               const int* route, cudaStream_t st) {
  const int I = P.n_experts;
  const long TD = 64 * 256;
  bool grouped = sizeof(AT) == 2;
  long w_rows = 0;
  MrnbTcHeads H{};
  if (grouped) {
    H.n_experts = I;
    for (int e = 0; e < I; ++e) {
      const long diff = (const char*)P.fc_w16[e] - (const char*)P.fc_w16[0];
      if (!logits[e] || !P.fc_w16[e] || diff < 0 || diff % 512 != 0 || diff / 512 > (1 << 24)) { grouped = false; break; }
      H.woff[e] = (int)(diff / 512); H.N[e] = P.n_class[e];
      H.out[e] = logits[e] + (size_t)b0 * 64 * ld_logits[e]; H.ldo[e] = ld_logits[e]; H.bias[e] = P.fc_b[e];
      if (H.woff[e] + H.N[e] > w_rows) w_rows = H.woff[e] + H.N[e];
    }
  }
  if (grouped) {
    H.route = route; H.rows_per_sample = 64; H.n_samples = bc;
    return mrnb_tc_heads(fa, 256, (long)bc * TD, P.fc_w16[0], w_rows, bc * 64, 256, H, st);
  }
  for (int e = 0; e < I; ++e) {
    if (!logits[e]) continue;
    LinearArgs fc{};
    fc.A = (const char*)fa + (size_t)e * bc * TD * sizeof(AT); fc.lda = 256;
    fc.W32 = P.fc_w[e]; fc.W16 = P.fc_w16[e]; fc.bias = P.fc_b[e];
    fc.out = logits[e] + (size_t)b0 * 64 * ld_logits[e]; fc.ldo = ld_logits[e]; fc.out_is_f32 = 1;
    fc.M = bc * 64; fc.N = P.n_class[e]; fc.K = 256; fc.groups = 1;
    MRNB_TRY(linear<AT>(fc, st));
  }
  return MRNB_OK;
}

template <typename AT>
int svtr_forward_t(const MrnbSvtrPack& P, const float* image, int B, int Bc, int bn_batch_stats, int update_running,
                   const float* drop_scales /*[I,12,2,B] or null*/, float* features /*[B,I,T,256]*/,
                   float* const* logits, const long* ld_logits, void* ws, size_t ws_bytes, cudaStream_t st) {
  const int I = P.n_experts;
  MRNB_CHECK_ARG(ws_bytes >= svtr_workspace_bytes_t<AT>(I, B, Bc), "svtr_forward: workspace too small (%zu < %zu)",
                 ws_bytes, svtr_workspace_bytes_t<AT>(I, B, Bc));
  SvtrWs<AT> wsp = carve_svtr<AT>(ws, ws_bytes, I, B, Bc);
  float* conv0 = wsp.conv0; __nv_bfloat16* act0p = wsp.act0p; float* conv1 = wsp.conv1; double* stats = wsp.stats; float* ss = wsp.ss;
  float* xall = wsp.xall; float* xb = wsp.xb; AT* lnout = wsp.lnout; AT* qkv = wsp.qkv; AT* att = wsp.att; AT* big = wsp.big;
  float* feat32 = wsp.feat32; AT* featat = wsp.featat;
  const size_t u = (size_t)I * Bc * 32768;
  (void)u;
  constexpr bool F32 = sizeof(AT) == 4;

  bool ln1_ready = false;      // the first norm1 of the coming stage has already been written to lnout
  // ---- patch embedding on the full batch (train-mode BN needs whole-batch statistics)
  double* st0 = stats; double* st1 = stats + (size_t)I * 32 * 2;
  float* ss0 = ss; float* ss1 = ss + (size_t)I * 32 * 2;
  if (bn_batch_stats) {
    cudaMemsetAsync(stats, 0, (size_t)I * 96 * 2 * sizeof(double), st);
  }
  mrnb_prof_begin(MRNB_PROF_CONV, st, 0.0, 0.0);
  if constexpr (sizeof(AT) == 2) {
    // ---- tensor-core mode: conv0 direct (K = 36) -> bf16 raw; conv1 as an implicit GEMM fed by TMA from the padded
    // NHWC activation (K = 3 kh x 128: {kw0,kw1} and {kw2, zero} 64-element slots), BN statistics from its fp32 output.
    __nv_bfloat16* raw0 = reinterpret_cast<__nv_bfloat16*>(conv0);
    conv0_rows2_kernel<__nv_bfloat16><<<dim3(8, B, I), 128, 0, st>>>(image, P.p[MRNB_P_CONV0_W], P.p[MRNB_P_CONV0_B], raw0,
                                                                      bn_batch_stats ? st0 : nullptr, B);
    MRNB_CHECK_LAUNCH("conv0_kernel");
    bn_finalize_kernel<<<cdiv(I * 32, 128), 128, 0, st>>>(st0, P.p[MRNB_P_BN0_W], P.p[MRNB_P_BN0_B],
                                                          (float*)P.p[MRNB_P_BN0_MEAN], (float*)P.p[MRNB_P_BN0_VAR], ss0, nullptr, I,
                                                          32, (double)B * 16 * 128, bn_batch_stats, update_running, 1e-5f);
    MRNB_CHECK_LAUNCH("bn_finalize_kernel");
    const long total8 = (long)I * B * 16 * 130 * 4;
    bn_gelu_pad_kernel<<<cdiv(total8, 256), 256, 0, st>>>(raw0, ss0, act0p, B, total8);
    MRNB_CHECK_LAUNCH("bn_gelu_pad_kernel");
    MRNB_CHECK_ARG(P.h[MRNB_P_CONV1_W], "svtr_forward: bf16 mode needs the GEMM-packed conv1 weight in h[MRNB_P_CONV1_W]");
    MrnbTcGemm g{};
    g.A = act0p; g.W = P.h[MRNB_P_CONV1_W]; g.ldw = 384; g.w_gstride = 64 * 384;
    g.bias = P.p[MRNB_P_CONV1_B]; g.bias_gstride = 64;
    g.out = conv1; g.ldo = 64; g.o_gstride = (long)B * 512 * 64; g.out_f32 = 1;
    g.M = B * 512; g.N = 64; g.K = 384; g.groups = I; g.rows_per_scale = 1;
    g.conv.enabled = 1;
    g.conv.dims[0] = 64; g.conv.dims[1] = 65; g.conv.dims[2] = 16; g.conv.dims[3] = (long)I * B;
    g.conv.strides[0] = 64; g.conv.strides[1] = 130 * 32; g.conv.strides[2] = 16L * 130 * 32;
    g.conv.box_h = 2; g.conv.box_img = 1; g.conv.sh = 2; g.conv.rows_per_img = 512; g.conv.per_kh = 2; g.conv.cch = 1;
    g.conv.pad_h = 1;
    g.conv.w_off = 0; g.conv.imgs_per_group = B;
    MRNB_TRY(mrnb_tc_gemm(g, st));
    if (bn_batch_stats) {
      bn_stats_rows_kernel<<<dim3(148, I), 256, 0, st>>>(conv1, (long)B * 512, st1);
      MRNB_CHECK_LAUNCH("bn_stats_rows_kernel");
    }
  } else {
    conv0_kernel<float><<<dim3(16, B, I), 128, 0, st>>>(image, P.p[MRNB_P_CONV0_W], P.p[MRNB_P_CONV0_B], conv0,
                                                         bn_batch_stats ? st0 : nullptr, B);
    MRNB_CHECK_LAUNCH("conv0_kernel");
    bn_finalize_kernel<<<cdiv(I * 32, 128), 128, 0, st>>>(st0, P.p[MRNB_P_BN0_W], P.p[MRNB_P_BN0_B],
                                                          (float*)P.p[MRNB_P_BN0_MEAN], (float*)P.p[MRNB_P_BN0_VAR], ss0, nullptr, I,
                                                          32, (double)B * 16 * 128, bn_batch_stats, update_running, 1e-5f);
    MRNB_CHECK_LAUNCH("bn_finalize_kernel");
    const size_t smem = (12872 + 288 * 64) * sizeof(float);
    static bool set = false;
    if (!set) { cudaFuncSetAttribute(conv1_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); set = true; }
    conv1_kernel<<<dim3(8, B, I), 256, smem, st>>>(conv0, ss0, P.p[MRNB_P_CONV1_W], P.p[MRNB_P_CONV1_B], conv1,
                                                    bn_batch_stats ? st1 : nullptr, B);
    MRNB_CHECK_LAUNCH("conv1_kernel");
  }
  bn_finalize_kernel<<<cdiv(I * 64, 128), 128, 0, st>>>(st1, P.p[MRNB_P_BN1_W], P.p[MRNB_P_BN1_B],
                                                        (float*)P.p[MRNB_P_BN1_MEAN], (float*)P.p[MRNB_P_BN1_VAR], ss1, nullptr, I,
                                                        64, (double)B * 8 * 64, bn_batch_stats, update_running, 1e-5f);
  MRNB_CHECK_LAUNCH("bn_finalize_kernel");
  {
    const long per_expert = (long)B * 32768;
    // tensor-core mode without batch chunking: blocks1.0.norm1 is emitted here as well (one pass over the tokens)
    ln1_ready = sizeof(AT) == 2 && Bc == B;
    embed_kernel<sizeof(AT) == 2><<<dim3(cdiv(per_expert / 4, 256), I), 256, 0, st>>>(
        conv1, ss1, P.p[MRNB_P_POS_EMBED], xall, per_expert, ln1_ready ? reinterpret_cast<__nv_bfloat16*>(lnout) : nullptr,
        P.p[MRNB_P_BLOCK0 + MRNB_PB_NORM1_W], P.p[MRNB_P_BLOCK0 + MRNB_PB_NORM1_B], 1e-6f);
    MRNB_CHECK_LAUNCH("embed_kernel");
  }
  mrnb_prof_end(MRNB_PROF_CONV, st);

  static const int DIMS[3] = {64, 128, 256}, DEPTH[3] = {3, 6, 3}, HEADS[3] = {2, 4, 8}, GH[3] = {8, 4, 2};
  static const int OUTS[3] = {128, 256, 512};
  {
    static bool set = false;
    if (!set) {
      const int mx = 2 * 512 * KV_LD * 4;
      cudaFuncSetAttribute(attention_kernel<AT, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx);
      cudaFuncSetAttribute(attention_kernel<AT, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx);
      set = true;
    }
  }

  for (int b0 = 0; b0 < B; b0 += Bc) {
    const int bc = (B - b0 < Bc) ? (B - b0) : Bc;
    // x for expert e, chunk: xall[e][b0 .. b0+bc) : group stride B*32768, rows contiguous inside a group
    float* x = xall + (size_t)b0 * 32768;
    long x_gs = (long)B * 32768;           // group (expert) stride of the current residual stream
    int blk = 0;
    for (int sidx = 0; sidx < 3; ++sidx) {
      const int d = DIMS[sidx], N = 32768 / d, heads = HEADS[sidx], H = GH[sidx], Wd = 64;
      const long rows_g = (long)bc * N;          // rows per expert in this chunk
      for (int j = 0; j < DEPTH[sidx]; ++j, ++blk) {
        const int pb = MRNB_P_BLOCK0 + blk * MRNB_PB_COUNT;
        const bool local = blk < 6;
        // tensor-core mode, d <= 128: the residual GEMMs (proj, fc2) own whole rows and emit the following LayerNorm
        const bool fuse_ln = sizeof(AT) == 2 && d <= 128 && (rows_g % 128) == 0;
        // LN1 (per expert: x groups are strided, outputs packed [I, rows_g, d]); fused into the previous block's fc2
        if (!(fuse_ln && j > 0) && !(j == 0 && ln1_ready))
          MRNB_TRY(launch_layernorm<AT>(x, x_gs, lnout, rows_g * d, P.p[pb + MRNB_PB_NORM1_W], P.p[pb + MRNB_PB_NORM1_B],
                                        rows_g * I, rows_g, d, 1e-6f, st));
        if (j == 0) ln1_ready = false;
        if (sizeof(AT) == 2 && use_fused_mixer(d)) {
          // tensor-core mode: the whole first branch (qkv GEMM -> attention -> proj + DropPath + residual [+ norm2]) is
          // one persistent kernel; q, k, v, scores and probabilities never reach HBM (mixer_tc.cu)
          MrnbMixer mx{};
          mx.A = lnout; mx.Wqkv = P.h[pb + MRNB_PB_QKV_W]; mx.bqkv = P.p[pb + MRNB_PB_QKV_B];
          mx.Wproj = P.h[pb + MRNB_PB_PROJ_W]; mx.bproj = P.p[pb + MRNB_PB_PROJ_B];
          mx.x = x; mx.x_gstride = x_gs;
          if (drop_scales) { mx.rowscale = drop_scales + ((size_t)blk * 2 + 0) * B + b0; mx.rowscale_gstride = (long)12 * 2 * B; }
          if (fuse_ln) { mx.ln_out = lnout; mx.ln_gamma = P.p[pb + MRNB_PB_NORM2_W]; mx.ln_beta = P.p[pb + MRNB_PB_NORM2_B]; mx.ln_eps = 1e-6f; }
          mx.D = d; mx.groups = I; mx.units_per_group = bc; mx.local = local ? 1 : 0;
          MRNB_TRY(mrnb_mixer_tc(mx, st));
        } else {
          LinearArgs a{};
          a.A = lnout; a.lda = d; a.a_gstride = rows_g * d;
          a.W32 = P.p[pb + MRNB_PB_QKV_W]; a.W16 = P.h[pb + MRNB_PB_QKV_W]; a.w_gstride = (long)3 * d * d;
          a.bias = P.p[pb + MRNB_PB_QKV_B]; a.bias_gstride = 3 * d;
          a.out = qkv; a.ldo = 3 * d; a.o_gstride = rows_g * 3 * d; a.out_is_f32 = F32;
          a.M = (int)rows_g; a.N = 3 * d; a.K = d; a.groups = I;
          MRNB_TRY(linear<AT>(a, st));
          {
            const size_t smem = (size_t)2 * N * KV_LD * sizeof(float);
            dim3 grid(I * bc, heads);
            double pairs = (double)N * N;
            if (local) {
              double sh = 0, sw = 0;
              for (int h = 0; h < H; ++h) sh += (h + 3 < H ? h + 3 : H - 1) - (h - 3 > 0 ? h - 3 : 0) + 1;
              for (int w2 = 0; w2 < Wd; ++w2) sw += (w2 + 5 < Wd ? w2 + 5 : Wd - 1) - (w2 - 5 > 0 ? w2 - 5 : 0) + 1;
              pairs = sh * sw;
            }
            MrnbProfScope prof(MRNB_PROF_ATTN, st, 4.0 * 32 * pairs * heads * I * bc,
                               (double)I * bc * N * d * 4 * sizeof(AT));
            if constexpr (sizeof(AT) == 2) {
              MRNB_TRY(mrnb_attention_tc(qkv, att, I * bc, N, d, heads, H, Wd, local ? 1 : 0, st));     // tcgen05 path
            } else {
              if (local) attention_kernel<AT, true><<<grid, N, smem, st>>>(qkv, att, N, d, heads, H, Wd);
              else attention_kernel<AT, false><<<grid, N, smem, st>>>(qkv, att, N, d, heads, H, Wd);
              MRNB_CHECK_LAUNCH("attention_kernel");
            }
          }
          // proj + DropPath scale + residual (in place on x)
          LinearArgs pr{};
          pr.A = att; pr.lda = d; pr.a_gstride = rows_g * d;
          pr.W32 = P.p[pb + MRNB_PB_PROJ_W]; pr.W16 = P.h[pb + MRNB_PB_PROJ_W]; pr.w_gstride = (long)d * d;
          pr.bias = P.p[pb + MRNB_PB_PROJ_B]; pr.bias_gstride = d;
          pr.out = x; pr.ldo = d; pr.o_gstride = x_gs; pr.out_is_f32 = 1; pr.res = x;
          if (drop_scales) {
            pr.rowscale = drop_scales + ((size_t)blk * 2 + 0) * B + b0; pr.rows_per_scale = N;
            pr.rowscale_gstride = (long)12 * 2 * B;
          }
          pr.M = (int)rows_g; pr.N = d; pr.K = d; pr.groups = I;
          if (fuse_ln) { pr.ln_out = lnout; pr.ln_gamma = P.p[pb + MRNB_PB_NORM2_W]; pr.ln_beta = P.p[pb + MRNB_PB_NORM2_B]; pr.ln_eps = 1e-6f; }
          MRNB_TRY(linear<AT>(pr, st));
        }
        if (!fuse_ln)
          MRNB_TRY(launch_layernorm<AT>(x, x_gs, lnout, rows_g * d, P.p[pb + MRNB_PB_NORM2_W], P.p[pb + MRNB_PB_NORM2_B],
                                        rows_g * I, rows_g, d, 1e-6f, st));
        if constexpr (sizeof(AT) == 2) {
          // fused MLP branch: fc1 -> GELU -> fc2 -> DropPath -> +residual (-> next LN1), hidden kept on chip
          MrnbMlp mp{};
          mp.A = lnout; mp.W1 = P.h[pb + MRNB_PB_FC1_W]; mp.W2 = P.h[pb + MRNB_PB_FC2_W];
          mp.b1 = P.p[pb + MRNB_PB_FC1_B]; mp.b2 = P.p[pb + MRNB_PB_FC2_B];
          mp.x = x; mp.x_gstride = x_gs;
          if (drop_scales) {
            mp.rowscale = drop_scales + ((size_t)blk * 2 + 1) * B + b0; mp.rows_per_scale = N;
            mp.rowscale_gstride = (long)12 * 2 * B;
          }
          if (fuse_ln && j + 1 < DEPTH[sidx]) {
            const int pn = pb + MRNB_PB_COUNT;
            mp.ln_out = lnout; mp.ln_gamma = P.p[pn + MRNB_PB_NORM1_W]; mp.ln_beta = P.p[pn + MRNB_PB_NORM1_B]; mp.ln_eps = 1e-6f;
          }
          if (j + 1 == DEPTH[sidx]) mp.cast_out = att;      // bf16 copy of the stage output = A operand of the SubSample conv
          mp.M = (int)rows_g; mp.D = d; mp.groups = I;
          MRNB_TRY(mrnb_mlp_tc(mp, st));
        } else {
          LinearArgs f1{};
          f1.A = lnout; f1.lda = d; f1.a_gstride = rows_g * d;
          f1.W32 = P.p[pb + MRNB_PB_FC1_W]; f1.W16 = P.h[pb + MRNB_PB_FC1_W]; f1.w_gstride = (long)4 * d * d;
          f1.bias = P.p[pb + MRNB_PB_FC1_B]; f1.bias_gstride = 4 * d;
          f1.out = big; f1.ldo = 4 * d; f1.o_gstride = rows_g * 4 * d; f1.out_is_f32 = F32; f1.gelu = 1;
          f1.M = (int)rows_g; f1.N = 4 * d; f1.K = d; f1.groups = I;
          MRNB_TRY(linear<AT>(f1, st));
          LinearArgs f2{};
          f2.A = big; f2.lda = 4 * d; f2.a_gstride = rows_g * 4 * d;
          f2.W32 = P.p[pb + MRNB_PB_FC2_W]; f2.W16 = P.h[pb + MRNB_PB_FC2_W]; f2.w_gstride = (long)4 * d * d;
          f2.bias = P.p[pb + MRNB_PB_FC2_B]; f2.bias_gstride = d;
          f2.out = x; f2.ldo = d; f2.o_gstride = x_gs; f2.out_is_f32 = 1; f2.res = x;
          if (drop_scales) {
            f2.rowscale = drop_scales + ((size_t)blk * 2 + 1) * B + b0; f2.rows_per_scale = N;
            f2.rowscale_gstride = (long)12 * 2 * B;
          }
          f2.M = (int)rows_g; f2.N = d; f2.K = 4 * d; f2.groups = I;
          if (fuse_ln && j + 1 < DEPTH[sidx]) {      // next block's norm1
            const int pn = pb + MRNB_PB_COUNT;
            f2.ln_out = lnout; f2.ln_gamma = P.p[pn + MRNB_PB_NORM1_W]; f2.ln_beta = P.p[pn + MRNB_PB_NORM1_B]; f2.ln_eps = 1e-6f;
          }
          MRNB_TRY(linear<AT>(f2, st));
        }
      }
      // SubSample: im2col -> conv GEMM (+bias) -> LN(eps 1e-5)
      const int Co = OUTS[sidx];
      const long orows_g = (long)bc * (H / 2) * Wd;
      const int ps = MRNB_P_SUB0 + sidx * MRNB_PS_COUNT;
      float* cv = (x == xb) ? xall : xb;          // conv output buffer distinct from x
      // (xall chunk region is free to reuse once x has moved to xb and vice versa)
      float* cvx = (cv == xall) ? xall + (size_t)b0 * 32768 : xb;
      const long cv_gs = (cv == xall) ? (long)B * 32768 : (long)bc * 32768;
      if constexpr (sizeof(AT) == 2) {
        // implicit GEMM: bf16 copy of the NHWC residual stream, A tiles gathered by TMA (zero fill = padding)
        // (att already holds the bf16 copy of x: written by the last block's fused-MLP epilogue)
        MrnbTcGemm g{};
        g.A = att; g.W = P.h[ps + MRNB_PS_CONV_W]; g.ldw = 9 * d; g.w_gstride = (long)Co * 9 * d;
        g.bias = P.p[ps + MRNB_PS_CONV_B]; g.bias_gstride = Co;
        g.out = cvx; g.ldo = Co; g.o_gstride = cv_gs; g.out_f32 = 1;
        g.M = (int)orows_g; g.N = Co; g.K = 9 * d; g.groups = I; g.rows_per_scale = 1;
        g.conv.enabled = 1;
        g.conv.dims[0] = d; g.conv.dims[1] = Wd; g.conv.dims[2] = H; g.conv.dims[3] = (long)I * bc;
        g.conv.strides[0] = d; g.conv.strides[1] = (long)Wd * d; g.conv.strides[2] = (long)H * Wd * d;
        const int Ho = H / 2;
        g.conv.box_h = Ho >= 2 ? 2 : 1; g.conv.box_img = Ho >= 2 ? 1 : 2; g.conv.sh = 2; g.conv.pad_h = 1;
        g.conv.rows_per_img = Ho * Wd; g.conv.per_kh = 3 * (d / 64); g.conv.cch = d / 64; g.conv.w_off = -1;
        g.conv.imgs_per_group = bc;
        MRNB_TRY(mrnb_tc_gemm(g, st));
      } else {
      {
        const long total4 = (long)I * orows_g * 9 * d / 4;
        im2col_kernel<AT><<<cdiv(total4, 256), 256, 0, st>>>(x, x_gs, bc, big, H, Wd, d, total4);
        MRNB_CHECK_LAUNCH("im2col_kernel");
      }
      LinearArgs cvl{};
      cvl.A = big; cvl.lda = 9 * d; cvl.a_gstride = orows_g * 9 * d;
      cvl.W32 = P.p[ps + MRNB_PS_CONV_W]; cvl.W16 = P.h[ps + MRNB_PS_CONV_W]; cvl.w_gstride = (long)Co * 9 * d;
      cvl.bias = P.p[ps + MRNB_PS_CONV_B]; cvl.bias_gstride = Co;
      cvl.out = cvx; cvl.ldo = Co; cvl.o_gstride = cv_gs; cvl.out_is_f32 = 1;
      cvl.M = (int)orows_g; cvl.N = Co; cvl.K = 9 * d; cvl.groups = I;
      MRNB_TRY(linear<AT>(cvl, st));
      }
      if (sidx < 2) {
        // LN in place (fp32 -> fp32) : next stage's residual stream
        if constexpr (sizeof(AT) == 2) {
          // SubSample norm in place + the next stage's first norm1 in the same pass
          const int pn = MRNB_P_BLOCK0 + (blk) * MRNB_PB_COUNT;      // blk already points at the next stage's first block
          MRNB_TRY(launch_layernorm2(cvx, cv_gs, cvx, cv_gs, P.p[ps + MRNB_PS_NORM_W], P.p[ps + MRNB_PS_NORM_B], 1e-5f,
                                     reinterpret_cast<__nv_bfloat16*>(lnout), orows_g * Co, P.p[pn + MRNB_PB_NORM1_W],
                                     P.p[pn + MRNB_PB_NORM1_B], 1e-6f, orows_g * I, orows_g, Co, st));
          ln1_ready = true;
        } else {
          MRNB_TRY(launch_layernorm<float>(cvx, cv_gs, cvx, cv_gs, P.p[ps + MRNB_PS_NORM_W], P.p[ps + MRNB_PS_NORM_B],
                                           orows_g * I, orows_g, Co, 1e-5f, st));
        }
        x = cvx; x_gs = cv_gs;
      } else {
        // last merge: LN -> AT [I, bc*64, 512] visual feature (model.py:88-95 relabel), then Linear 512->256
        MRNB_TRY(launch_layernorm<AT>(cvx, cv_gs, lnout, orows_g * Co, P.p[ps + MRNB_PS_NORM_W], P.p[ps + MRNB_PS_NORM_B],
                                      orows_g * I, orows_g, Co, 1e-5f, st));
        LinearArgs sq{};
        sq.A = lnout; sq.lda = 512; sq.a_gstride = orows_g * 512;
        sq.W32 = P.p[MRNB_P_SEQ_W]; sq.W16 = P.h[MRNB_P_SEQ_W]; sq.w_gstride = 256 * 512;
        sq.bias = P.p[MRNB_P_SEQ_B]; sq.bias_gstride = 256;
        sq.out = feat32; sq.ldo = 256; sq.o_gstride = orows_g * 256; sq.out_is_f32 = 1;
        sq.M = (int)orows_g; sq.N = 256; sq.K = 512; sq.groups = I;
        MRNB_TRY(linear<AT>(sq, st));
      }
    }
    // features -> router layout; classifier heads (ragged N = C_i)
    {
      const long TD = 64 * 256;
      const long total4 = (long)I * bc * TD / 4;
      const void* fa = feat32;
      if (features || !F32) {
        feature_scatter_kernel<<<cdiv(total4, 256), 256, 0, st>>>(feat32, features ? features + (size_t)b0 * I * TD : nullptr,
                                                                  F32 ? nullptr : reinterpret_cast<__nv_bfloat16*>(featat), I, bc, TD);
        MRNB_CHECK_LAUNCH("feature_scatter_kernel");
        if (!F32) fa = featat;
      }
      if (logits) {
        bool any = false;
        for (int e = 0; e < I; ++e) any = any || logits[e] != nullptr;
        if (any) MRNB_TRY(svtr_heads<AT>(P, fa, bc, b0, logits, ld_logits, nullptr, st));
      }
    }
  }
  return MRNB_OK;
}

}  // namespace

extern "C" size_t mrnb_svtr_workspace_bytes(int n_experts, int B, int chunk, int prec) {
  if (chunk <= 0 || chunk > B) chunk = B;
  return prec == MRNB_PREC_BF16 ? svtr_workspace_bytes_t<__nv_bfloat16>(n_experts, B, chunk)
                                : svtr_workspace_bytes_t<float>(n_experts, B, chunk);
}

extern "C" int mrnb_svtr_experts_forward(const MrnbSvtrPack* pack, const float* image, int B, int chunk, int prec,
                                         int bn_batch_stats, int update_running, const float* drop_scales,
                                         float* features, float* const* logits, const long* ld_logits, void* workspace,
                                         size_t workspace_bytes, cudaStream_t stream) {
  MRNB_CHECK_ARG(pack && image && workspace && B > 0, "svtr_experts_forward: null/empty argument");
  MRNB_CHECK_ARG(pack->n_experts >= 1 && pack->n_experts <= MRNB_MAX_EXPERTS, "svtr_experts_forward: n_experts out of range");
  MRNB_CHECK_ARG(!bn_batch_stats || B * 16 * 128 > 1, "svtr_experts_forward: batch statistics need more than one value");
  if (chunk <= 0 || chunk > B) chunk = B;
  for (int k = 0; k < MRNB_P_COUNT; ++k) MRNB_CHECK_ARG(pack->p[k], "svtr_experts_forward: parameter slot %d is null", k);
  if (prec == MRNB_PREC_BF16) {
    return svtr_forward_t<__nv_bfloat16>(*pack, image, B, chunk, bn_batch_stats, update_running, drop_scales, features,
                                         logits, ld_logits, workspace, workspace_bytes, stream);
  } else if (prec == MRNB_PREC_FP32) {
    return svtr_forward_t<float>(*pack, image, B, chunk, bn_batch_stats, update_running, drop_scales, features, logits,
                                 ld_logits, workspace, workspace_bytes, stream);
  }
  mrnb_set_error("svtr_experts_forward: unknown precision %d", prec);
  return MRNB_ERR_ARG;
}

// Classifier heads on the features left in `workspace` by the last mrnb_svtr_experts_forward call (chunk = 0) with the
// same (pack, B, prec).  route_index: NULL = every expert for every sample; device int32 [B] = hard route
// (modules/model.py:383-393): only the routed expert's head is evaluated per sample, logits rows of the other
// (expert, sample) pairs are left untouched (mrnb_gate_combine never reads them for a one-hot gate).
extern "C" int mrnb_svtr_heads(const MrnbSvtrPack* pack, int B, int prec, const int* route_index, float* const* logits,
                               const long* ld_logits, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  MRNB_CHECK_ARG(pack && logits && ld_logits && workspace && B > 0, "svtr_heads: null/empty argument");
  MRNB_CHECK_ARG(pack->n_experts >= 1 && pack->n_experts <= MRNB_MAX_EXPERTS, "svtr_heads: n_experts out of range");
  const int I = pack->n_experts;
  if (prec == MRNB_PREC_BF16) {
    MRNB_CHECK_ARG(workspace_bytes >= svtr_workspace_bytes_t<__nv_bfloat16>(I, B, B), "svtr_heads: workspace too small");
    SvtrWs<__nv_bfloat16> w = carve_svtr<__nv_bfloat16>(workspace, workspace_bytes, I, B, B);
    return svtr_heads<__nv_bfloat16>(*pack, w.featat, B, 0, logits, ld_logits, route_index, stream);
  } else if (prec == MRNB_PREC_FP32) {
    MRNB_CHECK_ARG(workspace_bytes >= svtr_workspace_bytes_t<float>(I, B, B), "svtr_heads: workspace too small");
    SvtrWs<float> w = carve_svtr<float>(workspace, workspace_bytes, I, B, B);
    // parity mode: plain fp32 GEMMs for every (expert, sample) pair (identical logits; the route only saves work)
    return svtr_heads<float>(*pack, w.feat32, B, 0, logits, ld_logits, nullptr, stream);
  }
  mrnb_set_error("svtr_heads: unknown precision %d", prec);
  return MRNB_ERR_ARG;
}

// Stand-alone ops for the tests.
extern "C" int mrnb_layernorm_f32(const float* x, float* y, const float* gamma, const float* beta, long rows, int D,
                                  float eps, cudaStream_t stream) {
  MRNB_CHECK_ARG(x && y && gamma && beta && rows > 0, "layernorm: bad argument");
  return launch_layernorm<float>(x, 0, y, 0, gamma, beta, rows, rows, D, eps, stream);
}

extern "C" int mrnb_svtr_attention_f32(const float* qkv, float* out, int groups, int N, int d, int heads, int H, int W,
                                       int local, cudaStream_t stream) {
  MRNB_CHECK_ARG(qkv && out && groups > 0 && N > 0 && N <= 512 && d == heads * 32 && H * W == N, "svtr_attention: bad argument");
  const size_t smem = (size_t)2 * N * KV_LD * sizeof(float);
  static bool set = false;
  if (!set) {
    const int mx = 2 * 512 * KV_LD * 4;
    cudaFuncSetAttribute(attention_kernel<float, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx);
    cudaFuncSetAttribute(attention_kernel<float, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx);
    set = true;
  }
  dim3 grid(groups, heads);
  if (local) attention_kernel<float, true><<<grid, N, smem, stream>>>(qkv, out, N, d, heads, H, W);
  else attention_kernel<float, false><<<grid, N, smem, stream>>>(qkv, out, N, d, heads, H, W);
  MRNB_CHECK_LAUNCH("attention_kernel");
  return MRNB_OK;
}
