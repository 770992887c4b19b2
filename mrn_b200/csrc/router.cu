// DM-Router + gate head: forward and the full parameter backward of the router-training stage.
//
// Reference (paths relative to /root/reference):
//   modules/dm_router.py:50-67   DM_Router.forward          :11-17 SpatialDomainGating   :26-33 ChannelDomainGating
//   modules/model.py:402-406     gate head (rearrange -> channel_route -> route -> softmax), :371-377 eval argmax
//   il_modules/mrn.py:342,360    taski_loss = CrossEntropy(gate, domain); loss = 15*CTC + taski_loss
//
// Math (SURVEY.md Appendix A.2/A.3), x in [B,I,T,D], rows m = (b,i,t), token n = i*T+t, channel k = i*D+c:
//   xn = LN_D(x); a1 = xn W1^T + b1; [u|v] = GELU(a1); vn = LN_D(v)
//   v2[b,n,:] = sum_m Ws[n,m] vn[b,m,:] + bs[n];  g1 = u*v2;  y = g1 W2^T + b2 + x
//   gn[b,k,:] = LN_T(y[b,k,:]);  g2[b,k,t] = sum_j Wc[k,j] gn[b,j,t] + bc[k];  y2 = y*g2;  out = y2 W3^T + b3 + x
//   s[b,t,j] = sum_k out[b,k,t] Wcr[j,k] + bcr[j];  r[b,j] = sum_t wr[t] s[b,t,j] + br;  gate = softmax(r)
// Every rearrange/permute of the reference is a two-level stride of the GEMM descriptors (no copies).
// Two GEMM engines.  fp32: the CUDA-core GEMM (gemm_f32.cu), the parity mode held to 1e-4.  bf16 with 32 <= T <= 64:
// tcgen05 (gemm_tc.cu for the forward row Linears, gemm_tc2.cu for the token / channel mixing and every backward GEMM)
// with bf16 operands and fp32 accumulation, CRNN's T = 63 padded to 64 frames.  The gate head (N = I) is an fp32 GEMV in
// both.
#include "common.cuh"
#include <stdlib.h>
#include "gemm_f32.h"
#include "gemm_tc2.h"
#include "gemm_tc.h"
#include "../../include/mrn_b200.h"

namespace {

constexpr int RD = 256;   // router channel width (opt.hidden_size)

enum { R_ROUTE_W, R_ROUTE_B, R_CR_W, R_CR_B, R_N_W, R_N_B, R_P1_W, R_P1_B, R_SN_W, R_SN_B, R_SP_W, R_SP_B,
       R_CN_W, R_CN_B, R_CP_W, R_CP_B, R_P2_W, R_P2_B, R_P3_W, R_P3_B };

// element count of each parameter slot, in R_* order
void router_sizes(int I, int T, int D, long* sz) {
  const long s[MRNB_ROUTER_NPARAMS] = {T, 1, (long)I * I * D, I, D, D, 2L * D * D, 2L * D, D, D,
                                       (long)I * T * I * T, (long)I * T, T, T, (long)I * D * I * D, (long)I * D,
                                       (long)D * D, D, (long)D * D, D};
  for (int k = 0; k < MRNB_ROUTER_NPARAMS; ++k) sz[k] = s[k];
}

long router_offsets(int I, int T, int D, long* off) {
  long sz[MRNB_ROUTER_NPARAMS];
  router_sizes(I, T, D, sz);
  // every slot starts on a 32-byte boundary (8 floats) so the bf16 shadow of a weight is a legal TMA base;
  // padding elements stay zero (zero gradient, untouched by Adam)
  long o = 0;
  for (int k = 0; k < MRNB_ROUTER_NPARAMS; ++k) { off[k] = o; o += (sz[k] + 7) / 8 * 8; }
  off[MRNB_ROUTER_NPARAMS] = o;
  return o;
}

// ---- row LayerNorm over D=256 with saved statistics (warp per row) ------------------------------
__global__ void __launch_bounds__(256)
ln_rows_fwd_kernel(const float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta,
                   float* __restrict__ y, __nv_bfloat16* __restrict__ y16, float* __restrict__ stats, long rows, float eps) {
  const long row = (long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  float v[8];
  const float* xr = x + row * RD;
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    const float4 t = *reinterpret_cast<const float4*>(xr + c * 128 + lane * 4);
    v[c * 4] = t.x; v[c * 4 + 1] = t.y; v[c * 4 + 2] = t.z; v[c * 4 + 3] = t.w;
  }
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < 8; ++j) s += v[j];
  const float mean = warp_sum(s) * (1.0f / RD);
  float q = 0.f;
#pragma unroll
  for (int j = 0; j < 8; ++j) { const float d = v[j] - mean; q = fmaf(d, d, q); }
  const float rstd = rsqrtf(warp_sum(q) * (1.0f / RD) + eps);
  if (lane == 0) { stats[row * 2] = mean; stats[row * 2 + 1] = rstd; }
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    const int idx = c * 128 + lane * 4;
    float4 o = make_float4((v[c * 4] - mean) * rstd, (v[c * 4 + 1] - mean) * rstd, (v[c * 4 + 2] - mean) * rstd, (v[c * 4 + 3] - mean) * rstd);
    if (gamma) {                                        // gamma == nullptr: plain x-hat (the affine is folded into the next Linear)
      const float4 g4 = __ldg(reinterpret_cast<const float4*>(gamma + idx)), b4 = __ldg(reinterpret_cast<const float4*>(beta + idx));
      o = make_float4(o.x * g4.x + b4.x, o.y * g4.y + b4.y, o.z * g4.z + b4.z, o.w * g4.w + b4.w);
    }
    if (y) *reinterpret_cast<float4*>(y + row * RD + idx) = o;
    if (y16) {
      __nv_bfloat162 h0 = __floats2bfloat162_rn(o.x, o.y), h1 = __floats2bfloat162_rn(o.z, o.w);
      *reinterpret_cast<uint2*>(y16 + row * RD + idx) = make_uint2(*reinterpret_cast<uint32_t*>(&h0), *reinterpret_cast<uint32_t*>(&h1));
    }
  }
}

// Tensor-core mode folds LayerNorm 1's affine into proj_1 (xn W1^T + b1 = xhat (W1 diag(gamma))^T + (b1 + W1 beta)):
//   forward:  W16[n,c] = bf16(W1[n,c] gamma[c]),  b1f[n] = b1[n] + sum_c W1[n,c] beta[c]            (block per output row n)
__global__ void __launch_bounds__(RD)
fold_ln_w1_kernel(const float* __restrict__ W1, const float* __restrict__ b1, const float* __restrict__ gamma,
                  const float* __restrict__ beta, __nv_bfloat16* __restrict__ W16, float* __restrict__ b1f) {
  __shared__ float sh[8];
  const int n = blockIdx.x, c = threadIdx.x;
  const float wv = W1[(long)n * RD + c];
  W16[(long)n * RD + c] = __float2bfloat16_rn(wv * gamma[c]);
  float s = warp_sum(wv * beta[c]);
  if ((c & 31) == 0) sh[c >> 5] = s;
  __syncthreads();
  if (c == 0) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += sh[k];
    b1f[n] = b1[n] + t;
  }
}
//   backward: with S = da1^T xhat [2D, D]:  dW1 = S diag(gamma) + db1 (x) beta,  dgamma[c] = sum_n W1[n,c] S[n,c],
//             dbeta[c] = sum_n db1[n] W1[n,c]   -- the M-row GEMM dxn = da1 W1 and the LayerNorm-backward pass over x are
//             not needed for the parameter gradients.   grid = row chunks of 32 output rows, thread = c
__global__ void __launch_bounds__(RD)
fold_ln_w1_bwd_kernel(const float* __restrict__ S, const float* __restrict__ db1, const float* __restrict__ W1,
                      const float* __restrict__ gamma, const float* __restrict__ beta, int nrows, float* __restrict__ dW1,
                      float* __restrict__ dgamma, float* __restrict__ dbeta) {
  const int c = threadIdx.x, n0 = blockIdx.x * 32;
  const float g = gamma[c], bt = beta[c];
  float ag = 0.f, ab = 0.f;
  for (int n = n0; n < n0 + 32 && n < nrows; ++n) {
    const float sv = S[(long)n * RD + c], wv = W1[(long)n * RD + c], d = db1[n];
    dW1[(long)n * RD + c] = fmaf(sv, g, d * bt);
    ag = fmaf(wv, sv, ag); ab = fmaf(d, wv, ab);
  }
  atomicAdd(dgamma + c, ag); atomicAdd(dbeta + c, ab);
}

__device__ __forceinline__ void store_bf16x4(__nv_bfloat16* p, float4 v) {
  __nv_bfloat162 h0 = __floats2bfloat162_rn(v.x, v.y), h1 = __floats2bfloat162_rn(v.z, v.w);
  *reinterpret_cast<uint2*>(p) = make_uint2(*reinterpret_cast<uint32_t*>(&h0), *reinterpret_cast<uint32_t*>(&h1));
}
// a1 [rows, 2D] -> u = GELU(a1[:, :D]) ; vn = LN_D(GELU(a1[:, D:])) + stats.   FAST: minimax-tanh GELU (tensor-core mode,
// the values end as bf16 operands; the backward recomputes with the same form)
template <bool FAST>
__global__ void __launch_bounds__(256)
gelu_ln_fwd_kernel(const float* __restrict__ a1, const float* __restrict__ gamma, const float* __restrict__ beta,
                   float* __restrict__ u, float* __restrict__ vn, __nv_bfloat16* __restrict__ vn16,
                   float* __restrict__ stats, long rows, float eps) {
  const long row = (long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* ar = a1 + row * 2 * RD;
  auto act = [](float x) { return FAST ? gelu_fast(x) : gelu_erf(x); };
  float v[8];
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    const float4 tu = *reinterpret_cast<const float4*>(ar + c * 128 + lane * 4);
    *reinterpret_cast<float4*>(u + row * RD + c * 128 + lane * 4) = make_float4(act(tu.x), act(tu.y), act(tu.z), act(tu.w));
    const float4 tv = *reinterpret_cast<const float4*>(ar + RD + c * 128 + lane * 4);
    v[c * 4] = act(tv.x); v[c * 4 + 1] = act(tv.y); v[c * 4 + 2] = act(tv.z); v[c * 4 + 3] = act(tv.w);
  }
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < 8; ++j) s += v[j];
  const float mean = warp_sum(s) * (1.0f / RD);
  float q = 0.f;
#pragma unroll
  for (int j = 0; j < 8; ++j) { const float d = v[j] - mean; q = fmaf(d, d, q); }
  const float rstd = rsqrtf(warp_sum(q) * (1.0f / RD) + eps);
  if (lane == 0) { stats[row * 2] = mean; stats[row * 2 + 1] = rstd; }
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    const int idx = c * 128 + lane * 4;
    const float4 g4 = __ldg(reinterpret_cast<const float4*>(gamma + idx)), b4 = __ldg(reinterpret_cast<const float4*>(beta + idx));
    const float4 o = make_float4((v[c * 4] - mean) * rstd * g4.x + b4.x, (v[c * 4 + 1] - mean) * rstd * g4.y + b4.y,
                                 (v[c * 4 + 2] - mean) * rstd * g4.z + b4.z, (v[c * 4 + 3] - mean) * rstd * g4.w + b4.w);
    if (vn) *reinterpret_cast<float4*>(vn + row * RD + idx) = o;
    if (vn16) store_bf16x4(vn16 + row * RD + idx, o);
  }
}

__global__ void mul_kernel(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ c,
                           __nv_bfloat16* __restrict__ c16, long n4) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n4) return;
  const float4 x = reinterpret_cast<const float4*>(a)[i], y = reinterpret_cast<const float4*>(b)[i];
  const float4 r = make_float4(x.x * y.x, x.y * y.y, x.z * y.z, x.w * y.w);
  if (c) reinterpret_cast<float4*>(c)[i] = r;
  if (c16) store_bf16x4(c16 + i * 4, r);
}
// c = a*b ; d = a*e      (shared first factor)
__global__ void mul2_kernel(const float* __restrict__ a, const float* __restrict__ b, const float* __restrict__ e,
                            float* __restrict__ c, float* __restrict__ d, __nv_bfloat16* __restrict__ d16, long n4) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n4) return;
  const float4 x = reinterpret_cast<const float4*>(a)[i], y = reinterpret_cast<const float4*>(b)[i],
               z = reinterpret_cast<const float4*>(e)[i];
  reinterpret_cast<float4*>(c)[i] = make_float4(x.x * y.x, x.y * y.y, x.z * y.z, x.w * y.w);
  const float4 r = make_float4(x.x * z.x, x.y * z.y, x.z * z.z, x.w * z.w);
  reinterpret_cast<float4*>(d)[i] = r;
  if (d16) store_bf16x4(d16 + i * 4, r);
}

// T == 64 (every SVTR / padded CRNN router): the 64 frames of a channel stay in registers -- one pass over y with all
// loads in flight instead of three dependent passes
__global__ void __launch_bounds__(RD)
lnT_fwd64_kernel(const float* __restrict__ y, const float* __restrict__ gamma /*[64]*/, const float* __restrict__ beta,
                 float* __restrict__ gn, __nv_bfloat16* __restrict__ gn16, float* __restrict__ stats /*[B*I, D, 2]*/, int Tv,
                 float eps) {
  const long bi = blockIdx.x;
  const int c = threadIdx.x;
  const float* yp = y + bi * 64 * RD + c;
  float v[64];
#pragma unroll
  for (int t = 0; t < 64; ++t) v[t] = yp[(long)t * RD];
  float s = 0.f;
#pragma unroll
  for (int t = 0; t < 64; ++t) s += t < Tv ? v[t] : 0.f;   // same summation order as the generic kernel
  const float mean = s / Tv;
  float q = 0.f;
#pragma unroll
  for (int t = 0; t < 64; ++t) { const float d = v[t] - mean; q = t < Tv ? fmaf(d, d, q) : q; }
  const float rstd = rsqrtf(q / Tv + eps);
  stats[(bi * RD + c) * 2] = mean; stats[(bi * RD + c) * 2 + 1] = rstd;
#pragma unroll
  for (int t = 0; t < 64; ++t) {
    const float o = t < Tv ? (v[t] - mean) * rstd * __ldg(gamma + t) + __ldg(beta + t) : 0.f;
    if (gn) gn[bi * 64 * RD + (long)t * RD + c] = o;
    if (gn16) gn16[bi * 64 * RD + (long)t * RD + c] = __float2bfloat16_rn(o);
  }
}

// LayerNorm over the patch axis T for every (b,i,c): block per (b,i), thread per c (ChannelDomainGating.norm)
__global__ void __launch_bounds__(RD)
lnT_fwd_kernel(const float* __restrict__ y, const float* __restrict__ gamma /*[T]*/, const float* __restrict__ beta,
               float* __restrict__ gn, __nv_bfloat16* __restrict__ gn16, float* __restrict__ stats /*[B*I, D, 2]*/, int T,
               int Tv, float eps) {
  // T = stored frames per (b,i); Tv <= T = valid frames (the tensor-core engine pads T = 63 to 64): padded frames
  // are excluded from the statistics and normalise to 0
  const long bi = blockIdx.x;
  const int c = threadIdx.x;
  const float* yp = y + bi * T * RD + c;
  float s = 0.f;
  for (int t = 0; t < Tv; ++t) s += yp[(long)t * RD];
  const float mean = s / Tv;
  float q = 0.f;
  for (int t = 0; t < Tv; ++t) { const float d = yp[(long)t * RD] - mean; q = fmaf(d, d, q); }
  const float rstd = rsqrtf(q / Tv + eps);
  stats[(bi * RD + c) * 2] = mean; stats[(bi * RD + c) * 2 + 1] = rstd;
  for (int t = 0; t < T; ++t) {
    const float o = t < Tv ? (yp[(long)t * RD] - mean) * rstd * gamma[t] + beta[t] : 0.f;
    if (gn) gn[bi * T * RD + (long)t * RD + c] = o;
    if (gn16) gn16[bi * T * RD + (long)t * RD + c] = __float2bfloat16_rn(o);
  }
}

// backward of lnT: dy += rstd*(dxh - mean(dxh) - xh*mean(dxh*xh)), dgamma[t] += sum dgn*xh, dbeta[t] += sum dgn
// block per (b,i), thread per channel c; the per-frame sums over c go through warp_reduce16 in groups of 8 frames
__global__ void __launch_bounds__(RD)
lnT_bwd_kernel(const float* __restrict__ y, const float* __restrict__ stats, const float* __restrict__ gamma,
               const float* __restrict__ dgn, float* __restrict__ dy /* accumulated */, __nv_bfloat16* __restrict__ dy16,
               float* __restrict__ dgamma, float* __restrict__ dbeta, int T, int Tv) {
  extern __shared__ float sh[];        // [T][2] block partials
  const long bi = blockIdx.x;
  const int c = threadIdx.x, lane = c & 31;
  for (int k = c; k < 2 * T; k += RD) sh[k] = 0.f;
  __syncthreads();
  const float mean = stats[(bi * RD + c) * 2], rstd = stats[(bi * RD + c) * 2 + 1];
  const float* yp = y + bi * T * RD + c;
  const float* dp = dgn + bi * T * RD + c;
  float m1 = 0.f, m2 = 0.f;
  for (int t0 = 0; t0 < Tv; t0 += 8) {
    float v[16];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int t = t0 + u;
      float xh = 0.f, d = 0.f;
      if (t < Tv) {
        xh = (yp[(long)t * RD] - mean) * rstd; d = dp[(long)t * RD];
        const float dxh = d * gamma[t];
        m1 += dxh; m2 = fmaf(dxh, xh, m2);
      }
      v[u] = d * xh; v[8 + u] = d;
    }
    const float tot = warp_reduce16(v, lane);
    if ((lane & 1) == 0) {
      const int idx = (lane >> 1) & 15;                    // 0..7: sum d*xh of frame t0+idx ; 8..15: sum d of frame t0+idx-8
      const int t = t0 + (idx & 7);
      if (t < Tv) atomicAdd(&sh[t * 2 + (idx >> 3)], tot);
    }
  }
  m1 /= Tv; m2 /= Tv;
  float* op = dy + bi * T * RD + c;
  for (int t = 0; t < T; ++t) {
    const float xh = (yp[(long)t * RD] - mean) * rstd;
    const float dxh = dp[(long)t * RD] * gamma[t];
    const float o = op[(long)t * RD] + (t < Tv ? rstd * (dxh - m1 - xh * m2) : 0.f);
    op[(long)t * RD] = o;
    if (dy16) dy16[bi * T * RD + (long)t * RD + c] = __float2bfloat16_rn(o);
  }
  __syncthreads();
  for (int k = c; k < T; k += RD) { atomicAdd(dgamma + k, sh[k * 2]); atomicAdd(dbeta + k, sh[k * 2 + 1]); }
}

// Row-LN backward (D=256, warp per row).  xin is the LN input (or its pre-GELU activation when GELU_IN):
//   dxin = LNbwd(dyn) [* GELU'(pre)]  (+ add1 + add2);  dgamma/dbeta accumulated with block partials + atomics.
template <bool GELU_IN, bool FAST = false>
__global__ void __launch_bounds__(256)
ln_rows_bwd_kernel(const float* __restrict__ xin, long ldx, const float* __restrict__ stats,
                   const float* __restrict__ gamma, const float* __restrict__ dyn, float* __restrict__ dxin,
                   __nv_bfloat16* __restrict__ dxin16, long lddx, const float* __restrict__ add1, const float* __restrict__ add2, float* __restrict__ dgamma,
                   float* __restrict__ dbeta, long rows, float* __restrict__ dcol = nullptr) {
  // dcol (optional): column sums of the produced gradient dxin (the bias gradient of the Linear that made xin)
  __shared__ float sg[RD], sb[RD], sc[RD];
  for (int k = threadIdx.x; k < RD; k += 256) { sg[k] = 0.f; sb[k] = 0.f; sc[k] = 0.f; }
  __syncthreads();
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  float ag[8], ab[8], ac[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { ag[j] = 0.f; ab[j] = 0.f; ac[j] = 0.f; }
  for (long row = (long)blockIdx.x * 8 + w; row < rows; row += (long)gridDim.x * 8) {
    const float mean = stats[row * 2], rstd = stats[row * 2 + 1];
    float xh[8], dxh[8], pre[8];
    float m1 = 0.f, m2 = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int idx = (j / 4) * 128 + lane * 4 + (j % 4);
      pre[j] = xin[row * ldx + idx];
      const float xv = GELU_IN ? (FAST ? gelu_fast(pre[j]) : gelu_erf(pre[j])) : pre[j];
      xh[j] = (xv - mean) * rstd;
      const float d = dyn[row * RD + idx];
      dxh[j] = gamma ? d * gamma[idx] : d;
      ag[j] = fmaf(d, xh[j], ag[j]); ab[j] += d;
      m1 += dxh[j]; m2 = fmaf(dxh[j], xh[j], m2);
    }
    m1 = warp_sum(m1) * (1.0f / RD); m2 = warp_sum(m2) * (1.0f / RD);
    if (dxin || dxin16) {
      float g[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int idx = (j / 4) * 128 + lane * 4 + (j % 4);
        g[j] = rstd * (dxh[j] - m1 - xh[j] * m2);
        if (GELU_IN) g[j] *= FAST ? gelu_fast_grad(pre[j]) : gelu_erf_grad(pre[j]);
        if (add1) g[j] += add1[row * RD + idx];
        if (add2) g[j] += add2[row * RD + idx];
        ac[j] += g[j];
      }
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        const long o = row * lddx + c * 128 + lane * 4;
        if (dxin) *reinterpret_cast<float4*>(dxin + o) = make_float4(g[c * 4], g[c * 4 + 1], g[c * 4 + 2], g[c * 4 + 3]);
        if (dxin16) store_bf16x4(dxin16 + o, make_float4(g[c * 4], g[c * 4 + 1], g[c * 4 + 2], g[c * 4 + 3]));
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int idx = (j / 4) * 128 + lane * 4 + (j % 4);
    if (dgamma) { atomicAdd(&sg[idx], ag[j]); atomicAdd(&sb[idx], ab[j]); }
    if (dcol) atomicAdd(&sc[idx], ac[j]);
  }
  __syncthreads();
  for (int k = threadIdx.x; k < RD; k += 256) {
    if (dgamma) { atomicAdd(dgamma + k, sg[k]); atomicAdd(dbeta + k, sb[k]); }
    if (dcol) atomicAdd(dcol + k, sc[k]);
  }
}

// da1[:, :D] = du * GELU'(a1[:, :D])
__global__ void gelu_bwd_kernel(const float* __restrict__ a1, const float* __restrict__ du, float* __restrict__ da1,
                                __nv_bfloat16* __restrict__ da1_16, long rows) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * RD) return;
  const long row = i / RD; const int c = (int)(i % RD);
  const float o = du[i] * gelu_erf_grad(a1[row * 2 * RD + c]);
  da1[row * 2 * RD + c] = o;
  if (da1_16) da1_16[row * 2 * RD + c] = __float2bfloat16_rn(o);
}

// dout[b,i,t,c] = sum_j ds[b,t,j] * Wcr[j,(i,c)]   (gate-head input gradient, K = I is tiny) + bf16 copy
__global__ void dout_kernel(const float* __restrict__ ds, const float* __restrict__ Wcr, int I, int T, long total4,
                            float* __restrict__ dout, __nv_bfloat16* __restrict__ dout16) {
  const long i4 = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i4 >= total4) return;
  const long e = i4 * 4;
  const int c = (int)(e % RD);
  const int t = (int)((e / RD) % T);
  const int i = (int)((e / ((long)RD * T)) % I);
  const long b = e / ((long)RD * T * I);
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int j = 0; j < I; ++j) {
    const float d = ds[(b * T + t) * I + j];
    const float4 w = *reinterpret_cast<const float4*>(Wcr + (long)j * I * RD + (long)i * RD + c);
    acc.x = fmaf(d, w.x, acc.x); acc.y = fmaf(d, w.y, acc.y); acc.z = fmaf(d, w.z, acc.z); acc.w = fmaf(d, w.w, acc.w);
  }
  *reinterpret_cast<float4*>(dout + e) = acc;
  if (dout16) store_bf16x4(dout16 + e, acc);
}

__global__ void cast16_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ y, long n) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) y[i] = __float2bfloat16_rn(x[i]);
}

// out[n] (+)= sum_m X(m, n) with two-level axes; grid (cdiv(N,32), msplit)
__global__ void colsum_kernel(const float* __restrict__ X, MrnbAxis am, MrnbAxis an, int M, int N, float* __restrict__ out) {
  __shared__ float sh[8][33];
  const int n = blockIdx.x * 32 + (threadIdx.x & 31);
  const int ty = threadIdx.x >> 5;
  const int per = (M + gridDim.y - 1) / gridDim.y;
  const int m0 = blockIdx.y * per, m1 = min(M, m0 + per);
  float s = 0.f;
  if (n < N) {
    const long on = (long)(n / an.inner) * an.so + (long)(n % an.inner) * an.si;
    for (int m = m0 + ty; m < m1; m += 8) s += X[(long)(m / am.inner) * am.so + (long)(m % am.inner) * am.si + on];
  }
  sh[ty][threadIdx.x & 31] = s;
  __syncthreads();
  if (ty == 0 && n < N) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += sh[k][threadIdx.x];
    atomicAdd(out + n, t);
  }
}

// gate head GEMV (N = I <= 8): s[(b,t), j] = sum_(i,c) out[b,i,t,c] * Wcr[j,(i,c)] + bcr[j].  One warp per (b,t) row;
// `out` is streamed exactly once (modules/model.py:402-403: rearrange 'b h w c -> b w (h c)' + channel_route).
template <int I>
__global__ void __launch_bounds__(256)
gate_head_fwd_kernel(const float* __restrict__ out, const float* __restrict__ Wcr, const float* __restrict__ bcr, int B,
                     int T, float* __restrict__ s) {
  // four consecutive rows per warp: every weight fragment (L1-resident, 36 KiB in all) is loaded once per four rows --
  // with one row per warp the kernel was bound by the 72 weight loads per lane and row, not by the stream of `out`
  constexpr int R = 4;
  const long row0 = ((long)blockIdx.x * 8 + (threadIdx.x >> 5)) * R;      // row = b*T + t
  const int lane = threadIdx.x & 31;
  const long nrows = (long)B * T;
  if (row0 >= nrows) return;
  float acc[R][I];
#pragma unroll
  for (int r = 0; r < R; ++r)
#pragma unroll
    for (int j = 0; j < I; ++j) acc[r][j] = 0.f;
#pragma unroll
  for (int i = 0; i < I; ++i) {
    float4 z0[R], z1[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const long row = row0 + r < nrows ? row0 + r : nrows - 1;
      const long b = row / T, t = row % T;
      const float* zp = out + ((b * I + i) * T + t) * RD + lane * 8;
      z0[r] = *reinterpret_cast<const float4*>(zp); z1[r] = *reinterpret_cast<const float4*>(zp + 4);
    }
#pragma unroll
    for (int j = 0; j < I; ++j) {
      const float* wp = Wcr + (long)j * I * RD + i * RD + lane * 8;
      const float4 w0 = __ldg(reinterpret_cast<const float4*>(wp)), w1 = __ldg(reinterpret_cast<const float4*>(wp + 4));
#pragma unroll
      for (int r = 0; r < R; ++r)
        acc[r][j] += z0[r].x * w0.x + z0[r].y * w0.y + z0[r].z * w0.z + z0[r].w * w0.w + z1[r].x * w1.x + z1[r].y * w1.y + z1[r].z * w1.z + z1[r].w * w1.w;
    }
  }
#pragma unroll
  for (int r = 0; r < R; ++r)
#pragma unroll
    for (int j = 0; j < I; ++j) {
      const float v = warp_sum(acc[r][j]);
      if (lane == 0 && row0 + r < nrows) s[(row0 + r) * I + j] = v + bcr[j];
    }
}

// dWcr[j,(i,c)] += sum_(b,t) ds[(b,t),j] * out[b,i,t,c].  grid (row chunks of 128, I); thread = channel c.
template <int I>
__global__ void __launch_bounds__(RD)
gate_head_dw_kernel(const float* __restrict__ ds, const float* __restrict__ out, int B, int T, float* __restrict__ dW) {
  __shared__ float sds[128 * I];
  const int i = blockIdx.y, c = threadIdx.x;
  const long row0 = (long)blockIdx.x * 128, nrows = (long)B * T;
  for (int k = threadIdx.x; k < 128 * I; k += RD) sds[k] = (row0 + k / I < nrows) ? ds[row0 * I + k] : 0.f;
  __syncthreads();
  float acc[I];
#pragma unroll
  for (int j = 0; j < I; ++j) acc[j] = 0.f;
  for (int r = 0; r < 128; ++r) {
    const long row = row0 + r;
    if (row >= nrows) break;
    const long b = row / T, t = row % T;
    const float z = out[((b * I + i) * T + t) * RD + c];
#pragma unroll
    for (int j = 0; j < I; ++j) acc[j] = fmaf(sds[r * I + j], z, acc[j]);
  }
#pragma unroll
  for (int j = 0; j < I; ++j) atomicAdd(dW + (long)j * I * RD + i * RD + c, acc[j]);
}

template <int I>
int launch_gate_head(const float* out, const float* Wcr, const float* bcr, int B, int T, float* s, cudaStream_t st) {
  gate_head_fwd_kernel<I><<<cdiv((long)B * T, 32), 256, 0, st>>>(out, Wcr, bcr, B, T, s);
  MRNB_CHECK_LAUNCH("gate_head_fwd_kernel");
  return MRNB_OK;
}
template <int I>
int launch_gate_head_dw(const float* ds, const float* out, int B, int T, float* dW, cudaStream_t st) {
  gate_head_dw_kernel<I><<<dim3(cdiv((long)B * T, 128), I), RD, 0, st>>>(ds, out, B, T, dW);
  MRNB_CHECK_LAUNCH("gate_head_dw_kernel");
  return MRNB_OK;
}
#define MRNB_DISPATCH_I(fn, I_, ...)                                                                   \
  switch (I_) {                                                                                         \
    case 1: MRNB_TRY(fn<1>(__VA_ARGS__)); break; case 2: MRNB_TRY(fn<2>(__VA_ARGS__)); break;           \
    case 3: MRNB_TRY(fn<3>(__VA_ARGS__)); break; case 4: MRNB_TRY(fn<4>(__VA_ARGS__)); break;           \
    case 5: MRNB_TRY(fn<5>(__VA_ARGS__)); break; case 6: MRNB_TRY(fn<6>(__VA_ARGS__)); break;           \
    case 7: MRNB_TRY(fn<7>(__VA_ARGS__)); break; default: MRNB_TRY(fn<8>(__VA_ARGS__)); break;          \
  }

// gate head finish: r[b,j] = sum_t wr[t] s[b,t,j] + br ; gate = softmax(r) ; index = first argmax
__global__ void __launch_bounds__(256)
gate_finish_kernel(const float* __restrict__ s, const float* __restrict__ wr, const float* __restrict__ br,
                   int B, int T, int I, float* __restrict__ r, float* __restrict__ gate, int* __restrict__ index) {
  // one warp per sample: lanes stride the (t, j) pairs of s[b] (contiguous), then a shuffle reduction per expert
  const int b = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (b >= B) return;
  float part[MRNB_MAX_EXPERTS];
#pragma unroll
  for (int j = 0; j < MRNB_MAX_EXPERTS; ++j) part[j] = 0.f;
  const float* sb = s + (long)b * T * I;
  for (int t = lane; t < T; t += 32) {
    const float w = wr[t];
#pragma unroll
    for (int j = 0; j < MRNB_MAX_EXPERTS; ++j)
      if (j < I) part[j] = fmaf(w, sb[t * I + j], part[j]);
  }
  float rr[MRNB_MAX_EXPERTS];
  float mx = -INFINITY; int am = 0;
#pragma unroll
  for (int j = 0; j < MRNB_MAX_EXPERTS; ++j) {
    if (j < I) {
      const float a = warp_sum(part[j]) + br[0];
      rr[j] = a;
      if (a > mx) { mx = a; am = j; }
    }
  }
  if (lane != 0) return;
  float sum = 0.f;
#pragma unroll
  for (int j = 0; j < MRNB_MAX_EXPERTS; ++j) if (j < I) sum += expf(rr[j] - mx);
#pragma unroll
  for (int j = 0; j < MRNB_MAX_EXPERTS; ++j) {
    if (j < I) {
      if (r) r[b * I + j] = rr[j];
      if (gate) gate[b * I + j] = expf(rr[j] - mx) / sum;
    }
  }
  if (index) index[b] = am;
}

// dL/dr from dL/dgate (CTC part) + CrossEntropy(gate, domain) applied to the softmaxed gate; also the CE loss.
// domain == NULL: dgate_ctc is the whole dL/dgate (no CE term, ce_loss untouched).
__global__ void gate_bwd_kernel(const float* __restrict__ gate, const float* __restrict__ dgate_ctc,
                                const long long* __restrict__ domain, int B, int I, float* __restrict__ dr,
                                float* __restrict__ ce_loss) {
  __shared__ double sh[8];
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  double lossb = 0.0;
  if (b < B && !domain) {
    float g[MRNB_MAX_EXPERTS];
    float dot = 0.f;
    for (int j = 0; j < I; ++j) { g[j] = gate[b * I + j]; dot = fmaf(g[j], dgate_ctc[b * I + j], dot); }
    for (int j = 0; j < I; ++j) dr[b * I + j] = g[j] * (dgate_ctc[b * I + j] - dot);
  } else if (b < B) {
    float g[MRNB_MAX_EXPERTS], dg[MRNB_MAX_EXPERTS];
    float mx = -INFINITY;
    for (int j = 0; j < I; ++j) { g[j] = gate[b * I + j]; mx = fmaxf(mx, g[j]); }
    float sum = 0.f;
    for (int j = 0; j < I; ++j) sum += expf(g[j] - mx);
    const int dom = (int)domain[b];
    float dot = 0.f;
    for (int j = 0; j < I; ++j) {
      const float sm = expf(g[j] - mx) / sum;
      dg[j] = (dgate_ctc ? dgate_ctc[b * I + j] : 0.f) + (sm - (j == dom ? 1.f : 0.f)) / (float)B;
      dot = fmaf(g[j], dg[j], dot);
    }
    lossb = -(double)(g[dom] - mx - logf(sum)) / (double)B;
    for (int j = 0; j < I; ++j) dr[b * I + j] = g[j] * (dg[j] - dot);
  }
  lossb = warp_sum_d(lossb);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = lossb;
  __syncthreads();
  if (threadIdx.x == 0 && domain) {
    double t = 0.0;
    for (int k = 0; k < (int)(blockDim.x >> 5); ++k) t += sh[k];
    atomicAdd(ce_loss, (float)t);
  }
}

// ds[b,t,j] = dr[b,j]*wr[t];  dwr[t] = sum_{b,j} dr[b,j] s[b,t,j];  dbr = sum dr      (block per t)
__global__ void route_bwd_kernel(const float* __restrict__ dr, const float* __restrict__ s, const float* __restrict__ wr,
                                 int B, int T, int I, float* __restrict__ ds, float* __restrict__ dwr, float* __restrict__ dbr) {
  __shared__ float sh[2][8];
  const int t = blockIdx.x;
  float a = 0.f, c = 0.f;
  const float w = wr[t];
  for (int k = threadIdx.x; k < B * I; k += blockDim.x) {
    const int b = k / I, j = k % I;
    const float d = dr[k];
    ds[((long)b * T + t) * I + j] = d * w;
    a = fmaf(d, s[((long)b * T + t) * I + j], a);
    c += d;
  }
  a = warp_sum(a); c = warp_sum(c);
  if ((threadIdx.x & 31) == 0) { sh[0][threadIdx.x >> 5] = a; sh[1][threadIdx.x >> 5] = c; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float ta = 0.f, tc = 0.f;
    for (int k = 0; k < (int)(blockDim.x >> 5); ++k) { ta += sh[0][k]; tc += sh[1][k]; }
    dwr[t] = ta;
    if (t == 0) dbr[0] = tc;
  }
}

inline size_t al(size_t v) { return (v + 255) / 256 * 256; }

typedef __nv_bfloat16 bf16;

struct RouterWs {
  // forward (kept for backward)
  float *stats1, *xn, *a1, *u, *vn, *stats2, *v2, *g1, *y, *statsT, *gn, *g2, *y2, *out, *s;
  // backward temporaries
  float *dr, *ds, *dout, *dy2, *dy, *dg2, *dgn, *dg1, *du, *dv2, *dvn, *da1, *dxn;
  float *gp, *ow; bf16 *gq16, *y2w16;   // gate-head driven backward: [B*I, D] each
  float *b1f, *S1;                      // folded proj_1 bias [2D]; S = da1^T xhat [2D, D]
  // bf16 shadows (tensor-core mode): GEMM operands only
  bf16 *w16, *xn16, *vn16, *g116, *gn16, *y216, *dout16, *dg216, *dy16, *dv216, *da116;
  size_t bytes;
};

RouterWs carve(char* base, int B, int I, int T, int D, bool bwd) {
  RouterWs w{};
  size_t o = 0;
  const size_t M = (size_t)B * I * T, MD = M * D;
  long off[MRNB_ROUTER_NPARAMS + 1];
  const size_t nparam = (size_t)router_offsets(I, T, D, off);
  auto take = [&](size_t n) { float* p = base ? (float*)(base + o) : nullptr; o = al(o + n * 4); return p; };
  auto take16 = [&](size_t n) { bf16* p = base ? (bf16*)(base + o) : nullptr; o = al(o + n * 2); return p; };
  w.stats1 = take(M * 2); w.xn = take(MD); w.a1 = take(MD * 2); w.u = take(MD); w.vn = take(MD); w.stats2 = take(M * 2);
  w.v2 = take(MD); w.g1 = take(MD); w.y = take(MD); w.statsT = take((size_t)B * I * D * 2); w.gn = take(MD);
  w.g2 = take(MD); w.y2 = take(MD); w.out = take(MD); w.s = take((size_t)B * T * I);
  w.w16 = take16(nparam); w.xn16 = take16(MD); w.vn16 = take16(MD); w.g116 = take16(MD); w.gn16 = take16(MD);
  w.y216 = take16(MD); w.b1f = take((size_t)2 * D);
  if (bwd) {
    w.dr = take((size_t)B * I); w.ds = take((size_t)B * T * I); w.dout = take(MD); w.dy2 = take(MD); w.dy = take(MD);
    w.dg2 = take(MD); w.dgn = take(MD); w.dg1 = take(MD); w.du = take(MD); w.dv2 = take(MD); w.dvn = take(MD);
    w.da1 = take(MD * 2); w.dxn = take(MD);
    w.dout16 = take16(MD); w.dg216 = take16(MD); w.dy16 = take16(MD); w.dv216 = take16(MD); w.da116 = take16(MD * 2);
    w.S1 = take((size_t)2 * D * D);
    const size_t rows_p = ((size_t)B * I + 127) / 128 * 128;   // the collapsed GEMMs run on B*I rows padded to a row tile
    w.gp = take(rows_p * D); w.ow = take((size_t)B * I * D); w.gq16 = take16(rows_p * D); w.y2w16 = take16(rows_p * D);
  }
  w.bytes = o + 256;
  return w;
}

#define LAUNCH_EW(kernel, n, ...)                                      \
  do {                                                                 \
    kernel<<<cdiv((n), 256), 256, 0, st>>>(__VA_ARGS__);               \
    MRNB_CHECK_LAUNCH(#kernel);                                        \
  } while (0)
// grid of the grid-stride row kernels (ln_rows_bwd_kernel, dg1_fused_kernel): 8 warps per block, 16 rows per warp
inline int rows16_grid(long rows) { const int g = (int)((rows + 8 * 16 - 1) / (8 * 16)); return g > 0 ? g : 1; }

// column sums for n-contiguous layouts: 64 x float4 columns per block, 4 row lanes, 4 rows in flight per thread
__global__ void __launch_bounds__(256)
colsum_vec_kernel(const float* __restrict__ X, MrnbAxis am, MrnbAxis an, int M, int N, float* __restrict__ out) {
  __shared__ float4 sh[4][64];
  const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;
  const int n = (blockIdx.x * 64 + tx) * 4;
  const int per = (M + gridDim.y - 1) / gridDim.y;
  const int m0 = blockIdx.y * per, m1 = min(M, m0 + per);
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  if (n < N) {
    const float* base = X + (long)(n / an.inner) * an.so + (long)(n % an.inner);
    int m = m0 + ty;
    for (; m + 12 < m1; m += 16) {
      float4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int mm = m + 4 * u;
        v[u] = *reinterpret_cast<const float4*>(base + (long)(mm / am.inner) * am.so + (long)(mm % am.inner) * am.si);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) { s.x += v[u].x; s.y += v[u].y; s.z += v[u].z; s.w += v[u].w; }
    }
    for (; m < m1; m += 4) {
      const float4 v = *reinterpret_cast<const float4*>(base + (long)(m / am.inner) * am.so + (long)(m % am.inner) * am.si);
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
  }
  sh[ty][tx] = s;
  __syncthreads();
  if (ty == 0 && n < N) {
    float4 t = sh[0][tx];
#pragma unroll
    for (int k = 1; k < 4; ++k) { t.x += sh[k][tx].x; t.y += sh[k][tx].y; t.z += sh[k][tx].z; t.w += sh[k][tx].w; }
    atomicAdd(out + n, t.x); atomicAdd(out + n + 1, t.y); atomicAdd(out + n + 2, t.z); atomicAdd(out + n + 3, t.w);
  }
}

// out[r % period] += sum_c X[r, 0..255]  for contiguous rows of 256 (token sums over (b, c)): one warp per (n, b-chunk)
__global__ void __launch_bounds__(256)
rowsum256_kernel(const float* __restrict__ X, int period, int reps, float* __restrict__ out) {
  const int n = blockIdx.x, lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int per = (reps + gridDim.y * 8 - 1) / (gridDim.y * 8);
  const int b0 = (blockIdx.y * 8 + w) * per, b1 = min(reps, b0 + per);
  float s = 0.f;
  for (int b = b0; b < b1; ++b) {
    const float* row = X + ((long)b * period + n) * RD;
    const float4 u = *reinterpret_cast<const float4*>(row + lane * 4), v = *reinterpret_cast<const float4*>(row + 128 + lane * 4);
    s += (u.x + u.y) + (u.z + u.w) + (v.x + v.y) + (v.z + v.w);
  }
  s = warp_sum(s);
  if (lane == 0 && b1 > b0) atomicAdd(out + n, s);
}

int colsum(const float* X, MrnbAxis am, MrnbAxis an, int M, int N, float* out, cudaStream_t st) {
  int msplit = M / 512; if (msplit < 1) msplit = 1; if (msplit > 64) msplit = 64;
  MrnbProfScope prof(MRNB_PROF_ROUTER_EW, st);
  const bool vec = an.si == 1 && (an.inner % 4 == 0) && (N % 4 == 0) && (an.so % 4 == 0) && (am.si % 4 == 0) && (am.so % 4 == 0) &&
                   ((reinterpret_cast<uintptr_t>(X) & 15) == 0);
  if (vec) {
    const int gx = cdiv(N, 256);
    int gy = 1184 / gx; if (gy < 1) gy = 1; if (gy > M / 16) gy = M / 16 > 0 ? M / 16 : 1;      // ~8 blocks per SM
    colsum_vec_kernel<<<dim3(gx, gy), 256, 0, st>>>(X, am, an, M, N, out);
    MRNB_CHECK_LAUNCH("colsum_vec_kernel");
    return MRNB_OK;
  }
  colsum_kernel<<<dim3(cdiv(N, 32), msplit), 256, 0, st>>>(X, am, an, M, N, out);
  MRNB_CHECK_LAUNCH("colsum_kernel");
  return MRNB_OK;
}

// =====================================================================================================================
// Gate-head driven backward of the training step (tensor-core mode).
//
// The only consumer of the router output in training is the gate head (modules/model.py:402-405): s = out Wcr^T + bcr over
// k = (i,c), then r = s^T wr + br over the frames.  Its input gradient is therefore RANK ONE along the frame axis:
//     dout[b,i,t,c] = wr[t] * q[b,(i,c)],    q[b,:] = dr[b,:] Wcr                                     (q: [B, I*D])
// and every contraction of the last Linear (out = y2 W3^T + b3 + x) collapses from M = B*I*T rows to B*I rows:
//     dy2[b,i,t,:] = wr[t] * p[b,i,:],  p = q W3          dW3 = q^T y2w,  y2w[b,i,:] = sum_t wr[t] y2[b,i,t,:]
//     db3 = (sum_t wr[t]) * sum_(b,i) q[b,i,:]             dWcr[j,(i,c)] = sum_b dr[b,j] ow[b,i,c],  ow = sum_t wr[t] out
//     dbcr[j] = (sum_t wr[t]) * sum_b dr[b,j]
// so dout / dy2 are never materialised, two M-row GEMMs and four passes over [M, D] tensors disappear, and the frame-
// weighted sums ow / y2w ride in the pass that produces dg2 = dy2 * y.
// =====================================================================================================================

// q[b,i,:] = sum_j dr[b,j] Wcr[j,(i,:)] (fp32 + bf16 GEMM operand) ;  db3 += wsum * q ;  dbcr += wsum * dr   (block per (b,i))
__global__ void __launch_bounds__(RD)
gate_q_kernel(const float* __restrict__ dr, const float* __restrict__ Wcr, const float* __restrict__ wr, int I, int T,
              __nv_bfloat16* __restrict__ q16, float* __restrict__ db3, float* __restrict__ dbcr) {
  __shared__ float swsum;
  const int bi = blockIdx.x, b = bi / I, i = bi % I, c = threadIdx.x;
  if (threadIdx.x < 32) {
    float s = 0.f;
    for (int t = threadIdx.x; t < T; t += 32) s += wr[t];
    s = warp_sum(s);
    if (threadIdx.x == 0) swsum = s;
  }
  float acc = 0.f;
  for (int j = 0; j < I; ++j) acc = fmaf(dr[b * I + j], Wcr[(long)j * I * RD + (long)i * RD + c], acc);
  q16[(long)bi * RD + c] = __float2bfloat16_rn(acc);
  __syncthreads();
  const float wsum = swsum;
  atomicAdd(db3 + c, acc * wsum);
  if (i == 0 && c < I) atomicAdd(dbcr + c, dr[b * I + c] * wsum);
}

// One pass over out / y2 / y per (b,i):  ow = sum_t wr[t] out,  y2w = sum_t wr[t] y2 (bf16 GEMM operand),  dg2 = wr[t] p y (bf16),
// dbc[(i,c)] += sum_t dg2.   128 threads x 2 channels.
__global__ void __launch_bounds__(128)
tsum_dg2_kernel(const float* __restrict__ out, const __nv_bfloat16* __restrict__ y216, const float* __restrict__ y,
                const float* __restrict__ p, const float* __restrict__ wr, int I, int T, float* __restrict__ ow,
                __nv_bfloat16* __restrict__ y2w16, __nv_bfloat16* __restrict__ dg216, float* __restrict__ dbc) {
  __shared__ float swr[128];
  const long bi = blockIdx.x;
  const int i = (int)(bi % I), c = threadIdx.x * 2;
  if (threadIdx.x < T) swr[threadIdx.x] = wr[threadIdx.x];
  __syncthreads();
  const float2 pp = *reinterpret_cast<const float2*>(p + bi * RD + c);
  float2 aow = make_float2(0.f, 0.f), ay = make_float2(0.f, 0.f), ad = make_float2(0.f, 0.f);
  const long base = bi * T * RD + c;
#pragma unroll 4
  for (int t = 0; t < T; ++t) {
    const float w = swr[t];
    const long o = base + (long)t * RD;
    const float2 ov = *reinterpret_cast<const float2*>(out + o);
    const float2 hv = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(y216 + o));
    const float2 yv = *reinterpret_cast<const float2*>(y + o);
    aow.x = fmaf(w, ov.x, aow.x); aow.y = fmaf(w, ov.y, aow.y);
    ay.x = fmaf(w, hv.x, ay.x); ay.y = fmaf(w, hv.y, ay.y);
    const float dx = w * pp.x * yv.x, dy = w * pp.y * yv.y;
    ad.x += dx; ad.y += dy;
    *reinterpret_cast<__nv_bfloat162*>(dg216 + o) = __floats2bfloat162_rn(dx, dy);
  }
  *reinterpret_cast<float2*>(ow + bi * RD + c) = aow;
  *reinterpret_cast<__nv_bfloat162*>(y2w16 + bi * RD + c) = __floats2bfloat162_rn(ay.x, ay.y);
  atomicAdd(dbc + (long)i * RD + c, ad.x);
  atomicAdd(dbc + (long)i * RD + c + 1, ad.y);
}

// dWcr[j, k] += sum_b dr[b,j] ow[b,k]   (k = (i,c) over I*D; grid (cdiv(ID,256), b-chunks))
__global__ void __launch_bounds__(256)
gate_dwcr_kernel(const float* __restrict__ dr, const float* __restrict__ ow, int B, int I, long ID, float* __restrict__ dW) {
  const long k = (long)blockIdx.x * 256 + threadIdx.x;
  const int per = (B + gridDim.y - 1) / gridDim.y;
  const int b0 = blockIdx.y * per, b1 = min(B, b0 + per);
  if (k >= ID) return;
  float acc[MRNB_MAX_EXPERTS];
#pragma unroll
  for (int j = 0; j < MRNB_MAX_EXPERTS; ++j) acc[j] = 0.f;
  for (int b = b0; b < b1; ++b) {
    const float z = ow[(long)b * ID + k];
#pragma unroll
    for (int j = 0; j < MRNB_MAX_EXPERTS; ++j)
      if (j < I) acc[j] = fmaf(__ldg(dr + b * I + j), z, acc[j]);
  }
#pragma unroll
  for (int j = 0; j < MRNB_MAX_EXPERTS; ++j)
    if (j < I) atomicAdd(dW + (long)j * ID + k, acc[j]);
}

// Backward of gn = LN_T(y) with the upstream gradient of y = y * g2 recomputed in place (dy_a = wr[t] p g2):
//   dy = wr[t] p g2 + rstd (dxh - mean_t dxh - xh mean_t(dxh xh)),  dxh = dgn gamma[t]
//   -> dy16 (bf16 GEMM operand);  dgamma[t] += sum d xh;  dbeta[t] += sum d;  db2[c] += sum_(b,i,t) dy   (bias of W2's Linear)
// block per (b,i), 128 threads x 2 channels, two passes over the 64 frames (the second one hits L2).
__global__ void __launch_bounds__(128)
lnT_bwd2_kernel(const float* __restrict__ y, const float* __restrict__ stats, const float* __restrict__ gamma,
                const float* __restrict__ dgn, const float* __restrict__ g2, const float* __restrict__ p,
                const float* __restrict__ wr, __nv_bfloat16* __restrict__ dy16, float* __restrict__ dgamma,
                float* __restrict__ dbeta, float* __restrict__ db2, int T, int Tv) {
  __shared__ float sh[128 * 2];        // [T][2] block partials
  __shared__ float sgam[128], swr[128];
  const long bi = blockIdx.x;
  const int c = threadIdx.x * 2, lane = threadIdx.x & 31;
  for (int k = threadIdx.x; k < 2 * T; k += 128) sh[k] = 0.f;
  if (threadIdx.x < T) { sgam[threadIdx.x] = gamma[threadIdx.x]; swr[threadIdx.x] = wr[threadIdx.x]; }
  __syncthreads();
  const float4 st4 = *reinterpret_cast<const float4*>(stats + (bi * RD + c) * 2);     // mean0, rstd0, mean1, rstd1
  const float2 pp = *reinterpret_cast<const float2*>(p + bi * RD + c);
  const long base = bi * T * RD + c;
  float m1x = 0.f, m2x = 0.f, m1y = 0.f, m2y = 0.f;
  for (int t0 = 0; t0 < Tv; t0 += 8) {
    float v[16];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int t = t0 + u;
      float a = 0.f, d = 0.f;
      if (t < Tv) {
        const float2 yv = *reinterpret_cast<const float2*>(y + base + (long)t * RD);
        const float2 dv = *reinterpret_cast<const float2*>(dgn + base + (long)t * RD);
        const float xh0 = (yv.x - st4.x) * st4.y, xh1 = (yv.y - st4.z) * st4.w;
        const float g = sgam[t];
        const float dx0 = dv.x * g, dx1 = dv.y * g;
        m1x += dx0; m2x = fmaf(dx0, xh0, m2x); m1y += dx1; m2y = fmaf(dx1, xh1, m2y);
        a = fmaf(dv.x, xh0, dv.y * xh1); d = dv.x + dv.y;
      }
      v[u] = a; v[8 + u] = d;
    }
    const float tot = warp_reduce16(v, lane);
    if ((lane & 1) == 0) {
      const int idx = (lane >> 1) & 15;                    // 0..7: sum d*xh of frame t0+idx ; 8..15: sum d of frame t0+idx-8
      const int t = t0 + (idx & 7);
      if (t < Tv) atomicAdd(&sh[t * 2 + (idx >> 3)], tot);
    }
  }
  const float inv = 1.0f / Tv;
  m1x *= inv; m2x *= inv; m1y *= inv; m2y *= inv;
  float sx = 0.f, sy = 0.f;
#pragma unroll 4
  for (int t = 0; t < T; ++t) {
    const long o = base + (long)t * RD;
    const float2 gv = *reinterpret_cast<const float2*>(g2 + o);
    const float w = swr[t];
    float ox = w * pp.x * gv.x, oy = w * pp.y * gv.y;
    if (t < Tv) {
      const float2 yv = *reinterpret_cast<const float2*>(y + o);
      const float2 dv = *reinterpret_cast<const float2*>(dgn + o);
      const float xh0 = (yv.x - st4.x) * st4.y, xh1 = (yv.y - st4.z) * st4.w;
      const float g = sgam[t];
      ox += st4.y * (dv.x * g - m1x - xh0 * m2x);
      oy += st4.w * (dv.y * g - m1y - xh1 * m2y);
    }
    sx += ox; sy += oy;
    *reinterpret_cast<__nv_bfloat162*>(dy16 + o) = __floats2bfloat162_rn(ox, oy);
  }
  atomicAdd(db2 + c, sx); atomicAdd(db2 + c + 1, sy);
  __syncthreads();
  for (int k = threadIdx.x; k < T; k += 128) { atomicAdd(dgamma + k, sh[k * 2]); atomicAdd(dbeta + k, sh[k * 2 + 1]); }
}

// g1 = u * v2 and u = GELU(a1[:, :D]) in one pass (warp per row, grid-stride):
//   du = dg1 v2 -> da1[:, :D] = du GELU'(a1[:, :D]) (bf16) ; dv2 = dg1 u (bf16) ; dbs[n] += sum_c dv2 ; db1[:D] += sum_rows da1
__global__ void __launch_bounds__(256)
dg1_fused_kernel(const float* __restrict__ dg1, const float* __restrict__ v2, const float* __restrict__ u,
                 const float* __restrict__ a1, __nv_bfloat16* __restrict__ da116, __nv_bfloat16* __restrict__ dv216,
                 float* __restrict__ dbs, float* __restrict__ db1, long rows, int IT) {
  __shared__ float sc[RD];
  for (int k = threadIdx.x; k < RD; k += 256) sc[k] = 0.f;
  __syncthreads();
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  float ac[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) ac[j] = 0.f;
  for (long row = (long)blockIdx.x * 8 + w; row < rows; row += (long)gridDim.x * 8) {
    float rs = 0.f;
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      const long o = row * RD + c * 128 + lane * 4, o2 = row * 2 * RD + c * 128 + lane * 4;
      const float4 g = *reinterpret_cast<const float4*>(dg1 + o), vv = *reinterpret_cast<const float4*>(v2 + o),
                   uu = *reinterpret_cast<const float4*>(u + o), aa = *reinterpret_cast<const float4*>(a1 + o2);
      const float4 da = make_float4(g.x * vv.x * gelu_fast_grad(aa.x), g.y * vv.y * gelu_fast_grad(aa.y),
                                    g.z * vv.z * gelu_fast_grad(aa.z), g.w * vv.w * gelu_fast_grad(aa.w));
      const float4 dv = make_float4(g.x * uu.x, g.y * uu.y, g.z * uu.z, g.w * uu.w);
      ac[c * 4] += da.x; ac[c * 4 + 1] += da.y; ac[c * 4 + 2] += da.z; ac[c * 4 + 3] += da.w;
      rs += (dv.x + dv.y) + (dv.z + dv.w);
      store_bf16x4(da116 + o2, da);
      store_bf16x4(dv216 + o, dv);
    }
    rs = warp_sum(rs);
    if (lane == 0) atomicAdd(dbs + (int)(row % IT), rs);
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) atomicAdd(&sc[(j / 4) * 128 + lane * 4 + (j % 4)], ac[j]);
  __syncthreads();
  for (int k = threadIdx.x; k < RD; k += 256) atomicAdd(db1 + k, sc[k]);
}

// Dimensions shared by every contraction of the router.
struct Dims {
  int B, I, T, D;
  long M, IT, ID, TD, ITD;
  bool tc;              // tensor-core (bf16 operand) engine
  int Tv;               // valid frames (<= T): T = 63 is carried padded to 64 by the tensor-core engine
  Dims(int b, int i, int t, int d, bool tc_, int tv = 0) : B(b), I(i), T(t), D(d), M((long)b * i * t), IT((long)i * t),
                                                           ID((long)i * d), TD((long)t * d), ITD((long)i * t * d), tc(tc_),
                                                           Tv(tv > 0 ? tv : t) {}
};

// ---- TMA views of the [B,I,T,D] activation tensors (bf16) --------------------------------------------------
// rows m = (b,t), k = (i,c): K-major, box = 64 c x 64 t x 1 i x 2 b  (a 128-row tile = two samples; needs T == 64)
MrnbTcOperand op_bt_ic_kmajor(const bf16* p, const Dims& d) {
  MrnbTcOperand o{};
  o.ptr = p; o.mn_major = 0;
  o.dims[0] = d.D; o.dims[1] = d.T; o.dims[2] = d.I; o.dims[3] = d.B;
  o.strides[0] = d.D; o.strides[1] = d.TD; o.strides[2] = d.ITD;
  o.box[0] = 64; o.box[1] = 64; o.box[2] = 1; o.box[3] = 2;
  o.recipe = MrnbTmaRecipe{{MRNB_SRC_K, MRNB_SRC_ZERO, MRNB_SRC_K, MRNB_SRC_MN}, {1, 1, d.D, d.T}, {d.D, 0, 0, 0}};
  return o;
}
// m / n = (i,c) contiguous in c, k = (b,t): MN-major, box = 64 c x 64 t x 1 x 1 per 64-wide chunk
MrnbTcOperand op_ic_bt_mnmajor(const bf16* p, const Dims& d) {
  MrnbTcOperand o{};
  o.ptr = p; o.mn_major = 1;
  o.dims[0] = d.D; o.dims[1] = d.T; o.dims[2] = d.I; o.dims[3] = d.B;
  o.strides[0] = d.D; o.strides[1] = d.TD; o.strides[2] = d.ITD;
  o.box[0] = 64; o.box[1] = 64; o.box[2] = 1; o.box[3] = 1;
  o.recipe = MrnbTmaRecipe{{MRNB_SRC_MN, MRNB_SRC_ZERO, MRNB_SRC_MN, MRNB_SRC_K}, {1, 1, d.D, d.T}, {d.D, 0, 0, 0}};
  return o;
}
// per-sample [IT, D] activations as the MN-major B operand of a token-mixing GEMM: n = c contiguous, k = token, g = b
MrnbTcOperand op_tok_c_mnmajor(const bf16* p, const Dims& d) {
  return mrnb_operand_mn2d(p, d.D, d.IT, d.D, d.B, d.ITD);
}
// rows = token n, k = (b,c): K-major with the sample folded into k, box = 64 c x box_rows n x 1 b
MrnbTcOperand op_tok_bc_kmajor(const bf16* p, const Dims& d, int box_rows) {
  MrnbTcOperand o{};
  o.ptr = p; o.mn_major = 0;
  o.dims[0] = d.D; o.dims[1] = d.IT; o.dims[2] = d.B; o.dims[3] = 1;
  o.strides[0] = d.D; o.strides[1] = d.ITD; o.strides[2] = d.ITD * d.B;
  o.box[0] = 64; o.box[1] = box_rows; o.box[2] = 1; o.box[3] = 1;
  o.recipe = MrnbTmaRecipe{{MRNB_SRC_K, MRNB_SRC_MN, MRNB_SRC_K, MRNB_SRC_ZERO}, {1, 1, d.D, 1}, {d.D, 0, 0, 0}};
  return o;
}
MrnbTcOperand nogroup(MrnbTcOperand o) {          // shared weight: ignore the group index
  for (int j = 0; j < 4; ++j) if (o.recipe.src[j] == MRNB_SRC_G) o.recipe.src[j] = MRNB_SRC_ZERO;
  return o;
}
inline int bn_for(int N) { return N >= 128 ? 128 : 64; }
// split-K factor of a weight-gradient GEMM with `tiles` output tiles: the largest split whose tiles x split work items
// still fit ONE wave of the 2 x 148 persistent CTAs (a second, partly filled wave costs a whole tile duration)
inline int splitk_for(int tiles) { const int s = 296 / (tiles > 0 ? tiles : 1); return s < 1 ? 1 : s; }

// out[rows, Nout] = A[rows, K] . W[Nout, K]^T (+bias, +res)   -- plain row-major Linear
int linear_rows(const Dims& d, const float* A32, const bf16* A16, long lda, const float* W32, const bf16* W16, int Nout, int K,
                const float* bias, const float* res, float* out, long ldo, cudaStream_t st) {
  if (d.tc) {
    // plain row-major Linear: the persistent TMEM-double-buffered kernel of the expert path (coalesced epilogue)
    MrnbTcGemm g{};
    g.A = A16; g.lda = lda; g.a_gstride = d.M * lda;
    g.W = W16; g.ldw = K; g.w_gstride = (long)Nout * K;
    g.bias = bias; g.out = out; g.ldo = ldo; g.o_gstride = d.M * ldo; g.out_f32 = 1; g.res = res;
    g.M = (int)d.M; g.N = Nout; g.K = K; g.groups = 1; g.rows_per_scale = 1;
    return mrnb_tc_gemm(g, st);
  }
  MrnbGemm g = mrnb_gemm_nt(A32, lda, W32, K, out, ldo, (int)d.M, Nout, K);
  g.bias_n = bias; g.res = res;
  return mrnb_sgemm(g, st);
}
// dX[rows, Nin] = dY[rows, Nout] . W[Nout, Nin]
int dx_rows(const Dims& d, const float* dY32, const bf16* dY16, long ldy, int Nout, const float* W32, const bf16* W16, int Nin,
            float* dX, long lddx, cudaStream_t st) {
  if (d.tc) {
    MrnbTcGemm2 g{};
    g.a = mrnb_operand_k2d(dY16, d.M, Nout, ldy, 128, 1);
    g.b = mrnb_operand_mn2d(W16, Nin, Nout, Nin, 1);
    g.out32 = dX; g.cm = mrnb_axis(lddx); g.cn = mrnb_axis(1);
    g.M = (int)d.M; g.N = Nin; g.K = Nout; g.groups = 1; g.alpha = 1.f;
    return mrnb_tc_gemm2(g, st);
  }
  MrnbGemm g{};
  g.A = dY32; g.am = mrnb_axis(ldy); g.ak = mrnb_axis(1); g.a_kfast = 1;
  g.B = W32; g.bk = mrnb_axis(Nin); g.bn = mrnb_axis(1); g.b_kfast = 0;
  g.C = dX; g.cm = mrnb_axis(lddx); g.cn = mrnb_axis(1);
  g.M = (int)d.M; g.N = Nin; g.K = Nout; g.batch = 1; g.splitk = 1; g.alpha = 1.f; g.rows_per_scale = 1;
  return mrnb_sgemm(g, st);
}
// dW[Nout, Nin] += dY[rows, Nout]^T . X[rows, Nin]      (K = rows, split-K into the zeroed gradient arena)
int dw_rows(const Dims& d, const float* dY32, const bf16* dY16, long ldy, int Nout, const float* X32, const bf16* X16, long ldx,
            int Nin, float* dW, cudaStream_t st) {
  if (d.tc) {
    MrnbTcGemm2 g{};
    g.a = mrnb_operand_mn2d(dY16, Nout, d.M, ldy, 1);
    g.b = mrnb_operand_mn2d(X16, Nin, d.M, ldx, 1);
    g.out32 = dW; g.cm = mrnb_axis(Nin); g.cn = mrnb_axis(1);
    g.M = Nout; g.N = Nin; g.K = (int)d.M; g.groups = 1; g.alpha = 1.f;
    g.splitk = splitk_for(cdiv(Nout, 128) * cdiv(Nin, bn_for(Nin)));
    return mrnb_tc_gemm2(g, st);
  }
  MrnbGemm g{};
  g.A = dY32; g.am = mrnb_axis(1); g.ak = mrnb_axis(ldy); g.a_kfast = 0;
  g.B = X32; g.bk = mrnb_axis(ldx); g.bn = mrnb_axis(1); g.b_kfast = 0;
  g.C = dW; g.cm = mrnb_axis(Nin); g.cn = mrnb_axis(1);
  g.M = Nout; g.N = Nin; g.K = (int)d.M; g.batch = 1; g.alpha = 1.f; g.rows_per_scale = 1;
  g.splitk = (int)((d.M + 2047) / 2048); if (g.splitk > 64) g.splitk = 64; if (g.splitk < 1) g.splitk = 1;
  return mrnb_sgemm(g, st);
}

// v2[b] = Ws . vn[b] + bs   (token mixing over n = i*T+t)
int token_mix_fwd(const Dims& d, const float* Ws32, const bf16* Ws16, const float* bs, const float* vn32, const bf16* vn16,
                  float* v2, cudaStream_t st) {
  if (d.tc) {
    MrnbTcGemm2 g{};
    g.a = nogroup(mrnb_operand_k2d(Ws16, d.IT, d.IT, d.IT, 128, 1));
    g.b = op_tok_c_mnmajor(vn16, d);
    g.out32 = v2; g.cm = mrnb_axis(d.D); g.cn = mrnb_axis(1); g.c_gstride = d.ITD;
    g.bias_m = bs; g.M = (int)d.IT; g.N = d.D; g.K = (int)d.IT; g.groups = d.B; g.alpha = 1.f;
    return mrnb_tc_gemm2(g, st);
  }
  MrnbGemm g{};
  g.A = Ws32; g.am = mrnb_axis(d.IT); g.ak = mrnb_axis(1); g.a_kfast = 1; g.sAb = 0;
  g.B = vn32; g.bk = mrnb_axis(d.D); g.bn = mrnb_axis(1); g.b_kfast = 0; g.sBb = d.ITD;
  g.C = v2; g.cm = mrnb_axis(d.D); g.cn = mrnb_axis(1); g.sCb = d.ITD;
  g.M = (int)d.IT; g.N = d.D; g.K = (int)d.IT; g.batch = d.B; g.splitk = 1; g.alpha = 1.f; g.rows_per_scale = 1;
  g.bias_m = bs;
  return mrnb_sgemm(g, st);
}
// dvn[b,m,:] = sum_n Ws[n,m] dv2[b,n,:] ;  dWs[n,m] += sum_(b,c) dv2[b,n,c] vn[b,m,c]
int token_mix_bwd(const Dims& d, const float* Ws32, const bf16* Ws16, const float* dv2_32, const bf16* dv2_16,
                  const float* vn32, const bf16* vn16, float* dvn, float* dWs, cudaStream_t st) {
  if (d.tc) {
    MrnbTcGemm2 g{};
    g.a = nogroup(mrnb_operand_mn2d(Ws16, d.IT, d.IT, d.IT, 1));
    g.b = op_tok_c_mnmajor(dv2_16, d);
    g.out32 = dvn; g.cm = mrnb_axis(d.D); g.cn = mrnb_axis(1); g.c_gstride = d.ITD;
    g.M = (int)d.IT; g.N = d.D; g.K = (int)d.IT; g.groups = d.B; g.alpha = 1.f;
    MRNB_TRY(mrnb_tc_gemm2(g, st));
    MrnbTcGemm2 h{};
    h.a = op_tok_bc_kmajor(dv2_16, d, 128);
    h.b = op_tok_bc_kmajor(vn16, d, bn_for((int)d.IT));
    h.out32 = dWs; h.cm = mrnb_axis(d.IT); h.cn = mrnb_axis(1);
    h.M = (int)d.IT; h.N = (int)d.IT; h.K = d.B * d.D; h.groups = 1; h.alpha = 1.f;
    h.splitk = splitk_for(cdiv(d.IT, 128) * cdiv(d.IT, bn_for((int)d.IT)));
    return mrnb_tc_gemm2(h, st);
  }
  MrnbGemm g{};
  g.A = Ws32; g.am = mrnb_axis(1); g.ak = mrnb_axis(d.IT); g.a_kfast = 0; g.sAb = 0;
  g.B = dv2_32; g.bk = mrnb_axis(d.D); g.bn = mrnb_axis(1); g.b_kfast = 0; g.sBb = d.ITD;
  g.C = dvn; g.cm = mrnb_axis(d.D); g.cn = mrnb_axis(1); g.sCb = d.ITD;
  g.M = (int)d.IT; g.N = d.D; g.K = (int)d.IT; g.batch = d.B; g.splitk = 1; g.alpha = 1.f; g.rows_per_scale = 1;
  MRNB_TRY(mrnb_sgemm(g, st));
  MrnbGemm h{};
  h.A = dv2_32; h.am = mrnb_axis(d.D); h.ak = mrnb_axis2(d.D, 1, d.ITD); h.a_kfast = 1;
  h.B = vn32; h.bn = mrnb_axis(d.D); h.bk = mrnb_axis2(d.D, 1, d.ITD); h.b_kfast = 1;
  h.C = dWs; h.cm = mrnb_axis(d.IT); h.cn = mrnb_axis(1);
  h.M = (int)d.IT; h.N = (int)d.IT; h.K = d.B * d.D; h.batch = 1; h.alpha = 1.f; h.rows_per_scale = 1;
  h.splitk = (d.B * d.D + 2047) / 2048; if (h.splitk > 32) h.splitk = 32; if (h.splitk < 1) h.splitk = 1;
  return mrnb_sgemm(h, st);
}

// g2[(b,t),(i,c)] = sum_(i',c') gn[(b,t),(i',c')] Wc[(i,c),(i',c')] + bc   (channel mixing over k = i*D+c, K = N = I*D)
// On tcgen05 every channel-mix GEMM runs 128 x 128 tiles at two CTAs per SM.  128 x 256 tiles at one CTA per SM (4-stage
// ring) measured slower: forward 135 -> 137 us, dgn 164 -> 204 us, dWc 165 -> 218 us, and in an earlier measurement
// forward 175 -> 246 us.  The second co-resident CTA hides more latency than the wider tile saves in L2 traffic.
int channel_mix_fwd(const Dims& d, const float* Wc32, const bf16* Wc16, const float* bc, const float* gn32, const bf16* gn16,
                    float* g2, cudaStream_t st) {
  if (d.tc) {
    MrnbTcGemm2 g{};
    g.a = op_bt_ic_kmajor(gn16, d);
    g.b = mrnb_operand_k2d(Wc16, d.ID, d.ID, d.ID, 128, 1);
    g.out32 = g2; g.cm = mrnb_axis2(d.T, d.D, d.ITD); g.cn = mrnb_axis2(d.D, 1, d.TD);
    g.bias_n = bc; g.M = d.B * d.T; g.N = (int)d.ID; g.K = (int)d.ID; g.groups = 1; g.alpha = 1.f;
    return mrnb_tc_gemm2(g, st);
  }
  MrnbGemm g{};
  g.A = gn32; g.am = mrnb_axis2(d.T, d.D, d.ITD); g.ak = mrnb_axis2(d.D, 1, d.TD); g.a_kfast = 1;
  g.B = Wc32; g.bn = mrnb_axis(d.ID); g.bk = mrnb_axis(1); g.b_kfast = 1;
  g.C = g2; g.cm = mrnb_axis2(d.T, d.D, d.ITD); g.cn = mrnb_axis2(d.D, 1, d.TD);
  g.M = d.B * d.T; g.N = (int)d.ID; g.K = (int)d.ID; g.batch = 1; g.splitk = 1; g.alpha = 1.f; g.rows_per_scale = 1;
  g.bias_n = bc;
  return mrnb_sgemm(g, st);
}
// dgn[(b,t), j] = sum_k dg2[(b,t),k] Wc[k,j] ;  dWc[k,j] += sum_(b,t) dg2[(b,t),k] gn[(b,t),j]
int channel_mix_bwd(const Dims& d, const float* Wc32, const bf16* Wc16, const float* dg2_32, const bf16* dg2_16,
                    const float* gn32, const bf16* gn16, float* dgn, float* dWc, cudaStream_t st) {
  if (d.tc) {
    MrnbTcGemm2 g{};
    g.a = op_bt_ic_kmajor(dg2_16, d);
    g.b = mrnb_operand_mn2d(Wc16, d.ID, d.ID, d.ID, 1);
    g.out32 = dgn; g.cm = mrnb_axis2(d.T, d.D, d.ITD); g.cn = mrnb_axis2(d.D, 1, d.TD);
    g.M = d.B * d.T; g.N = (int)d.ID; g.K = (int)d.ID; g.groups = 1; g.alpha = 1.f;
    MRNB_TRY(mrnb_tc_gemm2(g, st));
    MrnbTcGemm2 h{};
    h.a = op_ic_bt_mnmajor(dg2_16, d);
    h.b = op_ic_bt_mnmajor(gn16, d);
    h.out32 = dWc; h.cm = mrnb_axis(d.ID); h.cn = mrnb_axis(1);
    h.M = (int)d.ID; h.N = (int)d.ID; h.K = d.B * d.T; h.groups = 1; h.alpha = 1.f;
    h.splitk = splitk_for(cdiv(d.ID, 128) * cdiv(d.ID, 128));
    return mrnb_tc_gemm2(h, st);
  }
  MrnbGemm g{};
  g.A = dg2_32; g.am = mrnb_axis2(d.T, d.D, d.ITD); g.ak = mrnb_axis2(d.D, 1, d.TD); g.a_kfast = 1;
  g.B = Wc32; g.bk = mrnb_axis(d.ID); g.bn = mrnb_axis(1); g.b_kfast = 0;
  g.C = dgn; g.cm = mrnb_axis2(d.T, d.D, d.ITD); g.cn = mrnb_axis2(d.D, 1, d.TD);
  g.M = d.B * d.T; g.N = (int)d.ID; g.K = (int)d.ID; g.batch = 1; g.splitk = 1; g.alpha = 1.f; g.rows_per_scale = 1;
  MRNB_TRY(mrnb_sgemm(g, st));
  MrnbGemm h{};
  h.A = dg2_32; h.am = mrnb_axis2(d.D, 1, d.TD); h.ak = mrnb_axis2(d.T, d.D, d.ITD); h.a_kfast = 0;
  h.B = gn32; h.bk = mrnb_axis2(d.T, d.D, d.ITD); h.bn = mrnb_axis2(d.D, 1, d.TD); h.b_kfast = 0;
  h.C = dWc; h.cm = mrnb_axis(d.ID); h.cn = mrnb_axis(1);
  h.M = (int)d.ID; h.N = (int)d.ID; h.K = d.B * d.T; h.batch = 1; h.alpha = 1.f; h.rows_per_scale = 1;
  const int tiles = cdiv(d.ID, 128) * cdiv(d.ID, 128);
  h.splitk = tiles >= 120 ? 1 : (tiles >= 30 ? 4 : 16);
  if ((long)d.B * d.T < 64L * h.splitk) h.splitk = 1;
  return mrnb_sgemm(h, st);
}

int router_forward(const float* P, const float* x, const Dims& d, float* out_user, float* scores, float* gate, int* index,
                   RouterWs& w, cudaStream_t st) {
  long off[MRNB_ROUTER_NPARAMS + 1];
  const long nparam = router_offsets(d.I, d.T, d.D, off);
  const int B = d.B, I = d.I, T = d.T, D = d.D;
  const long M = d.M;
  const bool tc = d.tc;
  const bf16* W16 = w.w16;
  float* out = w.out;   // kept in the workspace for the backward; copied to the caller's buffer at the end
  {
    MrnbProfScope prof(MRNB_PROF_ROUTER_EW, st);
    if (tc) {
      LAUNCH_EW(cast16_kernel, nparam, P, w.w16, nparam);
      fold_ln_w1_kernel<<<2 * D, RD, 0, st>>>(P + off[R_P1_W], P + off[R_P1_B], P + off[R_N_W], P + off[R_N_B],
                                              w.w16 + off[R_P1_W], w.b1f);
      MRNB_CHECK_LAUNCH("fold_ln_w1_kernel");
    }
    // tensor-core mode: xn16 holds the plain x-hat, LayerNorm 1's affine lives in the folded proj_1 weights / bias
    ln_rows_fwd_kernel<<<cdiv(M, 8), 256, 0, st>>>(x, tc ? nullptr : P + off[R_N_W], P + off[R_N_B], tc ? nullptr : w.xn,
                                                   tc ? w.xn16 : nullptr, w.stats1, M, 1e-5f);
    MRNB_CHECK_LAUNCH("ln_rows_fwd_kernel");
  }
  // a1 = xn W1^T + b1
  MRNB_TRY(linear_rows(d, w.xn, w.xn16, D, P + off[R_P1_W], W16 + off[R_P1_W], 2 * D, D, tc ? w.b1f : P + off[R_P1_B], nullptr,
                       w.a1, 2 * D, st));
  {
    MrnbProfScope prof(MRNB_PROF_ROUTER_EW, st);
    if (tc) gelu_ln_fwd_kernel<true><<<cdiv(M, 8), 256, 0, st>>>(w.a1, P + off[R_SN_W], P + off[R_SN_B], w.u, nullptr, w.vn16, w.stats2, M, 1e-5f);
    else gelu_ln_fwd_kernel<false><<<cdiv(M, 8), 256, 0, st>>>(w.a1, P + off[R_SN_W], P + off[R_SN_B], w.u, w.vn, nullptr, w.stats2, M, 1e-5f);
    MRNB_CHECK_LAUNCH("gelu_ln_fwd_kernel");
  }
  MRNB_TRY(token_mix_fwd(d, P + off[R_SP_W], W16 + off[R_SP_W], P + off[R_SP_B], w.vn, w.vn16, w.v2, st));
  {   // g1 = u * v2 (a separate streaming pass: measured faster than a multiplier read in the GEMM's row-per-thread epilogue)
    MrnbProfScope prof(MRNB_PROF_ROUTER_EW, st);
    LAUNCH_EW(mul_kernel, M * D / 4, w.u, w.v2, tc ? nullptr : w.g1, tc ? w.g116 : nullptr, M * D / 4);
  }
  // y = g1 W2^T + b2 + x
  MRNB_TRY(linear_rows(d, w.g1, w.g116, D, P + off[R_P2_W], W16 + off[R_P2_W], D, D, P + off[R_P2_B], x, w.y, D, st));
  {
    MrnbProfScope prof(MRNB_PROF_ROUTER_EW, st);
    if (T == 64)
      lnT_fwd64_kernel<<<B * I, RD, 0, st>>>(w.y, P + off[R_CN_W], P + off[R_CN_B], tc ? nullptr : w.gn, tc ? w.gn16 : nullptr,
                                             w.statsT, d.Tv, 1e-5f);
    else
      lnT_fwd_kernel<<<B * I, RD, 0, st>>>(w.y, P + off[R_CN_W], P + off[R_CN_B], tc ? nullptr : w.gn, tc ? w.gn16 : nullptr,
                                           w.statsT, T, d.Tv, 1e-5f);
    MRNB_CHECK_LAUNCH("lnT_fwd_kernel");
  }
  MRNB_TRY(channel_mix_fwd(d, P + off[R_CP_W], W16 + off[R_CP_W], P + off[R_CP_B], w.gn, w.gn16, w.g2, st));
  {
    MrnbProfScope prof(MRNB_PROF_ROUTER_EW, st);
    LAUNCH_EW(mul_kernel, M * D / 4, w.y, w.g2, tc ? nullptr : w.y2, tc ? w.y216 : nullptr, M * D / 4);
  }
  // out = y2 W3^T + b3 + x
  MRNB_TRY(linear_rows(d, w.y2, w.y216, D, P + off[R_P3_W], W16 + off[R_P3_W], D, D, P + off[R_P3_B], x, out, D, st));
  if (scores || gate || index) {
    {   // s[(b,t), j] = sum_(i,c) out[b,i,t,c] Wcr[j,(i,c)] + bcr[j]     (N = I: fp32 GEMV, one pass over `out`)
      MrnbProfScope prof(MRNB_PROF_ROUTER_EW, st);
      MRNB_DISPATCH_I(launch_gate_head, I, out, P + off[R_CR_W], P + off[R_CR_B], B, T, w.s, st);
    }
    gate_finish_kernel<<<cdiv(B, 8), 256, 0, st>>>(w.s, P + off[R_ROUTE_W], P + off[R_ROUTE_B], B, T, I, scores, gate, index);
    MRNB_CHECK_LAUNCH("gate_finish_kernel");
  }
  if (out_user) cudaMemcpyAsync(out_user, out, (size_t)M * D * sizeof(float), cudaMemcpyDeviceToDevice, st);
  return MRNB_OK;
}

// Tensor-core mode, proj_1 + LayerNorm 1 parameter gradients from da1 (bf16) and db1 = G[R_P1_B] (complete):
// S = da1^T xhat on tcgen05 (split-K), then the [2D, D] fold kernel.
int ln1_fold_backward(const float* P, const long* off, const Dims& d, float* G, RouterWs& w, cudaStream_t st) {
  const int D = d.D;
  cudaMemsetAsync(w.S1, 0, (size_t)2 * D * D * sizeof(float), st);
  MRNB_TRY(dw_rows(d, nullptr, w.da116, 2 * D, 2 * D, nullptr, w.xn16, D, D, w.S1, st));
  MrnbProfScope prof(MRNB_PROF_ROUTER_EW, st);
  fold_ln_w1_bwd_kernel<<<cdiv(2 * D, 32), RD, 0, st>>>(w.S1, G + off[R_P1_B], P + off[R_P1_W], P + off[R_N_W], P + off[R_N_B],
                                                        2 * D, G + off[R_P1_W], G + off[R_N_W], G + off[R_N_B]);
  MRNB_CHECK_LAUNCH("fold_ln_w1_bwd_kernel");
  return MRNB_OK;
}

// Backward through DM_Router given d_out in w.dout (+ w.dout16 in tensor-core mode).  G = zeroed gradient arena.
int dm_router_backward_core(const float* P, const float* x, const Dims& d, float* G, float* dx, RouterWs& w, cudaStream_t st) {
  long off[MRNB_ROUTER_NPARAMS + 1];
  router_offsets(d.I, d.T, d.D, off);
  const int B = d.B, I = d.I, T = d.T, D = d.D;
  const long M = d.M, IT = d.IT, ID = d.ID, TD = d.TD, ITD = d.ITD;
  const long n4 = M * D / 4;
  const bool tc = d.tc;
  const bf16* W16 = w.w16;
  // out = y2 W3^T + b3 + x
  MRNB_TRY(dx_rows(d, w.dout, w.dout16, D, D, P + off[R_P3_W], W16 + off[R_P3_W], D, w.dy2, D, st));
  MRNB_TRY(dw_rows(d, w.dout, w.dout16, D, D, w.y2, w.y216, D, D, G + off[R_P3_W], st));
  MRNB_TRY(colsum(w.dout, mrnb_axis(D), mrnb_axis(1), (int)M, D, G + off[R_P3_B], st));
  {  // y2 = y * g2 : dy = dy2*g2 ; dg2 = dy2*y
    MrnbProfScope prof(MRNB_PROF_ROUTER_EW, st);
    LAUNCH_EW(mul2_kernel, n4, w.dy2, w.g2, w.y, w.dy, w.dg2, tc ? w.dg216 : nullptr, n4);
  }
  MRNB_TRY(channel_mix_bwd(d, P + off[R_CP_W], W16 + off[R_CP_W], w.dg2, w.dg216, w.gn, w.gn16, w.dgn, G + off[R_CP_W], st));
  MRNB_TRY(colsum(w.dg2, mrnb_axis2(T, D, ITD), mrnb_axis2(D, 1, TD), B * T, (int)ID, G + off[R_CP_B], st));
  {  // gn = LN_T(y)
    MrnbProfScope prof(MRNB_PROF_ROUTER_EW, st);
    lnT_bwd_kernel<<<B * I, RD, 2 * T * sizeof(float), st>>>(w.y, w.statsT, P + off[R_CN_W], w.dgn, w.dy, tc ? w.dy16 : nullptr,
                                                              G + off[R_CN_W], G + off[R_CN_B], T, d.Tv);
    MRNB_CHECK_LAUNCH("lnT_bwd_kernel");
  }
  // y = g1 W2^T + b2 + x
  MRNB_TRY(dx_rows(d, w.dy, w.dy16, D, D, P + off[R_P2_W], W16 + off[R_P2_W], D, w.dg1, D, st));
  MRNB_TRY(dw_rows(d, w.dy, w.dy16, D, D, w.g1, w.g116, D, D, G + off[R_P2_W], st));
  MRNB_TRY(colsum(w.dy, mrnb_axis(D), mrnb_axis(1), (int)M, D, G + off[R_P2_B], st));
  {  // g1 = u * v2 : du = dg1*v2 ; dv2 = dg1*u
    MrnbProfScope prof(MRNB_PROF_ROUTER_EW, st);
    LAUNCH_EW(mul2_kernel, n4, w.dg1, w.v2, w.u, w.du, w.dv2, tc ? w.dv216 : nullptr, n4);
  }
  MRNB_TRY(token_mix_bwd(d, P + off[R_SP_W], W16 + off[R_SP_W], w.dv2, w.dv216, w.vn, w.vn16, w.dvn, G + off[R_SP_W], st));
  {  // dbs[n] = sum_(b,c) dv2[b,n,c]
    MrnbProfScope prof(MRNB_PROF_ROUTER_EW, st);
    rowsum256_kernel<<<dim3((int)IT, B >= 64 ? 2 : 1), 256, 0, st>>>(w.dv2, (int)IT, B, G + off[R_SP_B]);
    MRNB_CHECK_LAUNCH("rowsum256_kernel");
  }
  {  // vn = LN_D(GELU(a1v)); u = GELU(a1u)
    MrnbProfScope prof(MRNB_PROF_ROUTER_EW, st);
    if (tc) ln_rows_bwd_kernel<true, true><<<rows16_grid(M), 256, 0, st>>>(w.a1 + D, 2 * D, w.stats2, P + off[R_SN_W], w.dvn,
                                                                           w.da1 + D, w.da116 + D, 2 * D, nullptr, nullptr,
                                                                           G + off[R_SN_W], G + off[R_SN_B], M);
    else ln_rows_bwd_kernel<true><<<rows16_grid(M), 256, 0, st>>>(w.a1 + D, 2 * D, w.stats2, P + off[R_SN_W], w.dvn, w.da1 + D,
                                                                  nullptr, 2 * D, nullptr, nullptr,
                                                                  G + off[R_SN_W], G + off[R_SN_B], M);
    MRNB_CHECK_LAUNCH("ln_rows_bwd_kernel");
    LAUNCH_EW(gelu_bwd_kernel, M * D, w.a1, w.du, w.da1, tc ? w.da116 : nullptr, M);
  }
  // a1 = xn W1^T + b1
  MRNB_TRY(colsum(w.da1, mrnb_axis(2 * D), mrnb_axis(1), (int)M, 2 * D, G + off[R_P1_B], st));
  if (tc) {
    MRNB_TRY(ln1_fold_backward(P, off, d, G, w, st));
    if (dx) {   // dxhat = da1 (W1 diag(gamma)): the folded bf16 weights already carry gamma
      MRNB_TRY(dx_rows(d, w.da1, w.da116, 2 * D, 2 * D, P + off[R_P1_W], W16 + off[R_P1_W], D, w.dxn, D, st));
      MrnbProfScope prof(MRNB_PROF_ROUTER_EW, st);
      ln_rows_bwd_kernel<false><<<rows16_grid(M), 256, 0, st>>>(x, D, w.stats1, nullptr, w.dxn, dx, nullptr, D, w.dy, w.dout,
                                                                nullptr, nullptr, M);
      MRNB_CHECK_LAUNCH("ln_rows_bwd_kernel");
    }
    return MRNB_OK;
  }
  MRNB_TRY(dw_rows(d, w.da1, w.da116, 2 * D, 2 * D, w.xn, w.xn16, D, D, G + off[R_P1_W], st));
  MRNB_TRY(dx_rows(d, w.da1, w.da116, 2 * D, 2 * D, P + off[R_P1_W], W16 + off[R_P1_W], D, w.dxn, D, st));
  {  // xn = LN_D(x): dgamma/dbeta (+ dx = LNbwd + dy + dout when requested)
    MrnbProfScope prof(MRNB_PROF_ROUTER_EW, st);
    ln_rows_bwd_kernel<false><<<rows16_grid(M), 256, 0, st>>>(x, D, w.stats1, P + off[R_N_W], w.dxn, dx, nullptr, D,
                                                              dx ? w.dy : nullptr, dx ? w.dout : nullptr,
                                                              G + off[R_N_W], G + off[R_N_B], M);
    MRNB_CHECK_LAUNCH("ln_rows_bwd_kernel");
  }
  return MRNB_OK;
}

// Training-step backward with d_out materialised: gate head from dL/ds (w.ds), then the generic DM_Router backward on
// dout.  The fp32 engine always runs it; the tensor-core engine runs it when the input gradient dx [B,I,T,D] is asked for
// (its own rank-one path never forms dx).  G = zeroed gradient arena.
int router_backward_gate_dout(const float* P, const float* x, const Dims& d, float* G, float* dx, RouterWs& w, cudaStream_t st) {
  long off[MRNB_ROUTER_NPARAMS + 1];
  router_offsets(d.I, d.T, d.D, off);
  {  // dWcr[j,(i,c)] = sum_(b,t) ds[(b,t),j] out[b,i,t,c]
    MrnbProfScope prof(MRNB_PROF_ROUTER_EW, st);
    MRNB_DISPATCH_I(launch_gate_head_dw, d.I, w.ds, w.out, d.B, d.T, G + off[R_CR_W], st);
  }
  MRNB_TRY(colsum(w.ds, mrnb_axis(d.I), mrnb_axis(1), d.B * d.T, d.I, G + off[R_CR_B], st));
  {  // dout[b,i,t,c] = sum_j ds[(b,t),j] Wcr[j,(i,c)]
    MrnbProfScope prof(MRNB_PROF_ROUTER_EW, st);
    const long total4 = d.M * d.D / 4;
    LAUNCH_EW(dout_kernel, total4, w.ds, P + off[R_CR_W], d.I, d.T, total4, w.dout, d.tc ? w.dout16 : nullptr);
  }
  return dm_router_backward_core(P, x, d, G, dx, w, st);
}

// Training-step backward in tensor-core mode: gate head + DM_Router parameter gradients from dL/dr (w.dr), with the
// rank-one structure of the gate head's input gradient exploited (see the kernel section above).  18 launches; no
// [M, D] fp32 gradient is written except the four GEMM outputs (dgn, dg1, dvn, dxn).  G = zeroed gradient arena.
int router_backward_gate_tc(const float* P, const float* x, const Dims& d, float* G, RouterWs& w, cudaStream_t st) {
  long off[MRNB_ROUTER_NPARAMS + 1];
  router_offsets(d.I, d.T, d.D, off);
  const int B = d.B, I = d.I, T = d.T, D = d.D;
  const long M = d.M, IT = d.IT, ID = d.ID;
  const bf16* W16 = w.w16;
  const float* wr = P + off[R_ROUTE_W];
  Dims dq = d;                        // the collapsed last Linear: B*I rows (zero-padded to a 128-row tile) instead of B*I*T
  dq.M = ((long)B * I + 127) / 128 * 128;
  if (dq.M > (long)B * I) {
    cudaMemsetAsync(w.gq16 + (long)B * I * D, 0, (size_t)(dq.M - (long)B * I) * D * sizeof(bf16), st);
    cudaMemsetAsync(w.y2w16 + (long)B * I * D, 0, (size_t)(dq.M - (long)B * I) * D * sizeof(bf16), st);
  }
  {
    MrnbProfScope prof(MRNB_PROF_ROUTER_EW, st);
    gate_q_kernel<<<B * I, RD, 0, st>>>(w.dr, P + off[R_CR_W], wr, I, T, w.gq16, G + off[R_P3_B], G + off[R_CR_B]);
    MRNB_CHECK_LAUNCH("gate_q_kernel");
  }
  // p = q W3   ([B*I, D] x [D, D], W3 read MN-major where it lies)
  MRNB_TRY(dx_rows(dq, nullptr, w.gq16, D, D, P + off[R_P3_W], W16 + off[R_P3_W], D, w.gp, D, st));
  {
    MrnbProfScope prof(MRNB_PROF_ROUTER_EW, st);
    tsum_dg2_kernel<<<B * I, 128, 0, st>>>(w.out, w.y216, w.y, w.gp, wr, I, T, w.ow, w.y2w16, w.dg216, G + off[R_CP_B]);
    MRNB_CHECK_LAUNCH("tsum_dg2_kernel");
    gate_dwcr_kernel<<<dim3(cdiv(ID, 256), B >= 64 ? 32 : 1), 256, 0, st>>>(w.dr, w.ow, B, I, ID, G + off[R_CR_W]);
    MRNB_CHECK_LAUNCH("gate_dwcr_kernel");
  }
  // dW3[n,k] = sum_(b,i) q[(b,i),n] y2w[(b,i),k]
  MRNB_TRY(dw_rows(dq, nullptr, w.gq16, D, D, nullptr, w.y2w16, D, D, G + off[R_P3_W], st));
  MRNB_TRY(channel_mix_bwd(d, nullptr, W16 + off[R_CP_W], nullptr, w.dg216, nullptr, w.gn16, w.dgn, G + off[R_CP_W], st));
  {
    MrnbProfScope prof(MRNB_PROF_ROUTER_EW, st);
    // (capping the resident blocks so that the second pass over y / dgn hits L2 cut the DRAM reads from 500 to 400 MB but
    // ran slower -- 147 vs 121 us: too few loads in flight per SM)
    lnT_bwd2_kernel<<<B * I, 128, 0, st>>>(w.y, w.statsT, P + off[R_CN_W], w.dgn, w.g2, w.gp, wr, w.dy16, G + off[R_CN_W],
                                           G + off[R_CN_B], G + off[R_P2_B], T, d.Tv);
    MRNB_CHECK_LAUNCH("lnT_bwd2_kernel");
  }
  // y = g1 W2^T + b2 + x
  MRNB_TRY(dx_rows(d, nullptr, w.dy16, D, D, P + off[R_P2_W], W16 + off[R_P2_W], D, w.dg1, D, st));
  MRNB_TRY(dw_rows(d, nullptr, w.dy16, D, D, nullptr, w.g116, D, D, G + off[R_P2_W], st));
  {
    MrnbProfScope prof(MRNB_PROF_ROUTER_EW, st);
    dg1_fused_kernel<<<rows16_grid(M), 256, 0, st>>>(w.dg1, w.v2, w.u, w.a1, w.da116, w.dv216, G + off[R_SP_B],
                                                     G + off[R_P1_B], M, (int)IT);
    MRNB_CHECK_LAUNCH("dg1_fused_kernel");
  }
  MRNB_TRY(token_mix_bwd(d, nullptr, W16 + off[R_SP_W], nullptr, w.dv216, nullptr, w.vn16, w.dvn, G + off[R_SP_W], st));
  {  // vn = LN_D(GELU(a1v)): da1[:, D:] (bf16 only), db1[D:], dgamma / dbeta
    MrnbProfScope prof(MRNB_PROF_ROUTER_EW, st);
    ln_rows_bwd_kernel<true, true><<<rows16_grid(M), 256, 0, st>>>(w.a1 + D, 2 * D, w.stats2, P + off[R_SN_W], w.dvn, nullptr,
                                                                   w.da116 + D, 2 * D, nullptr, nullptr, G + off[R_SN_W],
                                                                   G + off[R_SN_B], M, G + off[R_P1_B] + D);
    MRNB_CHECK_LAUNCH("ln_rows_bwd_kernel");
  }
  // a1 = xhat (W1 gamma)^T + b1f: proj_1 and LayerNorm 1 gradients from S = da1^T xhat (no M-row dxn GEMM, no pass over x)
  MRNB_TRY(ln1_fold_backward(P, off, d, G, w, st));
  return MRNB_OK;
}

}  // namespace

extern "C" long mrnb_router_param_offsets(int n_experts, int T, int D, long* offsets) {
  long tmp[MRNB_ROUTER_NPARAMS + 1];
  const long n = router_offsets(n_experts, T, D, tmp);
  if (offsets) for (int k = 0; k <= MRNB_ROUTER_NPARAMS; ++k) offsets[k] = tmp[k];
  return n;
}

#define ROUTER_ARGCHECK(name)                                                                                   \
  MRNB_CHECK_ARG(params && x && workspace && B > 0 && T > 0, name ": null/empty argument");                      \
  MRNB_CHECK_ARG(n_experts >= 1 && n_experts <= MRNB_MAX_EXPERTS, name ": n_experts %d out of range", n_experts); \
  MRNB_CHECK_ARG(D == RD, name ": only D == 256 (opt.hidden_size) is supported, got %d", D);                     \
  MRNB_CHECK_ARG(prec == MRNB_PREC_FP32 || prec == MRNB_PREC_BF16, name ": unknown precision %d", prec);

// The tensor-core engine tiles rows (b,t) as 2 samples x 64 frames: SVTR's T = 64 (modules/model.py:324) runs as is;
// CRNN's T = 63 (:322-323) runs PADDED to 64 frames: the activations get a zero frame, the T-dependent parameters
// (route.weight, spatial_gating.proj.{weight,bias}, channel_gating.norm.{weight,bias}) get zero rows / columns, the
// LayerNorm over frames masks the pad (Dims::Tv), and the gradient arena is un-padded at the end.  With those zeros the
// pad frame contributes exactly nothing to any valid output or gradient (see DESIGN.md §3).
static inline bool use_tc(int prec, int T) { return prec == MRNB_PREC_BF16 && T <= 64 && T >= 32; }
static inline int padded_T(int prec, int T) { return use_tc(prec, T) ? 64 : T; }

namespace {

struct RepackTable { long off[MRNB_ROUTER_NPARAMS + 1]; long offp[MRNB_ROUTER_NPARAMS + 1]; long sz[MRNB_ROUTER_NPARAMS]; };

// unpadded arena index i  <->  padded arena index; to_padded: dst[pad(i)] = src[i] (dst pre-zeroed), else dst[i] = src[pad(i)]
__global__ void repack_arena_kernel(const float* __restrict__ src, float* __restrict__ dst, RepackTable tb, int I, int T,
                                    int Tp, long n, int to_padded) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int k = 0;
  while (k + 1 < MRNB_ROUTER_NPARAMS && i >= tb.off[k + 1]) ++k;
  const long j = i - tb.off[k];
  if (j >= tb.sz[k]) { if (!to_padded) dst[i] = 0.f; return; }
  long jp = j;
  if (k == R_SP_W) {
    const long IT = (long)I * T, ITp = (long)I * Tp;
    const long r = j / IT, c = j % IT;
    jp = ((r / T) * Tp + r % T) * ITp + (c / T) * Tp + c % T;
  } else if (k == R_SP_B) {
    jp = (j / T) * Tp + j % T;
  }
  if (to_padded) dst[tb.offp[k] + jp] = src[i];
  else dst[i] = src[tb.offp[k] + jp];
}

// [B*I, T, D] <-> [B*I, Tp, D] (zero pad frame), one float4 per thread over the padded index space
__global__ void pad_frames_kernel(const float* __restrict__ src, float* __restrict__ dst, int T, int Tp, long total4, int to_padded) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total4) return;
  const int c4 = (int)(i % (RD / 4));
  const long r = i / (RD / 4);
  const int t = (int)(r % Tp);
  const long bi = r / Tp;
  if (to_padded) {
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (t < T) v = reinterpret_cast<const float4*>(src)[(bi * T + t) * (RD / 4) + c4];
    reinterpret_cast<float4*>(dst)[i] = v;
  } else if (t < T) {
    reinterpret_cast<float4*>(dst)[(bi * T + t) * (RD / 4) + c4] = reinterpret_cast<const float4*>(src)[i];
  }
}

RepackTable make_table(int I, int T, int Tp, int D) {
  RepackTable tb{};
  router_offsets(I, T, D, tb.off);
  router_offsets(I, Tp, D, tb.offp);
  router_sizes(I, T, D, tb.sz);
  return tb;
}

// workspace tail of the padded mode: padded input, padded parameters, padded gradients.  It sits behind the
// backward-sized carve whatever the call, so that both backward entry points find Pp / xp where mrnb_router_forward
// wrote them.
struct PadWs { float *xp, *Pp, *Gp; size_t bytes; };
PadWs carve_pad(char* base, int B, int I, int Tp, int D) {
  PadWs p{};
  size_t o = al(carve(nullptr, B, I, Tp, D, true).bytes);
  long offp[MRNB_ROUTER_NPARAMS + 1];
  const size_t np = (size_t)router_offsets(I, Tp, D, offp);
  auto take = [&](size_t n) { float* q = base ? (float*)(base + o) : nullptr; o = al(o + n * 4); return q; };
  p.xp = take((size_t)B * I * Tp * D); p.Pp = take(np); p.Gp = take(np);
  p.bytes = o + 256;
  return p;
}

// One call's engine, frame count and workspace: T -> Tp, the carve, the padded tail and the bytes they need.
struct RouterRun {
  Dims d;               // d.T = frames as run (Tp), d.Tv = the caller's frames
  RouterWs w;
  PadWs pw;             // padded mode only
  bool padded;
  size_t bytes;
  RouterRun(void* ws, int B, int I, int T, int D, int prec, bool bwd)
      : d(B, I, padded_T(prec, T), D, use_tc(prec, T), T), w(carve((char*)ws, B, I, d.T, D, bwd)), pw{}, padded(d.T != T) {
    if (padded) pw = carve_pad((char*)ws, B, I, d.T, D);
    bytes = padded ? pw.bytes : w.bytes;
  }
};

int pad_inputs(const float* params, const float* x, const RouterRun& r, cudaStream_t st) {
  MrnbProfScope prof(MRNB_PROF_ROUTER_EW, st);
  const Dims& d = r.d;
  const RepackTable tb = make_table(d.I, d.Tv, d.T, d.D);
  cudaMemsetAsync(r.pw.Pp, 0, (size_t)tb.offp[MRNB_ROUTER_NPARAMS] * sizeof(float), st);
  const long n = tb.off[MRNB_ROUTER_NPARAMS];
  LAUNCH_EW(repack_arena_kernel, n, params, r.pw.Pp, tb, d.I, d.Tv, d.T, n, 1);
  const long total4 = d.M * d.D / 4;
  LAUNCH_EW(pad_frames_kernel, total4, x, r.pw.xp, d.Tv, d.T, total4, 1);
  return MRNB_OK;
}

// padded [B*I, Tp, D] activations -> the caller's [B*I, T, D]
int unpad_frames(const RouterRun& r, const float* src, float* dst, cudaStream_t st) {
  MrnbProfScope prof(MRNB_PROF_ROUTER_EW, st);
  const long total4 = r.d.M * r.d.D / 4;
  LAUNCH_EW(pad_frames_kernel, total4, src, dst, r.d.Tv, r.d.T, total4, 0);
  return MRNB_OK;
}

// padded gradient arena -> the caller's arena
int unpad_grads(const RouterRun& r, float* grads, cudaStream_t st) {
  MrnbProfScope prof(MRNB_PROF_ROUTER_EW, st);
  const RepackTable tb = make_table(r.d.I, r.d.Tv, r.d.T, r.d.D);
  const long n = tb.off[MRNB_ROUTER_NPARAMS];
  LAUNCH_EW(repack_arena_kernel, n, r.pw.Gp, grads, tb, r.d.I, r.d.Tv, r.d.T, n, 0);
  return MRNB_OK;
}

}  // namespace

extern "C" size_t mrnb_router_workspace_bytes(int B, int n_experts, int T, int D, int with_backward) {
  // enough for either precision: the fp32 engine never pads the frames, the tensor-core engine may
  const size_t f32 = RouterRun(nullptr, B, n_experts, T, D, MRNB_PREC_FP32, with_backward != 0).bytes;
  const size_t b16 = RouterRun(nullptr, B, n_experts, T, D, MRNB_PREC_BF16, with_backward != 0).bytes;
  return f32 > b16 ? f32 : b16;
}

extern "C" int mrnb_router_forward(const float* params, const float* x, int B, int n_experts, int T, int D, int prec,
                                   float* out, float* scores, float* gate, int* index, void* workspace,
                                   size_t workspace_bytes, cudaStream_t stream) {
  ROUTER_ARGCHECK("router_forward");
  RouterRun r(workspace, B, n_experts, T, D, prec, false);
  MRNB_CHECK_ARG(workspace_bytes >= r.bytes, "router_forward: workspace too small (%zu < %zu)", workspace_bytes, r.bytes);
  if (!r.padded) return router_forward(params, x, r.d, out, scores, gate, index, r.w, stream);
  MRNB_TRY(pad_inputs(params, x, r, stream));
  MRNB_TRY(router_forward(r.pw.Pp, r.pw.xp, r.d, nullptr, scores, gate, index, r.w, stream));
  return out ? unpad_frames(r, r.w.out, out, stream) : MRNB_OK;
}

// Both training-step backward entries: dx == nullptr is mrnb_router_backward (the tensor-core engine keeps its rank-one
// path, which forms no input gradient).
static int router_backward(const float* params, const float* x, const float* gate, const float* dgate_ctc,
                           const long long* domain, int B, int n_experts, int T, int D, int prec, float* grads, float* dx,
                           float* taski_loss, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  ROUTER_ARGCHECK("router_backward");
  MRNB_CHECK_ARG(gate && grads, "router_backward: null argument");
  MRNB_CHECK_ARG(domain ? taski_loss != nullptr : dgate_ctc != nullptr,
                 "router_backward: a domain needs taski_loss; without one, dgate_ctc is the whole dL/dgate and is required");
  RouterRun r(workspace, B, n_experts, T, D, prec, true);
  MRNB_CHECK_ARG(workspace_bytes >= r.bytes, "router_backward: workspace too small (%zu < %zu)", workspace_bytes, r.bytes);
  if (r.padded) { params = r.pw.Pp; x = r.pw.xp; }   // written by mrnb_router_forward on the same workspace
  float* G = r.padded ? r.pw.Gp : grads;
  const Dims& d = r.d;
  RouterWs& w = r.w;
  cudaStream_t st = stream;
  long off[MRNB_ROUTER_NPARAMS + 1];
  const long nparam = router_offsets(d.I, d.T, d.D, off);
  cudaMemsetAsync(G, 0, nparam * sizeof(float), st);
  if (taski_loss) cudaMemsetAsync(taski_loss, 0, sizeof(float), st);
  {
    MrnbProfScope prof(MRNB_PROF_ROUTER_EW, st);
    gate_bwd_kernel<<<cdiv(B, 256), 256, 0, st>>>(gate, dgate_ctc, domain, B, d.I, w.dr, taski_loss);
    MRNB_CHECK_LAUNCH("gate_bwd_kernel");
    route_bwd_kernel<<<d.T, 256, 0, st>>>(w.dr, w.s, params + off[R_ROUTE_W], B, d.T, d.I, w.ds, G + off[R_ROUTE_W],
                                          G + off[R_ROUTE_B]);
    MRNB_CHECK_LAUNCH("route_bwd_kernel");
  }
  float* dxp = (dx && r.padded) ? w.dg2 : dx;   // padded dx: dg2 is dead by the time the core's last kernel writes dx
  if (d.tc && !dx) MRNB_TRY(router_backward_gate_tc(params, x, d, G, w, st));
  else MRNB_TRY(router_backward_gate_dout(params, x, d, G, dxp, w, st));
  if (!r.padded) return MRNB_OK;
  MRNB_TRY(unpad_grads(r, grads, st));
  return dx ? unpad_frames(r, dxp, dx, st) : MRNB_OK;
}

extern "C" int mrnb_router_backward(const float* params, const float* x, const float* gate, const float* dgate_ctc,
                                    const long long* domain, int B, int n_experts, int T, int D, int prec, float* grads,
                                    float* taski_loss, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  return router_backward(params, x, gate, dgate_ctc, domain, B, n_experts, T, D, prec, grads, nullptr, taski_loss, workspace,
                         workspace_bytes, stream);
}

extern "C" int mrnb_router_backward_dx(const float* params, const float* x, const float* gate, const float* dgate_ctc,
                                       const long long* domain, int B, int n_experts, int T, int D, int prec, float* grads,
                                       float* dx, float* taski_loss, void* workspace, size_t workspace_bytes,
                                       cudaStream_t stream) {
  MRNB_CHECK_ARG(dx, "router_backward_dx: null dx");
  return router_backward(params, x, gate, dgate_ctc, domain, B, n_experts, T, D, prec, grads, dx, taski_loss, workspace,
                         workspace_bytes, stream);
}

extern "C" int mrnb_dm_router_backward(const float* params, const float* x, const float* d_out, int B, int n_experts,
                                       int T, int D, int prec, float* grads, float* dx, void* workspace,
                                       size_t workspace_bytes, cudaStream_t stream) {
  ROUTER_ARGCHECK("dm_router_backward");
  MRNB_CHECK_ARG(d_out && grads, "dm_router_backward: null argument");
  RouterRun r(workspace, B, n_experts, T, D, prec, true);
  MRNB_CHECK_ARG(workspace_bytes >= r.bytes, "dm_router_backward: workspace too small (%zu < %zu)", workspace_bytes, r.bytes);
  const Dims& d = r.d;
  RouterWs& w = r.w;
  cudaStream_t st = stream;
  long off[MRNB_ROUTER_NPARAMS + 1];
  const long nparam = router_offsets(d.I, d.T, d.D, off);
  cudaMemsetAsync(r.padded ? r.pw.Gp : grads, 0, nparam * sizeof(float), st);
  if (!r.padded) {
    cudaMemcpyAsync(w.dout, d_out, (size_t)d.M * D * sizeof(float), cudaMemcpyDeviceToDevice, st);
    if (d.tc) LAUNCH_EW(cast16_kernel, d.M * D, d_out, w.dout16, d.M * D);
    return dm_router_backward_core(params, x, d, grads, dx, w, st);
  }
  {
    MrnbProfScope prof(MRNB_PROF_ROUTER_EW, st);
    const long total4 = d.M * D / 4;
    LAUNCH_EW(pad_frames_kernel, total4, d_out, w.dout, T, d.T, total4, 1);
    LAUNCH_EW(cast16_kernel, d.M * D, w.dout, w.dout16, d.M * D);
  }
  float* dxp = dx ? w.dg2 : nullptr;        // padded dx: dg2 is dead by the time the core's last kernel writes dx
  MRNB_TRY(dm_router_backward_core(r.pw.Pp, r.pw.xp, d, r.pw.Gp, dxp, w, st));
  MRNB_TRY(unpad_grads(r, grads, st));
  return dx ? unpad_frames(r, dxp, dx, st) : MRNB_OK;
}
