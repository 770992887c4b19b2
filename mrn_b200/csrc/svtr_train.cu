// Stage-0 expert training for ONE SVTR expert: activation-keeping forward and the full backward to every parameter.
//
// Reference (paths relative to /root/reference):
//   il_modules/mrn.py:225-279   _init_train: preds = model(image, cross=False)['logits'] (last expert only,
//                               modules/model.py:351-353) -> log_softmax -> CTCLoss(mean, zero_infinity) -> backward ->
//                               clip_grad_norm_(5) -> Adam -> OneCycleLR
//   modules/svtr.py:500-528     SVTR.forward_features (train mode: BatchNorm batch statistics, DropPath per sample)
//   modules/svtr.py:200-204     Block.forward        modules/svtr.py:133-152  Attention.forward
//   modules/svtr.py:246-254     PatchEmbed           modules/svtr.py:285-312  SubSample
//   modules/model.py:82-101,133-148   Model_Extractor.forward / Model.forward (Linear 512->256, CTC head)
// torch.autograd derives the backward in the reference; here every gradient is written out by hand.
//
// Layout: token-major [sample][token][channel]; fp32 residual stream; GEMM operands AT (fp32 parity mode, bf16
// tensor-core mode).  Parameters and gradients use the MrnbSvtrPack slot layout with n_experts == 1, so one flat arena
// serves Adam and the NCCL all-reduce.  The workspace keeps every activation the backward needs (~25 MB / sample fp32).
#include "common.cuh"
#include "gemm_f32.h"
#include "gemm_tc.h"
#include "gemm_tc2.h"
#include "train_util.cuh"
#include "svtr.h"

// attn_train_tc.cu: fused score / softmax and dP / dS kernels
int mrnb_attn_scores_softmax(const void* qkv, void* P, int B, int N, int d, int heads, int W, int local, float scale,
                             cudaStream_t st);
int mrnb_attn_dp_ds(const void* dO16, const void* qkv, const float* dO, const void* O, const void* P, void* dS, int B, int N,
                    int d, int heads, cudaStream_t st);

namespace {

constexpr int KV_LD = 36;
constexpr float ATT_SCALE = 0.17677669529663688110f;      // 32^-0.5: head_dim is 32 in every stage

static const int DIMS[3] = {64, 128, 256}, DEPTH[3] = {3, 6, 3}, HEADS[3] = {2, 4, 8}, GH[3] = {8, 4, 2};
static const int OUTS[3] = {128, 256, 512};

// ------------------------------------------------------------------------------------------------
// conv0 im2col of the NCHW image
// ------------------------------------------------------------------------------------------------
// conv0 (4->32, 3x3 s2 p1) on the NCHW image: col[(b,oh,ow), c*9 + kh*3 + kw]  (nn.Conv2d weight order)
__global__ void im2col_img_kernel(const float* __restrict__ img, float* __restrict__ col, long total) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int k = (int)(i % 36);
  long r = i / 36;
  const int ow = (int)(r % 128); r /= 128;
  const int oh = (int)(r % 16);
  const long b = r / 16;
  const int c = k / 9, kh = (k % 9) / 3, kw = k % 3;
  const int ih = oh * 2 - 1 + kh, iw = ow * 2 - 1 + kw;
  col[i] = (ih >= 0 && ih < 32 && iw >= 0 && iw < 256) ? __ldg(img + ((b * 4 + c) * 32 + ih) * 256 + iw) : 0.f;
}

// the same columns in bf16, zero-padded from 36 to K = 64 (one swizzled k-block of the tensor-core GEMM); thread = 8 columns
__global__ void im2col_img_pad64_kernel(const float* __restrict__ img, __nv_bfloat16* __restrict__ col, long rows) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * 8) return;
  const int j = (int)(i & 7);
  long r = i >> 3;
  const int ow = (int)(r % 128); r /= 128;
  const int oh = (int)(r % 16);
  const long b = r / 16;
  uint32_t pk[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    float v[2];
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int k = j * 8 + u * 2 + e;
      v[e] = 0.f;
      if (k < 36) {
        const int c = k / 9, kh = (k % 9) / 3, kw = k % 3;
        const int ih = oh * 2 - 1 + kh, iw = ow * 2 - 1 + kw;
        if (ih >= 0 && ih < 32 && iw >= 0 && iw < 256) v[e] = __ldg(img + ((b * 4 + c) * 32 + ih) * 256 + iw);
      }
    }
    __nv_bfloat162 hh = __floats2bfloat162_rn(v[0], v[1]);
    pk[u] = *reinterpret_cast<uint32_t*>(&hh);
  }
  *reinterpret_cast<uint4*>(col + i * 8) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
}
// ------------------------------------------------------------------------------------------------
// BatchNorm (train) with GELU on top (finalize: expert_util.cuh, backward apply pass: train_util.cuh)
// ------------------------------------------------------------------------------------------------
// act = GELU(raw * sc + sh) (+ pos[(row % pos_rows), c])      [rows, C] fp32, C % 4 == 0
__global__ void bn_gelu_kernel(const float* __restrict__ raw, const float* __restrict__ ss, const float* __restrict__ pos,
                               int pos_rows, float* __restrict__ act, int C, long total4) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total4) return;
  const int c = (int)((i * 4) % C);
  const float4 r = *reinterpret_cast<const float4*>(raw + i * 4);
  const float* s = ss + c * 2;
  float4 o;
  o.x = gelu_erf(fmaf(r.x, s[0], s[1])); o.y = gelu_erf(fmaf(r.y, s[2], s[3]));
  o.z = gelu_erf(fmaf(r.z, s[4], s[5])); o.w = gelu_erf(fmaf(r.w, s[6], s[7]));
  if (pos) {
    const long n = ((i * 4) / C) % pos_rows;
    const float4 p = *reinterpret_cast<const float4*>(pos + n * C + c);
    o.x += p.x; o.y += p.y; o.z += p.z; o.w += p.w;
  }
  *reinterpret_cast<float4*>(act + i * 4) = o;
}

// backward through GELU and the normalisation: dz = dact * GELU'(raw*sc+sh) (written in place over d), and per-channel
// sums S1 = sum dz, S2 = sum dz * xhat (fp64 atomics).   block (32, 8), grid (C/32, chunks)
__global__ void __launch_bounds__(256)
bn_bwd_reduce_kernel(const float* __restrict__ raw, float* __restrict__ d, const float* __restrict__ ss,
                     const float* __restrict__ mr, long rows, int C, double* __restrict__ sums) {
  __shared__ double sh[8][32][2];
  const int c = blockIdx.x * 32 + threadIdx.x, ty = threadIdx.y;
  const long per = (rows + gridDim.y - 1) / gridDim.y;
  const long r0 = (long)blockIdx.y * per, r1 = (r0 + per < rows) ? r0 + per : rows;
  const float sc = ss[c * 2], sf = ss[c * 2 + 1], mean = mr[c * 2], rstd = mr[c * 2 + 1];
  double s1 = 0.0, s2 = 0.0;
  for (long r = r0 + ty; r < r1; r += 8) {
    const float x = raw[r * C + c];
    const float dz = d[r * C + c] * gelu_erf_grad(fmaf(x, sc, sf));
    d[r * C + c] = dz;
    s1 += dz; s2 += (double)dz * ((x - mean) * rstd);
  }
  sh[ty][threadIdx.x][0] = s1; sh[ty][threadIdx.x][1] = s2;
  __syncthreads();
  if (ty == 0) {
    double a = 0.0, b = 0.0;
#pragma unroll
    for (int k = 0; k < 8; ++k) { a += sh[k][threadIdx.x][0]; b += sh[k][threadIdx.x][1]; }
    atomicAdd(sums + c * 2, a); atomicAdd(sums + c * 2 + 1, b);
  }
}

// dpos[n,c] = sum_b dx[b,n,c]
__global__ void pos_grad_kernel(const float* __restrict__ dx, float* __restrict__ dpos, int B, long per) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= per) return;
  float s = 0.f;
  for (int b = 0; b < B; ++b) s += dx[(long)b * per + i];
  dpos[i] = s;
}

// ------------------------------------------------------------------------------------------------
// LayerNorm forward / backward (one warp per row, lane owns columns lane + 32 j)
// ------------------------------------------------------------------------------------------------
template <typename OT, int D>
__global__ void __launch_bounds__(256)
ln_fwd_kernel(const float* __restrict__ x, OT* __restrict__ y, const float* __restrict__ gamma,
              const float* __restrict__ beta, long rows, float eps) {
  constexpr int VPT = D / 32;
  const long row = (long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  float v[VPT];
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < VPT; ++j) { v[j] = x[row * D + lane + 32 * j]; s += v[j]; }
  const float mean = warp_sum(s) * (1.0f / D);
  float q = 0.f;
#pragma unroll
  for (int j = 0; j < VPT; ++j) { const float d = v[j] - mean; q = fmaf(d, d, q); }
  const float rstd = rsqrtf(warp_sum(q) * (1.0f / D) + eps);
#pragma unroll
  for (int j = 0; j < VPT; ++j) {
    const int c = lane + 32 * j;
    y[row * D + c] = from_f32<OT>((v[j] - mean) * rstd * gamma[c] + beta[c]);
  }
}

template <typename OT>
int launch_ln_fwd(const float* x, OT* y, const float* gamma, const float* beta, long rows, int D, float eps, cudaStream_t st) {
  const int grid = cdiv(rows, 8);
  MrnbProfScope prof(MRNB_PROF_LN, st, 0.0, (double)rows * D * (4 + sizeof(OT)));
  switch (D) {
    case 64: ln_fwd_kernel<OT, 64><<<grid, 256, 0, st>>>(x, y, gamma, beta, rows, eps); break;
    case 128: ln_fwd_kernel<OT, 128><<<grid, 256, 0, st>>>(x, y, gamma, beta, rows, eps); break;
    case 256: ln_fwd_kernel<OT, 256><<<grid, 256, 0, st>>>(x, y, gamma, beta, rows, eps); break;
    case 512: ln_fwd_kernel<OT, 512><<<grid, 256, 0, st>>>(x, y, gamma, beta, rows, eps); break;
    default: mrnb_set_error("ln_fwd: unsupported D=%d", D); return MRNB_ERR_UNSUPPORTED;
  }
  MRNB_CHECK_LAUNCH("ln_fwd_kernel");
  return MRNB_OK;
}

// dx = add + rstd * (g*dy - mean(g*dy) - xhat * mean(g*dy*xhat));  dgamma += sum dy*xhat;  dbeta += sum dy.
// `add` (the gradient arriving over the residual connection) may be null and may alias dx.  Optional 16-bit copy of dx.
template <int D>
__global__ void __launch_bounds__(256)
ln_bwd_kernel(const float* __restrict__ x, const float* __restrict__ dy, const float* __restrict__ gamma,
              const float* add, float* dx, __nv_bfloat16* __restrict__ dx16, float* __restrict__ dgamma,
              float* __restrict__ dbeta, long rows, float eps, const float* __restrict__ scale16, int rows_per_scale) {
  constexpr int VPT = D / 32;
  __shared__ float red[8][D];
  const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
  float g[VPT], ag[VPT], ab[VPT];
#pragma unroll
  for (int j = 0; j < VPT; ++j) { g[j] = gamma[lane + 32 * j]; ag[j] = 0.f; ab[j] = 0.f; }
  for (long row = (long)blockIdx.x * 8 + wp; row < rows; row += (long)gridDim.x * 8) {
    float v[VPT], d[VPT];
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < VPT; ++j) { v[j] = x[row * D + lane + 32 * j]; d[j] = dy[row * D + lane + 32 * j]; s += v[j]; }
    const float mean = warp_sum(s) * (1.0f / D);
    float q = 0.f;
#pragma unroll
    for (int j = 0; j < VPT; ++j) { v[j] -= mean; q = fmaf(v[j], v[j], q); }
    const float rstd = rsqrtf(warp_sum(q) * (1.0f / D) + eps);
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int j = 0; j < VPT; ++j) {
      v[j] *= rstd;                                  // xhat
      ag[j] = fmaf(d[j], v[j], ag[j]); ab[j] += d[j];
      d[j] *= g[j];                                  // dxhat
      s1 += d[j]; s2 = fmaf(d[j], v[j], s2);
    }
    s1 = warp_sum(s1) * (1.0f / D); s2 = warp_sum(s2) * (1.0f / D);
#pragma unroll
    for (int j = 0; j < VPT; ++j) {
      const long o = row * D + lane + 32 * j;
      float r = rstd * (d[j] - s1 - v[j] * s2);
      if (add) r += add[o];
      dx[o] = r;
      if (dx16) dx16[o] = __float2bfloat16_rn(scale16 ? r * scale16[row / rows_per_scale] : r);
    }
  }
#pragma unroll
  for (int j = 0; j < VPT; ++j) red[wp][lane + 32 * j] = ag[j];
  __syncthreads();
  for (int c = threadIdx.x; c < D; c += 256) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += red[k][c];
    atomicAdd(dgamma + c, t);
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < VPT; ++j) red[wp][lane + 32 * j] = ab[j];
  __syncthreads();
  for (int c = threadIdx.x; c < D; c += 256) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += red[k][c];
    atomicAdd(dbeta + c, t);
  }
}

// dx16 (optional): 16-bit copy of dx, multiplied by scale16[row / rows_per_scale] when given -- the DropPath-scaled GEMM
// operand of the branch that consumes dx next
int launch_ln_bwd(const float* x, const float* dy, const float* gamma, const float* add, float* dx, __nv_bfloat16* dx16,
                  float* dgamma, float* dbeta, long rows, int D, float eps, cudaStream_t st, const float* scale16 = nullptr,
                  int rows_per_scale = 1) {
  int grid = cdiv(rows, 8 * 8);
  if (grid > 148 * 4) grid = 148 * 4;
  if (grid < 1) grid = 1;
  MrnbProfScope prof(MRNB_PROF_LN, st, 0.0, (double)rows * D * 16);
  switch (D) {
    case 64: ln_bwd_kernel<64><<<grid, 256, 0, st>>>(x, dy, gamma, add, dx, dx16, dgamma, dbeta, rows, eps, scale16, rows_per_scale); break;
    case 128: ln_bwd_kernel<128><<<grid, 256, 0, st>>>(x, dy, gamma, add, dx, dx16, dgamma, dbeta, rows, eps, scale16, rows_per_scale); break;
    case 256: ln_bwd_kernel<256><<<grid, 256, 0, st>>>(x, dy, gamma, add, dx, dx16, dgamma, dbeta, rows, eps, scale16, rows_per_scale); break;
    case 512: ln_bwd_kernel<512><<<grid, 256, 0, st>>>(x, dy, gamma, add, dx, dx16, dgamma, dbeta, rows, eps, scale16, rows_per_scale); break;
    default: mrnb_set_error("ln_bwd: unsupported D=%d", D); return MRNB_ERR_UNSUPPORTED;
  }
  MRNB_CHECK_LAUNCH("ln_bwd_kernel");
  return MRNB_OK;
}

// ------------------------------------------------------------------------------------------------
// Elementwise: GELU forward / backward, DropPath row scaling
// ------------------------------------------------------------------------------------------------
template <typename AT>
__global__ void gelu_fwd_kernel(const AT* __restrict__ pre, AT* __restrict__ act, long n4) {       // four elements per thread
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n4) return;
  if constexpr (sizeof(AT) == 4) {
    const float4 p = reinterpret_cast<const float4*>(pre)[i];
    reinterpret_cast<float4*>(act)[i] = make_float4(gelu_erf(p.x), gelu_erf(p.y), gelu_erf(p.z), gelu_erf(p.w));
  } else {
    const uint2 p = reinterpret_cast<const uint2*>(pre)[i];
    const __nv_bfloat162 a = *reinterpret_cast<const __nv_bfloat162*>(&p.x), b = *reinterpret_cast<const __nv_bfloat162*>(&p.y);
    __nv_bfloat162 h0 = __floats2bfloat162_rn(gelu_erf(__bfloat162float(a.x)), gelu_erf(__bfloat162float(a.y)));
    __nv_bfloat162 h1 = __floats2bfloat162_rn(gelu_erf(__bfloat162float(b.x)), gelu_erf(__bfloat162float(b.y)));
    reinterpret_cast<uint2*>(act)[i] = make_uint2(*reinterpret_cast<uint32_t*>(&h0), *reinterpret_cast<uint32_t*>(&h1));
  }
}
// d * GELU'(pre): fp32 in place (fp32 mode) or bf16 only (bf16 mode: the result is a GEMM operand and the source of the
// bias sum; the fp32 tensor is not written back).  Four elements per thread.
template <typename AT>
__global__ void gelu_bwd_kernel(const AT* __restrict__ pre, float* __restrict__ d, __nv_bfloat16* __restrict__ d16, long n4) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n4) return;
  const float4 g = reinterpret_cast<const float4*>(d)[i];
  float x[4];
  if constexpr (sizeof(AT) == 4) {
    const float4 p = reinterpret_cast<const float4*>(pre)[i];
    x[0] = p.x; x[1] = p.y; x[2] = p.z; x[3] = p.w;
  } else {
    const uint2 p = reinterpret_cast<const uint2*>(pre)[i];
    const __nv_bfloat162 a = *reinterpret_cast<const __nv_bfloat162*>(&p.x), b = *reinterpret_cast<const __nv_bfloat162*>(&p.y);
    x[0] = __bfloat162float(a.x); x[1] = __bfloat162float(a.y); x[2] = __bfloat162float(b.x); x[3] = __bfloat162float(b.y);
  }
  const float v0 = g.x * gelu_erf_grad(x[0]), v1 = g.y * gelu_erf_grad(x[1]), v2 = g.z * gelu_erf_grad(x[2]),
              v3 = g.w * gelu_erf_grad(x[3]);
  if (d16) {
    __nv_bfloat162 h0 = __floats2bfloat162_rn(v0, v1), h1 = __floats2bfloat162_rn(v2, v3);
    reinterpret_cast<uint2*>(d16)[i] = make_uint2(*reinterpret_cast<uint32_t*>(&h0), *reinterpret_cast<uint32_t*>(&h1));
  } else {
    reinterpret_cast<float4*>(d)[i] = make_float4(v0, v1, v2, v3);
  }
}
// bf16 mode: d16 <- d16 * GELU'(pre) in place (the fc2 input gradient leaves its GEMM as bf16; eight elements per thread)
__global__ void gelu_bwd16_kernel(const __nv_bfloat16* __restrict__ pre, __nv_bfloat16* __restrict__ d16, long n8) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n8) return;
  const uint4 p = reinterpret_cast<const uint4*>(pre)[i];
  uint4 g = reinterpret_cast<uint4*>(d16)[i];
  const uint32_t pw[4] = {p.x, p.y, p.z, p.w};
  uint32_t gw[4] = {g.x, g.y, g.z, g.w};
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const __nv_bfloat162 x = *reinterpret_cast<const __nv_bfloat162*>(&pw[k]);
    const __nv_bfloat162 d = *reinterpret_cast<const __nv_bfloat162*>(&gw[k]);
    __nv_bfloat162 o = __floats2bfloat162_rn(__bfloat162float(d.x) * gelu_erf_grad(__bfloat162float(x.x)),
                                             __bfloat162float(d.y) * gelu_erf_grad(__bfloat162float(x.y)));
    gw[k] = *reinterpret_cast<uint32_t*>(&o);
  }
  reinterpret_cast<uint4*>(d16)[i] = make_uint4(gw[0], gw[1], gw[2], gw[3]);
}
// y[r,:] = x[r,:] * scale[r / rows_per_scale]   (+ optional 16-bit copy); scale may be null (copy / cast only)
__global__ void scale_rows_kernel(const float* __restrict__ x, const float* __restrict__ scale, int rows_per_scale, int D,
                                  float* __restrict__ y, __nv_bfloat16* __restrict__ y16, long n) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float v = x[i] * (scale ? scale[(i / D) / rows_per_scale] : 1.f);
  if (y) y[i] = v;
  if (y16) y16[i] = __float2bfloat16_rn(v);
}

// ------------------------------------------------------------------------------------------------
// Attention, training flavour.  Forward = svtr.cu's attention_kernel + the row log-sum-exp; backward in two passes:
//   pass Q (thread per query, K/V of the head in smem):  D = dO.O,  dq = scale * sum_k p (dO.v_k - D) k_k
//   pass K (thread per key, scaled Q / dO of the head in smem): dv = sum_q p dO_q,  dk = sum_q p (dO_q.v - D_q) q_q
// with p = exp(q.k - lse_q).  The Local window (|dh| <= 3, |dw| <= 5, modules/svtr.py:116-128) is symmetric, so the
// queries that see key m are exactly the window around m.
// ------------------------------------------------------------------------------------------------
template <typename AT, bool LOCAL>
__global__ void __launch_bounds__(256)
attn_fwd_train_kernel(const AT* __restrict__ qkv, AT* __restrict__ out, float* __restrict__ lse, int N, int d, int heads,
                      int H, int W) {
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
  for (int n = tid; n < N; n += blockDim.x) {
    float q[32], acc[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) { q[j] = to_f32<AT>(base[(long)n * 3 * d + h * 32 + j]) * ATT_SCALE; acc[j] = 0.f; }
    float m = -INFINITY, l = 0.f;
    auto step = [&](int key) {
      const float4* kr = reinterpret_cast<const float4*>(sK + key * KV_LD);
      float s = 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 kk = kr[j];
        s = fmaf(q[4 * j], kk.x, s); s = fmaf(q[4 * j + 1], kk.y, s);
        s = fmaf(q[4 * j + 2], kk.z, s); s = fmaf(q[4 * j + 3], kk.w, s);
      }
      float p;
      if (s > m) {
        const float corr = expf(m - s);
        l *= corr;
#pragma unroll
        for (int j = 0; j < 32; ++j) acc[j] *= corr;
        m = s; p = 1.f;
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
      const int h0 = max(qh - 3, 0), h1 = min(qh + 3, H - 1), w0 = max(qw - 5, 0), w1 = min(qw + 5, W - 1);
      for (int kh = h0; kh <= h1; ++kh)
        for (int kw = w0; kw <= w1; ++kw) step(kh * W + kw);
    } else {
      for (int key = 0; key < N; ++key) step(key);
    }
    const float inv = 1.0f / l;
    AT* o = out + ((long)g * N + n) * d + h * 32;
#pragma unroll
    for (int j = 0; j < 32; ++j) o[j] = from_f32<AT>(acc[j] * inv);
    lse[((long)g * heads + h) * N + n] = m + logf(l);
  }
}

template <typename AT, typename GT, bool LOCAL>
__global__ void __launch_bounds__(256)
attn_bwd_q_kernel(const AT* __restrict__ qkv, const AT* __restrict__ o, const float* __restrict__ dO,
                  const float* __restrict__ lse, float* __restrict__ Dbuf, GT* __restrict__ dqkv, int N, int d, int heads,
                  int H, int W) {
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
  for (int n = tid; n < N; n += blockDim.x) {
    float q[32], go[32], dq[32];
    float Dn = 0.f;
    const long orow = ((long)g * N + n) * d + h * 32;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      q[j] = to_f32<AT>(base[(long)n * 3 * d + h * 32 + j]) * ATT_SCALE;
      go[j] = dO[orow + j];
      Dn = fmaf(go[j], to_f32<AT>(o[orow + j]), Dn);
      dq[j] = 0.f;
    }
    const float ls = lse[((long)g * heads + h) * N + n];
    Dbuf[((long)g * heads + h) * N + n] = Dn;
    auto step = [&](int key) {
      const float4* kr = reinterpret_cast<const float4*>(sK + key * KV_LD);
      const float4* vr = reinterpret_cast<const float4*>(sV + key * KV_LD);
      float s = 0.f, dp = 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 kk = kr[j], vv = vr[j];
        s = fmaf(q[4 * j], kk.x, s); s = fmaf(q[4 * j + 1], kk.y, s);
        s = fmaf(q[4 * j + 2], kk.z, s); s = fmaf(q[4 * j + 3], kk.w, s);
        dp = fmaf(go[4 * j], vv.x, dp); dp = fmaf(go[4 * j + 1], vv.y, dp);
        dp = fmaf(go[4 * j + 2], vv.z, dp); dp = fmaf(go[4 * j + 3], vv.w, dp);
      }
      const float ds = expf(s - ls) * (dp - Dn);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 kk = kr[j];
        dq[4 * j] = fmaf(ds, kk.x, dq[4 * j]); dq[4 * j + 1] = fmaf(ds, kk.y, dq[4 * j + 1]);
        dq[4 * j + 2] = fmaf(ds, kk.z, dq[4 * j + 2]); dq[4 * j + 3] = fmaf(ds, kk.w, dq[4 * j + 3]);
      }
    };
    if constexpr (LOCAL) {
      const int qh = n / W, qw = n % W;
      const int h0 = max(qh - 3, 0), h1 = min(qh + 3, H - 1), w0 = max(qw - 5, 0), w1 = min(qw + 5, W - 1);
      for (int kh = h0; kh <= h1; ++kh)
        for (int kw = w0; kw <= w1; ++kw) step(kh * W + kw);
    } else {
      for (int key = 0; key < N; ++key) step(key);
    }
    GT* dst = dqkv + ((long)g * N + n) * 3 * d + h * 32;
#pragma unroll
    for (int j = 0; j < 32; ++j) dst[j] = from_f32<GT>(dq[j] * ATT_SCALE);
  }
}

template <typename AT, typename GT, bool LOCAL>
__global__ void __launch_bounds__(256)
attn_bwd_kv_kernel(const AT* __restrict__ qkv, const float* __restrict__ dO, const float* __restrict__ lse,
                   const float* __restrict__ Dbuf, GT* __restrict__ dqkv, int N, int d, int heads, int H, int W) {
  extern __shared__ float sm[];
  float* sQ = sm;                                  // scaled queries
  float* sG = sm + (size_t)N * KV_LD;              // dO
  float* sL = sm + (size_t)2 * N * KV_LD;          // lse
  float* sD = sL + N;                              // D
  const int g = blockIdx.x, h = blockIdx.y, tid = threadIdx.x;
  const AT* base = qkv + (long)g * N * 3 * d;
  for (int k = tid; k < N * 32; k += blockDim.x) {
    const int n = k >> 5, j = k & 31;
    sQ[n * KV_LD + j] = to_f32<AT>(base[(long)n * 3 * d + h * 32 + j]) * ATT_SCALE;
    sG[n * KV_LD + j] = dO[((long)g * N + n) * d + h * 32 + j];
  }
  for (int n = tid; n < N; n += blockDim.x) {
    sL[n] = lse[((long)g * heads + h) * N + n];
    sD[n] = Dbuf[((long)g * heads + h) * N + n];
  }
  __syncthreads();
  for (int m = tid; m < N; m += blockDim.x) {
    float kx[32], vx[32], dk[32], dv[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      kx[j] = to_f32<AT>(base[(long)m * 3 * d + d + h * 32 + j]);
      vx[j] = to_f32<AT>(base[(long)m * 3 * d + 2 * d + h * 32 + j]);
      dk[j] = 0.f; dv[j] = 0.f;
    }
    auto step = [&](int qn) {
      const float4* qr = reinterpret_cast<const float4*>(sQ + qn * KV_LD);
      const float4* gr = reinterpret_cast<const float4*>(sG + qn * KV_LD);
      float s = 0.f, dp = 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 qq = qr[j], gg = gr[j];
        s = fmaf(qq.x, kx[4 * j], s); s = fmaf(qq.y, kx[4 * j + 1], s);
        s = fmaf(qq.z, kx[4 * j + 2], s); s = fmaf(qq.w, kx[4 * j + 3], s);
        dp = fmaf(gg.x, vx[4 * j], dp); dp = fmaf(gg.y, vx[4 * j + 1], dp);
        dp = fmaf(gg.z, vx[4 * j + 2], dp); dp = fmaf(gg.w, vx[4 * j + 3], dp);
      }
      const float p = expf(s - sL[qn]);
      const float ds = p * (dp - sD[qn]);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 qq = qr[j], gg = gr[j];
        dv[4 * j] = fmaf(p, gg.x, dv[4 * j]); dv[4 * j + 1] = fmaf(p, gg.y, dv[4 * j + 1]);
        dv[4 * j + 2] = fmaf(p, gg.z, dv[4 * j + 2]); dv[4 * j + 3] = fmaf(p, gg.w, dv[4 * j + 3]);
        dk[4 * j] = fmaf(ds, qq.x, dk[4 * j]); dk[4 * j + 1] = fmaf(ds, qq.y, dk[4 * j + 1]);
        dk[4 * j + 2] = fmaf(ds, qq.z, dk[4 * j + 2]); dk[4 * j + 3] = fmaf(ds, qq.w, dk[4 * j + 3]);
      }
    };
    if constexpr (LOCAL) {
      const int kh = m / W, kw = m % W;
      const int h0 = max(kh - 3, 0), h1 = min(kh + 3, H - 1), w0 = max(kw - 5, 0), w1 = min(kw + 5, W - 1);
      for (int qh = h0; qh <= h1; ++qh)
        for (int qw = w0; qw <= w1; ++qw) step(qh * W + qw);
    } else {
      for (int qn = 0; qn < N; ++qn) step(qn);
    }
    GT* dst = dqkv + ((long)g * N + m) * 3 * d + h * 32;
#pragma unroll
    for (int j = 0; j < 32; ++j) { dst[d + j] = from_f32<GT>(dk[j]); dst[2 * d + j] = from_f32<GT>(dv[j]); }
  }
}

template <typename AT>
int attention_train_fwd(const AT* qkv, AT* out, float* lse, int G, int N, int d, int heads, int H, int W, bool local,
                        cudaStream_t st) {
  const size_t smem = (size_t)2 * N * KV_LD * sizeof(float);
  static bool set = false;
  if (!set) {
    const int mx = 2 * 512 * KV_LD * 4;
    cudaFuncSetAttribute(attn_fwd_train_kernel<AT, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx);
    cudaFuncSetAttribute(attn_fwd_train_kernel<AT, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx);
    set = true;
  }
  MrnbProfScope prof(MRNB_PROF_ATTN, st, 0.0, 0.0);
  dim3 grid(G, heads);
  if (local) attn_fwd_train_kernel<AT, true><<<grid, 256, smem, st>>>(qkv, out, lse, N, d, heads, H, W);
  else attn_fwd_train_kernel<AT, false><<<grid, 256, smem, st>>>(qkv, out, lse, N, d, heads, H, W);
  MRNB_CHECK_LAUNCH("attn_fwd_train_kernel");
  return MRNB_OK;
}

template <typename AT, typename GT>
int attention_train_bwd(const AT* qkv, const AT* o, const float* dO, const float* lse, float* Dbuf, GT* dqkv, int G, int N,
                        int d, int heads, int H, int W, bool local, cudaStream_t st) {
  const size_t smem_q = (size_t)2 * N * KV_LD * sizeof(float);
  const size_t smem_k = smem_q + (size_t)2 * N * sizeof(float);
  static bool set = false;
  if (!set) {
    const int mq = 2 * 512 * KV_LD * 4, mk = mq + 2 * 512 * 4;
    cudaFuncSetAttribute(attn_bwd_q_kernel<AT, GT, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, mq);
    cudaFuncSetAttribute(attn_bwd_q_kernel<AT, GT, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, mq);
    cudaFuncSetAttribute(attn_bwd_kv_kernel<AT, GT, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, mk);
    cudaFuncSetAttribute(attn_bwd_kv_kernel<AT, GT, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, mk);
    set = true;
  }
  MrnbProfScope prof(MRNB_PROF_ATTN, st, 0.0, 0.0);
  dim3 grid(G, heads);
  if (local) {
    attn_bwd_q_kernel<AT, GT, true><<<grid, 256, smem_q, st>>>(qkv, o, dO, lse, Dbuf, dqkv, N, d, heads, H, W);
    MRNB_CHECK_LAUNCH("attn_bwd_q_kernel");
    attn_bwd_kv_kernel<AT, GT, true><<<grid, 256, smem_k, st>>>(qkv, dO, lse, Dbuf, dqkv, N, d, heads, H, W);
  } else {
    attn_bwd_q_kernel<AT, GT, false><<<grid, 256, smem_q, st>>>(qkv, o, dO, lse, Dbuf, dqkv, N, d, heads, H, W);
    MRNB_CHECK_LAUNCH("attn_bwd_q_kernel");
    attn_bwd_kv_kernel<AT, GT, false><<<grid, 256, smem_k, st>>>(qkv, dO, lse, Dbuf, dqkv, N, d, heads, H, W);
  }
  MRNB_CHECK_LAUNCH("attn_bwd_kv_kernel");
  return MRNB_OK;
}

// ------------------------------------------------------------------------------------------------
// Attention on the tensor cores (bf16 mode): probabilities materialised per (sample, head), every contraction a batched
// tcgen05 GEMM over groups g = b * heads + h (gemm_tc2.cu reads Q / K / V / dO as 32-wide head slices of the token rows).
//   forward : S = scale Q K^T (fp32) -> P = softmax(S + Local mask) (bf16, kept for the backward) -> O = P V
//   backward: dP = dO V^T -> dS = P (dP - D), D = dO.O -> dV = P^T dO, dQ = scale dS K, dK = scale dS^T Q
// The Local mixer (modules/svtr.py:116-128) is the same dense path with masked probabilities set to zero.
// ------------------------------------------------------------------------------------------------
int attn_tc_forward(const bf16* qkv, bf16* P, bf16* att, int B, int N, int d, int heads, int W, bool local, cudaStream_t st) {
  const long GH = (long)B * heads;
  // P = softmax(scale Q K^T + Local mask): scores accumulate in TMEM and the row epilogue is fused (attn_train_tc.cu)
  MRNB_TRY(mrnb_attn_scores_softmax(qkv, P, B, N, d, heads, W, local ? 1 : 0, ATT_SCALE, st));
  MrnbTcGemm2 o{};
  o.a = mrnb_operand_k2d(P, N, N, N, 128, GH);
  o.b = mrnb_operand_head(qkv + 2 * d, N, 3L * d, heads, B, 1, 64);
  o.out16 = att; o.cm = mrnb_axis(d); o.cn = mrnb_axis(1); o.g_inner = heads; o.c_gstride = (long)N * d; o.c_gstride2 = 32;
  o.M = N; o.N = 32; o.K = N; o.groups = (int)GH; o.splitk = 1; o.alpha = 1.f;
  return mrnb_tc_gemm2(o, st);
}

int attn_tc_backward(const bf16* qkv, const bf16* att, const float* dO, const bf16* dO16, const bf16* P, bf16* dS,
                     bf16* dqkv, int B, int N, int d, int heads, cudaStream_t st) {
  const long GH = (long)B * heads;
  // dS = P (dO V^T - dO.O): dP accumulates in TMEM, fused row epilogue
  MRNB_TRY(mrnb_attn_dp_ds(dO16, qkv, dO, att, P, dS, B, N, d, heads, st));
  auto head_out = [&](MrnbTcGemm2& q, int col0, float alpha) {
    q.out16 = dqkv + col0; q.cm = mrnb_axis(3L * d); q.cn = mrnb_axis(1); q.g_inner = heads; q.c_gstride = (long)N * 3 * d;
    q.c_gstride2 = 32; q.M = N; q.N = 32; q.K = N; q.groups = (int)GH; q.splitk = 1; q.alpha = alpha;
  };
  MrnbTcGemm2 dv{};                                   // dV = P^T dO
  dv.a = mrnb_operand_mn2d(P, N, N, N, GH);
  dv.b = mrnb_operand_head(dO16, N, d, heads, B, 1, 64);
  head_out(dv, 2 * d, 1.f);
  MRNB_TRY(mrnb_tc_gemm2(dv, st));
  MrnbTcGemm2 dq{};                                   // dQ = scale dS K
  dq.a = mrnb_operand_k2d(dS, N, N, N, 128, GH);
  dq.b = mrnb_operand_head(qkv + d, N, 3L * d, heads, B, 1, 64);
  head_out(dq, 0, ATT_SCALE);
  MRNB_TRY(mrnb_tc_gemm2(dq, st));
  MrnbTcGemm2 dk{};                                   // dK = scale dS^T Q
  dk.a = mrnb_operand_mn2d(dS, N, N, N, GH);
  dk.b = mrnb_operand_head(qkv, N, 3L * d, heads, B, 1, 64);
  head_out(dk, d, ATT_SCALE);
  return mrnb_tc_gemm2(dk, st);
}

// ------------------------------------------------------------------------------------------------
// Workspace
// ------------------------------------------------------------------------------------------------
template <typename AT>
struct TrainWs {
  float *colf, *raw0, *act0, *raw1, *ss, *mr;
  double *stats, *bsums;
  float* stage_in[3];
  float *xmid[12], *xout[12], *lse[12];
  AT *ln1[12], *ln2[12], *qkv[12], *att[12], *hpre[12], *hact[12];
  float* cv[3];
  AT *vis, *feat, *big;
  // backward scratch
  float *dxa, *dy, *dbig, *dqkv, *datt, *dln, *Dbuf, *dfeat;
  bf16 *dy16, *dbig16, *dqkv16, *dfeat16, *dlog16, *datt16;   // bf16 mode: GEMM-operand copies of the gradients
  bf16 *P[12], *dS16;                                    // bf16 mode: attention probabilities (kept), dS scratch
  bf16* w0pad16; float* dw0pad;                          // bf16 mode: conv0 weight [32,64] (36 taps zero padded) / its gradient
  size_t bytes;
};

template <typename AT>
TrainWs<AT> carve_train_ws(char* base, int B, int n_class) {
  TrainWs<AT> w{};
  Workspace W{base, 0, (size_t)-1};
  const size_t u = (size_t)B * 32768;
  w.colf = W.take<float>(u * 9 / 2);
  w.raw0 = W.take<float>((size_t)B * 2048 * 32);
  w.act0 = W.take<float>((size_t)B * 2048 * 32);
  w.raw1 = W.take<float>(u);
  w.ss = W.take<float>(96 * 2);
  w.mr = W.take<float>(96 * 2);
  w.stats = W.take<double>(96 * 2);
  w.bsums = W.take<double>(96 * 2);
  for (int s = 0; s < 3; ++s) { w.stage_in[s] = W.take<float>(u); w.cv[s] = W.take<float>(u); }
  for (int k = 0; k < 12; ++k) {
    w.xmid[k] = W.take<float>(u); w.xout[k] = W.take<float>(u); w.lse[k] = W.take<float>(u / 32);
    w.ln1[k] = W.take<AT>(u); w.ln2[k] = W.take<AT>(u); w.qkv[k] = W.take<AT>(u * 3); w.att[k] = W.take<AT>(u);
    w.hpre[k] = W.take<AT>(u * 4); w.hact[k] = W.take<AT>(u * 4);
  }
  w.vis = W.take<AT>(u);
  w.feat = W.take<AT>((size_t)B * 64 * 256);
  w.big = W.take<AT>(u * 9 / 2);
  w.dxa = W.take<float>(u); w.dy = W.take<float>(u * 2); w.dbig = W.take<float>(u * 9 / 2);
  w.datt = W.take<float>(u); w.dln = W.take<float>(u); w.Dbuf = W.take<float>(u / 32);
  w.dfeat = W.take<float>((size_t)B * 64 * 256);
  if (sizeof(AT) == 4) {
    w.dqkv = W.take<float>(u * 3);
  } else {
    w.dy16 = W.take<bf16>(u); w.dbig16 = W.take<bf16>(u * 4); w.dqkv16 = W.take<bf16>(u * 3);
    w.dfeat16 = W.take<bf16>((size_t)B * 64 * 256);
    w.dlog16 = W.take<bf16>((size_t)B * 64 * ((n_class + 7) / 8 * 8));
    w.datt16 = W.take<bf16>(u);
    int k = 0;
    for (int s = 0; s < 3; ++s)
      for (int j = 0; j < DEPTH[s]; ++j, ++k) w.P[k] = W.take<bf16>((size_t)B * 32768 / DIMS[s] * (32768 / DIMS[s]) * HEADS[s]);
    w.dS16 = W.take<bf16>((size_t)B * 2 * 512 * 512);
    w.w0pad16 = W.take<bf16>(32 * 64); w.dw0pad = W.take<float>(32 * 64);
  }
  w.bytes = W.off + 4096;
  return w;
}

inline float* gp(const MrnbSvtrPack& G, int slot) { return const_cast<float*>(G.p[slot]); }

// ------------------------------------------------------------------------------------------------
// Forward
// ------------------------------------------------------------------------------------------------
template <typename AT>
int train_forward_t(const MrnbSvtrPack& P, const float* image, int B, int bn_batch, int update_running,
                    const float* drop /*[12,2,B] or null*/, float* logits, long ld, void* ws, size_t ws_bytes,
                    cudaStream_t st) {
  TrainWs<AT> w = carve_train_ws<AT>((char*)ws, B, P.n_class[0]);
  MRNB_CHECK_ARG(ws_bytes >= w.bytes, "svtr_train_forward: workspace too small (%zu < %zu)", ws_bytes, w.bytes);
  const long u = (long)B * 32768;
  // ---- patch embedding: conv0 -> BN -> GELU -> conv1 -> BN -> GELU -> + pos_embed.  bf16 mode: both convolutions are
  //      bf16 im2col x tcgen05 GEMM (K = 36 zero-padded to 64, K = 288 rounded up by TMA zero-fill) with fp32 outputs;
  //      the BatchNorm statistics are taken from those fp32 outputs in fp64.
  if (bn_batch) cudaMemsetAsync(w.stats, 0, 96 * 2 * sizeof(double), st);
  {
    mrnb_prof_begin(MRNB_PROF_CONV, st, 0.0, 0.0);
    if constexpr (sizeof(AT) == 2) {
      // conv0 (K = 36) on the tensor cores: bf16 im2col zero-padded to one 64-wide k-block, N = 32 inside a 64-wide tile
      const long rows0 = (long)B * 2048;
      im2col_img_pad64_kernel<<<cdiv(rows0 * 8, 256), 256, 0, st>>>(image, w.big, rows0);
      MRNB_CHECK_LAUNCH("im2col_img_pad64_kernel");
      pad_w0_kernel<<<8, 256, 0, st>>>(P.p[MRNB_P_CONV0_W], w.w0pad16, 32);
      MRNB_CHECK_LAUNCH("pad_w0_kernel");
      MrnbTcGemm2 g0{};
      g0.a = mrnb_operand_k2d(w.big, rows0, 64, 64, 128, 1);
      g0.b = mrnb_operand_k2d(w.w0pad16, 32, 64, 64, 64, 1);
      g0.out32 = w.raw0; g0.cm = mrnb_axis(32); g0.cn = mrnb_axis(1); g0.bias_n = P.p[MRNB_P_CONV0_B];
      g0.M = (int)rows0; g0.N = 32; g0.K = 64; g0.groups = 1; g0.splitk = 1; g0.alpha = 1.f;
      MRNB_TRY(mrnb_tc_gemm2(g0, st));
    } else {
      const long total = (long)B * 2048 * 36;
      im2col_img_kernel<<<cdiv(total, 256), 256, 0, st>>>(image, w.colf, total);
      MRNB_CHECK_LAUNCH("im2col_img_kernel");
      MrnbGemm g = mrnb_gemm_nt(w.colf, 36, P.p[MRNB_P_CONV0_W], 36, w.raw0, 32, B * 2048, 32, 36);
      g.bias_n = P.p[MRNB_P_CONV0_B];
      MRNB_TRY(mrnb_sgemm(g, st));
    }
    if (bn_batch) MRNB_TRY(launch_colstats(w.raw0, (long)B * 2048, 32, w.stats, st));
    bn_finalize_kernel<<<1, 64, 0, st>>>(w.stats, P.p[MRNB_P_BN0_W], P.p[MRNB_P_BN0_B], (float*)P.p[MRNB_P_BN0_MEAN],
                                         (float*)P.p[MRNB_P_BN0_VAR], w.ss, w.mr, 1, 32, (double)B * 2048, bn_batch != 0,
                                         update_running != 0, 1e-5f);
    MRNB_CHECK_LAUNCH("bn_finalize_kernel");
    const long t4 = (long)B * 2048 * 32 / 4;
    bn_gelu_kernel<<<cdiv(t4, 256), 256, 0, st>>>(w.raw0, w.ss, nullptr, 1, w.act0, 32, t4);
    MRNB_CHECK_LAUNCH("bn_gelu_kernel");
    if constexpr (sizeof(AT) == 2) {
      // conv1 (K = 288) on the tensor cores: bf16 im2col, the contraction rounded up to 320 (TMA zero-fills both operands)
      MRNB_CHECK_ARG(P.h[MRNB_P_CONV1_W], "svtr_train: bf16 mode needs the 16-bit weight shadow");
      MRNB_TRY(launch_im2col<AT>(w.act0, w.big, 16, 128, 32, 3, 3, 1, 2, 2, 8, 64, (long)B * 512, st));
      MrnbTcGemm2 g1{};
      g1.a = mrnb_operand_k2d(w.big, (long)B * 512, 288, 288, 128, 1);
      g1.b = mrnb_operand_k2d(P.h[MRNB_P_CONV1_W], 64, 288, 288, 64, 1);
      g1.out32 = w.raw1; g1.cm = mrnb_axis(64); g1.cn = mrnb_axis(1); g1.bias_n = P.p[MRNB_P_CONV1_B];
      g1.M = B * 512; g1.N = 64; g1.K = 320; g1.groups = 1; g1.splitk = 1; g1.alpha = 1.f;
      MRNB_TRY(mrnb_tc_gemm2(g1, st));
    } else {
      MRNB_TRY(launch_im2col<float>(w.act0, w.colf, 16, 128, 32, 3, 3, 1, 2, 2, 8, 64, (long)B * 512, st));
      MrnbGemm g1 = mrnb_gemm_nt(w.colf, 288, P.p[MRNB_P_CONV1_W], 288, w.raw1, 64, B * 512, 64, 288);
      g1.bias_n = P.p[MRNB_P_CONV1_B];
      MRNB_TRY(mrnb_sgemm(g1, st));
    }
    if (bn_batch) MRNB_TRY(launch_colstats(w.raw1, (long)B * 512, 64, w.stats + 64, st));
    bn_finalize_kernel<<<1, 64, 0, st>>>(w.stats + 64, P.p[MRNB_P_BN1_W], P.p[MRNB_P_BN1_B], (float*)P.p[MRNB_P_BN1_MEAN],
                                         (float*)P.p[MRNB_P_BN1_VAR], w.ss + 64, w.mr + 64, 1, 64, (double)B * 512,
                                         bn_batch != 0, update_running != 0, 1e-5f);
    MRNB_CHECK_LAUNCH("bn_finalize_kernel");
    bn_gelu_kernel<<<cdiv(u / 4, 256), 256, 0, st>>>(w.raw1, w.ss + 64, P.p[MRNB_P_POS_EMBED], 512, w.stage_in[0], 64, u / 4);
    MRNB_CHECK_LAUNCH("bn_gelu_kernel");
    mrnb_prof_end(MRNB_PROF_CONV, st);
  }
  int blk = 0;
  for (int s = 0; s < 3; ++s) {
    const int d = DIMS[s], N = 32768 / d, heads = HEADS[s], H = GH[s], Wd = 64;
    const int rows = B * N;
    for (int j = 0; j < DEPTH[s]; ++j, ++blk) {
      const int pb = MRNB_P_BLOCK0 + blk * MRNB_PB_COUNT;
      const float* xin = j == 0 ? w.stage_in[s] : w.xout[blk - 1];
      MRNB_TRY(launch_ln_fwd<AT>(xin, w.ln1[blk], P.p[pb + MRNB_PB_NORM1_W], P.p[pb + MRNB_PB_NORM1_B], rows, d, 1e-6f, st));
      MRNB_TRY(lin<AT>(w.ln1[blk], d, P.p[pb + MRNB_PB_QKV_W], P.h[pb + MRNB_PB_QKV_W], P.p[pb + MRNB_PB_QKV_B], w.qkv[blk],
                       3 * d, false, rows, 3 * d, d, nullptr, nullptr, 1, st));
      if constexpr (sizeof(AT) == 2)
        MRNB_TRY(attn_tc_forward(w.qkv[blk], w.P[blk], w.att[blk], B, N, d, heads, Wd, blk < 6, st));
      else
        MRNB_TRY(attention_train_fwd<AT>(w.qkv[blk], w.att[blk], w.lse[blk], B, N, d, heads, H, Wd, blk < 6, st));
      MRNB_TRY(lin<AT>(w.att[blk], d, P.p[pb + MRNB_PB_PROJ_W], P.h[pb + MRNB_PB_PROJ_W], P.p[pb + MRNB_PB_PROJ_B],
                       w.xmid[blk], d, true, rows, d, d, xin, drop ? drop + ((size_t)blk * 2 + 0) * B : nullptr, N, st));
      MRNB_TRY(launch_ln_fwd<AT>(w.xmid[blk], w.ln2[blk], P.p[pb + MRNB_PB_NORM2_W], P.p[pb + MRNB_PB_NORM2_B], rows, d, 1e-6f, st));
      MRNB_TRY(lin<AT>(w.ln2[blk], d, P.p[pb + MRNB_PB_FC1_W], P.h[pb + MRNB_PB_FC1_W], P.p[pb + MRNB_PB_FC1_B], w.hpre[blk],
                       4 * d, false, rows, 4 * d, d, nullptr, nullptr, 1, st));
      const long n4 = (long)rows * d;                      // rows * 4d elements, four per thread
      gelu_fwd_kernel<AT><<<cdiv(n4, 256), 256, 0, st>>>(w.hpre[blk], w.hact[blk], n4);
      MRNB_CHECK_LAUNCH("gelu_fwd_kernel");
      MRNB_TRY(lin<AT>(w.hact[blk], 4 * d, P.p[pb + MRNB_PB_FC2_W], P.h[pb + MRNB_PB_FC2_W], P.p[pb + MRNB_PB_FC2_B],
                       w.xout[blk], d, true, rows, d, 4 * d, w.xmid[blk], drop ? drop + ((size_t)blk * 2 + 1) * B : nullptr, N, st));
    }
    // SubSample: conv 3x3 stride (2,1) -> LN(eps 1e-5)
    const int Co = OUTS[s], Ho = H / 2;
    const int orows = B * Ho * Wd;
    const int ps = MRNB_P_SUB0 + s * MRNB_PS_COUNT;
    MRNB_TRY(launch_im2col<AT>(w.xout[blk - 1], w.big, H, Wd, d, 3, 3, 1, 2, 1, Ho, Wd, (long)orows, st));
    MRNB_TRY(lin<AT>(w.big, 9 * d, P.p[ps + MRNB_PS_CONV_W], P.h[ps + MRNB_PS_CONV_W], P.p[ps + MRNB_PS_CONV_B], w.cv[s], Co,
                     true, orows, Co, 9 * d, nullptr, nullptr, 1, st));
    if (s < 2) MRNB_TRY(launch_ln_fwd<float>(w.cv[s], w.stage_in[s + 1], P.p[ps + MRNB_PS_NORM_W], P.p[ps + MRNB_PS_NORM_B], orows, Co, 1e-5f, st));
    else MRNB_TRY(launch_ln_fwd<AT>(w.cv[s], w.vis, P.p[ps + MRNB_PS_NORM_W], P.p[ps + MRNB_PS_NORM_B], orows, Co, 1e-5f, st));
  }
  const int M = B * 64;
  MRNB_TRY(lin<AT>(w.vis, 512, P.p[MRNB_P_SEQ_W], P.h[MRNB_P_SEQ_W], P.p[MRNB_P_SEQ_B], w.feat, 256, false, M, 256, 512,
                   nullptr, nullptr, 1, st));
  MRNB_TRY(lin<AT>(w.feat, 256, P.fc_w[0], P.fc_w16[0], P.fc_b[0], logits, ld, true, M, P.n_class[0], 256, nullptr, nullptr, 1, st));
  return MRNB_OK;
}

// ------------------------------------------------------------------------------------------------
// Backward.  G holds the gradient pointers in the same slots; the caller passes the flat gradient arena so that it is
// zeroed with one memset (split-K GEMMs, LayerNorm / bias sums accumulate with atomics).
// ------------------------------------------------------------------------------------------------
template <typename AT>
int train_backward_t(const MrnbSvtrPack& P, const MrnbSvtrPack& G, const float* image, const float* dlogits, long ldg,
                     int B, int bn_batch, const float* drop, float* grad_arena, long n_arena, void* ws, size_t ws_bytes,
                     cudaStream_t st) {
  constexpr bool TC = sizeof(AT) == 2;
  TrainWs<AT> w = carve_train_ws<AT>((char*)ws, B, P.n_class[0]);
  MRNB_CHECK_ARG(ws_bytes >= w.bytes, "svtr_train_backward: workspace too small (%zu < %zu)", ws_bytes, w.bytes);
  cudaMemsetAsync(grad_arena, 0, (size_t)n_arena * sizeof(float), st);
  const long u = (long)B * 32768;
  const int M = B * 64, C = P.n_class[0];
  // ---- CTC head and the 512 -> 256 Linear
  Grad dlog{dlogits, nullptr, ldg};
  if (TC) {
    const long ld16 = (C + 7) / 8 * 8;
    const long total = (long)M * ld16;
    cast_pad_rows_kernel<<<cdiv(total / 8, 256), 256, 0, st>>>(dlogits, ldg, C, w.dlog16, ld16, total);
    MRNB_CHECK_LAUNCH("cast_pad_rows_kernel");
    dlog = Grad{dlogits, w.dlog16, ld16};
  }
  MRNB_TRY(launch_colsum<float>(dlogits, ldg, M, C, const_cast<float*>(G.fc_b[0]), st));
  MRNB_TRY(gemm_dw<AT>(dlog, w.feat, 256, const_cast<float*>(G.fc_w[0]), M, C, 256, st));
  MRNB_TRY(gemm_dx<AT>(dlog, P.fc_w[0], P.fc_w16[0], w.dfeat, w.dfeat16, 256, M, C, 256, st));
  Grad dfe{w.dfeat, w.dfeat16, 256};
  MRNB_TRY(launch_colsum<float>(w.dfeat, 256, M, 256, gp(G, MRNB_P_SEQ_B), st));
  MRNB_TRY(gemm_dw<AT>(dfe, w.vis, 512, gp(G, MRNB_P_SEQ_W), M, 256, 512, st));
  MRNB_TRY(gemm_dx<AT>(dfe, P.p[MRNB_P_SEQ_W], P.h[MRNB_P_SEQ_W], w.dln, nullptr, 512, M, 256, 512, st));       // d vis
  float* dx = w.dxa;          // gradient w.r.t. the residual stream
  float* dcv = w.dy;          // gradient w.r.t. a SubSample conv output (+ its 16-bit copy in dy16)
  {
    const int ps = MRNB_P_SUB0 + 2 * MRNB_PS_COUNT;
    MRNB_TRY(launch_ln_bwd(w.cv[2], w.dln, P.p[ps + MRNB_PS_NORM_W], nullptr, dcv, w.dy16, gp(G, ps + MRNB_PS_NORM_W),
                           gp(G, ps + MRNB_PS_NORM_B), M, 512, 1e-5f, st));
  }
  int blk = 12;
  bool dy16_ready = false;      // bf16 mode: w.dy16 already holds the scaled operand of the next branch
  for (int s = 2; s >= 0; --s) {
    const int d = DIMS[s], N = 32768 / d, heads = HEADS[s], H = GH[s], Wd = 64;
    const int rows = B * N;
    const int Co = OUTS[s], Ho = H / 2;
    dy16_ready = false;         // the stage starts from the col2im output
    const int orows = B * Ho * Wd;
    const int ps = MRNB_P_SUB0 + s * MRNB_PS_COUNT;
    // ---- SubSample conv backward (im2col recomputed from the stage output)
    {
      Grad gcv{dcv, w.dy16, Co};
      MRNB_TRY(launch_colsum<float>(dcv, Co, orows, Co, gp(G, ps + MRNB_PS_CONV_B), st));
      MRNB_TRY(launch_im2col<AT>(w.xout[blk - 1], w.big, H, Wd, d, 3, 3, 1, 2, 1, Ho, Wd, (long)orows, st));
      MRNB_TRY(gemm_dw<AT>(gcv, w.big, 9 * d, gp(G, ps + MRNB_PS_CONV_W), orows, Co, 9 * d, st));
      MRNB_TRY(gemm_dx<AT>(gcv, P.p[ps + MRNB_PS_CONV_W], P.h[ps + MRNB_PS_CONV_W], w.dbig, nullptr, 9 * d, orows, Co, 9 * d, st));
      col2im_nhwc_kernel<3, 3><<<cdiv(u / 4, 256), 256, 0, st>>>(w.dbig, dx, H, Wd, d, 1, 2, 1, Ho, Wd, u / 4);
      MRNB_CHECK_LAUNCH("col2im_nhwc_kernel");
    }
    for (int j = DEPTH[s] - 1; j >= 0; --j) {
      --blk;
      const int pb = MRNB_P_BLOCK0 + blk * MRNB_PB_COUNT;
      const float* xin = j == 0 ? w.stage_in[s] : w.xout[blk - 1];
      // ---- MLP branch: xout = xmid + ds1 * (GELU(LN2(xmid) W1^T + b1) W2^T + b2)
      Grad gy{dx, w.dy16, d};
      if (TC && dy16_ready) {
        // the LayerNorm backward that produced dx already wrote its DropPath-scaled bf16 copy
      } else if (drop || TC) {
        scale_rows_kernel<<<cdiv(u, 256), 256, 0, st>>>(dx, drop ? drop + ((size_t)blk * 2 + 1) * B : nullptr, N, d,
                                                        (drop && !TC) ? w.dy : nullptr, w.dy16, u);
        MRNB_CHECK_LAUNCH("scale_rows_kernel");
        if (drop && !TC) gy.f = w.dy;
      }
      if constexpr (TC) MRNB_TRY(launch_colsum<bf16>(w.dy16, d, rows, d, gp(G, pb + MRNB_PB_FC2_B), st));
      else MRNB_TRY(launch_colsum<float>(gy.f, d, rows, d, gp(G, pb + MRNB_PB_FC2_B), st));
      MRNB_TRY(gemm_dw<AT>(gy, w.hact[blk], 4 * d, gp(G, pb + MRNB_PB_FC2_W), rows, d, 4 * d, st));
      if constexpr (TC) {
        // d(GELU output) leaves the GEMM as bf16 only; GELU' is applied in place on the bf16 tensor
        MRNB_TRY(gemm_dx_tc(gy.h, gy.ld, P.h[pb + MRNB_PB_FC2_W], nullptr, w.dbig16, 4 * d, rows, d, 4 * d, st));
        gelu_bwd16_kernel<<<cdiv(u / 2, 256), 256, 0, st>>>(w.hpre[blk], w.dbig16, u / 2);
        MRNB_CHECK_LAUNCH("gelu_bwd16_kernel");
      } else {
        MRNB_TRY(gemm_dx<AT>(gy, P.p[pb + MRNB_PB_FC2_W], P.h[pb + MRNB_PB_FC2_W], w.dbig, nullptr, 4 * d, rows, d, 4 * d, st));
        gelu_bwd_kernel<AT><<<cdiv(u, 256), 256, 0, st>>>(w.hpre[blk], w.dbig, w.dbig16, u);
        MRNB_CHECK_LAUNCH("gelu_bwd_kernel");
      }
      Grad gh{w.dbig, w.dbig16, 4L * d};
      if constexpr (TC) MRNB_TRY(launch_colsum<bf16>(w.dbig16, 4 * d, rows, 4 * d, gp(G, pb + MRNB_PB_FC1_B), st));
      else MRNB_TRY(launch_colsum<float>(w.dbig, 4 * d, rows, 4 * d, gp(G, pb + MRNB_PB_FC1_B), st));
      MRNB_TRY(gemm_dw<AT>(gh, w.ln2[blk], d, gp(G, pb + MRNB_PB_FC1_W), rows, 4 * d, d, st));
      MRNB_TRY(gemm_dx<AT>(gh, P.p[pb + MRNB_PB_FC1_W], P.h[pb + MRNB_PB_FC1_W], w.dln, nullptr, d, rows, 4 * d, d, st));
      // (bf16 mode: the same pass emits the mixer branch's GEMM operand, dx * ds0, in bf16)
      MRNB_TRY(launch_ln_bwd(w.xmid[blk], w.dln, P.p[pb + MRNB_PB_NORM2_W], dx, dx, TC ? w.dy16 : nullptr,
                             gp(G, pb + MRNB_PB_NORM2_W), gp(G, pb + MRNB_PB_NORM2_B), rows, d, 1e-6f, st,
                             drop ? drop + ((size_t)blk * 2 + 0) * B : nullptr, N));
      // ---- mixer branch: xmid = xin + ds0 * (Attn(LN1(xin)) Wp^T + bp)
      gy = Grad{dx, w.dy16, d};
      if (drop && !TC) {
        scale_rows_kernel<<<cdiv(u, 256), 256, 0, st>>>(dx, drop + ((size_t)blk * 2 + 0) * B, N, d, w.dy, nullptr, u);
        MRNB_CHECK_LAUNCH("scale_rows_kernel");
        gy.f = w.dy;
      }
      if constexpr (TC) MRNB_TRY(launch_colsum<bf16>(w.dy16, d, rows, d, gp(G, pb + MRNB_PB_PROJ_B), st));
      else MRNB_TRY(launch_colsum<float>(gy.f, d, rows, d, gp(G, pb + MRNB_PB_PROJ_B), st));
      MRNB_TRY(gemm_dw<AT>(gy, w.att[blk], d, gp(G, pb + MRNB_PB_PROJ_W), rows, d, d, st));
      MRNB_TRY(gemm_dx<AT>(gy, P.p[pb + MRNB_PB_PROJ_W], P.h[pb + MRNB_PB_PROJ_W], w.datt, w.datt16, d, rows, d, d, st));
      Grad gq{w.dqkv, w.dqkv16, 3L * d};
      if constexpr (TC) {
        MRNB_TRY(attn_tc_backward(w.qkv[blk], w.att[blk], w.datt, w.datt16, w.P[blk], w.dS16, w.dqkv16, B, N, d, heads, st));
        MRNB_TRY(launch_colsum<bf16>(w.dqkv16, 3 * d, rows, 3 * d, gp(G, pb + MRNB_PB_QKV_B), st));
      } else {
        MRNB_TRY((attention_train_bwd<AT, float>(w.qkv[blk], w.att[blk], w.datt, w.lse[blk], w.Dbuf, w.dqkv, B, N, d, heads,
                                                 H, Wd, blk < 6, st)));
        MRNB_TRY(launch_colsum<float>(w.dqkv, 3 * d, rows, 3 * d, gp(G, pb + MRNB_PB_QKV_B), st));
      }
      MRNB_TRY(gemm_dw<AT>(gq, w.ln1[blk], d, gp(G, pb + MRNB_PB_QKV_W), rows, 3 * d, d, st));
      MRNB_TRY(gemm_dx<AT>(gq, P.p[pb + MRNB_PB_QKV_W], P.h[pb + MRNB_PB_QKV_W], w.dln, nullptr, d, rows, 3 * d, d, st));
      // (bf16 mode, not the first block of the stage: also emit dx * ds1 of the previous block, its MLP branch's operand)
      dy16_ready = TC && j > 0;
      MRNB_TRY(launch_ln_bwd(xin, w.dln, P.p[pb + MRNB_PB_NORM1_W], dx, dx, dy16_ready ? w.dy16 : nullptr,
                             gp(G, pb + MRNB_PB_NORM1_W), gp(G, pb + MRNB_PB_NORM1_B), rows, d, 1e-6f, st,
                             (drop && j > 0) ? drop + ((size_t)(blk - 1) * 2 + 1) * B : nullptr, N));
    }
    if (s > 0) {
      // stage input = LN(conv output of the previous merge)
      const int pq = MRNB_P_SUB0 + (s - 1) * MRNB_PS_COUNT;
      MRNB_TRY(launch_ln_bwd(w.cv[s - 1], dx, P.p[pq + MRNB_PS_NORM_W], nullptr, dcv, w.dy16, gp(G, pq + MRNB_PS_NORM_W),
                             gp(G, pq + MRNB_PS_NORM_B), rows, d, 1e-5f, st));
    }
  }
  // ---- patch embedding backward (fp32): dx is the gradient w.r.t. x0 = GELU(BN1(conv1)) + pos_embed
  {
    mrnb_prof_begin(MRNB_PROF_CONV, st, 0.0, 0.0);
    const long per = 512L * 64;
    pos_grad_kernel<<<cdiv(per, 256), 256, 0, st>>>(dx, gp(G, MRNB_P_POS_EMBED), B, per);
    MRNB_CHECK_LAUNCH("pos_grad_kernel");
    cudaMemsetAsync(w.bsums, 0, 96 * 2 * sizeof(double), st);
    const long r1 = (long)B * 512;
    int chunks = (int)(r1 / 256); if (chunks < 1) chunks = 1; if (chunks > 148) chunks = 148;
    bn_bwd_reduce_kernel<<<dim3(2, chunks), dim3(32, 8), 0, st>>>(w.raw1, dx, w.ss + 64, w.mr + 64, r1, 64, w.bsums + 64);
    MRNB_CHECK_LAUNCH("bn_bwd_reduce_kernel");
    bn_bwd_apply_kernel<<<cdiv(u, 256), 256, 0, st>>>(w.raw1, dx, w.ss + 64, w.mr + 64, w.bsums + 64, (double)r1, bn_batch,
                                                      gp(G, MRNB_P_BN1_W), gp(G, MRNB_P_BN1_B), 64, u, TC ? w.dy16 : nullptr);
    MRNB_CHECK_LAUNCH("bn_bwd_apply_kernel");
    MRNB_TRY(launch_colsum<float>(dx, 64, r1, 64, gp(G, MRNB_P_CONV1_B), st));
    if constexpr (TC) {
      MRNB_TRY(launch_im2col<AT>(w.act0, w.big, 16, 128, 32, 3, 3, 1, 2, 2, 8, 64, r1, st));
      MRNB_TRY(gemm_dw_tc(w.dy16, 64, w.big, 288, gp(G, MRNB_P_CONV1_W), (int)r1, 64, 288, st));
      MRNB_TRY(gemm_dx_tc(w.dy16, 64, P.h[MRNB_P_CONV1_W], w.dbig, nullptr, 288, (int)r1, 64, 288, st));
    } else {
      MRNB_TRY(launch_im2col<float>(w.act0, w.colf, 16, 128, 32, 3, 3, 1, 2, 2, 8, 64, r1, st));
      MRNB_TRY(gemm_dw_f32(dx, 64, w.colf, 288, gp(G, MRNB_P_CONV1_W), (int)r1, 64, 288, st));
      MRNB_TRY(gemm_dx_f32(dx, 64, P.p[MRNB_P_CONV1_W], w.dbig, 288, (int)r1, 64, 288, st));
    }
    float* dact0 = w.dy;                                   // [B,16,128,32]
    const long n0 = (long)B * 2048 * 32;
    col2im_nhwc_kernel<3, 3><<<cdiv(n0 / 4, 256), 256, 0, st>>>(w.dbig, dact0, 16, 128, 32, 1, 2, 2, 8, 64, n0 / 4);
    MRNB_CHECK_LAUNCH("col2im_nhwc_kernel");
    const long r0 = (long)B * 2048;
    chunks = (int)(r0 / 256); if (chunks < 1) chunks = 1; if (chunks > 148) chunks = 148;
    bn_bwd_reduce_kernel<<<dim3(1, chunks), dim3(32, 8), 0, st>>>(w.raw0, dact0, w.ss, w.mr, r0, 32, w.bsums);
    MRNB_CHECK_LAUNCH("bn_bwd_reduce_kernel");
    bn_bwd_apply_kernel<<<cdiv(n0, 256), 256, 0, st>>>(w.raw0, dact0, w.ss, w.mr, w.bsums, (double)r0, bn_batch,
                                                       gp(G, MRNB_P_BN0_W), gp(G, MRNB_P_BN0_B), 32, n0, TC ? w.dbig16 : nullptr);
    MRNB_CHECK_LAUNCH("bn_bwd_apply_kernel");
    MRNB_TRY(launch_colsum<float>(dact0, 32, r0, 32, gp(G, MRNB_P_CONV0_B), st));
    if constexpr (TC) {
      im2col_img_pad64_kernel<<<cdiv(r0 * 8, 256), 256, 0, st>>>(image, w.big, r0);
      MRNB_CHECK_LAUNCH("im2col_img_pad64_kernel");
      cudaMemsetAsync(w.dw0pad, 0, 32 * 64 * sizeof(float), st);
      MRNB_TRY(gemm_dw_tc(w.dbig16, 32, w.big, 64, w.dw0pad, (int)r0, 32, 64, st));
      unpad_dw0_kernel<<<5, 256, 0, st>>>(w.dw0pad, gp(G, MRNB_P_CONV0_W), 32);
      MRNB_CHECK_LAUNCH("unpad_dw0_kernel");
    } else {
      const long total = r0 * 36;
      im2col_img_kernel<<<cdiv(total, 256), 256, 0, st>>>(image, w.colf, total);
      MRNB_CHECK_LAUNCH("im2col_img_kernel");
      MRNB_TRY(gemm_dw_f32(dact0, 32, w.colf, 36, gp(G, MRNB_P_CONV0_W), (int)r0, 32, 36, st));
    }
    mrnb_prof_end(MRNB_PROF_CONV, st);
  }
  return MRNB_OK;
}

}  // namespace

extern "C" size_t mrnb_svtr_train_workspace_bytes(int B, int n_class, int prec) {
  return prec == MRNB_PREC_BF16 ? carve_train_ws<__nv_bfloat16>(nullptr, B, n_class).bytes
                                : carve_train_ws<float>(nullptr, B, n_class).bytes;
}

extern "C" int mrnb_svtr_train_forward(const MrnbSvtrPack* pack, const float* image, int B, int prec, int bn_batch_stats,
                                       int update_running, const float* drop_scales, float* logits, long ld_logits,
                                       void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  MRNB_CHECK_ARG(pack && image && logits && workspace && B > 0, "svtr_train_forward: null/empty argument");
  MRNB_CHECK_ARG(pack->n_experts == 1, "svtr_train_forward: the training pack holds exactly one expert");
  MRNB_CHECK_ARG(ld_logits >= pack->n_class[0], "svtr_train_forward: ld_logits < n_class");
  MRNB_CHECK_ARG(!bn_batch_stats || (long)B * 512 > 1, "svtr_train_forward: batch statistics need more than one value");
  for (int k = 0; k < MRNB_P_COUNT; ++k) MRNB_CHECK_ARG(pack->p[k], "svtr_train_forward: parameter slot %d is null", k);
  if (prec == MRNB_PREC_FP32)
    return train_forward_t<float>(*pack, image, B, bn_batch_stats, update_running, drop_scales, logits, ld_logits, workspace,
                                  workspace_bytes, stream);
  if (prec == MRNB_PREC_BF16)
    return train_forward_t<__nv_bfloat16>(*pack, image, B, bn_batch_stats, update_running, drop_scales, logits, ld_logits,
                                          workspace, workspace_bytes, stream);
  mrnb_set_error("svtr_train_forward: unknown precision %d", prec);
  return MRNB_ERR_ARG;
}

extern "C" int mrnb_svtr_train_backward(const MrnbSvtrPack* pack, const MrnbSvtrPack* grads, const float* image,
                                        const float* dlogits, long ld_dlogits, int B, int prec, int bn_batch_stats,
                                        const float* drop_scales, float* grad_arena, long n_arena, void* workspace,
                                        size_t workspace_bytes, cudaStream_t stream) {
  MRNB_CHECK_ARG(pack && grads && image && dlogits && grad_arena && workspace && B > 0, "svtr_train_backward: null/empty argument");
  MRNB_CHECK_ARG(pack->n_experts == 1 && grads->n_experts == 1, "svtr_train_backward: the training pack holds exactly one expert");
  for (int k = 0; k < MRNB_P_COUNT; ++k) {
    const bool stat = k == MRNB_P_BN0_MEAN || k == MRNB_P_BN0_VAR || k == MRNB_P_BN1_MEAN || k == MRNB_P_BN1_VAR;
    MRNB_CHECK_ARG(stat || grads->p[k], "svtr_train_backward: gradient slot %d is null", k);
  }
  MRNB_CHECK_ARG(grads->fc_w[0] && grads->fc_b[0], "svtr_train_backward: classifier gradient slots are null");
  if (prec == MRNB_PREC_FP32)
    return train_backward_t<float>(*pack, *grads, image, dlogits, ld_dlogits, B, bn_batch_stats, drop_scales, grad_arena,
                                   n_arena, workspace, workspace_bytes, stream);
  if (prec == MRNB_PREC_BF16)
    return train_backward_t<__nv_bfloat16>(*pack, *grads, image, dlogits, ld_dlogits, B, bn_batch_stats, drop_scales,
                                           grad_arena, n_arena, workspace, workspace_bytes, stream);
  mrnb_set_error("svtr_train_backward: unknown precision %d", prec);
  return MRNB_ERR_ARG;
}

// ---- C-ABI test entries: the bf16 training attention of one stage, forwarded unchanged to attn_tc_forward /
// attn_tc_backward so the score kernel and the four value-side head GEMMs can be compared with a reference on their own
extern "C" int mrnb_attn_tc_train_forward(const void* qkv, void* P, void* O, int B, int N, int d, int heads, int W, int local,
                                          cudaStream_t stream) {
  MRNB_CHECK_ARG(qkv && P && O && B > 0 && heads > 0 && d == 32 * heads, "attn_tc_train_forward: bad argument");
  return attn_tc_forward((const bf16*)qkv, (bf16*)P, (bf16*)O, B, N, d, heads, W, local != 0, stream);
}

extern "C" int mrnb_attn_tc_train_backward(const void* qkv, const void* O, const float* dO, const void* dO16, const void* P,
                                           void* dS, void* dqkv, int B, int N, int d, int heads, cudaStream_t stream) {
  MRNB_CHECK_ARG(qkv && O && dO && dO16 && P && dS && dqkv && B > 0 && heads > 0 && d == 32 * heads,
                 "attn_tc_train_backward: bad argument");
  return attn_tc_backward((const bf16*)qkv, (const bf16*)O, dO, (const bf16*)dO16, (const bf16*)P, (bf16*)dS, (bf16*)dqkv, B, N,
                          d, heads, stream);
}
