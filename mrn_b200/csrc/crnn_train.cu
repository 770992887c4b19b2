// Stage-0 expert training for ONE CRNN expert (VGG + 2 x BidirectionalLSTM + CTC head, T = 63): activation-keeping
// forward and the full backward -- convolution / pooling / BatchNorm gradients and BPTT through both LSTM layers.
//
// Reference (paths relative to /root/reference):
//   il_modules/mrn.py:225-279        _init_train (model(image, cross=False)['logits'] -> CTC -> backward)
//   modules/feature_extraction.py:19-47   VGG_FeatureExtractor (Sequential 0..19)
//   modules/sequence_modeling.py:4-22     BidirectionalLSTM (nn.LSTM bidirectional, gate order i,f,g,o; Linear 2H -> out)
//   modules/model.py:82-101,133-148       Model_Extractor.forward (permute / avg-pool over H = 1) / Model.forward (fc)
// torch.autograd derives the backward in the reference; here every gradient is written out by hand.
//
// Layout: activations NHWC fp32 [sample][h][w][c]; every convolution is im2col (AT: fp32 parity mode / bf16 tensor-core
// mode) x GEMM; LSTM tensors are [sample][t][...] with both directions side by side (gates [B,63,2048] = dir*1024 +
// gate*256 + unit, cell / hidden [B,63,512] = dir*256 + unit).  Parameters / gradients: MrnbCrnnTrainPack slots inside
// one flat arena (Adam, NCCL all-reduce); the two directions of each LSTM tensor are adjacent, so the input projection,
// its weight gradient and the input gradient are single GEMMs over both directions.
#include "common.cuh"
#include "train_util.cuh"
#include "svtr.h"

namespace {

constexpr int T63 = 63, HID = 256;

// ------------------------------------------------------------------------------------------------
// elementwise / layout kernels
// ------------------------------------------------------------------------------------------------
__global__ void nchw_to_nhwc4_kernel(const float* __restrict__ img, float* __restrict__ out, int HW, long total) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;       // one pixel
  if (i >= total) return;
  const long b = i / HW, p = i % HW;
  const float* s = img + b * 4 * HW + p;
  *reinterpret_cast<float4*>(out + i * 4) = make_float4(s[0], s[HW], s[2L * HW], s[3L * HW]);
}

// conv0 on the tensor cores (bf16 mode): 3x3 pad-1 im2col of the 4-channel NHWC image with the 36 taps zero-padded to
// K = 64 (one 128-byte swizzle row): col[(b,oh,ow), (kh,kw,c) | 0...].  Thread = (output pixel, group of 8 columns).
__global__ void im2col_c4_pad64_kernel(const float* __restrict__ x, bf16* __restrict__ col, int H, int W, long rows) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * 8) return;
  const int j = (int)(i & 7);
  long r = i >> 3;
  const int ow = (int)(r % W); r /= W;
  const int oh = (int)(r % H);
  const long b = r / H;
  float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int tap = 2 * j + h;
    if (tap < 9) {
      const int ih = oh - 1 + tap / 3, iw = ow - 1 + tap % 3;
      if (ih >= 0 && ih < H && iw >= 0 && iw < W) {
        const float4 t = *reinterpret_cast<const float4*>(x + ((b * H + ih) * W + iw) * 4);
        v[4 * h] = t.x; v[4 * h + 1] = t.y; v[4 * h + 2] = t.z; v[4 * h + 3] = t.w;
      }
    }
  }
  uint32_t pk[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    __nv_bfloat162 hh = __floats2bfloat162_rn(v[2 * u], v[2 * u + 1]);
    pk[u] = *reinterpret_cast<uint32_t*>(&hh);
  }
  *reinterpret_cast<uint4*>(col + i * 8) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
}
__global__ void relu_kernel(float* __restrict__ x, long n4) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n4) return;
  float4 v = reinterpret_cast<float4*>(x)[i];
  v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f);
  reinterpret_cast<float4*>(x)[i] = v;
}
// d <- d * (a > 0)   (+ optional 16-bit copy)
__global__ void relu_bwd_kernel(const float* __restrict__ a, float* __restrict__ d, bf16* __restrict__ d16, long n) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float v = a[i] > 0.f ? d[i] : 0.f;
  d[i] = v;
  if (d16) d16[i] = __float2bfloat16_rn(v);
}
// y = relu(raw * sc + sh)     [rows, C]
__global__ void bn_relu_kernel(const float* __restrict__ raw, const float* __restrict__ ss, float* __restrict__ y, int C, long n) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int c = (int)(i % C);
  y[i] = fmaxf(fmaf(raw[i], ss[c * 2], ss[c * 2 + 1]), 0.f);
}
// max-pool ph x pw (stride = window) over NHWC, four channels per thread
__global__ void maxpool_kernel(const float* __restrict__ x, float* __restrict__ y, int H, int W, int C, int ph, int pw, long total4) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total4) return;
  const int c4 = C / 4;
  const int c = (int)(i % c4) * 4;
  long r = i / c4;
  const int Wo = W / pw, Ho = H / ph;
  const int ow = (int)(r % Wo); r /= Wo;
  const int oh = (int)(r % Ho);
  const long b = r / Ho;
  float4 m = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
  for (int dy = 0; dy < ph; ++dy)
    for (int dx = 0; dx < pw; ++dx) {
      const float4 v = *reinterpret_cast<const float4*>(x + ((b * H + oh * ph + dy) * W + ow * pw + dx) * C + c);
      m.x = fmaxf(m.x, v.x); m.y = fmaxf(m.y, v.y); m.z = fmaxf(m.z, v.z); m.w = fmaxf(m.w, v.w);
    }
  *reinterpret_cast<float4*>(y + i * 4) = m;
}
// backward of relu -> max-pool: the first maximal element of each window receives the gradient if it is positive
// (windows do not overlap; ties among zeros are irrelevant because relu' = 0 there).  Four channels per thread.
__global__ void maxpool_relu_bwd_kernel(const float* __restrict__ a, const float* __restrict__ dy, float* __restrict__ da, int H,
                                        int W, int C, int ph, int pw, long total4) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total4) return;
  const int c4 = C / 4;
  const int c = (int)(i % c4) * 4;
  long r = i / c4;
  const int Wo = W / pw, Ho = H / ph;
  const int ow = (int)(r % Wo); r /= Wo;
  const int oh = (int)(r % Ho);
  const long b = r / Ho;
  float m[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
  int arg[4] = {0, 0, 0, 0};
  for (int dy_ = 0; dy_ < ph; ++dy_)
    for (int dx_ = 0; dx_ < pw; ++dx_) {
      const float4 v4 = *reinterpret_cast<const float4*>(a + ((b * H + oh * ph + dy_) * W + ow * pw + dx_) * C + c);
      const float v[4] = {v4.x, v4.y, v4.z, v4.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) if (v[k] > m[k]) { m[k] = v[k]; arg[k] = dy_ * pw + dx_; }
    }
  const float4 g4 = *reinterpret_cast<const float4*>(dy + i * 4);
  const float g[4] = {m[0] > 0.f ? g4.x : 0.f, m[1] > 0.f ? g4.y : 0.f, m[2] > 0.f ? g4.z : 0.f, m[3] > 0.f ? g4.w : 0.f};
  for (int dy_ = 0; dy_ < ph; ++dy_)
    for (int dx_ = 0; dx_ < pw; ++dx_) {
      const int p = dy_ * pw + dx_;
      *reinterpret_cast<float4*>(da + ((b * H + oh * ph + dy_) * W + ow * pw + dx_) * C + c) =
          make_float4(p == arg[0] ? g[0] : 0.f, p == arg[1] ? g[1] : 0.f, p == arg[2] ? g[2] : 0.f, p == arg[3] ? g[3] : 0.f);
    }
}

// BatchNorm backward (d already carries the relu mask): S1 = sum d, S2 = sum d * xhat per channel (fp64 atomics)
__global__ void __launch_bounds__(256)
bn_relu_bwd_reduce_kernel(const float* __restrict__ raw, const float* __restrict__ d, const float* __restrict__ mr, long rows,
                          int C, double* __restrict__ sums) {
  __shared__ double sh[8][32][2];
  const int c = blockIdx.x * 32 + threadIdx.x, ty = threadIdx.y;
  const long per = (rows + gridDim.y - 1) / gridDim.y;
  const long r0 = (long)blockIdx.y * per, r1 = (r0 + per < rows) ? r0 + per : rows;
  const float mean = mr[c * 2], rstd = mr[c * 2 + 1];
  double s1 = 0.0, s2 = 0.0;
  for (long r = r0 + ty; r < r1; r += 8) {
    const float dz = d[r * C + c];
    s1 += dz; s2 += (double)dz * ((raw[r * C + c] - mean) * rstd);
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
__global__ void add_vec_kernel(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ o, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) o[i] = a[i] + b[i];
}
// ------------------------------------------------------------------------------------------------
// LSTM cell, both directions per launch.  gates G [B,63,2048] hold the pre-activations on entry and the activated
// gates (sigmoid i, f, o; tanh g) on exit; c, rec [B,63,512].  Direction 0 walks t = s, direction 1 walks t = 62 - s.
// hseq (AT) [B,63,512] receives h at the NEXT position of each direction (the operand of the W_hh weight gradient).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }

template <typename AT>
__global__ void lstm_cell_fwd_kernel(float* __restrict__ G, float* __restrict__ c, float* __restrict__ rec, AT* __restrict__ hseq,
                                     int B, int s) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;            // (dir, b, j)
  if (i >= 2 * B * HID) return;
  const int j = i % HID, b = (i / HID) % B, dir = i / (HID * B);
  const int t = dir ? T63 - 1 - s : s, tp = dir ? t + 1 : t - 1, tn = dir ? t - 1 : t + 1;
  float* g = G + ((long)b * T63 + t) * 2048 + dir * 1024 + j;
  const float gi = sigmoidf_(g[0]), gf = sigmoidf_(g[HID]), gg = tanhf(g[2 * HID]), go = sigmoidf_(g[3 * HID]);
  g[0] = gi; g[HID] = gf; g[2 * HID] = gg; g[3 * HID] = go;
  const long o = ((long)b * T63 + t) * 512 + dir * HID + j;
  const float cp = s > 0 ? c[((long)b * T63 + tp) * 512 + dir * HID + j] : 0.f;
  const float cn = gf * cp + gi * gg;
  c[o] = cn;
  const float h = go * tanhf(cn);
  rec[o] = h;
  if (s < T63 - 1) hseq[((long)b * T63 + tn) * 512 + dir * HID + j] = from_f32<AT>(h);
}

// BPTT step s (direction 0 at t = 62 - s, direction 1 at t = s): dh = drec[t] + dh_next; writes the gate
// pre-activation gradients over the activated gates in G and carries dc.
__global__ void lstm_cell_bwd_kernel(float* __restrict__ G, const float* __restrict__ c, const float* __restrict__ drec,
                                     float* __restrict__ dhn, float* __restrict__ dcn, int B, int s,
                                     bf16* __restrict__ G16) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 2 * B * HID) return;
  const int j = i % HID, b = (i / HID) % B, dir = i / (HID * B);
  const int t = dir ? s : T63 - 1 - s, tp = dir ? t + 1 : t - 1;          // tp: the position this cell took c_prev from
  const bool has_prev = dir ? (t < T63 - 1) : (t > 0);
  float* g = G + ((long)b * T63 + t) * 2048 + dir * 1024 + j;
  const float gi = g[0], gf = g[HID], gg = g[2 * HID], go = g[3 * HID];
  const long o = ((long)b * T63 + t) * 512 + dir * HID + j;
  const float ct = c[o];
  const float cp = has_prev ? c[((long)b * T63 + tp) * 512 + dir * HID + j] : 0.f;
  const float dh = drec[o] + (s > 0 ? dhn[i] : 0.f);
  dhn[i] = 0.f;                       // the next step's split-K GEMM accumulates dh_next with reductions onto zero
  const float tc = tanhf(ct);
  const float dc = dh * go * (1.f - tc * tc) + (s > 0 ? dcn[i] : 0.f);
  const float ai = dc * gg * gi * (1.f - gi), af = dc * cp * gf * (1.f - gf), ag = dc * gi * (1.f - gg * gg),
              ao = dh * tc * go * (1.f - go);
  g[0] = ai; g[HID] = af; g[2 * HID] = ag; g[3 * HID] = ao;
  if (G16) {
    bf16* h = G16 + ((long)b * T63 + t) * 2048 + dir * 1024 + j;
    h[0] = __float2bfloat16_rn(ai); h[HID] = __float2bfloat16_rn(af); h[2 * HID] = __float2bfloat16_rn(ag);
    h[3 * HID] = __float2bfloat16_rn(ao);
  }
  dcn[i] = dc * gf;
}

// ------------------------------------------------------------------------------------------------
// Parameter slots (MrnbCrnnTrainPack in include/mrn_b200.h) and the VGG layer table
// ------------------------------------------------------------------------------------------------
struct ConvL { int H, W, Cin, Cout, KH, KW, pad, ph, pw, w_slot, b_slot, bn; };
static const ConvL LAYERS[7] = {
    {32, 256, 4, 64, 3, 3, 1, 2, 2, MRNB_T_CONV0_W, MRNB_T_CONV0_B, -1},
    {16, 128, 64, 128, 3, 3, 1, 2, 2, MRNB_T_CONV1_W, MRNB_T_CONV1_B, -1},
    {8, 64, 128, 256, 3, 3, 1, 1, 1, MRNB_T_CONV2_W, MRNB_T_CONV2_B, -1},
    {8, 64, 256, 256, 3, 3, 1, 2, 1, MRNB_T_CONV3_W, MRNB_T_CONV3_B, -1},
    {4, 64, 256, 512, 3, 3, 1, 1, 1, MRNB_T_CONV4_W, -1, 0},
    {4, 64, 512, 512, 3, 3, 1, 2, 1, MRNB_T_CONV5_W, -1, 1},
    {2, 64, 512, 512, 2, 2, 0, 1, 1, MRNB_T_CONV6_W, MRNB_T_CONV6_B, -1},
};
inline int out_h(const ConvL& l) { return l.H + 2 * l.pad - l.KH + 1; }
inline int out_w(const ConvL& l) { return l.W + 2 * l.pad - l.KW + 1; }

template <typename AT>
struct CrnnWs {
  float* img4;            // NHWC copy of the image
  float* act[7];          // post-activation conv outputs (pre-pool), NHWC
  float* raw[2];          // pre-BatchNorm outputs of conv4 / conv5
  float* pool[7];         // pooled outputs where the layer pools (else = act)
  float *ss, *mr; double *stats, *bsums;
  AT* col; float* dcol;   // im2col scratch / its gradient
  AT* vis16;              // conv6 output as a GEMM operand (bf16 mode)
  // LSTM (2 layers)
  float *G[2], *c[2], *rec[2]; AT *rec16[2], *hseq[2], *out16[2];
  float* bsum;            // [2][2048]  b_ih + b_hh
  float *dhn, *dcn;       // [2][B][256]
  float *d0, *d1;         // gradient ping-pong (largest activation)
  bf16 *d16, *dlog16, *dG16, *w0pad16;   // w0pad16: conv0 weight [64,64] (36 taps zero padded)
  float* dw0pad;                         // its gradient [64,64]
  float *dout, *drec;     // [B*63,256], [B*63,512]
  size_t bytes;
};

template <typename AT>
CrnnWs<AT> carve_crnn_ws(char* base, int B, int n_class) {
  CrnnWs<AT> w{};
  Workspace W{base, 0, (size_t)-1};
  const size_t b = (size_t)B;
  w.img4 = W.take<float>(b * 32 * 256 * 4);
  size_t max_act = 0, max_col = 0;
  for (int l = 0; l < 7; ++l) {
    const ConvL& L = LAYERS[l];
    const size_t n = b * out_h(L) * out_w(L) * L.Cout;
    w.act[l] = W.take<float>(n);
    if (L.bn >= 0) w.raw[L.bn] = W.take<float>(n);
    w.pool[l] = (L.ph * L.pw > 1) ? W.take<float>(n / (L.ph * L.pw)) : w.act[l];
    if (n > max_act) max_act = n;
    const size_t cn = b * out_h(L) * out_w(L) * L.KH * L.KW * L.Cin;
    if (cn > max_col) max_col = cn;
  }
  w.ss = W.take<float>(2 * 512 * 2); w.mr = W.take<float>(2 * 512 * 2);
  w.stats = W.take<double>(2 * 512 * 2); w.bsums = W.take<double>(2 * 512 * 2);
  w.col = W.take<AT>(max_col); w.dcol = W.take<float>(max_col);
  w.vis16 = W.take<AT>(b * T63 * 512);
  for (int k = 0; k < 2; ++k) {
    w.G[k] = W.take<float>(b * T63 * 2048); w.c[k] = W.take<float>(b * T63 * 512); w.rec[k] = W.take<float>(b * T63 * 512);
    w.rec16[k] = W.take<AT>(b * T63 * 512); w.hseq[k] = W.take<AT>(b * T63 * 512); w.out16[k] = W.take<AT>(b * T63 * 256);
  }
  w.bsum = W.take<float>(2 * 2048);
  w.dhn = W.take<float>(2 * b * HID); w.dcn = W.take<float>(2 * b * HID);
  w.d0 = W.take<float>(max_act); w.d1 = W.take<float>(max_act);
  w.dout = W.take<float>(b * T63 * 256); w.drec = W.take<float>(b * T63 * 512);
  if (sizeof(AT) == 2) {
    w.d16 = W.take<bf16>(max_act);
    w.dlog16 = W.take<bf16>(b * T63 * ((n_class + 7) / 8 * 8));
    w.dG16 = W.take<bf16>(b * T63 * 2048);
    w.w0pad16 = W.take<bf16>(64 * 64);
    w.dw0pad = W.take<float>(64 * 64);
  }
  w.bytes = W.off + 4096;
  return w;
}

inline float* gpt(const MrnbCrnnTrainPack& G, int slot) { return const_cast<float*>(G.p[slot]); }

// ------------------------------------------------------------------------------------------------
// Forward
// ------------------------------------------------------------------------------------------------
template <typename AT>
int crnn_train_forward_t(const MrnbCrnnTrainPack& P, const float* image, int B, int bn_batch, int update_running, float* logits,
                         long ld, void* ws, size_t ws_bytes, cudaStream_t st) {
  constexpr bool TC = sizeof(AT) == 2;
  CrnnWs<AT> w = carve_crnn_ws<AT>((char*)ws, B, P.n_class);
  MRNB_CHECK_ARG(ws_bytes >= w.bytes, "crnn_train_forward: workspace too small (%zu < %zu)", ws_bytes, w.bytes);
  {
    const long px = (long)B * 32 * 256;
    nchw_to_nhwc4_kernel<<<cdiv(px, 256), 256, 0, st>>>(image, w.img4, 32 * 256, px);
    MRNB_CHECK_LAUNCH("nchw_to_nhwc4_kernel");
  }
  if (bn_batch) cudaMemsetAsync(w.stats, 0, 2 * 512 * 2 * sizeof(double), st);
  const float* in = w.img4;
  for (int l = 0; l < 7; ++l) {
    const ConvL& L = LAYERS[l];
    const int Ho = out_h(L), Wo = out_w(L), K = L.KH * L.KW * L.Cin;
    const int rows = B * Ho * Wo;
    const long n = (long)rows * L.Cout;
    float* dst = L.bn >= 0 ? w.raw[L.bn] : w.act[l];
    if (l == 0 && TC) {    // K = 36 zero-padded to 64: one swizzled k-block on the tensor cores
      im2col_c4_pad64_kernel<<<cdiv((long)rows * 8, 256), 256, 0, st>>>(in, reinterpret_cast<bf16*>(w.col), L.H, L.W, rows);
      MRNB_CHECK_LAUNCH("im2col_c4_pad64_kernel");
      pad_w0_kernel<<<16, 256, 0, st>>>(P.p[L.w_slot], w.w0pad16, 64);
      MRNB_CHECK_LAUNCH("pad_w0_kernel");
      LinearArgs a{};
      a.A = w.col; a.lda = 64; a.a_gstride = (long)rows * 64;
      a.W16 = w.w0pad16; a.w_gstride = 64 * 64;
      a.bias = P.p[L.b_slot]; a.bias_gstride = 64;
      a.out = dst; a.ldo = 64; a.o_gstride = (long)rows * 64; a.out_is_f32 = 1; a.relu = 1;
      a.M = rows; a.N = 64; a.K = 64; a.groups = 1;
      MRNB_TRY(linear<AT>(a, st));
    } else if (l == 0) {   // fp32 mode: CUDA cores
      float* colf = reinterpret_cast<float*>(w.dcol);
      MRNB_TRY(launch_im2col<float>(in, colf, L.H, L.W, L.Cin, L.KH, L.KW, L.pad, 1, 1, Ho, Wo, rows, st));
      MrnbGemm g = mrnb_gemm_nt(colf, K, P.p[L.w_slot], K, dst, L.Cout, rows, L.Cout, K);
      g.bias_n = P.p[L.b_slot]; g.act = 2;
      MRNB_TRY(mrnb_sgemm(g, st));
    } else {
      MRNB_TRY(launch_im2col<AT>(in, w.col, L.H, L.W, L.Cin, L.KH, L.KW, L.pad, 1, 1, Ho, Wo, rows, st));
      MRNB_TRY(lin<AT>(w.col, K, P.p[L.w_slot], P.h[L.w_slot], L.b_slot >= 0 ? P.p[L.b_slot] : nullptr, dst, L.Cout, true, rows,
                       L.Cout, K, nullptr, nullptr, 1, st));
      if (L.bn < 0) {
        relu_kernel<<<cdiv(n / 4, 256), 256, 0, st>>>(dst, n / 4);
        MRNB_CHECK_LAUNCH("relu_kernel");
      }
    }
    if (L.bn >= 0) {
      const int q = L.bn;
      const int sw = q == 0 ? MRNB_T_BN4_W : MRNB_T_BN5_W;
      if (bn_batch) MRNB_TRY(launch_colstats(dst, rows, 512, w.stats + q * 1024, st));
      bn_finalize_kernel<<<2, 256, 0, st>>>(w.stats + q * 1024, P.p[sw], P.p[sw + 1], P.bn_mean[q], P.bn_var[q], w.ss + q * 1024,
                                            w.mr + q * 1024, 1, 512, (double)rows, bn_batch != 0, update_running != 0, 1e-5f);
      MRNB_CHECK_LAUNCH("bn_finalize_kernel");
      bn_relu_kernel<<<cdiv(n, 256), 256, 0, st>>>(dst, w.ss + q * 1024, w.act[l], 512, n);
      MRNB_CHECK_LAUNCH("bn_relu_kernel");
    }
    if (L.ph * L.pw > 1) {
      const long np = n / (L.ph * L.pw);
      maxpool_kernel<<<cdiv(np / 4, 256), 256, 0, st>>>(w.act[l], w.pool[l], Ho, Wo, L.Cout, L.ph, L.pw, np / 4);
      MRNB_CHECK_LAUNCH("maxpool_kernel");
    }
    in = w.pool[l];
  }
  // visual feature [B,63,512] = conv6 output (H = 1: permute / avg-pool / squeeze are relabelings, model.py:88-95)
  const int M = B * T63;
  const AT* x = nullptr;
  if (TC) {
    cast_kernel<AT><<<cdiv((long)M * 512, 256), 256, 0, st>>>(w.act[6], w.vis16, (long)M * 512);
    MRNB_CHECK_LAUNCH("cast_kernel");
    x = w.vis16;
  } else {
    x = reinterpret_cast<const AT*>(w.act[6]);
  }
  int Kin = 512;
  for (int k = 0; k < 2; ++k) {
    const int s0 = MRNB_T_LSTM0 + k * MRNB_TL_COUNT;
    add_vec_kernel<<<8, 256, 0, st>>>(P.p[s0 + MRNB_TL_BIH], P.p[s0 + MRNB_TL_BHH], w.bsum, 2048);
    MRNB_CHECK_LAUNCH("add_vec_kernel");
    // input projection of both directions: G = x [W_ih_f ; W_ih_r]^T + (b_ih + b_hh)
    MRNB_TRY(lin<AT>(x, Kin, P.p[s0 + MRNB_TL_WIH], P.h[s0 + MRNB_TL_WIH], w.bsum, w.G[k], 2048, true, M, 2048, Kin, nullptr,
                     nullptr, 1, st));
    cudaMemsetAsync(w.hseq[k], 0, (size_t)M * 512 * sizeof(AT), st);
    for (int s = 0; s < T63; ++s) {
      if (s > 0) {
        const int tf = s, tr = T63 - 1 - s;
        if constexpr (TC) {
          // G[:, t_dir, dir] += h_prev[dir] W_hh[dir]^T on the tensor cores: h_prev is the bf16 hidden sequence the
          // previous cell wrote at this position; the accumulate is the epilogue's residual at the output address
          // one launch for both directions (groups = 2): the two operand slices sit at different time positions, so the
          // A map walks them in address order and the recipe mirrors the group index when the reverse direction is lower
          const long pa[2] = {(long)tf * 512, (long)tr * 512 + HID};
          const long pc[2] = {(long)tf * 2048, (long)tr * 2048 + 1024};
          const bool up = pa[1] > pa[0];
          MrnbTcGemm2 g{};
          g.a = mrnb_operand_k2d(w.hseq[k] + (up ? pa[0] : pa[1]), B, HID, (long)T63 * 512, 128, 2, up ? pa[1] - pa[0] : pa[0] - pa[1]);
          if (!up) g.a.recipe.flip[2] = 2;
          g.b = mrnb_operand_k2d(P.h[s0 + MRNB_TL_WHH], 1024, HID, HID, 128, 2, 1024L * HID);
          float* c = w.G[k] + pc[0];
          g.out32 = c; g.res = c; g.cm = mrnb_axis((long)T63 * 2048); g.cn = mrnb_axis(1); g.c_gstride = pc[1] - pc[0];
          g.M = B; g.N = 1024; g.K = HID; g.groups = 2; g.splitk = 1; g.alpha = 1.f;
          MRNB_TRY(mrnb_tc_gemm2(g, st));
        } else {
          // both directions in one fp32 launch (batch = 2)
          MrnbGemm g = mrnb_gemm_nt(w.rec[k] + (long)(tf - 1) * 512, (long)T63 * 512, P.p[s0 + MRNB_TL_WHH], HID,
                                    w.G[k] + (long)tf * 2048, (long)T63 * 2048, B, 1024, HID);
          g.batch = 2; g.sAb = HID + (long)((tr + 1) - (tf - 1)) * 512; g.sBb = 1024L * HID;
          g.sCb = 1024 + (long)(tr - tf) * 2048; g.accumulate = 1;
          MRNB_TRY(mrnb_sgemm(g, st));
        }
      }
      lstm_cell_fwd_kernel<AT><<<cdiv(2 * B * HID, 256), 256, 0, st>>>(w.G[k], w.c[k], w.rec[k], w.hseq[k], B, s);
      MRNB_CHECK_LAUNCH("lstm_cell_fwd_kernel");
    }
    const AT* r = nullptr;
    if (TC) {
      cast_kernel<AT><<<cdiv((long)M * 512, 256), 256, 0, st>>>(w.rec[k], w.rec16[k], (long)M * 512);
      MRNB_CHECK_LAUNCH("cast_kernel");
      r = w.rec16[k];
    } else {
      r = reinterpret_cast<const AT*>(w.rec[k]);
    }
    MRNB_TRY(lin<AT>(r, 512, P.p[s0 + MRNB_TL_LIN_W], P.h[s0 + MRNB_TL_LIN_W], P.p[s0 + MRNB_TL_LIN_B], w.out16[k], 256, false, M,
                     256, 512, nullptr, nullptr, 1, st));
    x = w.out16[k]; Kin = 256;
  }
  MRNB_TRY(lin<AT>(w.out16[1], 256, P.p[MRNB_T_FC_W], P.h[MRNB_T_FC_W], P.p[MRNB_T_FC_B], logits, ld, true, M, P.n_class, 256,
                   nullptr, nullptr, 1, st));
  return MRNB_OK;
}

// ------------------------------------------------------------------------------------------------
// Backward
// ------------------------------------------------------------------------------------------------
template <typename AT>
int crnn_train_backward_t(const MrnbCrnnTrainPack& P, const MrnbCrnnTrainPack& G, const float* dlogits, long ldg, int B,
                          int bn_batch, float* grad_arena, long n_arena, void* ws, size_t ws_bytes, cudaStream_t st) {
  constexpr bool TC = sizeof(AT) == 2;
  CrnnWs<AT> w = carve_crnn_ws<AT>((char*)ws, B, P.n_class);
  MRNB_CHECK_ARG(ws_bytes >= w.bytes, "crnn_train_backward: workspace too small (%zu < %zu)", ws_bytes, w.bytes);
  cudaMemsetAsync(grad_arena, 0, (size_t)n_arena * sizeof(float), st);
  const int M = B * T63, C = P.n_class;
  // ---- CTC head
  Grad dlog{dlogits, nullptr, ldg};
  if (TC) {
    const long ld16 = (C + 7) / 8 * 8, total = (long)M * ld16;
    cast_pad_rows_kernel<<<cdiv(total / 8, 256), 256, 0, st>>>(dlogits, ldg, C, w.dlog16, ld16, total);
    MRNB_CHECK_LAUNCH("cast_pad_rows_kernel");
    dlog = Grad{dlogits, w.dlog16, ld16};
  }
  MRNB_TRY(launch_colsum<float>(dlogits, ldg, M, C, gpt(G, MRNB_T_FC_B), st));
  MRNB_TRY(gemm_dw<AT>(dlog, w.out16[1], 256, gpt(G, MRNB_T_FC_W), M, C, 256, st));
  bf16* dout16 = TC ? w.d16 : nullptr;
  MRNB_TRY(gemm_dx<AT>(dlog, P.p[MRNB_T_FC_W], P.h[MRNB_T_FC_W], w.dout, dout16, 256, M, C, 256, st));
  // ---- the two BidirectionalLSTMs, last first
  float* dxin = w.d0;                        // gradient w.r.t. the layer input [M, Kin]
  for (int k = 1; k >= 0; --k) {
    const int s0 = MRNB_T_LSTM0 + k * MRNB_TL_COUNT;
    const int Kin = k == 0 ? 512 : 256;
    Grad gout{w.dout, dout16, 256};
    const AT* r = TC ? w.rec16[k] : reinterpret_cast<const AT*>(w.rec[k]);
    MRNB_TRY(launch_colsum<float>(w.dout, 256, M, 256, gpt(G, s0 + MRNB_TL_LIN_B), st));
    MRNB_TRY(gemm_dw<AT>(gout, r, 512, gpt(G, s0 + MRNB_TL_LIN_W), M, 256, 512, st));
    MRNB_TRY(gemm_dx<AT>(gout, P.p[s0 + MRNB_TL_LIN_W], P.h[s0 + MRNB_TL_LIN_W], w.drec, nullptr, 512, M, 256, 512, st));
    // BPTT: direction 0 from t = 62 down, direction 1 from t = 0 up
    for (int s = 0; s < T63; ++s) {
      if (s > 0) {
        // dh_next[dir] = dgates[:, t_prev_processed, dir] . W_hh[dir]      (fp32; one split-K launch per direction so that
        // the [B,256] x K = 1024 product spreads over the SMs)
        const int tpos[2] = {T63 - s, s - 1};         // positions processed at step s - 1
        if constexpr (TC) {
          // bf16 gate gradients (written by the cell kernel) x W_hh read MN-major; both directions in one launch
          // (groups = 2, mirrored group index when the reverse direction's slice is lower), K = 1024 split 8 ways
          const long pa[2] = {(long)tpos[0] * 2048, (long)tpos[1] * 2048 + 1024};
          const bool up = pa[1] > pa[0];
          MrnbTcGemm2 g{};
          g.a = mrnb_operand_k2d(w.dG16 + (up ? pa[0] : pa[1]), B, 1024, (long)T63 * 2048, 128, 2, up ? pa[1] - pa[0] : pa[0] - pa[1]);
          if (!up) g.a.recipe.flip[2] = 2;
          g.b = mrnb_operand_mn2d(P.h[s0 + MRNB_TL_WHH], HID, 1024, HID, 2, 1024L * HID);
          g.out32 = w.dhn; g.cm = mrnb_axis(HID); g.cn = mrnb_axis(1); g.c_gstride = (long)B * HID;
          g.M = B; g.N = HID; g.K = 1024; g.groups = 2; g.splitk = 8; g.alpha = 1.f;
          MRNB_TRY(mrnb_tc_gemm2(g, st));
        } else {
          for (int dir = 0; dir < 2; ++dir) {
            MrnbGemm g{};
            g.A = w.G[k] + (long)tpos[dir] * 2048 + dir * 1024; g.am = mrnb_axis((long)T63 * 2048); g.ak = mrnb_axis(1); g.a_kfast = 1;
            g.B = P.p[s0 + MRNB_TL_WHH] + (long)dir * 1024 * HID; g.bk = mrnb_axis(HID); g.bn = mrnb_axis(1); g.b_kfast = 0;
            g.C = w.dhn + (long)dir * B * HID; g.cm = mrnb_axis(HID); g.cn = mrnb_axis(1);
            g.M = B; g.N = HID; g.K = 1024; g.batch = 1; g.splitk = 8; g.alpha = 1.f; g.rows_per_scale = 1;
            MRNB_TRY(mrnb_sgemm(g, st));
          }
        }
      }
      lstm_cell_bwd_kernel<<<cdiv(2 * B * HID, 256), 256, 0, st>>>(w.G[k], w.c[k], w.drec, w.dhn, w.dcn, B, s, TC ? w.dG16 : nullptr);
      MRNB_CHECK_LAUNCH("lstm_cell_bwd_kernel");
    }
    // G now holds d(gate pre-activations) [M, 2048] for both directions
    Grad gG{w.G[k], nullptr, 2048};
    if (TC) gG.h = w.dG16;                     // written step by step by the cell kernel
    MRNB_TRY(launch_colsum<float>(w.G[k], 2048, M, 2048, gpt(G, s0 + MRNB_TL_BIH), st));
    cudaMemcpyAsync(gpt(G, s0 + MRNB_TL_BHH), gpt(G, s0 + MRNB_TL_BIH), 2048 * sizeof(float), cudaMemcpyDeviceToDevice, st);
    const AT* xin = k == 0 ? (TC ? w.vis16 : reinterpret_cast<const AT*>(w.act[6])) : w.out16[0];
    MRNB_TRY(gemm_dw<AT>(gG, xin, Kin, gpt(G, s0 + MRNB_TL_WIH), M, 2048, Kin, st));
    for (int dir = 0; dir < 2; ++dir) {
      Grad gd{w.G[k] + dir * 1024, TC ? w.dG16 + dir * 1024 : nullptr, 2048};
      MRNB_TRY(gemm_dw<AT>(gd, w.hseq[k] + dir * HID, 512, gpt(G, s0 + MRNB_TL_WHH) + (long)dir * 1024 * HID, M, 1024, HID, st));
    }
    float* dx = k == 0 ? dxin : w.dout;        // layer 1's input gradient is layer 0's output gradient
    MRNB_TRY(gemm_dx<AT>(gG, P.p[s0 + MRNB_TL_WIH], P.h[s0 + MRNB_TL_WIH], dx, k == 1 ? dout16 : nullptr, Kin, M, 2048, Kin, st));
  }
  // ---- VGG, last layer first.  d = gradient w.r.t. the (pooled) output of layer l
  float* d = dxin;                             // [B,1,63,512] = d conv6 output (post-relu)
  float* other = w.d1;
  for (int l = 6; l >= 0; --l) {
    const ConvL& L = LAYERS[l];
    const int Ho = out_h(L), Wo = out_w(L), K = L.KH * L.KW * L.Cin;
    const int rows = B * Ho * Wo;
    const long n = (long)rows * L.Cout;
    bf16* d16 = TC ? w.d16 : nullptr;
    // through pool + relu (or relu alone) to the conv / BN output
    if (L.ph * L.pw > 1) {
      const long np = n / (L.ph * L.pw);
      maxpool_relu_bwd_kernel<<<cdiv(np / 4, 256), 256, 0, st>>>(w.act[l], d, other, Ho, Wo, L.Cout, L.ph, L.pw, np / 4);
      MRNB_CHECK_LAUNCH("maxpool_relu_bwd_kernel");
      float* t = d; d = other; other = t;
      if (d16 && L.bn < 0) {
        cast_kernel<bf16><<<cdiv(n, 256), 256, 0, st>>>(d, d16, n);
        MRNB_CHECK_LAUNCH("cast_kernel");
      }
    } else {
      relu_bwd_kernel<<<cdiv(n, 256), 256, 0, st>>>(w.act[l], d, L.bn < 0 ? d16 : nullptr, n);
      MRNB_CHECK_LAUNCH("relu_bwd_kernel");
    }
    if (L.bn >= 0) {
      const int q = L.bn, sw = q == 0 ? MRNB_T_BN4_W : MRNB_T_BN5_W;
      cudaMemsetAsync(w.bsums + q * 1024, 0, 1024 * sizeof(double), st);
      int chunks = rows / 256; if (chunks < 1) chunks = 1; if (chunks > 64) chunks = 64;
      bn_relu_bwd_reduce_kernel<<<dim3(16, chunks), dim3(32, 8), 0, st>>>(w.raw[q], d, w.mr + q * 1024, rows, 512, w.bsums + q * 1024);
      MRNB_CHECK_LAUNCH("bn_relu_bwd_reduce_kernel");
      bn_bwd_apply_kernel<<<cdiv(n, 256), 256, 0, st>>>(w.raw[q], d, w.ss + q * 1024, w.mr + q * 1024, w.bsums + q * 1024, (double)rows,
                                                        bn_batch, gpt(G, sw), gpt(G, sw + 1), 512, n, d16);
      MRNB_CHECK_LAUNCH("bn_bwd_apply_kernel");
    }
    // conv backward
    if (L.b_slot >= 0) MRNB_TRY(launch_colsum<float>(d, L.Cout, rows, L.Cout, gpt(G, L.b_slot), st));
    const float* in = l == 0 ? w.img4 : w.pool[l - 1];
    if (l == 0 && TC) {
      im2col_c4_pad64_kernel<<<cdiv((long)rows * 8, 256), 256, 0, st>>>(in, reinterpret_cast<bf16*>(w.col), L.H, L.W, rows);
      MRNB_CHECK_LAUNCH("im2col_c4_pad64_kernel");
      cudaMemsetAsync(w.dw0pad, 0, 64 * 64 * sizeof(float), st);
      MRNB_TRY(gemm_dw_tc(d16, 64, reinterpret_cast<const bf16*>(w.col), 64, w.dw0pad, rows, 64, 64, st));
      unpad_dw0_kernel<<<9, 256, 0, st>>>(w.dw0pad, gpt(G, L.w_slot), 64);
      MRNB_CHECK_LAUNCH("unpad_dw0_kernel");
      break;
    }
    if (l == 0) {
      float* colf = w.dcol;
      MRNB_TRY(launch_im2col<float>(in, colf, L.H, L.W, L.Cin, L.KH, L.KW, L.pad, 1, 1, Ho, Wo, rows, st));
      MRNB_TRY(gemm_dw_f32(d, L.Cout, colf, K, gpt(G, L.w_slot), rows, L.Cout, K, st));
      break;                                   // no gradient w.r.t. the image
    }
    Grad gd{d, d16, L.Cout};
    MRNB_TRY(launch_im2col<AT>(in, w.col, L.H, L.W, L.Cin, L.KH, L.KW, L.pad, 1, 1, Ho, Wo, rows, st));
    MRNB_TRY(gemm_dw<AT>(gd, w.col, K, gpt(G, L.w_slot), rows, L.Cout, K, st));
    MRNB_TRY(gemm_dx<AT>(gd, P.p[L.w_slot], P.h[L.w_slot], w.dcol, nullptr, K, rows, L.Cout, K, st));
    const long in4 = (long)B * L.H * L.W * L.Cin / 4;
    // LAYERS has 3 x 3 windows and the 2 x 2 of conv6
    const auto col2im = L.KH == 2 ? col2im_nhwc_kernel<2, 2> : col2im_nhwc_kernel<3, 3>;
    col2im<<<cdiv(in4, 256), 256, 0, st>>>(w.dcol, other, L.H, L.W, L.Cin, L.pad, 1, 1, Ho, Wo, in4);
    MRNB_CHECK_LAUNCH("col2im_nhwc_kernel");
    float* t = d; d = other; other = t;
  }
  return MRNB_OK;
}

}  // namespace

extern "C" size_t mrnb_crnn_train_workspace_bytes(int B, int n_class, int prec) {
  return prec == MRNB_PREC_BF16 ? carve_crnn_ws<__nv_bfloat16>(nullptr, B, n_class).bytes
                                : carve_crnn_ws<float>(nullptr, B, n_class).bytes;
}

extern "C" int mrnb_crnn_train_forward(const MrnbCrnnTrainPack* pack, const float* image, int B, int prec, int bn_batch_stats,
                                       int update_running, float* logits, long ld_logits, void* workspace,
                                       size_t workspace_bytes, cudaStream_t stream) {
  MRNB_CHECK_ARG(pack && image && logits && workspace && B > 0, "crnn_train_forward: null/empty argument");
  MRNB_CHECK_ARG(ld_logits >= pack->n_class && pack->n_class > 0, "crnn_train_forward: ld_logits < n_class");
  for (int k = 0; k < MRNB_T_COUNT; ++k) MRNB_CHECK_ARG(pack->p[k], "crnn_train_forward: parameter slot %d is null", k);
  MRNB_CHECK_ARG(pack->bn_mean[0] && pack->bn_mean[1] && pack->bn_var[0] && pack->bn_var[1], "crnn_train_forward: BN statistics missing");
  if (prec == MRNB_PREC_FP32)
    return crnn_train_forward_t<float>(*pack, image, B, bn_batch_stats, update_running, logits, ld_logits, workspace,
                                       workspace_bytes, stream);
  if (prec == MRNB_PREC_BF16)
    return crnn_train_forward_t<__nv_bfloat16>(*pack, image, B, bn_batch_stats, update_running, logits, ld_logits, workspace,
                                               workspace_bytes, stream);
  mrnb_set_error("crnn_train_forward: unknown precision %d", prec);
  return MRNB_ERR_ARG;
}

extern "C" int mrnb_crnn_train_backward(const MrnbCrnnTrainPack* pack, const MrnbCrnnTrainPack* grads, const float* dlogits,
                                        long ld_dlogits, int B, int prec, int bn_batch_stats, float* grad_arena, long n_arena,
                                        void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  MRNB_CHECK_ARG(pack && grads && dlogits && grad_arena && workspace && B > 0, "crnn_train_backward: null/empty argument");
  for (int k = 0; k < MRNB_T_COUNT; ++k) MRNB_CHECK_ARG(grads->p[k], "crnn_train_backward: gradient slot %d is null", k);
  if (prec == MRNB_PREC_FP32)
    return crnn_train_backward_t<float>(*pack, *grads, dlogits, ld_dlogits, B, bn_batch_stats, grad_arena, n_arena, workspace,
                                        workspace_bytes, stream);
  if (prec == MRNB_PREC_BF16)
    return crnn_train_backward_t<__nv_bfloat16>(*pack, *grads, dlogits, ld_dlogits, B, bn_batch_stats, grad_arena, n_arena,
                                                workspace, workspace_bytes, stream);
  mrnb_set_error("crnn_train_backward: unknown precision %d", prec);
  return MRNB_ERR_ARG;
}
