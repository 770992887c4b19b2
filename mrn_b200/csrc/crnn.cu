// CRNN expert recogniser forward (VGG feature extractor + 2 x BidirectionalLSTM + CTC head), grouped over the
// N per-task experts.
//
// Reference (paths relative to /root/reference):
//   modules/feature_extraction.py:19-47   VGG_FeatureExtractor (7 convolutions, ReLU, 4 max-pools, 2 BatchNorm2d)
//   modules/sequence_modeling.py:4-22     BidirectionalLSTM (nn.LSTM bidirectional + Linear 2H -> H)
//   modules/model.py:46-57,82-101         Model_Extractor (permute / avg-pool over H = 1 / two BiLSTMs)
//   modules/model.py:133-148,176-181      Model.forward (CTC head fc), T = 63 frames (modules/model.py:322-323)
//
// Layout: activations are NHWC [expert][sample][h][w][channel] in AT (float in the fp32 parity mode, bf16 in the
// tensor-core mode).  In bf16 mode every 3x3 / 2x2 convolution with Cin >= 64 is an implicit GEMM on tcgen05: the A
// tiles are gathered by TMA straight from the NHWC activation (zero fill outside the image = padding), see
// MrnbTcConv in gemm_tc.h; in fp32 mode it is im2col + the CUDA-core SGEMM.  The frame axis is carried padded to
// 64 rows per sample (row 63 is scratch) so that every GEMM tile holds whole samples; the LSTM walks rows 0..62.
// The LSTM recurrence is one grouped GEMM (h W_hh^T for all experts x directions) + one cell kernel per step.
#include "common.cuh"
#include <stdlib.h>
#include "expert_util.cuh"
#include "../../include/mrn_b200.h"

namespace {

constexpr int CT = 63;      // frames
constexpr int CTP = 64;     // padded frame rows
constexpr int LH = 256;     // LSTM hidden size (opt.hidden_size)

template <typename AT> __device__ __forceinline__ void load8(const AT* p, float (&v)[8]);
template <> __device__ __forceinline__ void load8<float>(const float* p, float (&v)[8]) {
  const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
template <> __device__ __forceinline__ void load8<__nv_bfloat16>(const __nv_bfloat16* p, float (&v)[8]) {
  const uint4 u = *reinterpret_cast<const uint4*>(p);
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const __nv_bfloat162 h = *reinterpret_cast<const __nv_bfloat162*>(&w[j]);
    v[2 * j] = __low2float(h); v[2 * j + 1] = __high2float(h);
  }
}
template <typename AT> __device__ __forceinline__ void store8(AT* p, const float (&v)[8]);
template <> __device__ __forceinline__ void store8<float>(float* p, const float (&v)[8]) {
  *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  *reinterpret_cast<float4*>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
}
template <> __device__ __forceinline__ void store8<__nv_bfloat16>(__nv_bfloat16* p, const float (&v)[8]) {
  uint32_t w[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
    w[j] = *reinterpret_cast<const uint32_t*>(&h);
  }
  *reinterpret_cast<uint4*>(p) = make_uint4(w[0], w[1], w[2], w[3]);
}

// ------------------------------------------------------------------------------------------------
// conv0: Conv2d(4 -> 64, 3x3, pad 1) + ReLU + MaxPool 2x2 (feature_extraction.py:20-22), K = 36: CUDA cores.
// image NCHW fp32 [B,4,32,256] -> NHWC [I,B,16,128,64].  grid (16 pooled rows, B, I); block 256 = 128 pooled
// columns x 2 halves of 32 output channels; the 4 input rows and the expert's weights are staged in shared memory.
// ------------------------------------------------------------------------------------------------
template <typename AT>
__global__ void __launch_bounds__(256)
vgg_conv0_kernel(const float* __restrict__ image, const float* __restrict__ w /*[I,64,4,3,3]*/,
                 const float* __restrict__ bias /*[I,64]*/, AT* __restrict__ out, int B) {
  __shared__ float s_in[4][4][260];      // [channel][row][col + 1], zero padded
  __shared__ __align__(16) float s_w[64 * 36 + 64];
  const int pr = blockIdx.x, b = blockIdx.y, e = blockIdx.z;
  for (int i = threadIdx.x; i < 4 * 4 * 260; i += 256) {
    const int col = i % 260, r = (i / 260) % 4, c = i / (260 * 4);
    const int ih = 2 * pr - 1 + r, iw = col - 1;
    float v = 0.f;
    if (ih >= 0 && ih < 32 && iw >= 0 && iw < 256) v = image[(((long)b * 4 + c) * 32 + ih) * 256 + iw];
    s_in[c][r][col] = v;
  }
  for (int i = threadIdx.x; i < 64 * 36; i += 256) s_w[i] = w[(long)e * 64 * 36 + i];
  if (threadIdx.x < 64) s_w[64 * 36 + threadIdx.x] = bias[e * 64 + threadIdx.x];
  __syncthreads();
  const int pc = threadIdx.x & 127, half = threadIdx.x >> 7;
  float win[4][4][4];                    // [channel][row][col]: input window of the 2x2 conv outputs
#pragma unroll
  for (int c = 0; c < 4; ++c)
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int k = 0; k < 4; ++k) win[c][r][k] = s_in[c][r][2 * pc + k];
  AT* op = out + ((((long)e * B + b) * 16 + pr) * 128 + pc) * 64 + half * 32;
#pragma unroll 1
  for (int c8 = 0; c8 < 4; ++c8) {
    float o[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int oc = half * 32 + c8 * 8 + u;
      const float4* wp4 = reinterpret_cast<const float4*>(s_w + oc * 36);     // 9 broadcast 16-byte loads per channel
      float wreg[36];
#pragma unroll
      for (int k4 = 0; k4 < 9; ++k4) {
        const float4 t = wp4[k4];
        wreg[k4 * 4] = t.x; wreg[k4 * 4 + 1] = t.y; wreg[k4 * 4 + 2] = t.z; wreg[k4 * 4 + 3] = t.w;
      }
      float a00 = 0.f, a01 = 0.f, a10 = 0.f, a11 = 0.f;
#pragma unroll
      for (int c = 0; c < 4; ++c)
#pragma unroll
        for (int kh = 0; kh < 3; ++kh)
#pragma unroll
          for (int kw = 0; kw < 3; ++kw) {
            const float wv = wreg[(c * 3 + kh) * 3 + kw];
            a00 = fmaf(wv, win[c][kh][kw], a00);
            a01 = fmaf(wv, win[c][kh][kw + 1], a01);
            a10 = fmaf(wv, win[c][kh + 1][kw], a10);
            a11 = fmaf(wv, win[c][kh + 1][kw + 1], a11);
          }
      o[u] = fmaxf(fmaxf(fmaxf(a00, a01), fmaxf(a10, a11)) + s_w[64 * 36 + oc], 0.f);
    }
    store8<AT>(op + c8 * 8, o);
  }
}

// Tensor-core mode of conv0: im2col of the NCHW image shared by all experts, K = 36 taps (c, kh, kw) zero-padded to 64,
// rows WINDOW-MAJOR: row = ((b*16 + ph)*128 + pw)*4 + (dy*2 + dx) is the conv output pixel (2ph+dy, 2pw+dx), so the
// 2x2 max-pool is a max over 4 consecutive GEMM rows (MrnbTcGemm::pool4).  One thread per (row, 8-tap group).
__global__ void __launch_bounds__(256)
vgg_im2col0_kernel(const float* __restrict__ image, __nv_bfloat16* __restrict__ col, unsigned total) {
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const unsigned kg = i & 7, row = i >> 3;
  const unsigned win = row & 3, pw = (row >> 2) & 127, ph = (row >> 9) & 15, b = row >> 13;
  const int oh = 2 * ph + (win >> 1), ow = 2 * pw + (win & 1);
  float v[8];
#pragma unroll
  for (int u = 0; u < 8; ++u) {
    const int k = kg * 8 + u;
    float x = 0.f;
    if (k < 36) {
      const int c = k / 9, kh = (k % 9) / 3, kw = k % 3;
      const int ih = oh - 1 + kh, iw = ow - 1 + kw;
      if (ih >= 0 && ih < 32 && iw >= 0 && iw < 256) x = __ldg(image + (((size_t)b * 4 + c) * 32 + ih) * 256 + iw);
    }
    v[u] = x;
  }
  store8<__nv_bfloat16>(col + (size_t)i * 8, v);
}

// MaxPool2d((ph, pw)) over NHWC, 8 channels per thread.  in [N,H,W,C] -> out [N,H/ph,W/pw,C]   (32-bit index math:
// the 8-channel group count stays below 2^31 for every supported batch)
template <typename AT>
__global__ void pool_kernel(const AT* __restrict__ in, AT* __restrict__ out, int H, int W, int C, int ph, int pw, unsigned total8) {
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total8) return;
  const unsigned c8 = C / 8, OW = W / pw, OH = H / ph;
  const unsigned c = (i % c8) * 8;
  unsigned r = i / c8;
  const unsigned ow = r % OW; r /= OW;
  const unsigned oh = r % OH;
  const unsigned n = r / OH;
  float m[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) m[j] = -INFINITY;
  for (int a = 0; a < ph; ++a)
    for (int b = 0; b < pw; ++b) {
      float v[8];
      load8<AT>(in + ((size_t)((n * H + oh * ph + a) * W) + ow * pw + b) * C + c, v);
#pragma unroll
      for (int j = 0; j < 8; ++j) m[j] = fmaxf(m[j], v[j]);
    }
  store8<AT>(out + (size_t)i * 8, m);
}

// per-channel sum / sum of squares over the rows of x [I][rows][512] (BatchNorm2d batch statistics), fp64 atomics
template <typename AT>
__global__ void __launch_bounds__(256)
bn_stats512_kernel(const AT* __restrict__ x, long rows, double* __restrict__ stats /*[I,512,2]*/) {
  const int e = blockIdx.y;
  const long per = (rows + gridDim.x - 1) / gridDim.x;
  const long r0 = (long)blockIdx.x * per, r1 = r0 + per < rows ? r0 + per : rows;
  const AT* xp = x + (long)e * rows * 512;
  double s1[2] = {0.0, 0.0}, s2[2] = {0.0, 0.0};
  for (long r = r0; r < r1; ++r) {
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const float v = to_f32<AT>(xp[r * 512 + k * 256 + threadIdx.x]);
      s1[k] += v; s2[k] += (double)v * v;
    }
  }
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    atomicAdd(stats + ((long)e * 512 + k * 256 + threadIdx.x) * 2, s1[k]);
    atomicAdd(stats + ((long)e * 512 + k * 256 + threadIdx.x) * 2 + 1, s2[k]);
  }
}

// y = ReLU(x * scale + shift) (+ MaxPool (2,1) when pool_h == 2).  x [I][B][H][64][512] -> y [I][B][H/pool_h][64][512]
// grid (row blocks, I); a thread owns 8 channels (scale / shift in registers) and walks output rows
template <typename AT>
__global__ void __launch_bounds__(256)
bn_relu_pool_kernel(const AT* __restrict__ x, const float* __restrict__ ss /*[I,512,2]*/, AT* __restrict__ y,
                    unsigned rows_out /* per expert: B * OH * 64 */, int H, int pool_h) {
  const int e = blockIdx.y;
  const int c = (threadIdx.x & 63) * 8;
  float sc[8], sh[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { sc[j] = ss[((size_t)e * 512 + c + j) * 2]; sh[j] = ss[((size_t)e * 512 + c + j) * 2 + 1]; }
  const unsigned OH = H / pool_h;
  const AT* xe = x + (size_t)e * rows_out * pool_h * 512;
  AT* ye = y + (size_t)e * rows_out * 512;
  for (unsigned orow = blockIdx.x * 4 + (threadIdx.x >> 6); orow < rows_out; orow += gridDim.x * 4) {
    const unsigned w = orow & 63, nh = orow >> 6;          // nh = b * OH + oh
    const unsigned n = nh / OH, oh = nh % OH;
    float m[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) m[j] = 0.f;
    for (int a = 0; a < pool_h; ++a) {
      float v[8];
      load8<AT>(xe + ((size_t)((n * H + oh * pool_h + a) * 64) + w) * 512 + c, v);
#pragma unroll
      for (int j = 0; j < 8; ++j) m[j] = fmaxf(m[j], fmaf(v[j], sc[j], sh[j]));     // max(0, .) == ReLU
    }
    store8<AT>(ye + (size_t)orow * 512 + c, m);
  }
}

// ------------------------------------------------------------------------------------------------
// LSTM cell, step s of every (expert, direction) chain.  gates [2I][B][4H] fp32 = h_{t-1} W_hh^T (ignored at s = 0),
// pre [I][B*64][2*4H] AT = x W_ih^T + b_ih + b_hh for both directions; gates i, f, g, o (nn.LSTM) interleaved per unit.
// Writes c (fp32), h (AT, the next step's GEMM operand) and the [fwd | bwd] output row rec [I][B*64][2H].
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float sigmoid_f(float x) { return 1.0f / (1.0f + __expf(-x)); }

// MRNB_LSTM_SEQ = 0 keeps one grouped GEMM launch per time step (read on every call: the parity test toggles it)
inline bool lstm_seq_enabled() {
  const char* e = getenv("MRNB_LSTM_SEQ");
  return !e || atoi(e) != 0;
}

template <typename AT>
__global__ void lstm_cell_kernel(const float* __restrict__ gates, const AT* __restrict__ pre, float* __restrict__ cst,
                                 AT* __restrict__ hst, AT* __restrict__ rec, int I, int B, int s, unsigned total) {
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int j = (int)(i % LH);
  const unsigned gb = i / LH;
  const int b = (int)(gb % (unsigned)B);
  const int g = (int)(gb / (unsigned)B);
  const int e = g >> 1, dir = g & 1;
  const int t = dir ? CT - 1 - s : s;
  // gate axis interleaved: column 4*j + {i, f, g, o} (the pack re-orders the LSTM weight rows accordingly)
  const AT* pp = pre + (((long)e * B + b) * CTP + t) * (8 * LH) + dir * 4 * LH + 4 * j;
  float a[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) a[k] = to_f32<AT>(pp[k]);
  float cprev = 0.f;
  if (s > 0) {
    const float4 gq = *reinterpret_cast<const float4*>(gates + ((long)g * B + b) * (4 * LH) + 4 * j);
    a[0] += gq.x; a[1] += gq.y; a[2] += gq.z; a[3] += gq.w;
    cprev = cst[i];
  }
  const float c = sigmoid_f(a[1]) * cprev + sigmoid_f(a[0]) * tanhf(a[2]);
  const float h = sigmoid_f(a[3]) * tanhf(c);
  cst[i] = c;
  hst[i] = from_f32<AT>(h);
  rec[(((long)e * B + b) * CTP + t) * (2 * LH) + dir * LH + j] = from_f32<AT>(h);
}

// contextual feature [I][B][64][256] fp32 -> router layout [B,I,63,256] fp32 and compact [I][B*63][256] AT (fc operand)
template <typename AT>
__global__ void crnn_feature_kernel(const float* __restrict__ src, float* __restrict__ features, AT* __restrict__ compact,
                                    int I, int B, long total4) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total4) return;
  const int d = (int)(i % 64) * 4;
  long r = i / 64;
  const int t = (int)(r % CT); r /= CT;
  const int b = (int)(r % B);
  const int e = (int)(r / B);
  const float4 v = *reinterpret_cast<const float4*>(src + (((long)e * B + b) * CTP + t) * 256 + d);
  if (features) *reinterpret_cast<float4*>(features + (((long)b * I + e) * CT + t) * 256 + d) = v;
  AT* o = compact + (((long)e * B + b) * CT + t) * 256 + d;
  o[0] = from_f32<AT>(v.x); o[1] = from_f32<AT>(v.y); o[2] = from_f32<AT>(v.z); o[3] = from_f32<AT>(v.w);
}

// ------------------------------------------------------------------------------------------------
// one convolution layer over all experts: in [I][B][H][W][Cin] -> out [I][B][OH][OWp][Cout]
// ------------------------------------------------------------------------------------------------
struct ConvSpec { int H, W, Cin, Cout, KS, pad, OH, OWp, relu; };

template <typename AT>
int conv_layer(const ConvSpec& c, int I, int B, const AT* in, const float* W32, const void* W16, const float* bias,
               AT* out, float* col, cudaStream_t st) {
  const int K = c.KS * c.KS * c.Cin;
  const long rows = (long)B * c.OH * c.OWp;
  if constexpr (sizeof(AT) == 2) {
    MRNB_CHECK_ARG(W16, "crnn_forward: bf16 mode needs the 16-bit convolution weights");
    MrnbTcGemm g{};
    g.A = in; g.W = W16; g.ldw = K; g.w_gstride = (long)c.Cout * K;
    g.bias = bias; g.bias_gstride = c.Cout;
    g.out = out; g.ldo = c.Cout; g.o_gstride = rows * c.Cout; g.out_f32 = 0;
    g.M = (int)rows; g.N = c.Cout; g.K = K; g.groups = I; g.rows_per_scale = 1; g.relu = c.relu;
    g.conv.enabled = 1;
    g.conv.dims[0] = c.Cin; g.conv.dims[1] = c.W; g.conv.dims[2] = c.H; g.conv.dims[3] = (long)I * B;
    g.conv.strides[0] = c.Cin; g.conv.strides[1] = (long)c.W * c.Cin; g.conv.strides[2] = (long)c.H * c.W * c.Cin;
    g.conv.box_w = c.OWp;
    g.conv.box_h = c.OWp == 128 ? 1 : (c.OH >= 2 ? 2 : 1);
    g.conv.box_img = 128 / (g.conv.box_w * g.conv.box_h);
    g.conv.sh = 1; g.conv.pad_h = c.pad; g.conv.w_off = -c.pad;
    g.conv.rows_per_img = c.OH * c.OWp; g.conv.per_kh = c.KS * (c.Cin / 64); g.conv.cch = c.Cin / 64;
    g.conv.imgs_per_group = B;
    return mrnb_tc_gemm(g, st);
  } else {
    for (int e = 0; e < I; ++e) {
      const long total4 = rows * K / 4;
      im2col_nhwc_kernel<float><<<cdiv(total4, 256), 256, 0, st>>>(reinterpret_cast<const float*>(in) + (long)e * B * c.H * c.W * c.Cin,
                                                                   col, c.H, c.W, c.Cin, c.KS, c.KS, c.pad, 1, 1, c.OH, c.OWp, total4);
      MRNB_CHECK_LAUNCH("im2col_nhwc_kernel");
      LinearArgs a{};
      a.A = col; a.lda = K; a.W32 = W32 + (long)e * c.Cout * K; a.bias = bias ? bias + (long)e * c.Cout : nullptr;
      a.out = reinterpret_cast<float*>(out) + (long)e * rows * c.Cout; a.ldo = c.Cout; a.out_is_f32 = 1;
      a.M = (int)rows; a.N = c.Cout; a.K = K; a.groups = 1; a.relu = c.relu;
      MRNB_TRY(linear<float>(a, st));
    }
    return MRNB_OK;
  }
}

template <typename AT>
int launch_pool(const AT* in, AT* out, long N, int H, int W, int C, int ph, int pw, cudaStream_t st) {
  const long total8 = N * (H / ph) * (W / pw) * C / 8;
  MRNB_CHECK_ARG(total8 < (1L << 31) && N * H * W < (1L << 31), "crnn_forward: batch too large for the pooling kernels");
  pool_kernel<AT><<<cdiv(total8, 256), 256, 0, st>>>(in, out, H, W, C, ph, pw, (unsigned)total8);
  MRNB_CHECK_LAUNCH("pool_kernel");
  return MRNB_OK;
}

template <typename AT>
size_t crnn_workspace_bytes_t(int I, int B) {
  const size_t u = (size_t)I * B;
  size_t s = 0;
  s += align_up((u * 262144 > (size_t)B * 524288 ? u * 262144 : (size_t)B * 524288) * sizeof(AT));      // X (also the conv0 im2col)
  s += align_up(u * 131072 * sizeof(AT));      // Y
  s += align_up(u * 131072 * sizeof(AT));      // Z
  if (sizeof(AT) == 4) s += align_up((size_t)B * 2048 * 576 * 4);   // im2col of one expert (largest: 1 179 648 per sample)
  s += align_up((size_t)I * 512 * 2 * sizeof(double)) + align_up((size_t)I * 512 * 2 * sizeof(float));   // BN stats / scale-shift
  s += align_up(u * 2 * 4 * LH * 4);           // gates fp32
  s += align_up(u * 2 * LH * 4);               // c state
  s += align_up(u * 2 * LH * sizeof(AT));      // h state
  s += align_up(u * CT * 256 * sizeof(AT));    // compact features (fc operand)
  return s + 4096;
}

template <typename AT>
int crnn_forward_t(const MrnbCrnnPack& P, const float* image, int B, int bn_batch_stats, int update_running,
                   float* features, float* const* logits, const long* ld_logits, void* ws, size_t ws_bytes, cudaStream_t st) {
  const int I = P.n_experts;
  MRNB_CHECK_ARG(ws_bytes >= crnn_workspace_bytes_t<AT>(I, B), "crnn_forward: workspace too small (%zu < %zu)", ws_bytes,
                 crnn_workspace_bytes_t<AT>(I, B));
  constexpr bool F32 = sizeof(AT) == 4;
  Workspace W{(char*)ws, 0, ws_bytes};
  const size_t u = (size_t)I * B;
  AT* X = W.take<AT>(u * 262144 > (size_t)B * 524288 ? u * 262144 : (size_t)B * 524288);
  AT* Y = W.take<AT>(u * 131072);
  AT* Z = W.take<AT>(u * 131072);
  float* col = F32 ? W.take<float>((size_t)B * 2048 * 576) : nullptr;
  double* stats = W.take<double>((size_t)I * 512 * 2);
  float* ss = W.take<float>((size_t)I * 512 * 2);
  float* gates = W.take<float>(u * 2 * 4 * LH);
  float* cst = W.take<float>(u * 2 * LH);
  AT* hst = W.take<AT>(u * 2 * LH);
  AT* compact = W.take<AT>(u * CT * 256);
  const long N = (long)I * B;

  // ---- VGG (feature_extraction.py:19-47); Sequential index in the comments
  if constexpr (!F32) {
    // 0-2 on the tensor cores: shared im2col (X, 64 bf16 per conv pixel) -> per expert GEMM [B*8192 x 64] x [64 x 64]
    // with bias + ReLU + 2x2 max-pool in the epilogue -> Y [16,128,64]
    MRNB_CHECK_ARG(P.h[MRNB_C_CONV0_W], "crnn_forward: bf16 mode needs the GEMM-packed conv0 weight in h[MRNB_C_CONV0_W]");
    MRNB_CHECK_ARG((long)B * 8192 * 8 < (1L << 32), "crnn_forward: batch too large for the conv0 im2col");
    mrnb_prof_begin(MRNB_PROF_CONV, st, 0.0, 0.0);
    const unsigned total = (unsigned)B * 8192u * 8u;
    vgg_im2col0_kernel<<<cdiv(total, 256), 256, 0, st>>>(image, reinterpret_cast<__nv_bfloat16*>(X), total);
    MRNB_CHECK_LAUNCH("vgg_im2col0_kernel");
    mrnb_prof_end(MRNB_PROF_CONV, st);
    for (int e = 0; e < I; ++e) {
      MrnbTcGemm g{};
      g.A = X; g.lda = 64; g.W = reinterpret_cast<const __nv_bfloat16*>(P.h[MRNB_C_CONV0_W]) + (size_t)e * 64 * 64; g.ldw = 64;
      g.bias = P.p[MRNB_C_CONV0_B] + e * 64;
      g.out = reinterpret_cast<__nv_bfloat16*>(Y) + (size_t)e * B * 2048 * 64; g.ldo = 64; g.out_f32 = 0;
      g.M = B * 8192; g.N = 64; g.K = 64; g.groups = 1; g.rows_per_scale = 1; g.pool4 = 1;
      MRNB_TRY(mrnb_tc_gemm(g, st));
    }
  } else {
    mrnb_prof_begin(MRNB_PROF_CONV, st, 0.0, 0.0);
    vgg_conv0_kernel<AT><<<dim3(16, B, I), 256, 0, st>>>(image, P.p[MRNB_C_CONV0_W], P.p[MRNB_C_CONV0_B], Y, B);   // 0-2 -> Y [16,128,64]
    MRNB_CHECK_LAUNCH("vgg_conv0_kernel");
    mrnb_prof_end(MRNB_PROF_CONV, st);
  }
  {
    const ConvSpec c1{16, 128, 64, 128, 3, 1, 16, 128, 1};                                                 // 3-4 -> X [16,128,128]
    MRNB_TRY(conv_layer<AT>(c1, I, B, Y, P.p[MRNB_C_CONV1_W], P.h[MRNB_C_CONV1_W], P.p[MRNB_C_CONV1_B], X, col, st));
    MRNB_TRY(launch_pool<AT>(X, Y, N, 16, 128, 128, 2, 2, st));                                            // 5   -> Y [8,64,128]
    const ConvSpec c2{8, 64, 128, 256, 3, 1, 8, 64, 1};                                                    // 6-7 -> Z [8,64,256]
    MRNB_TRY(conv_layer<AT>(c2, I, B, Y, P.p[MRNB_C_CONV2_W], P.h[MRNB_C_CONV2_W], P.p[MRNB_C_CONV2_B], Z, col, st));
    const ConvSpec c3{8, 64, 256, 256, 3, 1, 8, 64, 1};                                                    // 8-9 -> X [8,64,256]
    MRNB_TRY(conv_layer<AT>(c3, I, B, Z, P.p[MRNB_C_CONV3_W], P.h[MRNB_C_CONV3_W], P.p[MRNB_C_CONV3_B], X, col, st));
    MRNB_TRY(launch_pool<AT>(X, Y, N, 8, 64, 256, 2, 1, st));                                              // 10  -> Y [4,64,256]
    // 11-13: conv (no bias) -> BatchNorm2d -> ReLU
    const ConvSpec c4{4, 64, 256, 512, 3, 1, 4, 64, 0};                                                    // 11  -> Z raw [4,64,512]
    MRNB_TRY(conv_layer<AT>(c4, I, B, Y, P.p[MRNB_C_CONV4_W], P.h[MRNB_C_CONV4_W], nullptr, Z, col, st));
    const long rows4 = (long)B * 4 * 64;
    for (int layer = 0; layer < 2; ++layer) {
      const AT* raw = Z;
      const int bnw = layer == 0 ? MRNB_C_BN4_W : MRNB_C_BN5_W;
      if (layer == 1) {
        const ConvSpec c5{4, 64, 512, 512, 3, 1, 4, 64, 0};                                                // 14  X -> Z raw [4,64,512]
        MRNB_TRY(conv_layer<AT>(c5, I, B, X, P.p[MRNB_C_CONV5_W], P.h[MRNB_C_CONV5_W], nullptr, Z, col, st));
      }
      mrnb_prof_begin(MRNB_PROF_CONV, st, 0.0, 0.0);
      if (bn_batch_stats) {
        cudaMemsetAsync(stats, 0, (size_t)I * 512 * 2 * sizeof(double), st);
        bn_stats512_kernel<AT><<<dim3(rows4 / 64 < 64 ? (int)(rows4 / 64) : 64, I), 256, 0, st>>>(raw, rows4, stats);
        MRNB_CHECK_LAUNCH("bn_stats512_kernel");
      }
      bn_finalize_kernel<<<cdiv(I * 512, 128), 128, 0, st>>>(stats, P.p[bnw], P.p[bnw + 1], (float*)P.p[bnw + 2],
                                                             (float*)P.p[bnw + 3], ss, nullptr, I, 512, (double)rows4, bn_batch_stats,
                                                             update_running, 1e-5f);
      MRNB_CHECK_LAUNCH("bn_finalize_kernel");
      // layer 0: 12-13 -> X [4,64,512]; layer 1: 15-17 (+ MaxPool (2,1)) -> Y [2,64,512]
      const int pool_h = layer == 0 ? 1 : 2;
      const unsigned rows_out = (unsigned)B * (4 / pool_h) * 64;
      bn_relu_pool_kernel<AT><<<dim3(rows_out / 4 < 1184 ? rows_out / 4 : 1184, I), 256, 0, st>>>(raw, ss, layer == 0 ? X : Y, rows_out,
                                                                                                 4, pool_h);
      MRNB_CHECK_LAUNCH("bn_relu_pool_kernel");
      mrnb_prof_end(MRNB_PROF_CONV, st);
    }
    const ConvSpec c6{2, 64, 512, 512, 2, 0, 1, 64, 1};                                                    // 18-19 -> X [1,64(63),512]
    MRNB_TRY(conv_layer<AT>(c6, I, B, Y, P.p[MRNB_C_CONV6_W], P.h[MRNB_C_CONV6_W], P.p[MRNB_C_CONV6_B], X, col, st));
  }

  // ---- two BidirectionalLSTMs (sequence_modeling.py:12-22); visual feature = X [I][B*64][512]
  const long rowsT = (long)B * CTP;
  AT* seq_in = X; int Kin = 512;
  AT* pre = Z; AT* rec = Y;
  for (int layer = 0; layer < 2; ++layer) {
    const int pl = MRNB_C_LSTM0 + layer * MRNB_CL_COUNT;
    LinearArgs ip{};
    ip.A = seq_in; ip.lda = Kin; ip.a_gstride = rowsT * Kin;
    ip.W32 = P.p[pl + MRNB_CL_WIH]; ip.W16 = P.h[pl + MRNB_CL_WIH]; ip.w_gstride = 8L * LH * Kin;
    ip.bias = P.p[pl + MRNB_CL_BIAS]; ip.bias_gstride = 8 * LH;
    ip.out = pre; ip.ldo = 8 * LH; ip.o_gstride = rowsT * 8 * LH; ip.out_is_f32 = F32;
    ip.M = (int)rowsT; ip.N = 8 * LH; ip.K = Kin; ip.groups = I;
    MRNB_TRY(linear<AT>(ip, st));
    const long cells = (long)2 * I * B * LH;
    // tensor-core mode with whole 128-sample tiles: the cell runs inside the epilogue of the recurrent GEMM
    const bool fused_cell = !F32 && (B % 128) == 0;
    bool seq_done = false;                 // steps 1 .. CT-1 already ran in the persistent cluster kernel
    for (int s = 0; s < CT && !seq_done; ++s) {
      if (s == 1 && fused_cell && lstm_seq_enabled()) {
        // every remaining step of the layer in ONE launch: W_hh resident in shared memory, h exchanged inside 4-CTA clusters
        // (gemm_tc.cu: lstm_seq_kernel).  h ping-pongs between hst (h_0 from the cell kernel above) and the unused fp32
        // `gates` buffer.
        const int rc = mrnb_tc_lstm_seq(P.h[pl + MRNB_CL_WHH], pre, (long)CTP * 8 * LH, (long)B * CTP * 8 * LH, rec,
                                        (long)CTP * 2 * LH, (long)B * CTP * 2 * LH, cst, hst, gates, 2 * I, B, CT, 1, st);
        if (rc == MRNB_OK) { seq_done = true; break; }
        if (rc != MRNB_ERR_UNSUPPORTED) return rc;
      }
      if (s > 0 && fused_cell) {
        MrnbTcGemm g{};
        g.A = hst; g.lda = LH; g.a_gstride = (long)B * LH;
        g.W = P.h[pl + MRNB_CL_WHH]; g.ldw = LH; g.w_gstride = 4L * LH * LH;
        g.out = gates; g.ldo = 4 * LH; g.o_gstride = (long)B * 4 * LH; g.out_f32 = 1;      // not written in this mode
        g.M = B; g.N = 4 * LH; g.K = LH; g.groups = 2 * I; g.rows_per_scale = 1;
        g.lstm.enabled = 1; g.lstm.B = B;
        g.lstm.pre = pre; g.lstm.pre_row = (long)CTP * 8 * LH; g.lstm.pre_e = (long)B * CTP * 8 * LH;
        g.lstm.pre_off[0] = (long)s * 8 * LH; g.lstm.pre_off[1] = (long)(CT - 1 - s) * 8 * LH + 4 * LH;
        g.lstm.cst = cst; g.lstm.hst = hst;
        g.lstm.rec = rec; g.lstm.rec_row = (long)CTP * 2 * LH; g.lstm.rec_e = (long)B * CTP * 2 * LH;
        g.lstm.rec_off[0] = (long)s * 2 * LH; g.lstm.rec_off[1] = (long)(CT - 1 - s) * 2 * LH + LH;
        MRNB_TRY(mrnb_tc_gemm(g, st));
        continue;
      }
      if (s > 0) {
        LinearArgs hh{};
        hh.A = hst; hh.lda = LH; hh.a_gstride = (long)B * LH;
        hh.W32 = P.p[pl + MRNB_CL_WHH]; hh.W16 = P.h[pl + MRNB_CL_WHH]; hh.w_gstride = 4L * LH * LH;
        hh.out = gates; hh.ldo = 4 * LH; hh.o_gstride = (long)B * 4 * LH; hh.out_is_f32 = 1;
        hh.M = B; hh.N = 4 * LH; hh.K = LH; hh.groups = 2 * I;
        MRNB_TRY(linear<AT>(hh, st));
      }
      mrnb_prof_begin(MRNB_PROF_MISC, st, 0.0, 0.0);
      lstm_cell_kernel<AT><<<cdiv(cells, 256), 256, 0, st>>>(gates, pre, cst, hst, rec, I, B, s, (unsigned)cells);
      MRNB_CHECK_LAUNCH("lstm_cell_kernel");
      mrnb_prof_end(MRNB_PROF_MISC, st);
    }
    LinearArgs lo{};
    lo.A = rec; lo.lda = 2 * LH; lo.a_gstride = rowsT * 2 * LH;
    lo.W32 = P.p[pl + MRNB_CL_LIN_W]; lo.W16 = P.h[pl + MRNB_CL_LIN_W]; lo.w_gstride = 256L * 2 * LH;
    lo.bias = P.p[pl + MRNB_CL_LIN_B]; lo.bias_gstride = 256;
    lo.out = X; lo.ldo = 256; lo.o_gstride = rowsT * 256; lo.out_is_f32 = (layer == 1) ? 1 : F32;
    lo.M = (int)rowsT; lo.N = 256; lo.K = 2 * LH; lo.groups = I;
    MRNB_TRY(linear<AT>(lo, st));
    seq_in = X; Kin = 256;
  }

  // ---- contextual feature -> router layout + classifier heads (ragged N = C_i), T = 63 rows per sample
  {
    const long total4 = (long)I * B * CT * 64;
    mrnb_prof_begin(MRNB_PROF_MISC, st, 0.0, 0.0);
    crnn_feature_kernel<AT><<<cdiv(total4, 256), 256, 0, st>>>(reinterpret_cast<const float*>(X), features, compact, I, B, total4);
    MRNB_CHECK_LAUNCH("crnn_feature_kernel");
    mrnb_prof_end(MRNB_PROF_MISC, st);
    if (logits) {
      for (int e = 0; e < I; ++e) {
        if (!logits[e]) continue;
        LinearArgs fc{};
        fc.A = compact + (size_t)e * B * CT * 256; fc.lda = 256;
        fc.W32 = P.fc_w[e]; fc.W16 = P.fc_w16[e]; fc.bias = P.fc_b[e];
        fc.out = logits[e]; fc.ldo = ld_logits[e]; fc.out_is_f32 = 1;
        fc.M = B * CT; fc.N = P.n_class[e]; fc.K = 256; fc.groups = 1;
        MRNB_TRY(linear<AT>(fc, st));
      }
    }
  }
  return MRNB_OK;
}

}  // namespace

extern "C" size_t mrnb_crnn_workspace_bytes(int n_experts, int B, int prec) {
  return prec == MRNB_PREC_BF16 ? crnn_workspace_bytes_t<__nv_bfloat16>(n_experts, B) : crnn_workspace_bytes_t<float>(n_experts, B);
}

extern "C" int mrnb_crnn_experts_forward(const MrnbCrnnPack* pack, const float* image, int B, int prec, int bn_batch_stats,
                                         int update_running, float* features, float* const* logits, const long* ld_logits,
                                         void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  MRNB_CHECK_ARG(pack && image && workspace && B > 0, "crnn_experts_forward: null/empty argument");
  MRNB_CHECK_ARG(pack->n_experts >= 1 && pack->n_experts <= MRNB_MAX_EXPERTS, "crnn_experts_forward: n_experts out of range");
  for (int k = 0; k < MRNB_C_COUNT; ++k) MRNB_CHECK_ARG(pack->p[k], "crnn_experts_forward: parameter slot %d is null", k);
  if (prec == MRNB_PREC_BF16)
    return crnn_forward_t<__nv_bfloat16>(*pack, image, B, bn_batch_stats, update_running, features, logits, ld_logits,
                                         workspace, workspace_bytes, stream);
  if (prec == MRNB_PREC_FP32)
    return crnn_forward_t<float>(*pack, image, B, bn_batch_stats, update_running, features, logits, ld_logits, workspace,
                                 workspace_bytes, stream);
  mrnb_set_error("crnn_experts_forward: unknown precision %d", prec);
  return MRNB_ERR_ARG;
}
