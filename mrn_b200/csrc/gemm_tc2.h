// Internal descriptor of the general tcgen05 GEMM (gemm_tc2.cu).
#pragma once
#include <cuda_runtime.h>
#include "gemm_f32.h"

enum { MRNB_SRC_ZERO = 0, MRNB_SRC_MN = 1, MRNB_SRC_K = 2, MRNB_SRC_G = 3 };

// TMA coordinate j of a tile = ((value of src[j]) / div[j]) % mod[j]   (div <= 1: no division, mod == 0: no modulo);
// flip[j] > 0 mirrors it afterwards: flip[j] - 1 - coordinate (walks a dimension backwards, e.g. groups stored in
// descending address order)
struct MrnbTmaRecipe { int src[4]; int div[4]; int mod[4]; int flip[4]; };

// A bf16 operand seen through a rank-4 TMA tensor map (dim 0 contiguous, 64 elements = 128 B inner box).
struct MrnbTcOperand {
  const void* ptr;
  int mn_major;          // 0: dim 0 walks k (K-major); 1: dim 0 walks m / n (MN-major), one 64-wide chunk per TMA load
  long dims[4];
  long strides[3];       // elements, for dims 1..3
  int box[4];
  MrnbTmaRecipe recipe;
};

struct MrnbTcGemm2 {
  MrnbTcOperand a, b;
  float* out32; void* out16;            // fp32 and / or bf16 output at the same element offsets
  MrnbAxis cm, cn; long c_gstride;      // two-level output addressing (elements)
  int g_inner; long c_gstride2;         // g_inner > 0: group offset = (g / g_inner) * c_gstride + (g % g_inner) * c_gstride2
  const float* bias_n; const float* bias_m; const float* mul; const float* res;
  float* pre32;                         // optional fp32 copy of the value before `mul` / `res` (same element offsets)
  int M, N, K, groups, splitk, gelu;
  float alpha;
};

// [groups][rows][K] with k contiguous
static inline MrnbTcOperand mrnb_operand_k2d(const void* p, long rows, long K, long ld, int box_rows, long groups, long gstride = 0) {
  MrnbTcOperand o{};
  if (gstride == 0) gstride = rows * ld;
  o.ptr = p; o.mn_major = 0;
  o.dims[0] = K; o.dims[1] = rows; o.dims[2] = groups; o.dims[3] = 1;
  o.strides[0] = ld; o.strides[1] = gstride; o.strides[2] = gstride * groups;
  o.box[0] = 64; o.box[1] = box_rows; o.box[2] = 1; o.box[3] = 1;
  o.recipe = MrnbTmaRecipe{{MRNB_SRC_K, MRNB_SRC_MN, MRNB_SRC_G, MRNB_SRC_ZERO}, {1, 1, 1, 1}, {0, 0, 0, 0}};
  return o;
}
// [groups][K][MN] with m / n contiguous
static inline MrnbTcOperand mrnb_operand_mn2d(const void* p, long MN, long K, long ld, long groups, long gstride = 0) {
  MrnbTcOperand o{};
  if (gstride == 0) gstride = K * ld;
  o.ptr = p; o.mn_major = 1;
  o.dims[0] = MN; o.dims[1] = K; o.dims[2] = groups; o.dims[3] = 1;
  o.strides[0] = ld; o.strides[1] = gstride; o.strides[2] = gstride * groups;
  o.box[0] = 64; o.box[1] = 64; o.box[2] = 1; o.box[3] = 1;
  o.recipe = MrnbTmaRecipe{{MRNB_SRC_MN, MRNB_SRC_K, MRNB_SRC_G, MRNB_SRC_ZERO}, {1, 1, 1, 1}, {0, 0, 0, 0}};
  return o;
}

// One attention head of a [groups][rows][ld] tensor whose heads are 32-wide column slices: (row, k) of group g = b * heads + h
// is ptr[(b * rows + row) * ld + h * 32 + k].  K-major: k walks the head dimension; MN-major: the head dimension is m / n.
// The 64-wide TMA box is half outside the 32-wide slice: the hardware zero-fills it (the GEMM runs with K or N padded).
static inline MrnbTcOperand mrnb_operand_head(const void* p, long rows, long ld, int heads, long batch, int mn_major, int box_rows) {
  MrnbTcOperand o{};
  o.ptr = p; o.mn_major = mn_major;
  o.dims[0] = 32; o.dims[1] = rows; o.dims[2] = heads; o.dims[3] = batch;
  o.strides[0] = ld; o.strides[1] = 32; o.strides[2] = rows * ld;
  o.box[0] = 64; o.box[1] = mn_major ? 64 : box_rows; o.box[2] = 1; o.box[3] = 1;
  if (mn_major) o.recipe = MrnbTmaRecipe{{MRNB_SRC_MN, MRNB_SRC_K, MRNB_SRC_G, MRNB_SRC_G}, {1, 1, 1, heads}, {0, 0, heads, 0}};
  else o.recipe = MrnbTmaRecipe{{MRNB_SRC_K, MRNB_SRC_MN, MRNB_SRC_G, MRNB_SRC_G}, {1, 1, 1, heads}, {0, 0, heads, 0}};
  return o;
}

int mrnb_tc_gemm2(const MrnbTcGemm2& p, cudaStream_t st);
