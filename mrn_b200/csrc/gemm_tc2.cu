// General tcgen05 GEMM: the router's contractions (modules/dm_router.py:50-67 and their backward) on the tensor cores.
//
//   C(g, m, n) (+)= epi( sum_k A(g, m, k) * B(g, k, n) )
//
// Differences from gemm_tc.cu (the plain grouped Linear of the expert path):
//   * each operand is K-major (k contiguous in HBM) or MN-major (m / n contiguous): `X^T . Y` weight gradients and
//     `dY . W` input gradients read the tensors where they lie -- no transposed copies;
//   * operands are described by rank-4 TMA tensor maps plus a coordinate recipe, so the reference's rearranges
//     ('b d p c -> b (d p) c', 'b d p c -> b (d c) p') are box orientations, not copies;
//   * two-level output addressing (same MrnbAxis as gemm_f32.cu), split-K with fp32 atomics, and an epilogue with
//     bias over n or m, exact GELU, an elementwise multiplier and a residual at the output address.
// bf16 operands, fp32 accumulation in TMEM.  128 x BN output tiles, BN = 128 for N >= 128 and 64 below, walked by two
// persistent CTAs per SM (router GEMMs have K >= 256).
#include "gemm_f32.h"
#include "gemm_tc2.h"
#include "sm100.cuh"

namespace {

constexpr int BM = 128, BK = 64, UMMA_K = 16;
constexpr int STAGES = 3;              // operand ring: 3 x <= 32 KiB, so that two CTAs fit one SM
constexpr int A_BYTES = BM * BK * 2;

__device__ __forceinline__ void red_add_v4(float* p, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// the k-dependent coordinates only (dims sourced from k), the others are left as they are: the producer computes the
// m/n- and group-sourced coordinates once per tile and refreshes only these per k-block (a single thread issues every
// TMA of the CTA: its integer divisions were the limiter of the MN-major weight-gradient GEMMs)
__device__ __forceinline__ void recipe_coords_k(const MrnbTmaRecipe& r, int k, int (&c)[4]) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if (r.src[j] != MRNB_SRC_K) continue;
    int v = k;
    if (r.div[j] > 1) v /= r.div[j];
    if (r.mod[j] > 0) v %= r.mod[j];
    if (r.flip[j] > 0) v = r.flip[j] - 1 - v;
    c[j] = v;
  }
}
__device__ __forceinline__ void recipe_coords(const MrnbTmaRecipe& r, int mn, int k, int g, int (&c)[4]) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    int v = r.src[j] == MRNB_SRC_MN ? mn : (r.src[j] == MRNB_SRC_K ? k : (r.src[j] == MRNB_SRC_G ? g : 0));
    if (r.div[j] > 1) v /= r.div[j];
    if (r.mod[j] > 0) v %= r.mod[j];
    if (r.flip[j] > 0) v = r.flip[j] - 1 - v;
    c[j] = v;
  }
}

struct Epi2 {
  float* out32; __nv_bfloat16* out16;     // either or both
  MrnbAxis cm, cn; long c_gs;
  int g_inner; long c_gs2;
  const float* bias_n; const float* bias_m;
  const float* mul; const float* res;
  float* pre32;                           // optional: the value before `mul` / `res` (same element offsets)
  int M, N, KB_total, kb_per_split, splits, gelu;
  int tiles_n, tiles_m; long total_tiles;
  int simple;      // plain row-major output addressing: the lean epilogue (whole-line vector loads / stores / reductions)
  float alpha;
};

// Persistent: each CTA walks tiles t = blockIdx.x, blockIdx.x + gridDim.x, ... (n-tile fastest, then m-tile, then
// group x split).  Barriers, TMEM and the tensor-map prefetch are set up once; the accumulator is double buffered in
// TMEM (2 x BN columns) so the epilogue of tile i overlaps the loads and MMAs of tile i + 1 -- the router / backward
// GEMMs have 1..8 k-blocks per tile, where the per-tile fixed cost used to dominate.
template <int BN, bool A_MN, bool B_MN>
__global__ void __launch_bounds__(192)
tc_gemm2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                const MrnbTmaRecipe ra, const MrnbTmaRecipe rb, const Epi2 ep) {
  extern __shared__ uint8_t smem_raw[];
  constexpr int B_BYTES = BN * BK * 2;
  constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  uint8_t* smem = smem_raw + align_smem_1024_offset(smem_raw);
  __shared__ __align__(8) uint64_t full_bar[STAGES];
  __shared__ __align__(8) uint64_t empty_bar[STAGES];
  __shared__ __align__(8) uint64_t tmem_full_bar[2];
  __shared__ __align__(8) uint64_t tmem_empty_bar[2];
  __shared__ uint32_t tmem_base_sh;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tiles_n = ep.tiles_n, tiles_m = ep.tiles_m;
  const long total = ep.total_tiles;

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&tmem_full_bar[a], 1); mbar_init(&tmem_empty_bar[a], 4); }
    fence_mbarrier_init();
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
  }
  if (warp == 1) tmem_alloc(&tmem_base_sh, 2 * BN);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_sh;

  auto tile_coords = [&](long t, int& n0, int& m0, int& g, int& kb0, int& KB) {
    n0 = (int)(t % tiles_n) * BN;
    long r = t / tiles_n;
    m0 = (int)(r % tiles_m) * BM;
    const int z = (int)(r / tiles_m);
    g = z / ep.splits;
    const int split = z % ep.splits;
    kb0 = split * ep.kb_per_split;
    int kb1 = kb0 + ep.kb_per_split;
    if (kb1 > ep.KB_total) kb1 = ep.KB_total;
    KB = kb1 - kb0;                               // host guarantees KB >= 1
  };

  if (warp == 0) {
    if (lane == 0) {
      uint32_t it = 0;
      for (long t = blockIdx.x; t < total; t += gridDim.x) {
        int n0, m0, g, kb0, KB;
        tile_coords(t, n0, m0, g, kb0, KB);
        constexpr int ACH = A_MN ? BM / 64 : 1, BCH = B_MN ? BN / 64 : 1;
        int ca[ACH][4], cb[BCH][4];
#pragma unroll
        for (int ch = 0; ch < ACH; ++ch) recipe_coords(ra, m0 + ch * 64, kb0 * BK, g, ca[ch]);
#pragma unroll
        for (int ch = 0; ch < BCH; ++ch) recipe_coords(rb, n0 + ch * 64, kb0 * BK, g, cb[ch]);
        for (int i = 0; i < KB; ++i, ++it) {
          const int s = it % STAGES;
          const uint32_t ph = (it / STAGES) & 1u;
          const int k0 = (kb0 + i) * BK;
          if (i > 0) {
#pragma unroll
            for (int ch = 0; ch < ACH; ++ch) recipe_coords_k(ra, k0, ca[ch]);
#pragma unroll
            for (int ch = 0; ch < BCH; ++ch) recipe_coords_k(rb, k0, cb[ch]);
          }
          mbar_wait(&empty_bar[s], ph ^ 1u);
          mbar_expect_tx(&full_bar[s], STAGE_BYTES);
          uint8_t* sa = smem + (size_t)s * STAGE_BYTES;
#pragma unroll
          for (int ch = 0; ch < ACH; ++ch)
            tma_load_4d(sa + ch * (BK * 128), &tmA, &full_bar[s], ca[ch][0], ca[ch][1], ca[ch][2], ca[ch][3]);
#pragma unroll
          for (int ch = 0; ch < BCH; ++ch)
            tma_load_4d(sa + A_BYTES + ch * (BK * 128), &tmB, &full_bar[s], cb[ch][0], cb[ch][1], cb[ch][2], cb[ch][3]);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = umma_idesc(UMMA_BF16, BM, BN, A_MN, B_MN);
      uint32_t it = 0, ti = 0;
      for (long t = blockIdx.x; t < total; t += gridDim.x, ++ti) {
        int n0, m0, g, kb0, KB;
        tile_coords(t, n0, m0, g, kb0, KB);
        const uint32_t acc = ti & 1u;
        mbar_wait(&tmem_empty_bar[acc], ((ti >> 1) & 1u) ^ 1u);       // epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + acc * (uint32_t)BN;
        for (int i = 0; i < KB; ++i, ++it) {
          const int s = it % STAGES;
          const uint32_t ph = (it / STAGES) & 1u;
          mbar_wait(&full_bar[s], ph);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + (size_t)s * STAGE_BYTES);
          // 128B-swizzled tiles.  K-major: rows of 128 B (64 k), 8-row atoms 1024 B apart along M/N; MN-major: rows of
          // 128 B (64 m/n), one row per k, 8-k atoms 1024 B apart, 64-wide MN chunks BK * 128 B apart (LBO)
          const uint64_t adesc = umma_smem_desc(sa, A_MN ? BK * 128 : 16, 1024, UMMA_SWIZZLE_128B);
          const uint64_t bdesc = umma_smem_desc(sa + A_BYTES, B_MN ? BK * 128 : 16, 1024, UMMA_SWIZZLE_128B);
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) {
            // K-major: +32 B inside the swizzled row; MN-major: +16 k-rows of 128 B
            const uint64_t aoff = A_MN ? (uint64_t)(k * UMMA_K * 128 >> 4) : (uint64_t)(k * 2);
            const uint64_t boff = B_MN ? (uint64_t)(k * UMMA_K * 128 >> 4) : (uint64_t)(k * 2);
            umma_bf16(tmem_d, adesc + aoff, bdesc + boff, idesc, (i | k) != 0 ? 1u : 0u);
          }
          umma_commit(&empty_bar[s]);
        }
        umma_commit(&tmem_full_bar[acc]);
      }
    }
  } else {
    const int q = warp & 3;
    const bool plain = ep.splits == 1;
    uint32_t ti = 0;
    for (long t = blockIdx.x; t < total; t += gridDim.x, ++ti) {
      int n0, m0, g, kb0, KB;
      tile_coords(t, n0, m0, g, kb0, KB);
      const uint32_t acc = ti & 1u;
      const int row = m0 + q * 32 + lane;
      mbar_wait(&tmem_full_bar[acc], (ti >> 1) & 1u);
      tc_fence_after();
      const bool rok = row < ep.M;
      const long og = ep.g_inner > 0 ? (long)(g / ep.g_inner) * ep.c_gs + (long)(g % ep.g_inner) * ep.c_gs2 : (long)g * ep.c_gs;
      const long om = rok ? og + (long)(row / ep.cm.inner) * ep.cm.so + (long)(row % ep.cm.inner) * ep.cm.si : 0;
      const float bm = (ep.bias_m && rok) ? ep.bias_m[row] : 0.f;
      if (ep.simple) {
        // lean epilogue: 32 columns per TMEM load, a whole 128-byte line of the row per thread, no index arithmetic.
        // simple == 1: plain row-major output; simple == 2: two-level addressing whose BN columns of a tile are contiguous
        // (cn.si == 1, cn.inner a multiple of BN): the row base takes the two-level row offset + the tile's column base
        const long orow = ep.simple == 1 ? og + (long)row * ep.cm.si
                                         : om + (long)(n0 / ep.cn.inner) * ep.cn.so + (long)(n0 % ep.cn.inner) - n0;
#pragma unroll 1
        for (int c0 = 0; c0 < BN; c0 += 32) {
          const int col0 = n0 + c0;
          if (col0 >= ep.N) break;                                    // warp-uniform
          uint32_t r[32];
          tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + acc * (uint32_t)BN + (uint32_t)c0, r);
          if (!rok) continue;
          const long o = orow + col0;
          if (col0 + 32 <= ep.N && (o & 3) == 0) {
            if (!plain) {
#pragma unroll
              for (int j = 0; j < 32; j += 4)
                red_add_v4(ep.out32 + o + j, __uint_as_float(r[j]) * ep.alpha, __uint_as_float(r[j + 1]) * ep.alpha,
                           __uint_as_float(r[j + 2]) * ep.alpha, __uint_as_float(r[j + 3]) * ep.alpha);
            } else {
              float v[32];
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]) * ep.alpha + bm;
              if (ep.bias_n) {
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                  const float4 b4 = __ldg(reinterpret_cast<const float4*>(ep.bias_n + col0 + j));
                  v[j] += b4.x; v[j + 1] += b4.y; v[j + 2] += b4.z; v[j + 3] += b4.w;
                }
              }
              if (ep.gelu) {
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = gelu_erf(v[j]);
              }
              if (ep.pre32) {
#pragma unroll
                for (int j = 0; j < 32; j += 4)
                  *reinterpret_cast<float4*>(ep.pre32 + o + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
              }
              if (ep.mul) {
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                  const float4 m4 = *reinterpret_cast<const float4*>(ep.mul + o + j);
                  v[j] *= m4.x; v[j + 1] *= m4.y; v[j + 2] *= m4.z; v[j + 3] *= m4.w;
                }
              }
              if (ep.res) {
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                  const float4 r4 = *reinterpret_cast<const float4*>(ep.res + o + j);
                  v[j] += r4.x; v[j + 1] += r4.y; v[j + 2] += r4.z; v[j + 3] += r4.w;
                }
              }
              if (ep.out32) {
#pragma unroll
                for (int j = 0; j < 32; j += 4)
                  *reinterpret_cast<float4*>(ep.out32 + o + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
              }
              if (ep.out16) {
#pragma unroll
                for (int j = 0; j < 32; j += 8) {
                  uint32_t pk[4];
#pragma unroll
                  for (int u = 0; u < 4; ++u) {
                    __nv_bfloat162 h = __floats2bfloat162_rn(v[j + 2 * u], v[j + 2 * u + 1]);
                    pk[u] = *reinterpret_cast<uint32_t*>(&h);
                  }
                  *reinterpret_cast<uint4*>(ep.out16 + o + j) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                }
              }
            }
          } else {
            for (int j = 0; j < 32; ++j) {
              if (col0 + j >= ep.N) break;
              float x = __uint_as_float(r[j]) * ep.alpha;
              if (!plain) { atomicAdd(ep.out32 + o + j, x); continue; }
              x += bm;
              if (ep.bias_n) x += __ldg(ep.bias_n + col0 + j);
              if (ep.gelu) x = gelu_erf(x);
              if (ep.pre32) ep.pre32[o + j] = x;
              if (ep.mul) x *= ep.mul[o + j];
              if (ep.res) x += ep.res[o + j];
              if (ep.out32) ep.out32[o + j] = x;
              if (ep.out16) ep.out16[o + j] = __float2bfloat16_rn(x);
            }
          }
        }
      } else
#pragma unroll 1
      for (int c0 = 0; c0 < BN; c0 += 16) {
        uint32_t r[16];
        tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + acc * (uint32_t)BN + (uint32_t)c0, r);
        const int col0 = n0 + c0;
        if (!rok || col0 >= ep.N) continue;
        // contiguous run of 16 columns?
        const bool contig = ep.cn.si == 1 && (col0 % ep.cn.inner) + 16 <= ep.cn.inner && col0 + 16 <= ep.N;
        const long on0 = (long)(col0 / ep.cn.inner) * ep.cn.so + (long)(col0 % ep.cn.inner) * ep.cn.si;
        float v[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          float x = __uint_as_float(r[j]) * ep.alpha;
          if (plain) {
            x += bm;
            if (ep.bias_n && col0 + j < ep.N) x += __ldg(ep.bias_n + col0 + j);
            if (ep.gelu) x = gelu_erf(x);
          }
          v[j] = x;
        }
        if (!plain) {
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const int col = col0 + j;
            if (col >= ep.N) break;
            const long o = om + (contig ? on0 + j : (long)(col / ep.cn.inner) * ep.cn.so + (long)(col % ep.cn.inner) * ep.cn.si);
            atomicAdd(ep.out32 + o, v[j]);
          }
          continue;
        }
        if (contig && ((om + on0) & 3) == 0) {
          const long o = om + on0;
#pragma unroll
          for (int j = 0; j < 16; j += 4) {
            float4 tt = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
            if (ep.pre32) *reinterpret_cast<float4*>(ep.pre32 + o + j) = tt;
            if (ep.mul) { const float4 mm = *reinterpret_cast<const float4*>(ep.mul + o + j); tt.x *= mm.x; tt.y *= mm.y; tt.z *= mm.z; tt.w *= mm.w; }
            if (ep.res) { const float4 rr = *reinterpret_cast<const float4*>(ep.res + o + j); tt.x += rr.x; tt.y += rr.y; tt.z += rr.z; tt.w += rr.w; }
            if (ep.out32) *reinterpret_cast<float4*>(ep.out32 + o + j) = tt;
            if (ep.out16) {
              __nv_bfloat162 h0 = __floats2bfloat162_rn(tt.x, tt.y), h1 = __floats2bfloat162_rn(tt.z, tt.w);
              *reinterpret_cast<uint2*>(ep.out16 + o + j) = make_uint2(*reinterpret_cast<uint32_t*>(&h0), *reinterpret_cast<uint32_t*>(&h1));
            }
          }
        } else {
          for (int j = 0; j < 16; ++j) {
            const int col = col0 + j;
            if (col >= ep.N) break;
            const long o = om + (long)(col / ep.cn.inner) * ep.cn.so + (long)(col % ep.cn.inner) * ep.cn.si;
            float x = v[j];
            if (ep.pre32) ep.pre32[o] = x;
            if (ep.mul) x *= ep.mul[o];
            if (ep.res) x += ep.res[o];
            if (ep.out32) ep.out32[o] = x;
            if (ep.out16) ep.out16[o] = __float2bfloat16_rn(x);
          }
        }
      }
      // this warp has read its 32 lanes of the accumulator: hand the buffer back to the MMA warp
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty_bar[acc]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 2 * BN);
}

int encode(CUtensorMap* map, const MrnbTcOperand& op) {
  cuuint64_t dims[4], strides[3];
  cuuint32_t box[4], es[4] = {1, 1, 1, 1};
  for (int j = 0; j < 4; ++j) { dims[j] = (cuuint64_t)op.dims[j]; box[j] = (cuuint32_t)op.box[j]; }
  for (int j = 0; j < 3; ++j) strides[j] = (cuuint64_t)op.strides[j] * 2;       // bytes, dims 1..3
  if ((reinterpret_cast<uintptr_t>(op.ptr) & 15) || op.box[0] != 64) {
    mrnb_set_error("tc_gemm2: operand misaligned or inner box != 64");
    return MRNB_ERR_ARG;
  }
  for (int j = 0; j < 3; ++j)
    if ((op.strides[j] * 2) % 16) { mrnb_set_error("tc_gemm2: stride %d not a multiple of 16 bytes", j); return MRNB_ERR_ARG; }
  return encode_tensor_map("tc_gemm2", map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, op.ptr, dims, strides, box, es, CU_TENSOR_MAP_SWIZZLE_128B);
}

template <int BN, bool A_MN, bool B_MN>
int launch2(const MrnbTcGemm2& p, cudaStream_t st) {
  CUtensorMap tmA, tmB;
  MRNB_TRY(encode(&tmA, p.a));
  MRNB_TRY(encode(&tmB, p.b));
  Epi2 ep{};
  ep.out32 = p.out32; ep.out16 = (__nv_bfloat16*)p.out16; ep.cm = p.cm; ep.cn = p.cn; ep.c_gs = p.c_gstride;
  ep.g_inner = p.g_inner; ep.c_gs2 = p.c_gstride2;
  ep.bias_n = p.bias_n; ep.bias_m = p.bias_m; ep.mul = p.mul; ep.res = p.res; ep.pre32 = p.pre32;
  ep.M = p.M; ep.N = p.N; ep.gelu = p.gelu; ep.alpha = p.alpha == 0.f ? 1.f : p.alpha;
  ep.KB_total = p.K / BK;
  int splits = p.splitk > 1 ? p.splitk : 1;
  if (splits > ep.KB_total) splits = ep.KB_total;
  ep.kb_per_split = (ep.KB_total + splits - 1) / splits;
  splits = (ep.KB_total + ep.kb_per_split - 1) / ep.kb_per_split;     // no empty split
  ep.splits = splits;
  const size_t smem = 1024 + (size_t)STAGES * (A_BYTES + BN * BK * 2);
  static bool attr = false;
  if (!attr) { cudaFuncSetAttribute(tc_gemm2_kernel<BN, A_MN, B_MN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); attr = true; }
  ep.simple = (p.cn.si == 1 && p.cn.inner >= p.N && p.cm.inner >= p.M) ? 1 : 0;
  if (!ep.simple && p.cn.si == 1 && p.cn.inner % BN == 0 && p.N % BN == 0 && (p.cn.so % 4) == 0 && (p.cm.si % 4) == 0 &&
      (p.cm.so % 4) == 0 && p.splitk <= 1)
    ep.simple = 2;
  ep.tiles_n = cdiv(p.N, BN); ep.tiles_m = cdiv(p.M, BM);
  ep.total_tiles = (long)ep.tiles_n * ep.tiles_m * p.groups * splits;
  static int n_sm = 0;
  if (!n_sm) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev); if (n_sm <= 0) n_sm = 148; }
  // two CTAs per SM: 2 x (2 x BN <= 256) TMEM columns, 2 x <= 97 KiB smem
  const long cap = 2L * n_sm;
  const int grid = (int)(ep.total_tiles < cap ? ep.total_tiles : cap);
  tc_gemm2_kernel<BN, A_MN, B_MN><<<grid, 192, smem, st>>>(tmA, tmB, p.a.recipe, p.b.recipe, ep);
  MRNB_CHECK_LAUNCH("tc_gemm2_kernel");
  return MRNB_OK;
}

}  // namespace

int mrnb_tc_gemm2(const MrnbTcGemm2& p, cudaStream_t st) {
  MRNB_CHECK_ARG(p.a.ptr && p.b.ptr && (p.out32 || p.out16) && p.M > 0 && p.N > 0 && p.K > 0 && p.groups > 0, "tc_gemm2: bad argument");
  MRNB_CHECK_ARG(p.K % BK == 0, "tc_gemm2: K=%d must be a multiple of 64", p.K);
  MRNB_CHECK_ARG(p.splitk <= 1 || (p.out32 && !p.out16 && !p.pre32 && !p.bias_n && !p.bias_m && !p.mul && !p.res && !p.gelu),
                 "tc_gemm2: split-K supports a raw fp32 accumulate only");
  MrnbProfScope prof(MRNB_PROF_TCGEMM2, st, 2.0 * p.M * p.N * p.K * p.groups,
                     (double)p.groups * (2.0 * p.M * p.K + 2.0 * p.N * p.K + 4.0 * p.M * p.N));
#define GO(BN_)                                                                                   \
  if (p.a.mn_major && p.b.mn_major) return launch2<BN_, true, true>(p, st);                       \
  if (p.a.mn_major) return launch2<BN_, true, false>(p, st);                                      \
  if (p.b.mn_major) return launch2<BN_, false, true>(p, st);                                      \
  return launch2<BN_, false, false>(p, st);
  if (p.N >= 128) { GO(128) } else { GO(64) }
#undef GO
}

// ---- C-ABI test entry: plain 2-D operands in any of the four major-ness combinations -------------------------
//   a_mn = 0: A is [M,K] (k contiguous)   a_mn = 1: A is stored [K,M] (m contiguous)
//   b_mn = 0: B is [N,K] (k contiguous)   b_mn = 1: B is stored [K,N] (n contiguous)
extern "C" int mrnb_tc_gemm_general(const void* A, int a_mn, const void* B, int b_mn, float* out, int M, int N, int K,
                                    int splitk, cudaStream_t stream) {
  MrnbTcGemm2 g{};
  g.a = a_mn ? mrnb_operand_mn2d(A, M, K, M, 1) : mrnb_operand_k2d(A, M, K, K, BM, 1);
  const int bn = N >= 128 ? 128 : 64;
  g.b = b_mn ? mrnb_operand_mn2d(B, N, K, N, 1) : mrnb_operand_k2d(B, N, K, K, bn, 1);
  g.out32 = out; g.cm = mrnb_axis(N); g.cn = mrnb_axis(1);
  g.M = M; g.N = N; g.K = K; g.groups = 1; g.splitk = splitk; g.alpha = 1.f;
  return mrnb_tc_gemm2(g, stream);
}
