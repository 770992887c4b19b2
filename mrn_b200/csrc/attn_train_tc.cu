// Training attention, the score side on the tensor cores with the row-wise epilogue fused (bf16 mode of the stage-0 step).
//
//   FWD : S = scale * Q K^T for 128 queries x ALL N keys of one (sample, head) accumulated in TMEM (N <= 512 fp32
//         columns = the whole tensor memory of an SM at N = 512) -> the epilogue thread that owns a query row reads its
//         row back (tcgen05.ld), applies the Local window (modules/svtr.py:116-128), max / sum / normalise ->
//         P (bf16, kept for the backward).  The fp32 score matrix never reaches HBM.
//   BWD : dP = dO V^T the same way -> dS = P * (dP - D), D = dO . O per row -> dS (bf16).
// The value-side contractions (O = P V, dV = P^T dO, dQ = scale dS K, dK = scale dS^T Q) stay batched GEMMs on
// gemm_tc2.cu.  Reference: modules/svtr.py:133-152 (Attention.forward) and its autograd backward.
//
// One persistent CTA walks work items (g = b * heads + h, 128-query tile); operands arrive by TMA as 32-wide head slices
// of the [rows, ld] token tensors (64-wide box, the upper half zero-filled by the hardware, only the two non-zero
// k-steps are issued); shared memory is double buffered so the loads of item i + 1 overlap the epilogue of item i.
#include "gemm_tc2.h"
#include "sm100.cuh"

namespace {

constexpr int BM = 128, BK = 64;
typedef __nv_bfloat16 bf16;

struct SpArgs {
  bf16* P;                 // FWD: out probabilities; BWD: in probabilities      [GH][N][N]
  bf16* dS;                // BWD out
  const float* dO;         // BWD: [B*N, d] fp32 (for D)
  const bf16* O;           // BWD: [B*N, d] attention output
  int heads, d, wshift, local;   // key grid width W = 1 << wshift
  long items;              // GH * (N / 128)
  float scale;
};

// MODE 0: forward (scores -> softmax -> P).  MODE 1: backward (dP -> dS).
// Block: warp 0 = TMA producer, warp 1 = MMA issuer, warps 2..17 = epilogue.  Each TMEM lane quarter (32 query rows) is
// served by FOUR epilogue warps that split the N key columns; row maxima / sums are exchanged through shared memory.
constexpr int EPI_WARPS = 16, NTHREADS = 64 + EPI_WARPS * 32;

__device__ __forceinline__ void epi_sync() { asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory"); }

// MODE 0: forward, all keys visible.  MODE 2: forward, Local window.  MODE 1: backward (dP -> dS).
template <int N, int MODE>
__global__ void __launch_bounds__(NTHREADS)
attn_sp_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const SpArgs a) {
  extern __shared__ uint8_t smem_raw[];
  constexpr int A_BYTES = BM * BK * 2, B_BYTES = N * BK * 2, STAGE_BYTES = A_BYTES + B_BYTES;
  constexpr int MT = N / BM;
  uint8_t* smem = smem_raw + align_smem_1024_offset(smem_raw);
  __shared__ __align__(8) uint64_t full_bar[2];
  __shared__ __align__(8) uint64_t empty_bar[2];
  __shared__ __align__(8) uint64_t tmem_full_bar;
  __shared__ __align__(8) uint64_t tmem_empty_bar;
  __shared__ uint32_t tmem_base_sh;
  __shared__ float red_max[4][BM], red_sum[4][BM];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s < 2; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    mbar_init(&tmem_full_bar, 1); mbar_init(&tmem_empty_bar, EPI_WARPS);
    fence_mbarrier_init();
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
  }
  if (warp == 1) tmem_alloc(&tmem_base_sh, N);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_sh;

  if (warp == 0) {
    if (lane == 0) {
      uint32_t it = 0;
      for (long t = blockIdx.x; t < a.items; t += gridDim.x, ++it) {
        const int s = it & 1;
        const uint32_t ph = (it >> 1) & 1u;
        const int g = (int)(t / MT), m0 = (int)(t % MT) * BM;
        const int h = g % a.heads, b = g / a.heads;
        mbar_wait(&empty_bar[s], ph ^ 1u);
        mbar_expect_tx(&full_bar[s], STAGE_BYTES);
        uint8_t* sa = smem + (size_t)s * STAGE_BYTES;
        tma_load_4d(sa, &tmA, &full_bar[s], 0, m0, h, b);
#pragma unroll
        for (int j = 0; j < MT; ++j) tma_load_4d(sa + A_BYTES + j * (BM * BK * 2), &tmB, &full_bar[s], 0, j * BM, h, b);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr int UN = N >= 256 ? 256 : N;                      // columns per MMA instruction
      constexpr uint32_t idesc = umma_idesc(UMMA_BF16, BM, UN);
      uint32_t it = 0;
      for (long t = blockIdx.x; t < a.items; t += gridDim.x, ++it) {
        const int s = it & 1;
        mbar_wait(&tmem_empty_bar, (it & 1u) ^ 1u);               // the epilogue has drained the accumulator
        mbar_wait(&full_bar[s], (it >> 1) & 1u);
        tc_fence_after();
        const uint32_t sa = smem_u32(smem + (size_t)s * STAGE_BYTES);
        const uint64_t adesc = umma_desc_k128(sa);
#pragma unroll
        for (int nb = 0; nb < N / UN; ++nb) {
          const uint64_t bdesc = umma_desc_k128(sa + A_BYTES + nb * UN * BK * 2);
#pragma unroll
          for (int k = 0; k < 2; ++k)                              // head_dim 32 = two 16-wide k-steps; the rest of the box is zero
            umma_bf16(tmem_base + (uint32_t)(nb * UN), adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc, k != 0 ? 1u : 0u);
        }
        umma_commit(&empty_bar[s]);
        umma_commit(&tmem_full_bar);
      }
    }
  } else {
    const int q = warp & 3;                                        // TMEM lane quarter this warp may read
    const int cg = (warp - 2) >> 2;                                // which quarter of the key columns it owns
    constexpr int CW = N / 4;                                      // columns per thread
    const int rr = q * 32 + lane;                                  // row inside the tile
    uint32_t it = 0;
    for (long t = blockIdx.x; t < a.items; t += gridDim.x, ++it) {
      const int g = (int)(t / MT), m0 = (int)(t % MT) * BM;
      const int n = m0 + rr;                                       // query row inside the (sample, head)
      const long prow = ((long)g * N + n) * N;
      mbar_wait(&tmem_full_bar, it & 1u);
      tc_fence_after();
      const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16);
      if (MODE != 1) {
        constexpr bool LOCAL = MODE == 2;
        const float sc2 = a.scale * 1.4426950408889634f;            // exp(scale x - m) = 2^(sc2 x - m2)
        const int wmask = (1 << a.wshift) - 1;
        const int nh = n >> a.wshift, nw = n & wmask;
        // visibility of the 32 keys of chunk c0 as a bit mask (a chunk lies inside one row of the key grid: W >= 32)
        auto chunk_mask = [&](int c0) -> uint32_t {
          if (!LOCAL) return 0xffffffffu;
          const int dh = (c0 >> a.wshift) - nh;
          if (dh < -3 || dh > 3) return 0u;
          const int base = c0 & wmask;
          const int lo = max(nw - 5 - base, 0), hi = min(nw + 5 - base, 31);
          if (hi < lo) return 0u;
          return (0xffffffffu >> (31 - hi)) & (0xffffffffu << lo);
        };
        float mx = -INFINITY;
#pragma unroll 1
        for (int c0 = cg * CW; c0 < (cg + 1) * CW; c0 += 32) {
          uint32_t r[32];
          tmem_ld32(trow + (uint32_t)c0, r);
          const uint32_t vm = chunk_mask(c0);
          if (vm == 0u) continue;
#pragma unroll
          for (int j = 0; j < 32; ++j) if (!LOCAL || ((vm >> j) & 1u)) mx = fmaxf(mx, __uint_as_float(r[j]));
        }
        red_max[cg][rr] = mx;
        epi_sync();
        mx = fmaxf(fmaxf(red_max[0][rr], red_max[1][rr]), fmaxf(red_max[2][rr], red_max[3][rr])) * sc2;
        float sum = 0.f;
#pragma unroll 1
        for (int c0 = cg * CW; c0 < (cg + 1) * CW; c0 += 32) {
          uint32_t r[32];
          tmem_ld32(trow + (uint32_t)c0, r);
          const uint32_t vm = chunk_mask(c0);
          if (vm == 0u) continue;
#pragma unroll
          for (int j = 0; j < 32; ++j) if (!LOCAL || ((vm >> j) & 1u)) sum += ex2_approx(fmaf(__uint_as_float(r[j]), sc2, -mx));
        }
        red_sum[cg][rr] = sum;
        epi_sync();
        const float inv = 1.0f / ((red_sum[0][rr] + red_sum[1][rr]) + (red_sum[2][rr] + red_sum[3][rr]));
#pragma unroll 1
        for (int c0 = cg * CW; c0 < (cg + 1) * CW; c0 += 32) {
          uint32_t r[32];
          tmem_ld32(trow + (uint32_t)c0, r);
          const uint32_t vm = chunk_mask(c0);
          uint4* dst = reinterpret_cast<uint4*>(a.P + prow + c0);
          if (vm == 0u) {
#pragma unroll
            for (int u = 0; u < 4; ++u) dst[u] = make_uint4(0u, 0u, 0u, 0u);
            continue;
          }
          uint32_t pk[16];
#pragma unroll
          for (int j = 0; j < 32; j += 2) {
            const float p0 = (!LOCAL || ((vm >> j) & 1u)) ? ex2_approx(fmaf(__uint_as_float(r[j]), sc2, -mx)) * inv : 0.f;
            const float p1 = (!LOCAL || ((vm >> (j + 1)) & 1u)) ? ex2_approx(fmaf(__uint_as_float(r[j + 1]), sc2, -mx)) * inv : 0.f;
            __nv_bfloat162 hh = __floats2bfloat162_rn(p0, p1);
            pk[j >> 1] = *reinterpret_cast<uint32_t*>(&hh);
          }
#pragma unroll
          for (int u = 0; u < 4; ++u) dst[u] = make_uint4(pk[4 * u], pk[4 * u + 1], pk[4 * u + 2], pk[4 * u + 3]);
        }
      } else {
        // D = dO . O over the 32 channels of this head
        const int h = g % a.heads, b = g / a.heads;
        const long orow = ((long)b * N + n) * a.d + h * 32;
        float D = 0.f;
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          const float4 g4 = *reinterpret_cast<const float4*>(a.dO + orow + j);
          const uint2 o2 = *reinterpret_cast<const uint2*>(a.O + orow + j);
          const __nv_bfloat162 oa = *reinterpret_cast<const __nv_bfloat162*>(&o2.x), ob = *reinterpret_cast<const __nv_bfloat162*>(&o2.y);
          D = fmaf(g4.x, __bfloat162float(oa.x), D); D = fmaf(g4.y, __bfloat162float(oa.y), D);
          D = fmaf(g4.z, __bfloat162float(ob.x), D); D = fmaf(g4.w, __bfloat162float(ob.y), D);
        }
#pragma unroll 1
        for (int c0 = cg * CW; c0 < (cg + 1) * CW; c0 += 32) {
          uint32_t r[32];
          tmem_ld32(trow + (uint32_t)c0, r);
          const uint4* src = reinterpret_cast<const uint4*>(a.P + prow + c0);
          uint4* dst = reinterpret_cast<uint4*>(a.dS + prow + c0);
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const uint4 pv = src[u];
            const uint32_t pw[4] = {pv.x, pv.y, pv.z, pv.w};
            uint32_t ov[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const __nv_bfloat162 p2 = *reinterpret_cast<const __nv_bfloat162*>(&pw[e]);
              const int j = u * 8 + e * 2;
              __nv_bfloat162 hh = __floats2bfloat162_rn(__bfloat162float(p2.x) * (__uint_as_float(r[j]) - D),
                                                        __bfloat162float(p2.y) * (__uint_as_float(r[j + 1]) - D));
              ov[e] = *reinterpret_cast<uint32_t*>(&hh);
            }
            dst[u] = make_uint4(ov[0], ov[1], ov[2], ov[3]);
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty_bar);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, N);
}

// rows of one head: (k, row, head, sample) over a [B * rows, ld] bf16 tensor whose heads are 32-wide column slices
int encode_head(CUtensorMap* map, const void* ptr, long rows, long ld, int heads, long batch) {
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) || (ld * 2) % 16) { mrnb_set_error("attn_sp: misaligned operand"); return MRNB_ERR_ARG; }
  cuuint64_t dims[4] = {32, (cuuint64_t)rows, (cuuint64_t)heads, (cuuint64_t)batch};
  cuuint64_t strides[3] = {(cuuint64_t)ld * 2, 64, (cuuint64_t)rows * ld * 2};
  cuuint32_t box[4] = {64, 128, 1, 1}, es[4] = {1, 1, 1, 1};
  return encode_tensor_map("attn_sp", map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, ptr, dims, strides, box, es, CU_TENSOR_MAP_SWIZZLE_128B);
}

template <int N, int MODE>
int launch_sp(const CUtensorMap& tmA, const CUtensorMap& tmB, const SpArgs& a, cudaStream_t st) {
  const size_t smem = 1024 + 2 * (size_t)(BM * BK * 2 + N * BK * 2);
  static bool attr = false;
  if (!attr) { cudaFuncSetAttribute(attn_sp_kernel<N, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); attr = true; }
  static int n_sm = 0;
  if (!n_sm) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev); if (n_sm <= 0) n_sm = 148; }
  int per_sm = 512 / N;                                          // tensor memory: 512 columns per SM
  const int by_smem = (int)((227 * 1024) / (smem + 5 * 1024));
  if (per_sm > by_smem) per_sm = by_smem;
  if (per_sm > 2048 / NTHREADS) per_sm = 2048 / NTHREADS;         // resident threads per SM
  const long cap = (long)n_sm * per_sm;
  const int grid = (int)(a.items < cap ? a.items : cap);
  attn_sp_kernel<N, MODE><<<grid, NTHREADS, smem, st>>>(tmA, tmB, a);
  MRNB_CHECK_LAUNCH("attn_sp_kernel");
  return MRNB_OK;
}

}  // namespace

// qkv [B*N, 3d] bf16 -> P [B*heads, N, N] bf16 = softmax(scale Q K^T + Local mask)
int mrnb_attn_scores_softmax(const void* qkv, void* P, int B, int N, int d, int heads, int W, int local, float scale,
                             cudaStream_t st) {
  MRNB_CHECK_ARG(N == 128 || N == 256 || N == 512, "attn_scores_softmax: N=%d unsupported", N);
  CUtensorMap tmA, tmB;
  MRNB_TRY(encode_head(&tmA, qkv, N, 3L * d, heads, B));
  MRNB_TRY(encode_head(&tmB, (const bf16*)qkv + d, N, 3L * d, heads, B));
  SpArgs a{};
  int ws = 0;
  while ((1 << ws) < W) ++ws;
  MRNB_CHECK_ARG((1 << ws) == W, "attn_scores_softmax: key grid width %d must be a power of two", W);
  a.P = (bf16*)P; a.heads = heads; a.d = d; a.wshift = ws; a.local = local; a.scale = scale;
  a.items = (long)B * heads * (N / BM);
  MrnbProfScope prof(MRNB_PROF_ATTN, st, 2.0 * 2 * 32 * (double)N * N * B * heads / 2, (double)B * heads * N * N * 2);
  if (local) {
    if (N == 512) return launch_sp<512, 2>(tmA, tmB, a, st);
    if (N == 256) return launch_sp<256, 2>(tmA, tmB, a, st);
    return launch_sp<128, 2>(tmA, tmB, a, st);
  }
  if (N == 512) return launch_sp<512, 0>(tmA, tmB, a, st);
  if (N == 256) return launch_sp<256, 0>(tmA, tmB, a, st);
  return launch_sp<128, 0>(tmA, tmB, a, st);
}

// dO16 [B*N, d] bf16, V inside qkv -> dS [B*heads, N, N] bf16 = P * (dO V^T - dO.O)
int mrnb_attn_dp_ds(const void* dO16, const void* qkv, const float* dO, const void* O, const void* P, void* dS, int B, int N,
                    int d, int heads, cudaStream_t st) {
  MRNB_CHECK_ARG(N == 128 || N == 256 || N == 512, "attn_dp_ds: N=%d unsupported", N);
  CUtensorMap tmA, tmB;
  MRNB_TRY(encode_head(&tmA, dO16, N, d, heads, B));
  MRNB_TRY(encode_head(&tmB, (const bf16*)qkv + 2 * d, N, 3L * d, heads, B));
  SpArgs a{};
  a.P = (bf16*)const_cast<void*>(P); a.dS = (bf16*)dS; a.dO = dO; a.O = (const bf16*)O; a.heads = heads; a.d = d; a.scale = 1.f;
  a.items = (long)B * heads * (N / BM);
  MrnbProfScope prof(MRNB_PROF_ATTN, st, 2.0 * 32 * (double)N * N * B * heads, (double)B * heads * N * N * 4);
  if (N == 512) return launch_sp<512, 1>(tmA, tmB, a, st);
  if (N == 256) return launch_sp<256, 1>(tmA, tmB, a, st);
  return launch_sp<128, 1>(tmA, tmB, a, st);
}
