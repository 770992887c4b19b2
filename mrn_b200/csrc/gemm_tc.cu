// Grouped bf16 GEMM on the 5th-generation tensor cores: TMA-fed shared-memory tiles (128B swizzle), tcgen05.mma
// issued by one elected thread, fp32 accumulator in TMEM, epilogue warps read it back with tcgen05.ld and fuse
// bias / exact GELU / DropPath row scale / fp32 residual before the store.
//
//   out[g, m, n] = epi( sum_k A[g, m, k] * W[g, n, k] + bias[g, n] )      g = expert (blockIdx.z)
//
// This is the tensor-core mode of every nn.Linear / conv-as-GEMM on the expert path (reference call sites:
// modules/svtr.py:56-58,106-108,277; modules/model.py:75-78,164,181), one launch for all experts.
//
// Warp roles (192 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer, warps 2..5 = epilogue
// (TMEM lane quarter = warp_id % 4).  Pipelines: smem full/empty mbarriers (TMA <-> MMA) and one TMEM-full
// mbarrier (MMA -> epilogue).  sm_100a only.
#include "gemm_tc.h"
#include "sm100.cuh"

namespace {

constexpr int BM = 128, BK = 64, UMMA_K = 16;
constexpr int MAX_STAGES = 2;          // 2 x 32 KiB ring + 32 KiB staging: two persistent CTAs per SM
constexpr int A_STAGE_BYTES = BM * BK * 2;   // 16 KiB

// Output tensor maps of the TMA-store epilogue (MODE 3: one fp32 [M, C_e] map per expert, box 32 x 32, 128B swizzle)
struct TcOutMaps { CUtensorMap m[8]; };

struct TcEpi {
  const float* bias; long bias_gs;
  void* out; long ldo; long o_gs;
  const float* res;
  const float* rowscale; int rows_per_scale; long rowscale_gs;
  int M, N, KB, stages, gelu;
  int n_tiles, m_tiles, total_tiles;
  // fused LayerNorm of the output rows (LNF kernels): bf16 ln_out[g][row][N], gamma/beta [groups][N]
  __nv_bfloat16* ln_out; long ln_gs; const float* ln_gamma; const float* ln_beta; float ln_eps;
  // implicit-GEMM convolution (see MrnbTcConv)
  int conv, rows_per_img, per_kh, cch, w_off, sh, imgs_per_group, ow_shift, pad_h;
  int relu;
  MrnbTcLstm lstm;
  MrnbTcHeads heads;       // MODE 3: ragged classifier heads of all experts in one launch (+ hard-route tile skip)
  int tma_out;             // MODE 3: output tiles leave through TMA stores (every head 16-byte aligned with ldo % 4 == 0)
};

// MODE 3 tile decode: flat tile t -> (expert e, m0, n0); returns false when the hard route sends none of the tile's samples
// to expert e (the tile is skipped by all three warp roles alike).
__device__ __forceinline__ bool heads_tile(const MrnbTcHeads& H, int t, int& e, int& m0, int& n0) {
  e = 0;
#pragma unroll
  for (int k = 1; k < 8; ++k) if (k < H.n_experts && t >= H.tile_prefix[k]) e = k;
  const int tl = t - H.tile_prefix[e], nt = H.n_tiles[e];
  m0 = (tl / nt) * 128; n0 = (tl % nt) * 128;
  if (H.route) {
    const int s0 = m0 / H.rows_per_sample, s1 = (m0 + 127) / H.rows_per_sample;
    bool any = false;
    for (int sidx = s0; sidx <= s1 && sidx < H.n_samples; ++sidx) any = any || (H.route[sidx] == e);
    return any;
  }
  return true;
}

constexpr int EPI_WARPS = 8;                       // two warps per TMEM lane quarter, each owning half of the tile columns
constexpr int NTHREADS = 64 + EPI_WARPS * 32;      // warp 0 TMA, warp 1 MMA + TMEM, warps 2..9 epilogue
constexpr int STAGING_BYTES = EPI_WARPS * 32 * 32 * 4;    // 32x32 fp32 tile per epilogue warp, XOR-swizzled

// Persistent kernel: CTA c walks tiles c, c + gridDim.x, ... (n fastest so neighbouring CTAs share the A tile in L2).
// The smem ring runs across tile boundaries, and the accumulator is double buffered in TMEM so the MMAs of tile i+1
// overlap the epilogue of tile i.
__device__ __forceinline__ float sigmoid_fast(float x) { return __fdividef(1.0f, 1.0f + __expf(-x)); }
__device__ __forceinline__ float tanh_fast(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

template <int BN, bool OUT_F32, bool GELU, bool LNF, int MODE = 0>
__global__ void __launch_bounds__(NTHREADS, LNF ? 1 : 2)
tc_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW, const TcEpi ep,
               const __grid_constant__ TcOutMaps tmO) {
  extern __shared__ uint8_t smem_raw[];
  constexpr int B_STAGE_BYTES = BN * BK * 2;
  constexpr int STAGE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;
  constexpr int TMEM_COLS = 2 * BN;
  uint8_t* smem = smem_raw + align_smem_1024_offset(smem_raw);
  __shared__ __align__(8) uint64_t full_bar[MAX_STAGES];
  __shared__ __align__(8) uint64_t empty_bar[MAX_STAGES];
  __shared__ __align__(8) uint64_t tmem_full_bar[2];
  __shared__ __align__(8) uint64_t tmem_empty_bar[2];
  __shared__ uint32_t tmem_base_sh;
  __shared__ float ln_part[2][4][2][32];        // [pass][row quarter][column half][row]: LayerNorm partial sums

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int stages = ep.stages, KB = ep.KB;
  const int n_tiles = ep.n_tiles, m_tiles = ep.m_tiles;
  const int total = ep.total_tiles;
  const bool relu = ep.relu != 0;
  float* staging = reinterpret_cast<float*>(smem + (size_t)stages * STAGE_BYTES);

  if (threadIdx.x == 0) {
    for (int s = 0; s < stages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(&tmem_full_bar[b], 1); mbar_init(&tmem_empty_bar[b], EPI_WARPS); }
    fence_mbarrier_init();
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmW);
  }
  if (warp == 1) tmem_alloc(&tmem_base_sh, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_sh;

  if (warp == 0) {
    if (lane == 0) {
      uint32_t it = 0;
      for (int t = blockIdx.x; t < total; t += gridDim.x) {
        int n0 = (t % n_tiles) * BN, m0 = ((t / n_tiles) % m_tiles) * BM, g = t / (n_tiles * m_tiles);
        int wrow = n0, wg = g;
        if constexpr (MODE == 3) {
          if (!heads_tile(ep.heads, t, g, m0, n0)) continue;
          wrow = ep.heads.woff[g] + n0; wg = 0;                 // the heads' weights are one stacked [sum C_i, K] matrix
        }
        for (int kb = 0; kb < KB; ++kb, ++it) {
          const int s = it % stages;
          const uint32_t ph = (it / stages) & 1u;
          mbar_wait(&empty_bar[s], ph ^ 1u);
          mbar_expect_tx(&full_bar[s], STAGE_BYTES);
          uint8_t* sa = smem + (size_t)s * STAGE_BYTES;
          if (ep.conv) {
            const int img = g * ep.imgs_per_group + m0 / ep.rows_per_img;
            const int oh0 = (m0 % ep.rows_per_img) >> ep.ow_shift;     // 64 or 128 output columns per output row
            const int kh = kb / ep.per_kh, j = kb % ep.per_kh;
            tma_load_4d(sa, &tmA, &full_bar[s], (j % ep.cch) * 64, j / ep.cch + ep.w_off, oh0 * ep.sh - ep.pad_h + kh, img);
          } else {
            tma_load_3d(sa, &tmA, &full_bar[s], kb * BK, m0, g);
          }
          tma_load_3d(sa + A_STAGE_BYTES, &tmW, &full_bar[s], kb * BK, wrow, wg);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = umma_idesc(UMMA_BF16, BM, BN);
      uint32_t it = 0;
      int i = 0;
      for (int t = blockIdx.x; t < total; t += gridDim.x, ++i) {
        if constexpr (MODE == 3) {
          int e_, m_, n_;
          if (!heads_tile(ep.heads, t, e_, m_, n_)) { --i; continue; }         // skipped tiles do not consume an accumulator
        }
        const int buf = i & 1;
        mbar_wait(&tmem_empty_bar[buf], (((uint32_t)i >> 1) & 1u) ^ 1u);      // epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t acc = tmem_base + (uint32_t)(buf * BN);
        for (int kb = 0; kb < KB; ++kb, ++it) {
          const int s = it % stages;
          const uint32_t ph = (it / stages) & 1u;
          mbar_wait(&full_bar[s], ph);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + (size_t)s * STAGE_BYTES);
          const uint64_t adesc = umma_desc_k128(sa), bdesc = umma_desc_k128(sa + A_STAGE_BYTES);
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) {
            // advance 16 bf16 = 32 B along K inside the 128 B swizzle row: +2 in the (>>4) address field
            umma_bf16(acc, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc, (kb | k) != 0 ? 1u : 0u);
          }
          umma_commit(&empty_bar[s]);          // frees the smem slot once these MMAs have read it
        }
        umma_commit(&tmem_full_bar[buf]);      // accumulator complete
      }
    }
  } else {
    // ---- epilogue warps: quarter q = warp % 4 (TMEM lanes 32q..32q+31), column half ch = (warp - 2) / 4.
    // The warp's CW columns are processed in passes of 32:
    //   phase A: one accumulator row per thread (tcgen05.ld) parked in a 32x32 fp32 staging tile (4 KiB per warp,
    //            16-byte pieces XOR-swizzled by row: conflict-free without padding);
    //   phase B: lanes own columns (8 lanes x float4 per row, 4 rows per step), so bias sits in registers and the
    //            residual loads / output stores are coalesced 128-byte segments.
    // Residual rows are prefetched before they are needed (pass 0: before the accumulator wait).
    const int ew = warp - 2;
    const int q = warp & 3, ch = ew >> 2;
    constexpr int CW = BN / 2;                                 // columns per epilogue warp: 64 (BN=128) or 32 (BN=64)
    constexpr int NP = CW / 32;                                // passes
    float* stg = staging + (size_t)ew * 1024;
    const int p8 = lane & 7, rsel = lane >> 3;
    int i = 0;
    for (int t = blockIdx.x; t < total; t += gridDim.x, ++i) {
      int n0 = (t % n_tiles) * BN, m0 = ((t / n_tiles) % m_tiles) * BM, g = t / (n_tiles * m_tiles);
      // output of this tile: the launch-wide description, or (MODE 3) the head of expert g
      void* t_out = ep.out; long t_ldo = ep.ldo; int t_N = ep.N; long gbase = (long)g * ep.o_gs;
      const float* bias = ep.bias ? ep.bias + (long)g * ep.bias_gs : nullptr;
      if constexpr (MODE == 3) {
        if (!heads_tile(ep.heads, t, g, m0, n0)) { --i; continue; }
        t_out = ep.heads.out[g]; t_ldo = ep.heads.ldo[g]; t_N = ep.heads.N[g]; gbase = 0; bias = ep.heads.bias[g];
      }
      const int buf = i & 1;
      const int colw = n0 + ch * CW + p8 * 4;                  // this lane's first column in pass 0
      // interior tile with aligned rows: branch-free path (pointer increments, tile-uniform DropPath scale)
      const bool interior = (m0 + BM <= ep.M) && (n0 + BN <= t_N) && ((t_ldo & 3) == 0) && ((gbase & 3) == 0) &&
                            (!ep.rowscale || (ep.rows_per_scale % BM) == 0);
      const long o0 = gbase + (long)(m0 + q * 32 + rsel) * t_ldo + colw;
      const long ostep = 4L * t_ldo;
      const bool pre_res = MODE != 3 && OUT_F32 && interior && ep.res != nullptr;
      float4 rv[8];
      if (pre_res) {
#pragma unroll
        for (int itr = 0; itr < 8; ++itr) rv[itr] = *reinterpret_cast<const float4*>(ep.res + o0 + itr * ostep);
        if (NP > 1 && p8 == 0) {                               // later passes: start their trip to L2 now (one lane per 128 B)
#pragma unroll
          for (int ps = 1; ps < NP; ++ps)
#pragma unroll
            for (int itr = 0; itr < 8; ++itr) asm volatile("prefetch.global.L2 [%0];" ::"l"(ep.res + o0 + ps * 32 + itr * ostep));
        }
      }
      const float rs = (MODE != 3 && interior && ep.rowscale) ? ep.rowscale[(long)g * ep.rowscale_gs + m0 / ep.rows_per_scale] : 1.0f;
      mbar_wait(&tmem_full_bar[buf], ((uint32_t)i >> 1) & 1u);
      tc_fence_after();
      const uint32_t tcol = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * BN + ch * CW);
      float4 keep[LNF ? NP * 8 : 1];
#pragma unroll
      for (int ps = 0; ps < NP; ++ps) {
        if (pre_res && ps > 0) {                               // this pass' residual rows: in flight during the TMEM load / staging
#pragma unroll
          for (int itr = 0; itr < 8; ++itr) rv[itr] = *reinterpret_cast<const float4*>(ep.res + o0 + ps * 32 + itr * ostep);
        }
        {
          uint32_t r[32];
          tmem_ld32(tcol + (uint32_t)(ps * 32), r);
          if (ps == NP - 1) {
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tmem_empty_bar[buf]);  // this warp's share of the accumulator is out of TMEM
          }
          if constexpr (MODE == 3) {
            if (ep.tma_out) {
              // TMA-store epilogue: + bias in the accumulator layout (thread = row: the 32 bias values of the pass are
              // broadcast loads), the 32 x 32 fp32 tile is parked in the staging tile in the 128B-swizzled box layout
              // (the same conflict-free XOR as below) and leaves with ONE bulk tensor store per warp and pass -- whole
              // 128-byte lines, rows / columns beyond M / C_e clipped by the hardware, no per-thread address arithmetic
              const int c0 = n0 + ch * CW + ps * 32;
              if (c0 < t_N) {
                if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // the previous store has read the tile
                __syncwarp();
#pragma unroll
                for (int pc = 0; pc < 8; ++pc) {
                  float4 b4;
                  if (c0 + 4 * pc + 4 <= t_N) b4 = __ldg(reinterpret_cast<const float4*>(bias + c0 + 4 * pc));
                  else {
                    b4.x = c0 + 4 * pc < t_N ? bias[c0 + 4 * pc] : 0.f; b4.y = c0 + 4 * pc + 1 < t_N ? bias[c0 + 4 * pc + 1] : 0.f;
                    b4.z = c0 + 4 * pc + 2 < t_N ? bias[c0 + 4 * pc + 2] : 0.f; b4.w = 0.f;
                  }
                  *reinterpret_cast<float4*>(stg + lane * 32 + ((pc ^ (lane & 7)) * 4)) =
                      make_float4(__uint_as_float(r[4 * pc]) + b4.x, __uint_as_float(r[4 * pc + 1]) + b4.y,
                                  __uint_as_float(r[4 * pc + 2]) + b4.z, __uint_as_float(r[4 * pc + 3]) + b4.w);
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                __syncwarp();
                if (lane == 0) tma_store_2d(&tmO.m[g], stg, c0, m0 + q * 32);
              }
              continue;
            }
          }
#pragma unroll
          for (int pc = 0; pc < 8; ++pc)
            *reinterpret_cast<float4*>(stg + lane * 32 + ((pc ^ (lane & 7)) * 4)) =
                make_float4(__uint_as_float(r[4 * pc]), __uint_as_float(r[4 * pc + 1]), __uint_as_float(r[4 * pc + 2]), __uint_as_float(r[4 * pc + 3]));
        }
        __syncwarp();
        const int col = colw + ps * 32;
        const bool cfull = col + 4 <= t_N;
        float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (bias && col < t_N) {
          if (cfull) b4 = *reinterpret_cast<const float4*>(bias + col);
          else {
            b4.x = bias[col];
            if (col + 1 < t_N) b4.y = bias[col + 1];
            if (col + 2 < t_N) b4.z = bias[col + 2];
          }
        }
        if constexpr (MODE == 3) {
          // classifier heads: bias + store only (no residual / scale / activation); the ragged last column tile of an
          // expert (C_e % 128 != 0) keeps the vector path for its full float4s -- row pitches are multiples of 4 floats
          if ((m0 + BM <= ep.M) && ((t_ldo & 3) == 0)) {
            float* op = reinterpret_cast<float*>(t_out) + o0 + ps * 32;
            if (cfull) {
#pragma unroll
              for (int itr = 0; itr < 8; ++itr) {
                const int rl = itr * 4 + rsel;
                float4 x = *reinterpret_cast<const float4*>(stg + rl * 32 + ((p8 ^ (rl & 7)) * 4));
                x.x += b4.x; x.y += b4.y; x.z += b4.z; x.w += b4.w;
                *reinterpret_cast<float4*>(op + itr * ostep) = x;
              }
            } else if (col < t_N) {
#pragma unroll
              for (int itr = 0; itr < 8; ++itr) {
                const int rl = itr * 4 + rsel;
                const float4 x = *reinterpret_cast<const float4*>(stg + rl * 32 + ((p8 ^ (rl & 7)) * 4));
                float* o = op + itr * ostep;
                o[0] = x.x + b4.x;
                if (col + 1 < t_N) o[1] = x.y + b4.y;
                if (col + 2 < t_N) o[2] = x.z + b4.z;
              }
            }
            __syncwarp();
            continue;
          }
        }
        if (MODE != 3 && interior) {
          if constexpr (MODE == 1) {
            // fused LSTM cell: x = (i, f, g, o) pre-activations of hidden unit j for sample b
            const MrnbTcLstm& L = ep.lstm;
            const int e = g >> 1, dir = g & 1;
            const int col = colw + ps * 32;                    // interleaved gate column, multiple of 4
            const int j = col >> 2;
            const __nv_bfloat16* prep = reinterpret_cast<const __nv_bfloat16*>(L.pre) + (long)e * L.pre_e + L.pre_off[dir] + col;
            __nv_bfloat16* recp = reinterpret_cast<__nv_bfloat16*>(L.rec) + (long)e * L.rec_e + L.rec_off[dir] + j;
#pragma unroll
            for (int itr = 0; itr < 8; ++itr) {
              const int rl = itr * 4 + rsel;
              const int b = m0 + q * 32 + rl;
              float4 x = *reinterpret_cast<const float4*>(stg + rl * 32 + ((p8 ^ (rl & 7)) * 4));
              const uint2 pv = *reinterpret_cast<const uint2*>(prep + (long)b * L.pre_row);
              const __nv_bfloat162 p01 = *reinterpret_cast<const __nv_bfloat162*>(&pv.x), p23 = *reinterpret_cast<const __nv_bfloat162*>(&pv.y);
              x.x += __low2float(p01); x.y += __high2float(p01); x.z += __low2float(p23); x.w += __high2float(p23);
              const long ci = ((long)g * L.B + b) * 256 + j;
              const float c = fmaf(sigmoid_fast(x.y), L.cst[ci], sigmoid_fast(x.x) * tanh_fast(x.z));
              const float h = sigmoid_fast(x.w) * tanh_fast(c);
              L.cst[ci] = c;
              const __nv_bfloat16 hb = __float2bfloat16_rn(h);
              reinterpret_cast<__nv_bfloat16*>(L.hst)[ci] = hb;
              recp[(long)b * L.rec_row] = hb;
            }
          } else if constexpr (MODE == 2) {
            // bias + ReLU + max over each group of 4 consecutive rows (a 2x2 pooling window: the im2col rows are
            // window-major), bf16 output [M/4, N].  Rows 4*itr .. 4*itr+3 sit in the lanes rsel = 0..3 of one step.
            __nv_bfloat16* op = reinterpret_cast<__nv_bfloat16*>(ep.out) + gbase + (long)((m0 + q * 32) >> 2) * ep.ldo + colw + ps * 32;
#pragma unroll
            for (int itr = 0; itr < 8; ++itr) {
              const int rl = itr * 4 + rsel;
              float4 x = *reinterpret_cast<const float4*>(stg + rl * 32 + ((p8 ^ (rl & 7)) * 4));
#pragma unroll
              for (int o = 8; o <= 16; o <<= 1) {
                x.x = fmaxf(x.x, __shfl_xor_sync(0xffffffffu, x.x, o)); x.y = fmaxf(x.y, __shfl_xor_sync(0xffffffffu, x.y, o));
                x.z = fmaxf(x.z, __shfl_xor_sync(0xffffffffu, x.z, o)); x.w = fmaxf(x.w, __shfl_xor_sync(0xffffffffu, x.w, o));
              }
              if (rsel == 0) {
                __nv_bfloat162 h0 = __floats2bfloat162_rn(fmaxf(x.x + b4.x, 0.f), fmaxf(x.y + b4.y, 0.f));
                __nv_bfloat162 h1 = __floats2bfloat162_rn(fmaxf(x.z + b4.z, 0.f), fmaxf(x.w + b4.w, 0.f));
                *reinterpret_cast<uint2*>(op + (long)itr * ep.ldo) = make_uint2(*reinterpret_cast<uint32_t*>(&h0), *reinterpret_cast<uint32_t*>(&h1));
              }
            }
          } else if (OUT_F32) {
            float* op = reinterpret_cast<float*>(t_out) + o0 + ps * 32;
#pragma unroll
            for (int itr = 0; itr < 8; ++itr) {
              const int rl = itr * 4 + rsel;
              float4 x = *reinterpret_cast<const float4*>(stg + rl * 32 + ((p8 ^ (rl & 7)) * 4));
              x.x += b4.x; x.y += b4.y; x.z += b4.z; x.w += b4.w;
              if (GELU) { x.x = gelu_erf(x.x); x.y = gelu_erf(x.y); x.z = gelu_erf(x.z); x.w = gelu_erf(x.w); }
              if (relu) { x.x = fmaxf(x.x, 0.f); x.y = fmaxf(x.y, 0.f); x.z = fmaxf(x.z, 0.f); x.w = fmaxf(x.w, 0.f); }
              x.x *= rs; x.y *= rs; x.z *= rs; x.w *= rs;
              if (pre_res) { x.x += rv[itr].x; x.y += rv[itr].y; x.z += rv[itr].z; x.w += rv[itr].w; }
              *reinterpret_cast<float4*>(op + itr * ostep) = x;
              if (LNF) keep[ps * 8 + itr] = x;
            }
          } else {
            __nv_bfloat16* op = reinterpret_cast<__nv_bfloat16*>(t_out) + o0 + ps * 32;
#pragma unroll
            for (int itr = 0; itr < 8; ++itr) {
              const int rl = itr * 4 + rsel;
              float4 x = *reinterpret_cast<const float4*>(stg + rl * 32 + ((p8 ^ (rl & 7)) * 4));
              x.x += b4.x; x.y += b4.y; x.z += b4.z; x.w += b4.w;
              if (GELU) { x.x = gelu_fast(x.x); x.y = gelu_fast(x.y); x.z = gelu_fast(x.z); x.w = gelu_fast(x.w); }
              if (relu) { x.x = fmaxf(x.x, 0.f); x.y = fmaxf(x.y, 0.f); x.z = fmaxf(x.z, 0.f); x.w = fmaxf(x.w, 0.f); }
              x.x *= rs; x.y *= rs; x.z *= rs; x.w *= rs;
              __nv_bfloat162 h0 = __floats2bfloat162_rn(x.x, x.y), h1 = __floats2bfloat162_rn(x.z, x.w);
              *reinterpret_cast<uint2*>(op + itr * ostep) = make_uint2(*reinterpret_cast<uint32_t*>(&h0), *reinterpret_cast<uint32_t*>(&h1));
            }
          }
        } else {
          // edge tiles / unaligned outputs: guarded scalar path
          for (int itr = 0; itr < 8; ++itr) {
            const int rl = itr * 4 + rsel;
            const int row = m0 + q * 32 + rl;
            if (row >= ep.M || col >= t_N) continue;
            const float4 xs = *reinterpret_cast<const float4*>(stg + rl * 32 + ((p8 ^ (rl & 7)) * 4));
            float xv[4] = {xs.x + b4.x, xs.y + b4.y, xs.z + b4.z, xs.w + b4.w};
            const float rsr = ep.rowscale ? ep.rowscale[(long)g * ep.rowscale_gs + row / ep.rows_per_scale] : 1.0f;
            const long o = gbase + (long)row * t_ldo + col;
            for (int j = 0; j < 4 && col + j < t_N; ++j) {
              float x = xv[j];
              if (GELU) x = OUT_F32 ? gelu_erf(x) : gelu_fast(x);
              if (relu) x = fmaxf(x, 0.f);
              x *= rsr;
              if (OUT_F32) {
                if (ep.res) x += ep.res[o + j];
                reinterpret_cast<float*>(t_out)[o + j] = x;
              } else {
                reinterpret_cast<__nv_bfloat16*>(t_out)[o + j] = __float2bfloat16_rn(x);
              }
            }
          }
        }
        __syncwarp();                                          // staging tile is reused by the next pass / tile
      }
      if (LNF) {
        // Fused LayerNorm of the freshly written rows (the tile spans the whole row: N == BN).  Two-pass statistics;
        // the two warps that share a row (column halves) exchange partial sums through shared memory.
        const float invn = 1.0f / (float)BN;
        float mean[8], rstd[8];
#pragma unroll
        for (int itr = 0; itr < 8; ++itr) {
          float sres = 0.f;
#pragma unroll
          for (int ps = 0; ps < NP; ++ps) { const float4 x = keep[ps * 8 + itr]; sres += (x.x + x.y) + (x.z + x.w); }
#pragma unroll
          for (int o = 4; o > 0; o >>= 1) sres += __shfl_xor_sync(0xffffffffu, sres, o);
          if (p8 == 0) ln_part[0][q][ch][itr * 4 + rsel] = sres;
        }
        asm volatile("bar.sync %0, 64;" ::"r"(1 + q) : "memory");
#pragma unroll
        for (int itr = 0; itr < 8; ++itr) {
          const int rl = itr * 4 + rsel;
          mean[itr] = (ln_part[0][q][0][rl] + ln_part[0][q][1][rl]) * invn;
          float sq = 0.f;
#pragma unroll
          for (int ps = 0; ps < NP; ++ps) {
            const float4 x = keep[ps * 8 + itr];
            const float d0 = x.x - mean[itr], d1 = x.y - mean[itr], d2 = x.z - mean[itr], d3 = x.w - mean[itr];
            sq += fmaf(d0, d0, d1 * d1) + fmaf(d2, d2, d3 * d3);
          }
#pragma unroll
          for (int o = 4; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
          if (p8 == 0) ln_part[1][q][ch][rl] = sq;
        }
        asm volatile("bar.sync %0, 64;" ::"r"(1 + q) : "memory");
        __nv_bfloat16* lrow = ep.ln_out + (long)g * ep.ln_gs + (long)(m0 + q * 32 + rsel) * BN + ch * CW + p8 * 4;
#pragma unroll
        for (int itr = 0; itr < 8; ++itr) {
          const int rl = itr * 4 + rsel;
          rstd[itr] = rsqrtf((ln_part[1][q][0][rl] + ln_part[1][q][1][rl]) * invn + ep.ln_eps);
#pragma unroll
          for (int ps = 0; ps < NP; ++ps) {
            const int cc = ch * CW + ps * 32 + p8 * 4;
            const float4 g4 = *reinterpret_cast<const float4*>(ep.ln_gamma + (long)g * BN + cc);
            const float4 t4 = *reinterpret_cast<const float4*>(ep.ln_beta + (long)g * BN + cc);
            const float4 x = keep[ps * 8 + itr];
            __nv_bfloat162 h0 = __floats2bfloat162_rn((x.x - mean[itr]) * rstd[itr] * g4.x + t4.x, (x.y - mean[itr]) * rstd[itr] * g4.y + t4.y);
            __nv_bfloat162 h1 = __floats2bfloat162_rn((x.z - mean[itr]) * rstd[itr] * g4.z + t4.z, (x.w - mean[itr]) * rstd[itr] * g4.w + t4.w);
            *reinterpret_cast<uint2*>(lrow + ps * 32 + (long)itr * 4 * BN) = make_uint2(*reinterpret_cast<uint32_t*>(&h0), *reinterpret_cast<uint32_t*>(&h1));
          }
        }
      }
    }
  }
  if (MODE == 3 && warp >= 2 && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // bulk stores of this thread are complete
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, TMEM_COLS);
}

// ---- host side ---------------------------------------------------------------------------------
// ---------------------------------------------------------------------------------------------------------------------
// Persistent LSTM recurrence (modules/sequence_modeling.py:12-22, the nn.LSTM inside BidirectionalLSTM): every time step
// s_first .. CT-1 of all (expert, direction) chains of one layer in ONE launch, instead of one grouped GEMM launch per
// step (63 x ~20 us per layer, each bounded by launch + TMA + MMA + epilogue latency, not by work).
//
// A thread-block CLUSTER of four CTAs owns one (chain g, 128-sample tile): CTA nq of the cluster keeps the 256 gate
// columns (64 hidden units x i,f,g,o) nq of W_hh -- [256 x 256] bf16 = 128 KiB -- resident in shared memory for the whole
// sequence.  Per step: the eight epilogue warps copy h_{s-1} of the tile (128 x 256 bf16, written by all four CTAs in the
// previous step, read with ld.global.cg from L2) into a 128B-swizzled K-major operand tile; one thread issues the
// 16 tcgen05 MMAs (M128 N256 K256, accumulator in 256 TMEM columns); the epilogue applies the cell exactly as the per-step
// kernel (MODE 1) does and writes c (fp32), h_s (bf16, ping-pong buffer) and the [fwd | bwd] output row; a hardware
// cluster barrier (release / acquire) publishes h_s to the other three CTAs.  Nothing else crosses CTAs.
struct LstmSeqArgs {
  const __nv_bfloat16* pre; long pre_row, pre_e;   // [expert][sample * CTP + t][2 * 4H]
  __nv_bfloat16* rec; long rec_row, rec_e;         // [expert][sample * CTP + t][2H]
  float* cst;                                      // [chain][B][H]
  __nv_bfloat16* h0; __nv_bfloat16* h1;            // hidden state ping-pong [chain][B][H]: step s reads buffer (s-1) & 1, writes s & 1
  int B, CT, s_first;
};
constexpr int LSEQ_THREADS = 256;                  // eight warps: operand copy + cell; thread 0 also loads W_hh and issues the MMAs
                                                   // (ten warps would put three on one SM sub-partition: 168 registers per thread)
constexpr int LSEQ_W_BYTES = 4 * 256 * BK * 2, LSEQ_A_BYTES = 4 * BM * BK * 2;
constexpr int LSEQ_SMEM = 1024 + LSEQ_W_BYTES + LSEQ_A_BYTES + EPI_WARPS * 4096;

__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint4 ld_cg_v4(const void* p) {
  uint4 v;
  asm volatile("ld.global.cg.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
  return v;
}

__global__ void __cluster_dims__(4, 1, 1) __launch_bounds__(LSEQ_THREADS, 1)
lstm_seq_kernel(const __grid_constant__ CUtensorMap tmW, const LstmSeqArgs p) {
  constexpr int LH = 256;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + align_smem_1024_offset(smem_raw);
  uint8_t* sW = smem;                                        // 4 k-blocks x [256 gate rows x 64 k]
  uint8_t* sA = smem + LSEQ_W_BYTES;                         // 4 k-blocks x [128 samples x 64 k]
  float* staging = reinterpret_cast<float*>(smem + LSEQ_W_BYTES + LSEQ_A_BYTES);
  __shared__ __align__(8) uint64_t w_full, acc_full;
  __shared__ uint32_t tmem_base_sh;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nq = blockIdx.x & 3;                             // rank in the cluster == quarter of the gate columns
  const int tile = blockIdx.x >> 2, m_tiles = p.B / BM;
  const int m0 = (tile % m_tiles) * BM, g = tile / m_tiles;
  const int e = g >> 1, dir = g & 1;
  if (threadIdx.x == 0) {
    mbar_init(&w_full, 1); mbar_init(&acc_full, 1);
    fence_mbarrier_init();
    prefetch_tmap(&tmW);
  }
  if (warp == 0) tmem_alloc(&tmem_base_sh, 256);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_sh;
  if (threadIdx.x == 0) {
    mbar_expect_tx(&w_full, LSEQ_W_BYTES);
    for (int kb = 0; kb < 4; ++kb) tma_load_3d(sW + kb * (256 * BK * 2), &tmW, &w_full, kb * BK, nq * 256, g);
  }
  uint32_t it = 0;
  for (int s = p.s_first; s < p.CT; ++s, ++it) {
    const __nv_bfloat16* hin = ((s - 1) & 1) ? p.h1 : p.h0;
    __nv_bfloat16* hout = (s & 1) ? p.h1 : p.h0;
    {
      // h_{s-1} of the tile: 128 rows x 512 B, contiguous -> 16-byte chunk c = row * 32 + kc
      const char* src = reinterpret_cast<const char*>(hin + ((long)g * p.B + m0) * LH);
      constexpr int NCH = BM * 32 / (EPI_WARPS * 32);          // 16 chunks per thread: all loads in flight before the first store
      uint4 v[NCH];
#pragma unroll
      for (int u = 0; u < NCH; ++u) v[u] = ld_cg_v4(src + (size_t)(threadIdx.x + u * EPI_WARPS * 32) * 16);
#pragma unroll
      for (int u = 0; u < NCH; ++u) {
        const int c = threadIdx.x + u * EPI_WARPS * 32;
        const int row = c >> 5, kc = c & 31, kb = kc >> 3, cc = kc & 7;
        *reinterpret_cast<uint4*>(sA + kb * A_STAGE_BYTES + row * 128 + ((cc ^ (row & 7)) << 4)) = v[u];
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      if (it == 0) mbar_wait(&w_full, 0);
      tc_fence_after();
      constexpr uint32_t idesc = umma_idesc(UMMA_BF16, BM, 256);
      for (int kb = 0; kb < 4; ++kb) {
        const uint64_t ad = umma_desc_k128(smem_u32(sA + kb * A_STAGE_BYTES)), bd = umma_desc_k128(smem_u32(sW + kb * (256 * BK * 2)));
#pragma unroll
        for (int k = 0; k < BK / UMMA_K; ++k) umma_bf16(tmem_base, ad + (uint64_t)(k * 2), bd + (uint64_t)(k * 2), idesc, (kb | k) != 0 ? 1u : 0u);
      }
      umma_commit(&acc_full);
    }
    __syncwarp();
    {
      const int ew = warp, q = warp & 3, ch = ew >> 2;
      float* stg = staging + (size_t)ew * 1024;
      const int p8 = lane & 7, rsel = lane >> 3;
      const int t = dir ? p.CT - 1 - s : s;                    // frame of this step for the chain's direction
      const uint32_t tcol = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(ch * 128);
      // input pre-activations and cell states of a pass' eight rows are loaded one pass ahead (pass 0: before the
      // accumulator wait, i.e. during the MMAs), so that no pass waits for a global load
      const __nv_bfloat16* prep0 = p.pre + (long)e * p.pre_e + (long)t * (8 * LH) + dir * 4 * LH + nq * 256 + ch * 128 + p8 * 4;
      const long crow0 = ((long)g * p.B + m0 + q * 32 + rsel) * LH + ((nq * 256 + ch * 128 + p8 * 4) >> 2);
      uint2 pvv[8], pvn[8];
      float cprev[8];
#pragma unroll
      for (int itr = 0; itr < 8; ++itr) {
        pvv[itr] = *reinterpret_cast<const uint2*>(prep0 + (long)(m0 + q * 32 + itr * 4 + rsel) * p.pre_row);
      }
      mbar_wait(&acc_full, it & 1u);
      tc_fence_after();
#pragma unroll 1
      for (int ps = 0; ps < 4; ++ps) {
        const int col = nq * 256 + ch * 128 + ps * 32 + p8 * 4;  // interleaved gate column of the chain: unit j = col / 4
        const int j = col >> 2;
        if (ps + 1 < 4) {
#pragma unroll
          for (int itr = 0; itr < 8; ++itr) {
            pvn[itr] = *reinterpret_cast<const uint2*>(prep0 + (ps + 1) * 32 + (long)(m0 + q * 32 + itr * 4 + rsel) * p.pre_row);
          }
        }
#pragma unroll
        for (int itr = 0; itr < 8; ++itr) cprev[itr] = p.cst[crow0 + ps * 8 + (long)itr * 4 * LH];
        {
          uint32_t r[32];
          tmem_ld32(tcol + (uint32_t)(ps * 32), r);
#pragma unroll
          for (int pc = 0; pc < 8; ++pc)
            *reinterpret_cast<float4*>(stg + lane * 32 + ((pc ^ (lane & 7)) * 4)) =
                make_float4(__uint_as_float(r[4 * pc]), __uint_as_float(r[4 * pc + 1]), __uint_as_float(r[4 * pc + 2]), __uint_as_float(r[4 * pc + 3]));
        }
        __syncwarp();
        __nv_bfloat16* recp = p.rec + (long)e * p.rec_e + (long)t * (2 * LH) + dir * LH + j;
#pragma unroll
        for (int itr = 0; itr < 8; ++itr) {
          const int rl = itr * 4 + rsel;
          const int b = m0 + q * 32 + rl;
          float4 x = *reinterpret_cast<const float4*>(stg + rl * 32 + ((p8 ^ (rl & 7)) * 4));
          const uint2 pv = pvv[itr];
          const __nv_bfloat162 p01 = *reinterpret_cast<const __nv_bfloat162*>(&pv.x), p23 = *reinterpret_cast<const __nv_bfloat162*>(&pv.y);
          x.x += __low2float(p01); x.y += __high2float(p01); x.z += __low2float(p23); x.w += __high2float(p23);
          const long ci = ((long)g * p.B + b) * LH + j;
          const float c = fmaf(sigmoid_fast(x.y), cprev[itr], sigmoid_fast(x.x) * tanh_fast(x.z));
          const float h = sigmoid_fast(x.w) * tanh_fast(c);
          p.cst[ci] = c;
          const __nv_bfloat16 hb = __float2bfloat16_rn(h);
          hout[ci] = hb;
          recp[(long)b * p.rec_row] = hb;
        }
#pragma unroll
        for (int itr = 0; itr < 8; ++itr) pvv[itr] = pvn[itr];
        __syncwarp();
      }
      tc_fence_before();
      if (s + 1 < p.CT) {
        // next step's input pre-activations (128 rows x 512 B of this CTA's gate columns): HBM -> L2 while the barrier settles
        const int tn = dir ? p.CT - 2 - s : s + 1;
        const char* pn = reinterpret_cast<const char*>(p.pre + (long)e * p.pre_e + (long)tn * (8 * LH) + dir * 4 * LH + nq * 256);
        const int t2 = threadIdx.x;                            // 256 threads: row = t2 / 2, 256-byte half = t2 & 1 (two 128-byte lines)
        const char* a = pn + (long)(m0 + (t2 >> 1)) * p.pre_row * 2 + (t2 & 1) * 256;
        asm volatile("prefetch.global.L2 [%0];" ::"l"(a));
        asm volatile("prefetch.global.L2 [%0];" ::"l"(a + 128));
      }
    }
    // h_s of all four gate-column quarters becomes visible to the cluster; the accumulator and the operand tile are free
    cluster_sync_all();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, 256);
}

// 3-D map over a [groups][rows][K] bf16 operand (K contiguous): box = 64 x box_rows x 1, 128B swizzle, zero OOB fill
int make_map(CUtensorMap* map, const void* ptr, long K, long rows, long groups, long ld, long gstride, int box_rows) {
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) || (ld % 8) || (groups > 1 && gstride % 8)) {
    mrnb_set_error("tc_gemm: operand must be 16-byte aligned with ld %% 8 == 0 (ptr=%p ld=%ld gstride=%ld)", ptr, ld, gstride);
    return MRNB_ERR_ARG;
  }
  cuuint64_t dims[3] = {(cuuint64_t)K, (cuuint64_t)rows, (cuuint64_t)groups};
  cuuint64_t strides[2] = {(cuuint64_t)ld * 2, (cuuint64_t)(groups > 1 ? gstride : rows * ld) * 2};
  cuuint32_t box[3] = {(cuuint32_t)BK, (cuuint32_t)box_rows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  return encode_tensor_map("tc_gemm", map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, ptr, dims, strides, box, estr, CU_TENSOR_MAP_SWIZZLE_128B);
}

int make_conv_map(CUtensorMap* map, const void* ptr, const MrnbTcConv& c) {
  cuuint64_t dims[4], strides[3];
  for (int j = 0; j < 4; ++j) dims[j] = (cuuint64_t)c.dims[j];
  for (int j = 0; j < 3; ++j) strides[j] = (cuuint64_t)c.strides[j] * 2;
  // with a traversal stride s the box spans (n - 1) * s + 1 elements to pick up n of them
  const int bw = c.box_w > 0 ? c.box_w : 64;
  cuuint32_t box[4] = {64, (cuuint32_t)bw, (cuuint32_t)((c.box_h - 1) * c.sh + 1), (cuuint32_t)c.box_img};
  cuuint32_t estr[4] = {1, 1, (cuuint32_t)(c.box_h > 1 ? c.sh : 1), 1};
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) || c.box_h * c.box_img * bw != BM || (bw != 64 && bw != 128)) {
    mrnb_set_error("tc_gemm: bad convolution view");
    return MRNB_ERR_ARG;
  }
  return encode_tensor_map("tc_gemm (conv)", map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, ptr, dims, strides, box, estr,
                           CU_TENSOR_MAP_SWIZZLE_128B);
}

// 2-D map over an fp32 [rows][cols] output (row pitch ld floats): box 32 x 32, 128B swizzle -- the TMA-store epilogue
bool make_out_map(CUtensorMap* map, void* ptr, long cols, long rows, long ld) {
  EncodeTiledFn fn = tensor_map_encoder();
  if (!fn || (reinterpret_cast<uintptr_t>(ptr) & 15) || (ld % 4)) return false;
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 4};
  cuuint32_t box[2] = {32, 32};
  cuuint32_t estr[2] = {1, 1};
  return fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, ptr, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

template <int BN, bool OUT_F32, bool GELU, bool LNF, int MODE = 0>
int launch_tc(const MrnbTcGemm& p, cudaStream_t st) {
  CUtensorMap tmA, tmW;
  if (p.conv.enabled) MRNB_TRY(make_conv_map(&tmA, p.A, p.conv));
  else MRNB_TRY(make_map(&tmA, p.A, p.K, p.M, p.groups, p.lda, p.a_gstride, BM));
  MRNB_TRY(make_map(&tmW, p.W, p.K, p.N, p.groups, p.ldw, p.w_gstride, BN));
  TcEpi ep;
  ep.bias = p.bias; ep.bias_gs = p.bias_gstride;
  ep.out = p.out; ep.ldo = p.ldo; ep.o_gs = p.o_gstride;
  ep.res = p.res; ep.rowscale = p.rowscale; ep.rows_per_scale = p.rows_per_scale > 0 ? p.rows_per_scale : 1;
  ep.rowscale_gs = p.rowscale_gstride;
  ep.M = p.M; ep.N = p.N; ep.KB = p.K / BK; ep.gelu = p.gelu;
  ep.stages = ep.KB < MAX_STAGES ? ep.KB : MAX_STAGES;
  ep.ln_out = (__nv_bfloat16*)p.ln_out; ep.ln_gs = p.ln_gstride; ep.ln_gamma = p.ln_gamma; ep.ln_beta = p.ln_beta; ep.ln_eps = p.ln_eps;
  ep.conv = p.conv.enabled; ep.rows_per_img = p.conv.rows_per_img; ep.per_kh = p.conv.per_kh; ep.cch = p.conv.cch;
  ep.w_off = p.conv.w_off; ep.sh = p.conv.sh; ep.imgs_per_group = p.conv.imgs_per_group;
  ep.ow_shift = p.conv.box_w == 128 ? 7 : 6; ep.pad_h = p.conv.pad_h; ep.relu = p.relu;
  ep.lstm = p.lstm;
  ep.n_tiles = cdiv(p.N, BN); ep.m_tiles = cdiv(p.M, BM);
  ep.total_tiles = ep.n_tiles * ep.m_tiles * p.groups;
  const size_t smem = 1024 + (size_t)ep.stages * (A_STAGE_BYTES + BN * BK * 2) + STAGING_BYTES;
  static bool attr_set = false;
  static int num_sms = 148;
  if (!attr_set) {
    cudaFuncSetAttribute(tc_gemm_kernel<BN, OUT_F32, GELU, LNF, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                         1024 + MAX_STAGES * (A_STAGE_BYTES + BN * BK * 2) + STAGING_BYTES);
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
    attr_set = true;
  }
  const int slots = (LNF ? 1 : 2) * num_sms;                                  // persistent CTAs: two per SM (one with fused LN)
  const int grid = ep.total_tiles < slots ? ep.total_tiles : slots;
  static const TcOutMaps no_maps{};
  tc_gemm_kernel<BN, OUT_F32, GELU, LNF, MODE><<<grid, NTHREADS, smem, st>>>(tmA, tmW, ep, no_maps);
  MRNB_CHECK_LAUNCH("tc_gemm_kernel");
  return MRNB_OK;
}

}  // namespace

int mrnb_tc_gemm(const MrnbTcGemm& p, cudaStream_t st) {
  MRNB_CHECK_ARG(p.A && p.W && p.out && p.M > 0 && p.N > 0 && p.K > 0 && p.groups > 0, "tc_gemm: bad argument");
  MRNB_CHECK_ARG(p.K % BK == 0, "tc_gemm: K=%d must be a multiple of %d", p.K, BK);
  MRNB_CHECK_ARG(!p.res || p.out_f32, "tc_gemm: residual needs an fp32 output");
  MrnbProfScope prof(MRNB_PROF_TCGEMM, st, 2.0 * p.M * p.N * p.K * p.groups,
                     (double)p.groups * (2.0 * p.M * p.K + 2.0 * p.N * p.K + (double)p.M * p.N * (p.out_f32 ? 4 : 2) +
                                         (p.res ? 4.0 * p.M * p.N : 0.0)));
  const bool wide = p.N >= 128 && (p.N % 128 == 0 || p.N > 256);
  if (p.lstm.enabled) {
    MRNB_CHECK_ARG(p.M % BM == 0 && p.N % 128 == 0 && !p.bias && !p.res && !p.rowscale && !p.gelu && !p.relu && !p.ln_out &&
                   p.lstm.pre && p.lstm.cst && p.lstm.hst && p.lstm.rec && p.lstm.pre_row % 4 == 0 && p.lstm.pre_e % 4 == 0 &&
                   p.lstm.pre_off[0] % 4 == 0 && p.lstm.pre_off[1] % 4 == 0,
                   "tc_gemm: fused LSTM cell needs M %% 128 == 0, N %% 128 == 0 and 8-byte aligned pre-activations");
    return launch_tc<128, true, false, false, 1>(p, st);
  }
  if (p.pool4) {
    MRNB_CHECK_ARG(!p.out_f32 && p.M % BM == 0 && (p.N == 64 || p.N % 128 == 0) && p.ldo % 4 == 0 && p.o_gstride % 4 == 0 && !p.res &&
                   !p.rowscale && !p.gelu && !p.ln_out, "tc_gemm: pooled epilogue needs bf16 output, M %% 128 == 0, N == 64 or N %% 128 == 0");
    return p.N == 64 ? launch_tc<64, false, false, false, 2>(p, st) : launch_tc<128, false, false, false, 2>(p, st);
  }
  if (p.ln_out) {
    // fused LayerNorm: the tile must span whole rows and every tile must take the interior path
    MRNB_CHECK_ARG(p.out_f32 && !p.gelu && (p.N == 64 || p.N == 128) && p.M % BM == 0 && p.ldo % 4 == 0 && p.o_gstride % 4 == 0 &&
                   p.ln_gamma && p.ln_beta && (!p.rowscale || p.rows_per_scale % BM == 0),
                   "tc_gemm: fused LayerNorm needs N in {64,128}, M %% 128 == 0, aligned fp32 output");
    return p.N == 128 ? launch_tc<128, true, false, true>(p, st) : launch_tc<64, true, false, true>(p, st);
  }
#define MRNB_GO(BN_)                                                                                              \
  if (p.out_f32) return p.gelu ? launch_tc<BN_, true, true, false>(p, st) : launch_tc<BN_, true, false, false>(p, st);   \
  return p.gelu ? launch_tc<BN_, false, true, false>(p, st) : launch_tc<BN_, false, false, false>(p, st);
  if (wide) { MRNB_GO(128) }
  MRNB_GO(64)
#undef MRNB_GO
}

int mrnb_tc_heads(const void* A, long lda, long a_gstride, const void* Wall, long w_rows, int M, int K, MrnbTcHeads H, cudaStream_t st) {
  MRNB_CHECK_ARG(A && Wall && M > 0 && K > 0 && K % BK == 0 && H.n_experts >= 1 && H.n_experts <= 8, "tc_heads: bad argument");
  MRNB_CHECK_ARG(!H.route || (H.rows_per_sample > 0 && H.n_samples > 0), "tc_heads: route needs rows_per_sample / n_samples");
  const int m_tiles = cdiv(M, BM);
  double flops = 0, bytes = 0;
  H.tile_prefix[0] = 0;
  for (int e = 0; e < H.n_experts; ++e) {
    MRNB_CHECK_ARG(H.out[e] && H.N[e] > 0 && H.ldo[e] >= H.N[e] && H.woff[e] >= 0 && H.woff[e] + H.N[e] <= w_rows, "tc_heads: bad expert %d", e);
    H.n_tiles[e] = cdiv(H.N[e], 128);
    H.tile_prefix[e + 1] = H.tile_prefix[e] + H.n_tiles[e] * m_tiles;
    const double frac = H.route ? 1.0 / H.n_experts : 1.0;     // hard route: ~1 / I of the (expert, sample) pairs are computed
    flops += 2.0 * M * H.N[e] * K * frac;
    bytes += (2.0 * M * K + 2.0 * H.N[e] * K) + 4.0 * M * H.N[e] * frac;
  }
  MrnbProfScope prof(MRNB_PROF_TCGEMM, st, flops, bytes);
  CUtensorMap tmA, tmW;
  MRNB_TRY(make_map(&tmA, A, K, M, H.n_experts, lda, a_gstride, BM));
  MRNB_TRY(make_map(&tmW, Wall, K, w_rows, 1, K, 0, 128));
  TcEpi ep{};
  ep.M = M; ep.N = 0; ep.KB = K / BK; ep.stages = ep.KB < MAX_STAGES ? ep.KB : MAX_STAGES;
  ep.rows_per_scale = 1; ep.n_tiles = 1; ep.m_tiles = m_tiles; ep.total_tiles = H.tile_prefix[H.n_experts];
  ep.heads = H;
  TcOutMaps maps{};
  ep.tma_out = 1;
  { const char* e = getenv("MRNB_HEADS_TMA"); if (e && atoi(e) == 0) ep.tma_out = 0; }
  for (int e = 0; e < H.n_experts && ep.tma_out; ++e)
    if (!H.bias[e] || !make_out_map(&maps.m[e], H.out[e], H.N[e], M, H.ldo[e])) ep.tma_out = 0;
  constexpr int BN_ = 128;
  const size_t smem = 1024 + (size_t)ep.stages * (A_STAGE_BYTES + BN_ * BK * 2) + STAGING_BYTES;
  static bool attr_set = false;
  static int num_sms = 148;
  if (!attr_set) {
    cudaFuncSetAttribute(tc_gemm_kernel<BN_, true, false, false, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                         1024 + MAX_STAGES * (A_STAGE_BYTES + BN_ * BK * 2) + STAGING_BYTES);
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
    attr_set = true;
  }
  const int slots = 2 * num_sms;
  const int grid = ep.total_tiles < slots ? ep.total_tiles : slots;
  tc_gemm_kernel<BN_, true, false, false, 3><<<grid, NTHREADS, smem, st>>>(tmA, tmW, ep, maps);
  MRNB_CHECK_LAUNCH("tc_gemm_kernel");
  return MRNB_OK;
}

extern "C" int mrnb_linear_bf16(const void* A, const void* W, const float* bias, const float* residual, void* out,
                                int out_is_f32, int M, int N, int K, int act_gelu, cudaStream_t stream) {
  MrnbTcGemm g{};
  g.A = A; g.lda = K; g.W = W; g.ldw = K; g.bias = bias; g.out = out; g.ldo = N; g.out_f32 = out_is_f32;
  g.res = residual; g.M = M; g.N = N; g.K = K; g.groups = 1; g.gelu = act_gelu; g.rows_per_scale = 1;
  return mrnb_tc_gemm(g, stream);
}

// Persistent LSTM recurrence: steps s_first .. CT-1 of `groups` = 2 x experts chains in one cluster launch.
// Whh: bf16 [groups][4H = 1024 (gate-interleaved)][H = 256].  Returns MRNB_ERR_UNSUPPORTED when the shape does not fit
// (the caller falls back to one grouped GEMM per step).
int mrnb_tc_lstm_seq(const void* Whh, const void* pre, long pre_row, long pre_e, void* rec, long rec_row, long rec_e, float* cst,
                     void* h0, void* h1, int groups, int B, int CT, int s_first, cudaStream_t st) {
  if (B % BM != 0 || groups <= 0 || s_first < 1 || s_first >= CT) return MRNB_ERR_UNSUPPORTED;
  static int num_sms = 0;
  if (!num_sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
    if (cudaFuncSetAttribute(lstm_seq_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, LSEQ_SMEM) != cudaSuccess) { cudaGetLastError(); num_sms = -1; }
  }
  const int grid = groups * (B / BM) * 4;
  if (num_sms <= 0 || grid > num_sms) return MRNB_ERR_UNSUPPORTED;       // every cluster must be resident (one CTA per SM)
  CUtensorMap tmW;
  MRNB_TRY(make_map(&tmW, Whh, 256, 1024, groups, 256, 1024L * 256, 256));
  LstmSeqArgs a{};
  a.pre = (const __nv_bfloat16*)pre; a.pre_row = pre_row; a.pre_e = pre_e;
  a.rec = (__nv_bfloat16*)rec; a.rec_row = rec_row; a.rec_e = rec_e;
  a.cst = cst; a.h0 = (__nv_bfloat16*)h0; a.h1 = (__nv_bfloat16*)h1; a.B = B; a.CT = CT; a.s_first = s_first;
  MrnbProfScope prof(MRNB_PROF_TCGEMM, st, 2.0 * B * 1024.0 * 256.0 * groups * (CT - s_first), 0.0);
  lstm_seq_kernel<<<grid, LSEQ_THREADS, LSEQ_SMEM, st>>>(tmW, a);
  MRNB_CHECK_LAUNCH("lstm_seq_kernel");
  return MRNB_OK;
}
