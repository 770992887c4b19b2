// Fused transformer MLP branch of an SVTR block on the tensor cores (bf16 mode):
//
//     x <- x + rs * ( GELU( LN2(x) W1^T + b1 ) W2^T + b2 )            [ + LN1_next(x) for the following block ]
//
// Reference: modules/svtr.py:61-67 (Mlp), :200-204 (Block.forward second branch), DropPath :7-22.
// The 4d-wide hidden activation never leaves the SM: for every 128-row tile the kernel walks the hidden axis in
// chunks of 128:   S_c = A W1_c^T  (tcgen05, TMEM, double buffered)  ->  epilogue warps: +b1, GELU, bf16 -> smem P
//                  O  += P W2_c^T  (tcgen05, TMEM accumulator of width d)
// and the final epilogue adds b2, the DropPath scale and the fp32 residual, stores x in place and (d <= 128)
// emits the next LayerNorm.  Per tile HBM traffic: A (bf16) + x in + x out (+ LN out) instead of two GEMM round trips
// through a [M,4d] tensor.
// Warp roles (four warpgroups, register budgets re-balanced with setmaxnreg): WG0 = control (warp 0 TMA producer, warp 1
// TMEM + MMA issuer), WG1 / WG2 = the eight GELU warps (S_c -> P_c), WG3 = output epilogue (O -> x, LayerNorm).  The output
// epilogue of tile i runs while the GELU warps already work on tile i + 1 (ncu source view of the previous single-epilogue
// version: 31 % of the epilogue warps' samples sat in the O -> x / LayerNorm code, serialised with the GELU chunks); the
// O accumulator is double buffered in TMEM for d <= 128.
#include "mlp_tc.h"
#include "sm100.cuh"

namespace {

constexpr int BM = 128, BK = 64, HC = 128;       // rows per tile, k-block, hidden chunk
constexpr int EPI_WARPS = 8, NTHREADS = 512;
constexpr int REGS_CTRL = 80, REGS_GELU = 168, REGS_OUT = 96;       // 128 * (80 + 2 * 168 + 96) = 65536
constexpr int TILE16K = 128 * 64 * 2;

// 16-byte-chunk swizzle key of row rl in the staged fp32 tiles (row pitch a multiple of 128 B): a quarter warp touches
// rows {2k, 2k+1} x 4 consecutive chunks, so bit 2 separates the two rows and bits 0-1 the row pairs -> conflict free
__device__ __forceinline__ int xs_key(int rl) { return ((rl & 1) << 2) | ((rl >> 1) & 3); }
struct MlpParams {
  const float* b1; const float* b2; long b_gs1, b_gs2;        // [groups][4D], [groups][D]
  float* x; long x_gs;                                        // fp32 residual stream, in place: [g][rows][D]
  const float* rowscale; int rows_per_scale; long rowscale_gs;
  __nv_bfloat16* ln_out; long ln_gs; const float* ln_gamma; const float* ln_beta; float ln_eps;   // optional (D <= 128)
  __nv_bfloat16* cast_out;   // optional bf16 copy of the new rows, [g][M][D] (stride ln_gs)
  int m_tiles, total_tiles;
  unsigned long long* trace;      // optional debug timeline (CTA 0), see MRNB_TRACE
};

#define MRNB_TRACE(slot_, idx_)                                                                    \
  do {                                                                                             \
    if (ep.trace && blockIdx.x == 0 && (idx_) < 64) {                                              \
      unsigned long long now__;                                                                    \
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now__));                                    \
      ep.trace[(slot_) * 64 + (idx_)] = now__;                                                     \
    }                                                                                              \
  } while (0)

template <int D>
struct Cfg {
  static constexpr int KB = D / BK;                    // k-blocks of the first GEMM
  static constexpr int C = 4 * D / HC;                 // hidden chunks: 2, 4, 8
  static constexpr int SLOT = D > 128 ? 32768 : 16384; // ring slot: W1 k-block [128 x 64] or W2 k-block [D x 64]
  static constexpr int RS = D > 128 ? 3 : 4;           // ring slots.  D = 256 streams 1 MiB of weights per 128-row tile: that
                                                       // launch is L2-bandwidth bound (1.5 GB / launch), see DESIGN.md
  static constexpr int NH = 1;                         // N-splits of the second GEMM (UMMA N = D / NH)
  static constexpr int W2ROWS = D / NH;
  static constexpr int A_BYTES = KB * TILE16K;
  static constexpr int P_BYTES = 2 * TILE16K;          // [128 x 128] bf16 as two 64-wide K halves
  static constexpr int BIAS_BYTES = 4 * D * 4;
  static constexpr int STG_BYTES = 4 * 2048;           // output-epilogue staging: 32 rows x 16 fp32 per warp
  static constexpr int XT_BYTES = D <= 128 ? BM * D * 4 : 0;   // new rows of the tile for the fused LayerNorm (D <= 128)
  static constexpr int SMEM = 1024 + A_BYTES + P_BYTES + RS * SLOT + BIAS_BYTES + STG_BYTES + XT_BYTES;
  static constexpr uint32_t O_COL = 256;               // TMEM: S buffers at 0 / 128, O at 256 (+ D for the second buffer)
  static constexpr int OB = D <= 128 ? 2 : 1;          // O accumulators
};

template <int D, bool LNF>
__global__ void __launch_bounds__(NTHREADS, 1)
mlp_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW1,
              const __grid_constant__ CUtensorMap tmW2, const MlpParams ep) {
  using K = Cfg<D>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + align_smem_1024_offset(smem_raw);
  uint8_t* sA = smem;
  uint8_t* sP = smem + K::A_BYTES;
  uint8_t* ring = sP + K::P_BYTES;
  float* sb1 = reinterpret_cast<float*>(ring + K::RS * K::SLOT);
  uint8_t* sStg = reinterpret_cast<uint8_t*>(sb1 + 4 * D);
  float* sXt = reinterpret_cast<float*>(sStg + K::STG_BYTES);   // [128][D] fp32, 16-byte pieces XOR-swizzled by row (LNF only)
  __shared__ __align__(8) uint64_t a_full, a_empty, w_full[8], w_empty[8], s_full[2], s_empty[2], p_full, p_empty, o_full[2], o_empty[2];
  __shared__ uint32_t tmem_base_sh;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int total = ep.total_tiles, m_tiles = ep.m_tiles;

  if (threadIdx.x == 0) {
    mbar_init(&a_full, 1); mbar_init(&a_empty, 1);
    for (int s = 0; s < K::RS; ++s) { mbar_init(&w_full[s], 1); mbar_init(&w_empty[s], 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(&s_full[b], 1); mbar_init(&s_empty[b], EPI_WARPS); }
    mbar_init(&p_full, EPI_WARPS); mbar_init(&p_empty, 1);
    for (int b = 0; b < 2; ++b) { mbar_init(&o_full[b], 1); mbar_init(&o_empty[b], 4); }
    fence_mbarrier_init();
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmW1);
    prefetch_tmap(&tmW2);
  }
  if (warp == 1) tmem_alloc(&tmem_base_sh, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_sh;

  if (warp < 4) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_CTRL));
  if (warp == 0) {
    // ============================== TMA producer ==============================
    if (lane == 0) {
      uint32_t it = 0;
      auto load_w = [&](const CUtensorMap* map, int c0, int c1, int g, uint32_t bytes) {
        const int s = it % K::RS;
        mbar_wait_nohint(&w_empty[s], ((it / K::RS) & 1u) ^ 1u);
        mbar_expect_tx(&w_full[s], bytes);
        tma_load_3d(ring + (size_t)s * K::SLOT, map, &w_full[s], c0, c1, g);
        ++it;
      };
      // Ring order = consumption order of the MMA issuer: A_0, W1_0 ; then per tile, per chunk c:
      //   { W1_{c+1}  |  at the last chunk: A and W1_0 of the NEXT tile (its S_0 is issued before this tile's last P W2) } ; W2_c
      auto load_a = [&](int ti, int t) {
        const int g = t / m_tiles, m0 = (t % m_tiles) * BM;
        mbar_wait_nohint(&a_empty, ((uint32_t)ti & 1u) ^ 1u);
        mbar_expect_tx(&a_full, K::A_BYTES);
        for (int kb = 0; kb < K::KB; ++kb) tma_load_3d(sA + kb * TILE16K, &tmA, &a_full, kb * BK, m0, g);
        for (int kb = 0; kb < K::KB; ++kb) load_w(&tmW1, kb * BK, 0, g, TILE16K);
      };
      int i = 0;
      if ((int)blockIdx.x < total) load_a(0, blockIdx.x);
      for (int t = blockIdx.x; t < total; t += gridDim.x, ++i) {
        const int g = t / m_tiles;
        for (int c = 0; c < K::C; ++c) {
          if (c + 1 < K::C) {
            for (int kb = 0; kb < K::KB; ++kb) load_w(&tmW1, kb * BK, (c + 1) * HC, g, TILE16K);
          } else if (t + (int)gridDim.x < total) {
            load_a(i + 1, t + gridDim.x);
          }
          for (int kk = 0; kk < 2; ++kk)
            for (int nh = 0; nh < K::NH; ++nh) load_w(&tmW2, c * HC + kk * BK, nh * K::W2ROWS, g, K::W2ROWS * BK * 2);
        }
      }
    }
  } else if (warp == 1) {
    // ============================== MMA issuer ==============================
    if (lane == 0) {
      constexpr uint32_t idesc_s = umma_idesc(UMMA_BF16, BM, HC);
      constexpr uint32_t idesc_o = umma_idesc(UMMA_F16, BM, K::W2ROWS);      // second GEMM in f16 x f16: P (GELU output) and W2 are f16
      uint32_t it = 0;
      int i = 0;
      auto issue_s = [&](int ti, int c) {
          const int b = c & 1;
          const uint32_t u = (uint32_t)(ti * (K::C / 2) + (c >> 1));
          mbar_wait_nohint(&s_empty[b], (u & 1u) ^ 1u);
          tc_fence_after();
          for (int kb = 0; kb < K::KB; ++kb, ++it) {
            const int s = it % K::RS;
            mbar_wait_nohint(&w_full[s], (it / K::RS) & 1u);
            tc_fence_after();
            const uint64_t ad = umma_desc_k128(smem_u32(sA + kb * TILE16K)), bd = umma_desc_k128(smem_u32(ring + (size_t)s * K::SLOT));
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_bf16(tmem_base + (uint32_t)(b * HC), ad + (uint64_t)(k * 2), bd + (uint64_t)(k * 2), idesc_s, (kb | k) != 0);
            umma_commit(&w_empty[s]);
          }
          umma_commit(&s_full[b]);
      };
      if ((int)blockIdx.x < total) { mbar_wait_nohint(&a_full, 0u); issue_s(0, 0); }
      for (int t = blockIdx.x; t < total; t += gridDim.x, ++i) {
        for (int c = 0; c < K::C; ++c) {
          if (c + 1 < K::C) {
            issue_s(i, c + 1);
          } else if (t + (int)gridDim.x < total) {
            // S_0 of the NEXT tile goes out before this tile's last P W2: the GELU warps find it ready at the tile boundary
            mbar_wait_nohint(&a_full, (uint32_t)(i + 1) & 1u);
            issue_s(i + 1, 0);
          }
          if (c + 1 == K::C - 1) umma_commit(&a_empty);                   // last S of this tile issued: A is free once it retires
          const uint32_t up = (uint32_t)(i * K::C + c);
          MRNB_TRACE(0, (int)up);                          // MMA: S_{c+1} issued, start waiting for P_c
          mbar_wait_nohint(&p_full, up & 1u);
          MRNB_TRACE(1, (int)up);                          // MMA: P_c available
          // O accumulator of this tile: buffer i % OB, free once the output epilogue of tile i - OB has drained it
          const uint32_t ob = K::OB == 2 ? ((uint32_t)i & 1u) : 0u, on = K::OB == 2 ? ((uint32_t)i >> 1) : (uint32_t)i;
          if (c == 0) mbar_wait_nohint(&o_empty[ob], (on & 1u) ^ 1u);
          tc_fence_after();
          for (int kk = 0; kk < 2; ++kk) {
            for (int nh = 0; nh < K::NH; ++nh, ++it) {
              const int s = it % K::RS;
              mbar_wait_nohint(&w_full[s], (it / K::RS) & 1u);
              tc_fence_after();
              const uint64_t ad = umma_desc_k128(smem_u32(sP + kk * TILE16K)), bd = umma_desc_k128(smem_u32(ring + (size_t)s * K::SLOT));
#pragma unroll
              for (int k = 0; k < 4; ++k)
                umma_bf16(tmem_base + K::O_COL + ob * (uint32_t)D + (uint32_t)(nh * K::W2ROWS), ad + (uint64_t)(k * 2),
                          bd + (uint64_t)(k * 2), idesc_o, (c | kk | k) != 0);
              umma_commit(&w_empty[s]);
            }
          }
          umma_commit(&p_empty);
          MRNB_TRACE(2, (int)up);                          // MMA: PV_c issued
          if (c == K::C - 1) umma_commit(&o_full[ob]);
        }
      }
    }
  } else if (warp >= 4 && warp < 12) {
    // ============================== GELU warps: S_c -> +b1 -> GELU -> f16 P_c ==============================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(REGS_GELU));
    const int ew = warp - 4, q = warp & 3, ch = ew >> 2;
    const int r = q * 32 + lane;                               // row inside the tile == TMEM lane
    const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
    int i = 0;
    int cur_g = -1;
    for (int t = blockIdx.x; t < total; t += gridDim.x, ++i) {
      const int g = t / m_tiles;
      if (warp == 4 && lane == 0) MRNB_TRACE(9, i);                // epi: tile start
      if (g != cur_g) {                                        // (re)load the fc1 bias of this expert
        asm volatile("bar.sync 5, 256;" ::: "memory");         // everyone done with the previous expert's bias
        for (int k = threadIdx.x - 128; k < 4 * D; k += EPI_WARPS * 32) sb1[k] = ep.b1[(long)g * ep.b_gs1 + k];
        asm volatile("bar.sync 5, 256;" ::: "memory");
        cur_g = g;
      }
      for (int c = 0; c < K::C; ++c) {
        const int b = c & 1;
        const uint32_t u = (uint32_t)(i * (K::C / 2) + (c >> 1));
        if (warp == 4 && lane == 0) MRNB_TRACE(3, i * K::C + c);   // epi: start waiting for S_c
        mbar_wait_nohint(&s_full[b], u & 1u);
        if (warp == 4 && lane == 0) MRNB_TRACE(4, i * K::C + c);   // epi: S_c ready
        tc_fence_after();
        uint32_t v0[32], v1[32];
        tmem_ld32(lane_addr + (uint32_t)(b * HC + ch * 64), v0);
        tmem_ld32(lane_addr + (uint32_t)(b * HC + ch * 64 + 32), v1);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&s_empty[b]);
        // +b1 (fp32), then GELU two values at a time in f16x2; P is handed to the tensor core as an f16 operand
        const float4* bb4 = reinterpret_cast<const float4*>(sb1 + c * HC + ch * 64);
        uint32_t pk[32];
#pragma unroll
        for (int e4 = 0; e4 < 16; ++e4) {                       // 4 columns per step
          const float4 bq = bb4[e4];
          const int col = e4 * 4;
          const float a0 = __uint_as_float(col < 32 ? v0[col] : v1[col - 32]) + bq.x;
          const float a1 = __uint_as_float(col < 32 ? v0[col + 1] : v1[col + 1 - 32]) + bq.y;
          const float a2 = __uint_as_float(col < 32 ? v0[col + 2] : v1[col + 2 - 32]) + bq.z;
          const float a3 = __uint_as_float(col < 32 ? v0[col + 3] : v1[col + 3 - 32]) + bq.w;
          const __half2 g0 = gelu_fast_h2(__floats2half2_rn(a0, a1)), g1 = gelu_fast_h2(__floats2half2_rn(a2, a3));
          pk[e4 * 2] = *reinterpret_cast<const uint32_t*>(&g0);
          pk[e4 * 2 + 1] = *reinterpret_cast<const uint32_t*>(&g1);
        }
        const uint32_t up = (uint32_t)(i * K::C + c);
        if (warp == 4 && lane == 0) MRNB_TRACE(5, (int)up);        // epi: GELU done
        mbar_wait_nohint(&p_empty, (up & 1u) ^ 1u);                   // previous P has been consumed by its MMAs (GELU already done)
        if (warp == 4 && lane == 0) MRNB_TRACE(6, (int)up);        // epi: P buffer free
        uint8_t* prow = sP + ch * TILE16K + r * 128;
#pragma unroll
        for (int pc = 0; pc < 8; ++pc)                          // 8 pieces of 8 columns (16 B of bf16), XOR-swizzled by row
          *reinterpret_cast<uint4*>(prow + ((pc ^ (r & 7)) * 16)) = make_uint4(pk[pc * 4], pk[pc * 4 + 1], pk[pc * 4 + 2], pk[pc * 4 + 3]);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive(&p_full);
        if (warp == 4 && lane == 0) MRNB_TRACE(7, (int)up);        // epi: P_c published
      }
    }
  } else if (warp >= 12) {
    // ============================== output epilogue warpgroup ==============================
    // O -> +b2, DropPath scale, + fp32 residual -> x (in place) [+ bf16 copy | + LayerNorm of the next block], one warp
    // per TMEM lane quarter, while the other warpgroups already work on the next tile.  16 accumulator columns of the
    // warp's 32 rows are transposed through a 2 KiB staging tile (16-byte pieces XOR-swizzled by row) so that global
    // accesses are 64-byte row segments: lane = (row in a group of 8, float4 of the 16).  (32-column steps with 8 lanes per
    // row segment measured slower: register spills under the 96-register budget of this warpgroup.)
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_OUT));
    const int q = warp & 3;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
    float* stg = reinterpret_cast<float*>(sStg + q * 2048);
    const int rsub = lane >> 2, c4 = lane & 3;
    int i = 0;
    for (int t = blockIdx.x; t < total; t += gridDim.x, ++i) {
      const int g = t / m_tiles, m0 = (t % m_tiles) * BM;
      const uint32_t ob = K::OB == 2 ? ((uint32_t)i & 1u) : 0u, on = K::OB == 2 ? ((uint32_t)i >> 1) : (uint32_t)i;
      const float rs = ep.rowscale ? ep.rowscale[(long)g * ep.rowscale_gs + m0 / ep.rows_per_scale] : 1.0f;
      float* xt = ep.x + (long)g * ep.x_gs + (long)(m0 + q * 32) * D;        // the warp's 32 rows
      const float* b2p = ep.b2 + (long)g * ep.b_gs2;
      float* xs = sXt + (size_t)(q * 32) * D;                  // this warp's rows of the staged tile (D <= 128)
      if constexpr (LNF && K::XT_BYTES > 0) {
        // idle until the tile's last P W2 MMA retires: the residual rows (32 x D fp32) travel HBM -> shared memory now
        // (cp.async, swizzled like the LayerNorm tile they will be overwritten into), so that neither pass below waits
        // for a global load -- the ncu source view put both passes on long-scoreboard stalls of those loads
#pragma unroll
        for (int c = 0; c < D / 16; ++c)
#pragma unroll
          for (int it = 0; it < 4; ++it) {
            const int rl = it * 8 + rsub;
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(xs + rl * D + (((c * 4 + c4) ^ xs_key(rl)) * 4))),
                         "l"(xt + (long)rl * D + c * 16 + c4 * 4) : "memory");
          }
        asm volatile("cp.async.commit_group;" ::: "memory");
      } else {
        // idle until the tile's last P W2 MMA retires: start the trip of the residual rows (32 x D fp32) to L2 now
        const char* xl2 = reinterpret_cast<const char*>(xt);
#pragma unroll
        for (int k = 0; k < D / 32; ++k) asm volatile("prefetch.global.L2 [%0];" ::"l"(xl2 + (long)(k * 32 + lane) * 128));
      }
      mbar_wait_nohint(&o_full[ob], on & 1u);
      if (warp == 12 && lane == 0) MRNB_TRACE(8, i);               // out: O ready
      tc_fence_after();
      __nv_bfloat16* ct = (!LNF && ep.cast_out) ? ep.cast_out + (long)g * ep.ln_gs + (long)(m0 + q * 32) * D : nullptr;
      float sum[4] = {0.f, 0.f, 0.f, 0.f}, sq[4] = {0.f, 0.f, 0.f, 0.f};
      constexpr bool XS = LNF && K::XT_BYTES > 0;              // residual rows staged in shared memory (LayerNorm variants:
                                                               // without the LayerNorm the GELU warps are the bottleneck and the extra
                                                               // shared-memory traffic cost them 151 -> 162 us at d = 64)
      float4 xin[4], xnx[4];
      if constexpr (XS) {
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncwarp();
      } else {
#pragma unroll
        for (int it = 0; it < 4; ++it) xin[it] = *reinterpret_cast<const float4*>(xt + (long)(it * 8 + rsub) * D + c4 * 4);
      }
#pragma unroll 1
      for (int c = 0; c < D / 16; ++c) {
        if constexpr (XS) {
#pragma unroll
          for (int it = 0; it < 4; ++it) {
            const int rl = it * 8 + rsub;
            xin[it] = *reinterpret_cast<const float4*>(xs + rl * D + (((c * 4 + c4) ^ xs_key(rl)) * 4));
          }
        } else if (c + 1 < D / 16) {                           // residual rows of the next 16 columns: in flight during this step
#pragma unroll
          for (int it = 0; it < 4; ++it) xnx[it] = *reinterpret_cast<const float4*>(xt + (long)(it * 8 + rsub) * D + (c + 1) * 16 + c4 * 4);
        }
        uint32_t v[16];
        tmem_ld16(lane_addr + K::O_COL + ob * (uint32_t)D + (uint32_t)(c * 16), v);
        if (c == D / 16 - 1) {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&o_empty[ob]);            // accumulator drained: a later tile may overwrite it
        }
#pragma unroll
        for (int pc = 0; pc < 4; ++pc)
          *reinterpret_cast<float4*>(stg + lane * 16 + ((pc ^ ((lane >> 1) & 3)) * 4)) =
              make_float4(__uint_as_float(v[4 * pc]), __uint_as_float(v[4 * pc + 1]), __uint_as_float(v[4 * pc + 2]), __uint_as_float(v[4 * pc + 3]));
        __syncwarp();
        const float4 b4 = __ldg(reinterpret_cast<const float4*>(b2p + c * 16 + c4 * 4));
#pragma unroll
        for (int it = 0; it < 4; ++it) {
          const int rl = it * 8 + rsub;
          const float4 a = *reinterpret_cast<const float4*>(stg + rl * 16 + ((c4 ^ ((rl >> 1) & 3)) * 4));
          float4 o;
          o.x = fmaf(a.x + b4.x, rs, xin[it].x); o.y = fmaf(a.y + b4.y, rs, xin[it].y);
          o.z = fmaf(a.z + b4.z, rs, xin[it].z); o.w = fmaf(a.w + b4.w, rs, xin[it].w);
          *reinterpret_cast<float4*>(xt + (long)rl * D + c * 16 + c4 * 4) = o;
          if (LNF) {
            sum[it] += (o.x + o.y) + (o.z + o.w); sq[it] += fmaf(o.x, o.x, o.y * o.y) + fmaf(o.z, o.z, o.w * o.w);
            *reinterpret_cast<float4*>(xs + rl * D + (((c * 4 + c4) ^ xs_key(rl)) * 4)) = o;
          }
          if (!LNF && ct) {
            __nv_bfloat162 h0 = __floats2bfloat162_rn(o.x, o.y), h1 = __floats2bfloat162_rn(o.z, o.w);
            *reinterpret_cast<uint2*>(ct + (long)rl * D + c * 16 + c4 * 4) = make_uint2(*reinterpret_cast<uint32_t*>(&h0), *reinterpret_cast<uint32_t*>(&h1));
          }
        }
        if constexpr (!XS) {
#pragma unroll
          for (int it = 0; it < 4; ++it) xin[it] = xnx[it];
        }
        __syncwarp();
      }
      if (LNF) {
        // LayerNorm of the new rows for the next block: the four lanes of a row hold its partial sums; the second pass
        // reads the rows back from the warp's own shared-memory tile
        const float* gam = ep.ln_gamma + (long)g * D;
        const float* bet = ep.ln_beta + (long)g * D;
        float mean[4], rstd[4];
#pragma unroll
        for (int it = 0; it < 4; ++it) {
          float s1 = sum[it], s2 = sq[it];
          s1 += __shfl_xor_sync(0xffffffffu, s1, 1); s2 += __shfl_xor_sync(0xffffffffu, s2, 1);
          s1 += __shfl_xor_sync(0xffffffffu, s1, 2); s2 += __shfl_xor_sync(0xffffffffu, s2, 2);
          mean[it] = s1 * (1.0f / D);
          rstd[it] = rsqrtf(fmaxf(s2 * (1.0f / D) - mean[it] * mean[it], 0.f) + ep.ln_eps);
        }
        __nv_bfloat16* lt = ep.ln_out + (long)g * ep.ln_gs + (long)(m0 + q * 32) * D;
#pragma unroll 2
        for (int c = 0; c < D / 16; ++c) {
          const float4 g4 = __ldg(reinterpret_cast<const float4*>(gam + c * 16 + c4 * 4));
          const float4 t4 = __ldg(reinterpret_cast<const float4*>(bet + c * 16 + c4 * 4));
#pragma unroll
          for (int it = 0; it < 4; ++it) {
            const int rl = it * 8 + rsub;
            const float4 xv = *reinterpret_cast<const float4*>(xs + rl * D + (((c * 4 + c4) ^ xs_key(rl)) * 4));
            __nv_bfloat162 h0 = __floats2bfloat162_rn((xv.x - mean[it]) * rstd[it] * g4.x + t4.x, (xv.y - mean[it]) * rstd[it] * g4.y + t4.y);
            __nv_bfloat162 h1 = __floats2bfloat162_rn((xv.z - mean[it]) * rstd[it] * g4.z + t4.z, (xv.w - mean[it]) * rstd[it] * g4.w + t4.w);
            *reinterpret_cast<uint2*>(lt + (long)rl * D + c * 16 + c4 * 4) = make_uint2(*reinterpret_cast<uint32_t*>(&h0), *reinterpret_cast<uint32_t*>(&h1));
          }
        }
        __syncwarp();
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

int map3(CUtensorMap* map, const void* ptr, long K, long rows, long groups, long ld, long gstride, int box_rows) {
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) || (ld % 8) || (gstride % 8)) { mrnb_set_error("mlp_tc: misaligned operand"); return MRNB_ERR_ARG; }
  cuuint64_t dims[3] = {(cuuint64_t)K, (cuuint64_t)rows, (cuuint64_t)groups};
  cuuint64_t strides[2] = {(cuuint64_t)ld * 2, (cuuint64_t)gstride * 2};
  cuuint32_t box[3] = {64, (cuuint32_t)box_rows, 1}, es[3] = {1, 1, 1};
  return encode_tensor_map("mlp_tc", map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, ptr, dims, strides, box, es, CU_TENSOR_MAP_SWIZZLE_128B);
}

template <int D, bool LNF>
int launch_mlp(const MrnbMlp& p, cudaStream_t st) {
  using K = Cfg<D>;
  CUtensorMap tmA, tmW1, tmW2;
  MRNB_TRY(map3(&tmA, p.A, D, p.M, p.groups, D, (long)p.M * D, BM));
  MRNB_TRY(map3(&tmW1, p.W1, D, 4 * D, p.groups, D, (long)4 * D * D, HC));
  MRNB_TRY(map3(&tmW2, p.W2, 4 * D, D, p.groups, 4 * D, (long)4 * D * D, K::W2ROWS));
  MlpParams ep{};
  ep.b1 = p.b1; ep.b2 = p.b2; ep.b_gs1 = 4 * D; ep.b_gs2 = D;
  ep.x = p.x; ep.x_gs = p.x_gstride;
  ep.rowscale = p.rowscale; ep.rows_per_scale = p.rows_per_scale > 0 ? p.rows_per_scale : 1; ep.rowscale_gs = p.rowscale_gstride;
  ep.cast_out = (__nv_bfloat16*)p.cast_out;
  ep.ln_out = (__nv_bfloat16*)p.ln_out; ep.ln_gs = (long)p.M * D; ep.ln_gamma = p.ln_gamma; ep.ln_beta = p.ln_beta; ep.ln_eps = p.ln_eps;
  ep.m_tiles = p.M / BM; ep.total_tiles = ep.m_tiles * p.groups;
  ep.trace = (unsigned long long*)p.trace;
  static bool attr = false;
  static int num_sms = 148;
  if (!attr) {
    cudaFuncSetAttribute(mlp_tc_kernel<D, LNF>, cudaFuncAttributeMaxDynamicSharedMemorySize, K::SMEM);
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
    attr = true;
  }
  const int grid = ep.total_tiles < num_sms ? ep.total_tiles : num_sms;
  mlp_tc_kernel<D, LNF><<<grid, NTHREADS, K::SMEM, st>>>(tmA, tmW1, tmW2, ep);
  MRNB_CHECK_LAUNCH("mlp_tc_kernel");
  return MRNB_OK;
}

}  // namespace

int mrnb_mlp_tc(const MrnbMlp& p, cudaStream_t st) {
  MRNB_CHECK_ARG(p.A && p.W1 && p.W2 && p.b1 && p.b2 && p.x && p.M > 0 && p.groups > 0, "mlp_tc: null/empty argument");
  MRNB_CHECK_ARG(p.M % BM == 0 && (p.D == 64 || p.D == 128 || p.D == 256), "mlp_tc: need M %% 128 == 0 and D in {64,128,256}");
  MRNB_CHECK_ARG(!p.rowscale || p.rows_per_scale % BM == 0, "mlp_tc: DropPath scale must be uniform per 128-row tile");
  MRNB_CHECK_ARG(!p.ln_out || (p.D <= 128 && p.ln_gamma && p.ln_beta), "mlp_tc: fused LayerNorm needs D <= 128");
  MRNB_CHECK_ARG(!(p.ln_out && p.cast_out), "mlp_tc: cast_out and ln_out are exclusive");
  MRNB_CHECK_ARG(p.x_gstride % 4 == 0, "mlp_tc: misaligned residual stream");
  const double M = (double)p.M * p.groups;
  MrnbProfScope prof(MRNB_PROF_MLP, st, 16.0 * M * p.D * p.D, M * p.D * (2.0 + 8.0 + (p.ln_out ? 2.0 : 0.0)));
  switch (p.D) {
    case 64: return p.ln_out ? launch_mlp<64, true>(p, st) : launch_mlp<64, false>(p, st);
    case 128: return p.ln_out ? launch_mlp<128, true>(p, st) : launch_mlp<128, false>(p, st);
    default: return launch_mlp<256, false>(p, st);
  }
}

// C-ABI test entry: one group.  x [M,D] fp32 is updated in place; ln_out (bf16 [M,D]) optional.
static void* g_mlp_trace = nullptr;
extern "C" void mrnb_mlp_set_trace(void* device_buffer) { g_mlp_trace = device_buffer; }

extern "C" int mrnb_mlp_bf16(const void* A, const void* W1, const float* b1, const void* W2, const float* b2, float* x,
                             const float* rowscale, int rows_per_scale, void* ln_out, const float* ln_gamma,
                             const float* ln_beta, float ln_eps, int M, int D, cudaStream_t stream) {
  MrnbMlp p{};
  p.trace = g_mlp_trace;
  p.A = A; p.W1 = W1; p.W2 = W2; p.b1 = b1; p.b2 = b2; p.x = x; p.x_gstride = (long)M * D;
  p.rowscale = rowscale; p.rows_per_scale = rows_per_scale;
  p.ln_out = ln_out; p.ln_gamma = ln_gamma; p.ln_beta = ln_beta; p.ln_eps = ln_eps;
  p.M = M; p.D = D; p.groups = 1;
  return mrnb_mlp_tc(p, stream);
}
