// Fused SVTR mixer branch on the tensor cores (bf16 mode): one persistent kernel per Block does
//
//     q,k,v = A Wqkv^T + b      (A = LN1(x), bf16)        modules/svtr.py:138-141   (q scaled by head_dim^-0.5, :142)
//     P     = softmax(q k^T [+ Local 7x11 window])        modules/svtr.py:143-146   (mask :116-128 as index bounds)
//     x    <- x + rs * ( (P v) Wproj^T + b_proj )         modules/svtr.py:148-151, :201-203 (DropPath :7-22)
//     ln    = LN2(x)                      (D <= 128)      modules/svtr.py:203 (norm2 of the same Block)
//
// for every (expert, sample) unit.  q, k, v, the scores and the probabilities never reach HBM: per block the kernel
// reads A (bf16) and x (fp32) and writes x and LN2(x), instead of the three round trips (qkv GEMM -> attention ->
// proj GEMM) through a [M,3D] tensor.
//
// A unit = one sample of one expert = N = 32768 / D tokens (512 / 256 / 128), NT = N / 128 query tiles, D / 32 heads.
// TMEM (512 columns):
//     [0,256)   Y = proj accumulator of the whole unit (NT tiles x D columns), accumulated over heads by the MMA itself
//     [256,320) / [320,384)  S = q k^T of one (query tile, 64-key block), one per softmax stream
//     [384,416) / [416,448)  O = P v of the stream's query tile
//     [448,512) OVL: staging of the q|k / v parts of one 128-token tile (the non-OVL staging aliases the S / O columns)
// 512 threads in four warpgroups with their own register budgets (setmaxnreg): control (warp 0 TMA producer, warps 1 / 2
// MMA issuers of the two streams, warp 3 OVL q|k|v issuer), two softmax streams of four warps (one query row per
// thread), and a fourth warpgroup that is the Y epilogue (64-wide stage) or the q|k|v drain (OVL).
//   64-wide stage: A of the whole unit resident in smem (64 KiB); per head phase 1 = q|k|v of all tiles (MMA -> TMEM ->
//     all eight softmax warps -> bf16 swizzled smem), phase 2 = attention, stream s on query tiles s, s + 2, with S(p+1)
//     issued while the softmax of pair p runs; head output -> smem -> proj MMA into Y; the epilogue warpgroup adds bias,
//     DropPath scale and the fp32 residual, stores x in place and emits LN2 while the next unit is already running.
//   128-wide stage (MRNB_MIXER_OVL): q/k/v double buffered by head parity, A streamed one tile at a time; the q|k|v GEMM
//     and drain of head h+1 run under the attention of head h; each stream runs the Y epilogue of its own tile; the first
//     S of the next head is issued behind the last P V of the current one.
// Shared memory: A, q/k/v of one (OVL: two) head(s) for all tokens (3 x N x 64 B each), one probability / head-output
// tile per stream, the q|k|v and proj weights of the current head(s), epilogue staging.
#include "mixer_tc.h"
#include "sm100.cuh"
#include <stdlib.h>
#include <type_traits>

namespace {

#ifndef MRNB_MIXER_OVL
#define MRNB_MIXER_OVL 1
#endif
constexpr int HD = 32;
// Four warpgroups with re-balanced register budgets (setmaxnreg): WG0 = control (warp 0 TMA producer, warp 1 MMA issuer of
// stream 0 + phase 1, warp 2 MMA issuer of stream 1), WG1 / WG2 = softmax streams 0 / 1, WG3 = Y epilogue.
constexpr int EPI_WARPS = 8, NTHREADS = 512;
constexpr int REGS_CTRL = 80, REGS_SOFTMAX = 168, REGS_EPI = 96;       // 128 * (80 + 2 * 168 + 96) = 65536
// TMEM columns: Y accumulator; per-stream S (64 keys) and O (32 dims); phase-1 staging buffers alias the S / O columns
constexpr uint32_t Y_COL = 0, S0_COL = 256, S1_COL = 320, O0_COL = 384, O1_COL = 416, STG0_COL = 256, STG1_COL = 352;
constexpr uint32_t STGX_COL = 448;      // OVL: dedicated 64-column staging of the q|k (64) / v (32) parts of one 128-token tile

// named barrier 1 + q for the two partner warps (64 threads) of TMEM lane quarter q
__device__ __forceinline__ void pair_sync(int q) {
  switch (q) {
    case 0: asm volatile("bar.sync 1, 64;" ::: "memory"); break;
    case 1: asm volatile("bar.sync 2, 64;" ::: "memory"); break;
    case 2: asm volatile("bar.sync 3, 64;" ::: "memory"); break;
    default: asm volatile("bar.sync 4, 64;" ::: "memory"); break;
  }
}
template <int D>
struct MCfg {
  static constexpr int N = 32768 / D;                       // tokens per unit: 512 / 256 / 128
  static constexpr int NT = N / 128;                        // query tiles: 4 / 2 / 1
  static constexpr int KR = N / 64;                         // key blocks = rows of the 64-wide token grid: 8 / 4 / 2
  static constexpr int HEADS = D / HD;
  static constexpr int KB = D / 64;                         // k-blocks of the q|k|v GEMM
  static constexpr int A_BYTES = ((D == 128 && MRNB_MIXER_OVL) ? 128 : N) * D * 2;   // resident unit (64 KiB) or, OVL, one 128-token tile (32 KiB)
  static constexpr int HT_BYTES = 128 * HD * 2;             // one [128 x 32] bf16 head tile: 8 KiB
  // OVL (D = 128): the q|k|v GEMM + drain of head h + 1 overlaps the attention of head h.  q/k/v tiles are double buffered
  // by head parity, A is streamed one 128-token tile at a time (re-read per head from L2) instead of resident, a dedicated
  // thread issues the q|k|v MMAs into their own TMEM staging columns and the Y-epilogue warpgroup drains them.  (D = 64:
  // two q/k/v buffers of 96 KiB do not fit; D = 256 runs unfused.)
  static constexpr bool OVL = D == 128 && MRNB_MIXER_OVL;
  static constexpr int QKV1_BYTES = 3 * NT * HT_BYTES;      // q, k, v of one head for all tokens
  static constexpr int QKV_BYTES = (OVL ? 2 : 1) * QKV1_BYTES;
  static constexpr int P_TILE = 128 * 64 * 2;               // one stream's probability tile [128 q x 64 keys]: 16 KiB
  static constexpr int P_BYTES = 2 * P_TILE;
  static constexpr int WQ_KB_BYTES = 96 * 128;              // q|k|v rows of one head, one 64-wide k-block
  static constexpr int WQ_BYTES = KB * WQ_KB_BYTES;
  static constexpr int WP_BYTES = D * HD * 2;
  static constexpr int STG_BYTES = 4 * 2048;                // Y-epilogue staging: 32 rows x 16 fp32 per warp
  static constexpr int BIAS_BYTES = OVL ? 4 * 3 * D * 4 : 0; // OVL: q|k|v bias of the drained expert, one copy per drain warp
  static constexpr int SMEM = 1024 + A_BYTES + QKV_BYTES + P_BYTES + WQ_BYTES + 2 * WP_BYTES + STG_BYTES + BIAS_BYTES;
  static_assert(NT * D == 256, "Y accumulator spans 256 TMEM columns");
  static_assert(SMEM <= 227 * 1024, "shared memory budget");
};

struct MixParams {
  const float* bqkv; const float* bproj;
  float* x; long x_gs;
  const float* rowscale; long rs_gs;
  __nv_bfloat16* ln_out; const float* ln_gamma; const float* ln_beta; float ln_eps;
  int upg, total;                                           // units per group (expert), total units
  int dbg;                                                  // MRNB_MIXER_DBG bits (bottleneck experiments only; results are wrong)
  unsigned long long* trace;                                // optional debug timeline of CTA 0 (tools/mixer_trace.py): [16][256] globaltimer stamps
};

#define MIX_TRACE(slot_, idx_)                                                                     \
  do {                                                                                             \
    if (ep.trace && blockIdx.x == 0 && (idx_) < 256) {                                             \
      unsigned long long now__;                                                                    \
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now__));                                    \
      ep.trace[(slot_) * 256 + (idx_)] = now__;                                                    \
    }                                                                                              \
  } while (0)

// Y epilogue of ONE 128-token query tile for the 32 rows of the calling warp (TMEM lane quarter q):
//   x <- x + rs * (Y + b_proj) in place  [+ LayerNorm 2 -> ln_out (bf16)]
// 16 accumulator columns of the warp's 32 rows are transposed through a 2 KiB staging tile `stg` (row-major, 16-byte
// pieces XOR-swizzled by row) so that global accesses are 64-byte row segments: lane = (row in a group of 8, float4 of
// the 16).  The residual rows of the next step are prefetched.  `release` (optional mbarrier) is arrived on by lane 0
// once the tile's Y columns are out of TMEM.  Called by the Y-epilogue warpgroup (one warp per quarter, every tile) or,
// OVL, by the softmax warps of the stream that owns the tile.
template <int D, bool LNF, int LNU = 2>
__device__ __forceinline__ void y_tile_epilogue(const MixParams& ep, int e, long unit, int qt, int q, int lane, uint32_t y_addr,
                                                float* xt, float rs, float* stg, uint64_t* release) {
  const int rsub = lane >> 2, c4 = lane & 3;
  const float* bpj = ep.bproj + (long)e * D;
  float sum[4] = {0.f, 0.f, 0.f, 0.f}, sq[4] = {0.f, 0.f, 0.f, 0.f};
  float4 xin[4], xnx[4];                                 // residual rows of this / the next 16-column step
  if (!(ep.dbg & 2)) {
#pragma unroll
    for (int it = 0; it < 4; ++it) xin[it] = *reinterpret_cast<const float4*>(xt + (long)(it * 8 + rsub) * D + c4 * 4);
  }
#pragma unroll 1
  for (int c = 0; c < D / 16; ++c) {
    if (!(ep.dbg & 2) && c + 1 < D / 16) {
#pragma unroll
      for (int it = 0; it < 4; ++it) xnx[it] = *reinterpret_cast<const float4*>(xt + (long)(it * 8 + rsub) * D + (c + 1) * 16 + c4 * 4);
    }
    uint32_t v[16];
    tmem_ld16(y_addr + (uint32_t)(c * 16), v);
    if (c == D / 16 - 1) {
      tc_fence_before();
      __syncwarp();
      if (release && lane == 0) mbar_arrive(release);    // this tile's accumulator columns are drained
    }
    if (ep.dbg & 2) continue;
#pragma unroll
    for (int pc = 0; pc < 4; ++pc)
      *reinterpret_cast<float4*>(stg + lane * 16 + ((pc ^ ((lane >> 1) & 3)) * 4)) =
          make_float4(__uint_as_float(v[4 * pc]), __uint_as_float(v[4 * pc + 1]), __uint_as_float(v[4 * pc + 2]), __uint_as_float(v[4 * pc + 3]));
    __syncwarp();
    const float4 b4 = __ldg(reinterpret_cast<const float4*>(bpj + c * 16 + c4 * 4));
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      const int rl = it * 8 + rsub;
      const float4 a = *reinterpret_cast<const float4*>(stg + rl * 16 + ((c4 ^ ((rl >> 1) & 3)) * 4));
      float4 o;
      o.x = fmaf(a.x + b4.x, rs, xin[it].x); o.y = fmaf(a.y + b4.y, rs, xin[it].y);
      o.z = fmaf(a.z + b4.z, rs, xin[it].z); o.w = fmaf(a.w + b4.w, rs, xin[it].w);
      *reinterpret_cast<float4*>(xt + (long)rl * D + c * 16 + c4 * 4) = o;
      if (LNF) { sum[it] += (o.x + o.y) + (o.z + o.w); sq[it] += fmaf(o.x, o.x, o.y * o.y) + fmaf(o.z, o.z, o.w * o.w); }
    }
#pragma unroll
    for (int it = 0; it < 4; ++it) xin[it] = xnx[it];
    __syncwarp();
  }
  if (LNF && !(ep.dbg & (2 | 32))) {
    // row statistics: the four lanes of a row hold its partial sums; second pass over the rows just written
    // (the warp's own stores: L1 / L2 hits) -> LayerNorm 2 in bf16
    const float* gam = ep.ln_gamma + (long)e * D;
    const float* bet = ep.ln_beta + (long)e * D;
    float mean[4], rstd[4];
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      float s1 = sum[it], s2 = sq[it];
      s1 += __shfl_xor_sync(0xffffffffu, s1, 1); s2 += __shfl_xor_sync(0xffffffffu, s2, 1);
      s1 += __shfl_xor_sync(0xffffffffu, s1, 2); s2 += __shfl_xor_sync(0xffffffffu, s2, 2);
      mean[it] = s1 * (1.0f / D);
      rstd[it] = rsqrtf(fmaxf(s2 * (1.0f / D) - mean[it] * mean[it], 0.f) + ep.ln_eps);
    }
    __nv_bfloat16* lt = ep.ln_out + ((long)unit * (32768 / D) + qt * 128 + q * 32) * D;
    // LNU steps unrolled: LNU x 4 independent 16-byte loads of the just-written rows in flight (they come back from L2)
#pragma unroll LNU
    for (int c = 0; c < D / 16; ++c) {
      const float4 g4 = __ldg(reinterpret_cast<const float4*>(gam + c * 16 + c4 * 4));
      const float4 t4 = __ldg(reinterpret_cast<const float4*>(bet + c * 16 + c4 * 4));
#pragma unroll
      for (int it = 0; it < 4; ++it) {
        const int rl = it * 8 + rsub;
        const float4 xv = *reinterpret_cast<const float4*>(xt + (long)rl * D + c * 16 + c4 * 4);
        *reinterpret_cast<uint2*>(lt + (long)rl * D + c * 16 + c4 * 4) = make_uint2(
            pack_bf16((xv.x - mean[it]) * rstd[it] * g4.x + t4.x, (xv.y - mean[it]) * rstd[it] * g4.y + t4.y),
            pack_bf16((xv.z - mean[it]) * rstd[it] * g4.z + t4.z, (xv.w - mean[it]) * rstd[it] * g4.w + t4.w));
      }
    }
  }
}

// The Y epilogue of the OVL variant, run by the softmax warps of the stream that owns the tile (168 registers): each
// warp's 32 rows in passes of RG x 8 rows.  The updated residual values of a pass stay in registers (RG x 32 per thread)
// between the x update and LayerNorm 2 -- no second pass over rows just stored -- and ALL residual loads of a pass are
// in flight at once (the first pass' before `wait_bar`, the barrier that says Y is complete, is waited for).  The
// accumulator columns are read once per pass (tcgen05.ld delivers all 32 lanes; the other rows are dropped); `stg` is
// 4 KiB: two alternating 32 x 16 fp32 staging tiles, one __syncwarp per step (DBUF = false: one 2 KiB tile, two).
// `release` (optional) is arrived on once the last pass has left TMEM.  The 64-wide stage runs it from the Y-epilogue
// warpgroup (RG = 2: 32 registers of rows), where the second pass of `y_tile_epilogue` cost 43 of the 464 us a launch takes.
template <int D, bool LNF, int RG, bool DBUF = true>
__device__ __forceinline__ void y_tile_epilogue_regs(const MixParams& ep, int e, long unit, int qt, int q, int lane, uint32_t y_addr,
                                                     float* xt, float rs, float* stg, int g_begin, int n_pass,
                                                     uint64_t* wait_bar, uint32_t wait_parity, uint64_t* release) {
  constexpr int NS = D / 16;
  const int rsub = lane >> 2, c4 = lane & 3;
  const float* bpj = ep.bproj + (long)e * D;
  const float* gam = ep.ln_gamma + (long)e * D;
  const float* bet = ep.ln_beta + (long)e * D;
  __nv_bfloat16* lt = ep.ln_out + ((long)unit * (32768 / D) + qt * 128 + q * 32) * D;
#pragma unroll 1
  for (int ps = 0; ps < n_pass; ++ps) {
    const int g0 = g_begin + ps * RG;                          // first 8-row group of this pass
    float4 xo[NS][RG];
    float* xr = xt + (long)(g0 * 8 + rsub) * D + c4 * 4;
#pragma unroll
    for (int c = 0; c < NS; ++c)
#pragma unroll
      for (int g2 = 0; g2 < RG; ++g2) xo[c][g2] = *reinterpret_cast<const float4*>(xr + g2 * 8 * D + c * 16);
    if (ps == 0 && wait_bar) { mbar_wait(wait_bar, wait_parity); tc_fence_after(); }
    float sum[RG], sq[RG];
#pragma unroll
    for (int g2 = 0; g2 < RG; ++g2) { sum[g2] = 0.f; sq[g2] = 0.f; }
#pragma unroll
    for (int c = 0; c < NS; ++c) {
      uint32_t v[16];
      tmem_ld16(y_addr + (uint32_t)(c * 16), v);
      if (c == NS - 1 && ps == n_pass - 1 && release) {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(release);
      }
      float* sb = stg + (DBUF ? (c & 1) * 512 : 0);
      if (!DBUF && c > 0) __syncwarp();                        // single staging tile: the previous step's reads are done
#pragma unroll
      for (int pc = 0; pc < 4; ++pc)
        *reinterpret_cast<float4*>(sb + lane * 16 + ((pc ^ ((lane >> 1) & 3)) * 4)) =
            make_float4(__uint_as_float(v[4 * pc]), __uint_as_float(v[4 * pc + 1]), __uint_as_float(v[4 * pc + 2]), __uint_as_float(v[4 * pc + 3]));
      __syncwarp();
      const float4 b4 = __ldg(reinterpret_cast<const float4*>(bpj + c * 16 + c4 * 4));
#pragma unroll
      for (int g2 = 0; g2 < RG; ++g2) {
        const int rl = (g0 + g2) * 8 + rsub;
        const float4 a = *reinterpret_cast<const float4*>(sb + rl * 16 + ((c4 ^ ((rl >> 1) & 3)) * 4));
        float4 o = xo[c][g2];
        o.x = fmaf(a.x + b4.x, rs, o.x); o.y = fmaf(a.y + b4.y, rs, o.y);
        o.z = fmaf(a.z + b4.z, rs, o.z); o.w = fmaf(a.w + b4.w, rs, o.w);
        *reinterpret_cast<float4*>(xr + g2 * 8 * D + c * 16) = o;
        xo[c][g2] = o;
        if (LNF) { sum[g2] += (o.x + o.y) + (o.z + o.w); sq[g2] += fmaf(o.x, o.x, o.y * o.y) + fmaf(o.z, o.z, o.w * o.w); }
      }
    }
    if (LNF) {
      float mean[RG], rstd[RG];
#pragma unroll
      for (int g2 = 0; g2 < RG; ++g2) {
        float s1 = sum[g2], s2 = sq[g2];
        s1 += __shfl_xor_sync(0xffffffffu, s1, 1); s2 += __shfl_xor_sync(0xffffffffu, s2, 1);
        s1 += __shfl_xor_sync(0xffffffffu, s1, 2); s2 += __shfl_xor_sync(0xffffffffu, s2, 2);
        mean[g2] = s1 * (1.0f / D);
        rstd[g2] = rsqrtf(fmaxf(s2 * (1.0f / D) - mean[g2] * mean[g2], 0.f) + ep.ln_eps);
      }
      __nv_bfloat16* lr = lt + (long)(g0 * 8 + rsub) * D + c4 * 4;
#pragma unroll
      for (int c = 0; c < NS; ++c) {
        const float4 g4 = __ldg(reinterpret_cast<const float4*>(gam + c * 16 + c4 * 4));
        const float4 t4 = __ldg(reinterpret_cast<const float4*>(bet + c * 16 + c4 * 4));
#pragma unroll
        for (int g2 = 0; g2 < RG; ++g2) {
          const float4 xv = xo[c][g2];
          *reinterpret_cast<uint2*>(lr + g2 * 8 * D + c * 16) = make_uint2(
              pack_bf16((xv.x - mean[g2]) * rstd[g2] * g4.x + t4.x, (xv.y - mean[g2]) * rstd[g2] * g4.y + t4.y),
              pack_bf16((xv.z - mean[g2]) * rstd[g2] * g4.z + t4.z, (xv.w - mean[g2]) * rstd[g2] * g4.w + t4.w));
        }
      }
    }
    __syncwarp();
  }
}

template <int D, bool LOCAL, bool LNF>
__global__ void __launch_bounds__(NTHREADS, 1)
mixer_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmWq,
                const __grid_constant__ CUtensorMap tmWp, const MixParams ep) {
  using K = MCfg<D>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + align_smem_1024_offset(smem_raw);
  uint8_t* sA = smem;
  uint8_t* sQ = sA + K::A_BYTES;                            // [N rows x 64 B]; then sK, sV
  uint8_t* sK = sQ + K::NT * K::HT_BYTES;
  uint8_t* sV = sK + K::NT * K::HT_BYTES;
  uint8_t* sP = sQ + K::QKV_BYTES;                          // two streams x 16 KiB (also: head-output tile, epilogue staging)
  uint8_t* sWq = sP + K::P_BYTES;
  uint8_t* sWp = sWq + K::WQ_BYTES;
  uint8_t* sStg = sWp + 2 * K::WP_BYTES;
  float* sBias = reinterpret_cast<float*>(sStg + K::STG_BYTES);   // OVL: [4 drain warps][3 * D]
  __shared__ __align__(8) uint64_t a_full, a_empty, wq_full, wq_empty, wp_full[2], wp_empty[2], stg_full[2], stg_empty[2], qkv_ready,
      s_full[2], s_empty[2], p_full[2], o_full[2], so_full[2], so_empty[2], y_full, y_empty[4], st1_done, qkvr[2], qkvf[2], yd[2];
  __shared__ uint32_t tmem_base_sh;
  __shared__ float ln_part[2][4][2][32];

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int total = ep.total, upg = ep.upg;

  if (threadIdx.x == 0) {
    mbar_init(&a_full, 1); mbar_init(&a_empty, 1); mbar_init(&wq_full, 1); mbar_init(&wq_empty, 1);
    for (int b = 0; b < 2; ++b) {
      mbar_init(&wp_full[b], 1); mbar_init(&wp_empty[b], 2);
      mbar_init(&stg_full[b], 1); mbar_init(&stg_empty[b], K::OVL ? 4 : EPI_WARPS);
      mbar_init(&qkvr[b], 128); mbar_init(&qkvf[b], 2); mbar_init(&yd[b], 1);
      mbar_init(&s_full[b], 1); mbar_init(&s_empty[b], 128); mbar_init(&p_full[b], 128); mbar_init(&o_full[b], 1);
      mbar_init(&so_full[b], 128); mbar_init(&so_empty[b], 1);
    }
    mbar_init(&qkv_ready, EPI_WARPS * 32); mbar_init(&y_full, 2); mbar_init(&st1_done, 1);
    for (int b = 0; b < 4; ++b) mbar_init(&y_empty[b], 4);
    fence_mbarrier_init();
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmWq);
    prefetch_tmap(&tmWp);
  }
  if (warp == 1) tmem_alloc(&tmem_base_sh, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_sh;

  // Key blocks are single rows of the 64-wide token grid.  Query tile qt holds grid rows 2qt and 2qt+1; the Local window
  // spans |dh| <= 3 rows, so it visits rows 2qt-3 .. 2qt+4 (clipped); the Global mixer visits every row.
  auto kr_lo = [](int qt) { return LOCAL ? (2 * qt - 3 > 0 ? 2 * qt - 3 : 0) : 0; };
  auto kr_hi = [](int qt) { return LOCAL ? (2 * qt + 5 < K::KR ? 2 * qt + 5 : K::KR) : K::KR; };

  if (warp < 4) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_CTRL));
  if (warp == 0) {
    // ============================== TMA producer ==============================
    if (lane == 0) {
      if constexpr (K::OVL) {
        // per head: Wq_h, Wp_h, then the A tiles of the unit one at a time (consumed by the q|k|v issuer, warp 3)
        uint32_t hc = 0, tc = 0;
        for (int u = blockIdx.x; u < total; u += gridDim.x) {
          const int e = u / upg;
          for (int h = 0; h < K::HEADS; ++h, ++hc) {
            mbar_wait(&wq_empty, (hc & 1u) ^ 1u);
            mbar_expect_tx(&wq_full, K::WQ_BYTES);
            for (int kb = 0; kb < K::KB; ++kb)
              for (int part = 0; part < 3; ++part)
                tma_load_3d(sWq + kb * K::WQ_KB_BYTES + part * 4096, &tmWq, &wq_full, kb * 64, part * D + h * HD, e);
            const int buf = hc & 1u;
            mbar_wait(&wp_empty[buf], ((hc >> 1) & 1u) ^ 1u);
            mbar_expect_tx(&wp_full[buf], K::WP_BYTES);
            tma_load_3d(sWp + buf * K::WP_BYTES, &tmWp, &wp_full[buf], h * HD, 0, e);
            for (int mt = 0; mt < K::NT; ++mt, ++tc) {
              mbar_wait(&a_empty, (tc & 1u) ^ 1u);
              mbar_expect_tx(&a_full, K::A_BYTES);
              for (int kb = 0; kb < K::KB; ++kb) tma_load_3d(sA + kb * 16384, &tmA, &a_full, kb * 64, mt * 128, u);
            }
          }
        }
      } else {
      uint32_t hc = 0;
      int i = 0;
      for (int u = blockIdx.x; u < total; u += gridDim.x, ++i) {
        const int e = u / upg;
        mbar_wait(&a_empty, ((uint32_t)i & 1u) ^ 1u);
        mbar_expect_tx(&a_full, K::A_BYTES);
        for (int mt = 0; mt < K::NT; ++mt)
          for (int kb = 0; kb < K::KB; ++kb) tma_load_3d(sA + (mt * K::KB + kb) * 16384, &tmA, &a_full, kb * 64, mt * 128, u);
        for (int h = 0; h < K::HEADS; ++h, ++hc) {
          mbar_wait(&wq_empty, (hc & 1u) ^ 1u);
          mbar_expect_tx(&wq_full, K::WQ_BYTES);
          for (int kb = 0; kb < K::KB; ++kb)
            for (int part = 0; part < 3; ++part)
              tma_load_3d(sWq + kb * K::WQ_KB_BYTES + part * 4096, &tmWq, &wq_full, kb * 64, part * D + h * HD, e);
          const int buf = hc & 1u;
          mbar_wait(&wp_empty[buf], ((hc >> 1) & 1u) ^ 1u);
          mbar_expect_tx(&wp_full[buf], K::WP_BYTES);
          tma_load_3d(sWp + buf * K::WP_BYTES, &tmWp, &wp_full[buf], h * HD, 0, e);
        }
      }
      }
    }
  } else if (warp == 3) {
    // ============================== q|k|v MMA issuer (OVL) ==============================
    // Runs ahead of the attention: per head and 128-token tile two parts -- q|k (N = 64) and v (N = 32) -- into the
    // dedicated staging columns; the Y-epilogue warpgroup drains each part into the q/k/v buffer of the head's parity.
    if constexpr (K::OVL) {
      if (lane == 0) {
        constexpr uint32_t idesc_qk = umma_idesc(UMMA_BF16, 128, 64), idesc_v = umma_idesc(UMMA_BF16, 128, 32);
        uint32_t hc = 0, tc = 0, pc = 0;
        for (int u = blockIdx.x; u < total; u += gridDim.x) {
          for (int h = 0; h < K::HEADS; ++h, ++hc) {
            mbar_wait(&wq_full, hc & 1u);
            tc_fence_after();
            for (int mt = 0; mt < K::NT; ++mt, ++tc) {
              mbar_wait(&a_full, tc & 1u);
              tc_fence_after();
#pragma unroll
              for (int part = 0; part < 2; ++part, ++pc) {
                mbar_wait(&stg_empty[0], (pc & 1u) ^ 1u);
                tc_fence_after();
                for (int kb = 0; kb < K::KB; ++kb) {
                  const uint64_t ad = umma_desc_k128(smem_u32(sA + kb * 16384));
                  const uint64_t bd = umma_desc_k128(smem_u32(sWq + kb * K::WQ_KB_BYTES + part * 8192));
#pragma unroll
                  for (int k = 0; k < 4; ++k)
                    umma_bf16(tmem_base + STGX_COL, ad + (uint64_t)(k * 2), bd + (uint64_t)(k * 2), part ? idesc_v : idesc_qk, (kb | k) != 0);
                }
                umma_commit(&stg_full[0]);
              }
              umma_commit(&a_empty);                         // this A tile is free once its q|k and v MMAs retire
            }
            umma_commit(&wq_empty);
          }
        }
      }
    }
  } else if (warp == 1 || warp == 2) {
    // ============================== MMA issuers ==============================
    // warp 1: phase 1 (q|k|v tiles) + softmax stream 0; warp 2: softmax stream 1.  Each stream has its own issuing
    // thread, so every dependency edge is a hardware-sleeping mbarrier wait (no polling between the streams).
    if (lane == 0) {
      const int s = warp == 1 ? 0 : 1;
      constexpr uint32_t idesc_qkv = umma_idesc(UMMA_BF16, 128, 96), idesc_s = umma_idesc(UMMA_BF16, 128, 64);
      constexpr uint32_t idesc_o = umma_idesc(UMMA_BF16, 128, HD, false, true), idesc_y = umma_idesc(UMMA_BF16, 128, D);
      const uint32_t s_col = s ? S1_COL : S0_COL, o_col = s ? O1_COL : O0_COL;
      uint32_t hc = 0, mc = 0, pc = 0, qc = 0;
      bool s_early = false;                                    // OVL: the first S of the coming head is already issued
      int i = 0;
      for (int u = blockIdx.x; u < total; u += gridDim.x, ++i) {
        if (!K::OVL && s == 0) { mbar_wait(&a_full, (uint32_t)i & 1u); tc_fence_after(); }
        for (int h = 0; h < K::HEADS; ++h, ++hc) {
          if (!K::OVL && s == 0) {
            // ---- phase 1: q|k|v of this head for every 128-token tile -> staging columns (two buffers over the S / O
            // columns of both streams: stream 1 must have retired the previous head first)
            mbar_wait(&wq_full, hc & 1u);
            mbar_wait(&st1_done, (hc & 1u) ^ 1u);
            tc_fence_after();
            for (int mt = 0; mt < K::NT; ++mt, ++mc) {
              const uint32_t sb = mc & 1u, stg_col = sb ? STG1_COL : STG0_COL;
              mbar_wait(&stg_empty[sb], ((mc >> 1) & 1u) ^ 1u);
              tc_fence_after();
              for (int kb = 0; kb < K::KB; ++kb) {
                const uint64_t ad = umma_desc_k128(smem_u32(sA + (mt * K::KB + kb) * 16384));
                const uint64_t bd = umma_desc_k128(smem_u32(sWq + kb * K::WQ_KB_BYTES));
#pragma unroll
                for (int k = 0; k < 4; ++k) umma_bf16(tmem_base + stg_col, ad + (uint64_t)(k * 2), bd + (uint64_t)(k * 2), idesc_qkv, (kb | k) != 0);
              }
              umma_commit(&stg_full[sb]);
            }
            umma_commit(&wq_empty);                          // weights of this head's q|k|v are free once these MMAs retire
            if (h == K::HEADS - 1) umma_commit(&a_empty);    // ... and so is A after the last head
          }
          // ---- phase 2: this stream's query tiles s, s+2, ..
          const int buf = hc & 1u;
          if constexpr (K::OVL) { if (!s_early) mbar_wait(&qkvr[buf], (hc >> 1) & 1u); }   // q/k/v of this head drained into buffer hc % 2
          else mbar_wait(&qkv_ready, hc & 1u);
          mbar_wait(&wp_full[buf], (hc >> 1) & 1u);
          tc_fence_after();
          uint8_t* const sQh = sQ + (K::OVL ? buf * K::QKV1_BYTES : 0);
          uint8_t* const sKh = sK + (K::OVL ? buf * K::QKV1_BYTES : 0);
          uint8_t* const sVh = sV + (K::OVL ? buf * K::QKV1_BYTES : 0);
          auto issue_s_from = [&](const uint8_t* q_, const uint8_t* k_, int qt, int kr) {
            const uint64_t qd = umma_smem_desc(smem_u32(q_ + qt * K::HT_BYTES), 16, 512, UMMA_SWIZZLE_64B);
            const uint64_t kd = umma_smem_desc(smem_u32(k_ + kr * 4096), 16, 512, UMMA_SWIZZLE_64B);
#pragma unroll
            for (int k = 0; k < HD / 16; ++k) umma_bf16(tmem_base + s_col, qd + (uint64_t)(k * 2), kd + (uint64_t)(k * 2), idesc_s, k);
            umma_commit(&s_full[s]);
          };
          auto issue_s = [&](int qt, int kr) { issue_s_from(sQh, sKh, qt, kr); };
          if (s < K::NT) {
            int qt = s, kr = kr_lo(s);
            if (!s_early) issue_s(qt, kr);
            s_early = false;
            while (true) {
              int nqt = qt, nkr = kr + 1;
              if (nkr >= kr_hi(qt)) { nqt = qt + 2; nkr = nqt < K::NT ? kr_lo(nqt) : 0; }
              const bool has_next = nqt < K::NT, last_of_tile = nqt != qt, first_of_tile = kr == kr_lo(qt);
              if (s == 0) MIX_TRACE(0, pc);                    // MMA0: start of pair
              if (has_next) {
                mbar_wait(&s_empty[s], pc & 1u);             // the stream has pulled S of the current pair out of TMEM
                tc_fence_after();
                issue_s(nqt, nkr);
              }
              if (s == 0) MIX_TRACE(1, pc);                    // MMA0: S(next) issued, waiting for P
              mbar_wait(&p_full[s], pc & 1u);
              tc_fence_after();
              if (s == 0) MIX_TRACE(2, pc);                    // MMA0: P available
              {
                // O (+)= P V: the accumulator lives in TMEM for the whole query tile (the softmax warps rescale it in
                // place on the rare occasions the running reference maximum moves)
                const uint64_t pd = umma_desc_k128(smem_u32(sP + s * K::P_TILE));
                const uint64_t vd = umma_smem_desc(smem_u32(sVh + kr * 4096), 16, 512, UMMA_SWIZZLE_64B);
#pragma unroll
                for (int k = 0; k < 64 / 16; ++k)             // P: +32 B per 16 keys inside the 128 B row; V: +16 key rows of 64 B
                  umma_bf16(tmem_base + o_col, pd + (uint64_t)(k * 2), vd + (uint64_t)((k * 16 * 64) >> 4), idesc_o, (!first_of_tile) || k != 0);
                umma_commit(&o_full[s]);
              }
              if (s == 0) MIX_TRACE(3, pc);                    // MMA0: PV issued
              ++pc;
              if constexpr (K::OVL) {
                // last pair of the head (one tile per stream): if q/k/v of the NEXT head (possibly of the next unit) are
                // already drained, its first S is issued now, under the stream's O normalisation and this head's proj MMA
                // (never blocking: a late drain must not hold back the proj MMA the Y epilogue is waiting for)
                const bool more = !(h == K::HEADS - 1 && u + (int)gridDim.x >= total);
                const uint32_t nb = (hc + 1u) & 1u;
                if (!has_next && more && mbar_test(&qkvr[nb], ((hc + 1u) >> 1) & 1u)) {
                  mbar_wait(&s_empty[s], (pc - 1u) & 1u);    // the stream has pulled the last S out of TMEM
                  tc_fence_after();
                  issue_s_from(sQ + nb * K::QKV1_BYTES, sK + nb * K::QKV1_BYTES, s, kr_lo(s));
                  s_early = true;
                }
              }
              if (last_of_tile) {
                // the stream has normalised the head output of this query tile into its tile buffer:
                // Y[qt] (+)= O_h Wproj[:, h*32 : h*32+32]^T
                mbar_wait(&so_full[s], qc & 1u);
                tc_fence_after();
                // first head: the previous unit's epilogue must have drained THIS tile's Y columns (released tile by tile).
                // OVL: the stream's own softmax warps run that epilogue before they hand over this head output
                if (!K::OVL && h == 0) { mbar_wait(&y_empty[qt], ((uint32_t)i & 1u) ^ 1u); tc_fence_after(); }
                const uint64_t od = umma_smem_desc(smem_u32(sP + s * K::P_TILE), 16, 512, UMMA_SWIZZLE_64B);
                const uint64_t wd = umma_smem_desc(smem_u32(sWp + buf * K::WP_BYTES), 16, 512, UMMA_SWIZZLE_64B);
#pragma unroll
                for (int k = 0; k < HD / 16; ++k)
                  umma_bf16(tmem_base + Y_COL + (uint32_t)(qt * D), od + (uint64_t)(k * 2), wd + (uint64_t)(k * 2), idesc_y, (h | k) != 0);
                umma_commit(&so_empty[s]);
                if (K::OVL && h == K::HEADS - 1) umma_commit(&yd[s]);    // Y of this stream's tile is complete for the unit
                ++qc;
              }
              if (!has_next) break;
              qt = nqt; kr = nkr;
            }
          }
          umma_commit(&wp_empty[buf]);
          if (s == 1) umma_commit(&st1_done);
          if constexpr (K::OVL) umma_commit(&qkvf[buf]);      // this stream has retired the head: its q/k/v buffer may be refilled
        }
        if (!K::OVL) umma_commit(&y_full);
      }
    }
  } else if (warp >= 4 && warp < 12) {
    // ============================== softmax warps (phase 1 drain + phase 2) ==============================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(REGS_SOFTMAX));
    const int ew = warp - 4, q = warp & 3, ch = ew >> 2;       // ch = softmax stream (phase 2) / column half of the phase-1 drain
    const int r = q * 32 + lane;                               // row inside a 128-token tile == TMEM lane
    const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
    const int sw = (r >> 1) & 3;                               // 64B-swizzle XOR of this row's 16-byte chunks
    const float sl2 = 0.17677669529663688110f * 1.4426950408889634f;   // 32^-0.5 * log2(e), applied to the scores in the exp2 FFMA
    uint8_t* ptile = sP + ch * K::P_TILE;                      // this stream's probability / head-output tile
    // final-epilogue staging: exactly the 4 KiB of sP this warp itself writes P rows into (no cross-warp hazard)
    float* stg = reinterpret_cast<float*>(ptile + (size_t)q * 4096);
    const int p8 = lane & 7, rsel = lane >> 3;
    constexpr int OW = D / 2, NPASS = OW / 32;
    const uint32_t s_col = ch ? S1_COL : S0_COL, o_col = ch ? O1_COL : O0_COL;
    uint32_t hc = 0, mc = 0, pc = 0, qc = 0;
    int i = 0;
    for (int u = blockIdx.x; u < total; u += gridDim.x, ++i) {
      const int e = u / upg, b = u % upg;
      if constexpr (K::OVL) {
        // the residual rows of this stream's tile (64 KiB) start their trip from HBM to L2 now; they are needed by the
        // Y epilogue after the last head
        const char* xl2 = reinterpret_cast<const char*>(ep.x + (long)e * ep.x_gs + (long)b * K::N * D + (long)(ch * 128) * D);
#pragma unroll
        for (int k = 0; k < D / 32; ++k) asm volatile("prefetch.global.L2 [%0];" ::"l"(xl2 + (long)(k * 128 + q * 32 + lane) * 128));
      }
      for (int h = 0; h < K::HEADS; ++h, ++hc) {
        if constexpr (!K::OVL) {
        // ---- phase 1 (all eight warps): staging columns -> (+bias, q scaled) -> bf16 -> 64B-swizzled K-major head tiles
        float bias[3][16];
#pragma unroll
        for (int pi = 0; pi < 3; ++pi) {
          const int p = ch * 3 + pi;                           // 16-column piece: tensor p / 2 (q, k, v), half p % 2
          const float4* bp = reinterpret_cast<const float4*>(ep.bqkv + (long)e * 3 * D + (p >> 1) * D + h * HD + (p & 1) * 16);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float4 t = __ldg(bp + j);
            bias[pi][4 * j] = t.x; bias[pi][4 * j + 1] = t.y; bias[pi][4 * j + 2] = t.z; bias[pi][4 * j + 3] = t.w;
          }
        }
        for (int mt = 0; mt < K::NT; ++mt, ++mc) {
          const uint32_t sb = mc & 1u, stg_col = sb ? STG1_COL : STG0_COL;
          mbar_wait(&stg_full[sb], (mc >> 1) & 1u);
          tc_fence_after();
          uint32_t v[3][16];
#pragma unroll
          for (int pi = 0; pi < 3; ++pi) tmem_ld16(lane_addr + stg_col + (uint32_t)((ch * 3 + pi) * 16), v[pi]);
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&stg_empty[sb]);
#pragma unroll
          for (int pi = 0; pi < 3; ++pi) {
            const int p = ch * 3 + pi, t = p >> 1, half = p & 1;
            uint32_t pk[8];
#pragma unroll
            for (int j = 0; j < 8; ++j)
              pk[j] = pack_bf16(__uint_as_float(v[pi][2 * j]) + bias[pi][2 * j], __uint_as_float(v[pi][2 * j + 1]) + bias[pi][2 * j + 1]);
            uint8_t* row = (t == 0 ? sQ : (t == 1 ? sK : sV)) + mt * K::HT_BYTES + r * 64;
            *reinterpret_cast<uint4*>(row + (((half * 2) ^ sw) * 16)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
            *reinterpret_cast<uint4*>(row + (((half * 2 + 1) ^ sw) * 16)) = make_uint4(pk[4], pk[5], pk[6], pk[7]);
          }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        mbar_arrive(&qkv_ready);

        }
        // ---- phase 2: stream ch owns query tiles ch, ch+2, ..; one thread = one query row, one key block = 64 keys
        for (int qt = ch; qt < K::NT; qt += 2, ++qc, ++pc) {
          const int qh = 2 * qt + (r >> 6), qw = r & 63;       // grid row / column of this query
          float m = -INFINITY, l = 0.f;                        // running reference maximum (log2 units) / normaliser
          const int j0 = kr_lo(qt), j1 = kr_hi(qt);
          for (int kr = j0; kr < j1; ++kr) {
            if (kr > j0) ++pc;
            const bool tr = warp == 4 && lane == 0;
            if (tr) MIX_TRACE(4, pc);                          // softmax: start of pair (waiting for S)
            mbar_wait(&s_full[ch], pc & 1u);
            tc_fence_after();
            if (tr) MIX_TRACE(5, pc);                          // softmax: S ready
            // the 64 scores of this row go to registers once; TMEM is released at once so S of the next pair overlaps
            uint32_t sv[64];
            if (!(ep.dbg & 4)) {
              tmem_ld32(lane_addr + s_col, *reinterpret_cast<uint32_t(*)[32]>(&sv[0]));
              tmem_ld32(lane_addr + s_col + 32u, *reinterpret_cast<uint32_t(*)[32]>(&sv[32]));
            } else {
#pragma unroll
              for (int k2 = 0; k2 < 64; ++k2) sv[k2] = 0u;
            }
            tc_fence_before();
            mbar_arrive(&s_empty[ch]);
            if (tr) MIX_TRACE(6, pc);                          // softmax: S in registers
            // Local window: key column kw is visible from query column qw iff |kw - qw| <= 5, key row iff |kr - qh| <= 3
            uint32_t vmask[2] = {0xffffffffu, 0xffffffffu};
            if (LOCAL) {
              const int dh = kr - qh;
              const bool rowok = dh >= -3 && dh <= 3;
#pragma unroll
              for (int cc = 0; cc < 2; ++cc) {
                const int lo = qw - 5 - cc * 32, hi = qw + 5 - cc * 32;      // valid key columns of this chunk: [lo, hi]
                uint32_t mk = 0u;
                if (rowok && hi >= 0 && lo <= 31) {
                  const int l2 = lo < 0 ? 0 : lo, h2 = hi > 31 ? 31 : hi;
                  mk = (0xffffffffu >> (31 - h2)) & (0xffffffffu << l2);
                }
                vmask[cc] = mk;
              }
            }
            uint8_t* prow = ptile + r * 128;
            float bsum = 0.f;
            // One pair for the key columns [CB, CB + NC): the Global mixer takes all 64; in a Local block a warp's 32 queries
            // (consecutive grid columns qb .. qb+31) only see key columns qb-5 .. qb+36, i.e. 48 of the 64: columns 0..47 for
            // the warps on the left half of the grid row, 16..63 on the right half (warp-uniform, compile-time ranges).
            auto block = [&](auto cb_, auto nc_) {
              constexpr int CB = decltype(cb_)::value, NC = decltype(nc_)::value;
              // block maximum (unmasked inside the visited columns: any reference >= the true maximum is valid); 4 chains
              float b0 = -INFINITY, b1 = -INFINITY, b2 = -INFINITY, b3 = -INFINITY;
#pragma unroll
              for (int c = CB; c < CB + NC; c += 8) {
                b0 = max3(b0, __uint_as_float(sv[c]), __uint_as_float(sv[c + 1]));
                b1 = max3(b1, __uint_as_float(sv[c + 2]), __uint_as_float(sv[c + 3]));
                b2 = max3(b2, __uint_as_float(sv[c + 4]), __uint_as_float(sv[c + 5]));
                b3 = max3(b3, __uint_as_float(sv[c + 6]), __uint_as_float(sv[c + 7]));
              }
              float bmax = fmaxf(fmaxf(b0, b1), fmaxf(b2, b3)) * sl2;   // log2 units of the scaled scores (sl2 > 0 keeps the order)
              if (LOCAL && (vmask[0] | vmask[1]) == 0u) bmax = -INFINITY;   // nothing visible for this query in this key row
              // Lazy rescaling: O accumulates in TMEM against the reference m; p = 2^(s - m) may exceed 1 by up to 2^8
              // before the reference is moved.  Only then is the O row rescaled in place (tcgen05.ld / st), which is rare.
              float factor = 1.0f;
              bool move = false;
              if (m == -INFINITY) m = bmax;                    // nothing accumulated yet for this row (its O row is exactly 0)
              else if (bmax > m + 8.0f) { move = true; factor = ex2_approx(m - bmax); l *= factor; m = bmax; }
              if (tr) MIX_TRACE(7, pc);                        // softmax: max done, waiting for PV(prev)
              if (kr > j0) {
                mbar_wait(&o_full[ch], (pc - 1u) & 1u);        // P V of the previous block has retired: O is stable, the P tile is free
                tc_fence_after();
                if (__any_sync(0xffffffffu, move)) {
                  uint32_t o[32];
                  tmem_ld32(lane_addr + o_col, o);
#pragma unroll
                  for (int k2 = 0; k2 < HD; ++k2) o[k2] = __float_as_uint(__uint_as_float(o[k2]) * factor);
                  tmem_st32(lane_addr + o_col, o);
                  tc_fence_before();
                }
              } else {
                mbar_wait(&so_empty[ch], (qc & 1u) ^ 1u);      // first block of a query tile: the previous proj MMA has consumed
              }                                                // the tile buffer (waited here, not at the tile start: its latency hides behind the loads above)
              if (tr) MIX_TRACE(8, pc);                        // softmax: PV(prev) done
              const float nm = (m == -INFINITY) ? 0.f : -m;
#pragma unroll
              for (int pcs = 0; pcs < 8; ++pcs) {              // 16-byte pieces of 8 key columns
                uint32_t pk[4] = {0u, 0u, 0u, 0u};
                if (pcs * 8 >= CB && pcs * 8 < CB + NC) {
#pragma unroll
                  for (int k2 = 0; k2 < 8; k2 += 2) {
                    const int c = pcs * 8 + k2;
                    float p0 = ex2_approx(fmaf(__uint_as_float(sv[c]), sl2, nm));
                    float p1 = ex2_approx(fmaf(__uint_as_float(sv[c + 1]), sl2, nm));
                    if (LOCAL) {
                      if (!((vmask[c >> 5] >> (c & 31)) & 1u)) p0 = 0.f;
                      if (!((vmask[(c + 1) >> 5] >> ((c + 1) & 31)) & 1u)) p1 = 0.f;
                    }
                    bsum += p0 + p1;
                    pk[k2 >> 1] = pack_bf16(p0, p1);
                  }
                }
                *reinterpret_cast<uint4*>(prow + ((pcs ^ (r & 7)) * 16)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
              }
            };
            if (!LOCAL) block(std::integral_constant<int, 0>{}, std::integral_constant<int, 64>{});
            else if (q & 1) block(std::integral_constant<int, 16>{}, std::integral_constant<int, 48>{});
            else block(std::integral_constant<int, 0>{}, std::integral_constant<int, 48>{});
            if (tr) MIX_TRACE(9, pc);                          // softmax: exps + P stores issued
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            mbar_arrive(&p_full[ch]);
            if (tr) MIX_TRACE(10, pc);                         // softmax: P published
            l += bsum;
          }
          // last block of this query tile: O of the whole tile, normalise, head output -> tile buffer (64B-swizzled [128 x 32] bf16)
          mbar_wait(&o_full[ch], pc & 1u);
          tc_fence_after();
          float acc[HD];
          {
            uint32_t o[32];
            tmem_ld32(lane_addr + o_col, o);
#pragma unroll
            for (int k2 = 0; k2 < HD; ++k2) acc[k2] = __uint_as_float(o[k2]);
            tc_fence_before();
          }
          const float inv = 1.0f / l;
          {
            uint8_t* row = ptile + r * 64;
#pragma unroll
            for (int c4 = 0; c4 < 4; ++c4) {
              uint32_t pk[4];
#pragma unroll
              for (int k2 = 0; k2 < 4; ++k2) pk[k2] = pack_bf16(acc[c4 * 8 + 2 * k2] * inv, acc[c4 * 8 + 2 * k2 + 1] * inv);
              *reinterpret_cast<uint4*>(row + ((c4 ^ sw) * 16)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
            }
          }
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          mbar_arrive(&so_full[ch]);
          if constexpr (K::OVL) {
            if (h == K::HEADS - 1) {
              // OVL: Y epilogue of this stream's own tile, right after the unit's last proj MMA (the Y-epilogue warpgroup is
              // busy draining q|k|v of the next heads).  Staging = the 4 KiB of the P tile this warp itself writes: free once
              // that proj MMA (the last reader of the tile buffer) has retired, which yd signals too.
              if (warp == 4 && lane == 0) MIX_TRACE(11, i);    // stream 0: last head output published, waiting for Y
              const float rs = ep.rowscale ? ep.rowscale[(long)e * ep.rs_gs + b] : 1.0f;
              float* xt = ep.x + (long)e * ep.x_gs + (long)b * K::N * D + (long)(qt * 128 + q * 32) * D;
              if (ep.dbg == 0) {
                y_tile_epilogue_regs<D, LNF, 2>(ep, e, u, qt, q, lane, lane_addr + Y_COL + (uint32_t)(qt * D), xt, rs, stg, 0, 2, &yd[ch], (uint32_t)i & 1u, nullptr);
              } else {
                mbar_wait(&yd[ch], (uint32_t)i & 1u);
                tc_fence_after();
                y_tile_epilogue<D, LNF, 8>(ep, e, u, qt, q, lane, lane_addr + Y_COL + (uint32_t)(qt * D), xt, rs, stg, nullptr);
              }
              tc_fence_before();
              if (warp == 4 && lane == 0) MIX_TRACE(13, i);    // stream 0: Y epilogue of its tile done
            }
          }
        }
      }

    }
  } else if (warp >= 12) {
    // ============================== Y epilogue warpgroup ==============================
    // Y -> +b_proj, DropPath scale, + fp32 residual -> x (in place) [+ LayerNorm 2], one thread per token row, while the
    // other warpgroups already work on the next unit (Y is handed back through y_empty).
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_EPI));
    const int q = warp & 3;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
    // 16 accumulator columns of the warp's 32 rows are transposed through a 2 KiB staging tile (row-major, 16-byte pieces
    // XOR-swizzled by row), so that global accesses are 64-byte row segments: lane = (row in a group of 8, float4 of the 16)
    float* stg = reinterpret_cast<float*>(sStg + q * 2048);
    const int rsub = lane >> 2, c4 = lane & 3;
    // ---- OVL: this warpgroup drains the q|k|v staging parts (one warp per TMEM lane quarter) into the q/k/v buffer of
    // the head's parity: a drain runs when its part is complete in TMEM and (first part of a head) the target buffer has
    // been retired by both attention streams.
    int d_u = blockIdx.x, d_h = 0, d_part = 0, d_e = -1;       // next drain: unit, head, part (2 per 128-token tile)
    uint32_t d_pc = 0, d_hc = 0;                               // staging phase counter, global head counter
    float* wbias = sBias + q * 3 * D;                          // this warp's copy of the expert's q|k|v bias
    auto try_drain = [&]() -> bool {
      if constexpr (!K::OVL) return false;
      if (d_u >= total) return false;
      // hardware-suspended waits: this warpgroup has nothing else to do, and a polling loop (test + nanosleep) was 20 %
      // of the kernel's executed instructions, issued on the sub-partitions the softmax warps need
      mbar_wait(&stg_full[0], d_pc & 1u);
      const int hb = d_hc & 1u;
      if (d_part == 0) {
        mbar_wait(&qkvf[hb], ((d_hc >> 1) & 1u) ^ 1u);
        const int e = d_u / upg;
        if (e != d_e) {
          __syncwarp();
          for (int k = lane; k < 3 * D; k += 32) wbias[k] = ep.bqkv[(long)e * 3 * D + k];
          __syncwarp();
          d_e = e;
        }
      }
      tc_fence_after();
      const int mt = d_part >> 1, part = d_part & 1;
      const int r = q * 32 + lane, sw = (r >> 1) & 3;
      uint8_t* qkv = sQ + hb * K::QKV1_BYTES;
      const int nt = part ? 1 : 2;                             // 32-column tensors in this part: q, k | v
      for (int tt = 0; tt < nt; ++tt) {
        uint32_t v[32];
        tmem_ld32(lane_addr + STGX_COL + (uint32_t)(tt * 32), v);
        if (tt == nt - 1) {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&stg_empty[0]);           // this warp's rows of the part are out of TMEM
        }
        const int t = part ? 2 : tt;                           // 0 = q, 1 = k, 2 = v
        const float4* bp = reinterpret_cast<const float4*>(wbias + t * D + d_h * HD);
        uint8_t* row = qkv + (size_t)t * K::NT * K::HT_BYTES + mt * K::HT_BYTES + r * 64;
#pragma unroll
        for (int c = 0; c < 4; ++c) {                          // 16-byte chunks of 8 head dimensions
          const float4 b0 = bp[2 * c], b1 = bp[2 * c + 1];
          *reinterpret_cast<uint4*>(row + ((c ^ sw) * 16)) = make_uint4(
              pack_bf16(__uint_as_float(v[8 * c]) + b0.x, __uint_as_float(v[8 * c + 1]) + b0.y),
              pack_bf16(__uint_as_float(v[8 * c + 2]) + b0.z, __uint_as_float(v[8 * c + 3]) + b0.w),
              pack_bf16(__uint_as_float(v[8 * c + 4]) + b1.x, __uint_as_float(v[8 * c + 5]) + b1.y),
              pack_bf16(__uint_as_float(v[8 * c + 6]) + b1.z, __uint_as_float(v[8 * c + 7]) + b1.w));
        }
      }
      ++d_pc;
      if (++d_part == 2 * K::NT) {
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        mbar_arrive(&qkvr[hb]);                                // 128 arrivals: every row of every tile of the head is in place
        if (warp == 12 && lane == 0) MIX_TRACE(14, (int)d_hc); // epi: head d_hc drained
        d_part = 0; ++d_hc;
        if (++d_h == K::HEADS) { d_h = 0; d_u += gridDim.x; }
      }
      return true;
    };
    if constexpr (K::OVL) {
      // OVL: the attention streams run the Y epilogue of their own tile; this warpgroup only drains q|k|v parts
      while (d_u < total) try_drain();
    } else {
    int i = 0;
    for (int u = blockIdx.x; u < total; u += gridDim.x, ++i) {
      const int e = u / upg, b = u % upg;
      const float rs = ep.rowscale ? ep.rowscale[(long)e * ep.rs_gs + b] : 1.0f;
      float* xunit = ep.x + (long)e * ep.x_gs + (long)b * K::N * D;
      {
        // this warpgroup is idle until the unit's last proj MMA retires: start the trip of its residual rows (128 KiB)
        // from HBM to L2 now
        const char* xl2 = reinterpret_cast<const char*>(xunit);
#pragma unroll
        for (int k = 0; k < 8; ++k) asm volatile("prefetch.global.L2 [%0];" ::"l"(xl2 + ((long)(k * 128 + (threadIdx.x - 384))) * 128));
      }
      mbar_wait(&y_full, (uint32_t)i & 1u);
      tc_fence_after();
      if (warp == 12 && lane == 0) MIX_TRACE(11, i);           // epi: y_full observed
      for (int qt = 0; qt < K::NT; ++qt) {
        // Y is handed back tile by tile (y_empty[qt]): the next unit's first proj MMA of a tile only waits for that tile
        if constexpr (LNF)
          y_tile_epilogue_regs<D, LNF, 2, false>(ep, e, u, qt, q, lane, lane_addr + Y_COL + (uint32_t)(qt * D),
                                                 xunit + (long)(qt * 128 + q * 32) * D, rs, stg, 0, 2, nullptr, 0u, &y_empty[qt]);
        else
          y_tile_epilogue<D, LNF>(ep, e, u, qt, q, lane, lane_addr + Y_COL + (uint32_t)(qt * D), xunit + (long)(qt * 128 + q * 32) * D,
                                  rs, stg, &y_empty[qt]);
        if (warp == 12 && lane == 0 && qt == K::NT - 1) MIX_TRACE(12, i);     // epi: Y drained (+ LayerNorm of the last tile)
      }
      if (warp == 12 && lane == 0) MIX_TRACE(13, i);           // epi: unit done
    }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

void* g_mixer_trace = nullptr;

// [groups][rows][K] bf16, k contiguous: box = box_k x box_rows x 1
int map3(CUtensorMap* map, const void* ptr, long K, long rows, long groups, int box_k, int box_rows, CUtensorMapSwizzle sw) {
  if (reinterpret_cast<uintptr_t>(ptr) & 15) { mrnb_set_error("mixer_tc: misaligned operand"); return MRNB_ERR_ARG; }
  cuuint64_t dims[3] = {(cuuint64_t)K, (cuuint64_t)rows, (cuuint64_t)groups};
  cuuint64_t strides[2] = {(cuuint64_t)K * 2, (cuuint64_t)rows * K * 2};
  cuuint32_t box[3] = {(cuuint32_t)box_k, (cuuint32_t)box_rows, 1}, es[3] = {1, 1, 1};
  return encode_tensor_map("mixer_tc", map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, ptr, dims, strides, box, es, sw);
}

template <int D, bool LOCAL, bool LNF>
int launch_mixer(const MrnbMixer& p, cudaStream_t st) {
  using K = MCfg<D>;
  const long units = (long)p.groups * p.units_per_group;
  CUtensorMap tmA, tmWq, tmWp;
  MRNB_TRY(map3(&tmA, p.A, D, K::N, units, 64, 128, CU_TENSOR_MAP_SWIZZLE_128B));
  MRNB_TRY(map3(&tmWq, p.Wqkv, D, 3 * D, p.groups, 64, 32, CU_TENSOR_MAP_SWIZZLE_128B));
  MRNB_TRY(map3(&tmWp, p.Wproj, D, D, p.groups, 32, D, CU_TENSOR_MAP_SWIZZLE_64B));
  MixParams ep{};
  ep.bqkv = p.bqkv; ep.bproj = p.bproj; ep.x = p.x; ep.x_gs = p.x_gstride;
  ep.rowscale = p.rowscale; ep.rs_gs = p.rowscale_gstride;
  ep.ln_out = (__nv_bfloat16*)p.ln_out; ep.ln_gamma = p.ln_gamma; ep.ln_beta = p.ln_beta; ep.ln_eps = p.ln_eps;
  ep.upg = p.units_per_group; ep.total = (int)units;
  { const char* e = getenv("MRNB_MIXER_DBG"); ep.dbg = e ? atoi(e) : 0; }
  ep.trace = (unsigned long long*)g_mixer_trace;
  static bool attr = false;
  static int num_sms = 148;
  if (!attr) {
    cudaFuncSetAttribute(mixer_tc_kernel<D, LOCAL, LNF>, cudaFuncAttributeMaxDynamicSharedMemorySize, K::SMEM);
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
    attr = true;
  }
  const int grid = units < num_sms ? (int)units : num_sms;
  mixer_tc_kernel<D, LOCAL, LNF><<<grid, NTHREADS, K::SMEM, st>>>(tmA, tmWq, tmWp, ep);
  MRNB_CHECK_LAUNCH("mixer_tc_kernel");
  return MRNB_OK;
}

}  // namespace

int mrnb_mixer_tc(const MrnbMixer& p, cudaStream_t st) {
  MRNB_CHECK_ARG(p.A && p.Wqkv && p.bqkv && p.Wproj && p.bproj && p.x && p.groups > 0 && p.units_per_group > 0, "mixer_tc: null/empty argument");
  MRNB_CHECK_ARG(p.D == 64 || p.D == 128 || p.D == 256, "mixer_tc: D must be 64, 128 or 256");
  MRNB_CHECK_ARG(!p.ln_out || (p.D <= 128 && p.ln_gamma && p.ln_beta), "mixer_tc: fused LayerNorm needs D <= 128");
  MRNB_CHECK_ARG(!(p.local && p.D == 256), "mixer_tc: the Local mixer exists for the 64- and 128-wide stages only");
  MRNB_CHECK_ARG(p.x_gstride % 4 == 0, "mixer_tc: misaligned residual stream");
  const double units = (double)p.groups * p.units_per_group, N = 32768.0 / p.D;
  // dense-equivalent work: qkv + proj GEMMs (8 N D^2) + attention (4 N^2 D); traffic: A + x in + x out (+ LN out)
  MrnbProfScope prof(MRNB_PROF_MIXER, st, units * (8.0 * N * p.D * p.D + 4.0 * N * N * p.D),
                     units * N * p.D * (2.0 + 8.0 + (p.ln_out ? 2.0 : 0.0)));
#define MRNB_MIX(D_, LOC_) return p.ln_out ? launch_mixer<D_, LOC_, true>(p, st) : launch_mixer<D_, LOC_, false>(p, st);
  if (p.D == 64) { if (p.local) { MRNB_MIX(64, true) } MRNB_MIX(64, false) }
  if (p.D == 128) { if (p.local) { MRNB_MIX(128, true) } MRNB_MIX(128, false) }
  return launch_mixer<256, false, false>(p, st);
#undef MRNB_MIX
}

extern "C" void mrnb_mixer_set_trace(void* device_buffer) { g_mixer_trace = device_buffer; }

// C-ABI test entry: one group.  x [units][N][D] fp32 is updated in place; ln_out (bf16 [units][N][D]) optional.
extern "C" int mrnb_mixer_bf16(const void* A, const void* Wqkv, const float* bqkv, const void* Wproj, const float* bproj,
                               float* x, const float* rowscale, void* ln_out, const float* ln_gamma, const float* ln_beta,
                               float ln_eps, int units, int D, int local, cudaStream_t stream) {
  MrnbMixer p{};
  p.A = A; p.Wqkv = Wqkv; p.bqkv = bqkv; p.Wproj = Wproj; p.bproj = bproj; p.x = x; p.x_gstride = 0;
  p.rowscale = rowscale; p.rowscale_gstride = 0;
  p.ln_out = ln_out; p.ln_gamma = ln_gamma; p.ln_beta = ln_beta; p.ln_eps = ln_eps;
  p.D = D; p.groups = 1; p.units_per_group = units; p.local = local;
  return mrnb_mixer_tc(p, stream);
}
