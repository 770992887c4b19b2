// SVTR mixer attention on the tensor cores (bf16 mode).   Reference: modules/svtr.py:133-152 (Attention.forward),
// Local mixer mask :116-128.
//
// One CTA per (expert*sample, head, 128-query tile).  Key blocks of 128:
//   S_j = Q K_j^T      tcgen05.mma M128 N128 K32  (Q, K_j: TMA -> 64B-swizzled K-major smem tiles)      -> TMEM cols [0,128)
//   softmax warps: tcgen05.ld S_j, scale (+ Local window predicate on the index), running max / sum per query row
//                  (one row per thread), P_j = exp(S_j - m) as bf16 into a 128B-swizzled K-major smem tile
//   O_j = P_j V_j      tcgen05.mma M128 N32 K128  (V_j read where it lies: MN-major, 64B swizzle)       -> TMEM cols [128,160)
//   acc = acc * exp(m_old - m_new) + O_j in registers; out = acc / l.
// Warp roles: warp 0 TMA producer, warp 1 TMEM alloc + MMA issuer, warps 2..9 softmax / epilogue: two warps per TMEM
// lane quarter, each owning one 64-key half of the block (and one 16-dim half of O); the partners exchange their
// half-row maxima through shared memory.  The softmax chain is latency-bound, so the extra warps are what buys speed.
#include "sm100.cuh"

namespace {

constexpr int QT = 128, KT = 128, HD = 32;
constexpr int TILE_BYTES = 128 * HD * 2;        // 8 KiB: one Q / K / V tile
constexpr int P_BYTES = 128 * KT * 2;           // 32 KiB
constexpr int TMEM_COLS = 256;
constexpr uint32_t O_COL = 128;

// named barrier 1 + q for the two partner warps (64 threads) of TMEM lane quarter q; immediate ids keep the CTA at 5 barriers
__device__ __forceinline__ void pair_sync(int q) {
  switch (q) {
    case 0: asm volatile("bar.sync 1, 64;" ::: "memory"); break;
    case 1: asm volatile("bar.sync 2, 64;" ::: "memory"); break;
    case 2: asm volatile("bar.sync 3, 64;" ::: "memory"); break;
    default: asm volatile("bar.sync 4, 64;" ::: "memory"); break;
  }
}

constexpr int ATT_THREADS = 64 + 256;

// Persistent: CTA c walks the work items (query tile, head, unit) c, c + gridDim.x, ...  Barriers, TMEM and the tensor-map
// prefetch are set up once per CTA; key blocks are numbered across items (jc) so that the K/V ring, S, P and O keep one
// running phase each, and the Q tile is handed back through q_empty.  (One CTA per item spent more time in set-up and
// tear-down than in the two MMAs of a 128-token unit: 195 us per launch at d = 256.)
template <bool LOCAL>
__global__ void __launch_bounds__(ATT_THREADS)
attn_tc_kernel(const __grid_constant__ CUtensorMap tm, __nv_bfloat16* __restrict__ out, int N, int d, int heads, int total) {
  constexpr int W = 64;            // SVTR token grid width for 32x256 crops (modules/svtr.py:348): shifts, not divisions
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + align_smem_1024_offset(smem_raw);
  uint8_t* sQ = smem;                          // 8 KiB
  uint8_t* sKV = smem + TILE_BYTES;            // 2 slots x (K 8 KiB + V 8 KiB)
  uint8_t* sP = smem + TILE_BYTES + 4 * TILE_BYTES;   // 32 KiB, 1024-aligned (offset 40 KiB)
  __shared__ __align__(8) uint64_t q_full, q_empty, kv_full[2], kv_empty[2], s_full, s_empty, p_full, o_full;
  __shared__ uint32_t tmem_base_sh;
  __shared__ float xch[3][2][QT];              // [block parity | 2 = end of item][column half][row]: partner exchange

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nqt = N / QT, nb_all = N / KT;
  (void)W;
  // Local mixer: a 128-token block is two rows of the 64-wide token grid; rows further than 3 apart never interact,
  // so q-tile t only needs key blocks |t - j| <= 2 (CTA-uniform skip of MMAs, loads and softmax).
  auto item = [&](int w, int& qt, int& h, int& g, int& jb0, int& nb) {
    qt = w % nqt; h = (w / nqt) % heads; g = w / (nqt * heads);
    jb0 = LOCAL ? (qt - 2 > 0 ? qt - 2 : 0) : 0;
    const int jb1 = LOCAL ? (qt + 3 < nb_all ? qt + 3 : nb_all) : nb_all;
    nb = jb1 - jb0;
  };

  if (threadIdx.x == 0) {
    mbar_init(&q_full, 1); mbar_init(&q_empty, 1);
    for (int s = 0; s < 2; ++s) { mbar_init(&kv_full[s], 1); mbar_init(&kv_empty[s], 1); }
    mbar_init(&s_full, 1); mbar_init(&s_empty, 256); mbar_init(&p_full, 256); mbar_init(&o_full, 1);
    fence_mbarrier_init();
    prefetch_tmap(&tm);
  }
  if (warp == 1) tmem_alloc(&tmem_base_sh, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_sh;

  if (warp == 0) {
    if (lane == 0) {
      uint32_t it = 0, jc = 0;
      for (int w = blockIdx.x; w < total; w += gridDim.x, ++it) {
        int qt, h, g, jb0, nb;
        item(w, qt, h, g, jb0, nb);
        const long row0 = (long)g * N;
        mbar_wait(&q_empty, (it & 1u) ^ 1u);                      // every S MMA of the previous item has read its Q tile
        mbar_expect_tx(&q_full, TILE_BYTES);
        tma_load_2d(sQ, &tm, &q_full, h * HD, (int)(row0 + qt * QT));
        for (int j = 0; j < nb; ++j, ++jc) {
          const int s = jc & 1;
          mbar_wait(&kv_empty[s], ((jc >> 1) & 1u) ^ 1u);
          mbar_expect_tx(&kv_full[s], 2 * TILE_BYTES);
          tma_load_2d(sKV + s * 2 * TILE_BYTES, &tm, &kv_full[s], d + h * HD, (int)(row0 + (jb0 + j) * KT));
          tma_load_2d(sKV + s * 2 * TILE_BYTES + TILE_BYTES, &tm, &kv_full[s], 2 * d + h * HD, (int)(row0 + (jb0 + j) * KT));
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // S = Q K^T : M128 N128, A and B K-major ; O = P V : M128 N32, A K-major, B MN-major
      constexpr uint32_t idesc_s = umma_idesc(UMMA_BF16, QT, KT);
      constexpr uint32_t idesc_o = umma_idesc(UMMA_BF16, QT, HD, false, true);
      // Q, K, V tiles: rows of 64 B (SWIZZLE_64B), atoms 512 B apart
      const uint64_t qdesc = umma_smem_desc(smem_u32(sQ), 16, 512, UMMA_SWIZZLE_64B);
      const uint64_t pdesc = umma_desc_k128(smem_u32(sP));
      // blocks are numbered jc across items: S(jc + 1) goes out as soon as the softmax warps have pulled S(jc) out of TMEM
      // (for the first block of an item also: its Q tile has landed), then P(jc) V(jc)
      auto issue_s = [&](uint32_t jc) {
        const int s = jc & 1;
        mbar_wait(&kv_full[s], (jc >> 1) & 1u);
        tc_fence_after();
        const uint64_t kdesc = umma_smem_desc(smem_u32(sKV + s * 2 * TILE_BYTES), 16, 512, UMMA_SWIZZLE_64B);
#pragma unroll
        for (int k = 0; k < HD / 16; ++k) umma_bf16(tmem_base, qdesc + (uint64_t)(k * 2), kdesc + (uint64_t)(k * 2), idesc_s, k);
        umma_commit(&s_full);
      };
      uint32_t it = 0, jc = 0;
      int w = blockIdx.x;
      int qt, h, g, jb0, nb = 0;
      if (w < total) {
        item(w, qt, h, g, jb0, nb);
        mbar_wait(&q_full, 0);
        issue_s(0);
        if (nb == 1) umma_commit(&q_empty);
      }
      while (w < total) {
        for (int j = 0; j < nb; ++j, ++jc) {
          // next S of the same item goes out before P V of this block (the softmax warps then find it ready)
          if (j + 1 < nb) {
            mbar_wait(&s_empty, jc & 1u);
            issue_s(jc + 1);
            if (j + 2 == nb) umma_commit(&q_empty);               // last S of this item issued: Q is free once it retires
          }
          mbar_wait(&p_full, jc & 1u);
          tc_fence_after();
          const int s = jc & 1;
          const uint64_t vdesc = umma_smem_desc(smem_u32(sKV + s * 2 * TILE_BYTES + TILE_BYTES), 16, 512, UMMA_SWIZZLE_64B);
#pragma unroll
          for (int k = 0; k < KT / 16; ++k) {
            // P: two 64-key halves of 16 KiB, +32 B per 16 keys inside the 128 B row; V: +16 key rows of 64 B
            const uint64_t pa = pdesc + (uint64_t)(((k >> 2) * 16384 + (k & 3) * 32) >> 4);
            const uint64_t vb = vdesc + (uint64_t)((k * 16 * 64) >> 4);
            umma_bf16(tmem_base + O_COL, pa, vb, idesc_o, k);
          }
          umma_commit(&kv_empty[s]);
          umma_commit(&o_full);
          if (j + 1 == nb) {
            // last block of the item: the first S of the NEXT item follows its P V (the softmax warps still have the
            // item's normalisation and store ahead of them; p_full(jc) implies s_empty(jc))
            const int wn = w + gridDim.x;
            if (wn < total) {
              int qt2, h2, g2, jb2, nb2;
              item(wn, qt2, h2, g2, jb2, nb2);
              mbar_wait(&q_full, (it + 1) & 1u);
              mbar_wait(&s_empty, jc & 1u);
              issue_s(jc + 1);
              if (nb2 == 1) umma_commit(&q_empty);
            }
          }
        }
        w += gridDim.x; ++it;
        if (w < total) item(w, qt, h, g, jb0, nb);
      }
    }
  } else {
    const int q = warp & 3;
    const int ch = (warp - 2) >> 2;               // 64-key half of every block / 16-dim half of O owned by this warp
    const int r = q * 32 + lane;                  // query row inside the tile == TMEM lane
    const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
    const float sl2 = 0.17677669529663688110f * 1.4426950408889634f;     // 32^-0.5 * log2(e)
    uint32_t jc = 0;                              // key blocks are numbered across items (barrier phases)
    for (int w = blockIdx.x; w < total; w += gridDim.x) {
    int qt, h, g, jb0, nb;
    item(w, qt, h, g, jb0, nb);
    const long row0 = (long)g * N;
    const int n = qt * QT + r;                    // token index of this query
    const int qh = n >> 6, qw = n & 63;
    float m = -INFINITY, l = 0.f, corr_prev = 0.f;
    float acc[HD / 2];
#pragma unroll
    for (int j = 0; j < HD / 2; ++j) acc[j] = 0.f;
    for (int j = 0; j < nb; ++j, ++jc) {
      mbar_wait(&s_full, jc & 1u);
      tc_fence_after();
      // Local window as a 32-bit validity mask per 32-key chunk (a chunk lies inside one row of the token grid):
      // bit i set <=> |kh - qh| <= 3 and |kw0 + i - qw| <= 5.
      uint32_t vmask[2];
#pragma unroll
      for (int cc = 0; cc < 2; ++cc) {
        vmask[cc] = 0xffffffffu;
        if (LOCAL) {
          const int key0 = (jb0 + j) * KT + (ch * 2 + cc) * 32;
          const int dh = (key0 >> 6) - qh;
          const int lo = qw - 5 - (key0 & 63), hi = qw + 5 - (key0 & 63);       // valid i in [lo, hi]
          uint32_t mk = 0u;
          if (dh >= -3 && dh <= 3 && hi >= 0 && lo <= 31) {
            const int l2 = lo < 0 ? 0 : lo, h2 = hi > 31 ? 31 : hi;
            mk = (0xffffffffu >> (31 - h2)) & (0xffffffffu << l2);
          }
          vmask[cc] = mk;
        }
      }
      // pass 1: maximum over the visible keys of the chunks this warp visits.  The Local window mask must apply here:
      // a masked key next to the window can score tens of log2 units above every visible one (peaked scores), and a
      // reference that high flushes all visible exp2() terms to zero -> l = 0 and a NaN / inf output row.
      float bmax = -INFINITY;
#pragma unroll
      for (int cc = 0; cc < 2; ++cc) {
        if (LOCAL && __all_sync(0xffffffffu, vmask[cc] == 0u)) continue;       // warp-uniform: nothing visible here
        uint32_t v[32];
        tmem_ld32(lane_addr + (uint32_t)((ch * 2 + cc) * 32), v);
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
          float s0 = __uint_as_float(v[i]), s1 = __uint_as_float(v[i + 1]);
          if (LOCAL) {
            if (!((vmask[cc] >> i) & 1u)) s0 = -INFINITY;
            if (!((vmask[cc] >> (i + 1)) & 1u)) s1 = -INFINITY;
          }
          bmax = max3(bmax, s0, s1);
        }
      }
      xch[jc & 1][ch][r] = bmax;
      pair_sync(q);                                              // the two warps of this lane quarter
      bmax = fmaxf(bmax, xch[jc & 1][ch ^ 1][r]);
      const float mnew = fmaxf(m, bmax * sl2);
      const float mref = (mnew == -INFINITY) ? 0.f : mnew;       // nothing visible so far
      const float corr = ex2_approx(m - mref);                   // m = -inf -> 0
      float bsum = 0.f;
      if (j > 0) {
        // deferred accumulation of the previous block: O_{j-1} = P_{j-1} V_{j-1} had all of pass 1 to complete, and
        // its completion also frees the P tile that pass 2 below overwrites
        mbar_wait(&o_full, (jc - 1u) & 1u);
        tc_fence_after();
        uint32_t o[16];
        tmem_ld16(lane_addr + O_COL + (uint32_t)(ch * 16), o);
#pragma unroll
        for (int i = 0; i < HD / 2; ++i) acc[i] = fmaf(acc[i], corr_prev, __uint_as_float(o[i]));
        tc_fence_before();
      }
      // pass 2: P = exp2(s*scale*log2e - m) -> bf16 -> swizzled smem (this warp's 64-key half = one 16 KiB P tile half)
#pragma unroll
      for (int cc = 0; cc < 2; ++cc) {
        uint32_t pk[16];
        if (LOCAL && __all_sync(0xffffffffu, vmask[cc] == 0u)) {
#pragma unroll
          for (int i = 0; i < 16; ++i) pk[i] = 0u;
        } else {
          uint32_t v[32];
          tmem_ld32(lane_addr + (uint32_t)((ch * 2 + cc) * 32), v);
#pragma unroll
          for (int i = 0; i < 32; i += 2) {
            float p0 = ex2_approx(fmaf(__uint_as_float(v[i]), sl2, -mref));
            float p1 = ex2_approx(fmaf(__uint_as_float(v[i + 1]), sl2, -mref));
            if (LOCAL) {
              if (!((vmask[cc] >> i) & 1u)) p0 = 0.f;
              if (!((vmask[cc] >> (i + 1)) & 1u)) p1 = 0.f;
            }
            __nv_bfloat162 hb = __floats2bfloat162_rn(p0, p1);
            bsum += p0 + p1;          // fp32 normaliser (rounding of P to bf16 is unbiased: no systematic mismatch with PV)
            pk[i >> 1] = *reinterpret_cast<uint32_t*>(&hb);
          }
        }
        uint8_t* prow = sP + ch * 16384 + r * 128;
#pragma unroll
        for (int p4 = 0; p4 < 4; ++p4) {
          const int piece = (cc * 4 + p4) ^ (r & 7);
          *reinterpret_cast<uint4*>(prow + piece * 16) = make_uint4(pk[p4 * 4], pk[p4 * 4 + 1], pk[p4 * 4 + 2], pk[p4 * 4 + 3]);
        }
      }
      tc_fence_before();
      mbar_arrive(&s_empty);                                      // this warp's half of S_j is consumed
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); // generic-proxy smem writes -> visible to UMMA
      mbar_arrive(&p_full);
      l = l * corr + bsum;                                        // partial normaliser of this half (same reference m)
      m = mnew;
      corr_prev = corr;
    }
    {
      mbar_wait(&o_full, (jc - 1u) & 1u);
      tc_fence_after();
      uint32_t o[16];
      tmem_ld16(lane_addr + O_COL + (uint32_t)(ch * 16), o);
#pragma unroll
      for (int i = 0; i < HD / 2; ++i) acc[i] = fmaf(acc[i], corr_prev, __uint_as_float(o[i]));
      tc_fence_before();
    }
    xch[2][ch][r] = l;
    pair_sync(q);
    const float inv = 1.0f / (l + xch[2][ch ^ 1][r]);
    __nv_bfloat16* op = out + (row0 + n) * d + h * HD + ch * (HD / 2);
#pragma unroll
    for (int i = 0; i < HD / 2; i += 8) {
      uint32_t pk[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        __nv_bfloat162 hb = __floats2bfloat162_rn(acc[i + 2 * u] * inv, acc[i + 2 * u + 1] * inv);
        pk[u] = *reinterpret_cast<uint32_t*>(&hb);
      }
      *reinterpret_cast<uint4*>(op + i) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
    }
      pair_sync(q);                                                // xch[2] is rewritten by the next item
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, TMEM_COLS);
}

}  // namespace

// qkv [groups*N, 3d] bf16 -> out [groups*N, d] bf16 ; N % 128 == 0, head_dim 32
int mrnb_attention_tc(const void* qkv, void* out, int groups, int N, int d, int heads, int H, int W, int local, cudaStream_t st) {
  MRNB_CHECK_ARG(qkv && out && groups > 0 && N % 128 == 0 && d == heads * HD && H * W == N && W == 64, "attention_tc: bad argument (token grid width must be 64)");
  CUtensorMap tm;
  cuuint64_t dims[2] = {(cuuint64_t)(3 * d), (cuuint64_t)((long)groups * N)};
  cuuint64_t strides[1] = {(cuuint64_t)(3 * d) * 2};
  cuuint32_t box[2] = {HD, 128}, es[2] = {1, 1};
  MRNB_TRY(encode_tensor_map("attention_tc", &tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, qkv, dims, strides, box, es,
                             CU_TENSOR_MAP_SWIZZLE_64B));
  const size_t smem = 1024 + TILE_BYTES + 4 * TILE_BYTES + P_BYTES;
  static bool attr = false;
  if (!attr) {
    cudaFuncSetAttribute(attn_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    cudaFuncSetAttribute(attn_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    attr = true;
  }
  const long total = (long)(N / QT) * heads * groups;
  static int n_sm = 0;
  if (!n_sm) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev); if (n_sm <= 0) n_sm = 148; }
  const long cap = 2L * n_sm;                    // two persistent CTAs per SM (2 x 256 TMEM columns, 2 x 73 KiB shared memory)
  const int grid = (int)(total < cap ? total : cap);
  if (local) attn_tc_kernel<true><<<grid, ATT_THREADS, smem, st>>>(tm, (__nv_bfloat16*)out, N, d, heads, (int)total);
  else attn_tc_kernel<false><<<grid, ATT_THREADS, smem, st>>>(tm, (__nv_bfloat16*)out, N, d, heads, (int)total);
  MRNB_CHECK_LAUNCH("attn_tc_kernel");
  return MRNB_OK;
}

extern "C" int mrnb_svtr_attention_bf16(const void* qkv, void* out, int groups, int N, int d, int heads, int H, int W,
                                        int local, cudaStream_t stream) {
  return mrnb_attention_tc(qkv, out, groups, N, d, heads, H, W, local, stream);
}
