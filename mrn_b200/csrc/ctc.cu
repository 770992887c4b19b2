// Fused gated combine + row log-sum-exp + CTC alpha/beta + gate-gradient contraction + greedy decode.
//
// Replaces, for the CTC head of MRN (reference paths relative to /root/reference):
//   modules/model.py:361-364,410-423   pad_zeros_features (pads with ONES) + stack + gate-mul + sum
//   modules/model.py:383-393           hard route (one-hot gate)
//   il_modules/mrn.py:251-252,345-346  log_softmax(2).permute(1,0,2) -> CTCLoss(mean, zero_infinity)
//   test.py:211-221,257                preds.max(2), softmax-max confidence
//   tools/utils.py:62-76               collapse repeats / drop blank
//
// HBM plan (DESIGN.md "combine+CTC"): the ragged expert logits z_i[B,T,C_i] are read ONCE.  The row pass
// produces lse[b,t], the <=26 label-column log-probs the lattice needs, the per-expert label values, and
// E_i[b,t] = sum_c softmax(logits)[c] * pad_i[c].  With those, the router-stage gradient
//   dL/dgate[b,i] = scale_b * sum_t ( E_i[b,t] - sum_s occ[b,t,s] * pad_i[b,t,ext_s] )
// needs no second pass over the logits (SURVEY.md Appendix A.5 identity, re-associated).
#include "sm100.cuh"

namespace {

constexpr int ROW_THREADS = 256;
constexpr int S1_MAX = 32;   // blank + up to 31 labels (reference uses batch_max_length = 25)

struct RowPtrs {
  const float* z[MRNB_MAX_EXPERTS];
  long ld[MRNB_MAX_EXPERTS];
  int C[MRNB_MAX_EXPERTS];
};

struct RowAcc {
  float m, s;
  float A[MRNB_MAX_EXPERTS];
  float best;
  int besti;
};

template <int I>
__device__ __forceinline__ void acc_merge(float& m, float& s, float (&A)[I], float& best, int& besti,
                                          float m2, float s2, const float (&A2)[I], float best2, int besti2) {
  const float mn = fmaxf(m, m2);
  const float f1 = (m == -INFINITY) ? 0.f : __expf(m - mn);
  const float f2 = (m2 == -INFINITY) ? 0.f : __expf(m2 - mn);
  s = s * f1 + s2 * f2;
#pragma unroll
  for (int i = 0; i < I; ++i) A[i] = A[i] * f1 + A2[i] * f2;
  m = mn;
  if (best2 > best || (best2 == best && besti2 < besti)) { best = best2; besti = besti2; }
}

constexpr float LOG2E = 1.4426950408889634f;

// Vector pass over one charset segment [lo, hi) in which experts i < K are past their charset (pad value 1.0) and
// experts i >= K are valid: 4 columns per thread from 16-byte loads, no per-element predicates, one online-softmax
// rescale per 4 columns.  The <= 3 ragged columns at either end of the segment go through the scalar update.
template <int I>
__device__ __forceinline__ void row_update(float l, const float (&v)[I], int c, float& m, float& s, float (&A)[I],
                                           float& best, int& besti) {
  if (l > best || (l == best && c < besti)) { best = l; besti = c; }
  if (l > m) {
    const float f = ex2_approx((m - l) * LOG2E);
    s *= f;
#pragma unroll
    for (int i = 0; i < I; ++i) A[i] *= f;
    m = l;
  }
  const float e = ex2_approx((l - m) * LOG2E);
  s += e;
#pragma unroll
  for (int i = 0; i < I; ++i) A[i] = fmaf(e, v[i], A[i]);
}

template <int I, int K>
__device__ __forceinline__ void row_segment(const float* const (&zr)[I], const float (&g)[I], int lo, int hi, int tid,
                                            float* __restrict__ lrow, float& m, float& s, float (&A)[I], float& best,
                                            int& besti) {
  if (lo >= hi) return;
  float gk = 0.f;
#pragma unroll
  for (int i = 0; i < K; ++i) gk += g[i];
  const int lo4 = min((lo + 3) & ~3, hi), hi4 = max(hi & ~3, lo4);
  for (int c0 = lo4 + tid * 4; c0 < hi4; c0 += ROW_THREADS * 4) {
    float4 v[I];
#pragma unroll
    for (int i = K; i < I; ++i) v[i] = __ldg(reinterpret_cast<const float4*>(zr[i] + c0));
    float l0 = gk, l1 = gk, l2 = gk, l3 = gk;
#pragma unroll
    for (int i = K; i < I; ++i) {
      l0 = fmaf(g[i], v[i].x, l0); l1 = fmaf(g[i], v[i].y, l1); l2 = fmaf(g[i], v[i].z, l2); l3 = fmaf(g[i], v[i].w, l3);
    }
    if (lrow) *reinterpret_cast<float4*>(lrow + c0) = make_float4(l0, l1, l2, l3);
    // this thread visits columns in ascending order: strict > keeps the first maximum
    if (l0 > best) { best = l0; besti = c0; }
    if (l1 > best) { best = l1; besti = c0 + 1; }
    if (l2 > best) { best = l2; besti = c0 + 2; }
    if (l3 > best) { best = l3; besti = c0 + 3; }
    const float cm = fmaxf(fmaxf(l0, l1), fmaxf(l2, l3));
    if (cm > m) {
      const float f = ex2_approx((m - cm) * LOG2E);        // m = -inf -> 0
      s *= f;
#pragma unroll
      for (int i = 0; i < I; ++i) A[i] *= f;
      m = cm;
    }
    const float mb = -m * LOG2E;
    const float e0 = ex2_approx(fmaf(l0, LOG2E, mb)), e1 = ex2_approx(fmaf(l1, LOG2E, mb));
    const float e2 = ex2_approx(fmaf(l2, LOG2E, mb)), e3 = ex2_approx(fmaf(l3, LOG2E, mb));
    const float es = (e0 + e1) + (e2 + e3);
    s += es;
#pragma unroll
    for (int i = 0; i < K; ++i) A[i] += es;                // pad value 1.0
#pragma unroll
    for (int i = K; i < I; ++i) A[i] = fmaf(e0, v[i].x, fmaf(e1, v[i].y, fmaf(e2, v[i].z, fmaf(e3, v[i].w, A[i]))));
  }
  // ragged ends (and segments shorter than one vector)
  for (int part = 0; part < 2; ++part) {
    const int a = part == 0 ? lo : hi4, b = part == 0 ? lo4 : hi;
    const int c = a + tid;
    if (c < b) {
      float v[I];
      float l = gk;
#pragma unroll
      for (int i = 0; i < I; ++i) {
        v[i] = i < K ? 1.0f : __ldg(zr[i] + c);
        if (i >= K) l = fmaf(g[i], v[i], l);
      }
      if (lrow) lrow[c] = l;
      row_update<I>(l, v, c, m, s, A, best, besti);
    }
  }
}

template <int I, int K>
struct SegLoop {
  __device__ static __forceinline__ void run(const float* const (&zr)[I], const float (&g)[I], const RowPtrs& P, int tid,
                                             float* lrow, float& m, float& s, float (&A)[I], float& best, int& besti) {
    row_segment<I, K>(zr, g, K == 0 ? 0 : P.C[K - 1], P.C[K], tid, lrow, m, s, A, best, besti);
    SegLoop<I, K + 1>::run(zr, g, P, tid, lrow, m, s, A, best, besti);
  }
};
template <int I>
struct SegLoop<I, I> {
  __device__ static __forceinline__ void run(const float* const (&)[I], const float (&)[I], const RowPtrs&, int, float*, float&,
                                             float&, float (&)[I], float&, int&) {}
};

// One CTA per (b,t) row.  fast = 1 (host-checked: charsets ascending, 16-byte aligned rows) enables the segment /
// vector pass whenever every gate weight is non-zero (soft route); the hard route (one-hot gate) keeps the generic
// loop, which skips the loads of the unselected experts.
template <int I>
__global__ void __launch_bounds__(ROW_THREADS)
combine_row_kernel(RowPtrs P, const float* __restrict__ gate,   // [B,I]
                   int T, int C, int fast,
                   float* __restrict__ logits, long ldo,          // optional [B*T, ldo]
                   float* __restrict__ lse,                       // [B*T]
                   float* __restrict__ E,                         // optional [B*T, I]
                   int* __restrict__ amax, float* __restrict__ maxprob,   // optional [B*T]
                   const long long* __restrict__ targets, const int* __restrict__ tlen, int Lmax,
                   float* __restrict__ lpe,                       // optional [B*T, S1]
                   float* __restrict__ zlab,                      // optional [B*T, S1, I]
                   int S1) {
  const int row = blockIdx.x;
  const int b = row / T;
  const int tid = threadIdx.x;
  float g[I];
  const float* zr[I];
#pragma unroll
  for (int i = 0; i < I; ++i) {
    g[i] = gate[b * I + i];
    zr[i] = P.z[i] + (long)row * P.ld[i];
  }
  float m = -INFINITY, s = 0.f, best = -INFINITY;
  int besti = 0x7fffffff;
  float A[I];
#pragma unroll
  for (int i = 0; i < I; ++i) A[i] = 0.f;

  bool soft = fast != 0;
#pragma unroll
  for (int i = 0; i < I; ++i) soft = soft && (g[i] != 0.f);
  if (soft) {
    SegLoop<I, 0>::run(zr, g, P, tid, logits ? logits + (long)row * ldo : nullptr, m, s, A, best, besti);
  } else
  for (int c0 = tid; c0 < C; c0 += ROW_THREADS * 4) {
    float v[4][I];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int c = c0 + u * ROW_THREADS;
#pragma unroll
      for (int i = 0; i < I; ++i) {
        // gate == 0 only happens for the hard (one-hot) route: skip the load, contribution is exactly 0
        v[u][i] = (c < P.C[i]) ? ((g[i] != 0.f && c < C) ? __ldg(zr[i] + c) : 0.f) : 1.0f;
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int c = c0 + u * ROW_THREADS;
      if (c < C) {
        float l = 0.f;
#pragma unroll
        for (int i = 0; i < I; ++i) l = fmaf(g[i], v[u][i], l);
        if (logits) logits[(long)row * ldo + c] = l;
        if (l > best) { best = l; besti = c; }     // ascending c per thread: first maximum wins
        if (l > m) {
          const float f = __expf(m - l);           // m = -inf -> 0
          s *= f;
#pragma unroll
          for (int i = 0; i < I; ++i) A[i] *= f;
          m = l;
        }
        const float e = __expf(l - m);
        s += e;
#pragma unroll
        for (int i = 0; i < I; ++i) A[i] = fmaf(e, v[u][i], A[i]);
      }
    }
  }
  // warp reduce
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float m2 = __shfl_xor_sync(0xffffffffu, m, o);
    const float s2 = __shfl_xor_sync(0xffffffffu, s, o);
    const float b2 = __shfl_xor_sync(0xffffffffu, best, o);
    const int bi2 = __shfl_xor_sync(0xffffffffu, besti, o);
    float A2[I];
#pragma unroll
    for (int i = 0; i < I; ++i) A2[i] = __shfl_xor_sync(0xffffffffu, A[i], o);
    acc_merge<I>(m, s, A, best, besti, m2, s2, A2, b2, bi2);
  }
  __shared__ float sm_m[ROW_THREADS / 32], sm_s[ROW_THREADS / 32], sm_b[ROW_THREADS / 32];
  __shared__ int sm_bi[ROW_THREADS / 32];
  __shared__ float sm_A[ROW_THREADS / 32][I];
  __shared__ float sm_lse;
  const int w = tid >> 5, lane = tid & 31;
  if (lane == 0) {
    sm_m[w] = m; sm_s[w] = s; sm_b[w] = best; sm_bi[w] = besti;
#pragma unroll
    for (int i = 0; i < I; ++i) sm_A[w][i] = A[i];
  }
  __syncthreads();
  if (tid == 0) {
    for (int k = 1; k < ROW_THREADS / 32; ++k) {
      float A2[I];
#pragma unroll
      for (int i = 0; i < I; ++i) A2[i] = sm_A[k][i];
      acc_merge<I>(m, s, A, best, besti, sm_m[k], sm_s[k], A2, sm_b[k], sm_bi[k]);
    }
    const float l = m + logf(s);
    sm_lse = l;
    lse[row] = l;
    if (E) {
      const float inv = 1.0f / s;
#pragma unroll
      for (int i = 0; i < I; ++i) E[(long)row * I + i] = A[i] * inv;
    }
    if (amax) amax[row] = besti;
    if (maxprob) maxprob[row] = __expf(best - l);
  }
  if (lpe) {
    __syncthreads();
    if (tid < S1) {
      const int L = min(tlen[b], Lmax);
      float l = 0.f;
      long base = ((long)row * S1 + tid) * I;
      const bool valid = (tid == 0) || (tid - 1 < L);
      int col = 0;
      if (tid > 0 && valid) col = (int)targets[(long)b * Lmax + tid - 1];
      if (valid && col >= 0 && col < C) {
#pragma unroll
        for (int i = 0; i < I; ++i) {
          const float v = (col < P.C[i]) ? ((g[i] != 0.f) ? zr[i][col] : 0.f) : 1.0f;
          l = fmaf(g[i], v, l);
          if (zlab) zlab[base + i] = v;
        }
        lpe[(long)row * S1 + tid] = l - sm_lse;
      } else {
        lpe[(long)row * S1 + tid] = -INFINITY;
        if (zlab) {
#pragma unroll
          for (int i = 0; i < I; ++i) zlab[base + i] = 0.f;
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// TMA-staged persistent variant of the row pass (the one the training step runs).
//
// One CTA per SM walks rows r = blockIdx.x, blockIdx.x + gridDim.x, ...  A producer thread streams each row's ragged
// expert slices into shared memory with 1-D bulk copies (cp.async.bulk, mbarrier complete_tx): the row is cut into
// chunks of 3072 columns, chunk j always lands in stage j ([I][3072] floats), so the columns past an expert's charset
// are pre-filled with the pad value 1.0 ONCE and never overwritten.  Stage j is released as soon as the consumers have
// pulled it into registers, so the next row's chunk j is already in flight while this row is still being reduced: up to
// a whole row (I*C*4 bytes, 120 KB for MLT17) of loads is outstanding per SM, independent of the arithmetic.
// Experts with a zero gate (hard route) are not loaded at all.  24 consumer warps do the online-softmax pass from
// conflict-free LDS.128 reads (the per-chunk dependency chain is long: fewer warps leave the SM latency-bound); two
// epilogue warps finish alternate rows from the per-thread partials, off the streaming path.
// ---------------------------------------------------------------------------------------------
constexpr int TMA_CONSUMERS = 704;             // 22 consumer warps: the per-chunk dependency chain needs the parallelism
constexpr int TMA_CHUNK = 4 * TMA_CONSUMERS;   // columns per stage = 4 per consumer thread
constexpr int TMA_MAX_CHUNKS = 8;

constexpr int TMA_EPI_WARPS = 4;                          // epilogue warp e finishes rows it = e (mod 4)
constexpr int TMA_THREADS = TMA_CONSUMERS + 32 + 32 * TMA_EPI_WARPS;      // + producer warp + epilogue warps

template <int I>
__global__ void __launch_bounds__(TMA_THREADS, 1)
combine_row_tma_kernel(RowPtrs P, const float* __restrict__ gate, int T, int C, int rows, int nchunks,
                       float* __restrict__ logits, long ldo, float* __restrict__ lse, float* __restrict__ E,
                       int* __restrict__ amax, float* __restrict__ maxprob, const long long* __restrict__ targets,
                       const int* __restrict__ tlen, int Lmax, float* __restrict__ lpe, float* __restrict__ zlab, int S1) {
  extern __shared__ __align__(128) float stage[];           // [nchunks][I][TMA_CHUNK], then partials [2][4 + I][256]
  __shared__ __align__(8) uint64_t full_bar[TMA_MAX_CHUNKS], empty_bar[TMA_MAX_CHUNKS];
  __shared__ __align__(8) uint64_t rowdone_bar[TMA_EPI_WARPS], partfree_bar[2];   // row-done: one per epilogue warp
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  float* part = stage + (size_t)nchunks * I * TMA_CHUNK;    // per-thread row partials, SoA: part[buf][k][tid]
  constexpr int PK = 4 + I;

  for (int k = tid; k < nchunks * I * TMA_CHUNK; k += blockDim.x) stage[k] = 1.0f;      // pad value, written once
  if (tid == 0) {
    for (int j = 0; j < nchunks; ++j) { mbar_init(&full_bar[j], 1); mbar_init(&empty_bar[j], TMA_CONSUMERS / 32); }
    for (int k = 0; k < TMA_EPI_WARPS; ++k) mbar_init(&rowdone_bar[k], TMA_CONSUMERS / 32);
    for (int k = 0; k < 2; ++k) mbar_init(&partfree_bar[k], 1);
    fence_mbarrier_init();
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // generic-proxy fill before async-proxy (TMA) writes
  __syncthreads();

  if (warp == TMA_CONSUMERS / 32) {
    // ---------------- producer warp: lane i streams expert i's slice of every chunk (lane 0 posts the byte count)
    {
      uint32_t it = 0;
      float gn[I];                                               // next row's gate, fetched one row ahead
#pragma unroll
      for (int i = 0; i < I; ++i) gn[i] = blockIdx.x < rows ? __ldg(gate + (blockIdx.x / T) * I + i) : 0.f;
      const int me = lane < I ? lane : 0;
      const int myC = P.C[me];
      const long myld = P.ld[me];
      const float* myz = P.z[me];
      for (int row = blockIdx.x; row < rows; row += gridDim.x, ++it) {
        float g[I];
#pragma unroll
        for (int i = 0; i < I; ++i) g[i] = gn[i];
        if (row + (int)gridDim.x < rows) {
          const int bn = (row + gridDim.x) / T;
#pragma unroll
          for (int i = 0; i < I; ++i) gn[i] = __ldg(gate + bn * I + i);
        }
        float myg = 0.f;
#pragma unroll
        for (int i = 0; i < I; ++i) if (i == lane) myg = g[i];
        const float* src = myz + (long)row * myld;
        for (int j = 0; j < nchunks; ++j) {
          uint32_t total = 0;
#pragma unroll
          for (int i = 0; i < I; ++i) {
            int n = P.C[i] - j * TMA_CHUNK;
            n = n < 0 ? 0 : (n > TMA_CHUNK ? TMA_CHUNK : n);
            total += (g[i] != 0.f) ? (uint32_t)((n + 3) & ~3) * 4u : 0u;      // whole 16-byte pieces (ld is padded to 4)
          }
          int n = myC - j * TMA_CHUNK;
          n = n < 0 ? 0 : (n > TMA_CHUNK ? TMA_CHUNK : n);
          const uint32_t nb = (lane < I && myg != 0.f) ? (uint32_t)((n + 3) & ~3) * 4u : 0u;
          mbar_wait(&empty_bar[j], (it & 1u) ^ 1u);
          if (lane == 0) {
            if (total == 0) mbar_arrive(&full_bar[j]);
            else mbar_expect_tx(&full_bar[j], total);
          }
          __syncwarp();
          if (nb) bulk_load(stage + ((size_t)j * I + lane) * TMA_CHUNK, src + j * TMA_CHUNK, nb, &full_bar[j]);
        }
      }
    }
    return;
  }

  if (warp > TMA_CONSUMERS / 32) {
    // ---------------- epilogue warps: warp ew finishes rows it = ew, ew + 4, ... from the partials in buffer it & 1
    const int ew = warp - TMA_CONSUMERS / 32 - 1;
    const int e = ew & 1;
    const float* pb = part + (size_t)e * PK * TMA_CONSUMERS;
    for (uint32_t it = ew; ; it += TMA_EPI_WARPS) {
      const long row = (long)blockIdx.x + (long)it * gridDim.x;
      if (row >= rows) break;
      const int b = (int)(row / T);
      // label-column gather first: it does not depend on the row reduction, so its DRAM latency hides behind the
      // consumers still streaming this row (S1 <= 32: one lattice column per lane)
      float lq = 0.f;
      bool lvalid = false;
      if (lpe && lane < S1) {
        const int L = min(tlen[b], Lmax);
        const long base = (row * S1 + lane) * I;
        const bool valid = (lane == 0) || (lane - 1 < L);
        int col = 0;
        if (lane > 0 && valid) col = (int)targets[(long)b * Lmax + lane - 1];
        lvalid = valid && col >= 0 && col < C;
        if (lvalid) {
#pragma unroll
          for (int i = 0; i < I; ++i) {
            const float gi = __ldg(gate + b * I + i);
            const float v = (col < P.C[i]) ? ((gi != 0.f) ? __ldg(P.z[i] + row * P.ld[i] + col) : 0.f) : 1.0f;
            lq = fmaf(gi, v, lq);
            if (zlab) zlab[base + i] = v;
          }
        } else if (zlab) {
#pragma unroll
          for (int i = 0; i < I; ++i) zlab[base + i] = 0.f;
        }
      }
      mbar_wait(&rowdone_bar[ew], (it / TMA_EPI_WARPS) & 1u);
      float m = -INFINITY, s = 0.f, best = -INFINITY;
      int besti = 0x7fffffff;
      float A[I];
#pragma unroll
      for (int i = 0; i < I; ++i) A[i] = 0.f;
      for (int k = lane; k < TMA_CONSUMERS; k += 32) {
        float A2[I];
#pragma unroll
        for (int i = 0; i < I; ++i) A2[i] = pb[(4 + i) * TMA_CONSUMERS + k];
        acc_merge<I>(m, s, A, best, besti, pb[k], pb[TMA_CONSUMERS + k], A2, pb[2 * TMA_CONSUMERS + k],
                     __float_as_int(pb[3 * TMA_CONSUMERS + k]));
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&partfree_bar[e]);             // partial buffer e may be rewritten (row it + 2)
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float m2 = __shfl_xor_sync(0xffffffffu, m, o);
        const float s2 = __shfl_xor_sync(0xffffffffu, s, o);
        const float b2 = __shfl_xor_sync(0xffffffffu, best, o);
        const int bi2 = __shfl_xor_sync(0xffffffffu, besti, o);
        float A2[I];
#pragma unroll
        for (int i = 0; i < I; ++i) A2[i] = __shfl_xor_sync(0xffffffffu, A[i], o);
        acc_merge<I>(m, s, A, best, besti, m2, s2, A2, b2, bi2);
      }
      const float lrow_lse = m + logf(s);                        // every lane holds the full reduction
      if (lane == 0) {
        lse[row] = lrow_lse;
        if (E) {
          const float inv = 1.0f / s;
#pragma unroll
          for (int i = 0; i < I; ++i) E[row * I + i] = A[i] * inv;
        }
        if (amax) amax[row] = besti;
        if (maxprob) maxprob[row] = __expf(best - lrow_lse);
      }
      if (lpe && lane < S1) lpe[row * S1 + lane] = lvalid ? lq - lrow_lse : -INFINITY;
    }
    return;
  }

  // ---------------- consumers (4 columns each per chunk)
  // the one 4-column group per expert that straddles its charset boundary: lanes >= C_i % 4 take the pad value again
  uint32_t smask = 0;                                            // chunks in which this thread owns a straddling group
#pragma unroll
  for (int i = 0; i < I; ++i) {
    const int Ci = P.C[i];
    if ((Ci & 3) != 0 && ((Ci % TMA_CHUNK) >> 2) == tid) smask |= 1u << (Ci / TMA_CHUNK);
  }
  uint32_t it = 0;
  float gn[I];                                                   // next row's gate, fetched one row ahead
#pragma unroll
  for (int i = 0; i < I; ++i) gn[i] = blockIdx.x < rows ? __ldg(gate + (blockIdx.x / T) * I + i) : 0.f;
  for (int row = blockIdx.x; row < rows; row += gridDim.x, ++it) {
    float g[I];
    bool hard = false;
#pragma unroll
    for (int i = 0; i < I; ++i) { g[i] = gn[i]; hard = hard || (g[i] == 0.f); }
    if (row + (int)gridDim.x < rows) {
      const int bn = (row + gridDim.x) / T;
#pragma unroll
      for (int i = 0; i < I; ++i) gn[i] = __ldg(gate + bn * I + i);
    }
    float m = -INFINITY, s = 0.f, best = -INFINITY;
    int besti = 0x7fffffff;
    float A[I];
#pragma unroll
    for (int i = 0; i < I; ++i) A[i] = 0.f;
    float* lrow = logits ? logits + (long)row * ldo : nullptr;

    for (int j = 0; j < nchunks; ++j) {
      mbar_wait(&full_bar[j], it & 1u);
      const int c0 = j * TMA_CHUNK + tid * 4;
      float4 v[I];
#pragma unroll
      for (int i = 0; i < I; ++i) v[i] = *reinterpret_cast<const float4*>(stage + ((size_t)j * I + i) * TMA_CHUNK + tid * 4);
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty_bar[j]);              // stage j may be refilled with the next row
      if ((smask >> j) & 1u) {                                 // rare: re-impose the pad on the copied ld padding
#pragma unroll
        for (int i = 0; i < I; ++i) {
          const int Ci = P.C[i], sn = Ci & 3;
          if (sn != 0 && ((Ci % TMA_CHUNK) >> 2) == tid && Ci / TMA_CHUNK == j) {
            if (sn <= 1) v[i].y = 1.0f;
            if (sn <= 2) v[i].z = 1.0f;
            v[i].w = 1.0f;
          }
        }
      }
      if (c0 >= C) continue;
      if (hard) {                                              // one-hot gate: unselected stages hold stale (finite) data
#pragma unroll
        for (int i = 0; i < I; ++i) if (g[i] == 0.f) v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
      float l0 = 0.f, l1 = 0.f, l2 = 0.f, l3 = 0.f;
#pragma unroll
      for (int i = 0; i < I; ++i) {
        l0 = fmaf(g[i], v[i].x, l0); l1 = fmaf(g[i], v[i].y, l1); l2 = fmaf(g[i], v[i].z, l2); l3 = fmaf(g[i], v[i].w, l3);
      }
      if (c0 + 4 <= C) {
        if (lrow) *reinterpret_cast<float4*>(lrow + c0) = make_float4(l0, l1, l2, l3);
        if (l0 > best) { best = l0; besti = c0; }
        if (l1 > best) { best = l1; besti = c0 + 1; }
        if (l2 > best) { best = l2; besti = c0 + 2; }
        if (l3 > best) { best = l3; besti = c0 + 3; }
        const float cm = fmaxf(fmaxf(l0, l1), fmaxf(l2, l3));
        if (cm > m) {
          const float f = ex2_approx((m - cm) * LOG2E);
          s *= f;
#pragma unroll
          for (int i = 0; i < I; ++i) A[i] *= f;
          m = cm;
        }
        const float mb = -m * LOG2E;
        const float e0 = ex2_approx(fmaf(l0, LOG2E, mb)), e1 = ex2_approx(fmaf(l1, LOG2E, mb));
        const float e2 = ex2_approx(fmaf(l2, LOG2E, mb)), e3 = ex2_approx(fmaf(l3, LOG2E, mb));
        s += (e0 + e1) + (e2 + e3);
#pragma unroll
        for (int i = 0; i < I; ++i) A[i] = fmaf(e0, v[i].x, fmaf(e1, v[i].y, fmaf(e2, v[i].z, fmaf(e3, v[i].w, A[i]))));
      } else {
        // the last, partial group of the row (C % 4 != 0)
        const float lv[4] = {l0, l1, l2, l3};
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          if (c0 + u < C) {
            float vv[I];
#pragma unroll
            for (int i = 0; i < I; ++i) vv[i] = u == 0 ? v[i].x : (u == 1 ? v[i].y : (u == 2 ? v[i].z : v[i].w));
            if (lrow) lrow[c0 + u] = lv[u];
            row_update<I>(lv[u], vv, c0 + u, m, s, A, best, besti);
          }
        }
      }
    }
    // ---- hand the per-thread partials to this row's epilogue warp and move on to the next row
    const int buf = it & 1u;
    mbar_wait(&partfree_bar[buf], ((it >> 1) & 1u) ^ 1u);
    float* pw = part + (size_t)buf * PK * TMA_CONSUMERS + tid;
    pw[0] = m; pw[TMA_CONSUMERS] = s; pw[2 * TMA_CONSUMERS] = best; pw[3 * TMA_CONSUMERS] = __int_as_float(besti);
#pragma unroll
    for (int i = 0; i < I; ++i) pw[(4 + i) * TMA_CONSUMERS] = A[i];
    __syncwarp();
    if (lane == 0) mbar_arrive(&rowdone_bar[it % TMA_EPI_WARPS]);
  }
}

// ---------------------------------------------------------------------------------------------
// Backward of the gated combine for a dense upstream gradient dY [B,T,C]:
//   dgate[b,i] = sum_{t, c<C} dY[b,t,c] * pad_i[b,t,c],   pad_i = z_i below C_i and 1.0 past it.
// The logits do not depend on the gate beyond this product, so the gate itself is not an input.
//
// Persistent like combine_row_tma_kernel: one CTA per SM walks rows r = blockIdx.x, blockIdx.x + gridDim.x, ...  A
// producer warp streams each row in chunks of BWD_CHUNK columns through a ring of stages ([I + 1][BWD_CHUNK] floats:
// the I expert slices, then dY) with 1-D bulk copies on mbarriers; lane i copies expert i's slice, lane I the dY slice.
// Every expert is loaded whatever its gate (a zero-gate expert still has a gradient); a slice past an expert's charset
// is not copied and reads as the pad value.  Each consumer thread owns 4 columns of a chunk and keeps I running dot
// products; a row's partials are reduced in a fixed order (warp shuffles, then warp 0 over the warps) into
// rowout[row, I], and a second kernel sums the T rows of each sample in order: no atomics, the same bits every run.
// ---------------------------------------------------------------------------------------------
constexpr int BWD_CONSUMERS = 512;
constexpr int BWD_CHUNK = 4 * BWD_CONSUMERS;
constexpr int BWD_MAX_STAGES = 4;
constexpr int BWD_THREADS = BWD_CONSUMERS + 32;
constexpr size_t BWD_SMEM_BUDGET = 200 * 1024;

template <int I>
__global__ void __launch_bounds__(BWD_THREADS, 1)
combine_bwd_tma_kernel(RowPtrs P, const float* __restrict__ dY, long ldy, int C, int rows, int nchunks, int nstages,
                       float* __restrict__ rowout) {
  extern __shared__ __align__(128) float stage[];              // [nstages][I + 1][BWD_CHUNK]
  __shared__ __align__(8) uint64_t full_bar[BWD_MAX_STAGES], empty_bar[BWD_MAX_STAGES];
  __shared__ float part[2][BWD_CONSUMERS / 32][I];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  constexpr size_t SLOT = (size_t)(I + 1) * BWD_CHUNK;
  if (tid == 0) {
    for (int s = 0; s < nstages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], BWD_CONSUMERS / 32); }
    fence_mbarrier_init();
  }
  __syncthreads();

  if (warp == BWD_CONSUMERS / 32) {
    // ---------------- producer warp
    const int myC = lane < I ? P.C[lane] : C;
    const long myld = lane < I ? P.ld[lane] : ldy;
    const float* myz = lane < I ? P.z[lane] : dY;
    uint32_t q = 0;
    for (int row = blockIdx.x; row < rows; row += gridDim.x) {
      const float* src = myz + (long)row * myld;
      for (int j = 0; j < nchunks; ++j, ++q) {
        const int s = (int)(q % (uint32_t)nstages);
        uint32_t total = 0;
#pragma unroll
        for (int i = 0; i <= I; ++i) {
          int n = (i < I ? P.C[i] : C) - j * BWD_CHUNK;
          n = n < 0 ? 0 : (n > BWD_CHUNK ? BWD_CHUNK : n);
          total += (uint32_t)((n + 3) & ~3) * 4u;                 // whole 16-byte pieces (ld is padded to 4)
        }
        int n = myC - j * BWD_CHUNK;
        n = n < 0 ? 0 : (n > BWD_CHUNK ? BWD_CHUNK : n);
        const uint32_t nb = lane <= I ? (uint32_t)((n + 3) & ~3) * 4u : 0u;
        mbar_wait(&empty_bar[s], ((q / (uint32_t)nstages) & 1u) ^ 1u);
        if (lane == 0) mbar_expect_tx(&full_bar[s], total);        // total > 0: the dY slice of chunk j < nchunks
        __syncwarp();
        if (nb) bulk_load(stage + s * SLOT + (size_t)lane * BWD_CHUNK, src + (long)j * BWD_CHUNK, nb, &full_bar[s]);
      }
    }
    return;
  }

  // ---------------- consumers (4 columns each per chunk)
  uint32_t q = 0, it = 0;
  for (int row = blockIdx.x; row < rows; row += gridDim.x, ++it) {
    float acc[I];
#pragma unroll
    for (int i = 0; i < I; ++i) acc[i] = 0.f;
    for (int j = 0; j < nchunks; ++j, ++q) {
      const int s = (int)(q % (uint32_t)nstages);
      mbar_wait(&full_bar[s], (q / (uint32_t)nstages) & 1u);
      const float* st = stage + s * SLOT + tid * 4;
      const int c0 = j * BWD_CHUNK + tid * 4;
      float4 dy = make_float4(0.f, 0.f, 0.f, 0.f);
      float4 v[I];
#pragma unroll
      for (int i = 0; i < I; ++i) {
        v[i] = make_float4(1.f, 1.f, 1.f, 1.f);
        if (c0 < P.C[i]) v[i] = *reinterpret_cast<const float4*>(st + (size_t)i * BWD_CHUNK);
      }
      if (c0 < C) dy = *reinterpret_cast<const float4*>(st + (size_t)I * BWD_CHUNK);
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty_bar[s]);                 // stage s may be refilled
      if (c0 >= C) continue;
      if (c0 + 4 > C) {                                          // the row's last, partial group: ld padding is not dY
        if (c0 + 1 >= C) dy.y = 0.f;
        if (c0 + 2 >= C) dy.z = 0.f;
        dy.w = 0.f;
      }
      const float sdy = (dy.x + dy.y) + (dy.z + dy.w);
#pragma unroll
      for (int i = 0; i < I; ++i) {
        const int Ci = P.C[i];
        if (c0 >= Ci) {
          acc[i] += sdy;                                         // pad value 1.0
        } else {
          if (c0 + 4 > Ci) {                                     // the group straddling C_i: re-impose the pad
            if (c0 + 1 >= Ci) v[i].y = 1.f;
            if (c0 + 2 >= Ci) v[i].z = 1.f;
            v[i].w = 1.f;
          }
          acc[i] = fmaf(dy.x, v[i].x, fmaf(dy.y, v[i].y, fmaf(dy.z, v[i].z, fmaf(dy.w, v[i].w, acc[i]))));
        }
      }
    }
    // ---- row reduction in a fixed order: warp tree, then warp 0 over the consumer warps (double-buffered partials)
#pragma unroll
    for (int i = 0; i < I; ++i) acc[i] = warp_sum(acc[i]);
    const int buf = it & 1u;
    if (lane == 0) {
#pragma unroll
      for (int i = 0; i < I; ++i) part[buf][warp][i] = acc[i];
    }
    asm volatile("bar.sync 1, %0;" ::"r"(BWD_CONSUMERS) : "memory");
    if (warp == 0 && lane < I) {
      float sum = 0.f;
#pragma unroll
      for (int w = 0; w < BWD_CONSUMERS / 32; ++w) sum += part[buf][w][lane];
      rowout[(long)row * I + lane] = sum;
    }
  }
}

// dgate[b,i] = sum_t rowout[b,t,i], t ascending
__global__ void combine_bwd_finish_kernel(const float* __restrict__ rowout, int B, int T, int I, float* __restrict__ dgate) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= B * I) return;
  const int b = k / I, i = k - b * I;
  float s = 0.f;
  for (int t = 0; t < T; ++t) s += rowout[((long)b * T + t) * I + i];
  dgate[k] = s;
}

// ---------------------------------------------------------------------------------------------
// CTC lattice: one warp per sequence; lane l owns states 2l (blank) and 2l+1 (label l+1).
// ---------------------------------------------------------------------------------------------
constexpr int CTC_WARPS = 4;

__global__ void __launch_bounds__(CTC_WARPS * 32)
ctc_lattice_kernel(const float* __restrict__ lpe,    // [B,T,S1]
                   const float* __restrict__ zlab,   // optional [B,T,S1,I]
                   const float* __restrict__ E,      // optional [B,T,I]
                   const long long* __restrict__ targets, const int* __restrict__ tlen, int Lmax,
                   int B, int T, int S1, int I, float grad_scale,   // pi / B
                   float* __restrict__ nll,          // [B]
                   float* __restrict__ dgate,        // optional [B,I]  (CTC part of dL/dgate)
                   float* __restrict__ occ_col) {    // optional [B,T,S1] posterior mass per label column
  extern __shared__ float smem[];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * CTC_WARPS + w;
  if (b >= B) return;
  float* s_lp = smem + (size_t)w * (T * S1 + T * 64);
  float* s_alpha = s_lp + T * S1;
  const float* lp_b = lpe + (long)b * T * S1;
  for (int k = lane; k < T * S1; k += 32) s_lp[k] = lp_b[k];
  const int L = min(tlen[b], Lmax);
  const int S = 2 * L + 1;
  const int s0 = 2 * lane, s1 = 2 * lane + 1;
  const bool v0 = s0 < S, v1 = s1 < S;
  long long lab = -1, labp = -2;
  if (v1) lab = targets[(long)b * Lmax + lane];
  labp = __shfl_up_sync(0xffffffffu, lab, 1);
  const bool skip1 = v1 && lane > 0 && lab != labp;   // s1 may come from s1-2 (previous label)
  const int col1 = lane + 1;
  __syncwarp();

  float a0 = -INFINITY, a1 = -INFINITY;
  if (lane == 0) { a0 = s_lp[0]; if (v1) a1 = s_lp[col1]; }
  s_alpha[0 * 64 + s0] = a0; s_alpha[0 * 64 + s1] = a1;
  for (int t = 1; t < T; ++t) {
    const float p1 = __shfl_up_sync(0xffffffffu, a1, 1);      // alpha[t-1][s0-1] == alpha[t-1][s1-2]
    const float prev1 = (lane > 0) ? p1 : -INFINITY;
    const float lb = s_lp[t * S1], ll_ = (col1 < S1) ? s_lp[t * S1 + col1] : -INFINITY;
    float n0 = log_add(a0, prev1);
    float n1 = log_add(a1, a0);
    if (skip1) n1 = log_add(n1, prev1);
    a0 = v0 ? n0 + lb : -INFINITY;
    a1 = v1 ? n1 + ll_ : -INFINITY;
    s_alpha[t * 64 + s0] = a0; s_alpha[t * 64 + s1] = a1;
  }
  // total log-likelihood: states S-1 (blank, lane L) and S-2 (label L, lane L-1)
  float e_last = __shfl_sync(0xffffffffu, a0, L);
  float e_prev = (L > 0) ? __shfl_sync(0xffffffffu, a1, L - 1) : -INFINITY;
  const float ll = log_add(e_last, e_prev);
  // zero_infinity=True zeroes only an infinite loss (ll == -inf: no valid alignment), exactly like torch.nn.CTCLoss;
  // a NaN log-likelihood (non-finite logits upstream) must stay visible in the loss and in the gradient.
  const bool feasible = (ll != -INFINITY);
  if (lane == 0) nll[b] = feasible ? -ll : 0.f;
  if (!dgate && !occ_col) return;

  const float scale = feasible ? grad_scale / (float)max(L, 1) : 0.f;
  float acc[MRNB_MAX_EXPERTS];
#pragma unroll
  for (int i = 0; i < MRNB_MAX_EXPERTS; ++i) acc[i] = 0.f;
  // beta, walking backwards; occupancy on the fly
  const bool skipn = __shfl_down_sync(0xffffffffu, (int)skip1, 1) && lane < 31;   // s1 -> s1+2 allowed
  float b0 = -INFINITY, b1 = -INFINITY;
  {
    const int t = T - 1;
    if (lane == L) b0 = s_lp[t * S1];
    if (L > 0 && lane == L - 1) b1 = s_lp[t * S1 + col1];
  }
  for (int t = T - 1; t >= 0; --t) {
    const float lb = s_lp[t * S1], ll_ = (col1 < S1) ? s_lp[t * S1 + col1] : -INFINITY;
    if (t < T - 1) {
      const float nb0 = __shfl_down_sync(0xffffffffu, b0, 1);   // beta[t+1][s1+1]
      const float nb1 = __shfl_down_sync(0xffffffffu, b1, 1);   // beta[t+1][s1+2]
      const float x0 = (lane < 31) ? nb0 : -INFINITY;
      const float x1 = (lane < 31) ? nb1 : -INFINITY;
      float n0 = log_add(b0, b1);                 // blank: stay or step to own label state
      float n1 = log_add(b1, x0);                 // label: stay or step to next blank
      if (skipn) n1 = log_add(n1, x1);
      b0 = v0 ? n0 + lb : -INFINITY;
      b1 = v1 ? n1 + ll_ : -INFINITY;
    }
    if (feasible) {
      const float al0 = s_alpha[t * 64 + s0], al1 = s_alpha[t * 64 + s1];
      const float o0 = (v0 && al0 != -INFINITY && b0 != -INFINITY) ? __expf(al0 + b0 - lb - ll) : 0.f;
      const float o1 = (v1 && al1 != -INFINITY && b1 != -INFINITY) ? __expf(al1 + b1 - ll_ - ll) : 0.f;
      if (dgate) {
        const float* zl = zlab + ((long)(b * T + t) * S1) * I;
        for (int i = 0; i < I; ++i) {
          float c = o0 * zl[i];
          if (v1) c = fmaf(o1, zl[(long)col1 * I + i], c);
          acc[i] += c;
        }
      }
      if (occ_col) {
        const float ob = warp_sum(o0);
        if (lane == 0) occ_col[(long)(b * T + t) * S1] = ob;
        if (col1 < S1) occ_col[(long)(b * T + t) * S1 + col1] = o1;
      }
    } else if (occ_col) {
      if (lane == 0) occ_col[(long)(b * T + t) * S1] = 0.f;
      if (col1 < S1) occ_col[(long)(b * T + t) * S1 + col1] = 0.f;
    }
  }
  if (dgate) {
    for (int i = 0; i < I; ++i) {
      float es = 0.f;
      for (int t = lane; t < T; t += 32) es += E[(long)(b * T + t) * I + i];
      const float tot = warp_sum(es) - warp_sum(acc[i]);
      if (lane == 0) dgate[b * I + i] = scale * tot;
    }
  }
}

// loss = mean_b(nll_b / max(len_b,1))   (CTCLoss reduction='mean')
__global__ void ctc_mean_kernel(const float* __restrict__ nll, const int* __restrict__ tlen, int B, int Lmax,
                                float* __restrict__ loss) {
  __shared__ double sh[32];
  double v = 0.0;
  for (int b = threadIdx.x; b < B; b += blockDim.x) v += (double)nll[b] / (double)max(min(tlen[b], Lmax), 1);
  v = warp_sum_d(v);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int k = 0; k < (int)(blockDim.x >> 5); ++k) t += sh[k];
    loss[0] = (float)(t / (double)B);
  }
}

// Dense gradient of mean-CTC w.r.t. logits: G = scale_b * (softmax - occupancy).  One CTA per row.
__global__ void __launch_bounds__(ROW_THREADS)
ctc_dense_grad_kernel(const float* __restrict__ logits, long ldl, const float* __restrict__ lse,
                      const float* __restrict__ occ_col, const float* __restrict__ nll,
                      const long long* __restrict__ targets, const int* __restrict__ tlen, int Lmax,
                      int T, int C, int S1, float grad_scale, float* __restrict__ grad, long ldg) {
  const int row = blockIdx.x, b = row / T;
  const int L = min(tlen[b], Lmax);
  // infeasible samples have nll == 0 exactly AND zero occupancy everywhere -> zero gradient (zero_infinity)
  float occ0 = occ_col[(long)row * S1];
  bool feasible = true;
  {
    __shared__ float tot;
    if (threadIdx.x == 0) {
      float s = 0.f;
      for (int j = 0; j <= L && j < S1; ++j) s += occ_col[(long)row * S1 + j];
      tot = s;
    }
    __syncthreads();
    feasible = !(tot <= 0.5f);  // occupancies of a feasible row sum to 1; NaN occupancies (NaN loss) stay "feasible" and propagate
  }
  (void)occ0; (void)nll;
  const float scale = feasible ? grad_scale / (float)max(L, 1) : 0.f;
  const float l = lse[row];
  for (int c = threadIdx.x; c < C; c += ROW_THREADS)
    grad[(long)row * ldg + c] = scale * __expf(logits[(long)row * ldl + c] - l);
  __syncthreads();
  if (threadIdx.x == 0 && feasible) {
    grad[(long)row * ldg] -= scale * occ_col[(long)row * S1];
    for (int j = 1; j <= L && j < S1; ++j) {
      const int col = (int)targets[(long)b * Lmax + j - 1];
      if (col >= 0 && col < C) grad[(long)row * ldg + col] -= scale * occ_col[(long)row * S1 + j];
    }
  }
}

// Greedy CTC decode: one warp per sample.
__global__ void greedy_decode_kernel(const int* __restrict__ amax, const float* __restrict__ maxprob, int B, int T,
                                     int* __restrict__ out_ids, int* __restrict__ out_len, float* __restrict__ conf) {
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (b >= B) return;
  int n = 0;
  float p = 1.f;
  for (int t0 = 0; t0 < T; t0 += 32) {
    const int t = t0 + lane;
    int id = 0, prev = -1;
    if (t < T) {
      id = amax[b * T + t];
      prev = (t > 0) ? amax[b * T + t - 1] : -1;
      p *= maxprob[b * T + t];
    }
    const bool keep = (t < T) && id != 0 && id != prev;
    const unsigned mask = __ballot_sync(0xffffffffu, keep);
    if (keep) out_ids[b * T + n + __popc(mask & ((1u << lane) - 1u))] = id;
    n += __popc(mask);
  }
  for (int k = n + lane; k < T; k += 32) out_ids[b * T + k] = -1;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) p *= __shfl_xor_sync(0xffffffffu, p, o);
  if (lane == 0) { out_len[b] = n; conf[b] = p; }
}

template <int I>
int launch_combine(const RowPtrs& P, const float* gate, int B, int T, int C, float* logits, long ldo, float* lse,
                   float* E, int* amax, float* maxprob, const long long* targets, const int* tlen, int Lmax,
                   float* lpe, float* zlab, int S1, cudaStream_t st) {
  int fast = 1;
  for (int i = 0; i < I; ++i) {
    fast = fast && (P.ld[i] % 4 == 0) && ((reinterpret_cast<uintptr_t>(P.z[i]) & 15) == 0) && (i == 0 || P.C[i] >= P.C[i - 1]);
  }
  fast = fast && P.C[I - 1] == C && (!logits || (ldo % 4 == 0 && (reinterpret_cast<uintptr_t>(logits) & 15) == 0));
  const int nchunks = (C + TMA_CHUNK - 1) / TMA_CHUNK;
  const size_t smem = ((size_t)nchunks * I * TMA_CHUNK + 2 * (4 + I) * TMA_CONSUMERS) * sizeof(float);
  static int use_tma = -1;
  if (use_tma < 0) { const char* e = getenv("MRNB_COMBINE_TMA"); use_tma = (e && e[0] == '0') ? 0 : 1; }
  if (fast && use_tma && nchunks <= TMA_MAX_CHUNKS && smem <= 220 * 1024) {
    static bool attr_set = false;
    static int num_sms = 148;
    if (!attr_set) {
      cudaFuncSetAttribute(combine_row_tma_kernel<I>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024);
      int dev = 0;
      cudaGetDevice(&dev);
      cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
      attr_set = true;
    }
    const int rows = B * T;
    const int grid = rows < num_sms ? rows : num_sms;
    combine_row_tma_kernel<I><<<grid, TMA_THREADS, smem, st>>>(P, gate, T, C, rows, nchunks, logits, ldo, lse, E, amax,
                                                                       maxprob, targets, tlen, Lmax, lpe, zlab, S1);
    MRNB_CHECK_LAUNCH("combine_row_tma_kernel");
    return MRNB_OK;
  }
  combine_row_kernel<I><<<B * T, ROW_THREADS, 0, st>>>(P, gate, T, C, fast, logits, ldo, lse, E, amax, maxprob, targets,
                                                         tlen, Lmax, lpe, zlab, S1);
  MRNB_CHECK_LAUNCH("combine_row_kernel");
  return MRNB_OK;
}

template <int I>
int launch_combine_bwd(const RowPtrs& P, const float* dY, long ldy, int B, int T, int C, float* dgate, float* rowout,
                       cudaStream_t st) {
  const int nchunks = (C + BWD_CHUNK - 1) / BWD_CHUNK;
  const size_t slot_bytes = (size_t)(I + 1) * BWD_CHUNK * sizeof(float);
  const int nstages = (int)(BWD_SMEM_BUDGET / slot_bytes) < BWD_MAX_STAGES ? (int)(BWD_SMEM_BUDGET / slot_bytes) : BWD_MAX_STAGES;
  static bool attr_set = false;
  static int num_sms = 148;
  if (!attr_set) {
    cudaFuncSetAttribute(combine_bwd_tma_kernel<I>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)BWD_SMEM_BUDGET);
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
    attr_set = true;
  }
  const int rows = B * T;
  const int grid = rows < num_sms ? rows : num_sms;
  combine_bwd_tma_kernel<I><<<grid, BWD_THREADS, nstages * slot_bytes, st>>>(P, dY, ldy, C, rows, nchunks, nstages, rowout);
  MRNB_CHECK_LAUNCH("combine_bwd_tma_kernel");
  combine_bwd_finish_kernel<<<cdiv(B * I, 256), 256, 0, st>>>(rowout, B, T, I, dgate);
  MRNB_CHECK_LAUNCH("combine_bwd_finish_kernel");
  return MRNB_OK;
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// C-ABI (declared in include/mrn_b200.h)
// ---------------------------------------------------------------------------------------------
extern "C" int mrnb_gate_combine(const float* const* z, const long* ld, const int* Ci, int n_experts,
                                 const float* gate, int B, int T,
                                 float* logits, long ldo, float* lse, float* E, int* amax, float* maxprob,
                                 const long long* targets, const int* tlen, int Lmax, float* lpe, float* zlab,
                                 cudaStream_t stream) {
  MRNB_CHECK_ARG(n_experts >= 1 && n_experts <= MRNB_MAX_EXPERTS, "gate_combine: n_experts %d out of range", n_experts);
  MRNB_CHECK_ARG(B > 0 && T > 0 && z && ld && Ci && gate && lse, "gate_combine: null/empty argument");
  MRNB_CHECK_ARG(!lpe || (targets && tlen && Lmax >= 0 && Lmax + 1 <= S1_MAX), "gate_combine: Lmax %d unsupported", Lmax);
  RowPtrs P;
  for (int i = 0; i < n_experts; ++i) {
    P.z[i] = z[i]; P.ld[i] = ld[i]; P.C[i] = Ci[i];
    MRNB_CHECK_ARG(z[i] && Ci[i] > 0 && ld[i] >= Ci[i] && Ci[i] <= Ci[n_experts - 1], "gate_combine: bad expert %d", i);
  }
  const int C = Ci[n_experts - 1];
  MRNB_CHECK_ARG(!logits || ldo >= C, "gate_combine: ldo < C");
  const int S1 = Lmax + 1;
  double rb = 0;
  for (int i = 0; i < n_experts; ++i) rb += (double)Ci[i];
  MrnbProfScope prof(MRNB_PROF_COMBINE, stream, 0.0, 4.0 * B * T * (rb + (logits ? C : 0)));
#define MRNB_CASE(N) case N: return launch_combine<N>(P, gate, B, T, C, logits, ldo, lse, E, amax, maxprob, targets, tlen, Lmax, lpe, zlab, S1, stream);
  switch (n_experts) {
    MRNB_CASE(1) MRNB_CASE(2) MRNB_CASE(3) MRNB_CASE(4) MRNB_CASE(5) MRNB_CASE(6) MRNB_CASE(7) MRNB_CASE(8)
  }
#undef MRNB_CASE
  return MRNB_ERR_ARG;
}

extern "C" size_t mrnb_gate_combine_backward_workspace_bytes(int B, int T, int n_experts) {
  return (size_t)B * T * n_experts * sizeof(float);
}

extern "C" int mrnb_gate_combine_backward(const float* const* z, const long* ld, const int* Ci, int n_experts, int B, int T,
                                          const float* dY, long ldy, float* dgate, void* workspace,
                                          size_t workspace_bytes, cudaStream_t stream) {
  MRNB_CHECK_ARG(n_experts >= 1 && n_experts <= MRNB_MAX_EXPERTS, "gate_combine_backward: n_experts %d out of range",
                 n_experts);
  MRNB_CHECK_ARG(B > 0 && T > 0 && z && ld && Ci && dY && dgate && workspace, "gate_combine_backward: null/empty argument");
  const int C = Ci[n_experts - 1];
  RowPtrs P;
  for (int i = 0; i < n_experts; ++i) {
    P.z[i] = z[i]; P.ld[i] = ld[i]; P.C[i] = Ci[i];
    MRNB_CHECK_ARG(z[i] && Ci[i] > 0 && Ci[i] <= C && ld[i] >= Ci[i] && ld[i] % 4 == 0 &&
                   (reinterpret_cast<uintptr_t>(z[i]) & 15) == 0,
                   "gate_combine_backward: expert %d needs C_i <= C, a 16-byte aligned base and ld %% 4 == 0", i);
  }
  MRNB_CHECK_ARG(ldy >= C && ldy % 4 == 0 && (reinterpret_cast<uintptr_t>(dY) & 15) == 0,
                 "gate_combine_backward: dY needs ldy >= C, ldy %% 4 == 0 and a 16-byte aligned base");
  MRNB_CHECK_ARG(workspace_bytes >= mrnb_gate_combine_backward_workspace_bytes(B, T, n_experts),
                 "gate_combine_backward: workspace too small (%zu bytes)", workspace_bytes);
  double rb = C;
  for (int i = 0; i < n_experts; ++i) rb += (double)Ci[i];
  MrnbProfScope prof(MRNB_PROF_COMBINE, stream, 0.0, 4.0 * B * T * rb);
  float* rowout = static_cast<float*>(workspace);
#define MRNB_CASE(N) case N: return launch_combine_bwd<N>(P, dY, ldy, B, T, C, dgate, rowout, stream);
  switch (n_experts) {
    MRNB_CASE(1) MRNB_CASE(2) MRNB_CASE(3) MRNB_CASE(4) MRNB_CASE(5) MRNB_CASE(6) MRNB_CASE(7) MRNB_CASE(8)
  }
#undef MRNB_CASE
  return MRNB_ERR_ARG;
}

extern "C" int mrnb_ctc_lattice(const float* lpe, const float* zlab, const float* E, const long long* targets,
                                const int* tlen, int Lmax, int B, int T, int n_experts, float grad_scale,
                                float* nll, float* loss_mean, float* dgate, float* occ_col, cudaStream_t stream) {
  MRNB_CHECK_ARG(lpe && targets && tlen && nll && B > 0 && T > 0, "ctc_lattice: null/empty argument");
  MRNB_CHECK_ARG(Lmax >= 0 && Lmax + 1 <= S1_MAX, "ctc_lattice: Lmax %d unsupported (max %d)", Lmax, S1_MAX - 1);
  MRNB_CHECK_ARG(!dgate || (zlab && E && n_experts >= 1 && n_experts <= MRNB_MAX_EXPERTS), "ctc_lattice: dgate needs zlab and E");
  const int S1 = Lmax + 1;
  const size_t smem = (size_t)CTC_WARPS * (T * S1 + T * 64) * sizeof(float);
  MRNB_CHECK_ARG(smem <= 200 * 1024, "ctc_lattice: T=%d too long for the shared-memory lattice", T);
  static bool attr_set = false;
  if (!attr_set) {
    cudaFuncSetAttribute(ctc_lattice_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    attr_set = true;
  }
  MrnbProfScope prof(MRNB_PROF_CTC, stream);
  ctc_lattice_kernel<<<cdiv(B, CTC_WARPS), CTC_WARPS * 32, smem, stream>>>(lpe, zlab, E, targets, tlen, Lmax, B, T, S1,
                                                                             n_experts, grad_scale, nll, dgate, occ_col);
  MRNB_CHECK_LAUNCH("ctc_lattice_kernel");
  if (loss_mean) {
    ctc_mean_kernel<<<1, 256, 0, stream>>>(nll, tlen, B, Lmax, loss_mean);
    MRNB_CHECK_LAUNCH("ctc_mean_kernel");
  }
  return MRNB_OK;
}

extern "C" int mrnb_ctc_dense_grad(const float* logits, long ldl, const float* lse, const float* occ_col,
                                   const float* nll, const long long* targets, const int* tlen, int Lmax, int B, int T,
                                   int C, float grad_scale, float* grad, long ldg, cudaStream_t stream) {
  MRNB_CHECK_ARG(logits && lse && occ_col && targets && tlen && grad && B > 0 && T > 0 && C > 0, "ctc_dense_grad: bad argument");
  MRNB_CHECK_ARG(ldl >= C && ldg >= C && Lmax + 1 <= S1_MAX, "ctc_dense_grad: bad leading dimension");
  ctc_dense_grad_kernel<<<B * T, ROW_THREADS, 0, stream>>>(logits, ldl, lse, occ_col, nll, targets, tlen, Lmax, T, C,
                                                            Lmax + 1, grad_scale, grad, ldg);
  MRNB_CHECK_LAUNCH("ctc_dense_grad_kernel");
  return MRNB_OK;
}

extern "C" int mrnb_greedy_decode(const int* amax, const float* maxprob, int B, int T, int* out_ids, int* out_len,
                                  float* conf, cudaStream_t stream) {
  MRNB_CHECK_ARG(amax && maxprob && out_ids && out_len && conf && B > 0 && T > 0, "greedy_decode: bad argument");
  greedy_decode_kernel<<<cdiv(B, 4), 128, 0, stream>>>(amax, maxprob, B, T, out_ids, out_len, conf);
  MRNB_CHECK_LAUNCH("greedy_decode_kernel");
  return MRNB_OK;
}
