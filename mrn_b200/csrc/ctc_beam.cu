// CTC prefix beam search on the device: N-best decoding of the hard-routed (or any gated) combine.
//
// No counterpart in the reference, which decodes greedily (test.py:211-221, mrnb_greedy_decode here).  Two kernels:
//   ctc_topk_kernel  per (b,t) row, the K best non-blank classes of the combined logits, recomputed from the ragged
//                    expert table with the combine's own expression (so the union-charset row [B,T,C] is never
//                    materialised), as log-probs against the combine's lse;
//   ctc_beam_kernel  one warp per sample: CTC prefix beam search over those candidates, prefixes held in a
//                    (parent, label) trie in shared memory.
#include "common.cuh"

namespace {

constexpr int TOPK_WARPS = 8;     // one warp per row
constexpr int TOPK_UNROLL = 4;    // 4-column groups per lane and expert loaded before any is used
constexpr int MAX_K = 32;         // candidates per frame
constexpr int MAX_W = 32;         // beam width (one beam entry per lane)
constexpr int MAX_T = 128;

struct ExpertTable {
  const float* z[MRNB_MAX_EXPERTS];
  long ld[MRNB_MAX_EXPERTS];
  int C[MRNB_MAX_EXPERTS];
};

// Order-preserving image of a (non-NaN) float as an unsigned integer, and its inverse.
__device__ __forceinline__ uint32_t f2ord(float f) {
  const uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord2f(uint32_t o) { return __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o); }

// Candidate key: value in the high word, ~tie in the low word, so that a larger key is the better candidate and an
// equal value goes to the smaller tie code.  0 is "no candidate" (no real value maps to it).
__device__ __forceinline__ uint64_t make_key(float v, uint32_t tie) { return ((uint64_t)f2ord(v) << 32) | (uint32_t)~tie; }

// The best key over the warp (every lane gets it).
__device__ __forceinline__ uint64_t warp_max_key(uint64_t k) {
  const uint32_t hi = (uint32_t)(k >> 32), lo = (uint32_t)k;
  const uint32_t mhi = __reduce_max_sync(0xffffffffu, hi);
  const uint32_t mlo = __reduce_max_sync(0xffffffffu, hi == mhi ? lo : 0u);
  return ((uint64_t)mhi << 32) | mlo;
}

// 4 consecutive columns c0.. of one expert row, the pad value 1.0 past its charset (no load there).
__device__ __forceinline__ float4 load_group(const float* __restrict__ z, int c0, int Ci, bool vec) {
  if (vec && c0 + 4 <= Ci) return __ldg(reinterpret_cast<const float4*>(z + c0));
  float4 r;
  r.x = c0 < Ci ? __ldg(z + c0) : 1.0f;
  r.y = c0 + 1 < Ci ? __ldg(z + c0 + 1) : 1.0f;
  r.z = c0 + 2 < Ci ? __ldg(z + c0 + 2) : 1.0f;
  r.w = c0 + 3 < Ci ? __ldg(z + c0 + 3) : 1.0f;
  return r;
}

template <int KP>
__device__ __forceinline__ void list_insert(uint64_t (&key)[KP], uint64_t x) {   // key[] sorted descending
#pragma unroll
  for (int j = 0; j < KP; ++j) {
    const uint64_t k = key[j];
    key[j] = k > x ? k : x;
    x = k > x ? x : k;
  }
}

// One warp per (b,t) row.  Each lane keeps its KP >= K best (value, class) keys in registers, sorted; a warp-wide bound
// (the largest of the lanes' KP-th keys: that lane alone holds KP keys above it) rejects almost every column with one
// float compare.  The K best of the 32 lists are then drawn one at a time.  The combined value is the combine's
// expression, l = fma(g_i, v_i, l) over experts in order from l = +0; an expert with a zero gate adds exactly +0 to a
// sum that is never -0, so skipping it (and its loads) changes no bit.
template <int I, int KP>
__global__ void __launch_bounds__(TOPK_WARPS * 32, 1)
ctc_topk_kernel(ExpertTable P, const float* __restrict__ gate, const float* __restrict__ lse, int rows, int T, int C, int K,
                int vec, int* __restrict__ top_ids, float* __restrict__ top_lp, float* __restrict__ blank_lp) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * TOPK_WARPS + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int b = row / T;
  float g[I];
  const float* zr[I];
#pragma unroll
  for (int i = 0; i < I; ++i) {
    g[i] = __ldg(gate + (long)b * I + i);
    zr[i] = P.z[i] + (long)row * P.ld[i];
  }
  uint64_t key[KP];
#pragma unroll
  for (int j = 0; j < KP; ++j) key[j] = 0;
  float bound = -INFINITY;        // value part of the warp-wide bound
  float blank = 0.f;
  for (int base = 0; base < C; base += 128 * TOPK_UNROLL) {
    float l[TOPK_UNROLL][4];
#pragma unroll
    for (int u = 0; u < TOPK_UNROLL; ++u) l[u][0] = l[u][1] = l[u][2] = l[u][3] = 0.f;
#pragma unroll
    for (int i = 0; i < I; ++i) {
      if (g[i] == 0.f) continue;
      float4 v[TOPK_UNROLL];
#pragma unroll
      for (int u = 0; u < TOPK_UNROLL; ++u) v[u] = load_group(zr[i], base + 128 * u + 4 * lane, P.C[i], vec != 0);
#pragma unroll
      for (int u = 0; u < TOPK_UNROLL; ++u) {
        l[u][0] = fmaf(g[i], v[u].x, l[u][0]);
        l[u][1] = fmaf(g[i], v[u].y, l[u][1]);
        l[u][2] = fmaf(g[i], v[u].z, l[u][2]);
        l[u][3] = fmaf(g[i], v[u].w, l[u][3]);
      }
    }
#pragma unroll
    for (int u = 0; u < TOPK_UNROLL; ++u) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int c = base + 128 * u + 4 * lane + e;
        const float v = l[u][e];
        if (c < C && !(v < bound)) {
          const uint64_t k = make_key(v, (uint32_t)c);
          if (c == 0) blank = v;
          else if (k > key[KP - 1]) list_insert<KP>(key, k);
        }
      }
    }
    const uint64_t wb = warp_max_key(key[KP - 1]);
    bound = wb ? ord2f((uint32_t)(wb >> 32)) : -INFINITY;
  }
  uint64_t mine = 0;
  for (int r = 0; r < K; ++r) {
    const uint64_t best = warp_max_key(key[0]);
    if (best == 0) break;
    if (lane == r) mine = best;
    if (key[0] == best) {
#pragma unroll
      for (int j = 0; j < KP - 1; ++j) key[j] = key[j + 1];
      key[KP - 1] = 0;
    }
  }
  const float ls = lse[row];
  if (lane < K) {
    top_ids[(long)row * K + lane] = mine ? (int)~(uint32_t)mine : -1;
    top_lp[(long)row * K + lane] = mine ? ord2f((uint32_t)(mine >> 32)) - ls : -INFINITY;
  }
  if (lane == 0) blank_lp[row] = blank - ls;
}

// Shared memory of one sample's beam search.
struct BeamSmem {
  uint64_t* cand;        // [W*K + W] candidate keys of the frame: extensions q = j*K + k, then stays W*K + j
  int *parent, *label, *child, *sibling, *stamp, *depth;   // trie nodes [1 + T*W]; node 0 is the empty prefix
  int* f_id;             // [MAX_K] the frame's candidate classes
  float* f_lp;           // [MAX_K]
  unsigned* merged;      // [MAX_W] bit k of merged[j]: extension (j, k) is an existing entry's prefix
  int *sel_parent, *sel_label, *sel_node;   // [MAX_W] new entries of the frame
};

__host__ __device__ inline size_t beam_smem_bytes(int T, int K, int W) {
  const size_t nodes = 1 + (size_t)T * W;
  return (size_t)(W * K + W) * 8 + 6 * nodes * 4 + (2 * MAX_K + 4 * MAX_W) * 4;
}

__device__ inline BeamSmem beam_smem(unsigned char* raw, int T, int K, int W) {
  BeamSmem s;
  const int nodes = 1 + T * W;
  s.cand = reinterpret_cast<uint64_t*>(raw);
  int* p = reinterpret_cast<int*>(s.cand + W * K + W);
  s.parent = p; s.label = p + nodes; s.child = p + 2 * nodes; s.sibling = p + 3 * nodes; s.stamp = p + 4 * nodes;
  s.depth = p + 5 * nodes;
  p += 6 * nodes;
  s.f_id = p; s.f_lp = reinterpret_cast<float*>(p + MAX_K);
  s.merged = reinterpret_cast<unsigned*>(p + 2 * MAX_K);
  s.sel_parent = p + 2 * MAX_K + MAX_W; s.sel_label = s.sel_parent + MAX_W; s.sel_node = s.sel_label + MAX_W;
  return s;
}

// CTC prefix beam search, one warp (one CTA) per sample; lane j holds beam entry j (prefix = trie node, pb, pnb).
// Per frame, with e the last label of entry j and the frame's candidates {blank} + (id_k, lp_k):
//   stay j         pb' = score_j + blank_lp,  pnb' = pnb_j + lp_e if e is a candidate,
//   extension j,k  pnb = (id_k == e ? pb_j : score_j) + lp_k.
// An extension that spells an entry m's prefix (parent(m) = prefix_j, last(m) = id_k) is log-added into m's stay and is
// no candidate of its own.  The trie never holds two nodes with the same (parent, label), so prefixes compare as node
// numbers and parent(m) is found through the stamp of the node: (frame << 6 | slot) while it is in the beam.
// The W best candidates by (score desc, stay before extension, parent slot, class) form the next beam, in that order.
__global__ void __launch_bounds__(32)
ctc_beam_kernel(const int* __restrict__ top_ids, const float* __restrict__ top_lp, const float* __restrict__ blank_lp, int T,
                int K, int W, int n_best, int* __restrict__ out_ids, int* __restrict__ out_len, float* __restrict__ out_score) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const BeamSmem s = beam_smem(smem_raw, T, K, W);
  const unsigned FULL = 0xffffffffu;
  const int b = blockIdx.x, lane = threadIdx.x;
  const long frame0 = (long)b * T;

  if (lane == 0) {
    s.parent[0] = -1; s.label[0] = -1; s.child[0] = -1; s.sibling[0] = -1; s.stamp[0] = 0; s.depth[0] = 0;
  }
  int nnodes = 1, nbeam = 1;
  int node = 0, e = -1;
  float pb = lane == 0 ? 0.f : -INFINITY, pnb = -INFINITY;

  int nid = -1;
  float nlp = -INFINITY, nblank = __ldg(blank_lp + frame0);
  if (lane < K) { nid = __ldg(top_ids + frame0 * K + lane); nlp = __ldg(top_lp + frame0 * K + lane); }

  for (int t = 0; t < T; ++t) {
    const float blank = nblank;
    __syncwarp();
    if (lane < K) { s.f_id[lane] = nid; s.f_lp[lane] = nlp; }
    s.merged[lane] = 0u;
    if (t + 1 < T) {                                   // next frame's candidates load while this one is decoded
      const long f = frame0 + t + 1;
      nblank = __ldg(blank_lp + f);
      if (lane < K) { nid = __ldg(top_ids + f * K + lane); nlp = __ldg(top_lp + f * K + lane); }
    }
    __syncwarp();

    const bool live = lane < nbeam;
    const float sc = log_add(pb, pnb);
    int ke = -1;                                       // slot of my last label among the frame's candidates
    if (live && e >= 0)
      for (int k = 0; k < K; ++k)
        if (s.f_id[k] == e) { ke = k; break; }
    float spb = -INFINITY, spnb = -INFINITY;
    if (live) {
      spb = sc + blank;
      if (ke >= 0) spnb = pnb + s.f_lp[ke];
    }
    int jp = -1;                                       // beam slot of my parent prefix, if my prefix is its extension
    if (live && node != 0 && ke >= 0) {
      const int st = s.stamp[s.parent[node]];
      if ((st >> 6) == t) jp = st & 63;
    }
    {
      const int src = jp < 0 ? 0 : jp;
      const float p_pb = __shfl_sync(FULL, pb, src), p_sc = __shfl_sync(FULL, sc, src);
      const int p_e = __shfl_sync(FULL, e, src);
      if (jp >= 0) {
        spnb = log_add(spnb, (e == p_e ? p_pb : p_sc) + s.f_lp[ke]);
        atomicOr(&s.merged[jp], 1u << ke);
      }
    }
    const float ssc = log_add(spb, spnb);
    __syncwarp();

    // candidate keys; each lane remembers its best
    const int next = nbeam * K, ncand = next + nbeam;
    uint64_t best = 0;
    int bq = 0;
    for (int q0 = 0; q0 < ncand; q0 += 32) {
      const int q = q0 + lane;
      const bool ext = q < next;
      int j = ext ? q / K : q - next;
      j = j < 31 ? j : 31;
      const float j_pb = __shfl_sync(FULL, pb, j), j_sc = __shfl_sync(FULL, sc, j), j_ssc = __shfl_sync(FULL, ssc, j);
      const int j_e = __shfl_sync(FULL, e, j);
      if (q >= ncand) continue;
      uint64_t key = 0;
      if (ext) {
        const int k = q - j * K;
        const int id = s.f_id[k];
        const float v = (id == j_e ? j_pb : j_sc) + s.f_lp[k];
        if (id >= 0 && !((s.merged[j] >> k) & 1u) && v > -INFINITY)
          key = make_key(v, (1u << 31) | ((uint32_t)j << 26) | ((uint32_t)id & 0x3ffffffu));
      } else if (j_ssc > -INFINITY) {
        key = make_key(j_ssc, (uint32_t)j << 26);
      }
      s.cand[q] = key;
      if (key > best) { best = key; bq = q; }
    }
    __syncwarp();

    // the W best candidates, best first
    int my_q = -1;
    uint32_t my_hi = 0;
    int nsel = 0;
    for (; nsel < W; ++nsel) {
      const uint64_t top = warp_max_key(best);
      if (top == 0) break;
      const bool win = best == top;
      const int wq = __shfl_sync(FULL, bq, __ffs(__ballot_sync(FULL, win)) - 1);
      if (lane == nsel) { my_q = wq; my_hi = (uint32_t)(top >> 32); }
      if (win) {
        s.cand[bq] = 0;
        best = 0;
        for (int q = lane; q < ncand; q += 32) {
          const uint64_t k = s.cand[q];
          if (k > best) { best = k; bq = q; }
        }
      }
    }

    // the new beam: stays keep their node, extensions find or add the (parent, label) child
    const bool sel = lane < nsel;
    const bool stay = sel && my_q >= next;
    int j = sel ? (stay ? my_q - next : my_q / K) : 0;
    const int j_node = __shfl_sync(FULL, node, j);
    const float j_spb = __shfl_sync(FULL, spb, j), j_spnb = __shfl_sync(FULL, spnb, j);
    float npb = -INFINITY, npnb = -INFINITY;
    int nnode = 0;
    if (sel) {
      s.sel_parent[lane] = stay ? -1 : j_node;
      if (stay) { nnode = j_node; npb = j_spb; npnb = j_spnb; }
      else { s.sel_label[lane] = s.f_id[my_q - j * K]; npnb = ord2f(my_hi); }
    }
    __syncwarp();
    if (lane == 0) {
      for (int r = 0; r < nsel; ++r) {
        const int par = s.sel_parent[r];
        if (par < 0) continue;
        const int lab = s.sel_label[r];
        int c = s.child[par];
        while (c >= 0 && s.label[c] != lab) c = s.sibling[c];
        if (c < 0) {
          c = nnodes++;
          s.parent[c] = par; s.label[c] = lab; s.child[c] = -1; s.sibling[c] = s.child[par]; s.depth[c] = s.depth[par] + 1;
          s.child[par] = c;
        }
        s.sel_node[r] = c;
      }
    }
    nnodes = __shfl_sync(FULL, nnodes, 0);
    __syncwarp();
    if (sel && !stay) nnode = s.sel_node[lane];
    if (sel) s.stamp[nnode] = ((t + 1) << 6) | lane;
    node = nnode; pb = npb; pnb = npnb;
    e = sel ? s.label[nnode] : -1;
    nbeam = nsel;
  }
  __syncwarp();

  if (lane < n_best) {
    int* ids = out_ids + ((long)b * n_best + lane) * T;
    int d = 0;
    if (lane < nbeam) {
      d = s.depth[node];
      for (int x = node, p = d - 1; x != 0; x = s.parent[x], --p) ids[p] = s.label[x];
    }
    for (int p = d; p < T; ++p) ids[p] = -1;
    out_len[(long)b * n_best + lane] = d;
    out_score[(long)b * n_best + lane] = lane < nbeam ? log_add(pb, pnb) : -INFINITY;
  }
}

template <int I, int KP>
int launch_topk(const ExpertTable& P, const float* gate, const float* lse, int B, int T, int C, int K, int vec,
                int* top_ids, float* top_lp, float* blank_lp, cudaStream_t st) {
  const int rows = B * T;
  ctc_topk_kernel<I, KP><<<cdiv(rows, TOPK_WARPS), TOPK_WARPS * 32, 0, st>>>(P, gate, lse, rows, T, C, K, vec, top_ids,
                                                                            top_lp, blank_lp);
  MRNB_CHECK_LAUNCH("ctc_topk_kernel");
  return MRNB_OK;
}

template <int I>
int launch_topk_k(const ExpertTable& P, const float* gate, const float* lse, int B, int T, int C, int K, int vec,
                  int* top_ids, float* top_lp, float* blank_lp, cudaStream_t st) {
  if (K <= 16) return launch_topk<I, 16>(P, gate, lse, B, T, C, K, vec, top_ids, top_lp, blank_lp, st);
  return launch_topk<I, 32>(P, gate, lse, B, T, C, K, vec, top_ids, top_lp, blank_lp, st);
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// C-ABI (declared in include/mrn_b200.h)
// ---------------------------------------------------------------------------------------------
extern "C" int mrnb_ctc_topk(const float* const* z, const long* ld, const int* Ci, int n_experts, const float* gate,
                             const float* lse, int B, int T, int K, int* top_ids, float* top_lp, float* blank_lp,
                             cudaStream_t stream) {
  MRNB_CHECK_ARG(K >= 1 && K <= MAX_K, "ctc_topk: K = %d out of range [1, %d]", K, MAX_K);
  MRNB_CHECK_ARG(n_experts >= 1 && n_experts <= MRNB_MAX_EXPERTS, "ctc_topk: n_experts %d out of range", n_experts);
  MRNB_CHECK_ARG(B > 0 && T > 0 && z && ld && Ci && gate && lse && top_ids && top_lp && blank_lp,
                 "ctc_topk: null/empty argument");
  ExpertTable P;
  int vec = 1;
  for (int i = 0; i < n_experts; ++i) {
    P.z[i] = z[i]; P.ld[i] = ld[i]; P.C[i] = Ci[i];
    MRNB_CHECK_ARG(z[i] && Ci[i] > 0 && ld[i] >= Ci[i] && Ci[i] <= Ci[n_experts - 1], "ctc_topk: bad expert %d", i);
    vec = vec && ld[i] % 4 == 0 && (reinterpret_cast<uintptr_t>(z[i]) & 15) == 0;
  }
  const int C = Ci[n_experts - 1];
#define MRNB_CASE(N) case N: return launch_topk_k<N>(P, gate, lse, B, T, C, K, vec, top_ids, top_lp, blank_lp, stream);
  switch (n_experts) {
    MRNB_CASE(1) MRNB_CASE(2) MRNB_CASE(3) MRNB_CASE(4) MRNB_CASE(5) MRNB_CASE(6) MRNB_CASE(7) MRNB_CASE(8)
  }
#undef MRNB_CASE
  return MRNB_ERR_ARG;
}

extern "C" int mrnb_ctc_beam_search(const int* top_ids, const float* top_lp, const float* blank_lp, int B, int T, int K,
                                    int W, int n_best, int* out_ids, int* out_len, float* out_score, cudaStream_t stream) {
  MRNB_CHECK_ARG(K >= 1 && K <= MAX_K, "ctc_beam_search: K = %d out of range [1, %d]", K, MAX_K);
  MRNB_CHECK_ARG(W >= 1 && W <= MAX_W, "ctc_beam_search: beam width %d out of range [1, %d]", W, MAX_W);
  MRNB_CHECK_ARG(n_best >= 1 && n_best <= W, "ctc_beam_search: n_best = %d out of range [1, W = %d]", n_best, W);
  MRNB_CHECK_ARG(T >= 1 && T <= MAX_T, "ctc_beam_search: T = %d out of range [1, %d]", T, MAX_T);
  MRNB_CHECK_ARG(top_ids && top_lp && blank_lp && out_ids && out_len && out_score && B > 0, "ctc_beam_search: null/empty argument");
  const size_t smem = beam_smem_bytes(T, K, W);
  static bool attr_set = false;
  if (!attr_set) {
    cudaFuncSetAttribute(ctc_beam_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                         (int)beam_smem_bytes(MAX_T, MAX_K, MAX_W));
    attr_set = true;
  }
  ctc_beam_kernel<<<B, 32, smem, stream>>>(top_ids, top_lp, blank_lp, T, K, W, n_best, out_ids, out_len, out_score);
  MRNB_CHECK_LAUNCH("ctc_beam_kernel");
  return MRNB_OK;
}
