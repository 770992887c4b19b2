// sm_100a building blocks shared by the tensor-core kernels: mbarriers, TMA, tcgen05 (UMMA, TMEM) and the host-side
// tensor-map encode.  Everything has internal linkage, as when every kernel file carried its own copy.
#pragma once
#include "common.cuh"
#include <cuda.h>

namespace {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// 1 KiB alignment of dynamic shared memory by OFFSET: `smem_raw + align_smem_1024_offset(smem_raw)`.  Not by an integer
// round trip of the pointer: with the offset form the compiler keeps the shared address space, so staging / operand
// tiles are accessed with LDS / STS instead of generic LD / ST (DESIGN.md §4, "Shared-address-space fix": the
// round-trip form cost 0.5 ms per training step).  The helper returns the offset rather than the aligned pointer
// because the pointer-returning form changes how nvcc associates the tile address arithmetic (other SASS, more spills).
__device__ __forceinline__ uint32_t align_smem_1024_offset(const void* smem_raw) {
  return (1024u - ((uint32_t)__cvta_generic_to_shared(smem_raw) & 1023u)) & 1023u;
}

// ---- mbarriers ----------------------------------------------------------------------------------------------------

// Wall-clock guard for mbarrier waits: first call latches the start time, later calls report > MRNB_WAIT_TRAP_NS
// elapsed (default 2 s).  Builds for compute-sanitizer runs, whose instrumentation slows kernels by orders of
// magnitude, raise the limit with -DMRNB_WAIT_TRAP_NS=... (tools/sanitize.sh).
#ifndef MRNB_WAIT_TRAP_NS
#define MRNB_WAIT_TRAP_NS 2000000000ull
#endif
__device__ __forceinline__ bool mrnb_wait_expired(uint64_t& t0) {
  uint64_t now;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
  if (t0 == 0) { t0 = now; return false; }
  return now - t0 > (unsigned long long)(MRNB_WAIT_TRAP_NS);
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
// makes the initialised barriers visible to the async proxy (TMA, tcgen05.commit); thread 0 after its mbar_init calls
__device__ __forceinline__ void fence_mbarrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// Bounded wait with a suspend-time hint (the thread sleeps in hardware instead of spinning): a protocol bug traps
// (kernel error) after MRNB_WAIT_TRAP_NS instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint64_t t0 = 0;
  for (uint32_t spin = 0;; ++spin) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity), "r"(0x989680u) : "memory");
    if (ok) return;
    if ((spin & 63u) == 63u && mrnb_wait_expired(t0)) __trap();
  }
}
// The same bounded wait without the suspend-time hint: the form the fused MLP kernel has always used.  It has never
// been measured against mbar_wait on the B200, so it stays a separate variant rather than being folded in.
__device__ __forceinline__ void mbar_wait_nohint(uint64_t* bar, uint32_t parity) {
  uint64_t t0 = 0;
  for (uint32_t spin = 0;; ++spin) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    if (ok) return;
    if ((spin & 63u) == 63u && mrnb_wait_expired(t0)) __trap();
  }
}
// Non-blocking probe of a phase (never suspends).
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\tmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}

// ---- TMA / bulk copies --------------------------------------------------------------------------------------------

__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
               ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
// shared -> global tile store, committed as its own bulk group (wait with cp.async.bulk.wait_group[.read])
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, const void* smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1) : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
// 1-D bulk copy global -> shared (bytes a multiple of 16), completion counted on `bar`
__device__ __forceinline__ void bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(src)), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// ---- tcgen05: descriptors, MMA, tensor memory ---------------------------------------------------------------------

// Shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout, descriptor version 1).  Byte offsets:
//   K-major : rows of 128 B (SWIZZLE_128B) / 64 B (SWIZZLE_64B); SBO = distance between 8-row atoms; LBO unused (16).
//   MN-major: one row per k; SBO = distance between 8-k atoms; LBO = distance between 64-wide MN chunks.
// The start address is advanced by adding (bytes >> 4) to the descriptor.
constexpr uint32_t UMMA_SWIZZLE_128B = 2, UMMA_SWIZZLE_64B = 4;
__device__ __forceinline__ uint64_t umma_smem_desc(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout) {
  uint64_t d = 0;
  d |= (uint64_t)((addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)layout << 61;
  return d;
}
// the common case: K-major 128B-swizzled tile, rows of 128 B, 8-row atoms 1024 B apart
__device__ __forceinline__ uint64_t umma_desc_k128(uint32_t addr) { return umma_smem_desc(addr, 16, 1024, UMMA_SWIZZLE_128B); }

// kind::f16 instruction descriptor: fp32 accumulator, A and B both bf16 (or both f16), M x N, each operand K-major
// unless *_mn.
enum UmmaInput : uint32_t { UMMA_F16 = 0, UMMA_BF16 = 1 };
__host__ __device__ constexpr uint32_t umma_idesc(UmmaInput ab, int m, int n, bool a_mn = false, bool b_mn = false) {
  return (1u << 4) | ((uint32_t)ab << 7) | ((uint32_t)ab << 10) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) |
         ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// D[tmem] (+)= A[smem] * B[smem]^T (acc = 0: overwrite), one instruction issued by one thread
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}
// arrives on `bar` once every MMA issued so far by this thread has completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// ordering of tcgen05 operations across a thread synchronisation (mbarrier or bar.sync)
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// Allocates `cols` TMEM columns (one whole warp) and writes the base address to shared memory; the permit is given up
// at once so that a co-resident CTA can allocate too.  Read the address after tc_fence_before / sync / tc_fence_after.
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_shared, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_shared)), "r"(cols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
// by the warp that allocated, after every use of the columns
__device__ __forceinline__ void tmem_dealloc(uint32_t base, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(cols) : "memory");
}

// TMEM -> registers, 32 lanes x 16 / 32 columns; the _nowait form leaves the registers pending until tmem_ld_wait()
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  tmem_ld16_nowait(taddr, r);
  tmem_ld_wait();
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  tmem_ld_wait();
}
// registers -> TMEM, 32 lanes x 32 columns, waits for the store to complete
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
        "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]),
        "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]),
        "r"(r[30]), "r"(r[31])
      : "memory");
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

// ---- small arithmetic ---------------------------------------------------------------------------------------------

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float max3(float a, float b, float c) {
  float r;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));      // FMNMX3
  return r;
}
__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}

// ---- host: tensor maps --------------------------------------------------------------------------------------------

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
// cuTensorMapEncodeTiled from the driver, looked up once per translation unit; nullptr when the driver lacks it
inline EncodeTiledFn tensor_map_encoder() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}
// Encodes a tiled tensor map (no interleave, no out-of-bounds NaN fill: outside the tensor reads as zero).  On failure
// the error message names the caller `who` and the result is MRNB_ERR_UNSUPPORTED (no entry point) or MRNB_ERR_ARG.
inline int encode_tensor_map(const char* who, CUtensorMap* map, CUtensorMapDataType dtype, cuuint32_t rank, const void* ptr,
                             const cuuint64_t* dims, const cuuint64_t* strides, const cuuint32_t* box, const cuuint32_t* elem_strides,
                             CUtensorMapSwizzle swizzle, CUtensorMapL2promotion l2 = CU_TENSOR_MAP_L2_PROMOTION_L2_256B) {
  EncodeTiledFn fn = tensor_map_encoder();
  if (!fn) { mrnb_set_error("%s: cuTensorMapEncodeTiled unavailable", who); return MRNB_ERR_UNSUPPORTED; }
  CUresult r = fn(map, dtype, rank, const_cast<void*>(ptr), dims, strides, box, elem_strides, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, l2,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { mrnb_set_error("%s: cuTensorMapEncodeTiled failed (%d)", who, (int)r); return MRNB_ERR_ARG; }
  return MRNB_OK;
}

}  // namespace
