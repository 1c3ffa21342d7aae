// tc_ptx.cuh — inline-PTX wrappers for the Blackwell async machinery used by the tensor-core kernels:
// mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc / mma / commit / ld), UMMA descriptors.
#pragma once
#include "common.cuh"

namespace tcp {

// ---------------------------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
// programmatic dependent launch (see launch_pdl in common.cuh): block until every prerequisite grid has completed
// and its writes are visible; then let the next kernel in the stream start its own prologue
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// Bounded wait: a pipeline bug must surface as a trap (clean CUDA error), never as a hung GPU.
// try_wait suspends the thread for a hardware-bounded interval per probe; 2^22 failed probes is seconds.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done, spins = 0;
  do {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (!done && ++spins > (1u << 22)) __trap();
  } while (!done);
}
__device__ __forceinline__ void prefetch_tmap(const void* tm) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tm)) : "memory");
}
__device__ __forceinline__ void tma_load_5d(uint32_t smem_dst, const void* tm, uint32_t bar, int c0,
                                            int c1, int c2, int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
      ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(c0), "r"(c1), "r"(c2),
        "r"(c3), "r"(c4)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t smem_dst, const void* tm, uint32_t bar, int c0,
                                            int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
// D[tmem] (+)= A[smem] * B[smem], bf16 x bf16 -> fp32, single-CTA
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc,
                                          uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Same, with the two 64-bit descriptors passed as (lo, hi) halves: the hi halves are loop constants and
// advancing along K / rows is one 32-bit add on the lo half (the issuing thread is a single lane, so
// every instruction saved in the issue loop is tensor-pipe time gained).
__device__ __forceinline__ void umma_bf16_lh(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo,
                                             uint32_t b_hi, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      ".reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t"
      "}"
      ::"r"(d_tmem), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
// ---- warp-uniform variants -------------------------------------------------------------------
// The TMA / tcgen05 instructions take their operands from UNIFORM registers. Issued from inside a
// divergent `if (lane == 0)` region the compiler wraps every one of them in an ELECT/branch
// "waterfall" loop plus R2UR moves (~150 cycles per MMA for the single issuing lane). So the producer
// and MMA warps run their loops with all 32 lanes converged on warp-uniform values, and only the
// instruction itself is predicated on one elected lane, inside the asm block.
__device__ __forceinline__ void umma_bf16_lh_elect(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo,
                                                   uint32_t b_hi, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p, q;\n\t"
      ".reg .b64 da, db;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t"
      "}"
      ::"r"(d_tmem), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit_elect(uint32_t bar) {
  asm volatile(
      "{\n\t"
      ".reg .pred q;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t"
      "}"
      ::"r"(bar)
      : "memory");
}
__device__ __forceinline__ void mbar_arrive_elect(uint32_t bar) {
  asm volatile(
      "{\n\t"
      ".reg .pred q;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "@q mbarrier.arrive.shared::cta.b64 _, [%0];\n\t"
      "}"
      ::"r"(bar)
      : "memory");
}
__device__ __forceinline__ void mbar_expect_tx_elect(uint32_t bar, uint32_t bytes) {
  asm volatile(
      "{\n\t"
      ".reg .pred q;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "@q mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n\t"
      "}"
      ::"r"(bar), "r"(bytes)
      : "memory");
}
__device__ __forceinline__ void tma_load_5d_elect(uint32_t smem_dst, const void* tm, uint32_t bar, int c0, int c1,
                                                  int c2, int c3, int c4) {
  asm volatile(
      "{\n\t"
      ".reg .pred q;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "@q cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6, %7}], [%2];\n\t"
      "}"
      ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d_elect(uint32_t smem_dst, const void* tm, uint32_t bar, int c0, int c1,
                                                  int c2) {
  asm volatile(
      "{\n\t"
      ".reg .pred q;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "@q cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5}], [%2];\n\t"
      "}"
      ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_elect(uint32_t smem_dst, const void* tm, uint32_t bar, int c0, int c1) {
  asm volatile(
      "{\n\t"
      ".reg .pred q;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "@q cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n\t"
      "}"
      ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
// descriptor halves: lo = start address >> 4 | LBO field, hi = SBO field | version 1 | swizzle code
__device__ __forceinline__ uint32_t desc_lo(uint32_t saddr, uint32_t lbo_bytes) {
  return ((saddr & 0x3FFFFu) >> 4) | (((lbo_bytes >> 4) & 0x3FFFu) << 16);
}
__device__ __forceinline__ uint32_t desc_hi(uint32_t sbo_bytes, uint32_t layout_type) {
  return ((sbo_bytes >> 4) & 0x3FFFu) | (1u << 14) | ((layout_type & 7u) << 29);
}
// mbarrier arrives when all previously issued MMAs of this thread have completed
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar)
               : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t r[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, "
      "%13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]),
        "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
// zero 16 accumulator columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_st16_zero(uint32_t taddr) {
  const uint32_t z = 0u;
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1};"
      ::"r"(taddr), "r"(z)
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() {
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// UMMA shared-memory matrix descriptor (SM100 format, version 1).
//   bits [ 0,14) start address >> 4      bits [16,30) leading byte offset >> 4
//   bits [32,46) stride byte offset >> 4 bits [46,48) version = 1   bits [61,64) swizzle mode
// K-major swizzled tile (rows of 32/64/128 B): SBO = 8 rows, LBO unused (=1).
// MN-major swizzled tile (k-rows of 32/64/128 B holding MN-contiguous elements): SBO = 8 k-rows,
// LBO = distance between consecutive swizzle-wide MN blocks.
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes,
                                                   uint32_t sbo_bytes, uint32_t layout_type) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)(layout_type & 7u) << 61;
  return d;
}
// Instruction descriptor for kind::f16: D=f32 (bits 4-5 = 1), A=B=bf16 (bits 7-9, 10-12 = 1),
// a_major bit 15, b_major bit 16 (0 = K-major, 1 = MN-major), N>>3 bits 17-22, M>>4 bits 24-28.
__host__ __device__ constexpr uint32_t make_idesc(int M, int N, int a_mn, int b_mn) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}


// swizzle span in bytes -> UMMA layout_type code (SWIZZLE_128B = 2, 64B = 4, 32B = 6)
__host__ __device__ constexpr uint32_t layout_code(int row_bytes) {
  return row_bytes == 128 ? 2u : (row_bytes == 64 ? 4u : 6u);
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
constexpr int kMaxDynSmem = 227 * 1024;  // opt-in dynamic shared memory per block on sm_100

// the same swizzle span for the TMA tensor map (rows of 128 / 64 / 32 bytes)
inline CUtensorMapSwizzle swizzle_for_row_bytes(int row_bytes) {
  return row_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                          : (row_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
}

// cuTensorMapEncodeTiled through the runtime's driver entry-point query (no link against libcuda), looked up once;
// nullptr when the driver does not provide it
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
inline EncodeTiledFn encode_tiled() {
  static const EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    const bool ok = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
                    qres == cudaDriverEntryPointSuccess;
    return ok ? (EncodeTiledFn)p : nullptr;
  }();
  return fn;
}

}  // namespace tcp
