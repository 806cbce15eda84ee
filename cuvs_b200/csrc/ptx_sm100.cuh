// Thin inline-PTX wrappers for the sm_100a features the scan kernels use:
// mbarrier, TMA (cp.async.bulk[.tensor]), tcgen05 (alloc / mma / commit / ld / fences).
// Hand-written against the PTX ISA; descriptor bit layouts follow the UMMA conventions
// (start address >>4, LBO, SBO, version=1 @46, layout type @61; instruction descriptor:
// c_format @4, a/b_format @7/@10, a/b_major @15/@16, N>>3 @17, M>>4 @24).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cstdint>

namespace b200 {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p)
{
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ bool elect_one()
{
  uint32_t pred = 0;
  asm volatile(
    "{\n\t"
    ".reg .pred P;\n\t"
    "elect.sync _|P, 0xffffffff;\n\t"
    "selp.b32 %0, 1, 0, P;\n\t"
    "}\n"
    : "=r"(pred));
  return pred != 0;
}

// ------------------------------------------------------------------ mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count)
{
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init()
{
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async()
{
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes)
{
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar)
{
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity)
{
  uint32_t ok;
  asm volatile(
    "{\n\t"
    ".reg .pred P;\n\t"
    "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2, %3;\n\t"
    "selp.b32 %0, 1, 0, P;\n\t"
    "}\n"
    : "=r"(ok)
    : "r"(smem_u32(bar)), "r"(parity), "r"(0x989680u) /* suspend-time hint: sleep in hardware instead of spinning */
    : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
  while (!mbar_try_wait(bar, parity)) {}
}

// ------------------------------------------------------------------ TMA
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* m)
{
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// 2-D tile load: coordinates (c0 = innermost element offset, c1 = row)
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int32_t c0, int32_t c1)
{
  asm volatile(
    "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
    ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
    : "memory");
}
// 1-D bulk copy global -> shared (16-byte aligned, size multiple of 16)
__device__ __forceinline__ void bulk_load_1d(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar)
{
  asm volatile(
    "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
    ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(gsrc)), "r"(bytes), "r"(smem_u32(bar))
    : "memory");
}

// Bulk L2 prefetch (UBLKPF): one instruction asks the copy engine to pull `bytes` (multiple of 16, 16-byte aligned source)
// of global memory into L2.  No destination, no registers, no completion object: the later ordinary loads hit L2.
__device__ __forceinline__ void bulk_prefetch_l2(const void* gsrc, uint32_t bytes)
{
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(reinterpret_cast<uint64_t>(gsrc)), "r"(bytes) : "memory");
}

// ------------------------------------------------------------------ tcgen05
template <uint32_t NCols>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result)
{
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)), "n"(NCols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <uint32_t NCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr)
{
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(NCols) : "memory");
}
__device__ __forceinline__ void tc_fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem], bf16 inputs, fp32 accumulate, issued by ONE thread.  The two shared-memory descriptors are
// given as (lo, hi) 32-bit halves: consecutive K steps / stages differ only in the low word (start address >> 4), so the
// issuing thread spends one integer add per operand and MMA.
__device__ __forceinline__ void mma_bf16_ss_lohi(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                                 uint32_t idesc, uint32_t accumulate)
{
  asm volatile(
    "{\n\t"
    ".reg .pred p;\n\t"
    ".reg .b64 da, db;\n\t"
    "mov.b64 da, {%1, %2};\n\t"
    "mov.b64 db, {%3, %4};\n\t"
    "setp.ne.b32 p, %6, 0;\n\t"
    "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t"
    "}\n"
    ::"r"(tmem_d), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
    : "memory");
}
__device__ __forceinline__ uint32_t smem_desc_lo(uint32_t smem_addr) { return ((smem_addr & 0x3ffffu) >> 4) | (1u << 16); }
constexpr uint32_t kDescHiSw128 = (1024u >> 4) | (1u << 14) | (2u << 29);  // SBO 1024 B, version 1, SWIZZLE_128B
constexpr uint32_t kDescHiSw32  = (256u >> 4) | (1u << 14) | (6u << 29);   // SBO 256 B, version 1, SWIZZLE_32B
// arrive on an mbarrier once all previously issued tcgen05.mma of this thread have completed
__device__ __forceinline__ void mma_commit(uint64_t* bar)
{
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// TMEM -> registers: this warp's 32 lanes x 32 consecutive fp32 columns (lane i gets row i)
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32])
{
  asm volatile(
    "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
    "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
    "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
    : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
      "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
      "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
      "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
    : "r"(taddr)
    : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t nthreads)
{
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// kind::f16, A = B = bf16, D = fp32, both K-major, dense
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N)
{
  return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(N >> 3) << 17) | (static_cast<uint32_t>(M >> 4) << 24);
}

}  // namespace ptx
}  // namespace b200
