// tcgen05 / TMEM helpers (sm_100a inline PTX) of the tensor-core kernels of the library; the mbarrier and fence
// primitives they use are in gnca_ptx.cuh.
//
// Operand conventions used throughout (validated on a B200 by scratch/umma_probe.cu, profiles/r02_umma_probe.md):
//  * kind::tf32, cta_group::1, M = 128: accumulator row m lives in TMEM lane m, column n in TMEM column base + n.
//  * A operand from TENSOR MEMORY (row m = lane m, k = column): a thread of a 128-thread warpgroup owns one row, so
//    "thread t <-> cell t <-> lane t" needs no shared-memory staging of the activations at all.
//  * B operand from shared memory, K-major, NO swizzle: core matrix = 8 rows x 16 bytes stored as 128 contiguous bytes,
//    core matrices adjacent along K (leading byte offset 128), 8-row groups strided by (K/4)*128 bytes (stride byte
//    offset).  One MMA consumes K = 8 tf32 values = two core-matrix columns = 256 bytes of descriptor advance.
//  * The tensor core TRUNCATES fp32 inputs to tf32 (probe: 7e-7 against a truncating host model, 1.8e-3 against a
//    rounding one), so the 3xTF32 split rounds explicitly: hi = rna(x), lo = rna(x - hi); x*w ~ hi*whi + hi*wlo + lo*whi.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "gnca_ptx.cuh"

namespace gnca {
namespace tc {

// float index of element (r, k) of an [R x K] operand in the canonical no-swizzle K-major layout (R % 8 == 0, K % 4 == 0)
__host__ __device__ __forceinline__ int canon_idx(int r, int k, int K) {
  return (r >> 3) * (K >> 2) * 32 + (k >> 2) * 32 + (r & 7) * 4 + (k & 3);
}

__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3fff);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3fff) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3fff) << 32;
  d |= (uint64_t)1 << 46;          // descriptor version 1 (sm_100)
  return d;                        // base offset 0, layout type 0 = no swizzle
}
// instruction descriptor: D = f32, A = B = tf32, both K-major, dense
__host__ __device__ constexpr uint32_t idesc_tf32(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ void mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
               "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}\n"
               :: "r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void mma_ss(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
               "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n"
               :: "r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}
// arrive on an mbarrier when every MMA issued so far by this thread has completed (implies fence::before_thread_sync)
__device__ __forceinline__ void mma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(bar) : "memory");
}
__device__ __forceinline__ void fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// whole-warp: allocate / free `cols` TMEM columns (power of two >= 32); the base address lands in *slot (shared memory)
__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(slot)), "r"(cols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_free(uint32_t base, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(base), "r"(cols) : "memory");
}

// 32 lanes x 32 bit, 16 consecutive columns: lane (taddr >> 16) + laneid, columns (taddr & 0xffff) .. +15
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                 "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
               : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};\n"
               :: "r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
                  "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]) : "memory");
}

__device__ __forceinline__ uint32_t tf32_rna(float x) { uint32_t r; asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x)); return r; }
__device__ __forceinline__ void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
  hi = tf32_rna(x);
  lo = tf32_rna(x - __uint_as_float(hi));
}
// activation split of the tile kernels, 3 instructions instead of the 7 `cvt.rna.tf32` expands to twice on sm_100a:
// hi = x rounded to nearest (ties away) on the 13 dropped bits by an integer add + mask (finite x; an overflow rounds to
// inf like the cvt), lo = x - hi handed to the tensor core as it is -- the unit truncates its operands to tf32, and
// |lo| <= 2^-11 |x|, so the truncation of lo costs <= 2^-21 |x| (the cvt version 2^-22; the dropped lo*lo term 2^-22).
__device__ __forceinline__ void split_tf32_fast(float x, uint32_t& hi, uint32_t& lo) {
  hi = (__float_as_uint(x) + 0x1000u) & 0xffffe000u;
  lo = __float_as_uint(x - __uint_as_float(hi));
}

// named barriers (id 0 is __syncthreads)
__device__ __forceinline__ void bar_sync(int id, int nthreads) { asm volatile("bar.sync %0, %1;" :: "r"(id), "r"(nthreads) : "memory"); }
__device__ __forceinline__ void bar_arrive(int id, int nthreads) { asm volatile("bar.arrive %0, %1;" :: "r"(id), "r"(nthreads) : "memory"); }

}  // namespace tc
}  // namespace gnca
