// Inline-PTX synchronisation primitives (sm_100a) shared by the cluster and tensor-core kernels of the library:
// shared-memory addresses, mbarriers, the async-proxy fence and the cluster barriers.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace gnca {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarriers (shared::cta) -------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(bar), "r"(count) : "memory");
}
// makes the initialisations above visible to the async proxy and to the other CTAs of the cluster
__device__ __forceinline__ void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
// arrive once and add `tx` bytes to the transaction count the current phase waits for
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t tx) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(tx) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  do {
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
                 : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  } while (!ok);
}

// generic-proxy writes to shared memory -> visible to the async proxy (UMMA operand reads, bulk copies)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- cluster barriers --------------------------------------------------------------------------------------------
// Every arrive is a release: the DSMEM and global stores a thread issued before it are performed before a peer passes
// the wait.  The waits differ in whether they acquire.
//
// Split form without acquire: independent work can run between the arrive and the wait.
__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.aligned;" ::: "memory"); }

// Full barrier with acquire: for kernels whose CTAs hand each other data through global memory, which a plain load may
// serve from a stale L1 line unless the wait acquires.
__device__ __forceinline__ void cluster_sync_acquire() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;\n" ::: "memory");
}

// Full barrier WITHOUT acquire: an acquire makes ptxas emit CCTL.IVALL, which invalidates the whole L1 -- including the
// lines backing local memory (stack) -- at every barrier.  For kernels whose peers communicate through shared::cluster
// stores only (nothing exchanged inside the kernel travels through L1-cached global memory), the invalidation buys
// nothing.
__device__ __forceinline__ void cluster_sync_no_acquire() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.aligned;\n" ::: "memory");
}

}  // namespace gnca
