// Shared helpers for the sm_100a kernels of the wave-propagation hot path.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/fus_b200.h"

// ---- host-side error / bookkeeping (defined in api.cu) ---------------------
int fus_set_error(int code, const char* what);
void fus_count_launch(int n = 1);

#define FUS_CUDA(expr)                                        \
  do {                                                        \
    cudaError_t e__ = (expr);                                 \
    if (e__ != cudaSuccess) return fus_set_error((int)e__, #expr); \
  } while (0)

#define FUS_LAUNCH_CHECK(name)                                 \
  do {                                                         \
    cudaError_t e__ = cudaGetLastError();                      \
    if (e__ != cudaSuccess) return fus_set_error((int)e__, name); \
    fus_count_launch();                                        \
  } while (0)

int fus_num_sms();

// halo wait armed for the next stiffness launch of this host thread (api.cu)
struct FusHaloDev;
bool fus_take_armed_wait(const FusHaloDev** h, long long* first_interface_cell);

// ---- device-side PTX wrappers ---------------------------------------------
#ifdef __CUDACC__

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}

// make mbarrier.init visible to the async proxy (TMA unit)
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

// order prior generic-proxy accesses to shared memory before later async-proxy
// (bulk copy) accesses to the same locations
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}

__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1, 0x989680;\n\t"
      "@P1 bra WAIT_DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "WAIT_DONE:\n\t"
      "}" ::"r"(addr),
      "r"(parity)
      : "memory");
}

// TMA 1-D bulk copy global -> shared, completion signalled on an mbarrier.
// src, dst and bytes must be multiples of 16.
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes,
                                         uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
          "r"(smem_u32(dst_smem)),
      "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

// same, with an L2 eviction-priority hint (streamed-once data: evict_first)
__device__ __forceinline__ void bulk_g2s_hint(void* dst_smem, const void* src_gmem, uint32_t bytes,
                                              uint64_t* bar, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint "
      "[%0], [%1], %2, [%3], %4;" ::"r"(smem_u32(dst_smem)),
      "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
      : "memory");
}

__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}

#endif  // __CUDACC__
