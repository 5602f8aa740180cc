// Shared device/host helpers for the dasp_b200 kernels (sm_100a only).
//
//  * error plumbing for the C ABI (thread-local last-error string, no exceptions cross the ABI)
//  * 1-D TMA ("bulk async copy") + mbarrier wrappers: the recurrence kernels stage contiguous
//    fp32 tiles HBM -> shared memory with cp.async.bulk (SASS: UBLKCP) and write results back
//    with the shared -> global bulk form, so the hot loops contain no LDG/STG at all.
//  * warp reductions.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/dasp_b200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "dasp_b200 kernels are written for sm_100a (B200) only"
#endif

namespace dasp {

// ---------------------------------------------------------------- host: error handling
// status codes: DASP_OK / DASP_ERR_* macros from include/dasp_b200.h

void set_error(const char* fmt, ...);

#define DASP_REQUIRE(cond, ...)            \
  do {                                     \
    if (!(cond)) {                         \
      ::dasp::set_error(__VA_ARGS__);      \
      return DASP_ERR_INVALID;     \
    }                                      \
  } while (0)

#define DASP_CUDA_OK(expr)                                                              \
  do {                                                                                  \
    cudaError_t e__ = (expr);                                                           \
    if (e__ != cudaSuccess) {                                                           \
      ::dasp::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, \
                        __LINE__);                                                      \
      return DASP_ERR_CUDA;                                                     \
    }                                                                                   \
  } while (0)

#define DASP_LAUNCH_OK(name)                                                           \
  do {                                                                                 \
    cudaError_t e__ = cudaGetLastError();                                              \
    if (e__ != cudaSuccess) {                                                          \
      ::dasp::set_error("launch of %s failed: %s", name, cudaGetErrorString(e__));     \
      return DASP_ERR_CUDA;                                                    \
    }                                                                                  \
  } while (0)

static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

int sm_count();  // cached cudaDevAttrMultiProcessorCount of the current device

// Test hook (dasp_debug_force_warps): 0 = automatic; 1/2/4/8/16 pins the warps-per-row choice of the scan kernels
// (the EQ forward has 4/8/16, the compressor all five; a kernel family that has no such variant keeps its automatic
// choice) so that every kernel variant can be exercised at small, cheap-to-check batch sizes.
int debug_forced_warps();
// Test hook (dasp_debug_reverb_flat_filterbank): the spectral IR synthesis uses unit-impulse "filters", so the
// band-filtered noise it keeps for the backward IS the periodic white sequence w_k the generator draws; the parity
// test rebuilds the reference-style noise tensor from it and checks the default path against the oracle.
int debug_flat_filterbank();

// ---------------------------------------------------------------- device helpers
#ifdef __CUDACC__

constexpr float kLn10Over20 = 0.11512925464970228f;   // ln(10)/20
constexpr float kLog2Of10Over20 = 0.16609640474436813f;  // log2(10)/20 : 10^(d/20) = 2^(d*this)

__device__ __forceinline__ float db_to_lin(float db) { return exp2f(db * kLog2Of10Over20); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---- mbarrier (shared::cta, 64-bit) ----
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
// make barrier inits visible to the async (TMA) proxy
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
// order generic-proxy shared-memory writes before later async-proxy (bulk copy) accesses
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
// plain arrive (release semantics at CTA scope): completes one pending arrival of the current phase
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra WAIT_DONE;\n"
      "bra WAIT_LOOP;\n"
      "WAIT_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}

// ---- 1-D TMA bulk copies (addresses and byte counts must be multiples of 16) ----
__device__ __forceinline__ void tma_load_1d(void* smem_dst, const void* gmem_src, uint32_t bytes,
                                            uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(smem_dst)),
      "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void tma_store_1d(void* gmem_dst, const void* smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gmem_dst),
               "r"(smem_u32(smem_src)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// wait until at most N committed bulk-store groups still READ their shared-memory source
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait_all() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

#endif  // __CUDACC__

}  // namespace dasp
