// Shared device/host helpers for the sm_100a hot-path kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <utility>

#include "re2e_b200.h"

namespace re2e {

// ---- host side ------------------------------------------------------------------------------
extern std::atomic<unsigned long long> g_launches;  // defined in api.cu
inline void count_launch(int n = 1) { g_launches.fetch_add((unsigned long long)n, std::memory_order_relaxed); }

#define RE2E_CHECK_ARG(cond) \
  do {                       \
    if (!(cond)) return RE2E_E_ARG; \
  } while (0)

#define RE2E_CUDA(expr)                   \
  do {                                    \
    cudaError_t _e = (expr);              \
    if (_e != cudaSuccess) return (int)_e; \
  } while (0)

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) once per (kernel, size) -- cached so that steady-state
// launches (and CUDA-graph capture) issue no attribute calls.  Defined in api.cu.
int ensure_smem(const void *func, size_t bytes);

// cudaGetLastError (not Peek): a failed launch is reported once, by the call that made it, and does not poison
// the status of later calls
inline int launch_status() {
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? RE2E_OK : (int)e;
}

int num_sms();   // SM count of the CURRENT device (cached per device); defined in api.cu
// true when at least one cluster of cluster_x CTAs of `threads` threads and `smem` dynamic shared memory bytes can be
// resident on the current device (cudaOccupancyMaxActiveClusters, cached); true without a device.  Defined in api.cu.
bool cluster_fits(const void *func, int cluster_x, int threads, size_t smem);

// Launch of a thread-block-cluster kernel in clusters of cluster_x CTAs along x; counts the launch.
// pdl = true launches with programmatic stream serialisation: the grid may become resident while its predecessor in
// the stream is still running, so the kernel must execute pdl_wait() before it reads or writes anything the
// predecessor (or, transitively, anything earlier in the stream) may still touch.
template <typename... KArgs, typename... Args>
inline int launch_cluster(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, int cluster_x,
                          bool pdl, Args &&...args) {
  const void *fn = reinterpret_cast<const void *>(kern);
  int rc = ensure_smem(fn, smem);
  if (rc != RE2E_OK) return rc;
  if (cluster_x > 8) RE2E_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)cluster_x;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 2 : 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);
  count_launch();
  return e == cudaSuccess ? RE2E_OK : (int)e;
}

inline bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// ---- device side ----------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// tanh with ~1e-7 absolute error: 1 - 2/(e^{2x}+1).  ex2.approx has 2^-22 relative error and the
// form saturates cleanly to +-1 for |x| large (no NaN: e^{2x} -> inf gives 1, -> 0 gives -1).
__device__ __forceinline__ float tanh_fast(float x) {
  float e = __expf(2.0f * x);
  return 1.0f - __fdividef(2.0f, e + 1.0f);
}

// same function from the raw approximate units (5 instructions, no range fix-ups): ex2.approx of a huge argument gives
// +inf -> rcp gives 0 -> 1; of a very negative one gives 0 -> rcp(1) = 1 -> -1.  |error| ~1e-7 absolute.
__device__ __forceinline__ float tanh_ex2(float x) {
  float e, r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * 2.8853900817779268f));   // e^{2x} = 2^{2x log2 e}
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(e + 1.0f));
  return fmaf(-2.0f, r, 1.0f);
}

__device__ __forceinline__ float sigmoid_acc(float x) { return 1.0f / (1.0f + expf(-x)); }

// streaming 128-bit accesses (read-once / write-once data: keep it out of L1)
__device__ __forceinline__ float4 ld_stream4(const float *p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ float2 ld_stream2(const float *p) {
  float2 r;
  asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0,%1}, [%2];" : "=f"(r.x), "=f"(r.y) : "l"(p));
  return r;
}
__device__ __forceinline__ float ld_stream1(const float *p) {
  float r;
  asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(r) : "l"(p));
  return r;
}
__device__ __forceinline__ void st_stream4(float *p, float4 v) {
  asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y),
               "f"(v.z), "f"(v.w)
               : "memory");
}

// Programmatic dependent launch (PDL).  The step kernels are launched with programmatic stream serialisation, so
// a grid may become resident while its predecessor in the stream (normally the previous decoder step) is still
// running.  Everything before pdl_wait() touches only memory that was final before the predecessor STARTED:
// parameters, the per-utterance encoder tensors (pre, enc_h) and -- in the backward -- tensors saved by the
// forward pass.  griddepcontrol.wait returns once the predecessor grid has completed and flushed; all global
// writes and all reads of per-step inputs (att_prev / dec_z, dc / dw, accumulators) come after it.  A predecessor
// that never executes launch_dependents (any foreign kernel) degrades to ordinary stream order.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ---- mbarrier + bulk async copy (TMA 1-D, SASS UBLKCP) ----------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
  // make the inits visible to the async proxy (and to the cluster)
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "DONE:\n\t"
      "}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
// global -> shared bulk copy; bytes % 16 == 0, both addresses 16 B aligned.
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes,
                                         uint64_t *bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(dst_smem)),
      "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}
// shared -> global bulk reduce-add (fp32): the TMA unit does the read-modify-write at L2.
__device__ __forceinline__ void bulk_red_add_s2g(void *dst_gmem, const void *src_smem, uint32_t bytes) {
  asm volatile("cp.reduce.async.bulk.global.shared::cta.bulk_group.add.f32 [%0], [%1], %2;" ::"l"(dst_gmem),
               "r"(smem_u32(src_smem)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_s2g(void *dst_gmem, const void *src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem),
               "r"(smem_u32(src_smem)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void bulk_wait() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}
// generic-proxy smem writes -> visible to the async proxy (before a bulk store reads them)
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ---- thread-block cluster helpers -------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t cluster_nctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// address of `p` (a shared-memory pointer of THIS cta) in the shared window of cluster rank `rank`
__device__ __forceinline__ uint32_t dsmem_addr(const void *p, uint32_t rank) {
  uint32_t a = smem_u32(p), r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(rank));
  return r;
}
__device__ __forceinline__ float dsmem_ld(uint32_t addr) {
  float v;
  asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void dsmem_st(uint32_t addr, float v) {
  asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}
__device__ __forceinline__ void dsmem_st4(uint32_t addr, float a, float b, float c, float d) {
  asm volatile("st.shared::cluster.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

}  // namespace re2e
