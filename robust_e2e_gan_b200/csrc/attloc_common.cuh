// Helpers shared by the AttLoc kernels (attloc.cu: one step per launch; attloc_loop.cu: the whole decoder
// loop in one persistent cluster kernel).  sm_100a only.
#pragma once
#include "common.cuh"

namespace re2e {

constexpr int kTG = 5;        // conv outputs per thread (sliding window)
constexpr int kKQ = 5;        // K split (items = frame groups x C x kKQ = 500 of 512 threads at the default shape)

__host__ __device__ inline int round4(int v) { return (v + 3) & ~3; }

// sum 16 per-lane values across the warp with recursive halving (16 shuffles instead of 80); on return
// lane L (L even) holds in v[0] the total of value index  bit4*8 + bit3*4 + bit2*2 + bit1  of L.
__device__ __forceinline__ void warp_reduce16(float (&v)[16], int lane) {
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const bool up = lane & 16;
    const float send = up ? v[i] : v[i + 8], keep = up ? v[i + 8] : v[i];
    v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const bool up = lane & 8;
    const float send = up ? v[i] : v[i + 4], keep = up ? v[i + 4] : v[i];
    v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
  }
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const bool up = lane & 4;
    const float send = up ? v[i] : v[i + 2], keep = up ? v[i + 2] : v[i];
    v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
  }
  {
    const bool up = lane & 2;
    const float send = up ? v[0] : v[1], keep = up ? v[1] : v[0];
    v[0] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
  }
  v[0] += __shfl_xor_sync(0xffffffffu, v[0], 1);
}

__device__ __forceinline__ void mbar_arrive1(uint64_t *bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void cluster_arrive() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
}
__device__ __forceinline__ void cluster_wait() {
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void pair_bar(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// remote shared-memory store that signals the destination CTA's mbarrier (complete_tx of 4 bytes): the
// receiver waits on its own barrier -- no cluster-wide barrier, no release fence on the sender
__device__ __forceinline__ void st_async_f32(uint32_t remote_addr, float v, uint32_t remote_bar) {
  asm volatile("st.async.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];" ::"r"(remote_addr),
               "r"(__float_as_uint(v)), "r"(remote_bar)
               : "memory");
}
__device__ __forceinline__ void st_async_f32x4(uint32_t remote_addr, float a, float b, float c, float d, uint32_t remote_bar) {
  asm volatile("st.async.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%1, %2, %3, %4}, [%5];" ::"r"(remote_addr),
               "r"(__float_as_uint(a)), "r"(__float_as_uint(b)), "r"(__float_as_uint(c)), "r"(__float_as_uint(d)),
               "r"(remote_bar)
               : "memory");
}
__device__ __forceinline__ void cluster_arrive_relaxed() {
  asm volatile("barrier.cluster.arrive.relaxed.aligned;" ::: "memory");
}

// ---- host side ------------------------------------------------------------------------------
// shapes both kernel families take: A = 64 * APL attention channels, D <= 512 encoder channels, C <= 16, odd K
inline int check_dims(int B, int Th, int D, int A, int C, int K) {
  if (B <= 0 || Th <= 0 || D <= 0 || A <= 0 || C <= 0 || K <= 0) return RE2E_E_ARG;
  if ((K & 1) == 0) return RE2E_E_ARG;
  if (A % 64 != 0 || A > 512 || (D & 3) || D > 512 || C > 16) return RE2E_E_UNSUPPORTED;
  const int apl = A / 64;
  if (!(apl == 1 || apl == 2 || apl == 4 || apl == 5 || apl == 8)) return RE2E_E_UNSUPPORTED;
  return RE2E_OK;
}

// rc = NAME<APL, CP> ARGS for the instantiated (A / 64, C padded to 10 or 16) pairs
#define ATT_DISPATCH(NAME, APLV, CPV, ...)                                              \
  switch (APLV) {                                                                       \
    case 1: rc = (CPV) == 10 ? NAME<1, 10> __VA_ARGS__ : NAME<1, 16> __VA_ARGS__; break; \
    case 2: rc = (CPV) == 10 ? NAME<2, 10> __VA_ARGS__ : NAME<2, 16> __VA_ARGS__; break; \
    case 4: rc = (CPV) == 10 ? NAME<4, 10> __VA_ARGS__ : NAME<4, 16> __VA_ARGS__; break; \
    case 5: rc = (CPV) == 10 ? NAME<5, 10> __VA_ARGS__ : NAME<5, 16> __VA_ARGS__; break; \
    case 8: rc = (CPV) == 10 ? NAME<8, 10> __VA_ARGS__ : NAME<8, 16> __VA_ARGS__; break; \
    default: rc = RE2E_E_UNSUPPORTED;                                                   \
  }

}  // namespace re2e
