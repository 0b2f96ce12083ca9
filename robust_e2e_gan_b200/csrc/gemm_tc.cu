// fp32-accurate dense GEMM on the 5th-generation tensor cores (tcgen05 / TMEM / TMA), 3xTF32 split.
//
//   C[M,N] (+)= Aop[M,K] * Bop[N,K]^T (+ bias[N])
//
// used for the dense layers on the hot path whose fp32 parity (1e-4) rules out a single TF32/BF16
// pass: ctc_lo (model/e2e_ctc.py:51), mlp_enc (model/e2e_attention.py:256) and their backward
// products.  Each fp32 operand x is split as x = hi + lo with hi = the TF32 the tensor core sees
// when it reads x (top 19 bits) and lo = tf32_rn(x - hi); three MMAs accumulate
// hi*hi + lo*hi + hi*lo in an fp32 TMEM accumulator (the dropped lo*lo term is ~2^-22 relative).
//
// Structure (one CTA per 128 x BN output tile, 192 threads):
//   warp 0      : TMA producer  -- cp.async.bulk.tensor.2d (SWIZZLE_128B boxes) into a smem ring
//   warp 1      : MMA issuer    -- one elected lane issues tcgen05.mma.cta_group::1.kind::tf32
//   warps 2..5  : converters    -- read each landed stage, write the `lo` copies (same swizzled layout)
//                 then epilogue -- tcgen05.ld the accumulator, add bias, store C
// Operands may be K-major ([rows][K], the nn.Linear layout) or MN-major ([K][rows]); the latter is
// what the backward products need (dX = g W, dW = g^T X) and is expressed purely through the TMA box
// shape and the UMMA descriptors -- no transposed copies.
#include <cuda.h>

#include "common.cuh"
#include "tc_common.cuh"

namespace re2e {
namespace {

constexpr int kBM = 128;
constexpr int kBK = 32;                 // fp32 elements per k-block = one 128 B swizzle row
constexpr int kConvWarps = 8;              // converter warps; the first four double as the epilogue warps
constexpr int kGemmThreads = 64 + 32 * kConvWarps;

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void *p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// 2-D fp32 tensor map: `inner` contiguous elements, `outer` rows of pitch `ld` elements; box 32 x box_outer,
// 128 B swizzle, out-of-bounds elements read as zero.
// mn_major operands use the 128B-span / 32B-atom swizzle: the only shared-memory layout tcgen05 accepts for MN-major
// 32-bit (tf32) operands (UMMA LayoutType SWIZZLE_128B_BASE32B = Swizzle<2,5,2> on the byte address).
int make_tmap(CUtensorMap *tm, const float *ptr, long long inner, long long outer, long long ld, int box_outer,
              bool mn_major) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return RE2E_E_UNSUPPORTED;
  cuuint64_t gdim[2] = {(cuuint64_t)inner, (cuuint64_t)outer};
  cuuint64_t gstr[1] = {(cuuint64_t)ld * sizeof(float)};
  cuuint32_t box[2] = {(cuuint32_t)kBK, (cuuint32_t)box_outer};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float *>(ptr), gdim, gstr, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE,
                   mn_major ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? RE2E_OK : RE2E_E_ARG;
}

// ---- device helpers ------------------------------------------------------------------------------
__device__ __forceinline__ void tma_load_2d(void *dst, const CUtensorMap *tm, int c0, int c1, uint64_t *bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
          smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(smem_u32(bar))
      : "memory");
}
struct GemmParams {
  float *C;
  const float *bias;
  int M, N, K, ldc, accumulate;
  int tma_c;    // C is 16 B aligned with a 16 B row pitch: the epilogue goes through the TMA store / reduce unit
  int kb_per;   // k-blocks per split (gridDim.z splits); split > 1: partial tiles are added with red.global
};

// shared -> global 2-D tensor store / fp32 reduce-add of one 32 x 32 box (SWIZZLE_128B staging); partial boxes at
// the M / N edges are clipped by the TMA unit
__device__ __forceinline__ void tma_store_2d(const CUtensorMap *tm, int c0, int c1, const void *src) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];" ::"l"(
                   reinterpret_cast<uint64_t>(tm)),
               "r"(c0), "r"(c1), "r"(smem_u32(src))
               : "memory");
}
__device__ __forceinline__ void tma_reduce_add_2d(const CUtensorMap *tm, int c0, int c1, const void *src) {
  asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%1, %2}], [%3];" ::"l"(
                   reinterpret_cast<uint64_t>(tm)),
               "r"(c0), "r"(c1), "r"(smem_u32(src))
               : "memory");
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, float a, float b, float c, float d) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

__device__ __forceinline__ void red_add4(float *p, float4 v) {
  asm volatile("red.global.add.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
               : "memory");
}

template <bool A_MN, bool B_MN, int BN, int STAGES>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_tf32x3_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                   const __grid_constant__ CUtensorMap tmC, const GemmParams p) {
  extern __shared__ __align__(1024) unsigned char smraw[];
  constexpr int A_BYTES = kBM * kBK * 4;         // 16 KB
  constexpr int B_BYTES = BN * kBK * 4;
  constexpr int STAGE_BYTES = 2 * (A_BYTES + B_BYTES);
  constexpr uint32_t TMEM_COLS = BN <= 32 ? 32 : BN <= 64 ? 64 : BN <= 128 ? 128 : 256;
  // instruction descriptor: D=f32, A=B=tf32, majors, N>>3, M>>4
  constexpr uint32_t IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((A_MN ? 1u : 0u) << 15) |
                             ((B_MN ? 1u : 0u) << 16) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(kBM >> 4) << 24);
  // smem: [stages][A_hi | B_hi | A_lo | B_lo] then barriers
  unsigned char *stage0 = smraw;
  uint64_t *full = reinterpret_cast<uint64_t *>(smraw + (size_t)STAGES * STAGE_BYTES);
  uint64_t *conv = full + STAGES;
  uint64_t *empty = conv + STAGES;
  uint64_t *tmem_full = empty + STAGES;
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tmem_full + 1);
  float *bias_s = reinterpret_cast<float *>(smraw + (size_t)STAGES * STAGE_BYTES + 1024);   // [BN] this tile's bias

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m0 = blockIdx.x * kBM, n0 = blockIdx.y * BN;
  // this CTA's slice of the K loop (split-K over gridDim.z keeps every tensor-core accumulation chain
  // <= kb_per*32 products: the TMEM accumulator adds with truncation, whose bias grows linearly in K)
  const int kb_begin = blockIdx.z * p.kb_per;
  const int nkb = min((p.K + kBK - 1) / kBK - kb_begin, p.kb_per);
  const bool split = gridDim.z > 1;

  if (threadIdx.x == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmA)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmB)) : "memory");
    if (p.tma_c) asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmC)) : "memory");
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&conv[s], kConvWarps);
      mbar_init(&empty[s], 1);
    }
    mbar_init(tmem_full, 1);
    mbar_fence_init();
  }
  if (warp == 1) {  // TMEM allocation by one full warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"(TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (threadIdx.x >= 64) {   // bias of this tile's columns (zero when absent / not this split's job)
    const bool use_bias = p.bias != nullptr && blockIdx.z == 0;
    for (int i = threadIdx.x - 64; i < BN; i += kGemmThreads - 64)
      bias_s[i] = (use_bias && n0 + i < p.N) ? __ldg(p.bias + n0 + i) : 0.0f;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      for (int kb = 0; kb < nkb; ++kb) {
        const int s = kb % STAGES;
        if (kb >= STAGES) mbar_wait(&empty[s], (uint32_t)(((kb / STAGES) - 1) & 1));
        unsigned char *st = stage0 + (size_t)s * STAGE_BYTES;
        mbar_expect_tx(&full[s], A_BYTES + B_BYTES);
        const int k0 = (kb_begin + kb) * kBK;
        if (!A_MN) {
          tma_load_2d(st, &tmA, k0, m0, &full[s]);
        } else {
#pragma unroll
          for (int j = 0; j < kBM / 32; ++j) tma_load_2d(st + j * 4096, &tmA, m0 + 32 * j, k0, &full[s]);
        }
        if (!B_MN) {
          tma_load_2d(st + A_BYTES, &tmB, k0, n0, &full[s]);
        } else {
#pragma unroll
          for (int j = 0; j < BN / 32; ++j) tma_load_2d(st + A_BYTES + j * 4096, &tmB, n0 + 32 * j, k0, &full[s]);
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    if (lane == 0) {
      for (int kb = 0; kb < nkb; ++kb) {
        const int s = kb % STAGES;
        mbar_wait(&conv[s], (uint32_t)((kb / STAGES) & 1));
        tc_fence_after();
        const uint32_t a_hi = smem_u32(stage0 + (size_t)s * STAGE_BYTES);
        const uint32_t b_hi = a_hi + A_BYTES;
        const uint32_t a_lo = b_hi + B_BYTES;
        const uint32_t b_lo = a_lo + A_BYTES;
#pragma unroll
        for (int k = 0; k < kBK / 8; ++k) {
          // K-major (SWIZZLE_128B): 8 tf32 = 32 B further along the swizzled 128 B row, 8-row groups 1 KB apart.
          // MN-major (SWIZZLE_128B_BASE32B): a box is 32 k-rows x 128 B (32 mn); the canonical atom is 4 k-rows
          // (SBO = 512 B between 4-k groups), 32-mn blocks are LBO = 4 KB apart, one MMA (K = 8) = 1 KB.
          const uint32_t ao = A_MN ? k * 1024 : k * 32;
          const uint32_t bo = B_MN ? k * 1024 : k * 32;
          const uint64_t dah = A_MN ? umma_desc(a_hi + ao, 4096, 512, 1) : umma_desc(a_hi + ao, 16, 1024, 2);
          const uint64_t dal = A_MN ? umma_desc(a_lo + ao, 4096, 512, 1) : umma_desc(a_lo + ao, 16, 1024, 2);
          const uint64_t dbh = B_MN ? umma_desc(b_hi + bo, 4096, 512, 1) : umma_desc(b_hi + bo, 16, 1024, 2);
          const uint64_t dbl = B_MN ? umma_desc(b_lo + bo, 4096, 512, 1) : umma_desc(b_lo + bo, 16, 1024, 2);
          umma_tf32(tmem_base, dah, dbh, IDESC, (kb | k) ? 1u : 0u);
          umma_tf32(tmem_base, dal, dbh, IDESC, 1u);
          umma_tf32(tmem_base, dah, dbl, IDESC, 1u);
        }
        umma_commit(&empty[s]);  // frees the stage once these MMAs have read it
      }
      umma_commit(tmem_full);    // accumulator complete
    }
  } else {
    // ===== converters (lo = tf32(x - hi)), then epilogue =====
    const int ctid = threadIdx.x - 64;  // 0 .. 32*kConvWarps-1
    for (int kb = 0; kb < nkb; ++kb) {
      const int s = kb % STAGES;
      mbar_wait(&full[s], (uint32_t)((kb / STAGES) & 1));
      const float4 *hi = reinterpret_cast<const float4 *>(stage0 + (size_t)s * STAGE_BYTES);
      float4 *lo = reinterpret_cast<float4 *>(stage0 + (size_t)s * STAGE_BYTES + A_BYTES + B_BYTES);
      constexpr int N4 = (A_BYTES + B_BYTES) / 16;
#pragma unroll 4
      for (int i = ctid; i < N4; i += 32 * kConvWarps) {
        const float4 x = hi[i];
        lo[i] = make_float4(tf32_lo(x.x), tf32_lo(x.y), tf32_lo(x.z), tf32_lo(x.w));
      }
      fence_proxy_async_smem();  // generic-proxy writes -> visible to the tensor core's async-proxy reads
      __syncwarp();
      if (lane == 0) mbar_arrive(&conv[s]);
    }
    // epilogue (warps 2..5): warp w may touch TMEM lanes [32*(w%4), +32)
    if (warp < 6) {
    mbar_wait(tmem_full, 0);
    tc_fence_after();
    const int q = warp & 3;
    const int row = m0 + 32 * q + lane;
    if (p.tma_c) {
      // coalesced asynchronous epilogue: TMEM -> registers (+bias) -> 128 B-swizzled staging rows in the (now idle)
      // operand ring -> one TMA box store (or fp32 reduce-add for split-K / accumulate) per 32 x 32 block,
      // double buffered per warp.  The SM issues 8 conflict-minimal STS.128 per block instead of 8 row-strided
      // STG.128 (32 sectors each), and never waits for the global writes.
      unsigned char *ebuf = stage0 + (size_t)q * 8192;
      const bool add = split || p.accumulate;
      const bool rows_ok = m0 + 32 * q < p.M;
      const int n_al = p.N & ~3;
#pragma unroll 1
      for (int c = 0; c < BN / 32; ++c) {
        const int col0 = n0 + c * 32;
        if (col0 >= p.N) break;
        if (c >= 2) {
          if (lane == 0) bulk_wait_read<1>();   // the block staged two iterations ago has left shared memory
          __syncwarp();
        }
        float v[32];
        tmem_ld32(tmem_base + ((uint32_t)(32 * q) << 16) + (uint32_t)(c * 32), v);
        const uint32_t base = smem_u32(ebuf + (size_t)(c & 1) * 4096) + (uint32_t)lane * 128u;
#pragma unroll
        for (int j4 = 0; j4 < 8; ++j4) {
          const float4 b4 = *reinterpret_cast<const float4 *>(bias_s + c * 32 + 4 * j4);
          st_shared_v4(base + (uint32_t)((j4 ^ (lane & 7)) << 4), v[4 * j4] + b4.x, v[4 * j4 + 1] + b4.y,
                       v[4 * j4 + 2] + b4.z, v[4 * j4 + 3] + b4.w);
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0 && rows_ok && col0 < n_al) {
          if (add) tma_reduce_add_2d(&tmC, col0, m0 + 32 * q, ebuf + (size_t)(c & 1) * 4096);
          else tma_store_2d(&tmC, col0, m0 + 32 * q, ebuf + (size_t)(c & 1) * 4096);
          bulk_commit();
        }
        // ragged tail (N % 4 != 0): the TMA unit clips in 16 B units, so the tensor map ends at N & ~3 and the last
        // 1..3 columns are written from registers (one 32-column block of the whole matrix takes this branch)
        if (n_al < p.N && n_al >= col0 && n_al < col0 + 32 && row < p.M) {
          float *dst = p.C + (size_t)row * p.ldc + col0;
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (col0 + j >= n_al && col0 + j < p.N) {
              const float val = v[j] + bias_s[c * 32 + j];
              if (split) atomicAdd(dst + j, val);
              else dst[j] = p.accumulate ? dst[j] + val : val;
            }
        }
      }
      if (lane == 0) bulk_wait_read<0>();
      __syncwarp();
    } else {
    const bool vec = false;   // this path is only taken when C is not 16 B addressable
#pragma unroll 1
    for (int c = 0; c < BN / 32; ++c) {
      float v[32];
      tmem_ld32(tmem_base + ((uint32_t)(32 * q) << 16) + (uint32_t)(c * 32), v);
      const int col0 = n0 + c * 32;
      if (row < p.M && col0 < p.N) {
        float *dst = p.C + (size_t)row * p.ldc + col0;
        if (p.bias && blockIdx.z == 0) {
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (col0 + j < p.N) v[j] += __ldg(p.bias + col0 + j);
        }
        if (split) {  // C was zeroed by the host side unless `accumulate`
          if (vec && col0 + 32 <= p.N) {
#pragma unroll
            for (int j = 0; j < 32; j += 4) red_add4(dst + j, make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]));
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (col0 + j < p.N) atomicAdd(dst + j, v[j]);
          }
        } else if (vec && col0 + 32 <= p.N) {
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            float4 o = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
            if (p.accumulate) {
              const float4 old = *reinterpret_cast<const float4 *>(dst + j);
              o.x += old.x; o.y += old.y; o.z += old.z; o.w += old.w;
            }
            *reinterpret_cast<float4 *>(dst + j) = o;
          }
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (col0 + j < p.N) dst[j] = p.accumulate ? dst[j] + v[j] : v[j];
        }
      }
    }
    }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

// ------------------------------------------------------------------------------------------------
// Persistent variant: one CTA per SM loops over (m tile, n tile, k slice) work items; the fp32 accumulator is double
// buffered in TMEM (2 x BN columns), so the epilogue of item i (dedicated warps) and the prologue latency of item
// i+1 overlap the MMAs -- in the one-CTA-per-tile kernel above ~25-33 % of a CTA's life is setup + first-load latency
// + epilogue with the tensor pipe idle (profiles/r01_s4d_gemm_phases.txt).
//   warp 0       TMA producer (one lane)        warp 1        MMA issuer (one lane), TMEM alloc / dealloc
//   warps 2..9   converters (lo copies)         warps 10..13  epilogue (TMEM lane quarter = warp % 4)
// The epilogue writes straight from registers (16 B per lane and row; fp32 red.add for split-K / accumulate): it no
// longer sits on the critical path, and the operand ring keeps all of the shared memory.
// ------------------------------------------------------------------------------------------------
constexpr int kPersistThreads = 14 * 32;

template <bool A_MN, bool B_MN, int BN, int STAGES>
__global__ void __launch_bounds__(kPersistThreads, 1)
gemm_tf32x3_persist_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                           const GemmParams p, int MT, int NT, int n_items) {
  extern __shared__ __align__(1024) unsigned char smraw[];
  constexpr int A_BYTES = kBM * kBK * 4;
  constexpr int B_BYTES = BN * kBK * 4;
  constexpr int STAGE_BYTES = 2 * (A_BYTES + B_BYTES);
  constexpr uint32_t TMEM_COLS = 512;            // two BN-column accumulators (BN <= 256)
  constexpr uint32_t IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((A_MN ? 1u : 0u) << 15) |
                             ((B_MN ? 1u : 0u) << 16) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(kBM >> 4) << 24);
  unsigned char *stage0 = smraw;
  uint64_t *full = reinterpret_cast<uint64_t *>(smraw + (size_t)STAGES * STAGE_BYTES);
  uint64_t *conv = full + STAGES;
  uint64_t *empty = conv + STAGES;
  uint64_t *tmem_full = empty + STAGES;          // [2]
  uint64_t *tmem_empty = tmem_full + 2;          // [2]
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tmem_empty + 2);
  float *bias_s = reinterpret_cast<float *>(smraw + (size_t)STAGES * STAGE_BYTES + 1024);   // [2][BN]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nkb_total = (p.K + kBK - 1) / kBK;
  const bool split = nkb_total > p.kb_per;

  if (threadIdx.x == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmA)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmB)) : "memory");
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&conv[s], kConvWarps);
      mbar_init(&empty[s], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tmem_full[i], 1);
      mbar_init(&tmem_empty[i], 4);
    }
    mbar_fence_init();
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"(TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  auto decode = [&](int w, int &m0, int &n0, int &kb_begin, int &nkb) {
    const int mt = w % MT, r = w / MT, nt = r % NT, ks = r / NT;
    m0 = mt * kBM;
    n0 = nt * BN;
    kb_begin = ks * p.kb_per;
    nkb = min(nkb_total - kb_begin, p.kb_per);
  };

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      int it = 0;
      for (int w = blockIdx.x; w < n_items; w += gridDim.x) {
        int m0, n0, kb_begin, nkb;
        decode(w, m0, n0, kb_begin, nkb);
        for (int kb = 0; kb < nkb; ++kb, ++it) {
          const int s = it % STAGES;
          if (it >= STAGES) mbar_wait(&empty[s], (uint32_t)(((it / STAGES) - 1) & 1));
          unsigned char *st = stage0 + (size_t)s * STAGE_BYTES;
          mbar_expect_tx(&full[s], A_BYTES + B_BYTES);
          const int k0 = (kb_begin + kb) * kBK;
          if (!A_MN) {
            tma_load_2d(st, &tmA, k0, m0, &full[s]);
          } else {
#pragma unroll
            for (int j = 0; j < kBM / 32; ++j) tma_load_2d(st + j * 4096, &tmA, m0 + 32 * j, k0, &full[s]);
          }
          if (!B_MN) {
            tma_load_2d(st + A_BYTES, &tmB, k0, n0, &full[s]);
          } else {
#pragma unroll
            for (int j = 0; j < BN / 32; ++j) tma_load_2d(st + A_BYTES + j * 4096, &tmB, n0 + 32 * j, k0, &full[s]);
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    if (lane == 0) {
      int it = 0, li = 0;
      for (int w = blockIdx.x; w < n_items; w += gridDim.x, ++li) {
        int m0, n0, kb_begin, nkb;
        decode(w, m0, n0, kb_begin, nkb);
        const int buf = li & 1;
        mbar_wait(&tmem_empty[buf], (uint32_t)(((li >> 1) & 1) ^ 1));   // epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(buf * BN);
        for (int kb = 0; kb < nkb; ++kb, ++it) {
          const int s = it % STAGES;
          mbar_wait(&conv[s], (uint32_t)((it / STAGES) & 1));
          tc_fence_after();
          const uint32_t a_hi = smem_u32(stage0 + (size_t)s * STAGE_BYTES);
          const uint32_t b_hi = a_hi + A_BYTES;
          const uint32_t a_lo = b_hi + B_BYTES;
          const uint32_t b_lo = a_lo + A_BYTES;
#pragma unroll
          for (int k = 0; k < kBK / 8; ++k) {
            const uint32_t ao = A_MN ? k * 1024 : k * 32;
            const uint32_t bo = B_MN ? k * 1024 : k * 32;
            const uint64_t dah = A_MN ? umma_desc(a_hi + ao, 4096, 512, 1) : umma_desc(a_hi + ao, 16, 1024, 2);
            const uint64_t dal = A_MN ? umma_desc(a_lo + ao, 4096, 512, 1) : umma_desc(a_lo + ao, 16, 1024, 2);
            const uint64_t dbh = B_MN ? umma_desc(b_hi + bo, 4096, 512, 1) : umma_desc(b_hi + bo, 16, 1024, 2);
            const uint64_t dbl = B_MN ? umma_desc(b_lo + bo, 4096, 512, 1) : umma_desc(b_lo + bo, 16, 1024, 2);
            umma_tf32(d_tmem, dah, dbh, IDESC, (kb | k) ? 1u : 0u);
            umma_tf32(d_tmem, dal, dbh, IDESC, 1u);
            umma_tf32(d_tmem, dah, dbl, IDESC, 1u);
          }
          umma_commit(&empty[s]);
        }
        umma_commit(&tmem_full[buf]);
      }
    }
  } else if (warp < 2 + kConvWarps) {
    // ===== converters =====
    const int ctid = threadIdx.x - 64;
    int it = 0;
    for (int w = blockIdx.x; w < n_items; w += gridDim.x) {
      int m0, n0, kb_begin, nkb;
      decode(w, m0, n0, kb_begin, nkb);
      for (int kb = 0; kb < nkb; ++kb, ++it) {
        const int s = it % STAGES;
        mbar_wait(&full[s], (uint32_t)((it / STAGES) & 1));
        const float4 *hi = reinterpret_cast<const float4 *>(stage0 + (size_t)s * STAGE_BYTES);
        float4 *lo = reinterpret_cast<float4 *>(stage0 + (size_t)s * STAGE_BYTES + A_BYTES + B_BYTES);
        constexpr int N4 = (A_BYTES + B_BYTES) / 16;
#pragma unroll 4
        for (int i = ctid; i < N4; i += 32 * kConvWarps) {
          const float4 x = hi[i];
          lo[i] = make_float4(tf32_lo(x.x), tf32_lo(x.y), tf32_lo(x.z), tf32_lo(x.w));
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(&conv[s]);
      }
    }
  } else {
    // ===== epilogue warps =====
    const int q = warp & 3;
    const int etid = threadIdx.x - 32 * (2 + kConvWarps);   // 0..127
    const bool vec = ((p.ldc & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.C) & 15u) == 0);
    int li = 0;
    for (int w = blockIdx.x; w < n_items; w += gridDim.x, ++li) {
      int m0, n0, kb_begin, nkb;
      decode(w, m0, n0, kb_begin, nkb);
      const int buf = li & 1;
      float *bs = bias_s + buf * BN;
      // bias of this item's columns (the buffer was last read two items ago; every epilogue warp has passed the
      // barrier of the item in between)
      {
        const bool use_bias = p.bias != nullptr && kb_begin == 0;
        for (int i = etid; i < BN; i += 128) bs[i] = (use_bias && n0 + i < p.N) ? __ldg(p.bias + n0 + i) : 0.0f;
      }
      asm volatile("bar.sync 1, 128;" ::: "memory");
      mbar_wait(&tmem_full[buf], (uint32_t)((li >> 1) & 1));
      tc_fence_after();
      const int row = m0 + 32 * q + lane;
#pragma unroll 1
      for (int c = 0; c < BN / 32; ++c) {
        const int col0 = n0 + c * 32;
        if (col0 >= p.N) break;
        float v[32];
        tmem_ld32(tmem_base + ((uint32_t)(32 * q) << 16) + (uint32_t)(buf * BN + c * 32), v);
        if (row < p.M) {
          float *dst = p.C + (size_t)row * p.ldc + col0;
          if (vec && col0 + 32 <= p.N) {
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              const float4 b4 = *reinterpret_cast<const float4 *>(bs + c * 32 + j);
              float4 o = make_float4(v[j] + b4.x, v[j + 1] + b4.y, v[j + 2] + b4.z, v[j + 3] + b4.w);
              if (split) {
                red_add4(dst + j, o);
              } else {
                if (p.accumulate) {
                  const float4 old = *reinterpret_cast<const float4 *>(dst + j);
                  o.x += old.x; o.y += old.y; o.z += old.z; o.w += old.w;
                }
                *reinterpret_cast<float4 *>(dst + j) = o;
              }
            }
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (col0 + j < p.N) {
                const float val = v[j] + bs[c * 32 + j];
                if (split) atomicAdd(dst + j, val);
                else dst[j] = p.accumulate ? dst[j] + val : val;
              }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[buf]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

template <bool A_MN, bool B_MN, int BN, int STAGES>
int launch_gemm_persist(const CUtensorMap &ta, const CUtensorMap &tb, const GemmParams &prm, cudaStream_t st) {
  constexpr size_t smem = (size_t)STAGES * 2 * (kBM * kBK * 4 + BN * kBK * 4) + 1024 + 2 * BN * 4;
  auto kern = gemm_tf32x3_persist_kernel<A_MN, B_MN, BN, STAGES>;
  int rc = ensure_smem(reinterpret_cast<const void *>(kern), smem);
  if (rc != RE2E_OK) return rc;
  const int nkb = (prm.K + kBK - 1) / kBK;
  const int MT = (prm.M + kBM - 1) / kBM, NT = (prm.N + BN - 1) / BN, KS = (nkb + prm.kb_per - 1) / prm.kb_per;
  const long long items = (long long)MT * NT * KS;
  if (items > 0x7fffffff) return RE2E_E_UNSUPPORTED;
  if (KS > 1 && !prm.accumulate) {
    cudaError_t e = cudaMemset2DAsync(prm.C, sizeof(float) * (size_t)prm.ldc, 0, sizeof(float) * (size_t)prm.N,
                                      (size_t)prm.M, st);
    if (e != cudaSuccess) return (int)e;
  }
  const int grid = (int)(items < num_sms() ? items : num_sms());
  kern<<<grid, kPersistThreads, smem, st>>>(ta, tb, prm, MT, NT, (int)items);
  count_launch();
  return launch_status();
}

template <int BN, int STAGES>
int dispatch_major_persist(int a_mn, int b_mn, const CUtensorMap &ta, const CUtensorMap &tb, const GemmParams &prm,
                           cudaStream_t st) {
  if (!a_mn && !b_mn) return launch_gemm_persist<false, false, BN, STAGES>(ta, tb, prm, st);
  if (!a_mn && b_mn) return launch_gemm_persist<false, true, BN, STAGES>(ta, tb, prm, st);
  if (a_mn && !b_mn) return launch_gemm_persist<true, false, BN, STAGES>(ta, tb, prm, st);
  return launch_gemm_persist<true, true, BN, STAGES>(ta, tb, prm, st);
}

template <bool A_MN, bool B_MN, int BN, int STAGES>
int launch_gemm(const CUtensorMap &ta, const CUtensorMap &tb, const CUtensorMap &tc, const GemmParams &prm,
                cudaStream_t st) {
  constexpr size_t smem = (size_t)STAGES * 2 * (kBM * kBK * 4 + BN * kBK * 4) + 1024 + BN * 4;
  auto kern = gemm_tf32x3_kernel<A_MN, B_MN, BN, STAGES>;
  int rc = ensure_smem(reinterpret_cast<const void *>(kern), smem);
  if (rc != RE2E_OK) return rc;
  const int nkb = (prm.K + kBK - 1) / kBK;
  dim3 grid((prm.M + kBM - 1) / kBM, (prm.N + BN - 1) / BN, (nkb + prm.kb_per - 1) / prm.kb_per);
  if (grid.z > 1 && !prm.accumulate) {
    cudaError_t e = cudaMemset2DAsync(prm.C, sizeof(float) * (size_t)prm.ldc, 0, sizeof(float) * (size_t)prm.N,
                                      (size_t)prm.M, st);
    if (e != cudaSuccess) return (int)e;
  }
  kern<<<grid, kGemmThreads, smem, st>>>(ta, tb, tc, prm);
  count_launch();
  return launch_status();
}

template <int BN, int STAGES>
int dispatch_major(int a_mn, int b_mn, const CUtensorMap &ta, const CUtensorMap &tb, const CUtensorMap &tc,
                   const GemmParams &prm, cudaStream_t st) {
  if (!a_mn && !b_mn) return launch_gemm<false, false, BN, STAGES>(ta, tb, tc, prm, st);
  if (!a_mn && b_mn) return launch_gemm<false, true, BN, STAGES>(ta, tb, tc, prm, st);
  if (a_mn && !b_mn) return launch_gemm<true, false, BN, STAGES>(ta, tb, tc, prm, st);
  return launch_gemm<true, true, BN, STAGES>(ta, tb, tc, prm, st);
}

}  // namespace
}  // namespace re2e

using namespace re2e;

// C[M,N] (+)= Aop[M,K] * Bop[N,K]^T (+ bias[N]);  a_mn = 0: A is [M][lda>=K] (K contiguous), a_mn = 1: A is
// stored [K][lda>=M] (M contiguous).  Same for B with N.  lda, ldb multiples of 4; A, B 16 B aligned.
extern "C" int re2e_gemm_tf32x3(const float *A, int lda, int a_mn, const float *B, int ldb, int b_mn, float *C,
                                int ldc, const float *bias, int M, int N, int K, int accumulate, void *stream) {
  RE2E_CHECK_ARG(A && B && C && M > 0 && N > 0 && K > 0 && ldc >= N);
  RE2E_CHECK_ARG((lda & 3) == 0 && (ldb & 3) == 0 && aligned16(A) && aligned16(B));
  RE2E_CHECK_ARG(lda >= (a_mn ? M : K) && ldb >= (b_mn ? N : K));
  CUtensorMap ta, tb, tc;
  int rc;
  const int BN = (N % 256 == 0 || N > 1024) ? 256 : 160;
  if (!a_mn) rc = make_tmap(&ta, A, K, M, lda, kBM, false);
  else rc = make_tmap(&ta, A, M, K, lda, kBK, true);
  if (rc != RE2E_OK) return rc;
  if (!b_mn) rc = make_tmap(&tb, B, K, N, ldb, BN, false);
  else rc = make_tmap(&tb, B, N, K, ldb, kBK, true);
  if (rc != RE2E_OK) return rc;
  GemmParams prm;
  prm.C = C; prm.bias = bias; prm.M = M; prm.N = N; prm.K = K; prm.ldc = ldc; prm.accumulate = accumulate;
  const int nkb = (K + kBK - 1) / kBK;
  // K > 768: split-K (bounds the truncating TMEM accumulation chain to <= 640 products).  The slice length is chosen
  // per shape so that the CTA count fills whole waves of the machine: cost = waves * (k-blocks + fixed per-CTA
  // overhead of ~4 k-block times for prologue + epilogue).
  prm.kb_per = nkb;
  if (nkb > 24) {
    const int sms = num_sms();
    const long long tiles = (long long)((M + kBM - 1) / kBM) * ((N + BN - 1) / BN);
    long long best = -1;
    for (int kp = 12; kp <= 20; ++kp) {
      const long long ctas = tiles * ((nkb + kp - 1) / kp);
      const long long cost = ((ctas + sms - 1) / sms) * (kp + 4);
      if (best < 0 || cost < best) { best = cost; prm.kb_per = kp; }
    }
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  {
    // more work items than SMs: persistent tile loop with a double-buffered TMEM accumulator.  A single wave gains
    // nothing from the tile loop and runs the one-CTA-per-tile kernel below.
    const long long items = (long long)((M + kBM - 1) / kBM) * ((N + BN - 1) / BN) * ((nkb + prm.kb_per - 1) / prm.kb_per);
    if (items > num_sms()) {
      prm.tma_c = 0;
      if (BN == 256) return dispatch_major_persist<256, 2>(a_mn, b_mn, ta, tb, prm, st);
      return dispatch_major_persist<160, 3>(a_mn, b_mn, ta, tb, prm, st);
    }
  }
  // epilogue through the TMA store unit when C is TMA-addressable (16 B aligned, 16 B row pitch); 32 x 32 boxes
  prm.tma_c = ((ldc & 3) == 0 && aligned16(C) && N >= 4) ? 1 : 0;
  if (prm.tma_c) {
    if ((rc = make_tmap(&tc, C, N & ~3, M, ldc, 32, false)) != RE2E_OK) return rc;
  } else {
    tc = ta;   // unused
  }
  if (BN == 256) return dispatch_major<256, 2>(a_mn, b_mn, ta, tb, tc, prm, st);
  return dispatch_major<160, 3>(a_mn, b_mn, ta, tb, tc, prm, st);
}
