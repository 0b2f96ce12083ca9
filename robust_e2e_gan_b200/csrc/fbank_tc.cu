// Fused differentiable front-end on the 5th-generation tensor cores (tcgen05 / TMEM), sm_100a.
//
//   forward : x = act(mask) * valid * mag  ->  x^2  ->  P = x^2 . fc (F x M mel projection, 3xTF32)  ->  clamp, log, CMVN
//             (model/enhance_model.py:157-164 + model/feat_model.py:118-135)
//   backward: dP = dY * G ;  d(x^2) = dP . fc^T (3xTF32)  ;  d_in = d(x^2) * 2 x * d x/d in
//
// Why tensor cores here: the projection is 2*N*F*M = 0.53 GFLOP per pass at the bench shape; as fp32 FMAs fed from
// shared memory it costs ~5x the time the HBM stream needs (measured: 127 us vs 9 us), on tcgen05 it disappears
// behind the stream.  fp32 parity (1e-4) needs the 3xTF32 split: x = hi + lo (hi = the 19 bits the tensor core
// reads, lo = x - hi), D += hi*hi + lo*hi + hi*lo.
//
// Forward structure (one persistent CTA per SM, each owning a contiguous range of frames):
//   warps 0..15 : converters -- coalesced row-segment loads of mask / mag (rows are 1028 B: only 4 B aligned, so no
//                 TMA; 8 B per lane on rows of equal parity when F = 257, else 4 B per lane), register prefetch,
//                 sigmoid/mask/square, hi/lo split, store into the 128B-swizzled K-major A tiles (128 frames x 32 bins)
//                 of a shared-memory ring
//   warp 20     : one lane issues tcgen05.mma.kind::tf32, TWO per 8-bin k-step: A_hi x [B_hi | B_lo] (the filter bank
//                 is resident per chunk as one tile of hi rows followed by lo rows, N = 2 round8(mel)) and A_lo x B_hi
//                 into a second column range of one of two TMEM accumulators -- A_hi is fetched once, 12 KB of operands
//                 per k-step instead of 16.5 KB for three separate products (the MMAs share the shared-memory port with
//                 the converters' stores: profiles/r01_s5_frontend_phases.txt)
//   warps 16..19: epilogue -- tcgen05.ld the three column ranges of the finished accumulator (lane <-> frame), sum,
//                 clamp/log/CMVN, store Y and G
// Algorithmic HBM bytes: 4*N*(2F + 2M) masked with G, 4*N*(F + M) plain.
#include "common.cuh"
#include "tc_common.cuh"

namespace re2e {
namespace {

constexpr int kCW = 16;                          // converter warps
constexpr int kEW = 4;                           // epilogue warps (one per TMEM lane quarter)
constexpr int kTcThreads = (kCW + kEW + 1) * 32; // + MMA warp
constexpr int kRows = 128;                       // frames per MMA tile
constexpr int kKC = 32;                          // bins per k-chunk (one 128 B swizzle row)
constexpr int kATile = kRows * 128;              // bytes of one A tile (hi or lo)
constexpr float kClampTc = 1e-7f;
constexpr int kMaxStagesTc = 4;

struct FbTcParams {
  const float *mask, *mag, *fc, *cmvn;
  const int32_t *lens;
  float *Y, *G, *enh;
  int mask_is_logit, N, T, F, M;
  int NB;            // UMMA N: mel channels padded to a multiple of 16
  int MB;            // filter-bank rows kept per chunk in shared memory: mel channels padded to a multiple of 8 (one
                     // swizzle group).  The MMA reads NB rows: rows [MB, NB) alias the next chunk / the A ring -- they
                     // only reach accumulator columns >= M, which the epilogue never stores
  int nchunks;       // 32-bin chunks that go through the tensor core
  int ksteps_last;   // 8-bin MMA steps in the last chunk
  int ntail;         // trailing bins (<= 4, e.g. the Nyquist bin of F = 257) added by the epilogue as plain FMAs
  int rows_per_cta;
  int nstages;
};

__device__ __forceinline__ float tf32_trunc_lo(float x) {
  // the tensor core reads the top 19 bits of an fp32 operand; what it drops is re-fed as a second operand
  return x - __uint_as_float(__float_as_uint(x) & 0xFFFFE000u);
}
__device__ __forceinline__ float sigmoid_fast(float x) { return __fdividef(1.0f, 1.0f + __expf(-x)); }

// FC: compile-time number of bins (257) so that the row-strided loads get immediate offsets; 0 = run-time p.F
template <bool MASKED, int DEPTH, int FC, bool PAIR>
__global__ void __launch_bounds__(kTcThreads, 1) fbank_tc_fwd_kernel(const FbTcParams p) {
  extern __shared__ __align__(1024) unsigned char smraw_[];
  unsigned char *sm = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(smraw_) + 1023) & ~(uintptr_t)1023);
  const int NB = p.NB, NS = p.nstages, F = FC > 0 ? FC : p.F, M = p.M;
  const int Fmma = p.nchunks * kKC < F ? p.nchunks * kKC : F;   // bins [0, Fmma) on the tensor core, [Fmma, F) in the epilogue
  // filter bank, per 32-bin chunk: [hi rows 0..MB | lo rows 0..MB) -- ONE K-major tile of 2 MB rows, so that
  // A_hi x [B_hi | B_lo] is a single MMA of N = 2 MB; its first NB rows double as the B_hi operand of A_lo x B_hi
  const int fc_bytes = p.nchunks * p.MB * 128;          // bytes of the hi (or lo) rows of all chunks
  const int fc_chunk = 2 * p.MB * 128;
  unsigned char *fc_hi = sm;
  unsigned char *fc_lo = sm + p.MB * 128;
  unsigned char *stage0 = sm + 2 * fc_bytes;
  const int WD = 2 * p.MB + NB;                         // accumulator columns per buffer: [hi.hi | hi.lo | lo.hi]
  uint64_t *full = reinterpret_cast<uint64_t *>(stage0 + (size_t)NS * 2 * kATile);
  uint64_t *empty = full + kMaxStagesTc;
  uint64_t *tfull = empty + kMaxStagesTc;
  uint64_t *tempty = tfull + 2;
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tempty + 2);
  float *c0_s = reinterpret_cast<float *>(tmem_slot + 2);
  float *c1_s = c0_s + NB;
  float *fct_s = c1_s + NB;          // [ntail][NB] filter-bank rows of the trailing bins

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int row_begin = min(p.N, (int)blockIdx.x * p.rows_per_cta);
  const int row_end = min(p.N, row_begin + p.rows_per_cta);
  const int ntiles = (row_end - row_begin + kRows - 1) / kRows;
  const uint32_t tmem_cols = 2 * WD <= 32 ? 32u : 2 * WD <= 64 ? 64u : 2 * WD <= 128 ? 128u : 2 * WD <= 256 ? 256u : 512u;

  // ---- one-time setup: barriers, TMEM, filter bank (hi/lo, K-major, 128B swizzle), CMVN
  if (tid == 0) {
    for (int s = 0; s < NS; ++s) { mbar_init(&full[s], kCW); mbar_init(&empty[s], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], kEW); }
    mbar_fence_init();
  }
  if (warp == kCW + kEW) tmem_alloc(tmem_slot, tmem_cols);
  {
    float4 *z = reinterpret_cast<float4 *>(fc_hi);
    for (int i = tid; i < 2 * fc_bytes / 16; i += kTcThreads) z[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int i = tid; i < NB; i += kTcThreads) {
      c0_s[i] = (p.cmvn && i < M) ? __ldg(p.cmvn + i) : 0.0f;
      c1_s[i] = (p.cmvn && i < M) ? __ldg(p.cmvn + M + i) : 1.0f;
    }
    for (int i = tid; i < p.ntail * NB; i += kTcThreads) {
      const int kt = i / NB, m = i - kt * NB;
      fct_s[i] = m < M ? __ldg(p.fc + (size_t)(Fmma + kt) * M + m) : 0.0f;
    }
  }
  __syncthreads();
  for (int i = tid; i < Fmma * M; i += kTcThreads) {
    const int k = i / M, m = i - k * M;
    const float v = __ldg(p.fc + i);
    const int ch = k >> 5, kk = k & 31;
    const int off = ch * fc_chunk + (m >> 3) * 1024 + (m & 7) * 128 + ((((kk >> 2) ^ (m & 7))) << 4) + (kk & 3) * 4;
    *reinterpret_cast<float *>(fc_hi + off) = v;
    *reinterpret_cast<float *>(fc_lo + off) = tf32_trunc_lo(v);
  }
  fence_proxy_async_smem();   // the filter bank is read by the tensor core (async proxy)
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int nitems = ntiles * p.nchunks;

  if (PAIR && FC == 257 && warp < kCW) {
    // ================= converters, F = 257 (8 B per lane) =================
    // thread <-> (frames warp + 16 j, bins 64 g + 2 lane, +1): items of 64 bins that fill TWO ring stages, ONE 256 B
    // request per row and item instead of two of 128 B.  The SM accepts a limited number of load REQUESTS, not bytes
    // (tools/membench, profiles/r01_s5_membench.txt: 12.1 vs 17.4 us for the matrix from DRAM at equal registers).
    // A row starts at byte 1028 r, so only even rows are 8 B aligned.  The parity of warp + 16 j depends neither on j
    // nor on the tile: warps with odd rows load the pairs (2 lane + 1, 2 lane + 2) -- 8 B aligned again -- and store
    // the two bins to their own slots; lane 31's second bin belongs to the next item (for the last item it is the
    // Nyquist bin, which the epilogue handles), and bin 0 of every item comes from one extra 8-lane load (lane j <->
    // row j).  Needs four ring stages (see fbank_tc_fwd) -- with fewer the converters wait for the MMAs after every item.
    constexpr int PD = DEPTH / 2 > 0 ? DEPTH / 2 : 1;     // items in flight: the same registers as DEPTH 4 B items
    const int rr = warp & 7;
    const int hsel = lane >> 4;                           // this lane writes the item's first / second 32-bin chunk
    const uint32_t offp =
        (uint32_t)((warp >> 3) * 1024 + rr * 128 + ((((lane & 15) >> 1) ^ rr) << 4) + (lane & 1) * 8);
    const int par = (row_begin + warp) & 1;
    float2 mg[PD][8], mk[MASKED ? PD : 1][8];
    float eg[PD], ek[MASKED ? PD : 1];                    // element 0 of row j in lane j (first item of a tile, odd warps)
    const int npi = ntiles * 4;
    int l_row0 = row_begin, l_g = 0, l_item = 0;
    auto load = [&](float2 (&g)[8], float2 (&k)[8], float &e0g, float &e0k) {
      const int nj = max(0, (min(kRows, row_end - l_row0) - warp + 15) >> 4);
      const size_t base = (size_t)(l_row0 + warp) * 257 + 64 * l_g + 2 * lane + par;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const bool ok = j < nj;
        g[j] = ok ? ld_stream2(p.mag + base + j * 16 * 257) : make_float2(0.0f, 0.0f);
        if (MASKED) k[j] = ok ? ld_stream2(p.mask + base + j * 16 * 257) : make_float2(0.0f, 0.0f);
      }
      if (par) {
        const bool ok = lane < nj;
        const size_t b0 = (size_t)(l_row0 + warp + 16 * (lane & 7)) * 257 + 64 * l_g;
        e0g = ok ? ld_stream1(p.mag + b0) : 0.0f;
        if (MASKED) e0k = ok ? ld_stream1(p.mask + b0) : 0.0f;
      }
      ++l_item;
      if (++l_g == 4) { l_g = 0; l_row0 += kRows; }
    };
#pragma unroll
    for (int d = 0; d < PD; ++d) {
      eg[d] = 0.0f;
      ek[MASKED ? d : 0] = 0.0f;
      if (d < npi) load(mg[d], mk[MASKED ? d : 0], eg[d], ek[MASKED ? d : 0]);
    }

    int c_row0 = row_begin, c_g = 0, nj_c = 0, nchunk = 0;
    uint32_t vmask = 0xffu;
    int st = 0;
    uint32_t ph = 0;
    for (int q0 = 0; q0 < npi; q0 += PD) {
#pragma unroll
      for (int d = 0; d < PD; ++d) {
        const int q = q0 + d;
        if (q < npi) {
          if (c_g == 0) {   // new tile: rows of this warp inside it, and which of them are inside their utterance
            nj_c = max(0, (min(kRows, row_end - c_row0) - warp + 15) >> 4);
            if (MASKED && p.lens) {
              int row = c_row0 + warp;
              int b = row / p.T, t = row - b * p.T;
              int len = __ldg(p.lens + min(b, p.N / p.T - 1));
              vmask = 0;
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                vmask |= (t < len ? 1u : 0u) << j;
                t += 16;
                while (t >= p.T) { t -= p.T; ++b; len = __ldg(p.lens + min(b, p.N / p.T - 1)); }
              }
            }
          }
          const int s0 = st;
          const uint32_t ph0 = ph;
          if (++st == NS) { st = 0; ph ^= 1u; }
          const int s1 = st;
          const uint32_t ph1 = ph;
          if (++st == NS) { st = 0; ph ^= 1u; }
          if (nchunk >= NS) mbar_wait(&empty[s0], ph0 ^ 1u);
          if (nchunk + 1 >= NS) mbar_wait(&empty[s1], ph1 ^ 1u);
          nchunk += 2;
          unsigned char *sa = stage0 + (size_t)(hsel ? s1 : s0) * 2 * kATile + offp;
          const int kcol = 64 * c_g + 2 * lane;
          auto masked_x = [&](float g, float k, bool v) {
            if (!MASKED) return g;
            const float sg = p.mask_is_logit ? sigmoid_fast(k) : k;
            return v ? sg * g : 0.0f;
          };
          if (!par) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              if (j >= nj_c) break;   // warp-uniform: rows past the CTA's range (partial last tile) cost nothing
              const float2 g2 = mg[d][j], k2 = mk[MASKED ? d : 0][j];
              const bool v = (vmask >> j) & 1u;
              const float xa = masked_x(g2.x, k2.x, v), xb = masked_x(g2.y, k2.y, v);
              if (MASKED && p.enh) {
                float *eo = p.enh + (size_t)(c_row0 + warp + 16 * j) * 257 + kcol;
                eo[0] = xa;
                eo[1] = xb;
              }
              const float2 x2 = make_float2(xa * xa, xb * xb);
              *reinterpret_cast<float2 *>(sa + j * 2048) = x2;
              *reinterpret_cast<float2 *>(sa + kATile + j * 2048) = make_float2(tf32_trunc_lo(x2.x), tf32_trunc_lo(x2.y));
            }
          } else {
            // odd rows: the lane holds bins (2 lane + 1, 2 lane + 2) of the item; each goes to its own slot (lane 31's
            // second one belongs to the NEXT item, which fetches it itself: lane j < 8 holds bin 0 of row j in eg / ek)
            const int ka = 2 * lane + 1, kb = (2 * lane + 2) & 63;
            unsigned char *base0 = stage0 + (size_t)s0 * 2 * kATile, *base1 = stage0 + (size_t)s1 * 2 * kATile;
            const uint32_t rowoff = (uint32_t)((warp >> 3) * 1024 + rr * 128);
            unsigned char *pa = (ka >> 5 ? base1 : base0) + rowoff + (((((ka & 31) >> 2) ^ rr)) << 4) + (ka & 3) * 4;
            unsigned char *pb = (kb >> 5 ? base1 : base0) + rowoff + (((((kb & 31) >> 2) ^ rr)) << 4) + (kb & 3) * 4;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              if (j >= nj_c) break;
              const float2 g2 = mg[d][j], k2 = mk[MASKED ? d : 0][j];
              const bool v = (vmask >> j) & 1u;
              const float xa = masked_x(g2.x, k2.x, v), xb = masked_x(g2.y, k2.y, v);
              if (MASKED && p.enh) {
                float *eo = p.enh + (size_t)(c_row0 + warp + 16 * j) * 257 + kcol + 1;
                eo[0] = xa;
                if (lane < 31) eo[1] = xb;
              }
              const float xa2 = xa * xa, xb2 = xb * xb;
              *reinterpret_cast<float *>(pa + j * 2048) = xa2;
              *reinterpret_cast<float *>(pa + kATile + j * 2048) = tf32_trunc_lo(xa2);
              if (lane < 31) {
                *reinterpret_cast<float *>(pb + j * 2048) = xb2;
                *reinterpret_cast<float *>(pb + kATile + j * 2048) = tf32_trunc_lo(xb2);
              }
            }
            if (lane < nj_c) {   // bin 0 of the item for row `lane`
              const bool v = (vmask >> lane) & 1u;
              const float x0 = masked_x(eg[d], ek[MASKED ? d : 0], v);
              if (MASKED && p.enh) p.enh[(size_t)(c_row0 + warp + 16 * lane) * 257 + 64 * c_g] = x0;
              const float x02 = x0 * x0;
              unsigned char *p0 = base0 + rowoff + ((0 ^ rr) << 4) + lane * 2048;
              *reinterpret_cast<float *>(p0) = x02;
              *reinterpret_cast<float *>(p0 + kATile) = tf32_trunc_lo(x02);
            }
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) { mbar_arrive(&full[s0]); mbar_arrive(&full[s1]); }
          if (++c_g == 4) { c_g = 0; c_row0 += kRows; }
          if (l_item < npi) load(mg[d], mk[MASKED ? d : 0], eg[d], ek[MASKED ? d : 0]);
        }
      }
    }
  } else if (warp < kCW) {
    // ================= converters (any F) =================
    // thread <-> (frames warp + 16 j, bin 32 c + lane).  Frames past the CTA's range are skipped altogether (their
    // A rows stay uninitialised: a row of A only feeds the same row of D, which is never stored).
    const int rr = warp & 7;
    const uint32_t off0 = (uint32_t)((warp >> 3) * 1024 + rr * 128 + (((lane >> 2) ^ rr) << 4) + (lane & 3) * 4);
    float mg[DEPTH][8], mk[MASKED ? DEPTH : 1][8];
    // state of the load stream (runs DEPTH items ahead of the convert stream)
    int l_row0 = row_begin, l_c = 0, l_item = 0;
    auto load = [&](float (&g)[8], float (&k)[8]) {
      const int nj = max(0, (min(kRows, row_end - l_row0) - warp + 15) >> 4);
      const int kcol = l_c * kKC + lane;
      const size_t base = (size_t)(l_row0 + warp) * F + kcol;
      const float *pg = p.mag + base;
      const float *pk = MASKED ? p.mask + base : nullptr;
      const bool kin = kcol < Fmma;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const bool ok = kin && j < nj;
        g[j] = ok ? ld_stream1(pg + j * 16 * F) : 0.0f;
        if (MASKED) k[j] = ok ? ld_stream1(pk + j * 16 * F) : 0.0f;
      }
      ++l_item;
      if (++l_c == p.nchunks) { l_c = 0; l_row0 += kRows; }
    };
#pragma unroll
    for (int d = 0; d < DEPTH; ++d)
      if (d < nitems) load(mg[d], mk[MASKED ? d : 0]);

    int c_row0 = row_begin, c_c = 0, nj_c = 0;
    uint32_t vmask = 0xffu;
    int st = 0;
    uint32_t ph = 0;
    for (int q0 = 0; q0 < nitems; q0 += DEPTH) {
#pragma unroll
      for (int d = 0; d < DEPTH; ++d) {
        const int q = q0 + d;
        if (q < nitems) {
          if (c_c == 0) {   // new tile: rows of this warp inside it, and which of them are inside their utterance
            nj_c = max(0, (min(kRows, row_end - c_row0) - warp + 15) >> 4);
            if (MASKED && p.lens) {
              int row = c_row0 + warp;
              int b = row / p.T, t = row - b * p.T;
              int len = __ldg(p.lens + min(b, p.N / p.T - 1));
              vmask = 0;
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                vmask |= (t < len ? 1u : 0u) << j;
                t += 16;
                while (t >= p.T) { t -= p.T; ++b; len = __ldg(p.lens + min(b, p.N / p.T - 1)); }
              }
            }
          }
          if (q >= NS) mbar_wait(&empty[st], ph ^ 1u);
          unsigned char *sa = stage0 + (size_t)st * 2 * kATile + off0;
          const int kcol = c_c * kKC + lane;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            if (j >= nj_c) break;   // warp-uniform: rows past the CTA's range (partial last tile) cost nothing
            float x = mg[d][j];
            if (MASKED) {
              const float sg = p.mask_is_logit ? sigmoid_fast(mk[MASKED ? d : 0][j]) : mk[MASKED ? d : 0][j];
              x = (vmask >> j) & 1u ? sg * x : 0.0f;
              if (p.enh && kcol < Fmma && j < nj_c) p.enh[(size_t)(c_row0 + warp + 16 * j) * F + kcol] = x;
            }
            const float x2 = x * x;
            *reinterpret_cast<float *>(sa + j * 2048) = x2;
            *reinterpret_cast<float *>(sa + kATile + j * 2048) = tf32_trunc_lo(x2);
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) mbar_arrive(&full[st]);
          if (++st == NS) { st = 0; ph ^= 1u; }
          if (++c_c == p.nchunks) { c_c = 0; c_row0 += kRows; }
          if (l_item < nitems) load(mg[d], mk[MASKED ? d : 0]);
        }
      }
    }
  } else if (warp == kCW + kEW) {
    // ================= MMA issuer =================
    if (lane == 0) {
      const uint32_t idesc_cat = umma_idesc_tf32(kRows, 2 * p.MB, false, false);   // A_hi x [B_hi | B_lo]
      const uint32_t idesc_hi = umma_idesc_tf32(kRows, NB, false, false);          // A_lo x B_hi (rows >= MB: unused columns)
      int st = 0;
      uint32_t ph = 0;
      for (int t = 0; t < ntiles; ++t) {
        const int buf = t & 1;
        if (t >= 2) mbar_wait(&tempty[buf], (uint32_t)(((t >> 1) - 1) & 1));
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(buf * WD);
        for (int c = 0; c < p.nchunks; ++c) {
          mbar_wait(&full[st], ph);
          tc_fence_after();
          const uint32_t a_hi = smem_u32(stage0 + (size_t)st * 2 * kATile);
          const uint32_t a_lo = a_hi + kATile;
          const uint32_t b_cat = smem_u32(fc_hi + (size_t)c * fc_chunk);
          const int ks = c == p.nchunks - 1 ? p.ksteps_last : 4;
          for (int k = 0; k < ks; ++k) {
            const uint64_t dah = umma_desc(a_hi + k * 32, 16, 1024, 2), dal = umma_desc(a_lo + k * 32, 16, 1024, 2);
            const uint64_t db = umma_desc(b_cat + k * 32, 16, 1024, 2);
            umma_tf32(d_tmem, dah, db, idesc_cat, (c | k) ? 1u : 0u);
            umma_tf32(d_tmem + (uint32_t)(2 * p.MB), dal, db, idesc_hi, (c | k) ? 1u : 0u);
          }
          umma_commit(&empty[st]);   // the stage is free once these MMAs have read it
          if (++st == NS) { st = 0; ph ^= 1u; }
        }
        umma_commit(&tfull[buf]);    // accumulator of tile t complete
      }
    }
  } else {
    // ================= epilogue: TMEM lane <-> frame =================
    const int e = warp - kCW;        // == warp % 4: the TMEM lane quarter this warp may access
    for (int t = 0; t < ntiles; ++t) {
      const int buf = t & 1;
      const int row = row_begin + t * kRows + 32 * e + lane;
      const bool rok = row < row_end;
      // trailing bins of this frame (issued before the accumulator wait: their latency hides behind the MMAs)
      float xt2[4] = {0.f, 0.f, 0.f, 0.f};
      if (rok && p.ntail > 0) {
        bool valid = true;
        if (MASKED && p.lens) {
          const int b = row / p.T;
          valid = (row - b * p.T) < __ldg(p.lens + b);
        }
#pragma unroll
        for (int kt = 0; kt < 4; ++kt)
          if (kt < p.ntail) {
            float x = ld_stream1(p.mag + (size_t)row * F + Fmma + kt);
            if (MASKED) {
              const float mv = ld_stream1(p.mask + (size_t)row * F + Fmma + kt);
              const float sg = p.mask_is_logit ? sigmoid_fast(mv) : mv;
              x = valid ? sg * x : 0.0f;
              if (p.enh) p.enh[(size_t)row * F + Fmma + kt] = x;
            }
            xt2[kt] = x * x;
          }
      }
      mbar_wait(&tfull[buf], (uint32_t)((t >> 1) & 1));
      tc_fence_after();
      for (int c16 = 0; c16 < NB; c16 += 16) {
        if (c16 >= M) continue;
        float v[16];
        {
          float v1[16], v2[16];
          const uint32_t tb = tmem_base + ((uint32_t)(32 * e) << 16) + (uint32_t)(buf * WD + c16);
          tmem_ld16(tb, v);                                  // x2_hi . fc_hi
          tmem_ld16(tb + (uint32_t)p.MB, v1);                // x2_hi . fc_lo
          tmem_ld16(tb + (uint32_t)(2 * p.MB), v2);          // x2_lo . fc_hi
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] += v1[i] + v2[i];
        }
#pragma unroll
        for (int kt = 0; kt < 4; ++kt)
          if (kt < p.ntail) {
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = fmaf(xt2[kt], fct_s[kt * NB + c16 + i], v[i]);
          }
        float y[16], gg[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const float P = v[i];
          const bool clamped = P <= kClampTc;
          const float c1 = c1_s[c16 + i];
          y[i] = (__logf(clamped ? kClampTc : P) + c0_s[c16 + i]) * c1;   // lg2.approx path: <= 3 ulp, far inside 1e-4
          gg[i] = clamped ? 0.0f : __fdividef(c1, P);
        }
        if (rok) {
          float *yo = p.Y + (size_t)row * M + c16;
          float *go = p.G ? p.G + (size_t)row * M + c16 : nullptr;
          if ((M & 3) == 0) {
#pragma unroll
            for (int i = 0; i < 16; i += 4)
              if (c16 + i < M) {
                *reinterpret_cast<float4 *>(yo + i) = make_float4(y[i], y[i + 1], y[i + 2], y[i + 3]);
                if (go) *reinterpret_cast<float4 *>(go + i) = make_float4(gg[i], gg[i + 1], gg[i + 2], gg[i + 3]);
              }
          } else {
#pragma unroll
            for (int i = 0; i < 16; ++i)
              if (c16 + i < M) {
                yo[i] = y[i];
                if (go) go[i] = gg[i];
              }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[buf]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kCW + kEW) {
    tc_fence_after();
    tmem_dealloc(tmem_base, tmem_cols);
  }
}

// ------------------------------------------------------------------------------------------------
// backward:  dP = dY * G ;  d(x^2)^T = fc . dP^T  (bins on the MMA M side, frames on the N side) ;
//            d_in[n,k] = d(x^2)[n,k] * 2 x * dx/d_in
//
//   warps 0..15 : epilogue -- TMEM lane <-> BIN, column <-> frame: for a fixed frame the 32 lanes of a warp touch 32
//                 consecutive bins, so mask / mag loads and d_in stores are coalesced 128 B segments straight from the
//                 accumulator layout (no shared-memory transpose).  Warp e: lane quarter e%4, M tile (e/4)%2, frame
//                 half e/8 of the 128-frame tile.
//   warps 16..19: converters -- thread <-> frame: dP = dY*G (128-bit loads), hi/lo split into the K-major B tile,
//                 frame validity, and the trailing bins (k >= 256) as plain FMAs
//   warp 20     : MMA issue: A = fc (resident, hi/lo), 2 M tiles x ceil(M/8) k-steps x 3 MMAs of 128x128x8 per tile
// TMEM: 2 accumulator buffers x 2 M tiles x 128 columns = all 512 columns.
// ------------------------------------------------------------------------------------------------
constexpr int kBwdEpiWarps = 16;
constexpr int kBwdCvtWarps = 4;
constexpr int kBwdThreads = (kBwdEpiWarps + kBwdCvtWarps + 1) * 32;

struct FbTcBwdParams {
  const float *dY, *G, *mask, *mag, *fc;
  const int32_t *lens;
  float *d_in;
  int mask_is_logit, N, T, F, M;
  int nmt;           // M tiles of 128 bins on the tensor core (1 or 2)
  int Fmma;          // bins [0, Fmma) on the tensor core, [Fmma, F) as plain FMAs (<= 4)
  int nkc;           // 32-wide k chunks over the mel axis (1 or 2)
  int ksteps_last;   // 8-wide MMA steps in the last chunk
  int rows_per_cta;
};

template <bool MASKED>
__global__ void __launch_bounds__(kBwdThreads, 1) fbank_tc_bwd_kernel(const FbTcBwdParams p) {
  extern __shared__ __align__(1024) unsigned char smraw_[];
  unsigned char *sm = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(smraw_) + 1023) & ~(uintptr_t)1023);
  const int F = p.F, M = p.M, nmt = p.nmt, nkc = p.nkc, ntail = F - p.Fmma;
  const int a_chunk = nmt * 128 * 128;                    // bytes of one k-chunk of A (nmt x 128 bins x 128 B)
  unsigned char *a_hi = sm;
  unsigned char *a_lo = sm + (size_t)nkc * a_chunk;
  unsigned char *b_hi = sm + (size_t)2 * nkc * a_chunk;   // [nkc][128 frames][128 B]
  unsigned char *b_lo = b_hi + (size_t)nkc * kATile;
  uint64_t *bfull = reinterpret_cast<uint64_t *>(b_lo + (size_t)nkc * kATile);   // [2]
  uint64_t *bempty = bfull + 2;                                                   // [1]
  uint64_t *tfull = bempty + 1;                                                   // [2]
  uint64_t *tempty = tfull + 2;                                                   // [2]
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tempty + 2);
  float *fct_s = reinterpret_cast<float *>(tmem_slot + 2);   // [4][64] filter-bank rows of the trailing bins
  float *dtail_s = fct_s + 4 * 64;                           // [2][4][128] d(x^2) of the trailing bins
  int *vrow_s = reinterpret_cast<int *>(dtail_s + 2 * 4 * 128);   // [2][128] frame inside its utterance?

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int row_begin = min(p.N, (int)blockIdx.x * p.rows_per_cta);
  const int row_end = min(p.N, row_begin + p.rows_per_cta);
  const int ntiles = (row_end - row_begin + kRows - 1) / kRows;

  if (tid == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(&bfull[i], kBwdCvtWarps);
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], kBwdEpiWarps);
    }
    mbar_init(bempty, 1);
    mbar_fence_init();
  }
  if (warp == kBwdEpiWarps + kBwdCvtWarps) tmem_alloc(tmem_slot, 512);
  {
    float4 *z = reinterpret_cast<float4 *>(a_hi);
    for (int i = tid; i < 2 * nkc * a_chunk / 16; i += kBwdThreads) z[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int i = tid; i < 4 * 64; i += kBwdThreads) {
      const int kt = i >> 6, m = i & 63;
      fct_s[i] = (kt < ntail && m < M) ? __ldg(p.fc + (size_t)(p.Fmma + kt) * M + m) : 0.0f;
    }
  }
  __syncthreads();
  // A = fc[bin][mel], K-major (mel contiguous), 128B swizzle: chunk c, row k at c*a_chunk + (k>>3)*1024 + (k&7)*128
  for (int i = tid; i < p.Fmma * M; i += kBwdThreads) {
    const int k = i / M, m = i - k * M;
    const float v = __ldg(p.fc + i);
    const int ch = m >> 5, mm = m & 31;
    const int off = ch * a_chunk + (k >> 3) * 1024 + (k & 7) * 128 + ((((mm >> 2) ^ (k & 7))) << 4) + (mm & 3) * 4;
    *reinterpret_cast<float *>(a_hi + off) = v;
    *reinterpret_cast<float *>(a_lo + off) = tf32_trunc_lo(v);
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < kBwdEpiWarps) {
    // ================= epilogue =================
    const int q = warp & 3, mt = (warp >> 2) & 1, h = warp >> 3;
    const int k = 128 * mt + 32 * q + lane;               // this lane's bin
    const bool kok = mt < nmt && k < p.Fmma;
    for (int t = 0; t < ntiles; ++t) {
      const int buf = t & 1;
      const uint32_t par = (uint32_t)((t >> 1) & 1);
      const int row0 = row_begin + t * kRows;
      mbar_wait(&bfull[buf], par);      // frame validity / trailing bins of this tile are published
      mbar_wait(&tfull[buf], par);
      tc_fence_after();
      if (mt < nmt) {
        for (int cb = 0; cb < 64; cb += 16) {
          const int r0 = 64 * h + cb;                     // first frame (tile-relative) of this batch of 16
          if (row0 + r0 >= row_end) break;
          float v[16];
          tmem_ld16(tmem_base + ((uint32_t)(32 * q) << 16) + (uint32_t)(buf * 256 + mt * 128 + r0), v);
          const size_t gbase = (size_t)(row0 + r0) * F + k;
          float mg[16], mk[MASKED ? 16 : 1];
          uint32_t vm = 0;
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            const bool inr = row0 + r0 + i < row_end;
            const bool val = inr && (!MASKED || vrow_s[buf * 128 + r0 + i] != 0);
            vm |= (val ? 1u : 0u) << i;
            const bool ld = kok && val;
            mg[i] = ld ? ld_stream1(p.mag + gbase + (size_t)i * F) : 0.0f;
            if (MASKED) mk[i] = ld ? ld_stream1(p.mask + gbase + (size_t)i * F) : 0.0f;
          }
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            float fac;
            if (MASKED) {
              if (p.mask_is_logit) {
                const float sg = sigmoid_fast(mk[i]);
                fac = 2.0f * sg * mg[i] * mg[i] * sg * (1.0f - sg);   // 2 x * mag * s(1-s),  x = s*mag
              } else {
                fac = 2.0f * mk[i] * mg[i] * mg[i];                   // 2 x * mag,  x = mask*mag
              }
              if (!((vm >> i) & 1u)) fac = 0.0f;
            } else {
              fac = 2.0f * mg[i];
            }
            if (kok && row0 + r0 + i < row_end) p.d_in[gbase + (size_t)i * F] = v[i] * fac;
          }
        }
      }
      // trailing bins (k >= Fmma): thread <-> frame, a few strided accesses
      if (ntail > 0 && q == 0 && mt == 0) {
#pragma unroll
        for (int rr = 0; rr < 64; rr += 32) {
          const int r = 64 * h + rr + lane, row = row0 + r;
          if (row < row_end) {
            const bool val = !MASKED || vrow_s[buf * 128 + r] != 0;
            for (int kt = 0; kt < ntail; ++kt) {
              const size_t gi = (size_t)row * F + p.Fmma + kt;
              const float mgv = p.mag[gi];
              float fac;
              if (MASKED) {
                const float mv = p.mask[gi];
                if (p.mask_is_logit) {
                  const float sg = sigmoid_fast(mv);
                  fac = 2.0f * sg * mgv * mgv * sg * (1.0f - sg);
                } else {
                  fac = 2.0f * mv * mgv * mgv;
                }
                if (!val) fac = 0.0f;
              } else {
                fac = 2.0f * mgv;
              }
              p.d_in[gi] = dtail_s[(buf * 4 + kt) * 128 + r] * fac;
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[buf]);
    }
  } else if (warp < kBwdEpiWarps + kBwdCvtWarps) {
    // ================= converters: thread <-> frame =================
    const int r = (warp - kBwdEpiWarps) * 32 + lane;      // tile-relative frame
    const uint32_t roff = (uint32_t)((r >> 3) * 1024 + (r & 7) * 128);
    for (int t = 0; t < ntiles; ++t) {
      const int buf = t & 1;
      const int row = row_begin + t * kRows + r;
      const bool inr = row < row_end;
      if (t >= 1) mbar_wait(bempty, (uint32_t)((t - 1) & 1));            // MMAs of tile t-1 have read the B tile
      if (t >= 2) mbar_wait(&tempty[buf], (uint32_t)(((t >> 1) - 1) & 1));   // epilogue of tile t-2 left this buffer
      float tail[4] = {0.f, 0.f, 0.f, 0.f};
      if (inr) {
        const float *py = p.dY + (size_t)row * M, *pg = p.G + (size_t)row * M;
        for (int m0 = 0; m0 < M; m0 += 8) {               // one 8-wide k-step at a time (M % 4 == 0)
          float dp[8];
#pragma unroll
          for (int u = 0; u < 8; u += 4) {
            if (m0 + u < M) {
              const float4 a = ld_stream4(py + m0 + u), g4 = ld_stream4(pg + m0 + u);
              dp[u] = a.x * g4.x; dp[u + 1] = a.y * g4.y; dp[u + 2] = a.z * g4.z; dp[u + 3] = a.w * g4.w;
            } else {
              dp[u] = dp[u + 1] = dp[u + 2] = dp[u + 3] = 0.0f;
            }
          }
          const int ch = m0 >> 5, mm = m0 & 31;
#pragma unroll
          for (int u = 0; u < 8; u += 4) {
            const uint32_t off = (uint32_t)ch * kATile + roff + (uint32_t)((((mm + u) >> 2) ^ (r & 7)) << 4);
            *reinterpret_cast<float4 *>(b_hi + off) = make_float4(dp[u], dp[u + 1], dp[u + 2], dp[u + 3]);
            *reinterpret_cast<float4 *>(b_lo + off) = make_float4(tf32_trunc_lo(dp[u]), tf32_trunc_lo(dp[u + 1]),
                                                                  tf32_trunc_lo(dp[u + 2]), tf32_trunc_lo(dp[u + 3]));
          }
#pragma unroll
          for (int kt = 0; kt < 4; ++kt)
            if (kt < ntail) {
#pragma unroll
              for (int u = 0; u < 8; ++u)
                if (m0 + u < M) tail[kt] = fmaf(dp[u], fct_s[kt * 64 + m0 + u], tail[kt]);
            }
        }
      }
      int valid = inr ? 1 : 0;
      if (MASKED && inr && p.lens) {
        const int b = row / p.T;
        valid = (row - b * p.T) < __ldg(p.lens + b) ? 1 : 0;
      }
      vrow_s[buf * 128 + r] = valid;
#pragma unroll
      for (int kt = 0; kt < 4; ++kt) dtail_s[(buf * 4 + kt) * 128 + r] = tail[kt];
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bfull[buf]);
    }
  } else {
    // ================= MMA issuer =================
    if (lane == 0) {
      const uint32_t idesc = umma_idesc_tf32(128, 128, false, false);
      for (int t = 0; t < ntiles; ++t) {
        const int buf = t & 1;
        mbar_wait(&bfull[buf], (uint32_t)((t >> 1) & 1));
        tc_fence_after();
        for (int mt = 0; mt < nmt; ++mt) {
          const uint32_t d_tmem = tmem_base + (uint32_t)(buf * 256 + mt * 128);
          for (int c = 0; c < nkc; ++c) {
            const uint32_t ah = smem_u32(a_hi + (size_t)c * a_chunk + (size_t)mt * kATile);
            const uint32_t al = smem_u32(a_lo + (size_t)c * a_chunk + (size_t)mt * kATile);
            const uint32_t bh = smem_u32(b_hi + (size_t)c * kATile), bl = smem_u32(b_lo + (size_t)c * kATile);
            const int ks = c == nkc - 1 ? p.ksteps_last : 4;
            for (int kk = 0; kk < ks; ++kk) {
              const uint64_t dah = umma_desc(ah + kk * 32, 16, 1024, 2), dal = umma_desc(al + kk * 32, 16, 1024, 2);
              const uint64_t dbh = umma_desc(bh + kk * 32, 16, 1024, 2), dbl = umma_desc(bl + kk * 32, 16, 1024, 2);
              umma_tf32(d_tmem, dah, dbh, idesc, (c | kk) ? 1u : 0u);
              umma_tf32(d_tmem, dal, dbh, idesc, 1u);
              umma_tf32(d_tmem, dah, dbl, idesc, 1u);
            }
          }
        }
        umma_commit(bempty);         // B tile may be overwritten
        umma_commit(&tfull[buf]);    // accumulators of tile t complete
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kBwdEpiWarps + kBwdCvtWarps) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

inline size_t fwd_smem_bytes(int nchunks, int MB, int NB, int ns) {
  return 1024 + (size_t)2 * nchunks * MB * 128 + (size_t)ns * 2 * kATile + 512 + (size_t)6 * NB * 4;
}

}  // namespace

// Whether fbank_tc_fwd has a configuration for (F, M): two accumulator buffers of [hi.hi | hi.lo | lo.hi] columns fit
// tensor memory and one stage fits shared memory.  Pointer alignment is checked at launch.
bool fbank_tc_fwd_fits(int F, int M) {
  const int NB = (M + 15) / 16 * 16, MB = (M + 7) / 8 * 8;
  const int ntail = (F >= kKC && (F % kKC) >= 1 && (F % kKC) <= 4) ? F % kKC : 0;
  const int nchunks = (F - ntail + kKC - 1) / kKC;
  return 2 * (2 * MB + NB) <= 512 && fwd_smem_bytes(nchunks, MB, NB, 1) <= 226 * 1024;
}

// Returns RE2E_E_UNSUPPORTED when the shape does not fit the tensor-core path (caller falls back to the SIMT kernel).
int fbank_tc_fwd(const float *mask, int mask_is_logit, const float *mag, const float *fc, const float *cmvn,
                 const int32_t *lens, float *Y, float *G, float *enh_out, int B, int T, int F, int M,
                 cudaStream_t st) {
  FbTcParams p;
  p.mask = mask; p.mag = mag; p.fc = fc; p.cmvn = cmvn; p.lens = lens; p.Y = Y; p.G = G; p.enh = enh_out;
  p.mask_is_logit = mask_is_logit; p.N = B * T; p.T = T; p.F = F; p.M = M;
  p.NB = (M + 15) / 16 * 16;
  p.MB = (M + 7) / 8 * 8;
  p.ntail = (F >= kKC && (F % kKC) >= 1 && (F % kKC) <= 4) ? F % kKC : 0;
  p.nchunks = (F - p.ntail + kKC - 1) / kKC;
  p.ksteps_last = (F - p.ntail - (p.nchunks - 1) * kKC + 7) / 8;
  if (!fbank_tc_fwd_fits(F, M)) return RE2E_E_UNSUPPORTED;
  int ns = kMaxStagesTc;
  while (ns > 1 && fwd_smem_bytes(p.nchunks, p.MB, p.NB, ns) > 226 * 1024) --ns;
  p.nstages = ns;
  if (((M & 3) == 0) && !(aligned16(Y) && (!G || aligned16(G)))) return RE2E_E_UNSUPPORTED;
  const int sms = num_sms();
  int grid = (p.N + 63) / 64;
  if (grid > sms) grid = sms;
  p.rows_per_cta = (p.N + grid - 1) / grid;
  const size_t smem = fwd_smem_bytes(p.nchunks, p.MB, p.NB, ns);
  int rc;
#define RE2E_FB_LAUNCH(MASKED, DEPTH, FC, PAIR)                                                                          \
  do {                                                                                                                  \
    if ((rc = ensure_smem(reinterpret_cast<const void *>(fbank_tc_fwd_kernel<MASKED, DEPTH, FC, PAIR>), smem)) != RE2E_OK) \
      return rc;                                                                                                        \
    fbank_tc_fwd_kernel<MASKED, DEPTH, FC, PAIR><<<grid, kTcThreads, smem, st>>>(p);                                     \
  } while (0)
  const bool pair = F == 257 && p.nchunks == 8 && ns >= 4 && (reinterpret_cast<uintptr_t>(mag) & 7u) == 0 &&
                    (!mask || (reinterpret_cast<uintptr_t>(mask) & 7u) == 0);
  if (mask) {
    if (pair) RE2E_FB_LAUNCH(true, 2, 257, true);
    else if (F == 257) RE2E_FB_LAUNCH(true, 2, 257, false);
    else RE2E_FB_LAUNCH(true, 2, 0, false);
  } else {
    if (pair) RE2E_FB_LAUNCH(false, 4, 257, true);
    else if (F == 257) RE2E_FB_LAUNCH(false, 4, 257, false);
    else RE2E_FB_LAUNCH(false, 4, 0, false);
  }
#undef RE2E_FB_LAUNCH
  count_launch();
  return launch_status();
}


// d_in only (dfc of a trainable bank is handled by the SIMT kernel).  RE2E_E_UNSUPPORTED -> caller falls back.
int fbank_tc_bwd(const float *dY, const float *G, const float *mask, int mask_is_logit, const float *mag,
                 const float *fc, const int32_t *lens, float *d_in, int B, int T, int F, int M, cudaStream_t st) {
  if ((M & 3) || M > 64 || F < 8 || !aligned16(dY) || !aligned16(G)) return RE2E_E_UNSUPPORTED;
  FbTcBwdParams p;
  p.dY = dY; p.G = G; p.mask = mask; p.mag = mag; p.fc = fc; p.lens = lens; p.d_in = d_in;
  p.mask_is_logit = mask_is_logit; p.N = B * T; p.T = T; p.F = F; p.M = M;
  const int ntail = (F % 128 >= 1 && F % 128 <= 4 && F > 128) ? F % 128 : 0;
  p.Fmma = F - ntail;
  p.nmt = (p.Fmma + 127) / 128;
  if (p.nmt > 2) return RE2E_E_UNSUPPORTED;
  p.nkc = (M + 31) / 32;
  p.ksteps_last = (M - (p.nkc - 1) * 32 + 7) / 8;
  const size_t smem = 1024 + (size_t)2 * p.nkc * p.nmt * 128 * 128 + (size_t)2 * p.nkc * kATile + 256 +
                      sizeof(float) * (4 * 64 + 2 * 4 * 128) + sizeof(int) * 2 * 128;
  if (smem > 226 * 1024) return RE2E_E_UNSUPPORTED;
  const int sms = num_sms();
  int grid = (p.N + 63) / 64;
  if (grid > sms) grid = sms;
  p.rows_per_cta = (p.N + grid - 1) / grid;
  int rc;
  if (mask) {
    if ((rc = ensure_smem(reinterpret_cast<const void *>(fbank_tc_bwd_kernel<true>), smem)) != RE2E_OK) return rc;
    fbank_tc_bwd_kernel<true><<<grid, kBwdThreads, smem, st>>>(p);
  } else {
    if ((rc = ensure_smem(reinterpret_cast<const void *>(fbank_tc_bwd_kernel<false>), smem)) != RE2E_OK) return rc;
    fbank_tc_bwd_kernel<false><<<grid, kBwdThreads, smem, st>>>(p);
  }
  count_launch();
  return launch_status();
}

}  // namespace re2e
