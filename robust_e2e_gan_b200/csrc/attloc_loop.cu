// The attention decoder loop (model/e2e_decoder.py:114-122: `att_c, att_w = self.att(hpad, hlen, z, att_w)` for
// every output position, the alignment fed back) as ONE persistent thread-block-cluster kernel per direction,
// for sm_100a.  Arithmetic per step = AttLoc.forward (model/e2e_attention.py:258-299) and its backward.
//
// Why: as separate launches the loop is a chain of 2 x #steps latency-bound cluster kernels, each paying a
// prologue (re-load of the utterance's `pre` / `enc_h` rows, the conv / attention weights) and a grid drain.  Here a
// cluster of CL CTAs owns one utterance for the WHOLE loop:
//   * the CTA's rows of pre[b] and enc_h[b] are fetched once (two 1-D bulk copies in the forward; in the backward they
//     live in TENSOR MEMORY -- 256 KB per SM, idle otherwise -- as warp-private columns written with tcgen05.st and
//     read back with tcgen05.ld, which frees shared memory for the d pre tile);
//   * W_att stays in registers, W_conv in shared memory, for all steps;
//   * the alignment never leaves the cluster: every CTA pushes the scaled energies of its frames to all peers
//     (st.async + mbarrier complete_tx over DSMEM) and each CTA normalises the whole row itself -- the softmax needs
//     ONE exchange per step, which also carries the (max, sum) pair and the partial context;
//   * the decoder-state projection W_dec z_i is an INPUT (dec_proj, all steps at once from one tensor-core GEMM) --
//     see re2e_attloc_loop_fwd in the header for when the caller can provide it;
//   * the backward recomputes tanh(.) from the resident `pre` rows and the saved conv features (10 floats per frame)
//     instead of saving and re-reading #steps x (B,Th,A) activations; parameter gradients accumulate in REGISTERS
//     across all steps and are written once; d dec_proj of every step goes out as one (S,B,A) tensor, so d dec_z and
//     dW_dec are two dense GEMMs after the loop; the chain gradient d att_prev stays in shared memory.
// Receive buffers and their mbarriers are double-buffered by step parity: a CTA can only run ahead of a peer by
// less than one step (it needs the peer's push of step s to finish step s), so data of step s+2 never lands before
// the peer has consumed step s.
#include <math_constants.h>

#include "attloc_common.cuh"
#include "tc_common.cuh"

namespace re2e {
namespace {

__device__ __forceinline__ void cp_async4(void *dst_smem, const void *src_gmem) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(dst_smem)), "l"(src_gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// Sum 10 per-lane values across the warp in 12 shuffles (recursive halving on an uneven tree).  On return lane L holds
// in v[0] the total of value index  5*bit4 + (bit1 ? 2 : (bit2 ? (bit3 ? 4 : 1) : (bit3 ? 3 : 0)))  of L; the lanes with
// bit1 set hold index 5*bit4 + 2 four times over (any bit3, bit2).
__device__ __forceinline__ void warp_reduce10(float (&v)[10], int lane) {
  {
    const bool up = lane & 16;
#pragma unroll
    for (int i = 0; i < 5; ++i) {
      const float send = up ? v[i] : v[i + 5], keep = up ? v[i + 5] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
    }
  }
  {
    const bool up = lane & 8;
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const float send = up ? v[i] : v[i + 3], keep = up ? v[i + 3] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
    }
    v[2] += __shfl_xor_sync(0xffffffffu, v[2], 8);
  }
  {
    const bool up = lane & 4;
    const float send = up ? v[0] : v[1], keep = up ? v[1] : v[0];
    v[0] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
    v[2] += __shfl_xor_sync(0xffffffffu, v[2], 4);
  }
  {
    const bool up = lane & 2;
    const float send = up ? v[0] : v[2], keep = up ? v[2] : v[0];
    v[0] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
  }
  v[0] += __shfl_xor_sync(0xffffffffu, v[0], 1);
}

constexpr int kLP = 8;            // warp pairs = frames per chunk
constexpr int kLW = 2 * kLP;      // warps
constexpr int kLT = kLW * 32;     // threads
constexpr int kLMaxCL = 8;
constexpr int kKG = 12;           // dW_conv taps per thread

struct LoopGeom {
  int tloc_max, App, CKp, Thp, Dp;
  int col_enc, ncols;             // backward: first TMEM column of the enc_h region, total columns used
};

struct LoopFwdParams {
  const float *pre, *enc, *dec_proj, *att_init, *W_att, *W_conv, *gvec, *gvec_b;
  float scaling;
  float *c_all, *w_all, *conv_all;
  int S, B, Th, D, A, C, K;
  LoopGeom g;
};

struct LoopBwdParams {
  const float *pre, *enc, *dec_proj, *att_init, *w_all, *conv_all, *dc_all, *dw_all, *W_att, *W_conv, *gvec;
  float scaling;
  float *d_pre, *d_decproj, *acc_slots;
  int slot_stride;
  int S, B, Th, D, A, C, K;
  LoopGeom g;
};

// ------------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------------
template <int APL, int CP, int DPL>
__global__ void __launch_bounds__(kLT, 1) attloc_loop_fwd_kernel(const LoopFwdParams p) {
  constexpr int NT = kLT;
  constexpr int WP = CP + 1;             // odd pitch of the staged W_att rows: conflict-free lane <-> a reads
  constexpr int CPP = (CP + 3) & ~3;     // pitch of conv rows in shared memory (128-bit broadcast reads)
  extern __shared__ __align__(128) unsigned char smraw[];
  const LoopGeom g = p.g;
  const int C = CP == 10 ? 10 : p.C;
  const int Th = p.Th, D = p.D, A = p.A, K = p.K, S = p.S, B = p.B, filts = (p.K - 1) / 2;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, half = warp & 1, pair = warp >> 1;
  const int CL = (int)cluster_nctarank(), rank = (int)cluster_ctarank();
  const int b = blockIdx.x / CL;
  const int t0 = min(Th, rank * g.tloc_max), t1 = min(Th, t0 + g.tloc_max), tloc = t1 - t0;
  const int nch = (tloc + kLP - 1) / kLP;
  const int Dp = g.Dp, Dh = (D + 1) / 2;

  uint64_t *full = reinterpret_cast<uint64_t *>(smraw);      // the resident (pre | enc) tile has landed
  uint64_t *xbar = full + 1;                                  // [2] per-step exchange, by step parity
  uint64_t *tbar = xbar + 2;                                  // partial contexts of the last step (rank 0)
  float *tile = reinterpret_cast<float *>(smraw + 128);       // tloc_max*A pre rows, then tloc_max*D enc rows
  float *app = tile + (size_t)g.tloc_max * (A + D);           // App   zero padded alignment row, a[i] at filts+i
  float *wc_s = app + g.App;                                  // CKp
  float *watt_s = wc_s + g.CKp;                               // A*WP  (prologue only)
  float *convp = watt_s + A * WP;                             // round4(kKQ*tloc_max*CP)  conv partials
  float *conv_s = convp + round4(kKQ * g.tloc_max * CP);      // tloc_max*CPP
  float *e_all = conv_s + g.tloc_max * CPP;                   // 2*Thp  scaled energies of ALL frames, by parity
  float *epart = e_all + 2 * g.Thp;                           // round4(2*tloc_max)  per-half partial energies of my frames
  float *cred = epart + round4(2 * g.tloc_max);               // kLP*Dp        per-pair partial contexts
  float *cbuf = cred + kLP * Dp;                              // 2*kLMaxCL*Dp  partial contexts of every rank (used on rank 0)

  const uint32_t xbytes = (uint32_t)Th * 4u + (rank == 0 ? (uint32_t)CL * (uint32_t)D * 4u : 0u);
  if (tid == 0) {
    mbar_init(full, 1);
    mbar_init(&xbar[0], 1);
    mbar_init(&xbar[1], 1);
    mbar_init(tbar, 1);
    mbar_fence_init();
    mbar_expect_tx(&xbar[0], xbytes);
    mbar_expect_tx(&xbar[1], xbytes);
    if (rank == 0) mbar_expect_tx(tbar, (uint32_t)CL * (uint32_t)D * 4u);
  }
  cluster_arrive_relaxed();   // "this CTA is running and its barriers exist"
  // parameters (final before any predecessor kernel started)
  float gv[APL];
#pragma unroll
  for (int j = 0; j < APL; ++j) gv[j] = __ldg(p.gvec + half * (A / 2) + lane + 32 * j);
  const float gb = __ldg(p.gvec_b);
  for (int i = tid; i < C * K; i += NT) wc_s[i] = __ldg(p.W_conv + i);
  for (int i = tid; i < A * C; i += NT) { const int a = i / C; watt_s[a * WP + (i - a * C)] = __ldg(p.W_att + i); }
  // the encoder projection / dec_proj / initial alignment are produced by kernels earlier in the stream
  pdl_wait();
  if (tid == 0 && tloc > 0) {
    mbar_expect_tx(full, (uint32_t)tloc * (uint32_t)(A + D) * 4u);
    bulk_g2s(tile, p.pre + ((size_t)b * Th + t0) * A, (uint32_t)tloc * A * 4u, full);
    bulk_g2s(tile + (size_t)g.tloc_max * A, p.enc + ((size_t)b * Th + t0) * D, (uint32_t)tloc * D * 4u, full);
  }
  for (int i = tid; i < g.App; i += NT) {
    const int t = i - filts;
    app[i] = (t >= 0 && t < Th) ? __ldg(p.att_init + (size_t)b * Th + t) : 0.0f;
  }
  __syncthreads();
  // W_att rows of this lane's channels -> registers, two channels per 64-bit register pair (packed FFMA2)
  constexpr int APH = (APL + 1) / 2;
  float2 WattP[APH][CP];
#pragma unroll
  for (int jp = 0; jp < APH; ++jp) {
    const int a0 = half * (A / 2) + lane + 32 * (2 * jp), a1 = a0 + 32;
#pragma unroll
    for (int c = 0; c < CP; ++c)
      WattP[jp][c] = make_float2(c < C ? watt_s[a0 * WP + c] : 0.0f, (c < C && 2 * jp + 1 < APL) ? watt_s[a1 * WP + c] : 0.0f);
  }
  uint32_t dmask = 0;                        // which of this lane's DPL encoder channels exist
#pragma unroll
  for (int j = 0; j < DPL; ++j)
    if (lane + 32 * j < Dh && half * Dh + lane + 32 * j < D) dmask |= 1u << j;
  const int aoff = half * (A / 2) + lane;
  cluster_wait();                            // every peer CTA is resident, its mbarriers initialised
  if (tloc > 0) mbar_wait(full, 0);

  for (int s = 0; s < S; ++s) {
    const uint32_t par = (uint32_t)s & 1u, ph = ((uint32_t)s >> 1) & 1u;
    float *e_cur = e_all + par * g.Thp;
    float *cb = cbuf + par * kLMaxCL * Dp;
    // decoder-state projection of this step (consumed after the convolution: its L2 latency is hidden)
    float dp[APL];
#pragma unroll
    for (int j = 0; j < APL; ++j) dp[j] = __ldg(p.dec_proj + ((size_t)s * B + b) * A + aoff + 32 * j);

    // ---- location convolution: conv[t,c] = sum_k Wc[c,k] * a[t + k - filts]; item = (k part, channel, 5 frames)
    {
      const int ntg = (tloc + kTG - 1) / kTG;
      const int Kq = (K + kKQ - 1) / kKQ;
      const int nitems = ntg * C * kKQ;
      for (int item = tid; item < nitems; item += NT) {
        const int tg = item % ntg, rest = item / ntg, c = rest % C, kq = rest / C;
        const int k0 = kq * Kq, k1 = min(K, k0 + Kq);
        const float *wr = wc_s + c * K;
        const float *ar = app + t0 + kTG * tg;  // element (t, k) = ar[(t - 5tg) + k]
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f, a4 = 0.f;
        float x0 = ar[k0], x1 = ar[k0 + 1], x2 = ar[k0 + 2], x3 = ar[k0 + 3];
#pragma unroll 5
        for (int k = k0; k < k1; ++k) {
          const float x4 = ar[k + 4], wv2 = wr[k];
          a0 = fmaf(wv2, x0, a0); a1 = fmaf(wv2, x1, a1); a2 = fmaf(wv2, x2, a2);
          a3 = fmaf(wv2, x3, a3); a4 = fmaf(wv2, x4, a4);
          x0 = x1; x1 = x2; x2 = x3; x3 = x4;
        }
        float *o = convp + ((size_t)kq * g.tloc_max + kTG * tg) * CP + c;
        const int nv = min(kTG, tloc - kTG * tg);
        o[0] = a0;
        if (nv > 1) o[CP] = a1;
        if (nv > 2) o[2 * CP] = a2;
        if (nv > 3) o[3 * CP] = a3;
        if (nv > 4) o[4 * CP] = a4;
      }
    }
    __syncthreads();  // #1
    for (int i = tid; i < tloc * CPP; i += NT) {
      const int tl = i / CPP, c = i - tl * CPP;
      float v = 0.0f;
      if (c < C) {
#pragma unroll
        for (int kq = 0; kq < kKQ; ++kq) v += convp[((size_t)kq * g.tloc_max + tl) * CP + c];
        if (p.conv_all) p.conv_all[(((size_t)s * B + b) * Th + t0 + tl) * C + c] = v;
      }
      conv_s[i] = v;
    }
    __syncthreads();  // #2: conv_s visible

    // ---- energies of step s and, in the same sweep over the resident frames, the context of step s-1 from the
    //      normalised alignment that is still in `app` (the context does not feed the recurrence: it is taken off
    //      the critical path, and no online-softmax bookkeeping is needed).  pair <-> frame, lane <-> channel
    float acc[DPL];
#pragma unroll
    for (int j = 0; j < DPL; ++j) acc[j] = 0.0f;
#pragma unroll 2
    for (int q = 0; q < nch; ++q) {
      const int tl = kLP * q + pair;
      if (tl < tloc) {
        const float *cvp = conv_s + tl * CPP;
        float cv[CPP];
#pragma unroll
        for (int c4 = 0; c4 < CPP; c4 += 4) {
          const float4 t4 = *reinterpret_cast<const float4 *>(cvp + c4);
          cv[c4] = t4.x; cv[c4 + 1] = t4.y; cv[c4 + 2] = t4.z; cv[c4 + 3] = t4.w;
        }
        const float *row = tile + (size_t)tl * A + aoff;
        const float pw = app[filts + t0 + tl];           // alignment of step s-1 (initial alignment at s = 0: unused)
        const float *er = tile + (size_t)g.tloc_max * A + (size_t)tl * D + half * Dh + lane;
        float part = 0.0f;
#pragma unroll
        for (int jp = 0; jp < APH; ++jp) {
          const bool two = 2 * jp + 1 < APL;
          float2 u = make_float2(dp[2 * jp] + row[64 * jp], two ? dp[2 * jp + 1] + row[64 * jp + 32] : 0.0f);
#pragma unroll
          for (int c = 0; c < CP; ++c) u = __ffma2_rn(WattP[jp][c], make_float2(cv[c], cv[c]), u);
          part = fmaf(gv[2 * jp], tanh_ex2(u.x), part);
          if (two) part = fmaf(gv[2 * jp + 1], tanh_ex2(u.y), part);
        }
#pragma unroll
        for (int j = 0; j < DPL; ++j)
          if (dmask & (1u << j)) acc[j] = fmaf(pw, er[32 * j], acc[j]);
        part = warp_sum(part);
        if (lane == 0) epart[2 * tl + half] = part;
      }
    }
#pragma unroll
    for (int j = 0; j < DPL; ++j)
      if (dmask & (1u << j)) cred[pair * Dp + half * Dh + lane + 32 * j] = acc[j];
    __syncthreads();  // #3: partial energies and per-pair partial contexts published

    // ---- ONE push per step: context partial of step s-1 -> rank 0, my frames' scaled energies -> every CTA
    for (int d = tid; d < D; d += NT) {
      float sum = 0.0f;
#pragma unroll
      for (int pr = 0; pr < kLP; ++pr) sum += cred[pr * Dp + d];
      st_async_f32(dsmem_addr(cb + rank * Dp + d, 0u), s > 0 ? sum : 0.0f, dsmem_addr(&xbar[par], 0u));
    }
    for (int i = tid; i < tloc * CL; i += NT) {
      const int r = i / tloc, tl = i - r * tloc;
      const float e = p.scaling * ((epart[2 * tl] + epart[2 * tl + 1]) + gb);
      st_async_f32(dsmem_addr(e_cur + t0 + tl, (uint32_t)r), e, dsmem_addr(&xbar[par], (uint32_t)r));
    }
    mbar_wait(&xbar[par], ph);   // the scaled energies of ALL frames (on rank 0 also the partial contexts) are here
    // softmax statistics of the whole row, redundantly per warp (same order everywhere: bit-identical), no barrier
    float M = -CUDART_INF_F;
    for (int t = lane; t < Th; t += 32) M = fmaxf(M, e_cur[t]);
    M = warp_max(M);
    float Ssum = 0.0f;
    for (int t = lane; t < Th; t += 32) Ssum += __expf(e_cur[t] - M);
    Ssum = warp_sum(Ssum);
    const float inv = 1.0f / Ssum;
    // the normalised alignment of ALL frames: next step's convolution input; this CTA's frames go to HBM
    for (int t = tid; t < Th; t += NT) {
      const float w = __expf(e_cur[t] - M) * inv;
      app[filts + t] = w;
      if (t >= t0 && t < t1) p.w_all[((size_t)s * B + b) * Th + t] = w;
    }
    if (rank == 0 && s > 0) {
      for (int d = tid; d < D; d += NT) {
        float sum = 0.0f;
        for (int r = 0; r < CL; ++r) sum += cb[r * Dp + d];
        p.c_all[((size_t)(s - 1) * B + b) * D + d] = sum;
      }
    }
    if (tid == 0) mbar_expect_tx(&xbar[par], xbytes);   // re-arm this parity's barrier for step s+2
    __syncthreads();  // #5: alignment row complete; receive buffers of this parity consumed
  }
  // ---- tail: the context of the last step
  {
    float acc[DPL];
#pragma unroll
    for (int j = 0; j < DPL; ++j) acc[j] = 0.0f;
    for (int q = 0; q < nch; ++q) {
      const int tl = kLP * q + pair;
      if (tl < tloc) {
        const float pw = app[filts + t0 + tl];
        const float *er = tile + (size_t)g.tloc_max * A + (size_t)tl * D + half * Dh + lane;
#pragma unroll
        for (int j = 0; j < DPL; ++j)
          if (dmask & (1u << j)) acc[j] = fmaf(pw, er[32 * j], acc[j]);
      }
    }
#pragma unroll
    for (int j = 0; j < DPL; ++j)
      if (dmask & (1u << j)) cred[pair * Dp + half * Dh + lane + 32 * j] = acc[j];
    __syncthreads();
    float *cb = cbuf + ((uint32_t)S & 1u) * kLMaxCL * Dp;
    for (int d = tid; d < D; d += NT) {
      float sum = 0.0f;
#pragma unroll
      for (int pr = 0; pr < kLP; ++pr) sum += cred[pr * Dp + d];
      st_async_f32(dsmem_addr(cb + rank * Dp + d, 0u), sum, dsmem_addr(tbar, 0u));
    }
    if (rank == 0) {
      mbar_wait(tbar, 0);
      for (int d = tid; d < D; d += NT) {
        float sum = 0.0f;
        for (int r = 0; r < CL; ++r) sum += cb[r * Dp + d];
        p.c_all[((size_t)(S - 1) * B + b) * D + d] = sum;
      }
    }
  }
  // no trailing cluster barrier: a CTA leaves only after everything addressed to it has landed (its last wait)
  // and it never reads remote shared memory
}

// ------------------------------------------------------------------------------------------------
// TMEM as a warp-private resident operand store (backward).  Warp w owns TMEM lanes [32*(w%4), +32); lane i of the
// warp <-> TMEM lane, consecutive columns <-> consecutive registers (shape 32x32b).
// ------------------------------------------------------------------------------------------------
template <int N>
__device__ __forceinline__ void tmem_ldn(uint32_t taddr, float *v);
template <>
__device__ __forceinline__ void tmem_ldn<1>(uint32_t taddr, float *v) {
  uint32_t r0;
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(r0) : "r"(taddr));
  v[0] = __uint_as_float(r0);
}
template <>
__device__ __forceinline__ void tmem_ldn<2>(uint32_t taddr, float *v) {
  uint32_t r0, r1;
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=r"(r0), "=r"(r1) : "r"(taddr));
  v[0] = __uint_as_float(r0); v[1] = __uint_as_float(r1);
}
template <>
__device__ __forceinline__ void tmem_ldn<4>(uint32_t taddr, float *v) {
  uint32_t r0, r1, r2, r3;
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(taddr));
  v[0] = __uint_as_float(r0); v[1] = __uint_as_float(r1); v[2] = __uint_as_float(r2); v[3] = __uint_as_float(r3);
}
template <>
__device__ __forceinline__ void tmem_ldn<8>(uint32_t taddr, float *v) {
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
template <int N>
__device__ __forceinline__ void tmem_stn(uint32_t taddr, const float *v);
template <>
__device__ __forceinline__ void tmem_stn<1>(uint32_t taddr, const float *v) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x1.b32 [%0], {%1};" ::"r"(taddr), "r"(__float_as_uint(v[0])) : "memory");
}
template <>
__device__ __forceinline__ void tmem_stn<2>(uint32_t taddr, const float *v) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1, %2};" ::"r"(taddr), "r"(__float_as_uint(v[0])),
               "r"(__float_as_uint(v[1]))
               : "memory");
}
template <>
__device__ __forceinline__ void tmem_stn<4>(uint32_t taddr, const float *v) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr),
               "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])),
               "r"(__float_as_uint(v[3]))
               : "memory");
}
template <>
__device__ __forceinline__ void tmem_stn<8>(uint32_t taddr, const float *v) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr),
               "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])),
               "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])),
               "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7]))
               : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// N consecutive columns as power-of-two pieces (N <= 16)
template <int N>
__device__ __forceinline__ void tmem_load(uint32_t taddr, float *v) {
  if constexpr (N >= 8) { tmem_ldn<8>(taddr, v); if constexpr (N > 8) tmem_load<N - 8>(taddr + 8, v + 8); }
  else if constexpr (N >= 4) { tmem_ldn<4>(taddr, v); if constexpr (N > 4) tmem_load<N - 4>(taddr + 4, v + 4); }
  else if constexpr (N >= 2) { tmem_ldn<2>(taddr, v); if constexpr (N > 2) tmem_load<N - 2>(taddr + 2, v + 2); }
  else { tmem_ldn<1>(taddr, v); }
}
template <int N>
__device__ __forceinline__ void tmem_store(uint32_t taddr, const float *v) {
  if constexpr (N >= 8) { tmem_stn<8>(taddr, v); if constexpr (N > 8) tmem_store<N - 8>(taddr + 8, v + 8); }
  else if constexpr (N >= 4) { tmem_stn<4>(taddr, v); if constexpr (N > 4) tmem_store<N - 4>(taddr + 4, v + 4); }
  else if constexpr (N >= 2) { tmem_stn<2>(taddr, v); if constexpr (N > 2) tmem_store<N - 2>(taddr + 2, v + 2); }
  else { tmem_stn<1>(taddr, v); }
}

// ------------------------------------------------------------------------------------------------
// backward: steps S-1 .. 0 in one kernel.
//   TMEM         : pre rows in the pass-2 layout (pair <-> frame, lane <-> channel: APL columns per frame and warp),
//                  enc_h rows in the pass-1 layout (warp <-> frame, lane <-> d: DPL2 columns per frame and warp)
//   shared memory: the d pre tile of the current step (tloc x A), handed to the TMA unit per step (bulk store for the
//                  first processed step, cp.reduce.async.bulk.add.f32 afterwards); the channel-major d conv rows of
//                  ALL frames (pushed by the cluster, double-buffered); the chain gradient d att_prev of my frames
//   registers    : W_att (pairs along c), gvec; running dW_att row (threads < A) or dW_conv taps (threads >= A),
//                  running d gvec -- written once after the last step
// ------------------------------------------------------------------------------------------------
template <int APL, int CP, int DPL2>
__global__ void __launch_bounds__(kLT, 1) attloc_loop_bwd_kernel(const LoopBwdParams p) {
  constexpr int NT = kLT;
  constexpr int WP = CP + 1;
  constexpr int CPP = (CP + 3) & ~3;
  constexpr int CH2 = (CP + 1) / 2;
  extern __shared__ __align__(128) unsigned char smraw[];
  const LoopGeom g = p.g;
  const int C = CP == 10 ? 10 : p.C;
  const int Th = p.Th, D = p.D, A = p.A, K = p.K, S = p.S, B = p.B, filts = (p.K - 1) / 2;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, half = warp & 1, pair = warp >> 1;
  const int CL = (int)cluster_nctarank(), rank = (int)cluster_ctarank();
  const int b = blockIdx.x / CL;
  const int t0 = min(Th, rank * g.tloc_max), t1 = min(Th, t0 + g.tloc_max), tloc = t1 - t0;
  const int nchx = (tloc + kLP - 1) / kLP;        // pass-2 chunks (8 frames)
  const int nche = (tloc + kLW - 1) / kLW;        // pass-1 chunks (16 frames)
  const int nchx_max = (g.tloc_max + kLP - 1) / kLP, nche_max = (g.tloc_max + kLW - 1) / kLW;

  uint64_t *done_x = reinterpret_cast<uint64_t *>(smraw);    // every warp finished forming d pre in place
  uint64_t *xbar1 = done_x + 1;                               // [2] sum_t w dwt partials of every rank, by parity
  uint64_t *xbar2 = xbar1 + 2;                                // [2] d conv of every frame (+ d dec_proj partials on rank 0)
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(xbar2 + 2);
  float *xs = reinterpret_cast<float *>(smraw + 128);         // tloc_max*A    d pre tile of the current step
  float *dcvT = xs + (size_t)g.tloc_max * A;                  // 2*CP*App      channel-major zero padded d conv, by parity
  float *app = dcvT + 2 * CP * g.App;                         // App           padded att_prev of the current step
  float *wc_s = app + g.App;                                  // CKp
  float *conv_s = wc_s + g.CKp;                               // tloc_max*CPP
  float *w_s = conv_s + g.tloc_max * CPP;                     // round4(tloc_max)
  float *dwt_s = w_s + round4(g.tloc_max);                    // round4(tloc_max)
  float *de_s = dwt_s + round4(g.tloc_max);                   // round4(tloc_max)
  float *dwn_s = de_s + round4(g.tloc_max);                   // round4(tloc_max)  chain gradient (d att_prev of my frames)
  float *dcv_p = dwn_s + round4(g.tloc_max);                  // 2*tloc_max*16     per-half d conv partials
  float *ddp_w = dcv_p + 2 * g.tloc_max * 16;                 // kLW*(A/2)         per-warp d dec_proj partials
  float *scr = ddp_w + kLW * (A / 2);                         // max(A*WP, kKQ*CP*tloc_max): W_att staging, then d att_prev partials
  float *ddp_x = scr + max(A * WP, round4(kKQ * CP * g.tloc_max));   // 2*kLMaxCL*A   d dec_proj partials of every rank (rank 0)
  float *xch = ddp_x + 2 * kLMaxCL * A;                       // 2*kLMaxCL
  float *slot = p.acc_slots + (size_t)blockIdx.x * p.slot_stride;   // [dW_att A*C | dW_conv C*K | dgvec A | dgvec_b 1]

  const uint32_t x1bytes = (uint32_t)CL * 4u;
  const uint32_t x2bytes = (uint32_t)Th * (uint32_t)C * 4u + (rank == 0 ? (uint32_t)CL * (uint32_t)A * 4u : 0u);
  if (tid == 0) {
    mbar_init(done_x, kLW);
    for (int i = 0; i < 2; ++i) { mbar_init(&xbar1[i], 1); mbar_init(&xbar2[i], 1); }
    mbar_fence_init();
    for (int i = 0; i < 2; ++i) { mbar_expect_tx(&xbar1[i], x1bytes); mbar_expect_tx(&xbar2[i], x2bytes); }
  }
  cluster_arrive_relaxed();
  if (warp == 0) tmem_alloc(tmem_slot, 512);
  // parameters
  float gv[APL];
#pragma unroll
  for (int j = 0; j < APL; ++j) gv[j] = __ldg(p.gvec + half * (A / 2) + lane + 32 * j);
  for (int i = tid; i < C * K; i += NT) wc_s[i] = __ldg(p.W_conv + i);
  for (int i = tid; i < A * C; i += NT) { const int a = i / C; scr[a * WP + (i - a * C)] = __ldg(p.W_att + i); }
  {  // zero the pads of the channel-major d conv rows (the frames themselves are pushed by the cluster every step)
    const int padn = g.App - Th;
    for (int i = tid; i < 2 * CP * padn; i += NT) {
      const int c = i / padn, o = i - c * padn;
      dcvT[c * g.App + (o < filts ? o : Th + o)] = 0.0f;
    }
    // the per-step loads only write the C real channels of a conv row: pads must be (and stay) zero, they meet zero
    // weights in the recomputation
    for (int i = tid; i < g.tloc_max * CPP; i += NT) conv_s[i] = 0.0f;
    for (int i = tid; i < round4(g.tloc_max); i += NT) dwn_s[i] = 0.0f;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tbase = *tmem_slot + ((uint32_t)(32 * (warp & 3)) << 16);
  const uint32_t tcol_pre = tbase + (uint32_t)((warp >> 2) * nchx_max * APL);
  const uint32_t tcol_enc = tbase + (uint32_t)(g.col_enc + (warp >> 2) * nche_max * DPL2);
  // W_att rows of this lane's channels -> registers, as pairs along c (packed FFMA2 both ways)
  float2 WattC[APL][CH2];
#pragma unroll
  for (int j = 0; j < APL; ++j) {
    const int a = half * (A / 2) + lane + 32 * j;
#pragma unroll
    for (int c2 = 0; c2 < CH2; ++c2)
      WattC[j][c2] = make_float2(2 * c2 < C ? scr[a * WP + 2 * c2] : 0.0f, 2 * c2 + 1 < C ? scr[a * WP + 2 * c2 + 1] : 0.0f);
  }
  const int aoff = half * (A / 2) + lane;
  pdl_wait();
  // resident operands -> TMEM (coalesced 128 B row segments per warp, once per kernel)
  for (int q = 0; q < nchx; ++q) {
    const int tl = kLP * q + pair;
    float v[APL];
#pragma unroll
    for (int j = 0; j < APL; ++j) v[j] = tl < tloc ? __ldg(p.pre + ((size_t)b * Th + t0 + tl) * A + aoff + 32 * j) : 0.0f;
    tmem_store<APL>(tcol_pre + (uint32_t)(q * APL), v);
  }
  for (int q = 0; q < nche; ++q) {
    const int tl = kLW * q + warp;
    float v[DPL2];
#pragma unroll
    for (int j = 0; j < DPL2; ++j)
      v[j] = (tl < tloc && lane + 32 * j < D) ? __ldg(p.enc + ((size_t)b * Th + t0 + tl) * D + lane + 32 * j) : 0.0f;
    tmem_store<DPL2>(tcol_enc + (uint32_t)(q * DPL2), v);
  }
  tmem_wait_st();
  __syncthreads();   // scr (W_att staging) is free from here on
  cluster_wait();    // peers are resident: remote stores may start

  // running parameter gradients (registers, all steps)
  float pacc[kKG];
#pragma unroll
  for (int i = 0; i < kKG; ++i) pacc[i] = 0.0f;
  float dgv[APL];
#pragma unroll
  for (int j = 0; j < APL; ++j) dgv[j] = 0.0f;
  float dgb = 0.0f;
  const int nkg = (K + kKG - 1) / kKG;
  const bool conv_thread = tid >= A && tid - A < C * nkg;
  const int cw_c = conv_thread ? (tid - A) / nkg : 0, cw_kb = conv_thread ? ((tid - A) % nkg) * kKG : 0;

  for (int it = 0; it < S; ++it) {
    const int s = S - 1 - it;
    const uint32_t par = (uint32_t)it & 1u, ph = ((uint32_t)it >> 1) & 1u;
    float *dcv_cur = dcvT + par * CP * g.App;
    float *ddpx = ddp_x + par * kLMaxCL * A;
    float *xc = xch + par * kLMaxCL;
    const size_t sb = (size_t)s * B + b;
    // ---- per-step inputs: alignment (output of step s), its conv features, previous alignment (padded), gradients
    float dcr[DPL2];
#pragma unroll
    for (int j = 0; j < DPL2; ++j) dcr[j] = (p.dc_all && lane + 32 * j < D) ? __ldg(p.dc_all + sb * D + lane + 32 * j) : 0.0f;
    float dp[APL];
#pragma unroll
    for (int j = 0; j < APL; ++j) dp[j] = __ldg(p.dec_proj + sb * A + aoff + 32 * j);
    for (int i = tid; i < tloc; i += NT) {
      w_s[i] = __ldg(p.w_all + sb * Th + t0 + i);
      dwt_s[i] = dwn_s[i] + (p.dw_all ? __ldg(p.dw_all + sb * Th + t0 + i) : 0.0f);
    }
    for (int i = tid; i < tloc * C; i += NT) {
      const int tl = i / C;
      conv_s[tl * CPP + (i - tl * C)] = __ldg(p.conv_all + (sb * Th + t0) * C + i);
    }
    {
      const float *prev = s == 0 ? p.att_init + (size_t)b * Th : p.w_all + (sb - B) * Th;
      for (int i = tid; i < g.App; i += NT) {
        const int t = i - filts;
        app[i] = (t >= 0 && t < Th) ? __ldg(prev + t) : 0.0f;
      }
    }
    __syncthreads();  // #1

    // ---- pass 1: dwt[t] += enc_h[t,:] . dc   (warp per frame, lane <-> d, enc_h from TMEM)
    for (int q = 0; q < nche; ++q) {
      const int tl = kLW * q + warp;
      float ev[DPL2];
      tmem_load<DPL2>(tcol_enc + (uint32_t)(q * DPL2), ev);
      tmem_wait_ld();
      float dot = 0.0f;
#pragma unroll
      for (int j = 0; j < DPL2; ++j) dot = fmaf(dcr[j], ev[j], dot);
      dot = warp_sum(dot);
      if (lane == 0 && tl < tloc) dwt_s[tl] += dot;
    }
    __syncthreads();  // #2: dwt complete
    if (warp == 0) {
      float s1 = 0.0f;
      for (int tl = lane; tl < tloc; tl += 32) s1 = fmaf(w_s[tl], dwt_s[tl], s1);
      s1 = warp_sum(s1);
      if (lane < CL) st_async_f32(dsmem_addr(xc + rank, (uint32_t)lane), s1, dsmem_addr(&xbar1[par], (uint32_t)lane));
    }
    mbar_wait(&xbar1[par], ph);
    float Stot = 0.0f;
    for (int r = 0; r < CL; ++r) Stot += xc[r];
    for (int tl = tid; tl < tloc; tl += NT) de_s[tl] = p.scaling * w_s[tl] * (dwt_s[tl] - Stot);
    if (tid == 0) {
      mbar_expect_tx(&xbar1[par], x1bytes);
      if (it > 0) bulk_wait<0>();   // the previous step's d pre tile has left shared memory (and landed)
    }
    __syncthreads();  // #3

    // ---- pass 2: recompute x = tanh(W_att conv + pre + dec_proj), through tanh.  pair <-> frame, lane <-> channel
    float ddp[APL];
#pragma unroll
    for (int j = 0; j < APL; ++j) ddp[j] = 0.0f;
    // `pre` of chunk q+1 is requested from TMEM while chunk q is processed (the wait at the top of an iteration then
    // finds the data there); the empty asm pins the prefetch registers behind the wait
    float pn[APL];
    tmem_load<APL>(tcol_pre, pn);
#pragma unroll 1
    for (int q = 0; q < nchx; ++q) {
      const int tl = kLP * q + pair;
      tmem_wait_ld();
      float pv[APL];
#pragma unroll
      for (int j = 0; j < APL; ++j) {
        asm volatile("" : "+f"(pn[j]));
        pv[j] = pn[j];
      }
      if (q + 1 < nchx) tmem_load<APL>(tcol_pre + (uint32_t)((q + 1) * APL), pn);
      if (tl < tloc) {
        const float de = de_s[tl];
        const float *cvp = conv_s + tl * CPP;
        float cv[CPP];
#pragma unroll
        for (int c4 = 0; c4 < CPP; c4 += 4) {
          const float4 t4 = *reinterpret_cast<const float4 *>(cvp + c4);
          cv[c4] = t4.x; cv[c4 + 1] = t4.y; cv[c4 + 2] = t4.z; cv[c4 + 3] = t4.w;
        }
        float2 dcv2[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) dcv2[c] = make_float2(0.0f, 0.0f);
        float *row = xs + (size_t)tl * A + aoff;
#pragma unroll
        for (int j = 0; j < APL; ++j) {
          float2 u2 = make_float2(pv[j] + dp[j], 0.0f);
#pragma unroll
          for (int c2 = 0; c2 < CH2; ++c2)
            u2 = __ffma2_rn(WattC[j][c2], make_float2(cv[2 * c2], 2 * c2 + 1 < CPP ? cv[2 * c2 + 1] : 0.0f), u2);
          const float x = tanh_ex2(u2.x + u2.y);
          dgv[j] = fmaf(de, x, dgv[j]);
          const float dt = de * gv[j] * (1.0f - x * x);
          ddp[j] += dt;
          row[32 * j] = dt;  // d pre of this step
          const float2 dt2 = make_float2(dt, dt);
#pragma unroll
          for (int c2 = 0; c2 < CH2; ++c2) dcv2[c2] = __ffma2_rn(dt2, WattC[j][c2], dcv2[c2]);
        }
        if constexpr (CP == 10) {     // 10 channels: uneven halving tree, 12 shuffles instead of 31
          float dcv[10];
#pragma unroll
          for (int c = 0; c < 5; ++c) { dcv[2 * c] = dcv2[c].x; dcv[2 * c + 1] = dcv2[c].y; }
          warp_reduce10(dcv, lane);
          if ((lane & 1) == 0 && ((lane & 2) == 0 || (lane & 12) == 0)) {
            const int b4 = (lane >> 4) & 1, b3 = (lane >> 3) & 1, b2 = (lane >> 2) & 1;
            const int ci = 5 * b4 + ((lane & 2) ? 2 : (b2 ? (b3 ? 4 : 1) : (b3 ? 3 : 0)));
            dcv_p[(half * g.tloc_max + tl) * 16 + ci] = dcv[0];
          }
        } else {
          float dcv[16];
#pragma unroll
          for (int c = 0; c < 8; ++c) { dcv[2 * c] = dcv2[c].x; dcv[2 * c + 1] = dcv2[c].y; }
          warp_reduce16(dcv, lane);
          if ((lane & 1) == 0) {
            const int ci = ((lane >> 4) & 1) * 8 + ((lane >> 3) & 1) * 4 + ((lane >> 2) & 1) * 2 + ((lane >> 1) & 1);
            dcv_p[(half * g.tloc_max + tl) * 16 + ci] = dcv[0];
          }
        }
      }
    }
    fence_proxy_async_smem();   // this thread's tile writes -> visible to the bulk (async proxy) reads
    __syncwarp();
    if (lane == 0) mbar_arrive1(done_x);
    if (tid == 0 && tloc > 0) {  // hand the d pre tile to the TMA unit: d_pre[b, t0:t1, :] (+)= tile
      mbar_wait(done_x, (uint32_t)it & 1u);
      float *dst = p.d_pre + ((size_t)b * Th + t0) * A;
      const uint32_t total = (uint32_t)tloc * A * 4u;
      for (uint32_t o = 0; o < total; o += 32768u) {
        const uint32_t nb = total - o < 32768u ? total - o : 32768u;
        if (it > 0) bulk_red_add_s2g(reinterpret_cast<char *>(dst) + o, reinterpret_cast<char *>(xs) + o, nb);
        else bulk_s2g(reinterpret_cast<char *>(dst) + o, reinterpret_cast<char *>(xs) + o, nb);
      }
      bulk_commit();
    }
#pragma unroll
    for (int j = 0; j < APL; ++j) ddp_w[warp * (A / 2) + lane + 32 * j] = ddp[j];
    __syncthreads();  // #4: d pre tile complete, per-warp partials published

    // ---- post pass A: pushes first (their latency overlaps the parameter-gradient work below)
    for (int item = tid; item < tloc * C; item += NT) {   // d conv of my frames -> every CTA (channel-major, padded)
      const int c = item / tloc, tl = item - c * tloc;
      const float v = dcv_p[tl * 16 + c] + dcv_p[(g.tloc_max + tl) * 16 + c];
      for (int r = 0; r < CL; ++r)
        st_async_f32(dsmem_addr(dcv_cur + c * g.App + filts + t0 + tl, (uint32_t)r), v, dsmem_addr(&xbar2[par], (uint32_t)r));
    }
    for (int a = tid; a < A; a += NT) {                    // d dec_proj partial of this CTA -> rank 0
      const int h = a >= A / 2 ? 1 : 0, ai = a - h * (A / 2);
      float sd = 0.0f;
#pragma unroll
      for (int pr = 0; pr < kLP; ++pr) sd += ddp_w[(2 * pr + h) * (A / 2) + ai];
      st_async_f32(dsmem_addr(ddpx + rank * A + a, 0u), sd, dsmem_addr(&xbar2[par], 0u));
    }
    if (warp == kLW - 1) {   // d gvec.bias = sum_t de[t]  (analytically zero over the utterance; kept for fidelity)
      float s2 = 0.0f;
      for (int tl = lane; tl < tloc; tl += 32) s2 += de_s[tl];
      dgb += warp_sum(s2);
    }
    // parameter gradients that only need THIS CTA's frames, side by side on disjoint threads, into registers:
    //   threads [0, A)          : dW_att[a,c]  += sum_t d pre[t,a] conv[t,c]            (thread <-> a, from the tile)
    //   threads [A, A + C*nkg)  : dW_conv[c,k] += sum_t dconv[t,c] att_prev[t+k-filts]  (12 taps per thread)
    if (tid < A) {
#pragma unroll 5
      for (int tl = 0; tl < tloc; ++tl) {
        const float dt = xs[(size_t)tl * A + tid];
#pragma unroll
        for (int c4 = 0; c4 < CPP; c4 += 4) {
          const float4 t4 = *reinterpret_cast<const float4 *>(conv_s + tl * CPP + c4);
          if (c4 < CP) pacc[c4] = fmaf(dt, t4.x, pacc[c4]);
          if (c4 + 1 < CP) pacc[c4 + 1] = fmaf(dt, t4.y, pacc[c4 + 1]);
          if (c4 + 2 < CP) pacc[c4 + 2] = fmaf(dt, t4.z, pacc[c4 + 2]);
          if (c4 + 3 < CP) pacc[c4 + 3] = fmaf(dt, t4.w, pacc[c4 + 3]);
        }
      }
    } else if (conv_thread) {
      const float *ar = app + cw_kb;                  // att_prev[t + k - filts] = app[t + k]
      float x[kKG];
#pragma unroll
      for (int i = 0; i < kKG - 1; ++i) x[i] = ar[t0 + i];
#pragma unroll 12   // = kKG: the register window rotates back onto itself, no moves
      for (int tl = 0; tl < tloc; ++tl) {
        x[kKG - 1] = ar[t0 + tl + kKG - 1];
        const float dv = dcv_p[tl * 16 + cw_c] + dcv_p[(g.tloc_max + tl) * 16 + cw_c];   // d conv of MY frame tl
#pragma unroll
        for (int i = 0; i < kKG; ++i) pacc[i] = fmaf(dv, x[i], pacc[i]);
#pragma unroll
        for (int i = 0; i < kKG - 1; ++i) x[i] = x[i + 1];
      }
    }
    mbar_wait(&xbar2[par], ph);   // d conv of all Th frames (and on rank 0 every rank's d dec_proj partial) are here
    if (rank == 0) {
      for (int a = tid; a < A; a += NT) {
        float sd = 0.0f;
        for (int r = 0; r < CL; ++r) sd += ddpx[r * A + a];
        p.d_decproj[sb * A + a] = sd;
      }
    }
    // ---- d att_prev[t] = sum_c sum_k Wc[c,k] dconv[t - k + filts, c] for my frames: the chain gradient of step s-1
    if (s > 0) {
      const int nsg = (tloc + kTG - 1) / kTG;
      const int Kq = (K + kKQ - 1) / kKQ;
      const int nitems = nsg * C * kKQ;
      for (int item = tid; item < nitems; item += NT) {
        const int sg = item % nsg, rest = item / nsg, c = rest % C, kq = rest / C;
        const int k0 = kq * Kq, k1 = min(K, k0 + Kq);
        const float *wr = wc_s + c * K;
        // padded index of dconv[t - k + filts] is (t - k + 2*filts); outputs t = t0+5sg .. +4
        const float *dr = dcv_cur + c * g.App + (t0 + kTG * sg) + 2 * filts;
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f, a4 = 0.f;
        float x1 = dr[1 - k0], x2 = dr[2 - k0], x3 = dr[3 - k0], x4 = dr[4 - k0];
#pragma unroll 5
        for (int k = k0; k < k1; ++k) {
          const float x0 = dr[-k], wv = wr[k];
          a0 = fmaf(wv, x0, a0); a1 = fmaf(wv, x1, a1); a2 = fmaf(wv, x2, a2);
          a3 = fmaf(wv, x3, a3); a4 = fmaf(wv, x4, a4);
          x4 = x3; x3 = x2; x2 = x1; x1 = x0;
        }
        float *o = scr + ((size_t)(kq * C + c)) * g.tloc_max + kTG * sg;
        const int nv = min(kTG, tloc - kTG * sg);
        o[0] = a0;
        if (nv > 1) o[1] = a1;
        if (nv > 2) o[2] = a2;
        if (nv > 3) o[3] = a3;
        if (nv > 4) o[4] = a4;
      }
    }
    if (tid == 0) mbar_expect_tx(&xbar2[par], x2bytes);
    __syncthreads();  // #5
    if (s > 0) {
      for (int tl = tid; tl < tloc; tl += NT) {
        float sum = 0.0f;
        for (int i = 0; i < kKQ * C; ++i) sum += scr[(size_t)i * g.tloc_max + tl];
        dwn_s[tl] = sum;
      }
    }
    // the next iteration's barrier #1 orders dwn_s / scr / conv_s / app reuse
  }

  // ---- epilogue: running parameter gradients -> this CTA's private slot (plain stores; summed by acc_reduce)
  if (tid < A) {
#pragma unroll
    for (int c = 0; c < CP; ++c)
      if (c < C) slot[tid * C + c] = pacc[c];
  } else if (conv_thread) {
#pragma unroll
    for (int i = 0; i < kKG; ++i)
      if (cw_kb + i < K) slot[A * C + cw_c * K + cw_kb + i] = pacc[i];
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < APL; ++j) ddp_w[warp * (A / 2) + lane + 32 * j] = dgv[j];
  __syncthreads();
  for (int a = tid; a < A; a += NT) {
    const int h = a >= A / 2 ? 1 : 0, ai = a - h * (A / 2);
    float sg = 0.0f;
#pragma unroll
    for (int pr = 0; pr < kLP; ++pr) sg += ddp_w[(2 * pr + h) * (A / 2) + ai];
    slot[A * C + C * K + a] = sg;
  }
  if (warp == kLW - 1 && lane == 0) slot[A * C + C * K + A] = dgb;
  if (tid == 0) bulk_wait<0>();  // all d_pre traffic of this CTA has left shared memory / landed
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(*tmem_slot, 512);
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
inline int pick_cl(int B, int Th) {
  const int sms = num_sms();
  int CL = 1;
  while (CL < kLMaxCL && B * CL * 2 <= sms) CL *= 2;
  while (CL > 1 && (Th + CL - 1) / CL < kLP) CL /= 2;  // tiny Th: do not over-split
  return CL;
}

inline void loop_geom_common(int Th, int D, int C, int K, int CL, LoopGeom &g) {
  const int filts = (K - 1) / 2;
  g.tloc_max = (Th + CL - 1) / CL;
  g.App = round4(Th + 2 * filts + 8);
  g.CKp = round4(C * K);
  g.Thp = round4(Th);
  g.Dp = round4(D);
  g.col_enc = 0;
  g.ncols = 0;
}

// forward: the CTA's whole (pre | enc) frame range must be resident in shared memory
inline bool loop_geom_fwd(int B, int Th, int D, int A, int C, int K, int CP, int &CL, LoopGeom &g, size_t &smem) {
  CL = pick_cl(B, Th);
  const int CPP = round4(CP);
  for (;;) {
    loop_geom_common(Th, D, C, K, CL, g);
    const size_t floats = (size_t)g.tloc_max * (A + D) + g.App + g.CKp + (size_t)A * (CP + 1) +
                          round4(kKQ * g.tloc_max * CP) + (size_t)g.tloc_max * CPP + 2 * (size_t)g.Thp +
                          round4(g.tloc_max) + round4(2 * g.tloc_max) + 2 * kLW + (size_t)kLP * g.Dp +
                          2 * (size_t)kLMaxCL * g.Dp + 4 * kLMaxCL;
    smem = 128 + sizeof(float) * floats;
    if (smem <= 226 * 1024) return true;
    if (CL >= kLMaxCL || B * CL * 2 > num_sms()) return false;   // longer utterances: the per-step kernels stream instead
    CL *= 2;
  }
}

// backward: pre / enc rows in TMEM (512 columns), the d pre tile in shared memory
inline bool loop_geom_bwd(int B, int Th, int D, int A, int C, int K, int CP, int dpl2, int &CL, LoopGeom &g,
                          size_t &smem) {
  CL = pick_cl(B, Th);
  const int CPP = round4(CP);
  const int nkg = (K + kKG - 1) / kKG;
  if (A + C * nkg > kLT) return false;   // dW_att rows and dW_conv taps live side by side in registers
  for (;;) {
    loop_geom_common(Th, D, C, K, CL, g);
    const int nchx_max = (g.tloc_max + kLP - 1) / kLP, nche_max = (g.tloc_max + kLW - 1) / kLW;
    g.col_enc = 4 * nchx_max * (A / 64);
    g.ncols = g.col_enc + 4 * nche_max * dpl2;
    const size_t scr = (size_t)A * (CP + 1) > (size_t)round4(kKQ * CP * g.tloc_max) ? (size_t)A * (CP + 1)
                                                                                   : (size_t)round4(kKQ * CP * g.tloc_max);
    const size_t floats = (size_t)g.tloc_max * A + 2 * (size_t)CP * g.App + g.App + g.CKp + (size_t)g.tloc_max * CPP +
                          4 * (size_t)round4(g.tloc_max) + 2 * (size_t)g.tloc_max * 16 + (size_t)kLW * (A / 2) + scr +
                          2 * (size_t)kLMaxCL * A + 2 * kLMaxCL;
    smem = 128 + sizeof(float) * floats;
    if (smem <= 226 * 1024 && g.ncols <= 512) return true;
    if (CL >= kLMaxCL || B * CL * 2 > num_sms()) return false;
    CL *= 2;
  }
}

// launched with programmatic dependent launch, like the step kernels
template <int APL, int CP>
int run_loop_fwd(const LoopFwdParams &prm, int CL, size_t smem, cudaStream_t st) {
  const dim3 grid((unsigned)(prm.B * CL));
  if (prm.D == prm.A) return launch_cluster(attloc_loop_fwd_kernel<APL, CP, APL>, grid, dim3(kLT), smem, st, CL, true, prm);
  return launch_cluster(attloc_loop_fwd_kernel<APL, CP, 8>, grid, dim3(kLT), smem, st, CL, true, prm);
}
template <int APL, int CP>
int run_loop_bwd(const LoopBwdParams &prm, int CL, size_t smem, cudaStream_t st) {
  const dim3 grid((unsigned)(prm.B * CL));
  if (prm.D == prm.A) return launch_cluster(attloc_loop_bwd_kernel<APL, CP, 2 * APL>, grid, dim3(kLT), smem, st, CL, true, prm);
  return launch_cluster(attloc_loop_bwd_kernel<APL, CP, 16>, grid, dim3(kLT), smem, st, CL, true, prm);
}

}  // namespace
}  // namespace re2e

using namespace re2e;

extern "C" int re2e_attloc_loop_supported(int S, int B, int Th, int D, int A, int C, int K) {
  if (S <= 0 || check_dims(B, Th, D, A, C, K) != RE2E_OK) return 0;
  const int CP = C == 10 ? 10 : 16;
  int CLf, CLb;
  size_t smem;
  LoopGeom g;
  if (!loop_geom_fwd(B, Th, D, A, C, K, CP, CLf, g, smem)) return 0;
  if (!loop_geom_bwd(B, Th, D, A, C, K, CP, D == A ? 2 * (A / 64) : 16, CLb, g, smem)) return 0;
  return 1;
}

extern "C" int re2e_attloc_loop_slots(int S, int B, int Th, int D, int A, int C, int K) {
  RE2E_CHECK_ARG(S > 0);
  int rc = check_dims(B, Th, D, A, C, K);
  if (rc != RE2E_OK) return rc;
  int CL;
  size_t smem;
  LoopGeom g;
  if (!loop_geom_bwd(B, Th, D, A, C, K, C == 10 ? 10 : 16, D == A ? 2 * (A / 64) : 16, CL, g, smem))
    return RE2E_E_UNSUPPORTED;
  return B * CL;
}

extern "C" int re2e_attloc_loop_fwd(const float *pre, const float *enc_h, const float *dec_proj,
                                    const float *att_init, const float *W_att, const float *W_conv,
                                    const float *gvec, const float *gvec_b, float scaling, float *c_all,
                                    float *w_all, float *conv_all, int S, int B, int Th, int D, int A, int C,
                                    int K, void *stream) {
  RE2E_CHECK_ARG(pre && enc_h && dec_proj && att_init && W_att && W_conv && gvec && gvec_b && c_all && w_all && S > 0);
  int rc = check_dims(B, Th, D, A, C, K);
  if (rc != RE2E_OK) return rc;
  RE2E_CHECK_ARG(aligned16(pre) && aligned16(enc_h));
  const int CP = C == 10 ? 10 : 16;
  LoopFwdParams prm;
  prm.pre = pre; prm.enc = enc_h; prm.dec_proj = dec_proj; prm.att_init = att_init; prm.W_att = W_att;
  prm.W_conv = W_conv; prm.gvec = gvec; prm.gvec_b = gvec_b; prm.scaling = scaling; prm.c_all = c_all;
  prm.w_all = w_all; prm.conv_all = conv_all;
  prm.S = S; prm.B = B; prm.Th = Th; prm.D = D; prm.A = A; prm.C = C; prm.K = K;
  int CL;
  size_t smem;
  if (!loop_geom_fwd(B, Th, D, A, C, K, CP, CL, prm.g, smem)) return RE2E_E_UNSUPPORTED;
  ATT_DISPATCH(run_loop_fwd, A / 64, CP, (prm, CL, smem, static_cast<cudaStream_t>(stream)));
  return rc;
}

extern "C" int re2e_attloc_loop_bwd(const float *pre, const float *enc_h, const float *dec_proj,
                                    const float *att_init, const float *w_all, const float *conv_all,
                                    const float *dc_all, const float *dw_all, const float *W_att,
                                    const float *W_conv, const float *gvec, float scaling, float *d_pre,
                                    float *d_decproj, float *acc_slots, int n_slots, int S, int B, int Th, int D,
                                    int A, int C, int K, void *stream) {
  RE2E_CHECK_ARG(pre && enc_h && dec_proj && att_init && w_all && conv_all && W_att && W_conv && gvec);
  RE2E_CHECK_ARG(d_pre && d_decproj && acc_slots && S > 0);
  int rc = check_dims(B, Th, D, A, C, K);
  if (rc != RE2E_OK) return rc;
  RE2E_CHECK_ARG(aligned16(d_pre));
  const int CP = C == 10 ? 10 : 16;
  LoopBwdParams prm;
  prm.pre = pre; prm.enc = enc_h; prm.dec_proj = dec_proj; prm.att_init = att_init; prm.w_all = w_all;
  prm.conv_all = conv_all; prm.dc_all = dc_all; prm.dw_all = dw_all; prm.W_att = W_att; prm.W_conv = W_conv;
  prm.gvec = gvec; prm.scaling = scaling; prm.d_pre = d_pre; prm.d_decproj = d_decproj; prm.acc_slots = acc_slots;
  prm.slot_stride = (int)re2e_attloc_acc_floats(A, C, K);
  prm.S = S; prm.B = B; prm.Th = Th; prm.D = D; prm.A = A; prm.C = C; prm.K = K;
  int CL;
  size_t smem;
  if (!loop_geom_bwd(B, Th, D, A, C, K, CP, D == A ? 2 * (A / 64) : 16, CL, prm.g, smem)) return RE2E_E_UNSUPPORTED;
  if (n_slots < B * CL) return RE2E_E_WORKSPACE;
  ATT_DISPATCH(run_loop_bwd, A / 64, CP, (prm, CL, smem, static_cast<cudaStream_t>(stream)));
  return rc;
}
