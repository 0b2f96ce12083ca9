// Location-aware attention step (AttLoc.forward, model/e2e_attention.py:258-299) for sm_100a,
// forward and backward, one thread-block-cluster kernel each.
//
// Mapping.  One CLUSTER of CL CTAs per utterance b; CTA `rank` owns the encoder frames
// [t0,t1) = rank*ceil(Th/CL) ....  The big per-step operands pre[b,t0:t1,:] / enc_h[b,t0:t1,:] (and in
// the backward the saved tanh activations) are contiguous in HBM, so they are fetched with 1-D bulk
// async copies (TMA, cp.async.bulk -> SASS UBLKCP) in chunks of NW frames into a shared-memory ring,
// each chunk signalled on its own mbarrier; all loads are in flight while the CTA computes the location
// convolution.  Softmax statistics and the context vector are combined across the CTAs of the cluster
// through distributed shared memory (ld.shared::cluster) -- no global round trip, no second kernel.
// The forward writes tanh(.) in place into the ring and hands the chunk back to the TMA unit (bulk
// store) so the backward does not recompute W_att*conv + tanh; the backward forms d pre in place in
// the ring and lets the TMA unit accumulate it into HBM (cp.reduce.async.bulk.add.f32 -> UBLKRED): the
// SM never reads d_pre.
// Algorithmic bytes per step (fp32): fwd 4*B*Th*(A+D) read (+4*B*Th*A activation save when training);
// bwd 4*B*Th*(A+D) read + 4*B*Th*A reduce.
//
// Thread mapping (NW warps): for the energy part a frame is handled by a PAIR of warps, each owning
// half of the A attention channels, lane <-> channel (a = half*A/2 + lane + 32j): W_att (A x C) lives in
// registers (APL*CP floats per lane).  The 1 x K location convolution and its two transposes in the
// backward are register-blocked sliding-window FMAs (5 outputs per thread, K split 4 ways).
#include <math_constants.h>

#include "attloc_common.cuh"

namespace re2e {
namespace {

constexpr int kMaxStages = 30;

struct AttGeom {
  int tloc_max, nch, ns, stage_floats, Thp, CKp, App;  // App: padded alignment row Th + 2*filts + 8
  int ring_floats;                                     // backward: floats reserved for the enc_h ring / its aliases
};

struct AttFwdParams {
  const float *pre, *enc, *att_prev, *dec_z, *W_dec, *W_att, *W_conv, *gvec, *gvec_b;
  float scaling;
  float *c, *w, *dec_proj, *conv, *xsave;
  int B, Th, D, A, Z, C, K;
  AttGeom g;
};

struct AttBwdParams {
  const float *dc, *dw, *xsave, *enc, *att_prev, *w, *conv, *W_dec, *W_decT, *W_att, *W_conv, *gvec;
  float scaling;
  float *d_pre, *d_decproj, *d_dec_z, *d_att_prev, *acc_slots;
  int accumulate_pre, slot_stride;
  int B, Th, D, A, Z, C, K;
  AttGeom g;
};

// issue chunk `q` of the [first | second] operand sequence into ring stage q % ns
template <int NW>
__device__ __forceinline__ void issue_chunk(int q, int nch, const AttGeom &g, const float *first, int wfirst,
                                            const float *second, int wsecond, int b, int Th, int t0, int t1,
                                            float *stages, uint64_t *full) {
  const int st = q % g.ns;
  const bool is_first = q < nch;
  const int qq = is_first ? q : q - nch;
  const int r0 = t0 + NW * qq;
  const int rows = min(NW, t1 - r0);
  const int width = is_first ? wfirst : wsecond;
  const float *src = (is_first ? first : second) + ((size_t)b * Th + r0) * width;
  const uint32_t bytes = (uint32_t)rows * width * 4u;
  mbar_expect_tx(&full[st], bytes);
  bulk_g2s(stages + (size_t)st * g.stage_floats, src, bytes, &full[st]);
}

// ------------------------------------------------------------------------------------------------
// forward (v3): ONE pass over the CTA's frames with an online softmax.
//
//   thread 0         : producer -- initialises the mbarriers and issues the bulk copies of the
//                      (pre chunk | enc chunk) stages up front (the whole frame range when it fits); a ring
//                      shorter than the range is refilled once all 16 warps released the stage
//   warps 0..15      : 8 warp PAIRS; pair p owns frame 8q+p of chunk q; the two warps of a pair split the
//                      A attention channels (energy) and the D encoder channels (context), lane <-> channel
//   per frame        : u = W_att conv[t] + pre[t] + dec_proj ; x = tanh(u) (stored for the backward) ;
//                      e = g.x (warp shuffle + 64-thread named barrier inside the pair) ;
//                      running (max, sum, context) update -- no CTA-wide barrier inside the frame loop
//   mlp_dec          : dec_proj = W_dec dec_z is computed INSIDE the kernel: every CTA of the cluster
//                      produces A/CL channels and pushes them into its peers' shared memory (DSMEM)
//   cluster combine  : every CTA pushes (max, sum) to all peers and its partial context to rank 0; after
//                      one cluster barrier all reads are local
// ------------------------------------------------------------------------------------------------
constexpr int kFP = 8;                  // warp pairs = frames per chunk
constexpr int kFW = 2 * kFP;            // compute warps
constexpr int kFT = kFW * 32;
constexpr int kDpl = 8;                 // D <= 512: encoder channels per lane per half
static_assert(8 * (kMaxStages + 2) <= 256, "forward: the mbarriers must leave bytes 256..383 of the header to the exchange");
// rows of the partial-context buffer: 8 up to clusters of 8
inline int fwd_rank_rows(int CL) { return CL > 8 ? CL : 8; }

template <int APL, int CP, int DPL>
__global__ void __launch_bounds__(kFT, 1) attloc_fwd_kernel(const AttFwdParams p) {
  constexpr int NT = kFT;
  constexpr int WP = CP + 1;             // odd pitch of the staged W_att rows: conflict-free lane <-> a reads
  constexpr int CPP = (CP + 3) & ~3;     // pitch of conv rows in shared memory (128-bit broadcast reads)
  extern __shared__ __align__(128) unsigned char smraw[];
  const AttGeom g = p.g;
  const int C = CP == 10 ? 10 : p.C;     // the CP == 10 instantiation is only dispatched for C == 10
  const int Th = p.Th, D = p.D, A = p.A, K = p.K, Z = p.Z, filts = (p.K - 1) / 2;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, half = warp & 1, pair = warp >> 1;
  const int CL = (int)cluster_nctarank(), rank = (int)cluster_ctarank();
  const int b = blockIdx.x / CL;
  const int t0 = min(Th, rank * g.tloc_max), t1 = min(Th, t0 + g.tloc_max), tloc = t1 - t0;
  const int nch = (tloc + kFP - 1) / kFP;
  const int Dp = round4(D), Dh = (D + 1) / 2;

  uint64_t *full = reinterpret_cast<uint64_t *>(smraw);
  uint64_t *dpbar = full + kMaxStages;                    // dec_proj row complete (A floats pushed by the cluster)
  uint64_t *xbar = dpbar + 1;                              // softmax statistics (+ partial contexts on rank 0) complete
  float *stages = reinterpret_cast<float *>(smraw + 512);
  float *app = stages + (size_t)g.ns * g.stage_floats;     // App   zero padded alignment row, ap[i] at filts+i
  float *wc_s = app + g.App;                               // CKp
  float *watt_s = wc_s + g.CKp;                            // A*WP
  float *dz_s = watt_s + A * WP;                           // round4(Z)
  float *dp_s = dz_s + round4(Z);                          // A      dec_proj, pushed by the cluster
  float *convp = dp_s + A;                                 // kKQ*tloc_max*CP  conv partials
  float *conv_s = convp + round4(kKQ * g.tloc_max * CP);   // tloc_max*CPP
  float *e_s = conv_s + g.tloc_max * CPP;                  // round4(tloc_max)  scaled energies
  float *epart = e_s + round4(g.tloc_max);                 // 2*tloc_max  per-frame partial energies of the two halves
  float *wstat = epart + round4(2 * g.tloc_max);           // kFW*2
  float *cbuf = wstat + 2 * kFW;                           // max(CL,8)*Dp  partial contexts (used on rank 0)
  float *xch = reinterpret_cast<float *>(smraw + 256);     // 2*16   (max, sum) of every rank, behind the mbarriers
  float *cred = stages;                                    // kFP*Dp, aliases the ring once it is drained

  auto issue = [&](int q) {
    const int st = q % g.ns;
    const int r0 = t0 + kFP * q;
    const int rows = min(kFP, t1 - r0);
    float *dst = stages + (size_t)st * g.stage_floats;
    mbar_expect_tx(&full[st], (uint32_t)rows * (uint32_t)(A + D) * 4u);
    bulk_g2s(dst, p.pre + ((size_t)b * Th + r0) * A, (uint32_t)rows * A * 4u, &full[st]);
    bulk_g2s(dst + kFP * A, p.enc + ((size_t)b * Th + r0) * D, (uint32_t)rows * D * 4u, &full[st]);
  };

  // ---- every global load of the prologue is issued before the first use: ONE L2 round trip for the small
  //      operands (alignment row, W_conv, W_att, dec_z, gvec) and this warp's W_dec rows
  constexpr int kCPW = 5;                              // mlp_dec channels per warp per pass
  constexpr int kZQ = 3;                               // 128-bit quads per lane per pass (Z <= 384 in one pass)
  const int apc = A / CL, a_begin = rank * apc;        // this CTA's slice of the A mlp_dec channels
  const bool wvec = p.dec_z && ((Z & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.W_dec) & 15u) == 0);
  float4 wv[kCPW][kZQ];
  if (wvec) {
    const int zq = Z >> 2;
#pragma unroll
    for (int u = 0; u < kCPW; ++u) {
      const int ai = warp + kFW * u;
      const float4 *wr = reinterpret_cast<const float4 *>(p.W_dec + (size_t)(a_begin + min(ai, apc - 1)) * Z);
#pragma unroll
      for (int v = 0; v < kZQ; ++v) {
        const int z4 = lane + 32 * v;
        wv[u][v] = (ai < apc && z4 < zq) ? __ldg(wr + z4) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
  }
  float gv[APL];
#pragma unroll
  for (int j = 0; j < APL; ++j) gv[j] = __ldg(p.gvec + half * (A / 2) + lane + 32 * j);
  const float gb = __ldg(p.gvec_b);
  constexpr int IA = 2, IC = 4, IW = 8;                // first block of every array: loads batched in registers
  float va[IA], vc[IC], vw[IW], vz;
  {
#pragma unroll
    for (int u = 0; u < IC; ++u) {
      const int i = tid + u * NT;
      vc[u] = i < C * K ? __ldg(p.W_conv + i) : 0.0f;
    }
#pragma unroll
    for (int u = 0; u < IW; ++u) {
      const int i = tid + u * NT;
      vw[u] = i < A * C ? __ldg(p.W_att + i) : 0.0f;
    }
  }
  // thread 0: barriers first (peers may push as soon as the cluster handshake completes), then the bulk copies of
  // the (pre | enc) stages -- issued AFTER this warp's prologue loads are in flight, so the serial issue loop of
  // one lane does not delay the loads of its warp
  if (tid == 0) {
    for (int i = 0; i < g.ns; ++i) mbar_init(&full[i], 1);
    mbar_init(dpbar, 1);
    mbar_init(xbar, 1);
    mbar_fence_init();
    if (p.dec_z) mbar_expect_tx(dpbar, (uint32_t)A * 4u);
    mbar_expect_tx(xbar, (uint32_t)CL * 8u + (rank == 0 ? (uint32_t)CL * (uint32_t)D * 4u : 0u));
  }
  // "this CTA is running and its barriers exist": peers wait on it before their first remote store
  cluster_arrive_relaxed();
  // whole == the ring holds the CTA's entire frame range (the common case): pre[b, t0:t1, :] and enc_h[b, t0:t1, :]
  // are two contiguous spans, fetched by TWO bulk copies on ONE mbarrier, laid out [pre rows | enc rows] -- the
  // single issuing lane is on the critical path of the prologue (everyone waits for it at barrier #1).
  const bool whole = g.ns >= nch;
  if (tid == 0) {
    if (whole) {
      if (tloc > 0) {
        mbar_expect_tx(&full[0], (uint32_t)tloc * (uint32_t)(A + D) * 4u);
        bulk_g2s(stages, p.pre + ((size_t)b * Th + t0) * A, (uint32_t)tloc * A * 4u, &full[0]);
        bulk_g2s(stages + (size_t)g.tloc_max * A, p.enc + ((size_t)b * Th + t0) * D, (uint32_t)tloc * D * 4u, &full[0]);
      }
    } else {
      const int first = nch < g.ns ? nch : g.ns;
      for (int q = 0; q < first; ++q) issue(q);
    }
  }
  {
#pragma unroll
    for (int u = 0; u < IC; ++u)
      if (tid + u * NT < C * K) wc_s[tid + u * NT] = vc[u];
#pragma unroll
    for (int u = 0; u < IW; ++u) {
      const int i = tid + u * NT;
      if (i < A * C) { const int a = i / C; watt_s[a * WP + (i - a * C)] = vw[u]; }
    }
    for (int i = tid + IC * NT; i < C * K; i += NT) wc_s[i] = __ldg(p.W_conv + i);
    for (int i = tid + IW * NT; i < A * C; i += NT) { const int a = i / C; watt_s[a * WP + (i - a * C)] = __ldg(p.W_att + i); }
  }
  // ---- PDL boundary: the per-step inputs (previous alignment, decoder state) exist only once the predecessor
  //      grid has completed; the next step's grid may start its own prologue from here on
  pdl_wait();
  pdl_launch_dependents();
  {
#pragma unroll
    for (int u = 0; u < IA; ++u) {
      const int i = tid + u * NT, t = i - filts;
      va[u] = (i < g.App && t >= 0 && t < Th) ? __ldcg(p.att_prev + (size_t)b * Th + t) : 0.0f;
    }
    vz = (p.dec_z && tid < Z) ? __ldcg(p.dec_z + (size_t)b * Z + tid) : 0.0f;
#pragma unroll
    for (int u = 0; u < IA; ++u)
      if (tid + u * NT < g.App) app[tid + u * NT] = va[u];
    if (tid < Z) dz_s[tid] = vz;
    // remainders (shapes beyond the first block)
    for (int i = tid + IA * NT; i < g.App; i += NT) {
      const int t = i - filts;
      app[i] = (t >= 0 && t < Th) ? __ldcg(p.att_prev + (size_t)b * Th + t) : 0.0f;
    }
    for (int i = tid + NT; i < Z; i += NT) dz_s[i] = p.dec_z ? __ldcg(p.dec_z + (size_t)b * Z + i) : 0.0f;
  }
  __syncthreads();  // #1

  // ---- mlp_dec slice of this CTA: channels [rank*A/CL, (rank+1)*A/CL), one warp per channel, lane <-> z
  for (int base = 0; base < apc; base += kFW * kCPW) {
    float dots[kCPW];
#pragma unroll
    for (int u = 0; u < kCPW; ++u) dots[u] = 0.0f;
    if (p.dec_z) {
      if (wvec) {
        const int zq = Z >> 2;
        for (int zb = 0; zb < zq; zb += 32 * kZQ) {
          if (base != 0 || zb != 0) {   // later passes: reload (the first pass was issued in the prologue)
#pragma unroll
            for (int u = 0; u < kCPW; ++u) {
              const int ai = base + warp + kFW * u;
              const float4 *wr = reinterpret_cast<const float4 *>(p.W_dec + (size_t)(a_begin + min(ai, apc - 1)) * Z);
#pragma unroll
              for (int v = 0; v < kZQ; ++v) {
                const int z4 = zb + lane + 32 * v;
                wv[u][v] = (ai < apc && z4 < zq) ? __ldg(wr + z4) : make_float4(0.f, 0.f, 0.f, 0.f);
              }
            }
          }
#pragma unroll
          for (int v = 0; v < kZQ; ++v) {
            const int z4 = zb + lane + 32 * v;
            const float4 dz = z4 < zq ? *reinterpret_cast<const float4 *>(dz_s + 4 * z4) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int u = 0; u < kCPW; ++u)
              dots[u] = fmaf(wv[u][v].x, dz.x, fmaf(wv[u][v].y, dz.y, fmaf(wv[u][v].z, dz.z, fmaf(wv[u][v].w, dz.w, dots[u]))));
          }
        }
      } else {
#pragma unroll
        for (int u = 0; u < kCPW; ++u) {
          const int ai = base + warp + kFW * u;
          if (ai < apc) {
            const float *wr = p.W_dec + (size_t)(a_begin + ai) * Z;
            for (int z = lane; z < Z; z += 32) dots[u] = fmaf(__ldg(wr + z), dz_s[z], dots[u]);
          }
        }
      }
    }
#pragma unroll
    for (int u = 0; u < kCPW; ++u) dots[u] = warp_sum(dots[u]);
    if (base == 0) cluster_wait();  // every peer CTA is resident, its mbarriers initialised
    if (p.dec_z) {
#pragma unroll
      for (int u = 0; u < kCPW; ++u) {
        const int ai = base + warp + kFW * u;
        if (ai < apc && lane < CL)
          st_async_f32(dsmem_addr(dp_s + a_begin + ai, (uint32_t)lane), dots[u], dsmem_addr(dpbar, (uint32_t)lane));
        if (ai < apc && lane == 0 && p.dec_proj) p.dec_proj[(size_t)b * A + a_begin + ai] = dots[u];
      }
    }
  }

  // ---- location convolution: conv[t,c] = sum_k Wc[c,k] * att_prev[t + k - filts]  (zero padded).
  //      item = (k quarter, channel, group of 5 frames): 2 shared loads per 5 FMAs
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
  // W_att rows of this lane's channels -> registers (independent of the conv partials), two channels per 64-bit
  // register pair so that the K=C dot products run as packed FFMA2 (fma.rn.f32x2, sm_100)
  constexpr int APH = (APL + 1) / 2;
  float2 WattP[APH][CP];
#pragma unroll
  for (int jp = 0; jp < APH; ++jp) {
    const int a0 = half * (A / 2) + lane + 32 * (2 * jp), a1 = a0 + 32;
#pragma unroll
    for (int c = 0; c < CP; ++c)
      WattP[jp][c] = make_float2(c < C ? watt_s[a0 * WP + c] : 0.0f, (c < C && 2 * jp + 1 < APL) ? watt_s[a1 * WP + c] : 0.0f);
  }
  __syncthreads();  // #2
  for (int i = tid; i < tloc * CPP; i += NT) {
    const int tl = i / CPP, c = i - tl * CPP;
    float v = 0.0f;
    if (c < C) {
#pragma unroll
      for (int kq = 0; kq < kKQ; ++kq) v += convp[((size_t)kq * g.tloc_max + tl) * CP + c];
      if (p.conv) p.conv[((size_t)b * Th + t0 + tl) * C + c] = v;
    }
    conv_s[i] = v;
  }
  if (p.dec_z) mbar_wait(dpbar, 0);   // dp_s holds the full dec_proj row (A floats pushed by the CTAs of the cluster)
  __syncthreads();  // #3: conv_s visible

  float m_run = -CUDART_INF_F, s_run = 0.0f;
  float acc[DPL];
#pragma unroll
  for (int j = 0; j < DPL; ++j) acc[j] = 0.0f;
  {
    float dp[APL];
#pragma unroll
    for (int j = 0; j < APL; ++j) dp[j] = p.dec_z ? dp_s[half * (A / 2) + lane + 32 * j] : 0.0f;
    uint32_t dmask = 0;                        // which of this lane's DPL encoder channels exist
#pragma unroll
    for (int j = 0; j < DPL; ++j)
      if (lane + 32 * j < Dh && half * Dh + lane + 32 * j < D) dmask |= 1u << j;
    const int aoff = half * (A / 2) + lane;
    // The frame range is processed in groups of g.ns chunks (ONE group when the ring holds the whole range, the
    // common case).  Per group: (1) energies of all its frames back to back -- no barrier inside, so the shuffle
    // reduction of one frame overlaps the FMAs of the next; (2) one 64-thread barrier inside the pair; (3) local
    // softmax statistics + context over the group's frames.
    for (int qg = 0; qg < nch; qg += g.ns) {
      const int gsz = min(g.ns, nch - qg);
      const uint32_t ph = (uint32_t)((qg / g.ns) & 1);
      if (whole) { if (tloc > 0) mbar_wait(&full[0], 0); }
      else for (int i = 0; i < gsz; ++i) mbar_wait(&full[i], ph);
      // (1) partial energies of this warp's half of the channels
#pragma unroll 2
      for (int i = 0; i < gsz; ++i) {
        const int tl = kFP * (qg + i) + pair;
        if (tl < tloc) {
          const float *cvp = conv_s + tl * CPP;
          float cv[CPP];
#pragma unroll
          for (int c4 = 0; c4 < CPP; c4 += 4) {
            const float4 t4 = *reinterpret_cast<const float4 *>(cvp + c4);
            cv[c4] = t4.x; cv[c4 + 1] = t4.y; cv[c4 + 2] = t4.z; cv[c4 + 3] = t4.w;
          }
          const float *row = (whole ? stages + (size_t)tl * A : stages + (size_t)i * g.stage_floats + pair * A) + aoff;
          float *xs = p.xsave ? p.xsave + ((size_t)b * Th + t0 + tl) * A + aoff : nullptr;
          float part = 0.0f;
#pragma unroll
          for (int jp = 0; jp < APH; ++jp) {
            const bool two = 2 * jp + 1 < APL;
            float2 u = make_float2(dp[2 * jp] + row[64 * jp], two ? dp[2 * jp + 1] + row[64 * jp + 32] : 0.0f);
#pragma unroll
            for (int c = 0; c < CP; ++c) u = __ffma2_rn(WattP[jp][c], make_float2(cv[c], cv[c]), u);
            const float x0 = tanh_ex2(u.x);
            if (xs) xs[64 * jp] = x0;  // activation kept for the backward (coalesced 128 B per warp store)
            part = fmaf(gv[2 * jp], x0, part);
            if (two) {
              const float x1 = tanh_ex2(u.y);
              if (xs) xs[64 * jp + 32] = x1;
              part = fmaf(gv[2 * jp + 1], x1, part);
            }
          }
          part = warp_sum(part);
          if (lane == 0) epart[2 * tl + half] = part;
        }
      }
      pair_bar(1 + pair, 64);
      if (gsz <= 8) {
        // common case (<= 8 frames per pair and group): everything of steps (2) and (3) for the group's frames is
        // issued up front -- 16 broadcast LDS, 8 exponentials, 8*DPL independent LDS -- instead of one frame at a
        // time (the per-frame version is latency bound: LDS -> FADD -> EX2 -> FFMA chains back to back)
        float ev[8];
        float mg8 = m_run;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int tl = kFP * (qg + i) + pair;
          const bool ok = i < gsz && tl < tloc;
          ev[i] = ok ? p.scaling * ((epart[2 * tl] + epart[2 * tl + 1]) + gb) : -CUDART_INF_F;
          if (ok && half == 0 && lane == 0) e_s[tl] = ev[i];
          mg8 = fmaxf(mg8, ev[i]);
        }
        if (mg8 > m_run) {
          const float sc = __expf(m_run - mg8);   // exp(-inf) = 0 for the first group
          s_run *= sc;
#pragma unroll
          for (int j = 0; j < DPL; ++j) acc[j] *= sc;
          m_run = mg8;
        }
        const float *er0 = (whole ? stages + (size_t)g.tloc_max * A + (size_t)(kFP * qg + pair) * D
                                  : stages + kFP * A + pair * D) + half * Dh + lane;
        const size_t estride = whole ? (size_t)kFP * D : (size_t)g.stage_floats;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float pw = ev[i] == -CUDART_INF_F ? 0.0f : __expf(ev[i] - m_run);
          s_run += pw;
          if (ev[i] != -CUDART_INF_F) {
            const float *er = er0 + i * estride;
#pragma unroll
            for (int j = 0; j < DPL; ++j)
              if (dmask & (1u << j)) acc[j] = fmaf(pw, er[32 * j], acc[j]);
          }
        }
      } else {
      // (2) scaled energies of the group's frames, running maximum
      float mg = m_run;
      for (int i = 0; i < gsz; ++i) {
        const int tl = kFP * (qg + i) + pair;
        if (tl < tloc) {
          const float e = p.scaling * ((epart[2 * tl] + epart[2 * tl + 1]) + gb);
          if (half == 0 && lane == 0) e_s[tl] = e;
          mg = fmaxf(mg, e);
        }
      }
      if (mg > m_run) {
        const float sc = __expf(m_run - mg);   // exp(-inf) = 0 for the first group
        s_run *= sc;
#pragma unroll
        for (int j = 0; j < DPL; ++j) acc[j] *= sc;
        m_run = mg;
      }
      // (3) un-normalised softmax weights and context
#pragma unroll 2
      for (int i = 0; i < gsz; ++i) {
        const int tl = kFP * (qg + i) + pair;
        if (tl < tloc) {
          const float e = p.scaling * ((epart[2 * tl] + epart[2 * tl + 1]) + gb);
          const float pw = __expf(e - m_run);
          s_run += pw;
          const float *er = (whole ? stages + (size_t)g.tloc_max * A + (size_t)tl * D
                                   : stages + (size_t)i * g.stage_floats + kFP * A + pair * D) + half * Dh + lane;
          if (dmask == (1u << DPL) - 1u) {   // every lane owns DPL channels (D == 64*DPL): no per-channel predicate
#pragma unroll
            for (int j = 0; j < DPL; ++j) acc[j] = fmaf(pw, er[32 * j], acc[j]);
          } else {
#pragma unroll
            for (int j = 0; j < DPL; ++j)
              if (dmask & (1u << j)) acc[j] = fmaf(pw, er[32 * j], acc[j]);
          }
        }
      }
      }
      if (qg + g.ns < nch) {   // ring shorter than the frame range (long utterances): refill behind a CTA barrier
        __syncthreads();
        if (tid == 0) {
          const int nxt = min(g.ns, nch - (qg + g.ns));
          for (int i = 0; i < nxt; ++i) issue(qg + g.ns + i);
        }
      }
    }
    if (lane == 0) { wstat[2 * warp] = m_run; wstat[2 * warp + 1] = s_run; }
  }
  __syncthreads();  // #4: ring drained, per-warp statistics published

  // ---- CTA combine (deterministic order), then push to the cluster
  float Mc = -CUDART_INF_F;
#pragma unroll
  for (int w2 = 0; w2 < kFW; ++w2) Mc = fmaxf(Mc, wstat[2 * w2]);
  {
    const float sc = m_run == -CUDART_INF_F ? 0.0f : __expf(m_run - Mc);
#pragma unroll
    for (int j = 0; j < DPL; ++j)
      if (lane + 32 * j < Dh && half * Dh + lane + 32 * j < D) cred[pair * Dp + half * Dh + lane + 32 * j] = acc[j] * sc;
  }
  __syncthreads();  // #5
  for (int d = tid; d < D; d += NT) {
    float sum = 0.0f;
#pragma unroll
    for (int pr = 0; pr < kFP; ++pr) sum += cred[pr * Dp + d];
    st_async_f32(dsmem_addr(cbuf + rank * Dp + d, 0u), sum, dsmem_addr(xbar, 0u));
  }
  if (tid < CL) {
    float sc = 0.0f;
#pragma unroll
    for (int pr = 0; pr < kFP; ++pr) {
      const float mw = wstat[4 * pr];
      if (mw != -CUDART_INF_F) sc += wstat[4 * pr + 1] * __expf(mw - Mc);
    }
    st_async_f32(dsmem_addr(xch + 2 * rank, (uint32_t)tid), Mc, dsmem_addr(xbar, (uint32_t)tid));
    st_async_f32(dsmem_addr(xch + 2 * rank + 1, (uint32_t)tid), sc, dsmem_addr(xbar, (uint32_t)tid));
  }
  mbar_wait(xbar, 0);   // every rank's (max, sum) -- and on rank 0 every partial context -- has landed here
  float M = -CUDART_INF_F;
  for (int r = 0; r < CL; ++r) M = fmaxf(M, xch[2 * r]);
  float S = 0.0f;
  for (int r = 0; r < CL; ++r)
    if (xch[2 * r] != -CUDART_INF_F) S += xch[2 * r + 1] * __expf(xch[2 * r] - M);
  const float inv = 1.0f / S;
  for (int tl = tid; tl < tloc; tl += NT) p.w[(size_t)b * Th + t0 + tl] = __expf(e_s[tl] - M) * inv;
  if (rank == 0) {
    for (int d = tid; d < D; d += NT) {
      float sum = 0.0f;
      for (int r = 0; r < CL; ++r)
        if (xch[2 * r] != -CUDART_INF_F) sum += cbuf[r * Dp + d] * __expf(xch[2 * r] - M);
      p.c[(size_t)b * D + d] = sum * inv;
    }
  }
  // no trailing cluster barrier: a CTA leaves only after everything addressed to it has landed (xbar), and it
  // never reads remote shared memory
}

// ------------------------------------------------------------------------------------------------
// backward (v3).  One cluster per utterance, CTA `rank` owns frames [t0,t1).
//
//   shared memory : the saved activations x = tanh(.) of ALL the CTA's frames (fetched by bulk copies in 8-frame
//                   chunks, each on its own mbarrier) stay resident; d pre is formed IN PLACE and handed back to the
//                   TMA unit chunk by chunk (cp.reduce.async.bulk.add.f32: the SM never reads d_pre).  enc_h streams
//                   through a small ring (it is only needed for dwt[t] = dw[t] + enc_h[t].dc).
//   pass 1        : warp per frame, dwt[t]; softmax backward needs sum_t w[t] dwt[t] over the whole utterance:
//                   every CTA pushes its partial sum to its peers (st.async + mbarrier, no cluster barrier)
//   pass 2        : warp pair per frame, lane <-> attention channel: dt = de g (1 - x^2) -> d pre (in place),
//                   d dec_proj, d gvec, d conv (16-value butterfly reduction); no CTA barrier inside the loop
//   post pass     : dW_att = dt^T conv straight from the resident tile; d conv / d dec_proj partials exchanged over
//                   DSMEM; d att_prev (transposed conv), dW_conv, and d dec_z = d dec_proj W_dec (split over ranks)
//   parameter grads: accumulated WITHOUT atomics into this CTA's private slot of `acc_slots` (plain read-modify-write,
//                   L2 resident across the decoder loop); re2e_attloc_acc_reduce sums the slots once per loop.
// ------------------------------------------------------------------------------------------------
constexpr int kBP = 8;                  // warp pairs = frames per activation chunk
constexpr int kBW = 2 * kBP;            // warps
constexpr int kBT = kBW * 32;
constexpr int kMaxXChunks = 16;         // tloc_max <= 128 frames per CTA
constexpr int kMaxEStages = 8;

template <int APL, int CP, int DPL2>
__global__ void __launch_bounds__(kBT, 1) attloc_bwd_kernel(const AttBwdParams p) {
  constexpr int NT = kBT;
  constexpr int WP = CP + 1;
  constexpr int CPP = (CP + 3) & ~3;
  extern __shared__ __align__(128) unsigned char smraw[];
  const AttGeom g = p.g;
  const int C = CP == 10 ? 10 : p.C;
  const int Th = p.Th, D = p.D, A = p.A, K = p.K, Z = p.Z, filts = (p.K - 1) / 2;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, half = warp & 1, pair = warp >> 1;
  const int CL = (int)cluster_nctarank(), rank = (int)cluster_ctarank();
  const int b = blockIdx.x / CL;
  const int t0 = min(Th, rank * g.tloc_max), t1 = min(Th, t0 + g.tloc_max), tloc = t1 - t0;
  const int nchx = (tloc + kBP - 1) / kBP;       // activation chunks (8 frames)
  const int nche = (tloc + kBW - 1) / kBW;       // enc_h chunks (16 frames)

  uint64_t *full_x = reinterpret_cast<uint64_t *>(smraw);   // [kMaxXChunks]
  uint64_t *done_x = full_x + kMaxXChunks;                  // [1] every warp finished forming d pre in place
  uint64_t *full_e = done_x + kMaxXChunks;                  // [kMaxEStages]
  uint64_t *xbar1 = full_e + kMaxEStages;                   // sum_t w dwt partials of every rank
  uint64_t *xbar2 = xbar1 + 1;                              // d conv of every frame + d dec_proj partials of every rank
  float *xs = reinterpret_cast<float *>(smraw + 512);       // tloc_max*A   activations, then d pre in place
  float *ering = xs + (size_t)g.tloc_max * A;               // ns * kBW*D   enc_h ring; reused after pass 1:
  float *ddp_w = ering;                                     //   kBW*(A/2)  per-warp d dec_proj partials
  float *dgv_w = ddp_w + kBW * (A / 2);                     //   kBW*(A/2)  per-warp d gvec partials
  float *scr = dgv_w + kBW * (A / 2);                       //   kKQ*CP*tloc_max  d att_prev partials
  float *dzp = scr + kKQ * CP * g.tloc_max;                 //   kBW*round4(ceil(Z/CL))  d dec_z partials
  float *app = ering + (size_t)g.ring_floats;               // App      padded att_prev row
  float *wc_s = app + g.App;                                // CKp
  float *watt_s = wc_s + g.CKp;                             // A*WP
  float *conv_s = watt_s + A * WP;                          // tloc_max*CPP
  float *w_s = conv_s + g.tloc_max * CPP;                   // round4(tloc_max)
  float *dwt_s = w_s + round4(g.tloc_max);                  // round4(tloc_max)
  float *de_s = dwt_s + round4(g.tloc_max);                 // round4(tloc_max)
  float *dcv_p = de_s + round4(g.tloc_max);                 // 2*tloc_max*16   per-half d conv partials
  float *dcvT = dcv_p + 2 * g.tloc_max * 16;                // CP*App  channel-major zero padded d conv of ALL frames
  float *ddp_x = dcvT + CP * g.App;                         // CL*A    d dec_proj partials of every rank
  float *ddp_t = ddp_x + CL * A;                            // A       d dec_proj total
  float *xch = ddp_t + A;                                   // 16      sum_t w dwt partials of every rank
  float *slot = p.acc_slots + (size_t)blockIdx.x * p.slot_stride;   // [dW_att A*C | dW_conv C*K | dgvec A | dgvec_b 1]

  const bool whole_e = g.ns >= nche;   // the enc_h ring holds the CTA's whole frame range
  auto issue_e = [&](int q) {
    const int st = q % g.ns;
    const int r0 = t0 + kBW * q;
    const int rows = min(kBW, t1 - r0);
    mbar_expect_tx(&full_e[st], (uint32_t)rows * D * 4u);
    bulk_g2s(ering + (size_t)st * g.stage_floats, p.enc + ((size_t)b * Th + r0) * D, (uint32_t)rows * D * 4u, &full_e[st]);
  };
  if (tid == 0) {
    mbar_init(&full_x[0], 1);
    mbar_init(done_x, kBW);
    for (int i = 0; i < g.ns; ++i) mbar_init(&full_e[i], 1);
    mbar_init(xbar1, 1);
    mbar_init(xbar2, 1);
    mbar_fence_init();
    mbar_expect_tx(xbar1, (uint32_t)CL * 4u);
    mbar_expect_tx(xbar2, (uint32_t)Th * (uint32_t)C * 4u + (uint32_t)CL * (uint32_t)A * 4u);
  }
  cluster_arrive_relaxed();   // "this CTA is running and its barriers exist"

  // ---- prologue loads, batched in registers: one L2 round trip.  Everything read here was written by the
  //      FORWARD pass (or is a parameter), so it is issued before the PDL boundary below.
  float gv[APL];
#pragma unroll
  for (int j = 0; j < APL; ++j) gv[j] = __ldg(p.gvec + half * (A / 2) + lane + 32 * j);
  {
    constexpr int IA = 2, IC = 4, IW = 8, IV = 2;
    float va[IA], vc[IC], vw[IW], vv[IV], vws;
#pragma unroll
    for (int u = 0; u < IA; ++u) {
      const int i = tid + u * NT, t = i - filts;
      va[u] = (i < g.App && t >= 0 && t < Th) ? __ldcg(p.att_prev + (size_t)b * Th + t) : 0.0f;
    }
#pragma unroll
    for (int u = 0; u < IC; ++u) {
      const int i = tid + u * NT;
      vc[u] = i < C * K ? __ldg(p.W_conv + i) : 0.0f;
    }
#pragma unroll
    for (int u = 0; u < IW; ++u) {
      const int i = tid + u * NT;
      vw[u] = i < A * C ? __ldg(p.W_att + i) : 0.0f;
    }
#pragma unroll
    for (int u = 0; u < IV; ++u) {
      const int i = tid + u * NT;
      vv[u] = i < tloc * C ? __ldg(p.conv + ((size_t)b * Th + t0) * C + i) : 0.0f;
    }
    vws = tid < tloc ? __ldg(p.w + (size_t)b * Th + t0 + tid) : 0.0f;
    // the bulk copies (enc_h ring first: pass 1 needs it first; then every activation chunk) are issued by one
    // lane AFTER its warp's prologue loads are in flight
    if (tid == 0 && tloc > 0) {
      // one bulk copy for the enc_h range (when the ring holds it all) and ONE for the activations: the issuing lane
      // is on the prologue's critical path (everyone waits for it at barrier #1)
      if (whole_e) {
        mbar_expect_tx(&full_e[0], (uint32_t)tloc * D * 4u);
        bulk_g2s(ering, p.enc + ((size_t)b * Th + t0) * D, (uint32_t)tloc * D * 4u, &full_e[0]);
      } else {
        const int first = nche < g.ns ? nche : g.ns;
        for (int q = 0; q < first; ++q) issue_e(q);
      }
      mbar_expect_tx(&full_x[0], (uint32_t)tloc * A * 4u);
      bulk_g2s(xs, p.xsave + ((size_t)b * Th + t0) * A, (uint32_t)tloc * A * 4u, &full_x[0]);
    }
#pragma unroll
    for (int u = 0; u < IA; ++u)
      if (tid + u * NT < g.App) app[tid + u * NT] = va[u];
#pragma unroll
    for (int u = 0; u < IC; ++u)
      if (tid + u * NT < C * K) wc_s[tid + u * NT] = vc[u];
#pragma unroll
    for (int u = 0; u < IW; ++u) {
      const int i = tid + u * NT;
      if (i < A * C) { const int a = i / C; watt_s[a * WP + (i - a * C)] = vw[u]; }
    }
#pragma unroll
    for (int u = 0; u < IV; ++u) {
      const int i = tid + u * NT;
      if (i < tloc * C) { const int tl = i / C; conv_s[tl * CPP + (i - tl * C)] = vv[u]; }
    }
    if (tid < tloc) w_s[tid] = vws;
    for (int i = tid + IA * NT; i < g.App; i += NT) {
      const int t = i - filts;
      app[i] = (t >= 0 && t < Th) ? __ldcg(p.att_prev + (size_t)b * Th + t) : 0.0f;
    }
    for (int i = tid + IC * NT; i < C * K; i += NT) wc_s[i] = __ldg(p.W_conv + i);
    for (int i = tid + IW * NT; i < A * C; i += NT) { const int a = i / C; watt_s[a * WP + (i - a * C)] = __ldg(p.W_att + i); }
    for (int i = tid + IV * NT; i < tloc * C; i += NT) {
      const int tl = i / C;
      conv_s[tl * CPP + (i - tl * C)] = __ldg(p.conv + ((size_t)b * Th + t0) * C + i);
    }
    for (int i = tid + NT; i < tloc; i += NT) w_s[i] = __ldg(p.w + (size_t)b * Th + t0 + i);
    // zero the pads of the channel-major d conv rows (the frames themselves are pushed by the cluster)
    const int padn = g.App - Th;
    for (int i = tid; i < CP * padn; i += NT) {
      const int c = i / padn, o = i - c * padn;
      dcvT[c * g.App + (o < filts ? o : Th + o)] = 0.0f;
    }
    if (CPP > CP)
      for (int i = tid; i < tloc * (CPP - CP); i += NT) conv_s[(i / (CPP - CP)) * CPP + CP + i % (CPP - CP)] = 0.0f;
  }
  // ---- PDL boundary: the incoming gradients (dc, dw = the next step's d att_prev) are produced by the predecessor
  //      grid(s); every global write of this kernel (d pre reduce-add, accumulator slots, outputs) comes later
  pdl_wait();
  pdl_launch_dependents();
  float dcr[DPL2];
#pragma unroll
  for (int j = 0; j < DPL2; ++j) dcr[j] = (p.dc && lane + 32 * j < D) ? __ldcg(p.dc + (size_t)b * D + lane + 32 * j) : 0.0f;
  for (int i = tid; i < tloc; i += NT) dwt_s[i] = p.dw ? __ldcg(p.dw + (size_t)b * Th + t0 + i) : 0.0f;
  __syncthreads();  // #1

  // ---- pass 1: dwt[t] = dw[t] + enc_h[t,:] . dc   (warp per frame, lane <-> d)
  {
    int st = 0;
    uint32_t ph = 0;
    for (int q = 0; q < nche; ++q) {
      if (!whole_e) mbar_wait(&full_e[st], ph);
      else if (q == 0) mbar_wait(&full_e[0], 0);
      const int tl = kBW * q + warp;
      if (tl < tloc) {
        const float *row = ering + (size_t)st * g.stage_floats + warp * D + lane;
        float dot = 0.0f;
#pragma unroll
        for (int j = 0; j < DPL2; ++j)
          if (lane + 32 * j < D) dot = fmaf(dcr[j], row[32 * j], dot);
        dot = warp_sum(dot);
        if (lane == 0) dwt_s[tl] += dot;
      }
      if (g.ns < nche) {   // ring shorter than the frame range (long utterances): refill behind a CTA barrier
        __syncthreads();
        if (tid == 0 && q + g.ns < nche) issue_e(q + g.ns);
      }
      if (++st == g.ns) { st = 0; ph ^= 1u; }
    }
  }
  // W_att rows of this lane's channels -> registers, as pairs along c (packed FFMA2 in pass 2)
  constexpr int CH2 = (CP + 1) / 2;
  float2 WattC[APL][CH2];
#pragma unroll
  for (int j = 0; j < APL; ++j) {
    const int a = half * (A / 2) + lane + 32 * j;
#pragma unroll
    for (int c2 = 0; c2 < CH2; ++c2)
      WattC[j][c2] = make_float2(2 * c2 < C ? watt_s[a * WP + 2 * c2] : 0.0f, 2 * c2 + 1 < C ? watt_s[a * WP + 2 * c2 + 1] : 0.0f);
  }
  __syncthreads();  // #2: dwt complete; the enc ring is free
  cluster_wait();   // peers are resident: remote stores may start
  if (warp == 0) {
    float s1 = 0.0f;
    for (int tl = lane; tl < tloc; tl += 32) s1 = fmaf(w_s[tl], dwt_s[tl], s1);
    s1 = warp_sum(s1);
    if (lane < CL) st_async_f32(dsmem_addr(xch + rank, (uint32_t)lane), s1, dsmem_addr(xbar1, (uint32_t)lane));
  }
  mbar_wait(xbar1, 0);
  float Stot = 0.0f;
  for (int r = 0; r < CL; ++r) Stot += xch[r];
  for (int tl = tid; tl < tloc; tl += NT) de_s[tl] = p.scaling * w_s[tl] * (dwt_s[tl] - Stot);
  __syncthreads();  // #3

  // ---- pass 2: through tanh.  pair <-> frame, lane <-> channel
  float dgv[APL], ddp[APL];
#pragma unroll
  for (int j = 0; j < APL; ++j) { dgv[j] = 0.0f; ddp[j] = 0.0f; }
  {
    const int aoff = half * (A / 2) + lane;
    if (tloc > 0) mbar_wait(&full_x[0], 0);   // landed long ago (issued in the prologue)
    // no barrier inside the frame loop: the 16-value butterfly of one frame overlaps the FMAs of the next
#pragma unroll 2
    for (int q = 0; q < nchx; ++q) {
      const int tl = kBP * q + pair;
      if (tl < tloc) {
        const float de = de_s[tl];
        float2 dcv2[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) dcv2[c] = make_float2(0.0f, 0.0f);
        float *row = xs + (size_t)tl * A + aoff;
#pragma unroll
        for (int j = 0; j < APL; ++j) {
          const float x = row[32 * j];
          dgv[j] = fmaf(de, x, dgv[j]);
          const float dt = de * gv[j] * (1.0f - x * x);
          ddp[j] += dt;
          row[32 * j] = dt;  // d pre, in place
          const float2 dt2 = make_float2(dt, dt);
#pragma unroll
          for (int c2 = 0; c2 < CH2; ++c2) dcv2[c2] = __ffma2_rn(dt2, WattC[j][c2], dcv2[c2]);
        }
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
    fence_proxy_async_smem();   // this thread's in-place writes -> visible to the bulk (async proxy) reads
    __syncwarp();
    if (lane == 0) mbar_arrive1(done_x);
    if (tid == 0) {             // hand the d pre tile (formed in place) to the TMA unit: d_pre[b, t0:t1, :] (+)= tile
      mbar_wait(done_x, 0);
      float *dst = p.d_pre + ((size_t)b * Th + t0) * A;
      const uint32_t total = (uint32_t)tloc * A * 4u;
      for (uint32_t o = 0; o < total; o += 32768u) {
        const uint32_t nb = total - o < 32768u ? total - o : 32768u;
        if (p.accumulate_pre) bulk_red_add_s2g(reinterpret_cast<char *>(dst) + o, reinterpret_cast<char *>(xs) + o, nb);
        else bulk_s2g(reinterpret_cast<char *>(dst) + o, reinterpret_cast<char *>(xs) + o, nb);
      }
      bulk_commit();
    }
#pragma unroll
    for (int j = 0; j < APL; ++j) {
      ddp_w[warp * (A / 2) + lane + 32 * j] = ddp[j];
      dgv_w[warp * (A / 2) + lane + 32 * j] = dgv[j];
    }
  }
  __syncthreads();  // #4: all d pre tiles written, per-warp partials published

  // ---- d dec_z[z] = sum_a d dec_proj[a] W_dec[a,z] for this rank's slice of z, from the TRANSPOSED weight
  //      W_decT (Z x A, built once per decoder loop): row z is one contiguous, 16 B aligned run of A floats, so the
  //      slice is read with fully coalesced 128-bit loads (15 per thread at the default shape instead of 60 scalar
  //      ones), warp <-> z rows, lane <-> quad of a.  The loads are issued HERE -- they do not depend on the cluster
  //      exchange -- and consumed after it (post pass B), so their L2 latency hides behind post pass A.
  constexpr int AQ = 16 * APL;                      // float4 per W_decT row (A / 4)
  constexpr int MQ = (AQ + 31) / 32;                // quads per lane
  constexpr int ZR = APL <= 5 ? 5 : 3;              // z rows per warp held in registers per pass
  const int zc = (Z + CL - 1) / CL, z_begin = rank * zc, z_n = max(0, min(zc, Z - z_begin));
  float4 wz[ZR][MQ];
  auto load_wz = [&](int zb) {
#pragma unroll
    for (int r = 0; r < ZR; ++r) {
      const int zi = zb + warp + kBW * r;
      const float4 *wr = reinterpret_cast<const float4 *>(p.W_decT + (size_t)(z_begin + min(zi, max(z_n - 1, 0))) * A);
#pragma unroll
      for (int m = 0; m < MQ; ++m) {
        const int j = lane + 32 * m;
        wz[r][m] = (zi < z_n && j < AQ) ? __ldg(wr + j) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
  };
  if (p.d_dec_z) load_wz(0);

  // ---- post pass A (needs nothing from the other CTAs)
  // d conv of this CTA's frames -> every CTA of the cluster (channel-major, padded)
  for (int item = tid; item < tloc * C; item += NT) {
    const int c = item / tloc, tl = item - c * tloc;
    const float v = dcv_p[tl * 16 + c] + dcv_p[(g.tloc_max + tl) * 16 + c];
    for (int r = 0; r < CL; ++r)
      st_async_f32(dsmem_addr(dcvT + c * g.App + filts + t0 + tl, (uint32_t)r), v, dsmem_addr(xbar2, (uint32_t)r));
  }
  // d dec_proj / d gvec of this CTA (fixed summation order), d dec_proj partial -> every CTA
  for (int a = tid; a < A; a += NT) {
    const int h = a >= A / 2 ? 1 : 0, ai = a - h * (A / 2);
    const float sg0 = slot[A * C + C * K + a];   // consumed only after the pushes: its L2 latency is off the exchange path
    float sd = 0.0f, sg = 0.0f;
#pragma unroll
    for (int pr = 0; pr < kBP; ++pr) {
      sd += ddp_w[(2 * pr + h) * (A / 2) + ai];
      sg += dgv_w[(2 * pr + h) * (A / 2) + ai];
    }
    for (int r = 0; r < CL; ++r)
      st_async_f32(dsmem_addr(ddp_x + rank * A + a, (uint32_t)r), sd, dsmem_addr(xbar2, (uint32_t)r));
    slot[A * C + C * K + a] = sg0 + sg;
  }
  if (warp == kBW - 1) {   // d gvec.bias = sum_t de[t]  (analytically zero over the utterance; kept for fidelity)
    float s2 = 0.0f;
    for (int tl = lane; tl < tloc; tl += 32) s2 += de_s[tl];
    s2 = warp_sum(s2);
    if (lane == 0 && tloc > 0) slot[A * C + C * K + A] += s2;
  }
  // The two parameter gradients that only need THIS CTA's frames run side by side on disjoint sets of warps:
  //   threads [0, A)       : dW_att[a,c] += sum_t d pre[t,a] conv[t,c]   straight from the resident tile (thread <-> a)
  //   threads [A, NT)      : dW_conv[c,k] += sum_{t in mine} dconv[t,c] att_prev[t + k - filts]  (6 taps per item)
  if (tid < A) {
    const int a = tid;
    float acc[CP];    // starts from the slot's running total (loads overlap the frame loop)
#pragma unroll
    for (int c = 0; c < CP; ++c) acc[c] = c < C ? slot[a * C + c] : 0.0f;
#pragma unroll 5
    for (int tl = 0; tl < tloc; ++tl) {
      const float dt = xs[(size_t)tl * A + a];
#pragma unroll
      for (int c4 = 0; c4 < CPP; c4 += 4) {
        const float4 t4 = *reinterpret_cast<const float4 *>(conv_s + tl * CPP + c4);
        if (c4 < CP) acc[c4] = fmaf(dt, t4.x, acc[c4]);
        if (c4 + 1 < CP) acc[c4 + 1] = fmaf(dt, t4.y, acc[c4 + 1]);
        if (c4 + 2 < CP) acc[c4 + 2] = fmaf(dt, t4.z, acc[c4 + 2]);
        if (c4 + 3 < CP) acc[c4 + 3] = fmaf(dt, t4.w, acc[c4 + 3]);
      }
    }
#pragma unroll
    for (int c = 0; c < CP; ++c)
      if (c < C) slot[a * C + c] = acc[c];
  }
  {
    constexpr int KG = 12;   // taps per item: C * ceil(K / 12) = 170 items <= the 192 threads left beside dW_att
    const int nkg = (K + KG - 1) / KG;
    const int first = A < NT ? A : 0, nthr = A < NT ? NT - A : NT;   // A >= NT (A = 512): everyone, after dW_att
    if (tid >= first) {
      for (int item = tid - first; item < C * nkg; item += nthr) {
        const int kg = item % nkg, c = item / nkg;
        const int kb = kg * KG;
        const float *ar = app + kb;                  // att_prev[t + k - filts] = app[t + k]
        float acc6[KG];   // starts from the slot's running total: the loads overlap the tap loop
#pragma unroll
        for (int i = 0; i < KG; ++i) acc6[i] = kb + i < K ? slot[A * C + c * K + kb + i] : 0.0f;
        float x[KG];
#pragma unroll
        for (int i = 0; i < KG - 1; ++i) x[i] = ar[t0 + i];
#pragma unroll 12   // = KG: the register window rotates back onto itself, no moves
        for (int tl = 0; tl < tloc; ++tl) {
          x[KG - 1] = ar[t0 + tl + KG - 1];
          const float dv = dcv_p[tl * 16 + c] + dcv_p[(g.tloc_max + tl) * 16 + c];   // d conv of MY frame tl
#pragma unroll
          for (int i = 0; i < KG; ++i) acc6[i] = fmaf(dv, x[i], acc6[i]);
#pragma unroll
          for (int i = 0; i < KG - 1; ++i) x[i] = x[i + 1];
        }
#pragma unroll
        for (int i = 0; i < KG; ++i)
          if (kb + i < K) slot[A * C + c * K + kb + i] = acc6[i];
      }
    }
  }
  mbar_wait(xbar2, 0);
  for (int a = tid; a < A; a += NT) {
    float sd = 0.0f;
    for (int r = 0; r < CL; ++r) sd += ddp_x[r * A + a];
    ddp_t[a] = sd;
    if (rank == 0) p.d_decproj[(size_t)b * A + a] = sd;
  }
  __syncthreads();  // #5 (also: scr aliases the per-warp partials read above)

  // ---- post pass B
  // d dec_z from the prefetched W_decT rows: one dot product of length A per z row, reduced inside the warp
  if (p.d_dec_z) {
    for (int zb = 0; zb < z_n; zb += kBW * ZR) {
      if (zb > 0) load_wz(zb);
#pragma unroll
      for (int r = 0; r < ZR; ++r) {
        float s0 = 0.0f;
#pragma unroll
        for (int m = 0; m < MQ; ++m) {
          const int j = lane + 32 * m;
          if (j < AQ) {
            const float4 d4 = *reinterpret_cast<const float4 *>(ddp_t + 4 * j);
            s0 = fmaf(d4.x, wz[r][m].x, fmaf(d4.y, wz[r][m].y, fmaf(d4.z, wz[r][m].z, fmaf(d4.w, wz[r][m].w, s0))));
          }
        }
        s0 = warp_sum(s0);
        const int zi = zb + warp + kBW * r;
        if (lane == 0 && zi < z_n) p.d_dec_z[(size_t)b * Z + z_begin + zi] = s0;
      }
    }
  }
  // d att_prev[s] = sum_c sum_k Wc[c,k] * dconv[s - k + filts, c]   (sliding window, 5 outputs/thread)
  if (p.d_att_prev) {
    const int nsg = (tloc + kTG - 1) / kTG;
    const int Kq = (K + kKQ - 1) / kKQ;
    const int nitems = nsg * C * kKQ;
    for (int item = tid; item < nitems; item += NT) {
      const int sg = item % nsg, rest = item / nsg, c = rest % C, kq = rest / C;
      const int k0 = kq * Kq, k1 = min(K, k0 + Kq);
      const float *wr = wc_s + c * K;
      // padded index of dconv[s - k + filts] is (s - k + 2*filts); outputs s = s0 .. s0+4
      const float *dr = dcvT + c * g.App + (t0 + kTG * sg) + 2 * filts;
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
    __syncthreads();  // #6
    for (int tl = tid; tl < tloc; tl += NT) {
      float sum = 0.0f;
      for (int i = 0; i < kKQ * C; ++i) sum += scr[(size_t)i * g.tloc_max + tl];
      p.d_att_prev[(size_t)b * Th + t0 + tl] = sum;
    }
  }
  if (tid == 0) bulk_wait<0>();  // all d_pre traffic of this CTA has left shared memory / landed
}

// out[i] = sum_s slots[s*stride + i]   -- once per decoder loop, fixed summation order.
// block = 32 outputs x 8 slot groups; group g sums slots g, g+8, ...; the 8 partials are combined through smem.
__global__ void __launch_bounds__(256)
acc_reduce_kernel(const float *__restrict__ slots, int n_slots, int stride, int n, float *__restrict__ out) {
  __shared__ float part[8][33];
  const int lane = threadIdx.x & 31, grp = threadIdx.x >> 5;
  const int i = blockIdx.x * 32 + lane;
  float s0 = 0.f, s1 = 0.f;
  if (i < n) {
    int s = grp;
    for (; s + 8 < n_slots; s += 16) {
      s0 += __ldg(slots + (size_t)s * stride + i);
      s1 += __ldg(slots + (size_t)(s + 8) * stride + i);
    }
    if (s < n_slots) s0 += __ldg(slots + (size_t)s * stride + i);
  }
  part[grp][lane] = s0 + s1;
  __syncthreads();
  if (grp == 0 && i < n) {
    float t = 0.f;
#pragma unroll
    for (int g2 = 0; g2 < 8; ++g2) t += part[g2][lane];
    out[i] = t;
  }
}

// ------------------------------------------------------------------------------------------------
// small helpers
// ------------------------------------------------------------------------------------------------
__global__ void init_att_kernel(const int32_t *__restrict__ hlens, float *__restrict__ att, int B, int Th) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * Th) return;
  const int b = i / Th, t = i - b * Th;
  const int l = __ldg(hlens + b);
  att[i] = (t < l) ? 1.0f / (float)l : 0.0f;
}

// d_enc_h[b,t,:] (+)= sum_i w_all[i,b,t] * dc_all[i,b,:]   (rank-#steps update, once per decoder loop)
// CTA <-> (utterance, tile of tt frames); the utterance's dc rows [steps][D] and the tile's weights [steps][tt]
// are staged in shared memory; thread <-> (d, group of 8 frames): w broadcast, dc conflict free, 8 FMAs per 2 LDS.
constexpr int kEGThreads = 512;
__global__ void __launch_bounds__(kEGThreads)
enc_grad_kernel(const float *__restrict__ w_all, const float *__restrict__ dc_all,
                float *__restrict__ d_enc, int steps, int B, int Th, int D, int tt, int accumulate) {
  extern __shared__ __align__(16) float smem[];
  float *dc_s = smem;                     // [steps][D]
  float *w_s = smem + (size_t)round4(steps * D);  // [steps][tt]   (tt % 8 == 0)
  const int tiles = (Th + tt - 1) / tt;
  const int b = blockIdx.x / tiles, t0 = (blockIdx.x - b * tiles) * tt;
  const int rows = min(tt, Th - t0);
  const int tid = threadIdx.x;
  if ((D & 3) == 0) {
    const int D4 = D >> 2;
    for (int i = tid; i < steps * D4; i += kEGThreads) {
      const int s = i / D4, d4 = i - s * D4;
      reinterpret_cast<float4 *>(dc_s)[i] = __ldg(reinterpret_cast<const float4 *>(dc_all + ((size_t)s * B + b) * D) + d4);
    }
  } else {
    for (int i = tid; i < steps * D; i += kEGThreads) {
      const int s = i / D, d = i - s * D;
      dc_s[i] = __ldg(dc_all + ((size_t)s * B + b) * D + d);
    }
  }
  for (int i = tid; i < steps * tt; i += kEGThreads) {
    const int s = i / tt, r = i - s * tt;
    w_s[i] = r < rows ? __ldg(w_all + ((size_t)s * B + b) * Th + t0 + r) : 0.0f;
  }
  __syncthreads();
  const int ngr = (rows + 7) / 8;
  for (int item = tid; item < D * ngr; item += kEGThreads) {
    const int d = item % D, gr = item / D;
    float a[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int r = gr * 8 + i;
      a[i] = (accumulate && r < rows) ? d_enc[((size_t)b * Th + t0 + r) * D + d] : 0.0f;   // in flight during the loop
    }
#pragma unroll 4
    for (int s = 0; s < steps; ++s) {
      const float dv = dc_s[s * D + d];
      const float4 w0 = *reinterpret_cast<const float4 *>(w_s + s * tt + gr * 8);
      const float4 w1 = *reinterpret_cast<const float4 *>(w_s + s * tt + gr * 8 + 4);
      a[0] = fmaf(w0.x, dv, a[0]); a[1] = fmaf(w0.y, dv, a[1]); a[2] = fmaf(w0.z, dv, a[2]); a[3] = fmaf(w0.w, dv, a[3]);
      a[4] = fmaf(w1.x, dv, a[4]); a[5] = fmaf(w1.y, dv, a[5]); a[6] = fmaf(w1.z, dv, a[6]); a[7] = fmaf(w1.w, dv, a[7]);
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int r = gr * 8 + i;
      if (r < rows) d_enc[((size_t)b * Th + t0 + r) * D + d] = a[i];
    }
  }
}

// forward (v3) geometry: stage = kFP frames of (pre | enc); the ring holds the whole frame range when it fits
// Clusters of 16 are non-portable: the pickers ask the device whether one fits at the chosen shared-memory size.  Every
// instantiation of a direction runs the same block (__launch_bounds__(threads, 1), dynamic shared memory only), so the
// default-dims instantiation stands for all of them.
inline bool pick_geom_fwd(int B, int Th, int D, int A, int Z, int C, int K, int CP, int &CL, AttGeom &g,
                          size_t &smem) {
  const int sms = num_sms();
  CL = 1;
  while (CL < 8 && B * CL * 2 <= sms) CL *= 2;
  while (CL > 1 && (Th + CL - 1) / CL < kFP) CL /= 2;  // tiny Th: do not over-split
  const int filts = (K - 1) / 2;
  g.stage_floats = kFP * (A + D);
  g.Thp = round4(Th);
  g.CKp = round4(C * K);
  g.App = round4(Th + 2 * filts + 8);
  const size_t budget = 224 * 1024;
  const size_t stage_bytes = sizeof(float) * (size_t)g.stage_floats;
  size_t fixed;
  for (;;) {
    g.tloc_max = (Th + CL - 1) / CL;
    g.nch = (g.tloc_max + kFP - 1) / kFP;
    // the last 16 floats once held the (max, sum) exchange, now in the header: kept so that no size changes
    fixed = 512 + sizeof(float) * ((size_t)g.App + g.CKp + (size_t)A * (CP + 1) + round4(Z) + A +
                                   (size_t)round4(kKQ * g.tloc_max * CP) + (size_t)g.tloc_max * round4(CP) +
                                   round4(g.tloc_max) + round4(2 * g.tloc_max) +
                                   2 * kFW + (size_t)fwd_rank_rows(CL) * round4(D) + 16);
    if (fixed + 2 * stage_bytes <= budget) break;
    // long utterances: the per-frame part of the fixed area shrinks with the CTA's frame range -- split further, up to
    // the non-portable cluster size of 16 (the grid runs in waves when B*CL CTAs exceed the SMs: clusters do not wait
    // for each other)
    if (CL >= 16) return false;
    CL *= 2;
  }
  int ns = (int)((budget - fixed) / stage_bytes);
  if (ns > g.nch) ns = g.nch;
  if (ns > kMaxStages) ns = kMaxStages;
  if (ns < 1) ns = 1;
  g.ns = ns;
  smem = fixed + ns * stage_bytes;
  return CL <= 8 || cluster_fits(reinterpret_cast<const void *>(attloc_fwd_kernel<5, 10, 5>), CL, kFT, smem);
}

// backward (v3) geometry: all activations of the CTA resident, enc_h through a ring of kBW-frame stages
inline bool pick_geom_bwd(int B, int Th, int D, int A, int Z, int C, int K, int CP, int &CL, AttGeom &g,
                          size_t &smem) {
  const int sms = num_sms();
  CL = 1;
  while (CL < 8 && B * CL * 2 <= sms) CL *= 2;
  while (CL > 1 && (Th + CL - 1) / CL < kBP) CL /= 2;
  const int filts = (K - 1) / 2;
  const int CPP = round4(CP);
  g.stage_floats = kBW * D;
  g.Thp = round4(Th);
  g.CKp = round4(C * K);
  g.App = round4(Th + 2 * filts + 8);
  for (;;) {
    g.tloc_max = (Th + CL - 1) / CL;
    g.nch = (g.tloc_max + kBW - 1) / kBW;
    const size_t alias_floats = (size_t)kBW * A + (size_t)kKQ * CP * g.tloc_max +
                                (size_t)kBW * round4((Z + CL - 1) / CL);
    const size_t fixed = 512 + sizeof(float) * ((size_t)g.tloc_max * A + (size_t)g.App + g.CKp + (size_t)A * (CP + 1) +
                                                (size_t)g.tloc_max * CPP + 3 * (size_t)round4(g.tloc_max) +
                                                2 * (size_t)g.tloc_max * 16 + (size_t)CP * g.App + (size_t)(CL + 1) * A + 16);
    const size_t budget = 224 * 1024;
    const size_t stage_bytes = sizeof(float) * (size_t)g.stage_floats;
    const size_t alias_bytes = sizeof(float) * ((alias_floats + 3) & ~(size_t)3);
    const size_t min_ring = stage_bytes > alias_bytes ? stage_bytes : alias_bytes;
    if (g.tloc_max <= kMaxXChunks * kBP && fixed + min_ring <= budget) {
      int ns = (int)((budget - fixed) / stage_bytes);
      if (ns > g.nch) ns = g.nch;
      if (ns > kMaxEStages) ns = kMaxEStages;
      if (ns < 1) ns = 1;
      g.ns = ns;
      size_t ring = (size_t)ns * stage_bytes;
      if (ring < alias_bytes) ring = alias_bytes;
      g.ring_floats = (int)(ring / sizeof(float));
      smem = fixed + ring;
      return CL <= 8 || cluster_fits(reinterpret_cast<const void *>(attloc_bwd_kernel<5, 10, 10>), CL, kBT, smem);
    }
    // long utterances: split further, up to the non-portable cluster size of 16.  Only the CTAs of one cluster need to
    // be co-resident (they synchronise through DSMEM and the cluster barrier; nothing is shared across clusters), so
    // the grid may run in waves when B*CL exceeds the SMs.
    if (CL >= 16) return false;
    CL *= 2;
  }
}

// the step kernels are launched with programmatic dependent launch: the grid may start its prologue while the
// previous kernel of the stream drains (see pdl_wait())
template <int APL, int CP>
int run_fwd(const AttFwdParams &prm, int CL, size_t smem, cudaStream_t st) {
  const dim3 grid((unsigned)(prm.B * CL));
  // encoder channels per lane: the common D == A case gets an exact instantiation, anything else the general one
  if (prm.D == prm.A) return launch_cluster(attloc_fwd_kernel<APL, CP, APL>, grid, dim3(kFT), smem, st, CL, true, prm);
  return launch_cluster(attloc_fwd_kernel<APL, CP, kDpl>, grid, dim3(kFT), smem, st, CL, true, prm);
}
template <int APL, int CP>
int run_bwd(const AttBwdParams &prm, int CL, size_t smem, cudaStream_t st) {
  const dim3 grid((unsigned)(prm.B * CL));
  if (prm.D == prm.A) return launch_cluster(attloc_bwd_kernel<APL, CP, 2 * APL>, grid, dim3(kBT), smem, st, CL, true, prm);
  return launch_cluster(attloc_bwd_kernel<APL, CP, 2 * kDpl>, grid, dim3(kBT), smem, st, CL, true, prm);
}

}  // namespace
}  // namespace re2e

using namespace re2e;

extern "C" int re2e_attloc_init_att(const int32_t *hlens, float *att_prev, int B, int Th, void *stream) {
  RE2E_CHECK_ARG(hlens && att_prev && B > 0 && Th > 0);
  init_att_kernel<<<(B * Th + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(hlens, att_prev, B, Th);
  count_launch();
  return launch_status();
}

extern "C" int re2e_attloc_step_fwd(const float *pre, const float *enc_h, const float *dec_z,
                                    const float *att_prev, const float *W_dec, const float *W_att,
                                    const float *W_conv, const float *gvec, const float *gvec_b,
                                    float scaling, float *c, float *w, float *dec_proj, float *conv,
                                    float *xsave, int B, int Th, int D, int A, int Z, int C, int K,
                                    void *stream) {
  RE2E_CHECK_ARG(pre && enc_h && att_prev && W_dec && W_att && W_conv && gvec && gvec_b && c && w);
  int rc = check_dims(B, Th, D, A, C, K);
  if (rc != RE2E_OK) return rc;
  RE2E_CHECK_ARG(Z > 0 && aligned16(pre) && aligned16(enc_h));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int CP = C == 10 ? 10 : 16;
  AttFwdParams prm;
  prm.pre = pre; prm.enc = enc_h; prm.att_prev = att_prev; prm.dec_z = dec_z; prm.W_dec = W_dec; prm.W_att = W_att;
  prm.W_conv = W_conv; prm.gvec = gvec; prm.gvec_b = gvec_b; prm.scaling = scaling; prm.c = c; prm.w = w;
  prm.dec_proj = dec_proj; prm.conv = conv; prm.xsave = xsave;
  prm.B = B; prm.Th = Th; prm.D = D; prm.A = A; prm.Z = Z; prm.C = C; prm.K = K;
  int CL;
  size_t smem;
  if (!pick_geom_fwd(B, Th, D, A, Z, C, K, CP, CL, prm.g, smem)) return RE2E_E_UNSUPPORTED;
  ATT_DISPATCH(run_fwd, A / 64, CP, (prm, CL, smem, st));
  return rc;
}

extern "C" int re2e_attloc_step_supported(int B, int Th, int D, int A, int Z, int C, int K, int *cl_fwd_host,
                                          int *cl_bwd_host) {
  int clf = 0, clb = 0;
  if (check_dims(B, Th, D, A, C, K) == RE2E_OK && Z > 0) {
    const int CP = C == 10 ? 10 : 16;
    AttGeom g;
    size_t smem;
    int CL;
    if (pick_geom_fwd(B, Th, D, A, Z, C, K, CP, CL, g, smem)) clf = CL;
    if (pick_geom_bwd(B, Th, D, A, Z, C, K, CP, CL, g, smem)) clb = CL;
  }
  if (cl_fwd_host) *cl_fwd_host = clf;
  if (cl_bwd_host) *cl_bwd_host = clb;
  return clf > 0 && clb > 0;
}

extern "C" size_t re2e_attloc_acc_floats(int A, int C, int K) {
  return (size_t)round4(A * C + C * K + A + 1);
}
// one slot per CTA of the backward launch for this shape (B clusters of CL CTAs); < 0 if the shape is unsupported
extern "C" int re2e_attloc_acc_slots(int B, int Th, int D, int A, int Z, int C, int K) {
  int rc = check_dims(B, Th, D, A, C, K);
  if (rc != RE2E_OK) return rc;
  int CL;
  size_t smem;
  AttGeom g;
  if (!pick_geom_bwd(B, Th, D, A, Z, C, K, C == 10 ? 10 : 16, CL, g, smem)) return RE2E_E_UNSUPPORTED;
  return B * CL;
}

extern "C" int re2e_attloc_step_bwd(const float *dc, const float *dw, const float *xsave, const float *enc_h,
                                    const float *att_prev, const float *w, const float *conv, const float *W_dec,
                                    const float *W_decT, const float *W_att, const float *W_conv, const float *gvec,
                                    float scaling,
                                    float *d_pre, int accumulate_pre, float *d_decproj, float *d_dec_z,
                                    float *d_att_prev, float *acc_slots, int n_slots, int B, int Th, int D, int A,
                                    int Z, int C, int K, void *stream) {
  RE2E_CHECK_ARG(xsave && enc_h && att_prev && w && conv && W_dec && W_att && W_conv && gvec);
  RE2E_CHECK_ARG(d_pre && d_decproj && acc_slots && Z > 0);
  RE2E_CHECK_ARG(!d_dec_z || (W_decT && aligned16(W_decT)));
  int rc = check_dims(B, Th, D, A, C, K);
  if (rc != RE2E_OK) return rc;
  RE2E_CHECK_ARG(aligned16(xsave) && aligned16(enc_h) && aligned16(d_pre));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int CP = C == 10 ? 10 : 16;
  AttBwdParams prm;
  prm.dc = dc; prm.dw = dw; prm.xsave = xsave; prm.enc = enc_h; prm.att_prev = att_prev; prm.w = w;
  prm.conv = conv; prm.W_dec = W_dec; prm.W_decT = W_decT; prm.W_att = W_att; prm.W_conv = W_conv; prm.gvec = gvec;
  prm.scaling = scaling; prm.d_pre = d_pre; prm.d_decproj = d_decproj; prm.d_dec_z = d_dec_z;
  prm.d_att_prev = d_att_prev; prm.acc_slots = acc_slots; prm.accumulate_pre = accumulate_pre;
  prm.slot_stride = (int)re2e_attloc_acc_floats(A, C, K);
  prm.B = B; prm.Th = Th; prm.D = D; prm.A = A; prm.Z = Z; prm.C = C; prm.K = K;
  int CL;
  size_t smem;
  if (!pick_geom_bwd(B, Th, D, A, Z, C, K, CP, CL, prm.g, smem)) return RE2E_E_UNSUPPORTED;
  if (n_slots < B * CL) return RE2E_E_WORKSPACE;
  ATT_DISPATCH(run_bwd, A / 64, CP, (prm, CL, smem, st));
  return rc;
}

// out[0 .. A*C + C*K + A + 1) = sum over the n_slots private accumulators (layout [dW_att | dW_conv | dgvec | dgvec_b])
extern "C" int re2e_attloc_acc_reduce(const float *acc_slots, int n_slots, float *out, int A, int C, int K,
                                      void *stream) {
  RE2E_CHECK_ARG(acc_slots && out && n_slots > 0 && A > 0 && C > 0 && K > 0);
  const int n = A * C + C * K + A + 1;
  acc_reduce_kernel<<<(n + 31) / 32, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      acc_slots, n_slots, (int)re2e_attloc_acc_floats(A, C, K), n, out);
  count_launch();
  return launch_status();
}

extern "C" int re2e_attloc_enc_grad(const float *w_all, const float *dc_all, float *d_enc_h, int steps,
                                    int B, int Th, int D, int accumulate, void *stream) {
  RE2E_CHECK_ARG(w_all && dc_all && d_enc_h && steps > 0 && B > 0 && Th > 0 && D > 0);
  const int tt = 32;   // frames per CTA: the utterance's dc block (steps x D) is re-read Th/tt times from L2
  // The dc rows of the launch's steps are staged in shared memory (<= 200 KB).  A longer decoder loop runs as several
  // launches over equal runs of steps, the first with the caller's `accumulate`, the others adding to it: every
  // element still sums its steps in order, so the result does not depend on the split.
  const int max_steps = (200 * 1024 / (int)sizeof(float) - 3) / (D + tt);
  if (max_steps < 1) return RE2E_E_UNSUPPORTED;
  const int launches = (steps + max_steps - 1) / max_steps;
  const int per = (steps + launches - 1) / launches;
  {
    const size_t smem = sizeof(float) * ((size_t)round4(per * D) + (size_t)per * tt);
    int rc0 = ensure_smem(reinterpret_cast<const void *>(enc_grad_kernel), smem);
    if (rc0 != RE2E_OK) return rc0;
  }
  const int tiles = (Th + tt - 1) / tt;
  for (int s0 = 0; s0 < steps; s0 += per) {
    const int n = min(per, steps - s0);
    const size_t smem = sizeof(float) * ((size_t)round4(n * D) + (size_t)n * tt);
    enc_grad_kernel<<<B * tiles, kEGThreads, smem, static_cast<cudaStream_t>(stream)>>>(
        w_all + (size_t)s0 * B * Th, dc_all + (size_t)s0 * B * D, d_enc_h, n, B, Th, D, tt, s0 == 0 ? accumulate : 1);
    count_launch();
    const int rc = launch_status();
    if (rc != RE2E_OK) return rc;
  }
  return RE2E_OK;
}
