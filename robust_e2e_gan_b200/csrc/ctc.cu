// CTC loss (alpha/beta recursion) and its gradient, log-softmax, best path and batched prefix scoring
// for sm_100a.  Replaces the warp_ctc.CTCLoss call of model/e2e_ctc.py:30,63 (third-party
// warpctc_pytorch; algorithm restated from Graves et al. 2006), F.log_softmax at :75 and the
// per-hypothesis numpy loop of CTCPrefixScore.__call__ at :109-155.
//
// Three kernels per loss evaluation, all HBM-bound on the (B,Th,V) logits:
//   ctc_lse_kernel   : one warp per frame; 128-bit streaming loads, online log-sum-exp per lane,
//                      warp-shuffle merge; gathers the S = 2U+1 label log-probs lp[b,t,s] (compact).
//   ctc_ab_kernel    : one CTA per utterance; alpha (forward in t) and beta (backward in t) run
//                      concurrently in the two halves of the CTA on separate named barriers; the
//                      lattice column lives in shared memory, lp is register-prefetched 8 frames
//                      ahead.  The column is renormalised every 8 frames and the running offset kept
//                      in fp64, so |alpha| stays O(100) and fp32 rounding does not grow with T
//                      (plain fp32 log-domain CTC loses ~1e-4 at |alpha| ~ 1e3).
//   ctc_grad_kernel  : one warp per frame; grad = gscale * (softmax - occupancy), written once.
// Forced alignment (re2e_ctc_align) is ctc_lse_kernel followed by ctc_viterbi_warp_kernel: the forward recursion in the
// max-plus semiring with 2-bit backpointers in shared memory and an on-device backtrace.
// Algorithmic bytes: 4*V per valid frame (lse) + 2*4*V per frame (grad read + write).
#include <math_constants.h>

#include "common.cuh"

namespace re2e {
namespace {

constexpr int kWarpsPerCta = 8;
constexpr int kRenorm = 8;

struct CtcWs {
  unsigned int *counter;
  float *lse;      // (B,Th)
  float *lpmax;    // (B,Th)  max_s lp[b,t,s]: per-frame normaliser of the lattice column
  double *offA;    // (B,Th)
  double *offB;    // (B,Th)
  double *nll_d;   // (B) negative log-likelihood in fp64 (float nll loses 1e-4 at |nll| ~ 1e3)
  float *lpc;      // (B,Th,Smax)
  float *alpha;    // (B,Th,Smax)
  float *beta;     // (B,Th,Smax)
  size_t bytes;
};

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

inline CtcWs carve(void *ws, int B, int Th, int Smax) {
  CtcWs w;
  char *p = static_cast<char *>(ws);
  size_t off = 0;
  w.counter = reinterpret_cast<unsigned int *>(p + off); off += 256;
  w.offA = reinterpret_cast<double *>(p + off); off += align_up(sizeof(double) * (size_t)B * Th, 256);
  w.offB = reinterpret_cast<double *>(p + off); off += align_up(sizeof(double) * (size_t)B * Th, 256);
  w.nll_d = reinterpret_cast<double *>(p + off); off += align_up(sizeof(double) * (size_t)B, 256);
  w.lse = reinterpret_cast<float *>(p + off); off += align_up(sizeof(float) * (size_t)B * Th, 256);
  w.lpmax = reinterpret_cast<float *>(p + off); off += align_up(sizeof(float) * (size_t)B * Th, 256);
  size_t lat = align_up(sizeof(float) * (size_t)B * Th * Smax, 256);
  w.lpc = reinterpret_cast<float *>(p + off); off += lat;
  w.alpha = reinterpret_cast<float *>(p + off); off += lat;
  w.beta = reinterpret_cast<float *>(p + off); off += lat;
  w.bytes = off;
  return w;
}

// merge two (max, sum-of-exp) pairs
__device__ __forceinline__ void lse_merge(float &m, float &s, float m2, float s2) {
  float mn = fmaxf(m, m2);
  if (mn == -CUDART_INF_F) { m = mn; s = 0.f; return; }
  s = s * __expf(m - mn) + s2 * __expf(m2 - mn);
  m = mn;
}
__device__ __forceinline__ void lse_push(float &m, float &s, float x) {
  if (x > m) { s = s * __expf(m - x) + 1.0f; m = x; }
  else s += __expf(x - m);
}
__device__ __forceinline__ void lse_push4(float &m, float &s, float4 v) {
  float mx = fmaxf(fmaxf(v.x, v.y), fmaxf(v.z, v.w));
  if (mx > m) { s *= __expf(m - mx); m = mx; }
  s += __expf(v.x - m) + __expf(v.y - m) + __expf(v.z - m) + __expf(v.w - m);
}

// warp-cooperative (max, sumexp) over one row of V floats; row only 4 B aligned in general
__device__ __forceinline__ void warp_row_lse(const float *row, int V, int lane, float &m, float &s) {
  m = -CUDART_INF_F; s = 0.f;
  int head = (int)(((16u - (unsigned)(reinterpret_cast<uintptr_t>(row) & 15u)) & 15u) >> 2);
  if (head > V) head = V;
  if (lane < head) lse_push(m, s, ld_stream1(row + lane));
  const float *body = row + head;
  const int nvec = (V - head) >> 2;
  int i4 = lane;
  for (; i4 + 96 < nvec; i4 += 128) {
    float4 a = ld_stream4(body + 4 * i4), b = ld_stream4(body + 4 * (i4 + 32)),
           c = ld_stream4(body + 4 * (i4 + 64)), d = ld_stream4(body + 4 * (i4 + 96));
    lse_push4(m, s, a); lse_push4(m, s, b); lse_push4(m, s, c); lse_push4(m, s, d);
  }
  for (; i4 < nvec; i4 += 32) lse_push4(m, s, ld_stream4(body + 4 * i4));
  for (int i = head + 4 * nvec + lane; i < V; i += 32) lse_push(m, s, ld_stream1(row + i));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    float m2 = __shfl_xor_sync(0xffffffffu, m, o), s2 = __shfl_xor_sync(0xffffffffu, s, o);
    lse_merge(m, s, m2, s2);
  }
}

// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kWarpsPerCta * 32)
ctc_lse_kernel(const float *__restrict__ logits, long long stride_b, long long stride_t,
               const int32_t *__restrict__ labels, const int32_t *__restrict__ label_offs,
               const int32_t *__restrict__ label_lens, const int32_t *__restrict__ input_lens, int blank,
               float *__restrict__ lse, float *__restrict__ lpmax, float *__restrict__ lpc, int B, int Th,
               int V, int Smax) {
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5);
  if (row >= (long long)B * Th) return;
  const int b = (int)(row / Th), t = (int)(row - (long long)b * Th);
  if (t >= min(Th, __ldg(input_lens + b))) return;  // padded frame: never read
  const float *x = logits + b * stride_b + t * stride_t;
  float m, s;
  warp_row_lse(x, V, lane, m, s);
  const float l = m + logf(s);
  if (lane == 0) lse[row] = l;
  const int U = __ldg(label_lens + b), S = 2 * U + 1;
  const int32_t *lab = labels + __ldg(label_offs + b);
  float *out = lpc + row * Smax;
  float mx = -CUDART_INF_F;
  for (int i = lane; i < S; i += 32) {
    int v = (i & 1) ? __ldg(lab + (i >> 1)) : blank;
    const float lpv = __ldg(x + v) - l;   // row was just streamed: L2 hit
    out[i] = lpv;
    mx = fmaxf(mx, lpv);
  }
  mx = warp_max(mx);
  if (lane == 0) lpmax[row] = mx;
}

__device__ __forceinline__ void cp_async4(float *dst_smem, const float *src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// log(e^a + e^b + e^c) with -inf handling
// The recursion applies this once per frame on the critical path of a 200-step serial chain, so it is built from the
// raw approximate units (ex2 / lg2: 2^-22 relative / ~1e-7 absolute on [1,3]) instead of the range-reduced libm
// expf / logf (~150 instructions): the sum is in [1, 3] (the max term contributes exactly 1), no range fix-ups needed.
// Absolute error per call ~2e-7, i.e. a few 1e-6 over an utterance -- two orders below the 1e-4 parity tolerance.
__device__ __forceinline__ float lse3(float a, float b, float c) {
  // branch free (the lattice corners are -inf for many frames: a divergent early return would serialise the warp):
  // all three -inf -> m0 = 0, the sum is 0, lg2(0) = -inf and the result is -inf
  const float m = fmaxf(a, fmaxf(b, c));
  const float m0 = m == -CUDART_INF_F ? 0.0f : m;
  const float kLog2e = 1.4426950408889634f, kLn2 = 0.6931471805599453f;
  float ea, eb, ec, l;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(ea) : "f"((a - m0) * kLog2e));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(eb) : "f"((b - m0) * kLog2e));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(ec) : "f"((c - m0) * kLog2e));
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l) : "f"((ea + eb) + ec));
  return fmaf(l, kLn2, m0);
}

__device__ __forceinline__ void named_bar(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ---------------------------------------------------------------------------------------------
// alpha / beta with ONE WARP per direction (2 warps per utterance): lane l owns the SPL consecutive lattice states
// [l*SPL, (l+1)*SPL) in registers, the two neighbours a column update needs from the adjacent lane come through warp
// shuffles, and the SPL independent log-sum-exps per lane overlap in the pipeline.  No shared-memory column, no CTA
// barrier: the per-frame critical path is shuffle -> lse3 instead of STS -> bar.sync -> LDS -> lse3 (the CTA-wide
// version below remains for lattices wider than 32*8 states).  Same outputs / renormalisation scheme as below.
// ---------------------------------------------------------------------------------------------
template <int SPL>
__global__ void __launch_bounds__(32)
ctc_ab_warp_kernel(const float *__restrict__ lpc, const float *__restrict__ lpmax,
                   const int32_t *__restrict__ labels, const int32_t *__restrict__ label_offs,
                   const int32_t *__restrict__ label_lens, const int32_t *__restrict__ input_lens, int blank,
                   float *__restrict__ alpha, float *__restrict__ beta, double *__restrict__ offA,
                   double *__restrict__ offB, float *__restrict__ nll, double *__restrict__ nll_d,
                   float *__restrict__ loss, unsigned int *counter, int B, int Th, int Smax) {
  // grid (B, 2): blockIdx.y is the direction, so every branch on it is block-uniform (a direction per WARP of one
  // CTA makes the compiler wrap each shuffle in convergence barriers)
  constexpr int kRing = SPL <= 4 ? 32 : 16, kAhead = kRing - 8, kSlot = 32 * SPL + 1;
  __shared__ float ring[kRing * kSlot];        // [kRing][32*SPL states | frame max]
  const int b = blockIdx.x;
  const int half = blockIdx.y, lane = threadIdx.x;
  const int T = min(Th, max(0, __ldg(input_lens + b)));
  const int U = __ldg(label_lens + b), S = 2 * U + 1;
  const int32_t *lab = labels + __ldg(label_offs + b);
  const float NEG = -CUDART_INF_F;
  const unsigned FULL = 0xffffffffu;
  const int s0 = lane * SPL;
  bool live[SPL], skip[SPL], start[SPL];
#pragma unroll
  for (int k = 0; k < SPL; ++k) {
    const int s = s0 + k;
    live[k] = s < S;
    skip[k] = false;
    if (live[k] && (s & 1)) {
      if (half == 0) skip[k] = s >= 3 && __ldg(lab + (s >> 1)) != __ldg(lab + (s >> 1) - 1);
      else skip[k] = s + 2 < S && __ldg(lab + (s >> 1)) != __ldg(lab + (s >> 1) + 1);
    }
    start[k] = live[k] && (half == 0 ? (s < 2) : (s >= S - 2));
  }
  const float *lp_b = lpc + (size_t)b * Th * Smax;
  const float *lpm_b = lpmax + (size_t)b * Th;
  float *out_b = (half == 0 ? alpha : beta) + (size_t)b * Th * Smax;
  double *off_b = (half == 0 ? offA : offB) + (size_t)b * Th;
  const long long dir = half ? -1 : 1;
  const int t_first = half ? T - 1 : 0;
  const long long stepS = dir * Smax;

  // Prefetch through shared memory: every lane copies ITS states of frame i + kAhead with 4-byte cp.async (LDGSTS) into a
  // ring, one commit group per frame; cp.async.wait_group kAhead then guarantees frame i has landed.  Unlike a register
  // prefetch this costs no scoreboards (a warp has six, so a rolling register prefetch of 8 frames degenerates to one
  // full memory latency per frame) and no registers, and it runs 24 (wide lattices: 8) frames ahead.
  const float *src_p = lp_b + (long long)t_first * Smax + s0;     // frame being ISSUED (advances with the loop)
  const float *srcm_p = lpm_b + t_first;
  auto issue_frame = [&](int i) {
    if (i < T) {
      float *dst = ring + (i & (kRing - 1)) * kSlot;
#pragma unroll
      for (int k = 0; k < SPL; ++k)
        if (live[k]) cp_async4(dst + s0 + k, src_p + k);
      if (lane == 0) cp_async4(dst + 32 * SPL, srcm_p);
    }
    src_p += stepS;
    srcm_p += dir;
    cp_async_commit();
  };
  // states beyond this utterance's lattice are never copied: they read as -inf from the ring for the whole run, which
  // keeps their column entries at -inf without a per-frame select
#pragma unroll
  for (int k = 0; k < SPL; ++k)
    if (!live[k])
      for (int r = 0; r < kRing; ++r) ring[r * kSlot + s0 + k] = NEG;
  __syncwarp();
  for (int i = 0; i < kAhead; ++i) issue_frame(i);
  float *out_p = out_b + (long long)t_first * Smax + s0;
  double *off_p = off_b + t_first;
  double off = 0.0;
  float a[SPL];
#pragma unroll
  for (int k = 0; k < SPL; ++k) a[k] = NEG;
#pragma unroll 2
  for (int i = 0; i < T; ++i) {
    issue_frame(i + kAhead);
    cp_async_wait<kAhead>();
    __syncwarp();                                   // lane 0's copy of the frame max is visible to the warp
    const float *fr = ring + (i & (kRing - 1)) * kSlot;
    const float lpm = fr[32 * SPL];
    float lpv[SPL];
#pragma unroll
    for (int k = 0; k < SPL; ++k) lpv[k] = fr[s0 + k] - lpm;      // -inf for states outside the lattice
    if (lane == 0) off += (double)lpm;
    // neighbours from the adjacent lane: alpha needs states s-1, s-2 (previous lane's last two), beta s+1, s+2
    float n1, n2;
    if (half == 0) {
      n1 = __shfl_up_sync(FULL, a[SPL - 1], 1);
      n2 = SPL >= 2 ? __shfl_up_sync(FULL, a[SPL >= 2 ? SPL - 2 : 0], 1) : __shfl_up_sync(FULL, a[0], 2);
      if (lane == 0) { n1 = NEG; n2 = NEG; }
      if (SPL == 1 && lane == 1) n2 = NEG;
    } else {
      n1 = __shfl_down_sync(FULL, a[0], 1);
      n2 = SPL >= 2 ? __shfl_down_sync(FULL, a[SPL >= 2 ? 1 : 0], 1) : __shfl_down_sync(FULL, a[0], 2);
      if (lane == 31) { n1 = NEG; n2 = NEG; }
      if (SPL == 1 && lane == 30) n2 = NEG;
    }
    float v[SPL];
#pragma unroll
    for (int k = 0; k < SPL; ++k) {
      float x1, x2;   // the two neighbours of state k in this direction
      if (half == 0) {
        x1 = k >= 1 ? a[k >= 1 ? k - 1 : 0] : n1;
        x2 = k >= 2 ? a[k >= 2 ? k - 2 : 0] : (k == 1 ? n1 : n2);
      } else {
        x1 = k + 1 < SPL ? a[k + 1 < SPL ? k + 1 : 0] : n1;
        x2 = k + 2 < SPL ? a[k + 2 < SPL ? k + 2 : 0] : (k + 1 < SPL ? n1 : n2);
      }
      // frame 0: a = -inf everywhere, the recursion yields -inf and the start states are seeded instead
      const float r = lse3(a[k], x1, skip[k] ? x2 : NEG) + lpv[k];
      v[k] = (i == 0 && start[k]) ? lpv[k] : r;
    }
    if ((i & (kRenorm - 1)) == kRenorm - 1) {   // exact renormalisation: subtract the column max, remember it in fp64
      float m = v[0];
#pragma unroll
      for (int k = 1; k < SPL; ++k) m = fmaxf(m, v[k]);
      m = warp_max(m);
      if (m != NEG) {
#pragma unroll
        for (int k = 0; k < SPL; ++k) v[k] -= m;
        if (lane == 0) off += (double)m;
      }
    }
#pragma unroll
    for (int k = 0; k < SPL; ++k) {
      a[k] = v[k];
      if (live[k]) out_p[k] = v[k];
    }
    if (lane == 0) *off_p = off;
    out_p += stepS;
    off_p += dir;
    __syncwarp();   // every lane is done with this ring slot before it is refilled kRing - kAhead frames later
  }
  if (half == 0) {
    float *fin = ring;
#pragma unroll
    for (int k = 0; k < SPL; ++k) fin[s0 + k] = a[k];
    __syncwarp();
    if (lane == 0) {
      double r;
      if (T == 0) r = (U == 0) ? 0.0 : (double)CUDART_INF_F;
      else {
        float x = fin[S - 1], y = S > 1 ? fin[S - 2] : NEG;
        float m = fmaxf(x, y);
        if (m == NEG) r = (double)CUDART_INF_F;
        else r = -((double)m + (double)logf(expf(x - m) + expf(y - m)) + off);
      }
      nll[b] = (float)r;
      nll_d[b] = r;
      __threadfence();
      unsigned int done = atomicAdd(counter, 1u);
      if (done == (unsigned)B - 1) {      // last utterance to finish: deterministic ordered sum
        __threadfence();
        double acc = 0.0;
        for (int k = 0; k < B; ++k) acc += *(volatile double *)(nll_d + k);
        loss[0] = (float)(acc / (double)B);
        *counter = 0u;
      }
    }
  }
}

// one CTA per utterance; blockDim = 2*Sp (Sp = Smax rounded to 32): first half alpha, second beta
__global__ void __launch_bounds__(1024)
ctc_ab_kernel(const float *__restrict__ lpc, const float *__restrict__ lpmax,
              const int32_t *__restrict__ labels,
              const int32_t *__restrict__ label_offs, const int32_t *__restrict__ label_lens,
              const int32_t *__restrict__ input_lens, int blank, float *__restrict__ alpha,
              float *__restrict__ beta, double *__restrict__ offA, double *__restrict__ offB,
              float *__restrict__ nll, double *__restrict__ nll_d, float *__restrict__ loss,
              unsigned int *counter, int B, int Th, int Smax, int Sp) {
  extern __shared__ __align__(16) float smem[];
  const int b = blockIdx.x;
  const int half = threadIdx.x / Sp;     // warp-uniform (Sp % 32 == 0)
  const int s = threadIdx.x - half * Sp;
  const int pitch = Sp + 4;
  float *col = smem + half * 2 * pitch;  // [2][pitch], element s at index s+2
  float *wred = smem + 4 * pitch + half * 32;
  const int T = min(Th, max(0, __ldg(input_lens + b)));
  const int U = __ldg(label_lens + b), S = 2 * U + 1;
  const int32_t *lab = labels + __ldg(label_offs + b);
  const bool live = s < S;
  // skip transition allowed?  alpha: s-2 -> s ; beta: s+2 -> s
  bool skip = false;
  if (live && (s & 1)) {
    if (half == 0) skip = s >= 3 && __ldg(lab + (s >> 1)) != __ldg(lab + (s >> 1) - 1);
    else skip = s + 2 < S && __ldg(lab + (s >> 1)) != __ldg(lab + (s >> 1) + 1);
  }
  const float NEG = -CUDART_INF_F;
  if (s < 2) { col[s] = NEG; col[pitch + s] = NEG; col[Sp + 2 + s] = NEG; col[pitch + Sp + 2 + s] = NEG; }
  const float *lp_b = lpc + (size_t)b * Th * Smax;
  float *out_b = (half == 0 ? alpha : beta) + (size_t)b * Th * Smax;
  double *off_b = (half == 0 ? offA : offB) + (size_t)b * Th;
  const int nwarps = Sp >> 5;
  const int barid = 1 + half;

  const float *lpm_b = lpmax + (size_t)b * Th;
  float pf[kRenorm], pm[kRenorm];
#pragma unroll
  for (int j = 0; j < kRenorm; ++j) {
    int t = half ? T - 1 - j : j;
    pf[j] = (live && j < T) ? __ldg(lp_b + (size_t)t * Smax + s) : NEG;
    pm[j] = j < T ? __ldg(lpm_b + t) : 0.0f;
  }
  double off = 0.0;
  int cur = 0;
  // running pointers (one add per frame instead of 64-bit index arithmetic): frame t of this direction, and the frame
  // kRenorm steps ahead for the prefetch
  const long long dir = half ? -1 : 1;
  const int t_first = half ? T - 1 : 0;
  const float *pf_ptr = lp_b + ((long long)t_first + dir * kRenorm) * Smax + s;
  const float *pm_ptr = lpm_b + ((long long)t_first + dir * kRenorm);
  float *out_p = out_b + (long long)t_first * Smax + s;
  double *off_p = off_b + t_first;
  const long long stepS = dir * Smax;
  const int d1 = half == 0 ? -1 : 1;      // neighbour offsets inside the column
  const bool start = half == 0 ? (s < 2) : (s >= S - 2);
  for (int i0 = 0; i0 < T; i0 += kRenorm) {
#pragma unroll
    for (int j = 0; j < kRenorm; ++j) {
      const int i = i0 + j;
      if (i >= T) break;
      // every frame is shifted by its own max label log-prob (kept in `off`), so a column only drifts
      // by the gap to the best label between the exact renormalisations below
      const float lpm = pm[j];
      const float lpv = pf[j] - lpm;
      if (s == 0) off += (double)lpm;   // only the thread that stores / uses the offsets pays for the fp64 pipe
      {  // prefetch frame i + kRenorm
        const bool more = i + kRenorm < T;
        pf[j] = (live && more) ? __ldg(pf_ptr) : NEG;
        pm[j] = more ? __ldg(pm_ptr) : 0.0f;
        pf_ptr += stepS;
        pm_ptr += dir;
      }
      const float *c = col + cur * pitch + 2 + s;
      const float a0 = c[0], a1 = c[d1];
      const float a2 = skip ? c[2 * d1] : NEG;
      float v = lse3(a0, a1, a2) + lpv;                  // -inf columns stay -inf
      if (i == 0) v = start ? lpv : NEG;
      if (!live) v = NEG;
      float *n = col + (cur ^ 1) * pitch + 2;
      if (j == kRenorm - 1) {
        // renormalise: subtract the column max, remember it in fp64
        float wm = warp_max(v);
        if ((threadIdx.x & 31) == 0) wred[s >> 5] = wm;
        named_bar(barid, Sp);
        float gm = NEG;
        for (int w = 0; w < nwarps; ++w) gm = fmaxf(gm, wred[w]);
        if (gm != NEG) {
          v -= gm;
          if (s == 0) off += (double)gm;
        }
      }
      n[s] = v;
      if (live) *out_p = v;
      if (s == 0) *off_p = off;
      out_p += stepS;
      off_p += dir;
      cur ^= 1;
      named_bar(barid, Sp);
    }
  }
  if (half == 0 && s == 0) {
    double r;
    if (T == 0) r = (U == 0) ? 0.0 : (double)CUDART_INF_F;
    else {
      const float *c = col + cur * pitch + 2;
      float a = c[S - 1], bb = S > 1 ? c[S - 2] : NEG;
      float m = fmaxf(a, bb);
      if (m == NEG) r = (double)CUDART_INF_F;
      else r = -((double)m + (double)logf(expf(a - m) + expf(bb - m)) + off);
    }
    nll[b] = (float)r;
    nll_d[b] = r;
    __threadfence();
    unsigned int done = atomicAdd(counter, 1u);
    if (done == (unsigned)B - 1) {      // last utterance to finish: deterministic ordered sum
      __threadfence();
      double acc = 0.0;
      for (int k = 0; k < B; ++k) acc += *(volatile double *)(nll_d + k);
      loss[0] = (float)(acc / (double)B);
      *counter = 0u;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Forced alignment: the Viterbi path through the blank-interleaved lattice of a GIVEN transcript, i.e. the forward half
// of ctc_ab_warp_kernel in the max-plus semiring plus backpointers and a backtrace.  One CTA of one warp per utterance,
// lane l owns states [l*SPL, (l+1)*SPL) in registers, lp rows prefetched through the same cp.async ring.
//   v_t(s) = max(v(s), v(s-1), skip ? v(s-2) : -inf) + lp_t(s)        (no transcendental functions)
// Tie rule (also the oracle's, oracle/ctc_align.py ctc_viterbi): on equal values stay in s, then come from s-1, then from s-2;
// at the end take S-1 (final blank) over S-2.  As in alpha / beta, every frame is shifted by its lpmax and the column is
// renormalised every kRenorm frames (offsets in fp64): each subtracts one constant from all states, which keeps |v| and
// hence fp32 rounding small over long utterances and never reverses the order of two states.
// Backpointers: 2 bits per state (0 stay, 1 from s-1, 2 from s-2), one uint32 per lane and frame in dynamic shared
// memory (128 B per frame).  After the last frame lane 0 walks them back from the chosen end state and leaves the state
// of frame t in the same array; the warp then writes states / tokens / spans in parallel over frames.
template <int SPL>
struct ViterbiSmem {
  static constexpr int kRing = SPL <= 4 ? 32 : 16, kAhead = kRing - 8, kSlot = 32 * SPL + 1;
  static constexpr size_t ring_bytes = sizeof(float) * kRing * kSlot;    // multiple of 4 B: bp words follow directly
  static size_t bytes(int Th) { return ring_bytes + sizeof(uint32_t) * 32 * (size_t)Th; }
};

template <int SPL>
__global__ void __launch_bounds__(32)
ctc_viterbi_warp_kernel(const float *__restrict__ lpc, const float *__restrict__ lpmax,
                        const int32_t *__restrict__ labels, const int32_t *__restrict__ label_offs,
                        const int32_t *__restrict__ label_lens, const int32_t *__restrict__ input_lens, int blank,
                        int32_t *__restrict__ states, int32_t *__restrict__ tokens, int32_t *__restrict__ spans,
                        float *__restrict__ score, int Th, int Smax, int Umax) {
  static_assert(SPL <= 16, "2-bit backpointers of one lane must fit one uint32");
  using L = ViterbiSmem<SPL>;
  constexpr int kRing = L::kRing, kAhead = L::kAhead, kSlot = L::kSlot;
  extern __shared__ __align__(16) float vsm[];
  float *ring = vsm;                                                    // [kRing][32*SPL states | frame max]
  uint32_t *bp = reinterpret_cast<uint32_t *>(vsm + kRing * kSlot);     // [Th][32 lanes]
  const int b = blockIdx.x, lane = threadIdx.x;
  const int T = min(Th, max(0, __ldg(input_lens + b)));
  const int U = __ldg(label_lens + b), S = 2 * U + 1;
  const int32_t *lab = labels + __ldg(label_offs + b);
  const float NEG = -CUDART_INF_F;
  const unsigned FULL = 0xffffffffu;
  const int s0 = lane * SPL;
  uint32_t live = 0, skip = 0, start = 0;                               // one bit per state of this lane
#pragma unroll
  for (int k = 0; k < SPL; ++k) {
    const int s = s0 + k;
    if (s < S) {
      live |= 1u << k;
      if ((s & 1) && s >= 3 && __ldg(lab + (s >> 1)) != __ldg(lab + (s >> 1) - 1)) skip |= 1u << k;
      if (s < 2) start |= 1u << k;
    }
  }
  const float *lp_b = lpc + (size_t)b * Th * Smax;
  const float *src_p = lp_b + s0;               // frame being ISSUED (advances with the loop)
  const float *srcm_p = lpmax + (size_t)b * Th;
  auto issue_frame = [&](int i) {
    if (i < T) {
      float *dst = ring + (i & (kRing - 1)) * kSlot;
#pragma unroll
      for (int k = 0; k < SPL; ++k)
        if ((live >> k) & 1u) cp_async4(dst + s0 + k, src_p + k);
      if (lane == 0) cp_async4(dst + 32 * SPL, srcm_p);
    }
    src_p += Smax;
    srcm_p += 1;
    cp_async_commit();
  };
  // states beyond the lattice are never copied and read as -inf for the whole run
#pragma unroll
  for (int k = 0; k < SPL; ++k)
    if (!((live >> k) & 1u))
      for (int r = 0; r < kRing; ++r) ring[r * kSlot + s0 + k] = NEG;
  __syncwarp();
  for (int i = 0; i < kAhead; ++i) issue_frame(i);
  double off = 0.0;
  float a[SPL];
#pragma unroll
  for (int k = 0; k < SPL; ++k) a[k] = NEG;
  uint32_t *bp_p = bp + lane;
#pragma unroll 2
  for (int i = 0; i < T; ++i) {
    issue_frame(i + kAhead);
    cp_async_wait<kAhead>();
    __syncwarp();                                   // lane 0's copy of the frame max is visible to the warp
    const float *fr = ring + (i & (kRing - 1)) * kSlot;
    const float lpm = fr[32 * SPL];
    if (lane == 0) off += (double)lpm;
    float n1 = __shfl_up_sync(FULL, a[SPL - 1], 1);
    float n2 = SPL >= 2 ? __shfl_up_sync(FULL, a[SPL >= 2 ? SPL - 2 : 0], 1) : __shfl_up_sync(FULL, a[0], 2);
    if (lane == 0) { n1 = NEG; n2 = NEG; }
    if (SPL == 1 && lane == 1) n2 = NEG;
    float v[SPL];
    uint32_t word = 0;
#pragma unroll
    for (int k = 0; k < SPL; ++k) {
      const float x1 = k >= 1 ? a[k >= 1 ? k - 1 : 0] : n1;
      const float x2 = k >= 2 ? a[k >= 2 ? k - 2 : 0] : (k == 1 ? n1 : n2);
      float m = a[k];
      uint32_t d = 0;
      if (x1 > m) { m = x1; d = 1; }                                  // strict: ties stay
      if (((skip >> k) & 1u) && x2 > m) { m = x2; d = 2; }            // strict: ties come from s-1
      word |= d << (2 * k);
      const float lpv = fr[s0 + k] - lpm;                             // -inf for states outside the lattice
      // frame 0: the column is -inf everywhere and the start states are seeded instead
      v[k] = i == 0 ? (((start >> k) & 1u) ? lpv : NEG) : m + lpv;
    }
    *bp_p = word;
    bp_p += 32;
    if ((i & (kRenorm - 1)) == kRenorm - 1) {
      float m = v[0];
#pragma unroll
      for (int k = 1; k < SPL; ++k) m = fmaxf(m, v[k]);
      m = warp_max(m);
      if (m != NEG) {
#pragma unroll
        for (int k = 0; k < SPL; ++k) v[k] -= m;
        if (lane == 0) off += (double)m;
      }
    }
#pragma unroll
    for (int k = 0; k < SPL; ++k) a[k] = v[k];
    __syncwarp();   // every lane is done with this ring slot before it is refilled kRing - kAhead frames later
  }
  // final column -> shared memory (the ring is idle: every issued copy belonged to a frame < T and has landed)
#pragma unroll
  for (int k = 0; k < SPL; ++k) ring[s0 + k] = a[k];
  __syncwarp();
  int feasible = 0;
  if (lane == 0) {
    float sc;
    if (T == 0) {
      sc = U == 0 ? 0.0f : NEG;
    } else {
      const float x = ring[S - 1], y = S > 1 ? ring[S - 2] : NEG;
      int s = y > x ? S - 2 : S - 1;                                    // ties: final blank
      const float e = fmaxf(x, y);
      if (e == NEG) {
        sc = NEG;
      } else {
        sc = (float)(off + (double)e);
        feasible = 1;
        // serial walk; the state of frame t replaces word t % 32 of frame t once that frame has been read (a bank
        // per lane for the parallel pass below)
        for (int t = T - 1; t >= 0; --t) {
          const uint32_t w = bp[t * 32 + s / SPL];
          bp[t * 32 + (t & 31)] = (uint32_t)s;
          if (t > 0) s -= (int)((w >> (2 * (s % SPL))) & 3u);
        }
      }
    }
    score[b] = sc;
  }
  feasible = __shfl_sync(FULL, feasible, 0);   // also orders lane 0's shared-memory writes before the reads below
  __syncwarp();
  int32_t *st_b = states + (size_t)b * Th, *tk_b = tokens + (size_t)b * Th;
  int32_t *sp_b = spans + (size_t)b * Umax * 2;
  const int Tv = feasible ? T : 0;
  for (int t = lane; t < Th; t += 32) {
    int s = -1, tok = -1;
    if (t < Tv) {
      s = (int)bp[t * 32 + (t & 31)];
      tok = (s & 1) ? __ldg(lab + (s >> 1)) : blank;
      if (s & 1) {      // every label state is visited by one run of frames: its ends are written exactly once
        const int u = s >> 1;
        if (t == 0 || (int)bp[(t - 1) * 32 + ((t - 1) & 31)] != s) sp_b[2 * u] = t;
        if (t == Tv - 1 || (int)bp[(t + 1) * 32 + ((t + 1) & 31)] != s) sp_b[2 * u + 1] = t;
      }
    }
    st_b[t] = s;
    tk_b[t] = tok;
  }
  for (int u = (feasible ? U : 0) + lane; u < Umax; u += 32) {
    sp_b[2 * u] = -1;
    sp_b[2 * u + 1] = -1;
  }
}

// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kWarpsPerCta * 32)
ctc_grad_kernel(const float *__restrict__ logits, long long stride_b, long long stride_t,
                const int32_t *__restrict__ labels, const int32_t *__restrict__ label_offs,
                const int32_t *__restrict__ label_lens, const int32_t *__restrict__ input_lens, int blank,
                const double *__restrict__ nll_d, const float *__restrict__ grad_out,
                const float *__restrict__ lse, const float *__restrict__ lpc,
                const float *__restrict__ alpha, const float *__restrict__ beta,
                const double *__restrict__ offA, const double *__restrict__ offB, float *__restrict__ grad,
                int B, int Th, int V, int Smax, int vec_ok) {
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5);
  if (row >= (long long)B * Th) return;
  const int b = (int)(row / Th), t = (int)(row - (long long)b * Th);
  const float *x = logits + b * stride_b + t * stride_t;
  float *g = grad + b * stride_b + t * stride_t;
  const bool valid = t < min(Th, __ldg(input_lens + b));
  const float gs = (grad_out ? __ldg(grad_out) : 1.0f) / (float)B;
  const float l = valid ? lse[row] : 0.f;
  int head = (int)(((16u - (unsigned)(reinterpret_cast<uintptr_t>(g) & 15u)) & 15u) >> 2);
  if (!vec_ok || head > V) head = V;
  for (int i = lane; i < head; i += 32) g[i] = valid ? gs * __expf(ld_stream1(x + i) - l) : 0.f;
  const int nvec = (V - head) >> 2;
  const float *xb = x + head;
  float *gb = g + head;
  if (valid) {
    int i4 = lane;
    for (; i4 + 96 < nvec; i4 += 128) {
      float4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = ld_stream4(xb + 4 * (i4 + 32 * u));
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        float4 o = make_float4(gs * __expf(v[u].x - l), gs * __expf(v[u].y - l), gs * __expf(v[u].z - l),
                               gs * __expf(v[u].w - l));
        *reinterpret_cast<float4 *>(gb + 4 * (i4 + 32 * u)) = o;
      }
    }
    for (; i4 < nvec; i4 += 32) {
      float4 v = ld_stream4(xb + 4 * i4);
      *reinterpret_cast<float4 *>(gb + 4 * i4) = make_float4(
          gs * __expf(v.x - l), gs * __expf(v.y - l), gs * __expf(v.z - l), gs * __expf(v.w - l));
    }
  } else {
    for (int i4 = lane; i4 < nvec; i4 += 32) *reinterpret_cast<float4 *>(gb + 4 * i4) = make_float4(0, 0, 0, 0);
  }
  for (int i = head + 4 * nvec + lane; i < V; i += 32) g[i] = valid ? gs * __expf(ld_stream1(x + i) - l) : 0.f;
  if (!valid) return;
  const double nl = nll_d[b];
  if (!isfinite(nl)) return;  // infeasible labelling: leave softmax only
  __syncwarp();               // row stores above are ordered before the corrections below
  const int U = __ldg(label_lens + b), S = 2 * U + 1;
  const int32_t *lab = labels + __ldg(label_offs + b);
  const double base = offA[row] + offB[row] + nl;
  const size_t lo = (size_t)row * Smax;
  for (int i = lane; i < S; i += 32) {
    float a = alpha[lo + i], bt = beta[lo + i];
    if (a == -CUDART_INF_F || bt == -CUDART_INF_F) continue;
    float occ = expf((float)((double)a + (double)bt - (double)lpc[lo + i] + base));
    int v = (i & 1) ? __ldg(lab + (i >> 1)) : blank;
    atomicAdd(g + v, -gs * occ);
  }
}

// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kWarpsPerCta * 32)
log_softmax_kernel(const float *__restrict__ x, float *__restrict__ out, int32_t *__restrict__ best,
                   long long rows, int V) {
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5);
  if (row >= rows) return;
  const float *xr = x + row * V;
  float *o = out + row * V;
  float m = -CUDART_INF_F, s = 0.f;
  int am = 0x7fffffff;
  float av = -CUDART_INF_F;
  for (int i = lane; i < V; i += 32) {
    float v = xr[i];
    lse_push(m, s, v);
    if (v > av) { av = v; am = i; }
  }
#pragma unroll
  for (int of = 16; of > 0; of >>= 1) {
    float m2 = __shfl_xor_sync(0xffffffffu, m, of), s2 = __shfl_xor_sync(0xffffffffu, s, of);
    lse_merge(m, s, m2, s2);
    float av2 = __shfl_xor_sync(0xffffffffu, av, of);
    int am2 = __shfl_xor_sync(0xffffffffu, am, of);
    if (av2 > av || (av2 == av && am2 < am)) { av = av2; am = am2; }
  }
  const float l = m + logf(s);
  for (int i = lane; i < V; i += 32) o[i] = xr[i] - l;
  if (best && lane == 0) best[row] = am;
}

// ---------------------------------------------------------------------------------------------
// Cross-entropy of the attention decoder (model/e2e_decoder.py:155-157, F.cross_entropy with ignore_index, mean over
// the labelled positions) without materialising log-softmax: one pass per row gives lse, the row's nll and its arg-max
// (th_accuracy, model/e2e_common.py:198-205); the backward writes (softmax - onehot) * scale in one pass.  Rows may be
// pitched (`ld`, the padded layout the tensor-core GEMM writes).  One warp per row.
__global__ void __launch_bounds__(kWarpsPerCta * 32)
ce_fwd_kernel(const float *__restrict__ x, long long ld, const long long *__restrict__ target, long long ignore_id,
              long long rows, int V, float *__restrict__ lse, float *__restrict__ nll, int32_t *__restrict__ best) {
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5);
  if (row >= rows) return;
  const float *xr = x + row * ld;
  float m = -CUDART_INF_F, s = 0.f, av = -CUDART_INF_F;
  int am = 0x7fffffff;
  for (int i = lane; i < V; i += 32) {
    const float v = xr[i];
    lse_push(m, s, v);
    if (v > av) { av = v; am = i; }
  }
#pragma unroll
  for (int of = 16; of > 0; of >>= 1) {
    const float m2 = __shfl_xor_sync(0xffffffffu, m, of), s2 = __shfl_xor_sync(0xffffffffu, s, of);
    lse_merge(m, s, m2, s2);
    const float av2 = __shfl_xor_sync(0xffffffffu, av, of);
    const int am2 = __shfl_xor_sync(0xffffffffu, am, of);
    if (av2 > av || (av2 == av && am2 < am)) { av = av2; am = am2; }
  }
  if (lane == 0) {
    const float l = m + logf(s);
    const long long t = target[row];
    lse[row] = l;
    nll[row] = (t == ignore_id || t < 0 || t >= V) ? 0.f : l - xr[t];
    if (best) best[row] = am;
  }
}

__global__ void __launch_bounds__(kWarpsPerCta * 32)
ce_bwd_kernel(const float *__restrict__ x, long long ld, const long long *__restrict__ target, long long ignore_id,
              long long rows, int V, const float *__restrict__ lse, const float *__restrict__ scale,
              float *__restrict__ dx, long long ldd) {
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5);
  if (row >= rows) return;
  const long long t = target[row];
  const bool on = !(t == ignore_id || t < 0 || t >= V);
  const float l = lse[row], sc = on ? __ldg(scale) : 0.f;
  const float *xr = x + row * ld;
  float *dr = dx + row * ldd;
  for (int i = lane; i < V; i += 32) dr[i] = on ? (expf(xr[i] - l) - (i == t ? 1.f : 0.f)) * sc : 0.f;
}

// ---------------------------------------------------------------------------------------------
// Batched prefix scoring (model/e2e_ctc.py:109-155): one WARP per (hypothesis h, candidate j), lane <-> frame, 32 frames
// per block.  The recursion
//     r^n_t = (r^n_{t-1} + phi_{t-1}) x_t ,   r^b_t = (r^n_{t-1} + r^b_{t-1}) y_t        (probability domain)
// is linear in the state (r^n, r^b, 1): frame t is the matrix [[x, 0, x phi], [y, y, 0], [0, 0, 1]] and products of such
// matrices keep the shape [[a, 0, p], [b, d, q], [0, 0, 1]].  So instead of a 32-step dependent chain per block the warp
// runs an inclusive SCAN over the frames' matrices in the log semiring (5 shuffle steps, 4 logaddexp each) and applies
// every lane's prefix product to the state carried in from the previous block: ~12 dependent logaddexp per 32 frames
// instead of 32.  psi = logsumexp_t(phi_{t-1} + x_t) is a plain warp reduction.  Everything that does not depend on the
// recursion (phi, the two columns of lpz) is fetched one block ahead, coalesced.
// Arithmetic in base-2 logs with raw MUFU approximations (relative error 2^-22, far inside the parity tolerance);
// "log 0" is the reference's logzero, which absorbs every finite addend in fp32 exactly as it does there.
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float lg2_approx(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float lae2(float a, float b) {      // log2(2^a + 2^b)
  return fmaxf(a, b) + lg2_approx(1.0f + ex2_approx(-fabsf(a - b)));
}
constexpr int kPrefixWarps = 4;
__global__ void __launch_bounds__(kPrefixWarps * 32)
ctc_prefix_kernel(const float *__restrict__ lpz, const float *__restrict__ r_prev,
                  const int32_t *__restrict__ cs, const int32_t *__restrict__ last,
                  const int32_t *__restrict__ out_len, float *__restrict__ log_psi,
                  float *__restrict__ r_new, int T, int V, int H, int Cc, int blank, int eos) {
  const int lane = threadIdx.x & 31;
  const int idx = blockIdx.x * kPrefixWarps + (threadIdx.x >> 5);
  pdl_wait();
  pdl_launch_dependents();
  if (idx >= H * Cc) return;
  const int h = idx / Cc;
  const int c = __ldcg(cs + idx);        // (candidates, states: results of kernels this grid may overlap)
  const float LZ = -10000000000.0f, L2E = 1.4426950408889634f, LN2 = 0.6931471805599453f, LZ2 = LZ * L2E;
  const int ol = __ldcg(out_len + h);
  const float *rp = r_prev + (size_t)h * T * 2;
  float *rn = r_new + (size_t)idx * T * 2;
  const bool same = ol > 0 && c == __ldcg(last + h);
  const int start = ol > 1 ? ol : 1;
  for (int t = lane; t < min(start - 1, T); t += 32) *reinterpret_cast<float2 *>(rn + 2 * t) = make_float2(LZ, LZ);
  const float r0 = ol == 0 ? __ldg(lpz + c) : LZ;
  if (lane == 0 && start - 1 < T) *reinterpret_cast<float2 *>(rn + 2 * (start - 1)) = make_float2(r0, LZ);
  float n_in = r0 * L2E, b_in = LZ2;               // state after frame base-1, base-2 logs
  float psi = LZ2;                                 // this lane's share of logsumexp_t(phi_{t-1} + x_t)
  // operands of frame t of the current block, fetched one block ahead of their use
  float2 pv = make_float2(LZ, LZ);
  float xc = 0.f, xb = 0.f;
  if (start + lane < T) {
    const int t = start + lane;
    pv = __ldcg(reinterpret_cast<const float2 *>(rp + 2 * (t - 1)));
    xc = __ldg(lpz + (size_t)t * V + c);
    xb = __ldg(lpz + (size_t)t * V + blank);
  }
  for (int base = start; base < T; base += 32) {
    const int t = base + lane;
    const bool valid = t < T;
    const float phi = same ? pv.y * L2E : lae2(pv.x * L2E, pv.y * L2E);
    const float x = xc * L2E, y = xb * L2E;
    if (t + 32 < T) {                              // next block's operands
      pv = __ldcg(reinterpret_cast<const float2 *>(rp + 2 * (t + 31)));
      xc = __ldg(lpz + (size_t)(t + 32) * V + c);
      xb = __ldg(lpz + (size_t)(t + 32) * V + blank);
    }
    // this frame's matrix (identity beyond T): [[a, 0, p], [b, d, q], [0, 0, 1]] in logs
    float a = valid ? x : 0.f, b = valid ? y : LZ2, d = valid ? y : 0.f, p = valid ? x + phi : LZ2, q = LZ2;
    if (valid) psi = lae2(psi, x + phi);
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {       // mine (later frames) x theirs (earlier frames)
      const float a0 = __shfl_up_sync(0xffffffffu, a, off), b0 = __shfl_up_sync(0xffffffffu, b, off),
                  d0 = __shfl_up_sync(0xffffffffu, d, off), p0 = __shfl_up_sync(0xffffffffu, p, off),
                  q0 = __shfl_up_sync(0xffffffffu, q, off);
      if (lane >= off) {
        const float qn = lae2(lae2(b + p0, d + q0), q);
        const float bn = lae2(b + a0, d + b0);
        p = lae2(a + p0, p);
        a += a0;
        d += d0;
        b = bn;
        q = qn;
      }
    }
    const float nn = lae2(a + n_in, p);
    const float nb = lae2(lae2(b + n_in, d + b_in), q);
    if (valid) *reinterpret_cast<float2 *>(rn + 2 * t) = make_float2(fmaxf(nn * LN2, LZ), fmaxf(nb * LN2, LZ));
    n_in = __shfl_sync(0xffffffffu, nn, 31);
    b_in = __shfl_sync(0xffffffffu, nb, 31);
  }
#pragma unroll
  for (int of = 16; of > 0; of >>= 1) psi = lae2(psi, __shfl_xor_sync(0xffffffffu, psi, of));
  psi = lae2(psi, r0 * L2E);                       // the t = start-1 term the reference starts from
  psi = fmaxf(psi * LN2, LZ);
  if (c == eos) {
    const float a = __ldcg(rp + 2 * (T - 1)), b = __ldcg(rp + 2 * (T - 1) + 1);
    psi = fmaxf(lae2(a * L2E, b * L2E) * LN2, LZ);
  }
  if (lane == 0) log_psi[idx] = psi;
}

}  // namespace
}  // namespace re2e

using namespace re2e;

extern "C" size_t re2e_ctc_ws_bytes(int B, int Th, int V, int Umax) {
  (void)V;
  if (B <= 0 || Th <= 0 || Umax < 0) return 0;
  return carve(nullptr, B, Th, 2 * Umax + 1).bytes;
}

extern "C" int re2e_ctc_loss_fwd(const float *logits, long long stride_b, long long stride_t,
                                 const int32_t *labels, const int32_t *label_offs,
                                 const int32_t *label_lens, const int32_t *input_lens, int blank,
                                 float *nll, float *loss, void *ws, size_t ws_bytes, int B, int Th, int V,
                                 int Umax, void *stream) {
  RE2E_CHECK_ARG(logits && labels && label_offs && label_lens && input_lens && nll && loss && ws);
  RE2E_CHECK_ARG(B > 0 && Th > 0 && V > 0 && Umax >= 0 && blank >= 0 && blank < V);
  const int Smax = 2 * Umax + 1;
  const int Sp = (Smax + 31) & ~31;
  if (2 * Sp > 1024) return RE2E_E_UNSUPPORTED;
  CtcWs w = carve(ws, B, Th, Smax);
  if (ws_bytes < w.bytes) return RE2E_E_WORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  RE2E_CUDA(cudaMemsetAsync(w.counter, 0, 256, st));
  const long long rows = (long long)B * Th;
  const int grid = (int)((rows + kWarpsPerCta - 1) / kWarpsPerCta);
  ctc_lse_kernel<<<grid, kWarpsPerCta * 32, 0, st>>>(logits, stride_b, stride_t, labels, label_offs,
                                                     label_lens, input_lens, blank, w.lse, w.lpmax, w.lpc, B,
                                                     Th, V, Smax);
  count_launch();
  int rc = launch_status();
  if (rc != RE2E_OK) return rc;
  // lattices of up to 256 states: one warp per direction, the column in registers (SPL states per lane)
  const int spl = (Smax + 31) / 32;
#define RE2E_AB_WARP(SPLV)                                                                                          \
  ctc_ab_warp_kernel<SPLV><<<dim3(B, 2), 32, 0, st>>>(w.lpc, w.lpmax, labels, label_offs, label_lens, input_lens, blank,     \
                                             w.alpha, w.beta, w.offA, w.offB, nll, w.nll_d, loss, w.counter, B, Th, \
                                             Smax)
  if (spl <= 1) RE2E_AB_WARP(1);
  else if (spl == 2) RE2E_AB_WARP(2);
  else if (spl == 3) RE2E_AB_WARP(3);
  else if (spl == 4) RE2E_AB_WARP(4);
  else if (spl <= 6) RE2E_AB_WARP(6);
  else if (spl <= 8) RE2E_AB_WARP(8);
  else {
    const size_t smem = sizeof(float) * (4 * (size_t)(Sp + 4) + 64);
    ctc_ab_kernel<<<B, 2 * Sp, smem, st>>>(w.lpc, w.lpmax, labels, label_offs, label_lens, input_lens, blank, w.alpha,
                                           w.beta, w.offA, w.offB, nll, w.nll_d, loss, w.counter, B, Th, Smax, Sp);
  }
#undef RE2E_AB_WARP
  count_launch();
  return launch_status();
}

extern "C" int re2e_ctc_loss_bwd(const float *logits, long long stride_b, long long stride_t,
                                 const int32_t *labels, const int32_t *label_offs,
                                 const int32_t *label_lens, const int32_t *input_lens, int blank,
                                 const float *nll, const float *grad_out, const void *ws, size_t ws_bytes,
                                 float *grad, int B, int Th, int V, int Umax, void *stream) {
  RE2E_CHECK_ARG(logits && labels && label_offs && label_lens && input_lens && nll && ws && grad);
  RE2E_CHECK_ARG(B > 0 && Th > 0 && V > 0 && Umax >= 0);
  const int Smax = 2 * Umax + 1;
  CtcWs w = carve(const_cast<void *>(ws), B, Th, Smax);
  if (ws_bytes < w.bytes) return RE2E_E_WORKSPACE;
  const long long rows = (long long)B * Th;
  const int grid = (int)((rows + kWarpsPerCta - 1) / kWarpsPerCta);
  const int vec_ok = ((reinterpret_cast<uintptr_t>(logits) ^ reinterpret_cast<uintptr_t>(grad)) & 15u) == 0;
  ctc_grad_kernel<<<grid, kWarpsPerCta * 32, 0, static_cast<cudaStream_t>(stream)>>>(
      logits, stride_b, stride_t, labels, label_offs, label_lens, input_lens, blank, w.nll_d, grad_out, w.lse,
      w.lpc, w.alpha, w.beta, w.offA, w.offB, grad, B, Th, V, Smax, vec_ok);
  count_launch();
  return launch_status();
}

namespace re2e {
namespace {
template <int SPL>
int launch_viterbi(const CtcWs &w, const int32_t *labels, const int32_t *label_offs, const int32_t *label_lens,
                   const int32_t *input_lens, int blank, int32_t *states, int32_t *tokens, int32_t *spans, float *score,
                   int B, int Th, int Smax, int Umax, cudaStream_t st) {
  const size_t smem = ViterbiSmem<SPL>::bytes(Th);
  ctc_viterbi_warp_kernel<SPL><<<B, 32, smem, st>>>(w.lpc, w.lpmax, labels, label_offs, label_lens, input_lens, blank,
                                                    states, tokens, spans, score, Th, Smax, Umax);
  count_launch();
  return launch_status();
}
// the backpointers of the whole utterance live in shared memory: 128 B per frame next to the prefetch ring
template <int SPL>
int prepare_viterbi(int Th) {
  const size_t smem = ViterbiSmem<SPL>::bytes(Th);
  if (smem > 227 * 1024) return RE2E_E_UNSUPPORTED;
  return ensure_smem(reinterpret_cast<const void *>(&ctc_viterbi_warp_kernel<SPL>), smem);
}
}  // namespace
}  // namespace re2e

extern "C" int re2e_ctc_align(const float *logits, long long stride_b, long long stride_t, const int32_t *labels,
                              const int32_t *label_offs, const int32_t *label_lens, const int32_t *input_lens, int blank,
                              int32_t *states, int32_t *tokens, int32_t *spans, float *score, void *ws, size_t ws_bytes,
                              int B, int Th, int V, int Umax, void *stream) {
  RE2E_CHECK_ARG(logits && labels && label_offs && label_lens && input_lens && states && tokens && score && ws);
  RE2E_CHECK_ARG(B > 0 && Th > 0 && V > 0 && Umax >= 0 && blank >= 0 && blank < V && (spans || Umax == 0));
  if (Umax > 255) return RE2E_E_UNSUPPORTED;       // the loss's limit: Smax <= 511, at most 16 states per lane
  const int Smax = 2 * Umax + 1;
  const int spl = (Smax + 31) / 32;
  // every shape check comes before the first launch
#define RE2E_VIT(F)                                                                                                  \
  (spl <= 1 ? F<1> : spl == 2 ? F<2> : spl == 3 ? F<3> : spl == 4 ? F<4> : spl <= 6 ? F<6> : spl <= 8 ? F<8>         \
   : spl <= 12 ? F<12> : F<16>)
  int rc = RE2E_VIT(prepare_viterbi)(Th);
  if (rc != RE2E_OK) return rc;
  CtcWs w = carve(ws, B, Th, Smax);
  if (ws_bytes < w.bytes) return RE2E_E_WORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long rows = (long long)B * Th;
  const int grid = (int)((rows + kWarpsPerCta - 1) / kWarpsPerCta);
  ctc_lse_kernel<<<grid, kWarpsPerCta * 32, 0, st>>>(logits, stride_b, stride_t, labels, label_offs, label_lens,
                                                     input_lens, blank, w.lse, w.lpmax, w.lpc, B, Th, V, Smax);
  count_launch();
  rc = launch_status();
  if (rc != RE2E_OK) return rc;
  rc = RE2E_VIT(launch_viterbi)(w, labels, label_offs, label_lens, input_lens, blank, states, tokens, spans, score, B, Th,
                                Smax, Umax, st);
#undef RE2E_VIT
  return rc;
}

extern "C" int re2e_log_softmax(const float *logits, float *out, int32_t *best, long long rows, int V,
                                void *stream) {
  RE2E_CHECK_ARG(logits && out && rows > 0 && V > 0);
  const int grid = (int)((rows + kWarpsPerCta - 1) / kWarpsPerCta);
  log_softmax_kernel<<<grid, kWarpsPerCta * 32, 0, static_cast<cudaStream_t>(stream)>>>(logits, out, best,
                                                                                       rows, V);
  count_launch();
  return launch_status();
}

extern "C" int re2e_cross_entropy_fwd(const float *logits, long long ld, const long long *target, long long ignore_id,
                                      long long rows, int V, float *lse, float *nll, int32_t *best, void *stream) {
  RE2E_CHECK_ARG(logits && target && lse && nll && rows > 0 && V > 0 && ld >= V);
  const int grid = (int)((rows + kWarpsPerCta - 1) / kWarpsPerCta);
  ce_fwd_kernel<<<grid, kWarpsPerCta * 32, 0, static_cast<cudaStream_t>(stream)>>>(logits, ld, target, ignore_id, rows, V,
                                                                                  lse, nll, best);
  count_launch();
  return launch_status();
}

extern "C" int re2e_cross_entropy_bwd(const float *logits, long long ld, const long long *target, long long ignore_id,
                                      long long rows, int V, const float *lse, const float *scale, float *dlogits,
                                      long long ldd, void *stream) {
  RE2E_CHECK_ARG(logits && target && lse && scale && dlogits && rows > 0 && V > 0 && ld >= V && ldd >= V);
  const int grid = (int)((rows + kWarpsPerCta - 1) / kWarpsPerCta);
  ce_bwd_kernel<<<grid, kWarpsPerCta * 32, 0, static_cast<cudaStream_t>(stream)>>>(logits, ld, target, ignore_id, rows, V,
                                                                                  lse, scale, dlogits, ldd);
  count_launch();
  return launch_status();
}

extern "C" int re2e_ctc_prefix_score(const float *lpz, const float *r_prev, const int32_t *cs,
                                     const int32_t *last, const int32_t *out_len, float *log_psi,
                                     float *r_new, int T, int V, int H, int Ccand, int blank, int eos,
                                     void *stream) {
  RE2E_CHECK_ARG(lpz && r_prev && cs && last && out_len && log_psi && r_new);
  RE2E_CHECK_ARG(T > 0 && V > 0 && H > 0 && Ccand > 0);
  const int n = H * Ccand;
  cudaError_t e = launch_pdl(3, ctc_prefix_kernel, dim3((unsigned)((n + kPrefixWarps - 1) / kPrefixWarps)),
                             dim3(kPrefixWarps * 32), 0, static_cast<cudaStream_t>(stream), lpz, r_prev, cs, last, out_len,
                             log_psi, r_new, T, V, H, Ccand, blank, eos);
  count_launch();
  return e == cudaSuccess ? launch_status() : (int)e;
}
