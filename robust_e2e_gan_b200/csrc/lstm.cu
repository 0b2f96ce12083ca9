// LSTMCell step of the attention decoder (model/e2e_decoder.py:128 `self.decoder[0](ey, (z_list[0], c_list[0]))`,
// torch.nn.LSTMCell arithmetic, gate order i, f, g, o) as pieces that fit the decoder loop:
//   * the embedding half of the input product, W_ih[:, :Z] . embed(y_s) + b_ih + b_hh, does not depend on the recurrence:
//     ALL positions at once on the tensor-core GEMM before the loop (training), or a per-token table (beam search);
//   * per position ONE launch (lstm_step_kernel<true>): the two batch-sized products that do depend on it -- context .
//     W_ih[:, Z:]^T and h . W_hh^T -- reduced across a 4-CTA cluster, with the pointwise cell as the epilogue;
//   * backward per position: the pointwise kernel (gate gradients, d c_prev) + ONE product launch for d context | d h_prev
//     (lstm_step_kernel<false>, 8-CTA clusters); the weight gradients of all positions are two dense GEMMs after the loop;
//   * batch_nt_kernel: the generic batch-sized product (any dimensions; also the decoder's output layer in beam search);
//   * sample_tokens_kernel: the same product reduced to each row's arg-max (scheduled sampling in training).
#include "attloc_common.cuh"
#include "common.cuh"

namespace re2e {
namespace {

__device__ __forceinline__ float sigmoid_f(float x) { return 1.0f / (1.0f + __expf(-x)); }

// gates (B,4Z): in = the two recurrent products; out = the gate ACTIVATIONS (i, f, g, o), kept for the backward
__global__ void __launch_bounds__(256) lstm_pointwise_fwd_kernel(float *__restrict__ gates, const float *__restrict__ egate,
                                                                  const float *__restrict__ c_prev,
                                                                  float *__restrict__ c_out, float *__restrict__ h_out,
                                                                  int B, int Z) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * Z) return;
  const int m = idx / Z, u = idx - m * Z;
  float *g = gates + (size_t)m * 4 * Z + u;
  const float *e = egate ? egate + (size_t)m * 4 * Z + u : nullptr;
  const float pi = g[0] + (e ? e[0] : 0.0f), pf = g[Z] + (e ? e[Z] : 0.0f);
  const float pg = g[2 * Z] + (e ? e[2 * Z] : 0.0f), po = g[3 * Z] + (e ? e[3 * Z] : 0.0f);
  const float i = sigmoid_f(pi), f = sigmoid_f(pf), gg = tanhf(pg), o = sigmoid_f(po);
  const float c = f * (c_prev ? c_prev[idx] : 0.0f) + i * gg;
  g[0] = i; g[Z] = f; g[2 * Z] = gg; g[3 * Z] = o;
  c_out[idx] = c;
  h_out[idx] = o * tanhf(c);
}

// act (B,4Z) gate activations, c_new the cell state this step produced; dh / dc: gradients arriving at (h', c') (either may
// be NULL = zero).  dgates (B,4Z): gradient w.r.t. the PRE-activation gates; dc_prev (B,Z).
__global__ void __launch_bounds__(256) lstm_pointwise_bwd_kernel(const float *__restrict__ act, const float *__restrict__ c_prev,
                                                                  const float *__restrict__ c_new, const float *__restrict__ dh,
                                                                  const float *__restrict__ dc, float *__restrict__ dgates,
                                                                  float *__restrict__ dc_prev, int B, int Z) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * Z) return;
  const int m = idx / Z, u = idx - m * Z;
  const float *a = act + (size_t)m * 4 * Z + u;
  const float i = a[0], f = a[Z], g = a[2 * Z], o = a[3 * Z];
  const float tc = tanhf(c_new[idx]);
  const float dhv = dh ? dh[idx] : 0.0f;
  const float dct = (dc ? dc[idx] : 0.0f) + dhv * o * (1.0f - tc * tc);
  float *d = dgates + (size_t)m * 4 * Z + u;
  d[0] = dct * g * i * (1.0f - i);
  d[Z] = dct * (c_prev ? c_prev[idx] : 0.0f) * f * (1.0f - f);
  d[2 * Z] = dct * i * (1.0f - g * g);
  d[3 * Z] = dhv * tc * o * (1.0f - o);
  dc_prev[idx] = dct * f;
}

// out[m,n] (+)= sum_k X[m,k] * W[n,k] (+ bias[n])   for a batch-sized M (the decoder's per-position products: M =
// utterances or beam rows, N up to the vocabulary, K up to 4Z).  One CTA per 8 (or, for long N, 16) output columns so that
// all SMs stream the weight matrix once; warp <-> column.  Within a warp lane <-> (row, slice of the reduction): with M
// rows, 32 / M lanes share a row and split the staged chunk between them (M = 10 beam rows keep 30 lanes busy), combined
// by shuffles at the end.  The reduction runs in chunks of kBK columns staged in shared memory with 128-bit accesses on
// both sides: X rows at a pitch of kBK + 4 floats (conflict-free 128-bit reads with lane <-> row), the warp's W row as
// broadcast reads.  Four independent FMA chains per thread.
constexpr int kBK = 320;       // reduction chunk
constexpr int kBM = 32;        // rows per pass

// One pass of up to kBM rows: returns sum_k X[m0 + lane, k] * W[n, k] in lanes < rows (0 for a column n >= N).  Every
// thread of the CTA must call it (block barriers inside).
__device__ __forceinline__ float batch_nt_pass(const float *__restrict__ X, const float *__restrict__ W, float *x_s,
                                               float *w_s, int m0, int rows, int n, int N, int K, int vec) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int G = 32 / rows;                                     // lanes per row
  const int mrow = lane % rows, part = lane / rows;            // part >= G: idle lane
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  for (int k0 = 0; k0 < K; k0 += kBK) {
    const int kc = min(kBK, K - k0), kq = (kc + 3) >> 2;
    __syncthreads();                                           // previous chunk consumed
    if (vec) {                                                 // K % 4 == 0, 16 B aligned operands
      for (int r = warp; r < rows; r += nwarps)
        for (int q = lane; q < kq; q += 32)
          *reinterpret_cast<float4 *>(x_s + r * (kBK + 4) + 4 * q) =
              __ldcg(reinterpret_cast<const float4 *>(X + (size_t)(m0 + r) * K + k0) + q);   // (X: the predecessor's result)
      for (int q = lane; q < kq; q += 32)
        *reinterpret_cast<float4 *>(w_s + warp * kBK + 4 * q) =
            n < N ? __ldg(reinterpret_cast<const float4 *>(W + (size_t)n * K + k0) + q) : make_float4(0.f, 0.f, 0.f, 0.f);
    } else {                                                   // scalar staging, the chunk zero-padded to a quad
      for (int r = warp; r < rows; r += nwarps)
        for (int k = lane; k < 4 * kq; k += 32)
          x_s[r * (kBK + 4) + k] = k < kc ? __ldcg(X + (size_t)(m0 + r) * K + k0 + k) : 0.f;
      for (int k = lane; k < 4 * kq; k += 32)
        w_s[warp * kBK + k] = (n < N && k < kc) ? __ldg(W + (size_t)n * K + k0 + k) : 0.f;
    }
    __syncthreads();
    if (part < G) {
      const float4 *xr = reinterpret_cast<const float4 *>(x_s + mrow * (kBK + 4));
      const float4 *wr = reinterpret_cast<const float4 *>(w_s + warp * kBK);
#pragma unroll 4
      for (int q = part; q < kq; q += G) {
        const float4 x = xr[q], w = wr[q];
        a0 = fmaf(x.x, w.x, a0); a1 = fmaf(x.y, w.y, a1); a2 = fmaf(x.z, w.z, a2); a3 = fmaf(x.w, w.w, a3);
      }
    }
  }
  float v = (a0 + a1) + (a2 + a3);
  for (int g = 1; g < G; ++g) {
    const float o = __shfl_down_sync(0xffffffffu, v, g * rows);
    if (lane < rows) v += o;
  }
  return v;
}

__global__ void __launch_bounds__(512) batch_nt_kernel(const float *__restrict__ X, const float *__restrict__ W,
                                                      const float *__restrict__ bias, float *__restrict__ out, int M,
                                                      int N, int K, int accumulate, int vec) {
  extern __shared__ __align__(16) float batch_smem[];
  float *x_s = batch_smem, *w_s = batch_smem + kBM * (kBK + 4);
  const int lane = threadIdx.x & 31, n = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  pdl_wait();
  pdl_launch_dependents();
  for (int m0 = 0; m0 < M; m0 += kBM) {
    const int rows = min(kBM, M - m0);
    float v = batch_nt_pass(X, W, x_s, w_s, m0, rows, n, N, K, vec);
    if (lane < rows && n < N) {
      float *o = out + (size_t)(m0 + lane) * N + n;
      v += bias ? __ldg(bias + n) : 0.f;
      *o = accumulate ? __ldcg(o) + v : v;
    }
  }
}

// Scheduled sampling (model/e2e_decoder.py:123-127): tok[m] = argmax_n (X[m,:] . W[n,:] + bias[n]) when *flag != 0, the
// product of batch_nt_kernel without writing the logits.  A row's winner is the largest 64-bit key
//   (order-preserving bits of v + 0.0f) << 32 | (0xFFFFFFFF - n)
// -- larger value first, lower index on equal values, -0 == +0 -- so one atomicMax per (CTA, row) into ws[m] gives an exact
// result whatever order the CTAs finish in.  The last CTA to finish (fence + counter ws[M]) turns the keys into tokens and
// leaves ws zero again: the kernel needs no memset node in a CUDA graph.
__device__ __forceinline__ unsigned long long argmax_key(float v, int n) {
  uint32_t u = __float_as_uint(v + 0.0f);
  u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
  return ((unsigned long long)u << 32) | (unsigned long long)(0xFFFFFFFFu - (uint32_t)n);
}

__global__ void __launch_bounds__(512) sample_tokens_kernel(const float *__restrict__ X, const float *__restrict__ W,
                                                           const float *__restrict__ bias, const int32_t *__restrict__ flag,
                                                           int32_t *__restrict__ tok, unsigned long long *ws, int M,
                                                           int N, int K, int vec) {
  extern __shared__ __align__(16) float batch_smem[];
  __shared__ unsigned long long key_s[kBM];
  __shared__ int last_s;
  float *x_s = batch_smem, *w_s = batch_smem + kBM * (kBK + 4);
  const int tid = threadIdx.x, lane = tid & 31, n = blockIdx.x * (blockDim.x >> 5) + (tid >> 5);
  if (__ldcg(flag) == 0) return;                               // teacher token: tok[] stays as the caller filled it
  for (int m0 = 0; m0 < M; m0 += kBM) {
    const int rows = min(kBM, M - m0);
    if (tid < kBM) key_s[tid] = 0ull;                          // (ordered before the atomics by the pass's barriers)
    const float v = batch_nt_pass(X, W, x_s, w_s, m0, rows, n, N, K, vec);
    if (lane < rows && n < N) atomicMax(&key_s[lane], argmax_key(v + (bias ? __ldg(bias + n) : 0.f), n));
    __syncthreads();
    if (tid < rows) atomicMax(ws + m0 + tid, key_s[tid]);
  }
  __threadfence();
  __syncthreads();
  if (tid == 0) last_s = atomicAdd(ws + M, 1ull) == (unsigned long long)(gridDim.x - 1);
  __syncthreads();
  if (!last_s) return;
  __threadfence();
  for (int m = tid; m < M; m += blockDim.x) tok[m] = (int32_t)(0xFFFFFFFFu - (uint32_t)atomicExch(ws + m, 0ull));
  if (tid == 0) atomicExch(ws + M, 0ull);
}

// ---- one LSTMCell position per launch -----------------------------------------------------------------------------
// Both per-position products have batch-sized M (<= 32 rows per pass) against a 1.5-3 MB weight matrix that stays in
// L2 between positions, so the step is bound by how many SMs pull the weights and by launch latency, not by FLOPs.
// Layout: a cluster works on a tile of 32 X rows x 32 W rows and splits the REDUCTION over its CTAs; every CTA fetches
// its K slice of the 64 rows with one bulk copy per row (one mbarrier), multiplies with a 2-row x 4-column register tile
// per thread (lanes 0-15 <-> rows r / r + 16, half-warps <-> column quads: 6 128-bit shared loads per 32 FMAs), and
// stores its partial tile into rank 0's shared memory (st.shared::cluster); after one cluster barrier rank 0 adds the
// partials in rank order (deterministic) and runs the epilogue:
//   forward  -- the 32 W rows of cluster t are the four gates of hidden units 8t .. 8t+7, the reduction runs over
//               [context | h_prev] against [W_ih[:, Z:] | W_hh] (first half of the ranks <-> context, second half <->
//               h_prev): the epilogue adds the embedding-half gates and applies the cell's pointwise arithmetic, i.e.
//               the whole position is ONE launch on 38 x 4 = 152 CTAs for Z = 300;
//   backward -- W rows are 32 consecutive rows of the transposed matrix (D + Z, 4Z), the reduction runs over the 4Z gate
//               gradients in 8 slices (20 x 8 = 160 CTAs): the epilogue scatters the tile into d context / d h_prev.
constexpr int kSK = 320;           // longest K slice of one CTA
constexpr int kST = 32;            // tile edge (X rows, W rows)
constexpr int kSRP = 40;           // pitch of a partial tile in shared memory
constexpr int kSThreads = 256;     // warps 0-3: first half of the CTA's K slice, warps 4-7: second half

struct LstmStep {
  const float *X1, *X2;            // (M,K1), (M,K2); K2 = 0: one source
  const float *W;                  // rows of K1 + K2 floats
  int M, K1, K2, NW;               // NW: rows of W (forward 4Z, backward D + Z)
  int pitch;                       // shared row pitch in floats: longest slice + 4 or + 8 so that pitch / 4 is odd
                                   // (conflict-free 128-bit reads with lane <-> row)
  const float *egate, *c_prev;     // forward epilogue
  const int32_t *egate_row;        // row of `egate` for batch row m (NULL: m) -- the beam search looks the embedding half up by token
  float *act, *c_out, *h_out;
  int Z;
  float *out1, *out2;              // backward epilogue: columns [0,N1) -> out1 (M,N1), the rest -> out2 (M,NW-N1)
  int N1;
};

inline int lstm_step_pitch(int K1, int K2, int cl) {
  const int parts = K2 > 0 ? cl / 2 : cl;
  int per = round4((K1 + parts - 1) / parts);
  if (K2 > 0) per = max(per, round4((K2 + parts - 1) / parts));
  int pitch = per + 4;
  if (!((pitch >> 2) & 1)) pitch += 4;
  return pitch;
}
inline size_t lstm_step_smem(int pitch, int cl) { return sizeof(float) * (size_t)(2 * kST * pitch + cl * kST * kSRP); }

template <bool FWD>
__global__ void __launch_bounds__(kSThreads) lstm_step_kernel(const LstmStep p) {
  extern __shared__ __align__(16) float step_smem[];
  const int pitch = p.pitch;
  float *x_s = step_smem, *w_s = step_smem + kST * pitch, *red = step_smem + 2 * kST * pitch;
  __shared__ __align__(8) uint64_t bar[2], rbar;     // rbar (rank 0): the partial tiles of all ranks have landed
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, kh = warp >> 2, wq = warp & 3;
  const int rank = (int)cluster_ctarank(), CL = (int)cluster_nctarank();
  const int tile = blockIdx.x / CL;
  const int m0 = blockIdx.y * kST, rows = min(kST, p.M - m0);

  // this rank's slice of the reduction
  const bool second = p.K2 > 0 && rank >= CL / 2;
  const int parts = p.K2 > 0 ? CL / 2 : CL, part = second ? rank - CL / 2 : rank;
  const int Ksrc = second ? p.K2 : p.K1;
  const float *X = second ? p.X2 : p.X1;
  const int per = round4((Ksrc + parts - 1) / parts);
  const int k0 = min(part * per, Ksrc), ks = min(per, Ksrc - k0);
  const int ldw = p.K1 + p.K2, wofs = (second ? p.K1 : 0) + k0;
  const int kq = ks >> 2, kq0 = (kq + 1) >> 1;              // quads of the slice; the first kq0 belong to warps 0-3

  if (tid == 0) {
    mbar_init(&bar[0], 1);
    mbar_init(&bar[1], 1);
    mbar_init(&rbar, 1);
    mbar_fence_init();
    if (rank == 0) mbar_expect_tx(&rbar, (uint32_t)CL * kST * kST * 4u);
  }
  cluster_arrive_relaxed();        // (rank 0's barrier is initialised before anyone signals it)
  __syncthreads();
  // one bulk copy per (row, half): threads 0-31 / 64-95 X rows, 32-63 / 96-127 W rows.  The weights are constant, so their
  // copies go out before the PDL boundary; the X rows (and every other input) are the predecessor's results.
  const int half = (tid >> 6) & 1, r = tid & 31, is_w = (tid >> 5) & 1;
  const int off = half ? 4 * kq0 : 0, len = half ? 4 * (kq - kq0) : 4 * kq0;
  if (tid < 128 && len > 0) {
    const int wrow = FWD ? (r >> 3) * p.Z + tile * 8 + (r & 7) : tile * kST + r;
    const bool wvalid = FWD ? (tile * 8 + (r & 7) < p.Z) : (wrow < p.NW);
    if (r == 0 && !is_w) {
      const int nw = FWD ? 4 * min(8, p.Z - tile * 8) : min(kST, p.NW - tile * kST);
      mbar_expect_tx(&bar[half], (uint32_t)(rows + nw) * (uint32_t)len * 4u);
    }
    if (is_w && wvalid) bulk_g2s(w_s + r * pitch + off, p.W + (size_t)wrow * ldw + wofs + off, (uint32_t)len * 4u, &bar[half]);
  }
  pdl_wait();
  pdl_launch_dependents();
  if (tid < 128 && len > 0 && !is_w && r < rows)
    bulk_g2s(x_s + r * pitch + off, X + (size_t)(m0 + r) * Ksrc + k0 + off, (uint32_t)len * 4u, &bar[half]);
  // rank 0: this thread's epilogue inputs, fetched while the copies fly
  float ep[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
  if (FWD && rank == 0) {
    const int m = tid >> 3, u = tile * 8 + (tid & 7);
    if (m < rows && u < p.Z) {
      const size_t row = (size_t)(m0 + m);
      if (p.egate) {
        const size_t erow = p.egate_row ? (size_t)__ldcg(p.egate_row + row) : row;
#pragma unroll
        for (int g = 0; g < 4; ++g) ep[g] = __ldg(p.egate + erow * 4 * p.Z + (size_t)g * p.Z + u);
      }
      if (p.c_prev) ep[4] = __ldcg(p.c_prev + row * p.Z + u);
    }
  }

  const int hl = lane & 15, cg = lane >> 4;
  float2 acc[2][4];                // (even-k, odd-k) partial sums: the reduction runs as packed FFMA2
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = make_float2(0.f, 0.f);
  const int qb = kh ? kq0 : 0, qe = kh ? kq : kq0;
  if (qe > qb) {
    mbar_wait(&bar[kh], 0);
    const float4 *xa = reinterpret_cast<const float4 *>(x_s + hl * pitch);
    const float4 *xb = reinterpret_cast<const float4 *>(x_s + (hl + 16) * pitch);
    const float4 *wp = reinterpret_cast<const float4 *>(w_s + (8 * wq + 4 * cg) * pitch);
    const int p4 = pitch >> 2;
#pragma unroll 2
    for (int q = qb; q < qe; ++q) {
      const float4 a = xa[q], b = xb[q];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float4 w = wp[j * p4 + q];
        acc[0][j] = __ffma2_rn(make_float2(a.x, a.y), make_float2(w.x, w.y), acc[0][j]);
        acc[0][j] = __ffma2_rn(make_float2(a.z, a.w), make_float2(w.z, w.w), acc[0][j]);
        acc[1][j] = __ffma2_rn(make_float2(b.x, b.y), make_float2(w.x, w.y), acc[1][j]);
        acc[1][j] = __ffma2_rn(make_float2(b.z, b.w), make_float2(w.z, w.w), acc[1][j]);
      }
    }
  }
  float s[2][4];
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) s[i][j] = acc[i][j].x + acc[i][j].y;

  // the two K halves meet in this CTA's own slot; the sum goes to the same slot of rank 0 with stores that signal rank 0's
  // barrier (st.async ... complete_tx): the other ranks are done once the stores are issued, no cluster barrier
  float *mine = red + rank * kST * kSRP;
  const int col = 8 * wq + 4 * cg;
  if (kh) {
    *reinterpret_cast<float4 *>(mine + hl * kSRP + col) = make_float4(s[0][0], s[0][1], s[0][2], s[0][3]);
    *reinterpret_cast<float4 *>(mine + (hl + 16) * kSRP + col) = make_float4(s[1][0], s[1][1], s[1][2], s[1][3]);
  }
  __syncthreads();
  cluster_wait();
  if (!kh) {
    const float4 s0 = *reinterpret_cast<const float4 *>(mine + hl * kSRP + col);
    const float4 s1 = *reinterpret_cast<const float4 *>(mine + (hl + 16) * kSRP + col);
    const uint32_t dst = dsmem_addr(mine, 0), rb = dsmem_addr(&rbar, 0);
    st_async_f32x4(dst + 4u * (uint32_t)(hl * kSRP + col), s[0][0] + s0.x, s[0][1] + s0.y, s[0][2] + s0.z, s[0][3] + s0.w,
                   rb);
    st_async_f32x4(dst + 4u * (uint32_t)((hl + 16) * kSRP + col), s[1][0] + s1.x, s[1][1] + s1.y, s[1][2] + s1.z,
                   s[1][3] + s1.w, rb);
  }
  if (rank != 0) return;
  mbar_wait(&rbar, 0);

  if (FWD) {
    // (row m, hidden unit j of the tile): four gates, partials added in rank order, then the embedding-half gates
    const int m = tid >> 3, j = tid & 7, u = tile * 8 + j;
    if (m < rows && u < p.Z) {
      const size_t row = (size_t)(m0 + m);
      float pre[4];
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        float v = red[m * kSRP + g * 8 + j];
        for (int c = 1; c < CL; ++c) v += red[(c * kST + m) * kSRP + g * 8 + j];
        pre[g] = v + ep[g];
      }
      const float i = sigmoid_f(pre[0]), f = sigmoid_f(pre[1]), gg = tanhf(pre[2]), o = sigmoid_f(pre[3]);
      const float c = f * ep[4] + i * gg;
      float *a = p.act + row * 4 * p.Z + u;
      a[0] = i; a[p.Z] = f; a[2 * p.Z] = gg; a[3 * p.Z] = o;
      p.c_out[row * p.Z + u] = c;
      p.h_out[row * p.Z + u] = o * tanhf(c);
    }
  } else {
    for (int e = tid; e < kST * kST; e += kSThreads) {
      const int m = e >> 5, j = e & 31, n = tile * kST + j;
      if (m >= rows || n >= p.NW) continue;
      float v = red[m * kSRP + j];
      for (int c = 1; c < CL; ++c) v += red[(c * kST + m) * kSRP + j];
      if (n < p.N1) p.out1[(size_t)(m0 + m) * p.N1 + n] = v;
      else p.out2[(size_t)(m0 + m) * (p.NW - p.N1) + (n - p.N1)] = v;
    }
  }
}

template <bool FWD>
int launch_lstm_step(LstmStep prm, int tiles, int cl, cudaStream_t st) {
  auto kern = lstm_step_kernel<FWD>;
  prm.pitch = lstm_step_pitch(prm.K1, prm.K2, cl);
  const size_t smem = lstm_step_smem(prm.pitch, cl);
  int rc = ensure_smem(reinterpret_cast<const void *>(kern), smem);
  if (rc != RE2E_OK) return rc;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(tiles * cl), (unsigned)((prm.M + kST - 1) / kST));
  cfg.blockDim = dim3((unsigned)kSThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)cl;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = (pdl_enabled() && (pdl_mask() & 1)) ? 2 : 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, prm);
  count_launch();
  return e == cudaSuccess ? RE2E_OK : (int)e;
}

constexpr int kFwdCL = 4, kBwdCL = 8;

}  // namespace
}  // namespace re2e

using namespace re2e;

extern "C" int re2e_batch_nt(const float *X, const float *W, const float *bias, float *out, int M, int N, int K,
                             int accumulate, void *stream) {
  RE2E_CHECK_ARG(X && W && out && M > 0 && N > 0 && K > 0);
  const int vec = !(K & 3) && aligned16(X) && aligned16(W);
  const int cols = N >= 2048 ? 16 : 8;                         // columns (warps) per CTA
  const size_t smem = sizeof(float) * (kBM * (kBK + 4) + cols * kBK);
  int rc = ensure_smem(reinterpret_cast<const void *>(batch_nt_kernel), smem);
  if (rc != RE2E_OK) return rc;
  cudaError_t e = launch_pdl(1, batch_nt_kernel, dim3((unsigned)((N + cols - 1) / cols)), dim3((unsigned)(cols * 32)), smem,
                             static_cast<cudaStream_t>(stream), X, W, bias, out, M, N, K, accumulate, vec);
  count_launch();
  return e == cudaSuccess ? launch_status() : (int)e;
}

extern "C" int re2e_sample_tokens_ws_bytes(int M) { return M > 0 ? (int)sizeof(unsigned long long) * (M + 1) : 0; }

extern "C" int re2e_sample_tokens(const float *X, const float *W, const float *bias, const int32_t *flag, int32_t *tok,
                                  unsigned long long *ws, int M, int N, int K, void *stream) {
  RE2E_CHECK_ARG(X && W && flag && tok && ws && M > 0 && N > 0 && K > 0);
  const int vec = !(K & 3) && aligned16(X) && aligned16(W);
  const int cols = N >= 2048 ? 16 : 8;
  const size_t smem = sizeof(float) * (kBM * (kBK + 4) + cols * kBK);
  int rc = ensure_smem(reinterpret_cast<const void *>(sample_tokens_kernel), smem);
  if (rc != RE2E_OK) return rc;
  sample_tokens_kernel<<<(N + cols - 1) / cols, cols * 32, smem, static_cast<cudaStream_t>(stream)>>>(X, W, bias, flag, tok,
                                                                                                  ws, M, N, K, vec);
  count_launch();
  return launch_status();
}

extern "C" int re2e_lstm_step_supported(int B, int D, int Z) {
  return B > 0 && D > 0 && Z > 0 && !(D & 3) && !(Z & 3) && round4((D + 1) / 2) <= kSK && round4((Z + 1) / 2) <= kSK &&
         round4((4 * Z + kBwdCL - 1) / kBwdCL) <= kSK;
}

extern "C" int re2e_lstm_step_fwd(const float *ctx, const float *h_prev, const float *c_prev, const float *Wcat,
                                  const float *egate, const int32_t *egate_row, float *act, float *c_out,
                                  float *h_out, int B, int D, int Z, void *stream) {
  RE2E_CHECK_ARG(ctx && h_prev && Wcat && act && c_out && h_out && B > 0 && D > 0 && Z > 0);
  if (!re2e_lstm_step_supported(B, D, Z) || !aligned16(ctx) || !aligned16(h_prev) || !aligned16(Wcat))
    return RE2E_E_UNSUPPORTED;
  LstmStep p{};
  p.X1 = ctx; p.X2 = h_prev; p.W = Wcat; p.M = B; p.K1 = D; p.K2 = Z; p.NW = 4 * Z;
  p.egate = egate; p.egate_row = egate_row; p.c_prev = c_prev; p.act = act; p.c_out = c_out; p.h_out = h_out; p.Z = Z;
  return launch_lstm_step<true>(p, (Z + 7) / 8, kFwdCL, static_cast<cudaStream_t>(stream));
}

extern "C" int re2e_lstm_step_bwd(const float *dgates, const float *WcatT, float *d_ctx, float *d_hprev, int B, int D,
                                  int Z, void *stream) {
  RE2E_CHECK_ARG(dgates && WcatT && d_ctx && d_hprev && B > 0 && D > 0 && Z > 0);
  if (!re2e_lstm_step_supported(B, D, Z) || !aligned16(dgates) || !aligned16(WcatT)) return RE2E_E_UNSUPPORTED;
  LstmStep p{};
  p.X1 = dgates; p.X2 = nullptr; p.W = WcatT; p.M = B; p.K1 = 4 * Z; p.K2 = 0; p.NW = D + Z;
  p.out1 = d_ctx; p.out2 = d_hprev; p.N1 = D; p.Z = Z;
  return launch_lstm_step<false>(p, (D + Z + kST - 1) / kST, kBwdCL, static_cast<cudaStream_t>(stream));
}

extern "C" int re2e_lstm_pointwise_fwd(float *gates, const float *egate, const float *c_prev, float *c_out, float *h_out,
                                       int B, int Z, void *stream) {
  RE2E_CHECK_ARG(gates && c_out && h_out && B > 0 && Z > 0);
  const int n = B * Z;
  lstm_pointwise_fwd_kernel<<<(n + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(gates, egate, c_prev, c_out,
                                                                                          h_out, B, Z);
  count_launch();
  return launch_status();
}

extern "C" int re2e_lstm_pointwise_bwd(const float *act, const float *c_prev, const float *c_new, const float *dh,
                                       const float *dc, float *dgates, float *dc_prev, int B, int Z, void *stream) {
  RE2E_CHECK_ARG(act && c_new && dgates && dc_prev && B > 0 && Z > 0);
  const int n = B * Z;
  lstm_pointwise_bwd_kernel<<<(n + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(act, c_prev, c_new, dh, dc,
                                                                                          dgates, dc_prev, B, Z);
  count_launch();
  return launch_status();
}
