// Device side of ONE output position of the hybrid CTC/attention beam search (model/e2e_decoder.py:233-314, next rows N1
// and N2 of SURVEY 8f).  All W = beam hypothesis rows are advanced together; the host only merges W x beam candidates
// per position.  The position is this fixed sequence of launches over static buffers (so it replays from a CUDA graph):
//   beam_gather       parent rows of every recurrent state -> working copies           (this file)
//   attloc_step_fwd   attention context / alignment                                    (attloc.cu)
//   lstm_step_fwd     LSTMCell, embedding half looked up by token                      (lstm.cu)
//   batch_nt          output layer                                                     (lstm.cu)
//   log_softmax_topk  log-softmax + the ctc_beam (or beam) best tokens of every row    (this file)
//   ctc_prefix_score  CTC prefix scores of those candidates                            (ctc.cu)
//   beam_joint        (1-w) att + w (ctc - ctc_prev), best `beam` per row, + row score (this file)
#include <math_constants.h>

#include "common.cuh"

namespace re2e {
namespace {

// float <-> unsigned key with the same order (so that redux.sync max does the arg-max in one instruction)
__device__ __forceinline__ unsigned ord_key(float v) {
  const unsigned u = __float_as_uint(v);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord_val(unsigned k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// State tensors one gather can move: z and c of every decoder layer (2 per layer), the alignment and the two CTC states,
// so decoders of up to 6 layers fit with CTC.  The arrays are kernel parameters (400 B of the 4 KB parameter space).
constexpr int kMaxSeg = 16;
struct GatherArgs {
  const float *src[kMaxSeg];
  float *dst[kMaxSeg];
  int row_floats[kMaxSeg];
  int sub_count[kMaxSeg];          // > 0: source rows are indexed (parent, cand) with this many candidates per parent
  const int32_t *parent, *cand;
};

// dst_s[m, :] = src_s[parent[m] (, cand[m]), :] for every state tensor s: grid (W, segments)
__global__ void __launch_bounds__(128) beam_gather_kernel(const GatherArgs a) {
  const int m = blockIdx.x, s = blockIdx.y;
  const int n = a.row_floats[s], sub = a.sub_count[s];
  const int p = __ldg(a.parent + m);
  const size_t srow = sub > 0 ? (size_t)p * sub + __ldg(a.cand + m) : (size_t)p;
  const float *src = a.src[s] + srow * n;
  float *dst = a.dst[s] + (size_t)m * n;
  for (int i = threadIdx.x; i < n; i += blockDim.x) dst[i] = __ldg(src + i);
}

// ---- log-softmax of one row + its k largest entries (sorted, ties -> lower index), one CTA per row ------------------
constexpr int kTkThreads = 1024, kTkVPT = 8;

__device__ __forceinline__ float block_max(float v, float *sh) {
  v = warp_max(v);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = sh[threadIdx.x & 31];
  r = warp_max(r);
  __syncthreads();
  return r;
}
__device__ __forceinline__ float block_sum(float v, float *sh) {
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = sh[threadIdx.x & 31];
  r = warp_sum(r);
  __syncthreads();
  return r;
}

// Selection in two levels: every warp extracts the k best of its 256 entries (k rounds of a redux.sync arg-max, all 32
// warps in parallel, no block barrier), then warp 0 merges the 32 sorted lists (lane <-> list, k rounds over the heads).
__global__ void __launch_bounds__(kTkThreads) log_softmax_topk_kernel(const float *__restrict__ x, float *__restrict__ full,
                                                                      float *__restrict__ vals, int32_t *__restrict__ ids,
                                                                      int V, int k) {
  __shared__ float sh[32];
  __shared__ unsigned ckey[32][33];
  __shared__ int cidx[32][33];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const size_t row = blockIdx.x;
  const float *xr = x + row * V;
  pdl_wait();
  pdl_launch_dependents();
  float v[kTkVPT];
  float m = -CUDART_INF_F;
#pragma unroll
  for (int i = 0; i < kTkVPT; ++i) {
    const int idx = tid + kTkThreads * i;
    v[i] = idx < V ? __ldcg(xr + idx) : -CUDART_INF_F;
    m = fmaxf(m, v[i]);
  }
  m = block_max(m, sh);
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < kTkVPT; ++i)
    if (tid + kTkThreads * i < V) s += expf(v[i] - m);
  s = block_sum(s, sh);
  const float lse = m + logf(s);
  unsigned key[kTkVPT];
#pragma unroll
  for (int i = 0; i < kTkVPT; ++i) {
    const int idx = tid + kTkThreads * i;
    key[i] = 0u;                                   // below the key of every float
    if (idx < V) {
      const float o = v[i] - lse;
      if (full) full[row * V + idx] = o;
      key[i] = ord_key(o);
    }
  }
  for (int j = 0; j < k; ++j) {
    unsigned bk = 0u;
    int bi = 0x7fffffff;
#pragma unroll
    for (int i = 0; i < kTkVPT; ++i)
      if (key[i] > bk) { bk = key[i]; bi = tid + kTkThreads * i; }
    const unsigned mx = __reduce_max_sync(0xffffffffu, bk);
    const int win = (int)__reduce_min_sync(0xffffffffu, bk == mx ? (unsigned)bi : 0x7fffffffu);
    if (lane == 0) { ckey[warp][j] = mx; cidx[warp][j] = win; }
#pragma unroll
    for (int i = 0; i < kTkVPT; ++i)
      if (tid + kTkThreads * i == win) key[i] = 0u;
  }
  __syncthreads();
  if (warp == 0) {
    int p = 0;                                     // head of list `lane`
    for (int j = 0; j < k; ++j) {
      const unsigned hk = p < k ? ckey[lane][p] : 0u;
      const int hi = p < k ? cidx[lane][p] : 0x7fffffff;
      const unsigned mx = __reduce_max_sync(0xffffffffu, hk);
      const int win = (int)__reduce_min_sync(0xffffffffu, hk == mx ? (unsigned)hi : 0x7fffffffu);
      if (hk == mx && hi == win) ++p;
      if (lane == 0) {
        vals[row * k + j] = ord_val(mx);
        ids[row * k + j] = win;
      }
    }
  }
}

// ---- joint score + per-row top `beam` (one warp per hypothesis row) ------------------------------------------------
// local = w_att * att_top + w_ctc * (log_psi - psi_prev)   (model/e2e_decoder.py:284-286; separate roundings, as the
// reference's tensor expression), candidates out[0] = row score + local, out[1] = token id, out[2] = candidate index
__global__ void __launch_bounds__(128) beam_joint_kernel(const float *__restrict__ att_top, const int32_t *__restrict__ ids,
                                                         const float *__restrict__ log_psi,
                                                         const float *__restrict__ psi_prev, const float *__restrict__ sc,
                                                         float w_att, float w_ctc, int W, int Cb, int beam,
                                                         float *__restrict__ out) {
  const int lane = threadIdx.x & 31, h = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (h >= W) return;
  float val = -CUDART_INF_F;
  if (lane < Cb) {
    const float a = att_top[h * Cb + lane];
    val = log_psi ? __fadd_rn(__fmul_rn(w_att, a), __fmul_rn(w_ctc, __fsub_rn(log_psi[h * Cb + lane], psi_prev[h]))) : a;
  }
  const float base = sc[h];
  for (int b = 0; b < beam; ++b) {
    float bv = val;
    int bj = lane;
#pragma unroll
    for (int of = 16; of > 0; of >>= 1) {
      const float v2 = __shfl_xor_sync(0xffffffffu, bv, of);
      const int j2 = __shfl_xor_sync(0xffffffffu, bj, of);
      if (v2 > bv || (v2 == bv && j2 < bj)) { bv = v2; bj = j2; }
    }
    if (lane == 0) {
      out[(size_t)h * beam + b] = __fadd_rn(base, bv);
      out[(size_t)(W + h) * beam + b] = (float)ids[h * Cb + bj];
      out[(size_t)(2 * W + h) * beam + b] = (float)bj;
    }
    if (lane == bj) val = -CUDART_INF_F;
  }
}

// ---- merge of the W x beam candidates of one position (model/e2e_decoder.py:296-333), one warp ---------------------
// The reference extends the live hypotheses one by one and keeps a stable descending sort truncated to `beam`: that is
// the `beam` best of the n_live x beam candidates in (row, rank) order, ties to the lower flat index.  The winners are
// recorded for the host's bookkeeping (hist[pos]: score, parent row, token, candidate index); those that did not emit
// <eos> become the rows of the next position, in order, spare rows repeating the last one.  state = {n_live, pos}.
__global__ void __launch_bounds__(32) beam_merge_kernel(const float *__restrict__ out, int32_t *__restrict__ state,
                                                        int32_t *__restrict__ ctl, float *__restrict__ sc,
                                                        float *__restrict__ hist, int W, int beam, int eos, int maxlen) {
  __shared__ float vals[1024];
  __shared__ float row_sc[32];
  __shared__ int row_p[32], row_j[32], row_t[32];
  const int lane = threadIdx.x;
  const int n = state[0], pos = state[1];
  if (n <= 0 || pos >= maxlen) {
    if (lane == 0) state[1] = pos + 1;
    return;
  }
  const int total = n * beam;
  for (int i = lane; i < total; i += 32) vals[i] = out[i];
  __syncwarp();
  float my_sc = 0.f;
  int my_k = 0;
  for (int b = 0; b < beam; ++b) {
    float bv = -CUDART_INF_F;
    int bk = 0x7fffffff;
    for (int i = lane; i < total; i += 32) {
      const float v = vals[i];
      if (v > bv) { bv = v; bk = i; }
    }
#pragma unroll
    for (int of = 16; of > 0; of >>= 1) {
      const float v2 = __shfl_xor_sync(0xffffffffu, bv, of);
      const int k2 = __shfl_xor_sync(0xffffffffu, bk, of);
      if (v2 > bv || (v2 == bv && k2 < bk)) { bv = v2; bk = k2; }
    }
    if (bk == 0x7fffffff) bk = 0;                      // (every candidate -inf / NaN: keep indices valid)
    if (lane == b) { my_sc = bv; my_k = bk; }
    if (lane == 0) vals[bk] = -CUDART_INF_F;
    __syncwarp();
  }
  // lane b < beam holds winner b
  const bool have = lane < beam;
  const int r = have ? my_k / beam : 0, j = have ? my_k - r * beam : 0;
  const int tok = have ? (int)out[(size_t)(W + r) * beam + j] : eos;
  const int joint = have ? (int)out[(size_t)(2 * W + r) * beam + j] : 0;
  if (have) {
    float *hp = hist + (size_t)pos * 4 * beam;
    hp[lane] = my_sc;
    hp[beam + lane] = (float)r;
    hp[2 * beam + lane] = (float)tok;
    hp[3 * beam + lane] = (float)joint;
  }
  const bool alive = have && tok != eos && pos != maxlen - 1;
  const unsigned m = __ballot_sync(0xffffffffu, alive);
  const int n2 = __popc(m), rank = __popc(m & ((1u << lane) - 1u));
  if (alive) { row_sc[rank] = my_sc; row_p[rank] = r; row_j[rank] = joint; row_t[rank] = tok; }
  __syncwarp();
  if (n2 > 0 && lane < W) {
    const int s = min(lane, n2 - 1);
    ctl[lane] = row_p[s];
    ctl[W + lane] = row_j[s];
    ctl[2 * W + lane] = row_t[s];
    ctl[3 * W + lane] = pos + 1;
    sc[lane] = row_sc[s];
  }
  if (lane == 0) { state[0] = n2; state[1] = pos + 1; }
}

// ---- joint + merge + gather of one position in ONE launch (one CTA, a warp per row) ---------------------------------
// Phase 1 = beam_joint (candidates kept in shared memory), phase 2 = beam_merge on warp 0, phase 3 = beam_gather for the
// NEXT position with the rows just chosen.  Three launch latencies of a strictly serial chain become one.
struct AdvanceArgs {
  const float *att_top, *log_psi, *psi_prev;
  const int32_t *ids;
  float *sc;
  float w_att, w_ctc;
  int W, Cb, beam, eos, maxlen;
  int32_t *state, *ctl;
  float *hist;
  GatherArgs g;
  int nseg;
};

__global__ void __launch_bounds__(1024) beam_advance_kernel(const AdvanceArgs a) {
  __shared__ float s_out[3][1024];
  __shared__ float row_sc[32];
  __shared__ int row_p[32], row_j[32], row_t[32], s_ctl[2][32], s_n2, s_state[2];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int W = a.W, Cb = a.Cb, beam = a.beam;
  pdl_wait();
  pdl_launch_dependents();
  if (threadIdx.x == 1023) { s_state[0] = __ldcg(a.state); s_state[1] = __ldcg(a.state + 1); }     // (latency hidden behind phase 1)
  // phase 1: joint scores of row `warp`, its `beam` best in descending order (arg-max by redux.sync on ordered keys)
  if (warp < W) {
    const int h = warp;
    unsigned key = 0u;
    if (lane < Cb) {
      const float x = __ldcg(a.att_top + h * Cb + lane);
      const float val = a.log_psi ? __fadd_rn(__fmul_rn(a.w_att, x),
                                              __fmul_rn(a.w_ctc, __fsub_rn(__ldcg(a.log_psi + h * Cb + lane),
                                                                           __ldcg(a.psi_prev + h))))
                                  : x;
      key = ord_key(val);
    }
    const int my_id = lane < Cb ? __ldcg(a.ids + h * Cb + lane) : 0;
    const float base = __ldcg(a.sc + h);
    for (int b = 0; b < beam; ++b) {
      const unsigned mx = __reduce_max_sync(0xffffffffu, key);
      const int bj = (int)__reduce_min_sync(0xffffffffu, key == mx ? (unsigned)lane : 32u);
      if (lane == bj) {
        s_out[0][h * beam + b] = __fadd_rn(base, ord_val(mx));
        s_out[1][h * beam + b] = (float)my_id;
        s_out[2][h * beam + b] = (float)bj;
        key = 0u;
      }
    }
  }
  __syncthreads();
  // phase 2 (warp 0): the rows' lists are sorted, so the merge is a W-way merge over the list heads, lane <-> row
  if (warp == 0) {
    const int n = s_state[0], pos = s_state[1];
    int n2 = 0;
    if (n > 0 && pos < a.maxlen) {
      int p = 0;
      float my_sc = 0.f;
      int my_k = 0;
      for (int b = 0; b < beam; ++b) {
        const bool live = lane < n && p < beam;
        const unsigned hk = live ? ord_key(s_out[0][lane * beam + p]) : 0u;
        const unsigned mx = __reduce_max_sync(0xffffffffu, hk);
        const int wl = (int)__reduce_min_sync(0xffffffffu, (live && hk == mx) ? (unsigned)lane : 32u);   // lower flat index
        const int wk = __shfl_sync(0xffffffffu, lane * beam + p, wl & 31);
        if (lane == b) { my_sc = ord_val(mx); my_k = wk; }
        if (lane == wl) ++p;
      }
      const bool have = lane < beam;
      const int r = have ? my_k / beam : 0;
      const int tok = have ? (int)s_out[1][my_k] : a.eos;
      const int joint = have ? (int)s_out[2][my_k] : 0;
      if (have) {
        float *hp = a.hist + (size_t)pos * 4 * beam;
        hp[lane] = my_sc;
        hp[beam + lane] = (float)r;
        hp[2 * beam + lane] = (float)tok;
        hp[3 * beam + lane] = (float)joint;
      }
      const bool alive = have && tok != a.eos && pos != a.maxlen - 1;
      const unsigned m = __ballot_sync(0xffffffffu, alive);
      n2 = __popc(m);
      const int rank = __popc(m & ((1u << lane) - 1u));
      if (alive) { row_sc[rank] = my_sc; row_p[rank] = r; row_j[rank] = joint; row_t[rank] = tok; }
      __syncwarp();
      if (n2 > 0 && lane < W) {
        const int s = min(lane, n2 - 1);
        a.ctl[lane] = row_p[s];
        a.ctl[W + lane] = row_j[s];
        a.ctl[2 * W + lane] = row_t[s];
        a.ctl[3 * W + lane] = pos + 1;
        a.sc[lane] = row_sc[s];
        s_ctl[0][lane] = row_p[s];
        s_ctl[1][lane] = row_j[s];
      }
      if (lane == 0) a.state[0] = n2;
    }
    if (lane == 0) { a.state[1] = pos + 1; s_n2 = n2; }
  }
  __syncthreads();
  // phase 3: the chosen rows' states -> working copies of the next position (four independent loads in flight per
  // thread: the copy is latency-bound)
  if (s_n2 <= 0) return;
  const int nt = blockDim.x;
  for (int s = 0; s < a.nseg; ++s) {
    const int nf = a.g.row_floats[s], sub = a.g.sub_count[s], tot = W * nf;
    const float *src = a.g.src[s];
    float *dst = a.g.dst[s];
    for (int e0 = threadIdx.x; e0 < tot; e0 += 4 * nt) {
      float v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int e = e0 + u * nt;
        if (e < tot) {
          const int m = e / nf, i = e - m * nf;
          const size_t srow = sub > 0 ? (size_t)s_ctl[0][m] * sub + s_ctl[1][m] : (size_t)s_ctl[0][m];
          v[u] = __ldcg(src + srow * nf + i);
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int e = e0 + u * nt;
        if (e < tot) dst[e] = v[u];
      }
    }
  }
}

// ---- initial state of a search: the working copies every row starts from (model/e2e_decoder.py:205-231) -----------
// z = c = 0, alignment uniform over the Th frames (e2e_attention.py:264-268), CTC state r0 = (logzero, running sum of the
// blank column) (model/e2e_ctc.py:95-107, sequential fp32 as the reference's loop), row 0 live with token <sos>.
__global__ void __launch_bounds__(1024) beam_init_kernel(float *__restrict__ z_in, float *__restrict__ c_in,
                                                         float *__restrict__ a_in, float *__restrict__ r_in,
                                                         float *__restrict__ psi_in, const float *__restrict__ lpz,
                                                         int32_t *__restrict__ ctl, float *__restrict__ sc,
                                                         int32_t *__restrict__ state, int W, int Z, int Th, int V,
                                                         int blank, int sos) {
  const int tid = threadIdx.x, nt = blockDim.x;
  for (int i = tid; i < W * Z; i += nt) { z_in[i] = 0.f; c_in[i] = 0.f; }
  const float u = 1.0f / (float)Th;
  for (int i = tid; i < W * Th; i += nt) a_in[i] = u;
  if (tid < W) {
    ctl[tid] = 0; ctl[W + tid] = 0; ctl[2 * W + tid] = sos; ctl[3 * W + tid] = 0;
    sc[tid] = 0.f;
    if (psi_in) psi_in[tid] = 0.f;
  }
  if (tid == 0) { state[0] = 1; state[1] = 0; }
  if (r_in) {
    if (tid == 0) {
      float acc = 0.f;
      for (int t = 0; t < Th; ++t) {
        acc = t == 0 ? __ldg(lpz + blank) : acc + __ldg(lpz + (size_t)t * V + blank);
        r_in[2 * t] = -10000000000.0f;
        r_in[2 * t + 1] = acc;
      }
    }
    __syncthreads();
    for (int i = tid; i < (W - 1) * 2 * Th; i += nt) r_in[2 * Th + i] = r_in[i % (2 * Th)];
  }
}

}  // namespace
}  // namespace re2e

using namespace re2e;

extern "C" int re2e_beam_merge(const float *out, int32_t *state, int32_t *ctl, float *sc, float *hist, int W, int beam,
                               int eos, int maxlen, void *stream) {
  RE2E_CHECK_ARG(out && state && ctl && sc && hist && W > 0 && beam > 0 && maxlen > 0);
  if (W > 32 || beam > 32) return RE2E_E_UNSUPPORTED;
  beam_merge_kernel<<<1, 32, 0, static_cast<cudaStream_t>(stream)>>>(out, state, ctl, sc, hist, W, beam, eos, maxlen);
  count_launch();
  return launch_status();
}

extern "C" int re2e_beam_gather(const int32_t *parent, const int32_t *cand, int W, int nseg, const float *const *src,
                                float *const *dst, const int *row_floats, const int *sub_count, void *stream) {
  RE2E_CHECK_ARG(parent && src && dst && row_floats && sub_count && W > 0 && nseg > 0 && nseg <= kMaxSeg);
  GatherArgs a{};
  for (int s = 0; s < nseg; ++s) {
    RE2E_CHECK_ARG(src[s] && dst[s] && row_floats[s] > 0 && (sub_count[s] == 0 || cand));
    a.src[s] = src[s];
    a.dst[s] = dst[s];
    a.row_floats[s] = row_floats[s];
    a.sub_count[s] = sub_count[s];
  }
  a.parent = parent;
  a.cand = cand;
  beam_gather_kernel<<<dim3((unsigned)W, (unsigned)nseg), 128, 0, static_cast<cudaStream_t>(stream)>>>(a);
  count_launch();
  return launch_status();
}

extern "C" int re2e_log_softmax_topk(const float *logits, long long rows, int V, int k, float *full, float *vals,
                                     int32_t *ids, void *stream) {
  RE2E_CHECK_ARG(logits && vals && ids && rows > 0 && V > 0 && k > 0 && k <= V);
  if (V > kTkThreads * kTkVPT || k > 32) return RE2E_E_UNSUPPORTED;
  log_softmax_topk_kernel<<<(unsigned)rows, kTkThreads, 0, static_cast<cudaStream_t>(stream)>>>(logits, full, vals, ids, V, k);
  count_launch();
  return launch_status();
}

extern "C" int re2e_beam_joint(const float *att_top, const int32_t *ids, const float *log_psi, const float *psi_prev,
                               const float *sc, float w_att, float w_ctc, int W, int Cb, int beam, float *out,
                               void *stream) {
  RE2E_CHECK_ARG(att_top && ids && sc && out && W > 0 && Cb > 0 && beam > 0 && beam <= Cb && (!log_psi || psi_prev));
  if (Cb > 32) return RE2E_E_UNSUPPORTED;
  beam_joint_kernel<<<(W + 3) / 4, 128, 0, static_cast<cudaStream_t>(stream)>>>(att_top, ids, log_psi, psi_prev, sc, w_att,
                                                                              w_ctc, W, Cb, beam, out);
  count_launch();
  return launch_status();
}

extern "C" int re2e_beam_advance(const float *att_top, const int32_t *ids, const float *log_psi, const float *psi_prev,
                                 float *sc, float w_att, float w_ctc, int W, int Cb, int beam, int32_t *state,
                                 int32_t *ctl, float *hist, int eos, int maxlen, int nseg, const float *const *src,
                                 float *const *dst, const int *row_floats, const int *sub_count, void *stream) {
  RE2E_CHECK_ARG(att_top && ids && sc && state && ctl && hist && W > 0 && Cb > 0 && beam > 0 && beam <= Cb && maxlen > 0);
  RE2E_CHECK_ARG((!log_psi || psi_prev) && nseg >= 0 && nseg <= kMaxSeg && (nseg == 0 || (src && dst && row_floats && sub_count)));
  if (W > 32 || Cb > 32) return RE2E_E_UNSUPPORTED;
  AdvanceArgs a{};
  a.att_top = att_top; a.ids = ids; a.log_psi = log_psi; a.psi_prev = psi_prev; a.sc = sc;
  a.w_att = w_att; a.w_ctc = w_ctc; a.W = W; a.Cb = Cb; a.beam = beam; a.eos = eos; a.maxlen = maxlen;
  a.state = state; a.ctl = ctl; a.hist = hist; a.nseg = nseg;
  for (int s = 0; s < nseg; ++s) {
    RE2E_CHECK_ARG(src[s] && dst[s] && row_floats[s] > 0 && sub_count[s] >= 0);
    a.g.src[s] = src[s]; a.g.dst[s] = dst[s]; a.g.row_floats[s] = row_floats[s]; a.g.sub_count[s] = sub_count[s];
  }
  beam_advance_kernel<<<1, 1024, 0, static_cast<cudaStream_t>(stream)>>>(a);
  count_launch();
  return launch_status();
}

extern "C" int re2e_beam_init(float *z_in, float *c_in, float *a_in, float *r_in, float *psi_in, const float *lpz,
                              int32_t *ctl, float *sc, int32_t *state, int W, int Z, int Th, int V, int blank, int sos,
                              void *stream) {
  RE2E_CHECK_ARG(z_in && c_in && a_in && ctl && sc && state && W > 0 && Z > 0 && Th > 0 && (!r_in || (lpz && psi_in && V > 0)));
  if (W > 1024) return RE2E_E_UNSUPPORTED;
  beam_init_kernel<<<1, 1024, 0, static_cast<cudaStream_t>(stream)>>>(z_in, c_in, a_in, r_in, psi_in, lpz, ctl, sc, state, W,
                                                                      Z, Th, V, blank, sos);
  count_launch();
  return launch_status();
}
