// Fused differentiable front-end for sm_100a:
//   mask tail (model/enhance_model.py:157-164) -> power -> F x M mel projection -> clamp -> log -> CMVN
//   (model/feat_model.py:118-135), forward and backward, one kernel each.
//
// Data layout in HBM: mask / mag / d_in are (N = B*T, F) row-major fp32 (F = 257: rows are NOT 16 B
// aligned, so tiles are moved as flat, 16 B aligned spans of R rows with R % 4 == 0); Y / G / dY are
// (N, M).  Each CTA stages one R-row tile of x^2 (fwd) or of the chain-rule factor (bwd) plus the
// whole filter bank in shared memory, so every HBM byte is touched once per pass:
//   fwd  : 4*N*(2F + M) B  (+4*N*M when G is saved)      bwd : 4*N*(M [dY] + M [G] + 2F + F) B
// This file is the fp32-FMA implementation of the projection (bit-faithful to fp32 torch.mm up to
// summation order); see DESIGN.md for the tcgen05 3xTF32 variant.
#include "common.cuh"

namespace re2e {
namespace {

constexpr int kThreads = 256;
constexpr float kClamp = 1e-7f;

struct FbankGeom {
  int R;    // rows per tile (multiple of 4)
  int RG;   // row groups (threads along rows)
  int CG;   // column groups of 8 mel channels
  int Fp;   // padded row pitch of the x tile in smem (floats), Fp/4 odd
  int Mp;   // padded pitch of fc rows in smem: CG*8
  int Mq;   // padded pitch for the bwd layouts (floats), Mq/4 odd
};

template <int TR>
__host__ __device__ inline FbankGeom make_geom(int F, int M) {
  FbankGeom g;
  g.CG = (M + 7) / 8;
  g.RG = kThreads / g.CG;
  int R = g.RG * TR;
  R -= R % 4;
  g.RG = R / TR;  // keep R == RG*TR exactly (TR in {2,4} so R%4==0 keeps divisibility)
  g.R = g.RG * TR;
  g.Fp = (F + 3) & ~3;
  if (((g.Fp / 4) & 1) == 0) g.Fp += 4;
  g.Mp = g.CG * 8;
  g.Mq = g.Mp;
  if (((g.Mq / 4) & 1) == 0) g.Mq += 4;
  return g;
}

// x = act(mask) * valid * mag  (or mag when mask == nullptr); returns x, and s (activation) via ref
__device__ __forceinline__ float mask_x(const float *mask, int mask_is_logit, float magv, float maskv,
                                        bool valid, float &s) {
  if (mask == nullptr) {
    s = 1.0f;
    return magv;
  }
  s = mask_is_logit ? sigmoid_acc(maskv) : maskv;
  if (!valid) s = 0.0f;
  return s * magv;
}

// ------------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------------
template <int TR>
__global__ void __launch_bounds__(kThreads, 1)
fbank_fwd_kernel(const float *__restrict__ mask, int mask_is_logit, const float *__restrict__ mag,
                 const float *__restrict__ fc, const float *__restrict__ cmvn,
                 const int32_t *__restrict__ lens, float *__restrict__ Y, float *__restrict__ G,
                 float *__restrict__ enh_out, int N, int T, int F, int M, int vec_ok) {
  extern __shared__ __align__(16) float smem[];
  const FbankGeom g = make_geom<TR>(F, M);
  float *s_fc = smem;                    // [Fp][Mp]  (rows >= F and cols >= M are zero)
  float *s_x = smem + g.Fp * g.Mp;       // [R][Fp]   x^2
  const int tid = threadIdx.x;

  for (int i = tid; i < g.Fp * g.Mp; i += kThreads) {
    int k = i / g.Mp, m = i - k * g.Mp;
    s_fc[i] = (k < F && m < M) ? __ldg(fc + (size_t)k * M + m) : 0.0f;
  }
  const int cg = tid % g.CG, rg = tid / g.CG;
  const bool active = rg < g.RG;
  const int ntiles = (N + g.R - 1) / g.R;

  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int row0 = tile * g.R;
    const int rows = min(g.R, N - row0);
    __syncthreads();  // previous tile's readers are done with s_x (also covers the s_fc fill)
    // ---- stage: flat span [row0*F, (row0+rows)*F) -> s_x[r][k] = x^2 ; zero the k-padding
    {
      const size_t base = (size_t)row0 * F;
      const int span = rows * F;
      const float *pm = mag + base;
      const float *pk = mask ? mask + base : nullptr;
      float *pe = enh_out ? enh_out + base : nullptr;
      if (vec_ok) {
        const int span4 = span >> 2;  // rows%4==0 or last tile: tail handled below
        for (int i4 = tid; i4 < span4; i4 += kThreads) {
          float4 mv = ld_stream4(pm + 4 * i4);
          float4 kv = pk ? ld_stream4(pk + 4 * i4) : make_float4(0, 0, 0, 0);
          int idx = 4 * i4;
          int r = idx / F, k = idx - r * F;
          float xs[4];
          const float mvv[4] = {mv.x, mv.y, mv.z, mv.w};
          const float kvv[4] = {kv.x, kv.y, kv.z, kv.w};
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            int row = row0 + r;
            int b = row / T;
            bool valid = lens ? (row - b * T) < __ldg(lens + b) : true;
            float s;
            float x = mask_x(pk, mask_is_logit, mvv[j], kvv[j], valid, s);
            xs[j] = x;
            s_x[r * g.Fp + k] = x * x;
            if (++k == F) { k = 0; ++r; }
          }
          if (pe) st_stream4(pe + 4 * i4, make_float4(xs[0], xs[1], xs[2], xs[3]));
        }
        for (int idx = 4 * span4 + tid; idx < span; idx += kThreads) {
          int r = idx / F, k = idx - r * F;
          int row = row0 + r, b = row / T;
          bool valid = lens ? (row - b * T) < __ldg(lens + b) : true;
          float s;
          float x = mask_x(pk, mask_is_logit, pm[idx], pk ? pk[idx] : 0.f, valid, s);
          if (pe) pe[idx] = x;
          s_x[r * g.Fp + k] = x * x;
        }
      } else {
        for (int idx = tid; idx < span; idx += kThreads) {
          int r = idx / F, k = idx - r * F;
          int row = row0 + r, b = row / T;
          bool valid = lens ? (row - b * T) < __ldg(lens + b) : true;
          float s;
          float x = mask_x(pk, mask_is_logit, pm[idx], pk ? pk[idx] : 0.f, valid, s);
          if (pe) pe[idx] = x;
          s_x[r * g.Fp + k] = x * x;
        }
      }
      const int padk = g.Fp - F;
      for (int i = tid; i < g.R * padk; i += kThreads) {
        int r = i / padk, k = F + (i - r * padk);
        s_x[r * g.Fp + k] = 0.0f;
      }
      // rows beyond `rows` in the last tile: zero so the FMAs stay finite
      for (int i = rows * g.Fp + tid; i < g.R * g.Fp; i += kThreads) s_x[i] = 0.0f;
    }
    __syncthreads();
    // ---- projection: thread (rg,cg) owns rows {rg + i*RG} x cols [8cg, 8cg+8)
    if (active) {
      float acc[TR][8];
#pragma unroll
      for (int i = 0; i < TR; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.0f;
      const float *fcp = s_fc + cg * 8;
      for (int k4 = 0; k4 < g.Fp; k4 += 4) {
        float4 xv[TR];
#pragma unroll
        for (int i = 0; i < TR; ++i)
          xv[i] = *reinterpret_cast<const float4 *>(s_x + (rg + i * g.RG) * g.Fp + k4);
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
          const float4 f0 = *reinterpret_cast<const float4 *>(fcp + (k4 + kk) * g.Mp);
          const float4 f1 = *reinterpret_cast<const float4 *>(fcp + (k4 + kk) * g.Mp + 4);
#pragma unroll
          for (int i = 0; i < TR; ++i) {
            const float xk = kk == 0 ? xv[i].x : kk == 1 ? xv[i].y : kk == 2 ? xv[i].z : xv[i].w;
            acc[i][0] = fmaf(xk, f0.x, acc[i][0]);
            acc[i][1] = fmaf(xk, f0.y, acc[i][1]);
            acc[i][2] = fmaf(xk, f0.z, acc[i][2]);
            acc[i][3] = fmaf(xk, f0.w, acc[i][3]);
            acc[i][4] = fmaf(xk, f1.x, acc[i][4]);
            acc[i][5] = fmaf(xk, f1.y, acc[i][5]);
            acc[i][6] = fmaf(xk, f1.z, acc[i][6]);
            acc[i][7] = fmaf(xk, f1.w, acc[i][7]);
          }
        }
      }
      // ---- epilogue: clamp (<= 1e-7 -> 1e-7, zero gradient there), log, CMVN
#pragma unroll
      for (int i = 0; i < TR; ++i) {
        const int r = rg + i * g.RG;
        if (r >= rows) continue;
        const size_t o = (size_t)(row0 + r) * M + cg * 8;
        float y[8], gg[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int m = cg * 8 + j;
          const float P = acc[i][j];
          const bool clamped = P <= kClamp;
          float c0 = 0.f, c1 = 1.f;
          if (cmvn && m < M) { c0 = __ldg(cmvn + m); c1 = __ldg(cmvn + M + m); }
          y[j] = (logf(clamped ? kClamp : P) + c0) * c1;
          gg[j] = clamped ? 0.0f : c1 / P;
        }
        if ((M & 3) == 0 && cg * 8 + 8 <= M) {
          *reinterpret_cast<float4 *>(Y + o) = make_float4(y[0], y[1], y[2], y[3]);
          *reinterpret_cast<float4 *>(Y + o + 4) = make_float4(y[4], y[5], y[6], y[7]);
          if (G) {
            *reinterpret_cast<float4 *>(G + o) = make_float4(gg[0], gg[1], gg[2], gg[3]);
            *reinterpret_cast<float4 *>(G + o + 4) = make_float4(gg[4], gg[5], gg[6], gg[7]);
          }
        } else {
#pragma unroll
          for (int j = 0; j < 8; ++j)
            if (cg * 8 + j < M) {
              Y[o + j] = y[j];
              if (G) G[o + j] = gg[j];
            }
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// backward:  dP = dY * G ;  d(x^2) = dP @ fc^T ;  d_in = d(x^2) * fac,
//   fac = 2*x                      (single-input form, d/d mag)
//       = 2*x*mag*s(1-s)*valid     (mask_is_logit)       = 2*x*mag*valid (plain mask)
// ------------------------------------------------------------------------------------------------
template <int TK>  // k-columns per thread (4)
__global__ void __launch_bounds__(kThreads, 1)
fbank_bwd_kernel(const float *__restrict__ dY, const float *__restrict__ G,
                 const float *__restrict__ mask, int mask_is_logit, const float *__restrict__ mag,
                 const float *__restrict__ fc, const int32_t *__restrict__ lens,
                 float *__restrict__ d_in, int N, int T, int F, int M, int R, int vec_ok) {
  extern __shared__ __align__(16) float smem[];
  const FbankGeom g = make_geom<2>(F, M);
  const int Mq = g.Mq;                 // pitch (floats) of fc rows and dP rows, Mq/4 odd
  float *s_fc = smem;                  // [Fp][Mq]
  float *s_dp = s_fc + g.Fp * Mq;      // [R][Mq]
  float *s_f = s_dp + R * Mq;          // [R][Fp]  factor, overwritten in place by d_in
  const int tid = threadIdx.x;
  for (int i = tid; i < g.Fp * Mq; i += kThreads) {
    int k = i / Mq, m = i - k * Mq;
    s_fc[i] = (k < F && m < M) ? __ldg(fc + (size_t)k * M + m) : 0.0f;
  }
  const int KG = g.Fp / TK;            // k groups (Fp % 4 == 0)
  const int ntiles = (N + R - 1) / R;
  const int M4 = Mq / 4;

  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int row0 = tile * R;
    const int rows = min(R, N - row0);
    __syncthreads();
    // ---- stage dP = dY*G  (zero padded to Mq, rows beyond `rows` zero)
    for (int i = tid; i < R * Mq; i += kThreads) {
      int r = i / Mq, m = i - r * Mq;
      float v = 0.0f;
      if (r < rows && m < M) {
        size_t o = (size_t)(row0 + r) * M + m;
        v = ld_stream1(dY + o) * ld_stream1(G + o);
      }
      s_dp[i] = v;
    }
    // ---- stage factor tile
    {
      const size_t base = (size_t)row0 * F;
      const int span = rows * F;
      const float *pm = mag + base;
      const float *pk = mask ? mask + base : nullptr;
      const int span4 = vec_ok ? (span >> 2) : 0;
      for (int i4 = tid; i4 < span4; i4 += kThreads) {
        float4 mv = ld_stream4(pm + 4 * i4);
        float4 kv = pk ? ld_stream4(pk + 4 * i4) : make_float4(0, 0, 0, 0);
        int idx = 4 * i4;
        int r = idx / F, k = idx - r * F;
        const float mvv[4] = {mv.x, mv.y, mv.z, mv.w};
        const float kvv[4] = {kv.x, kv.y, kv.z, kv.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          int row = row0 + r, b = row / T;
          bool valid = lens ? (row - b * T) < __ldg(lens + b) : true;
          float s;
          float x = mask_x(pk, mask_is_logit, mvv[j], kvv[j], valid, s);
          float fac = 2.0f * x;
          if (pk) fac *= mvv[j] * (mask_is_logit ? s * (1.0f - s) : (valid ? 1.0f : 0.0f));
          s_f[r * g.Fp + k] = fac;
          if (++k == F) { k = 0; ++r; }
        }
      }
      for (int idx = 4 * span4 + tid; idx < span; idx += kThreads) {
        int r = idx / F, k = idx - r * F;
        int row = row0 + r, b = row / T;
        bool valid = lens ? (row - b * T) < __ldg(lens + b) : true;
        float s;
        float mvj = pm[idx];
        float x = mask_x(pk, mask_is_logit, mvj, pk ? pk[idx] : 0.f, valid, s);
        float fac = 2.0f * x;
        if (pk) fac *= mvj * (mask_is_logit ? s * (1.0f - s) : (valid ? 1.0f : 0.0f));
        s_f[r * g.Fp + k] = fac;
      }
    }
    __syncthreads();
    // ---- d(x^2)[r][k] = sum_m dP[r][m] fc[k][m]; thread owns 4 rows x TK k's per work item
    const int RB = (rows + 3) / 4;
    for (int item = tid; item < RB * KG; item += kThreads) {
      const int kg = item % KG, rb = item / KG;
      float acc[4][TK];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < TK; ++j) acc[i][j] = 0.0f;
      // k's are interleaved (k = kg + j*KG) so that a warp's fc rows are Mq floats apart (Mq/4 odd:
      // conflict-free 128-bit reads) and its factor-tile accesses are consecutive words.
      const float4 *fp = reinterpret_cast<const float4 *>(s_fc + kg * Mq);
      const float4 *dp = reinterpret_cast<const float4 *>(s_dp + (rb * 4) * Mq);
      for (int m4 = 0; m4 < M4; ++m4) {
        float4 d[4], f[TK];
#pragma unroll
        for (int i = 0; i < 4; ++i) d[i] = dp[i * M4 + m4];
#pragma unroll
        for (int j = 0; j < TK; ++j) f[j] = fp[(j * KG) * M4 + m4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < TK; ++j) {
            acc[i][j] = fmaf(d[i].x, f[j].x, acc[i][j]);
            acc[i][j] = fmaf(d[i].y, f[j].y, acc[i][j]);
            acc[i][j] = fmaf(d[i].z, f[j].z, acc[i][j]);
            acc[i][j] = fmaf(d[i].w, f[j].w, acc[i][j]);
          }
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int r = rb * 4 + i;
        if (r < rows) {
#pragma unroll
          for (int j = 0; j < TK; ++j) s_f[r * g.Fp + kg + j * KG] *= acc[i][j];
        }
      }
    }
    __syncthreads();
    // ---- flat coalesced store of the d_in tile
    {
      const size_t base = (size_t)row0 * F;
      const int span = rows * F;
      float *po = d_in + base;
      const int span4 = vec_ok ? (span >> 2) : 0;
      for (int i4 = tid; i4 < span4; i4 += kThreads) {
        int idx = 4 * i4;
        int r = idx / F, k = idx - r * F;
        float v[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          v[j] = s_f[r * g.Fp + k];
          if (++k == F) { k = 0; ++r; }
        }
        st_stream4(po + 4 * i4, make_float4(v[0], v[1], v[2], v[3]));
      }
      for (int idx = 4 * span4 + tid; idx < span; idx += kThreads) {
        int r = idx / F, k = idx - r * F;
        po[idx] = s_f[r * g.Fp + k];
      }
    }
  }
}

// dfc[k][m] += sum_n x[n,k]^2 * dP[n,m]   (only when the filter bank is trainable)
__global__ void __launch_bounds__(kThreads)
fbank_dfc_kernel(const float *__restrict__ dY, const float *__restrict__ G,
                 const float *__restrict__ mask, int mask_is_logit, const float *__restrict__ mag,
                 const int32_t *__restrict__ lens, float *__restrict__ dfc, int N, int T, int F, int M,
                 int rows_per_cta) {
  extern __shared__ __align__(16) float smem[];
  constexpr int RC = 16;               // rows per staged chunk
  float *s_x2 = smem;                  // [RC][F]
  float *s_dp = smem + RC * F;         // [RC][M]
  const int tid = threadIdx.x;
  const int row_begin = blockIdx.x * rows_per_cta;
  const int row_end = min(N, row_begin + rows_per_cta);
  const int outs = F * M;
  constexpr int kMaxPer = 48;          // supports F*M <= 48*256 = 12288 per pass
  for (int obase = 0; obase < outs; obase += kMaxPer * kThreads) {
    float acc[kMaxPer];
#pragma unroll
    for (int j = 0; j < kMaxPer; ++j) acc[j] = 0.0f;
    for (int r0 = row_begin; r0 < row_end; r0 += RC) {
      const int rows = min(RC, row_end - r0);
      __syncthreads();
      for (int i = tid; i < rows * F; i += kThreads) {
        int r = i / F;
        int row = r0 + r, b = row / T;
        bool valid = lens ? (row - b * T) < __ldg(lens + b) : true;
        size_t o = (size_t)r0 * F + i;
        float s;
        float x = mask_x(mask, mask_is_logit, mag[o], mask ? mask[o] : 0.f, valid, s);
        s_x2[i] = x * x;
      }
      for (int i = tid; i < rows * M; i += kThreads) {
        size_t o = (size_t)r0 * M + i;
        s_dp[i] = dY[o] * G[o];
      }
      __syncthreads();
#pragma unroll
      for (int j = 0; j < kMaxPer; ++j) {
        int o = obase + j * kThreads + tid;
        if (o < outs) {
          int k = o / M, m = o - k * M;
          float a = acc[j];
          for (int r = 0; r < rows; ++r) a = fmaf(s_x2[r * F + k], s_dp[r * M + m], a);
          acc[j] = a;
        }
      }
    }
#pragma unroll
    for (int j = 0; j < kMaxPer; ++j) {
      int o = obase + j * kThreads + tid;
      if (o < outs) atomicAdd(dfc + o, acc[j]);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// stand-alone mask tail
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads)
mask_apply_kernel(const float *__restrict__ logits, const float *__restrict__ mag,
                  const float *__restrict__ d_enh, const int32_t *__restrict__ lens,
                  float *__restrict__ out, long long total, int T, int F, int vec_ok) {
  // fwd (d_enh == nullptr): out = sigmoid(logits)*valid*mag ; bwd: out = d_enh*mag*s(1-s)*valid
  const long long tf = (long long)T * F;
  const long long stride = (long long)gridDim.x * blockDim.x;
  const long long i0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (vec_ok) {
    const long long total4 = total >> 2;
    for (long long i4 = i0; i4 < total4; i4 += stride) {
      float4 lv = ld_stream4(logits + 4 * i4), mv = ld_stream4(mag + 4 * i4);
      float4 dv = d_enh ? ld_stream4(d_enh + 4 * i4) : make_float4(0, 0, 0, 0);
      const float l[4] = {lv.x, lv.y, lv.z, lv.w}, m[4] = {mv.x, mv.y, mv.z, mv.w},
                  d[4] = {dv.x, dv.y, dv.z, dv.w};
      float o[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        long long idx = 4 * i4 + j;
        int b = (int)(idx / tf);
        int t = (int)((idx - (long long)b * tf) / F);
        bool valid = lens ? t < __ldg(lens + b) : true;
        float s = sigmoid_acc(l[j]);
        o[j] = !valid ? 0.0f : (d_enh ? d[j] * m[j] * s * (1.0f - s) : s * m[j]);
      }
      st_stream4(out + 4 * i4, make_float4(o[0], o[1], o[2], o[3]));
    }
    for (long long idx = 4 * total4 + i0; idx < total; idx += stride) {
      int b = (int)(idx / tf);
      int t = (int)((idx - (long long)b * tf) / F);
      bool valid = lens ? t < __ldg(lens + b) : true;
      float s = sigmoid_acc(logits[idx]);
      out[idx] = !valid ? 0.0f : (d_enh ? d_enh[idx] * mag[idx] * s * (1.0f - s) : s * mag[idx]);
    }
  } else {
    for (long long idx = i0; idx < total; idx += stride) {
      int b = (int)(idx / tf);
      int t = (int)((idx - (long long)b * tf) / F);
      bool valid = lens ? t < __ldg(lens + b) : true;
      float s = sigmoid_acc(logits[idx]);
      out[idx] = !valid ? 0.0f : (d_enh ? d_enh[idx] * mag[idx] * s * (1.0f - s) : s * mag[idx]);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// CMVN statistics over valid frames (fp64 accumulation on device)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads)
cmvn_stats_kernel(const float *__restrict__ Y, const int32_t *__restrict__ lens, double *sum,
                  double *sumsq, long long *frames, int B, int T, int M) {
  // grid.x = B * chunks; each CTA reduces a slab of frames of one utterance; thread -> (frame lane, m)
  const int chunks = gridDim.x / B;
  const int b = blockIdx.x / chunks, ch = blockIdx.x - b * chunks;
  const int len = min(T, max(0, __ldg(lens + b)));
  const int per = (len + chunks - 1) / chunks;
  const int t0 = ch * per, t1 = min(len, t0 + per);
  extern __shared__ __align__(16) float smem[];
  double *s_sum = reinterpret_cast<double *>(smem);     // [lanes][M]
  const int lanes = kThreads / M > 0 ? kThreads / M : 1;
  const int m = threadIdx.x % M, ln = threadIdx.x / M;
  double a = 0.0, q = 0.0;
  if (ln < lanes && threadIdx.x < lanes * M) {
    for (int t = t0 + ln; t < t1; t += lanes) {
      float v = Y[((size_t)b * T + t) * M + m];
      a += (double)v;
      q += (double)v * (double)v;
    }
  }
  double *s_sq = s_sum + lanes * M;
  if (threadIdx.x < lanes * M) { s_sum[ln * M + m] = a; s_sq[ln * M + m] = q; }
  __syncthreads();
  if (threadIdx.x < M) {
    double ta = 0.0, tq = 0.0;
    for (int l = 0; l < lanes; ++l) { ta += s_sum[l * M + threadIdx.x]; tq += s_sq[l * M + threadIdx.x]; }
    atomicAdd(sum + threadIdx.x, ta);
    atomicAdd(sumsq + threadIdx.x, tq);
  }
  if (threadIdx.x == 0 && ch == 0) atomicAdd(reinterpret_cast<unsigned long long *>(frames), (unsigned long long)len);
}

template <typename K>
int set_smem(K kernel, size_t bytes) {
  return ensure_smem(reinterpret_cast<const void *>(kernel), bytes);
}

}  // namespace
}  // namespace re2e

namespace re2e {
// fbank_tc.cu: tcgen05 path; RE2E_E_UNSUPPORTED when the shape does not fit it
int fbank_tc_fwd(const float *mask, int mask_is_logit, const float *mag, const float *fc, const float *cmvn,
                 const int32_t *lens, float *Y, float *G, float *enh_out, int B, int T, int F, int M,
                 cudaStream_t st);
int fbank_tc_bwd(const float *dY, const float *G, const float *mask, int mask_is_logit, const float *mag,
                 const float *fc, const int32_t *lens, float *d_in, int B, int T, int F, int M, cudaStream_t st);
bool fbank_tc_fwd_fits(int F, int M);

namespace {
constexpr size_t kBwdSmemBudget = 200 * 1024;   // SIMT backward: filter bank + as many row tiles as fit

// Shapes that BOTH directions run: a forward kernel (tcgen05, or the SIMT fallback) and the SIMT backward, which is
// the d_in path whenever the tcgen05 backward does not apply (M > 64, M % 4 != 0, F > 260, unaligned dY).
// re2e_fbank_fwd and re2e_fbank_bwd both reject everything else up front, so no shape takes a forward and then fails
// in its backward.  At F = 257 this is M <= 176: the SIMT forward tile of M = 177 needs 237,120 B of shared memory.
bool fbank_shape_ok(int F, int M) {
  if (M > 256) return false;
  const FbankGeom gf = M <= 48 ? make_geom<2>(F, M) : make_geom<4>(F, M);
  const size_t fwd_smem = sizeof(float) * ((size_t)gf.Fp * gf.Mp + (size_t)gf.R * gf.Fp);
  if (fwd_smem > 227 * 1024 && !fbank_tc_fwd_fits(F, M)) return false;
  const FbankGeom gb = make_geom<2>(F, M);
  return sizeof(float) * ((size_t)gb.Fp * gb.Mq + 4 * (size_t)(gb.Mq + gb.Fp)) <= kBwdSmemBudget;
}
}  // namespace
}  // namespace re2e

using namespace re2e;

extern "C" int re2e_fbank_fwd(const float *mask, int mask_is_logit, const float *mag, const float *fc,
                              const float *cmvn, const int32_t *lens, float *Y, float *G,
                              float *enh_out, int B, int T, int F, int M, void *stream) {
  RE2E_CHECK_ARG(mag && fc && Y && B > 0 && T > 0 && F > 0 && M > 0);
  if (!fbank_shape_ok(F, M)) return RE2E_E_UNSUPPORTED;
  const int N = B * T;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int vec_ok = aligned16(mag) && (!mask || aligned16(mask)) && (!enh_out || aligned16(enh_out));
  if (((M & 3) == 0) && !(aligned16(Y) && (!G || aligned16(G)))) return RE2E_E_ARG;
  int rc = fbank_tc_fwd(mask, mask_is_logit, mag, fc, cmvn, lens, Y, G, enh_out, B, T, F, M, st);
  if (rc != RE2E_E_UNSUPPORTED) return rc;   // tensor-core path taken (or a real error)
  if (M <= 48) {
    const FbankGeom g = make_geom<2>(F, M);
    size_t smem = sizeof(float) * ((size_t)g.Fp * g.Mp + (size_t)g.R * g.Fp);
    if ((rc = set_smem(fbank_fwd_kernel<2>, smem)) != RE2E_OK) return rc;
    int ntiles = (N + g.R - 1) / g.R;
    int grid = ntiles < num_sms() ? ntiles : num_sms();
    fbank_fwd_kernel<2><<<grid, kThreads, smem, st>>>(mask, mask_is_logit, mag, fc, cmvn, lens, Y, G,
                                                      enh_out, N, T, F, M, vec_ok);
  } else {
    const FbankGeom g = make_geom<4>(F, M);
    size_t smem = sizeof(float) * ((size_t)g.Fp * g.Mp + (size_t)g.R * g.Fp);
    if ((rc = set_smem(fbank_fwd_kernel<4>, smem)) != RE2E_OK) return rc;
    int ntiles = (N + g.R - 1) / g.R;
    int grid = ntiles < num_sms() ? ntiles : num_sms();
    fbank_fwd_kernel<4><<<grid, kThreads, smem, st>>>(mask, mask_is_logit, mag, fc, cmvn, lens, Y, G,
                                                      enh_out, N, T, F, M, vec_ok);
  }
  count_launch();
  return launch_status();
}

extern "C" int re2e_fbank_bwd(const float *dY, const float *G, const float *mask, int mask_is_logit,
                              const float *mag, const float *fc, const int32_t *lens, float *d_in,
                              float *dfc, int B, int T, int F, int M, void *stream) {
  RE2E_CHECK_ARG(dY && G && mag && fc && B > 0 && T > 0 && F > 0 && M > 0);
  RE2E_CHECK_ARG(d_in || dfc);
  if (!fbank_shape_ok(F, M)) return RE2E_E_UNSUPPORTED;
  const int N = B * T;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int rc;
  bool d_in_done = false;
  if (d_in) {
    rc = fbank_tc_bwd(dY, G, mask, mask_is_logit, mag, fc, lens, d_in, B, T, F, M, st);
    if (rc == RE2E_OK) d_in_done = true;
    else if (rc != RE2E_E_UNSUPPORTED) return rc;
  }
  if (d_in && !d_in_done) {
    const FbankGeom g = make_geom<2>(F, M);
    // rows per tile: fill what is left of ~200 KB after the filter bank, multiple of 4
    size_t fixed = sizeof(float) * (size_t)g.Fp * g.Mq;
    size_t per_row = sizeof(float) * (size_t)(g.Mq + g.Fp);
    size_t budget = kBwdSmemBudget;
    int R = (int)((budget - fixed) / per_row);
    R -= R % 4;
    if (R > 128) R = 128;
    // balance tiles over the SMs
    int ntiles = (N + R - 1) / R;
    int waves = (ntiles + num_sms() - 1) / num_sms();
    int R2 = (N + waves * num_sms() - 1) / (waves * num_sms());
    R2 = (R2 + 3) & ~3;
    if (R2 < R && R2 >= 16) R = R2;
    ntiles = (N + R - 1) / R;
    size_t smem = fixed + per_row * R;
    if ((rc = set_smem(fbank_bwd_kernel<4>, smem)) != RE2E_OK) return rc;
    const int vec_ok = aligned16(mag) && (!mask || aligned16(mask)) && aligned16(d_in);
    int grid = ntiles < num_sms() ? ntiles : num_sms();
    fbank_bwd_kernel<4><<<grid, kThreads, smem, st>>>(dY, G, mask, mask_is_logit, mag, fc, lens, d_in, N,
                                                      T, F, M, R, vec_ok);
    count_launch();
    if ((rc = launch_status()) != RE2E_OK) return rc;
  }
  if (dfc) {
    int ctas = num_sms();
    int rows_per_cta = (N + ctas - 1) / ctas;
    rows_per_cta = (rows_per_cta + 15) & ~15;
    ctas = (N + rows_per_cta - 1) / rows_per_cta;
    size_t smem = sizeof(float) * 16 * (size_t)(F + M);
    if ((rc = set_smem(fbank_dfc_kernel, smem)) != RE2E_OK) return rc;
    fbank_dfc_kernel<<<ctas, kThreads, smem, st>>>(dY, G, mask, mask_is_logit, mag, lens, dfc, N, T, F, M,
                                                   rows_per_cta);
    count_launch();
    if ((rc = launch_status()) != RE2E_OK) return rc;
  }
  return RE2E_OK;
}

extern "C" int re2e_mask_apply_fwd(const float *logits, const float *mag, const int32_t *lens,
                                   float *enh, int B, int T, int F, void *stream) {
  RE2E_CHECK_ARG(logits && mag && enh && B > 0 && T > 0 && F > 0);
  const long long total = (long long)B * T * F;
  const int vec_ok = aligned16(logits) && aligned16(mag) && aligned16(enh);
  long long want = (total / 4 + kThreads - 1) / kThreads;
  int grid = (int)(want < (long long)num_sms() * 8 ? (want > 0 ? want : 1) : num_sms() * 8);
  mask_apply_kernel<<<grid, kThreads, 0, static_cast<cudaStream_t>(stream)>>>(logits, mag, nullptr, lens,
                                                                              enh, total, T, F, vec_ok);
  count_launch();
  return launch_status();
}

extern "C" int re2e_mask_apply_bwd(const float *d_enh, const float *logits, const float *mag,
                                   const int32_t *lens, float *d_logits, int B, int T, int F,
                                   void *stream) {
  RE2E_CHECK_ARG(d_enh && logits && mag && d_logits && B > 0 && T > 0 && F > 0);
  const long long total = (long long)B * T * F;
  const int vec_ok = aligned16(logits) && aligned16(mag) && aligned16(d_enh) && aligned16(d_logits);
  long long want = (total / 4 + kThreads - 1) / kThreads;
  int grid = (int)(want < (long long)num_sms() * 8 ? (want > 0 ? want : 1) : num_sms() * 8);
  mask_apply_kernel<<<grid, kThreads, 0, static_cast<cudaStream_t>(stream)>>>(logits, mag, d_enh, lens,
                                                                              d_logits, total, T, F, vec_ok);
  count_launch();
  return launch_status();
}

extern "C" int re2e_cmvn_stats(const float *Y, const int32_t *lens, double *sum, double *sumsq,
                               long long *frames, int B, int T, int M, void *stream) {
  RE2E_CHECK_ARG(Y && lens && sum && sumsq && frames && B > 0 && T > 0 && M > 0);
  if (M > kThreads) return RE2E_E_UNSUPPORTED;
  int chunks = (num_sms() * 2 + B - 1) / B;
  if (chunks > (T + 31) / 32) chunks = (T + 31) / 32;
  if (chunks < 1) chunks = 1;
  const int lanes = kThreads / M;
  size_t smem = sizeof(double) * 2 * (size_t)lanes * M;
  cmvn_stats_kernel<<<B * chunks, kThreads, smem, static_cast<cudaStream_t>(stream)>>>(Y, lens, sum, sumsq,
                                                                                      frames, B, T, M);
  count_launch();
  return launch_status();
}
