/*
 * re2e_b200.h -- C ABI of the B200-native hot path for Robust_e2e_gan.
 *
 * The reference (bliunlpr/Robust_e2e_gan) has no FFI of its own: its hot path
 * is three Python nn.Modules that dispatch to ATen / cuDNN / warp-ctc.  This
 * header is the boundary a maintainer binds instead (ctypes stub shown in
 * INTEGRATION.md).  Each entry point cites the reference lines it replaces.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - fp32, row-major, contiguous unless a stride argument says otherwise;
 *   - `stream` is a cudaStream_t passed as void* (torch.cuda.current_stream().cuda_stream);
 *   - no entry point allocates, frees or synchronises; scratch comes in as `ws`;
 *   - return value: 0 = ok; < 0 = argument error (RE2E_E_*); > 0 = cudaError_t.
 *   - NULL for an optional pointer disables that input / output.
 */
#ifndef RE2E_B200_H_
#define RE2E_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RE2E_OK 0
#define RE2E_E_ARG (-1)        /* bad size / null pointer / misaligned buffer */
#define RE2E_E_UNSUPPORTED (-2) /* shape outside what the kernels were built for */
#define RE2E_E_WORKSPACE (-3)   /* ws_bytes too small; call the *_ws_bytes query */

/* ABI / build identification. */
int re2e_abi_version(void);              /* bumps on any signature change */
const char *re2e_build_info(void);       /* "sm_100a nvcc 12.9 ..." */
const char *re2e_error_string(int code); /* static string for RE2E_E_* or cudaGetErrorString */
/* Number of kernel launches this library has issued in this process (monotonic). */
unsigned long long re2e_launch_count(void);

/* --------------------------------------------------------------------------------------------
 * Front-end.  Replaces model/enhance_model.py:157-164 (mask tail) fused with
 * model/feat_model.py:118-135 (FbankModel.forward) and its autograd backward.
 *
 *   x[n,f]  = mask ? act(mask[n,f]) * [t < lens[b]] * mag[n,f] : mag[n,f]        n = b*T + t
 *   P[n,m]  = sum_f x[n,f]^2 * fc[f,m]
 *   Y[n,m]  = (log(max(P, 1e-7)) + cmvn[0,m]) * cmvn[1,m]            (cmvn optional)
 *   G[n,m]  = P > 1e-7 ? cmvn[1,m] / P : 0          (dY/dP; saved for the backward, optional)
 *
 * mask_is_logit: 1 -> act = sigmoid (mask holds linear_out), 0 -> act = identity.
 * enh_out (optional): receives x (the reference's `enhance_out`, (B,T,F)).
 * Shapes: re2e_fbank_fwd and re2e_fbank_bwd accept the same (F, M) and return RE2E_E_UNSUPPORTED for the rest before
 * launching anything -- M <= 176 at F = 257 (the SIMT forward's shared-memory tile above 80 filters is the limit).
 * ------------------------------------------------------------------------------------------ */
int re2e_fbank_fwd(const float *mask, int mask_is_logit, const float *mag, const float *fc,
                   const float *cmvn, const int32_t *lens, float *Y, float *G, float *enh_out,
                   int B, int T, int F, int M, void *stream);

/* dY (N,M) -> d_in (N,F): gradient w.r.t. `mask` when mask != NULL (through act and *mag),
 * else w.r.t. `mag` (the single-input FbankModel form).  G is the tensor saved by fwd.
 * dfc (optional, (F,M), ACCUMULATED into): gradient of a trainable filter bank
 * (feat_model.py:105-109 `fbank_opti_type == 'train'`). */
int re2e_fbank_bwd(const float *dY, const float *G, const float *mask, int mask_is_logit,
                   const float *mag, const float *fc, const int32_t *lens, float *d_in, float *dfc,
                   int B, int T, int F, int M, void *stream);

/* Banded filter bank (csrc/fbank_band.cu).  A triangular mel bank -- the reference's frozen 80-filter table
 * (model/feat_model.py:15-33: every FFT bin feeds <= 2 filters) or any bank generated like model/e2e_common.py:104-132
 * -- is banded; for it the front-end is a pure HBM stream (TMA bulk copies of 8-frame spans into a shared-memory ring,
 * ~450 MACs per frame instead of the dense 257 x M projection).  The caller detects the structure ONCE from fc (F,M)
 * and passes it as tables:
 *   flo[M] int32, fw[M*32] : filter m = sum_{k<32} fw[m*32+k] * P[flo[m]+k]   (its support lies in 32 consecutive bins,
 *                            flo[m] + 32 <= F)
 *   mlo[F] int32, bw[F*4]  : bin f feeds filters mlo[f] .. mlo[f]+3 with weights bw[f*4+k]   (mlo[f] + 4 <= M)
 * A bank that does not fit (a trained, dense fc) uses re2e_fbank_fwd / _bwd (tcgen05 dense projection).
 * Forward, up to three outputs per launch (joint_train.py:158-161 -- `mag` is read once for two of them):
 *   mask != NULL : Y_enh, G  from act(mask)*[t<lens]*mag   (as re2e_fbank_fwd);  Y_plain (optional) from plain mag
 *   mask == NULL : Y_enh, G  from plain mag (the single-input form; Y_plain must be NULL)
 *   mag2, Y2     : optional second plain input and its output (both or neither)
 * Backward: d_in as re2e_fbank_bwd (no dfc: a frozen bank).  Shapes: (B*T) % 8 == 0, 32 <= F, 4 <= M <= 80
 * (re2e_fbank_band_supported); inputs 16 B aligned. */
int re2e_fbank_band_supported(int B, int T, int F, int M);
int re2e_fbank_band_fwd(const float *mask, int mask_is_logit, const float *mag, const float *mag2,
                        const int32_t *flo, const float *fw, const float *cmvn, const int32_t *lens, float *Y_enh,
                        float *G, float *Y_plain, float *Y2, int B, int T, int F, int M, void *stream);
int re2e_fbank_band_bwd(const float *dY, const float *G, const float *mask, int mask_is_logit, const float *mag,
                        const int32_t *mlo, const float *bw, const int32_t *lens, float *d_in, int B, int T, int F,
                        int M, void *stream);

/* Stand-alone mask tail (enhance_model.py:157-164) forward / backward, for callers that
 * need `enhance_out` itself (e.g. the L1 mask loss at :166-172). */
int re2e_mask_apply_fwd(const float *logits, const float *mag, const int32_t *lens, float *enh,
                        int B, int T, int F, void *stream);
int re2e_mask_apply_bwd(const float *d_enh, const float *logits, const float *mag,
                        const int32_t *lens, float *d_logits, int B, int T, int F, void *stream);

/* CMVN statistics (feat_model.py:62-90 compute_cmvn): per-mel sum and sum of squares over the
 * valid frames t < lens[b] of Y (B,T,M); ACCUMULATES into sum[M], sumsq[M] (fp64 on device)
 * and frames[1] (int64).  Next-row N3 of SURVEY.md section 8f. */
int re2e_cmvn_stats(const float *Y, const int32_t *lens, double *sum, double *sumsq,
                    long long *frames, int B, int T, int M, void *stream);

/* --------------------------------------------------------------------------------------------
 * AttLoc.  Replaces model/e2e_attention.py:236-299 (forward) and its autograd backward.
 * Shapes: enc_h (B,Th,D)  pre (B,Th,A)  dec_z (B,Z)  att_prev,w (B,Th)  c (B,D)
 *         W_enc (A,D) b_enc (A)  W_dec (A,Z)  W_att (A,C)  W_conv (C,K) K = 2*filts+1
 *         gvec (A)  gvec_b (1)
 * ------------------------------------------------------------------------------------------ */

/* Uniform initial alignment, zero padded (e2e_attention.py:264-268). hlens on device. */
int re2e_attloc_init_att(const int32_t *hlens, float *att_prev, int B, int Th, void *stream);

/* One attention step (e2e_attention.py:258-299).  dec_z == NULL means zeros (:258-259).
 * mlp_dec (dec_z @ W_dec^T, :278) is computed inside the kernel (split over the CTAs of a cluster, exchanged
 * through distributed shared memory).  Optional outputs (NULL when not needed):
 *   dec_proj (B,A) = dec_z @ W_dec^T
 *   conv (B,Th,C)  = loc_conv(att_prev)                               (saved for the backward)
 *   xsave (B,Th,A) = tanh(mlp_att(conv) + pre + dec_proj)             (saved for the backward) */
int re2e_attloc_step_fwd(const float *pre, const float *enc_h, const float *dec_z,
                         const float *att_prev, const float *W_dec, const float *W_att,
                         const float *W_conv, const float *gvec, const float *gvec_b,
                         float scaling, float *c, float *w, float *dec_proj, float *conv, float *xsave,
                         int B, int Th, int D, int A, int Z, int C, int K, void *stream);

/* Backward of one step.  Inputs dc (B,D) / dw (B,Th) may be NULL (= zero); xsave / conv / w are the
 * tensors saved by the forward.
 *   d_pre (B,Th,A)       (+)= dE/dpre   accumulate_pre != 0: TMA reduce-add into d_pre (accumulated
 *                             across steps); == 0: plain store (first backward step, no zero-fill)
 *   d_decproj (B,A)       = dE/d(dec_z @ W_dec^T)        (kept for dW_dec = sum_steps d_decproj^T dec_z)
 *   d_dec_z (B,Z)         = d_decproj @ W_dec            (NULL to skip: first decoder step has no dec_z).  Read from
 *                           W_decT (Z,A) = W_dec^T, a 16 B aligned copy the caller builds once per decoder loop:
 *                           each cluster re-reads the whole matrix every step, the transposed rows make that
 *                           read fully coalesced (required when d_dec_z != NULL)
 *   d_att_prev (B,Th)     = dE/d att_prev                (NULL to skip, e.g. first decoder step)
 *   acc_slots             parameter-gradient accumulators, n_slots >= re2e_attloc_acc_slots(...) private slots of
 *                         re2e_attloc_acc_floats(A,C,K) floats each, layout [dW_att A*C | dW_conv C*K | dgvec A |
 *                         dgvec_b 1]; zero them once per decoder loop, every step ADDS into them without atomics
 *                         (one slot per CTA), re2e_attloc_acc_reduce sums the slots after the loop.
 * d enc_h is NOT produced here: sum_i w_i (x) dc_i is a rank-(#steps) update applied once by
 * re2e_attloc_enc_grad after the loop (no per-step read-modify-write of (B,Th,D)). */
size_t re2e_attloc_acc_floats(int A, int C, int K);
int re2e_attloc_acc_slots(int B, int Th, int D, int A, int Z, int C, int K);
int re2e_attloc_step_bwd(const float *dc, const float *dw, const float *xsave, const float *enc_h,
                         const float *att_prev, const float *w, const float *conv, const float *W_dec,
                         const float *W_decT, const float *W_att, const float *W_conv, const float *gvec,
                         float scaling,
                         float *d_pre, int accumulate_pre, float *d_decproj, float *d_dec_z,
                         float *d_att_prev, float *acc_slots, int n_slots, int B, int Th, int D, int A,
                         int Z, int C, int K, void *stream);
int re2e_attloc_acc_reduce(const float *acc_slots, int n_slots, float *out, int A, int C, int K,
                           void *stream);

/* d_enc_h[b,t,:] (+)= sum_i w_all[i,b,t] * dc_all[i,b,:]   (i < steps); accumulate != 0 adds. */
int re2e_attloc_enc_grad(const float *w_all, const float *dc_all, float *d_enc_h, int steps,
                         int B, int Th, int D, int accumulate, void *stream);

/* The attention decoder loop as ONE persistent cluster kernel per direction (csrc/attloc_loop.cu).  Replaces the S
 * consecutive calls `att_c, att_w = self.att(hpad, hlen, z_list[0], att_w)` of Decoder.forward
 * (model/e2e_decoder.py:114-122), i.e. S x model/e2e_attention.py:258-299 with the alignment fed back, and the
 * autograd backward of that chain.  Step-indexed tensors are (S, ...):
 *   dec_proj (S,B,A)  = dec_z_s @ W_dec^T for every step (row 0 zeros when the first dec_z is None): the caller
 *                       forms it with ONE dense product, which is possible whenever the decoder states of all steps
 *                       exist before the loop (the joint-step hot path feeds them; a teacher-forced decoder whose
 *                       recurrence does not see the context).  When z_s depends on c_{s-1} (LSTMCell fed with the
 *                       context, Decoder.forward) use the per-step entry points above.
 *   att_init (B,Th)   the alignment fed to step 0 (re2e_attloc_init_att)
 *   c_all (S,B,D), w_all (S,B,Th)   outputs of every step;  conv_all (S,B,Th,C) saved for the backward (NULL: skip)
 * Backward: dc_all (S,B,D) / dw_all (S,B,Th) are the incoming gradients of c_all / w_all (either may be NULL = zeros);
 * the gradient flowing back through the fed-back alignment is kept inside the kernel.
 *   d_pre (B,Th,A)      = sum over steps (written, not accumulated into)
 *   d_decproj (S,B,A)   = dE/d dec_proj           (d dec_z = d_decproj @ W_dec and dW_dec are dense products)
 *   acc_slots           n_slots >= re2e_attloc_loop_slots(...) slots of re2e_attloc_acc_floats floats, WRITTEN (no
 *                       zero-fill needed), summed by re2e_attloc_acc_reduce
 * d enc_h: re2e_attloc_enc_grad(w_all, dc_all, ...) as for the per-step path.
 * re2e_attloc_loop_supported: 1 when the shape fits (the CTA's frame range of one utterance resident on chip for
 * the whole loop), else 0 -- callers then use the per-step entry points. */
int re2e_attloc_loop_supported(int S, int B, int Th, int D, int A, int C, int K);
int re2e_attloc_loop_slots(int S, int B, int Th, int D, int A, int C, int K);
int re2e_attloc_loop_fwd(const float *pre, const float *enc_h, const float *dec_proj, const float *att_init,
                         const float *W_att, const float *W_conv, const float *gvec, const float *gvec_b,
                         float scaling, float *c_all, float *w_all, float *conv_all, int S, int B, int Th, int D,
                         int A, int C, int K, void *stream);
int re2e_attloc_loop_bwd(const float *pre, const float *enc_h, const float *dec_proj, const float *att_init,
                         const float *w_all, const float *conv_all, const float *dc_all, const float *dw_all,
                         const float *W_att, const float *W_conv, const float *gvec, float scaling, float *d_pre,
                         float *d_decproj, float *acc_slots, int n_slots, int S, int B, int Th, int D, int A,
                         int C, int K, void *stream);

/* Batch-sized ("skinny", M <= a few hundred rows) fp32 products on the per-step path:
 *   out[M,N] (+)= X[M,K] @ W[N,K]^T   (re2e_skinny_nt)   dec_proj = dec_z @ W_dec^T  (mlp_dec, :278)
 *   out[M,N] (+)= X[M,K] @ W[K,N]     (re2e_skinny_nn)   d_dec_z  = d_decproj @ W_dec */
int re2e_skinny_nt(const float *X, const float *W, float *out, int M, int N, int K, int accumulate,
                   void *stream);
int re2e_skinny_nn(const float *X, const float *W, float *out, int M, int N, int K, int accumulate,
                   void *stream);

/* LSTMCell step of the attention decoder (model/e2e_decoder.py:128, torch.nn.LSTMCell, gate order i,f,g,o), fused
 * pointwise part (csrc/lstm.cu).  The caller forms the recurrent products with re2e_skinny_nt into `gates` (B,4Z):
 *   gates = context @ W_ih[:, Z:]^T + h_prev @ W_hh^T ;  egate (B,4Z, optional) = embed(y) @ W_ih[:, :Z]^T + b_ih + b_hh
 * (the embedding half of every position comes from ONE dense product before the loop).
 *   fwd: gates <- gate activations (i,f,g,o) in place (saved for the backward); c_out, h_out (B,Z).  c_prev NULL = zeros.
 *   bwd: dh / dc = gradients arriving at (h_out, c_out), NULL = zero; dgates (B,4Z) w.r.t. the pre-activation gates
 *        (d context = dgates @ W_ih[:, Z:], d h_prev = dgates @ W_hh via re2e_skinny_nn; weight gradients of all steps are
 *        two dense products after the loop); dc_prev (B,Z). */
/* out[M,N] (+)= X[M,K] @ W[N,K]^T for a batch-sized M and long N / K (the decoder's per-position recurrent products,
 * N or K = 4Z): one CTA per 8 output columns so that all SMs stream the weight matrix once, reduction staged in chunks
 * (128-bit staging when K % 4 == 0 and X, W are 16 B aligned, scalar staging otherwise).  The backward uses it on transposed weight copies made once per loop. */
int re2e_batch_nt(const float *X, const float *W, const float *bias /* (N) or NULL */, float *out, int M, int N, int K,
                  int accumulate, void *stream);
/* Scheduled sampling (model/e2e_decoder.py:123-127): the next input token of every batch row, chosen on the device.
 *   *flag != 0: tok[m] = argmax_n (X[m,:] . W[n,:] + bias[n])   (lowest n among equal values; -0 and +0 are equal)
 *   *flag == 0: tok unchanged (the caller pre-fills the teacher tokens)
 * X (M,K) top-layer decoder state, W (N,K) output layer, bias (N) or NULL; flag: device int32 (read by the kernel, so one
 * captured graph serves any draw pattern); tok: device int32 (M).  The logits are never written.
 * ws: re2e_sample_tokens_ws_bytes(M) bytes, zero before the first call; every call leaves it zero (graph-replayable with
 * no memset).  One call at a time per ws. */
int re2e_sample_tokens_ws_bytes(int M);
int re2e_sample_tokens(const float *X, const float *W, const float *bias, const int32_t *flag, int32_t *tok,
                       unsigned long long *ws, int M, int N, int K, void *stream);
/* One LSTMCell position in one launch (after the embedding half): gates = egate + ctx @ Wcat[:, :D]^T + h_prev @
 * Wcat[:, D:]^T, then the cell's pointwise arithmetic -> act (B,4Z) gate activations (kept for the backward), c_out, h_out
 * (B,Z).  Wcat (4Z, D+Z) = [W_ih[:, E:] | W_hh].  Clusters of 4 CTAs split the reduction (deterministic order).
 * re2e_lstm_step_bwd: d_ctx (B,D) | d_hprev (B,Z) = dgates (B,4Z) @ Wcat, given WcatT (D+Z, 4Z) = Wcat^T (clusters of 8).
 * Supported: D % 4 == Z % 4 == 0, D, Z <= 640, 16 B aligned operands; else RE2E_E_UNSUPPORTED (callers then compose
 * re2e_batch_nt + re2e_lstm_pointwise_*). */
int re2e_lstm_step_supported(int B, int D, int Z);
int re2e_lstm_step_fwd(const float *ctx, const float *h_prev, const float *c_prev, const float *Wcat, const float *egate,
                       const int32_t *egate_row /* row of egate per batch row (token lookup), NULL: row m */, float *act,
                       float *c_out, float *h_out, int B, int D, int Z, void *stream);
int re2e_lstm_step_bwd(const float *dgates, const float *WcatT, float *d_ctx, float *d_hprev, int B, int D, int Z,
                       void *stream);
int re2e_lstm_pointwise_fwd(float *gates, const float *egate, const float *c_prev, float *c_out, float *h_out, int B,
                            int Z, void *stream);
int re2e_lstm_pointwise_bwd(const float *act, const float *c_prev, const float *c_new, const float *dh, const float *dc,
                            float *dgates, float *dc_prev, int B, int Z, void *stream);

/* fp32-accurate dense GEMM on tcgen05 tensor cores (3xTF32 split, fp32 TMEM accumulator; csrc/gemm_tc.cu):
 *   C[M,N] (+)= Aop[M,K] * Bop[N,K]^T (+ bias[N])
 * a_mn = 0: A stored [M][lda] (K contiguous)   a_mn = 1: A stored [K][lda] (M contiguous);  same for B / N.
 * Replaces the cuBLAS sgemm behind nn.Linear on the path: ctc_lo (model/e2e_ctc.py:51), mlp_enc
 * (model/e2e_attention.py:256) and their backward products (dX = g W : b_mn = 1;  dW = g^T X : a_mn = b_mn = 1).
 * lda, ldb multiples of 4 elements, A and B 16 B aligned (TMA); ldc >= N. */
int re2e_gemm_tf32x3(const float *A, int lda, int a_mn, const float *B, int ldb, int b_mn, float *C,
                     int ldc, const float *bias, int M, int N, int K, int accumulate, void *stream);

/* out[c] = sum_r X[r*ld + c]  (rows x cols, row pitch ld): the bias gradient of a dense layer (db = column sums of dY;
 * ctc_lo, model/e2e_ctc.py:28, and mlp_enc, model/e2e_attention.py:214).  Deterministic two-pass reduction;
 * partial: scratch of re2e_colsum_blocks(rows) * cols floats. */
int re2e_colsum_blocks(int rows);
int re2e_colsum(const float *X, long long ld, int rows, int cols, float *partial, float *out, void *stream);

/* --------------------------------------------------------------------------------------------
 * CTC.  Replaces the warp_ctc.CTCLoss call at model/e2e_ctc.py:30,63 (softmax + alpha/beta +
 * gradient; arithmetic of the un-vendored warpctc_pytorch) and F.log_softmax at :75.
 * logits: raw activations, element (b,t,v) at logits[b*stride_b + t*stride_t + v]
 *         ((B,Th,V) contiguous: stride_b = Th*V, stride_t = V; warp-ctc's (Th,B,V): stride_b = V,
 *         stride_t = B*V).  labels: flat int32, utterance b at labels[label_offs[b] ..+label_lens[b]).
 * blank = 0 in the reference.  Smax = 2*max(label_lens)+1.
 * ------------------------------------------------------------------------------------------ */
size_t re2e_ctc_ws_bytes(int B, int Th, int V, int Umax);

/* Forward: nll[b] = -log p(y_b | x_b[:input_lens[b]]), loss[0] = sum_b nll[b] / B  (size_average
 * over the batch, e2e_ctc.py:30).  Fills ws with lse (B,Th), alpha/beta (B,Th,Smax) for bwd. */
int re2e_ctc_loss_fwd(const float *logits, long long stride_b, long long stride_t,
                      const int32_t *labels, const int32_t *label_offs, const int32_t *label_lens,
                      const int32_t *input_lens, int blank, float *nll, float *loss, void *ws,
                      size_t ws_bytes, int B, int Th, int V, int Umax, void *stream);

/* Backward: grad[b,t,v] = gscale * (softmax(x)[v] - occupancy[b,t,v]) for t < input_lens[b], else 0,
 * gscale = (grad_out ? grad_out[0] : 1) / B.   grad has the same strides as logits. */
int re2e_ctc_loss_bwd(const float *logits, long long stride_b, long long stride_t,
                      const int32_t *labels, const int32_t *label_offs, const int32_t *label_lens,
                      const int32_t *input_lens, int blank, const float *nll, const float *grad_out,
                      const void *ws, size_t ws_bytes, float *grad, int B, int Th, int V, int Umax,
                      void *stream);

/* Forced alignment: the single most likely path of each transcript through its blank-interleaved lattice (Viterbi,
 * max-plus forward recursion + backtrace on the device; no reference counterpart).  Inputs as re2e_ctc_loss_fwd, the
 * same workspace (re2e_ctc_ws_bytes); logits may also be log-probabilities (a per-frame constant does not move the path).
 * Two launches (the loss's log-sum-exp / lattice gather, then one warp per utterance); no host synchronisation.
 *   states (B,Th) int32   lattice state s in [0, 2U] of every frame (even = blank, odd 2u+1 = label u)
 *   tokens (B,Th) int32   blank or labels[u] for that state
 *   spans (B,Umax,2)      first and last frame of each label
 *   score (B) fp32        log-probability of the path under softmax(logits)
 * Tie rule: on equal scores a state prefers staying (s), then s-1, then s-2; at the last frame S-1 (final blank) is
 * preferred to S-2.  Frames t >= min(input_lens[b], Th), labels u >= label_lens[b] and every entry of an infeasible
 * utterance (input_lens[b] < U + adjacent repeats) are -1; an infeasible utterance scores -inf.  U = 0 gives the all-blank
 * path; input_lens[b] <= 0 gives score 0 if U = 0, else -inf.
 * Umax <= 255 and Th up to ~1550..1680 (the backpointers, 128 B per frame, live in shared memory), else
 * RE2E_E_UNSUPPORTED before anything is launched. */
int re2e_ctc_align(const float *logits, long long stride_b, long long stride_t, const int32_t *labels,
                   const int32_t *label_offs, const int32_t *label_lens, const int32_t *input_lens, int blank,
                   int32_t *states, int32_t *tokens, int32_t *spans, float *score, void *ws, size_t ws_bytes, int B,
                   int Th, int V, int Umax, void *stream);

/* out = log_softmax(logits, dim=-1) over rows of length V (e2e_ctc.py:68-75 after ctc_lo);
 * best (optional, int32 per row) = argmax_v  ("CTC best-path alignment", lowest index on ties). */
int re2e_log_softmax(const float *logits, float *out, int32_t *best, long long rows, int V,
                     void *stream);

/* Batched CTC prefix scoring (model/e2e_ctc.py:109-155, one call per live hypothesis there).
 * lpz (T,V) log-probs of one utterance; H hypotheses x Ccand candidates each.
 *   r_prev (H,T,2); cs (H,Ccand) int32 candidate ids; last (H) int32 = y[-1]; out_len (H) = len(y)-1
 *   log_psi (H,Ccand); r_new (H,Ccand,T,2)  (rows < max(out_len,1)-1 are set to logzero). */
int re2e_ctc_prefix_score(const float *lpz, const float *r_prev, const int32_t *cs,
                          const int32_t *last, const int32_t *out_len, float *log_psi,
                          float *r_new, int T, int V, int H, int Ccand, int blank, int eos,
                          void *stream);

/* Cross-entropy of the attention decoder (model/e2e_decoder.py:155-157: F.cross_entropy, ignore_index, mean) in one pass
 * per direction.  logits (rows, V) with row pitch ld floats; target int64 (rows); rows whose target is ignore_id (or out
 * of range) contribute nll = 0 / a zero gradient row.  fwd: lse (rows), nll (rows) = lse - logits[target], best (rows)
 * = arg-max (NULL to skip; th_accuracy of model/e2e_common.py:198-205).  bwd: dlogits (rows, V) pitch ldd =
 * (softmax - onehot) * *scale, scale a device scalar (incoming gradient / number of labelled rows). */
int re2e_cross_entropy_fwd(const float *logits, long long ld, const long long *target, long long ignore_id, long long rows,
                           int V, float *lse, float *nll, int32_t *best, void *stream);
int re2e_cross_entropy_bwd(const float *logits, long long ld, const long long *target, long long ignore_id, long long rows,
                           int V, const float *lse, const float *scale, float *dlogits, long long ldd, void *stream);

/* ------------------------------------------------------------------------------------------
 * Beam search, one output position for all W = beam hypothesis rows (model/e2e_decoder.py:233-314; SURVEY 8f N1/N2).
 * The reference advances one hypothesis at a time (beam x B=1 calls) and scores CTC prefixes in a host loop over T;
 * here a position is gather -> re2e_attloc_step_fwd -> re2e_lstm_step_fwd -> re2e_batch_nt (output layer) ->
 * re2e_log_softmax_topk -> re2e_ctc_prefix_score -> re2e_beam_joint over static buffers (graph-replayable).
 *
 * re2e_beam_gather: for each of nseg state tensors, dst[s][m, :] = src[s][parent[m] (, cand[m]), :] (row_floats[s] floats;
 *   sub_count[s] > 0: the source has that many candidate sub-rows per parent row, e.g. the CTC states (W, ctc_beam, T, 2)).
 * re2e_log_softmax_topk: per row log-softmax (optionally written to `full` (rows,V)) and its k largest entries, sorted
 *   descending, ties to the lower index -- what torch.topk(log_softmax(x), k) returns (model/e2e_decoder.py:262,276).
 *   V <= 8192 and k <= 32, else RE2E_E_UNSUPPORTED.
 * re2e_beam_joint: local = w_att * att_top + w_ctc * (log_psi - psi_prev[row]) (log_psi NULL: local = att_top), the `beam`
 *   best of the Cb <= 32 candidates per row; out (3, W, beam) fp32 = {row score + local, token id, candidate index}
 *   (model/e2e_decoder.py:284-292). */
/* Initial working state of a search (model/e2e_decoder.py:205-231): z_in = c_in = 0 (W,Z), a_in uniform over Th (W,Th),
 * r_in (W,Th,2) = CTCPrefixScore.initial_state (model/e2e_ctc.py:95-107; r_in / psi_in / lpz NULL without CTC), psi_in = 0,
 * ctl = {parent 0, candidate 0, token sos, position 0}, sc = 0, state = {1 live hypothesis, position 0}. */
int re2e_beam_init(float *z_in, float *c_in, float *a_in, float *r_in, float *psi_in, const float *lpz, int32_t *ctl,
                   float *sc, int32_t *state, int W, int Z, int Th, int V, int blank, int sos, void *stream);
int re2e_beam_gather(const int32_t *parent, const int32_t *cand, int W, int nseg, const float *const *src,
                     float *const *dst, const int *row_floats, const int *sub_count, void *stream);
int re2e_log_softmax_topk(const float *logits, long long rows, int V, int k, float *full, float *vals, int32_t *ids,
                          void *stream);
int re2e_beam_joint(const float *att_top, const int32_t *ids, const float *log_psi, const float *psi_prev, const float *sc,
                    float w_att, float w_ctc, int W, int Cb, int beam, float *out, void *stream);
/* Merge of one position on the device (model/e2e_decoder.py:296-333): the `beam` best of the first n_live x beam
 * candidates of `out` (stable descending order), recorded in hist[pos] (4, beam) = {score, parent row, token, candidate
 * index} for the host's hypothesis bookkeeping; the winners whose token is not <eos> become the rows of position pos+1
 * (ctl (4,W) int32 = parent, candidate, token, position; sc (W) row scores), none survive at pos = maxlen-1.
 * state int32[2] = {n_live, pos} is advanced.  With this the host reads the history back every few positions instead of
 * synchronising at each one.  W, beam <= 32. */
int re2e_beam_merge(const float *out, int32_t *state, int32_t *ctl, float *sc, float *hist, int W, int beam, int eos,
                    int maxlen, void *stream);
/* re2e_beam_joint + re2e_beam_merge + re2e_beam_gather (for the NEXT position, with the rows just chosen) in one launch
 * of one CTA: the tail of a position is a strictly serial chain of three tiny kernels, i.e. three launch latencies. */
int re2e_beam_advance(const float *att_top, const int32_t *ids, const float *log_psi, const float *psi_prev, float *sc,
                      float w_att, float w_ctc, int W, int Cb, int beam, int32_t *state, int32_t *ctl, float *hist,
                      int eos, int maxlen, int nseg, const float *const *src, float *const *dst, const int *row_floats,
                      const int *sub_count, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* RE2E_B200_H_ */
