"""Oracle (CPU restatement) of the CTC pieces.  TEST INFRASTRUCTURE ONLY.

Follows /root/reference/model/e2e_ctc.py:
  * CTC.forward ......... :33-66   (ctc_lo Linear, always-on F.dropout, (T,B,V) logits,
                                    loss = sum_b nll_b / B, blank = 0)
  * CTC.log_softmax ..... :68-75
  * CTCPrefixScore ...... :78-155  (Watanabe et al. Alg. 2, label-vectorised)

The loss arithmetic itself is NOT in the reference tree: it is delegated to the
third-party ``warpctc_pytorch`` (un-vendored, un-pinned -> PARITY UNPINNED for
this piece).  It is restated here twice, independently:
  (1) ``ctc_loss_torch``  -- torch.nn.functional.ctc_loss on log_softmax (autograd grads);
  (2) ``ctc_alpha_beta``  -- the published alpha/beta recursion (Graves et al. 2006,
      eqs. 6-8, 10-11, 16) in float64 numpy with the closed-form gradient
      softmax - occupancy, which is what warp-ctc documents computing.
tests/test_oracle.py checks (1) == (2).  Gradients follow autograd semantics
(scaled by grad_output), see SURVEY.md section 8c caveat.
"""
import numpy as np
import torch
import torch.nn.functional as F


# ----------------------------------------------------------------------------- loss
def ctc_loss_torch(logits_btv, hlens, ys, blank=0):
    """logits (B,Th,V) raw activations; ys list of 1-D int tensors. Returns (loss(1,), nll(B,))."""
    B = logits_btv.shape[0]
    lp = F.log_softmax(logits_btv.transpose(0, 1), dim=2)
    olens = torch.tensor([int(y.numel()) for y in ys], dtype=torch.long)
    flat = torch.cat([y.reshape(-1) for y in ys]).long() if len(ys) else torch.zeros(0, dtype=torch.long)
    nll = F.ctc_loss(lp, flat, torch.as_tensor(list(map(int, hlens)), dtype=torch.long), olens,
                     blank=blank, reduction="none", zero_infinity=False)
    return (nll.sum() / B).view(1), nll


def ctc_module_forward(ctc_lo_w, ctc_lo_b, hs_pad, hlens, ys_pad, dropout_rate=0.0, ignore_id=-1):
    """e2e_ctc.py:33-66."""
    ys = [y[y != ignore_id] for y in ys_pad]
    ys_hat = F.linear(F.dropout(hs_pad, p=dropout_rate), ctc_lo_w, ctc_lo_b)
    loss, _ = ctc_loss_torch(ys_hat, hlens, ys)
    return loss


def log_softmax(ctc_lo_w, ctc_lo_b, hs_pad):
    """e2e_ctc.py:68-75."""
    return F.log_softmax(F.linear(hs_pad, ctc_lo_w, ctc_lo_b), dim=2)


def _logsumexp(*xs):
    m = max(xs)
    if m == -np.inf:
        return -np.inf
    return m + np.log(sum(np.exp(x - m) for x in xs))


def ctc_alpha_beta(logits_tv, labels, blank=0):
    """One utterance. logits (T,V) float, labels 1-D ints (may be empty).
    Returns dict(nll, grad (T,V) = d nll / d logits, alpha, beta (T,S) log-domain, lp (T,V))."""
    x = np.asarray(logits_tv, dtype=np.float64)
    T, V = x.shape
    m = x.max(axis=1, keepdims=True)
    lp = x - (m + np.log(np.exp(x - m).sum(axis=1, keepdims=True)))
    lab = [int(v) for v in labels]
    U = len(lab)
    S = 2 * U + 1
    ext = [blank] * S
    for u in range(U):
        ext[2 * u + 1] = lab[u]
    NEG = -np.inf
    alpha = np.full((T, S), NEG)
    beta = np.full((T, S), NEG)
    alpha[0, 0] = lp[0, ext[0]]
    if S > 1:
        alpha[0, 1] = lp[0, ext[1]]
    for t in range(1, T):
        for s in range(S):
            a = alpha[t - 1, s]
            b = alpha[t - 1, s - 1] if s >= 1 else NEG
            c = alpha[t - 1, s - 2] if (s >= 2 and ext[s] != blank and ext[s] != ext[s - 2]) else NEG
            alpha[t, s] = _logsumexp(a, b, c) + lp[t, ext[s]]
    beta[T - 1, S - 1] = lp[T - 1, ext[S - 1]]
    if S > 1:
        beta[T - 1, S - 2] = lp[T - 1, ext[S - 2]]
    for t in range(T - 2, -1, -1):
        for s in range(S):
            a = beta[t + 1, s]
            b = beta[t + 1, s + 1] if s + 1 < S else NEG
            c = beta[t + 1, s + 2] if (s + 2 < S and ext[s] != blank and ext[s] != ext[s + 2]) else NEG
            beta[t, s] = _logsumexp(a, b, c) + lp[t, ext[s]]
    ll = _logsumexp(alpha[T - 1, S - 1], alpha[T - 1, S - 2] if S > 1 else NEG)
    grad = np.exp(lp)
    for t in range(T):
        for s in range(S):
            v = alpha[t, s] + beta[t, s]
            if v > NEG:
                grad[t, ext[s]] -= np.exp(v - lp[t, ext[s]] - ll)
    return {"nll": -ll, "grad": grad, "alpha": alpha, "beta": beta, "lp": lp}


def best_path(lp_btv):
    """north_star 'CTC alignments': argmax_v log_softmax(h)[b,t,:] (SURVEY.md 8a-4)."""
    return lp_btv.argmax(dim=2)


# ----------------------------------------------------------------------------- prefix score
class CTCPrefixScoreOracle(object):
    """Restatement of e2e_ctc.py:78-155 in numpy (logzero = -1e10).  ``dtype``: float32 is the reference's own
    arithmetic; float64 gives the high-precision truth the device kernel is judged against."""

    def __init__(self, x, blank, eos, dtype=np.float32):
        self.logzero = -10000000000.0
        self.blank = blank
        self.eos = eos
        self.dtype = dtype
        self.input_length = len(x)
        self.x = np.asarray(x, dtype=dtype)

    def initial_state(self):
        """:95-107 -- r[t,1] = cumulative blank log-prob, r[t,0] = logzero."""
        T = self.input_length
        r = np.full((T, 2), self.logzero, dtype=self.dtype)
        acc = self.dtype(0.0)
        for t in range(T):
            acc = self.dtype(acc + self.x[t, self.blank]) if t > 0 else self.x[0, self.blank]
            r[t, 1] = acc
        return r

    def __call__(self, y, cs, r_prev):
        """:109-155.  Rows r[0 .. start-2] are left uninitialised by the reference
        (np.ndarray); here they are set to logzero -- do not compare them."""
        T = self.input_length
        cs = np.asarray(cs)
        n = len(cs)
        output_length = len(y) - 1
        r = np.full((T, 2, n), self.logzero, dtype=self.dtype)
        xs = self.x[:, cs]
        if output_length == 0:
            r[0, 0] = xs[0]
            r[0, 1] = self.logzero
        r_sum = np.logaddexp(r_prev[:, 0], r_prev[:, 1]).astype(self.dtype)
        last = y[-1]
        log_phi = np.repeat(r_sum[:, None], n, axis=1)
        if output_length > 0:
            for i in range(n):
                if cs[i] == last:
                    log_phi[:, i] = r_prev[:, 1]
        start = max(output_length, 1)
        log_psi = r[start - 1, 0].copy()
        for t in range(start, T):
            r[t, 0] = np.logaddexp(r[t - 1, 0], log_phi[t - 1]) + xs[t]
            r[t, 1] = np.logaddexp(r[t - 1, 0], r[t - 1, 1]) + self.x[t, self.blank]
            log_psi = np.logaddexp(log_psi, log_phi[t - 1] + xs[t])
        eos_pos = np.where(cs == self.eos)[0]
        if len(eos_pos) > 0:
            log_psi[eos_pos] = r_sum[-1]
        return log_psi.astype(self.dtype), np.moveaxis(r, 2, 0), start
