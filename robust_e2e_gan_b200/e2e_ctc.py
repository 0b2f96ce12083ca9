"""Drop-in ``CTC`` and ``CTCPrefixScore`` (reference: model/e2e_ctc.py) on sm_100a kernels.

``CTC(odim, eprojs, dropout_rate)`` keeps the reference's constructor, ``ctc_lo`` Linear
(state_dict keys ``ctc_lo.weight`` / ``ctc_lo.bias``), ``forward(hs_pad, hlens, ys_pad)`` -> (1,)
loss = sum_b nll_b / B with blank = 0, and ``log_softmax(hs_pad)``.  The softmax + alpha/beta +
gradient that the reference delegates to the third-party ``warpctc_pytorch`` (e2e_ctc.py:11,30,63)
run in csrc/ctc.cu on the (B,Th,V) logits in place (no (Th,B,V) transpose copy).  Gradients follow
autograd semantics (scaled by grad_output).  ``ctc_forced_align`` / ``CTC.forced_align`` add what the reference
lacks: the forced (Viterbi) alignment of a given transcript, computed on the device.
"""
import collections

import numpy as np
import torch
import torch.nn.functional as F

from . import _lib
from .linear import linear as _linear_tc


class PreparedTargets(object):
    """Flat int32 labels + offsets/lengths already on the device (skips the per-call host parse)."""

    def __init__(self, labels, offs, lens, umax, nutt):
        self.labels, self.offs, self.lens, self.umax, self.nutt = labels, offs, lens, umax, nutt


def prepare_targets(ys, device, ignore_id=-1):
    """ys: padded LongTensor (B,Lmax) with ``ignore_id`` padding, or a list of 1-D tensors
    (model/e2e_ctc.py:43 ``ys = [y[y != ignore_id] for y in ys_pad]``).  One D2H copy at most."""
    if torch.is_tensor(ys):
        rows = ys.detach().cpu().numpy()
        seqs = [r[r != ignore_id] for r in rows]
    else:
        sizes = [int(y.numel()) for y in ys]
        flat = torch.cat([y.reshape(-1) for y in ys]).detach().cpu().numpy() if sum(sizes) else np.zeros(0, np.int64)
        seqs, o = [], 0
        for n in sizes:
            r = flat[o:o + n]
            seqs.append(r[r != ignore_id])
            o += n
    lens = np.array([len(s) for s in seqs], dtype=np.int32)
    offs = np.zeros(len(seqs), dtype=np.int32)
    if len(seqs) > 1:
        offs[1:] = np.cumsum(lens[:-1])
    flat = np.concatenate(seqs).astype(np.int32) if lens.sum() else np.zeros(1, np.int32)
    dev = torch.device(device)
    to = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev, non_blocking=True)
    return PreparedTargets(to(flat), to(offs), to(lens), int(lens.max()) if len(lens) else 0, len(seqs))


class _CTCLossFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits, hlens_dev, tgt, blank):
        L = _lib.lib()
        x = logits if _strided_ok(logits) else _lib.f32c(logits)
        B, Th, V = x.shape
        dev = x.device
        sb, st = x.stride(0), x.stride(1)
        nbytes = int(L.re2e_ctc_ws_bytes(B, Th, V, tgt.umax))
        ws = torch.empty(nbytes, device=dev, dtype=torch.uint8)
        nll = torch.empty(B, device=dev, dtype=torch.float32)
        loss = torch.empty(1, device=dev, dtype=torch.float32)
        with _lib.on(dev):
            _lib.check(L.re2e_ctc_loss_fwd(_lib.ptr(x), sb, st, _lib.ptr(tgt.labels), _lib.ptr(tgt.offs),
                                           _lib.ptr(tgt.lens), _lib.ptr(hlens_dev), int(blank), _lib.ptr(nll),
                                           _lib.ptr(loss), _lib.ptr(ws), nbytes, B, Th, V, tgt.umax,
                                           _lib.stream_ptr()), "re2e_ctc_loss_fwd")
        ctx.save_for_backward(x, hlens_dev, tgt.labels, tgt.offs, tgt.lens, nll, ws)
        ctx.meta = (int(blank), tgt.umax)
        ctx.mark_non_differentiable(nll)
        return loss, nll

    @staticmethod
    def backward(ctx, g, _g_nll):
        L = _lib.lib()
        x, hlens_dev, labels, offs, lens, nll, ws = ctx.saved_tensors
        blank, umax = ctx.meta
        B, Th, V = x.shape
        sb, st = x.stride(0), x.stride(1)
        # same (possibly row-padded) layout as the logits: the tcgen05 backward GEMMs read it through TMA
        grad = torch.empty_strided((B, Th, V), x.stride(), device=x.device, dtype=torch.float32)
        g = _lib.f32c(g.reshape(-1)[:1], x.device)
        with _lib.on(x.device):
            _lib.check(L.re2e_ctc_loss_bwd(_lib.ptr(x), sb, st, _lib.ptr(labels), _lib.ptr(offs),
                                           _lib.ptr(lens), _lib.ptr(hlens_dev), blank, _lib.ptr(nll), _lib.ptr(g),
                                           _lib.ptr(ws), ws.numel(), _lib.ptr(grad), B, Th, V, umax,
                                           _lib.stream_ptr()), "re2e_ctc_loss_bwd")
        return grad, None, None, None


def _strided_ok(t):
    """fp32 CUDA (B,Th,V) with unit inner stride and non-overlapping rows (a row-padded GEMM output)."""
    return (t.dtype == torch.float32 and t.is_cuda and t.dim() == 3 and t.stride(2) == 1
            and t.stride(1) >= t.shape[2] and t.stride(0) >= t.stride(1) * t.shape[1])


def _device_hlens(hlens, dev):
    """int32 CUDA lengths from host ints or a CUDA int tensor (the latter without a copy or a synchronisation)."""
    if torch.is_tensor(hlens) and hlens.is_cuda:
        return hlens.to(torch.int32).contiguous()
    return torch.from_numpy(np.fromiter((int(h) for h in hlens), dtype=np.int32)).to(dev, non_blocking=True)


def ctc_loss(logits, hlens, targets, blank=0):
    """logits (B,Th,V) raw activations on CUDA; hlens host ints (or int32 CUDA tensor);
    targets: PreparedTargets or anything prepare_targets accepts.  Returns (loss (1,), nll (B,))."""
    dev = logits.device
    if not isinstance(targets, PreparedTargets):
        targets = prepare_targets(targets, dev)
    hl = _device_hlens(hlens, dev)
    assert targets.nutt == logits.shape[0] and hl.numel() == logits.shape[0]
    return _CTCLossFunction.apply(logits, hl, targets, blank)


CTCAlignment = collections.namedtuple("CTCAlignment", ["states", "tokens", "spans", "score"])
CTCAlignment.__doc__ = """Forced CTC alignment of a batch (``ctc_forced_align``); -1 marks padding and infeasible
    utterances.
    states (B,Th) int32  lattice state per frame (2u: blank before label u, 2u+1: label u)
    tokens (B,Th) int32  blank id or the label emitted by that state
    spans (B,Umax,2) int32  first and last frame of each label
    score (B) fp32  log-probability of the path under softmax(logits) (-inf when no path exists)"""


def ctc_forced_align(logits, hlens, targets, blank=0):
    """Viterbi path of each transcript through its CTC lattice, on the device (csrc/ctc.cu ctc_viterbi_warp_kernel).
    logits (B,Th,V) fp32 CUDA raw activations or log-probabilities (rows may be pitched, like the ctc_lo GEMM output);
    hlens host ints or an int CUDA tensor (clamped to Th); targets: PreparedTargets or anything prepare_targets
    accepts.  On equal scores a state stays, then comes from s-1, then from s-2; the path ends in the final blank
    when that ties with the last label.  Returns CTCAlignment; takes no part in autograd.  With PreparedTargets and
    device hlens the call never synchronises with the host and can be captured into a CUDA graph."""
    L = _lib.lib()
    dev = logits.device
    if not isinstance(targets, PreparedTargets):
        targets = prepare_targets(targets, dev)
    hl = _device_hlens(hlens, dev)
    x = logits.detach()
    x = x if _strided_ok(x) else _lib.f32c(x)
    B, Th, V = x.shape
    assert targets.nutt == B and hl.numel() == B
    umax = targets.umax
    nbytes = int(L.re2e_ctc_ws_bytes(B, Th, V, umax))
    ws = torch.empty(nbytes, device=dev, dtype=torch.uint8)
    states = torch.empty(B, Th, device=dev, dtype=torch.int32)
    tokens = torch.empty(B, Th, device=dev, dtype=torch.int32)
    spans = torch.empty(B, umax, 2, device=dev, dtype=torch.int32)
    score = torch.empty(B, device=dev, dtype=torch.float32)
    with _lib.on(dev):
        _lib.check(L.re2e_ctc_align(_lib.ptr(x), x.stride(0), x.stride(1), _lib.ptr(targets.labels),
                                    _lib.ptr(targets.offs), _lib.ptr(targets.lens), _lib.ptr(hl), int(blank),
                                    _lib.ptr(states), _lib.ptr(tokens), _lib.ptr(spans) if umax else None,
                                    _lib.ptr(score), _lib.ptr(ws), nbytes, B, Th, V, umax, _lib.stream_ptr()),
                   "re2e_ctc_align")
    return CTCAlignment(states, tokens, spans, score)


def log_softmax_rows(logits, want_best=False):
    """log_softmax over the last dim with the warp-per-row kernel (+ argmax = CTC best path)."""
    L = _lib.lib()
    x = _lib.f32c(logits.detach())
    V = x.shape[-1]
    rows = x.numel() // V
    out = torch.empty_like(x)
    best = torch.empty(x.shape[:-1], device=x.device, dtype=torch.int32) if want_best else None
    with _lib.on(x.device):
        _lib.check(L.re2e_log_softmax(_lib.ptr(x), _lib.ptr(out), _lib.ptr(best), rows, V, _lib.stream_ptr()),
                   "re2e_log_softmax")
    return (out, best) if want_best else out


class CTC(torch.nn.Module):
    """model/e2e_ctc.py:17-75."""

    def __init__(self, odim, eprojs, dropout_rate):
        super(CTC, self).__init__()
        self.dropout_rate = dropout_rate
        self.loss = None
        self.ctc_lo = torch.nn.Linear(eprojs, odim)
        self.loss_fn = ctc_loss          # the reference holds warp_ctc.CTCLoss(size_average=True) here
        self.ignore_id = -1

    def forward(self, hs_pad, hlens, ys_pad):
        """hs_pad (B,Tmax,D); hlens (B) host ints; ys_pad padded (B,Lmax) tensor, list of 1-D
        LongTensors, or PreparedTargets.  Returns the (1,) loss (sum of utterance NLLs / B)."""
        self.loss = None
        dev = self.ctc_lo.weight.device
        if hs_pad.device != dev:
            hs_pad = hs_pad.to(dev)
        # model/e2e_ctc.py:51 -- functional dropout, active regardless of .training (quirk 6)
        ys_hat = _linear_tc(F.dropout(hs_pad, p=self.dropout_rate), self.ctc_lo.weight, self.ctc_lo.bias)
        tgt = ys_pad if isinstance(ys_pad, PreparedTargets) else prepare_targets(ys_pad, dev, self.ignore_id)
        self.loss, self.nll = ctc_loss(ys_hat, hlens, tgt, blank=0)
        return self.loss

    def log_softmax(self, hs_pad):
        """model/e2e_ctc.py:68-75 (decode-time only; returned tensor carries no graph)."""
        dev = self.ctc_lo.weight.device
        with torch.no_grad():
            return log_softmax_rows(_linear_tc(hs_pad.to(dev), self.ctc_lo.weight, self.ctc_lo.bias))

    def forced_align(self, hs_pad, hlens, ys_pad):
        """Forced alignment of ys_pad (padded tensor with ignore_id, list of 1-D tensors or PreparedTargets) to
        ctc_lo(hs_pad) without dropout; see ctc_forced_align.  Returns CTCAlignment."""
        dev = self.ctc_lo.weight.device
        tgt = ys_pad if isinstance(ys_pad, PreparedTargets) else prepare_targets(ys_pad, dev, self.ignore_id)
        with torch.no_grad():
            ys_hat = _linear_tc(hs_pad.to(dev), self.ctc_lo.weight, self.ctc_lo.bias)
            return ctc_forced_align(ys_hat, hlens, tgt, blank=0)

    def best_path(self, hs_pad):
        """argmax_v log_softmax(ctc_lo(h))[b,t,:] -- the 'CTC alignment' of the north star."""
        dev = self.ctc_lo.weight.device
        with torch.no_grad():
            return log_softmax_rows(_linear_tc(hs_pad.to(dev), self.ctc_lo.weight, self.ctc_lo.bias),
                                    want_best=True)[1]


def ctc_prefix_score_batch(lpz, r_prev, cs, last, out_len, blank, eos):
    """Device-resident batched prefix scoring (H hypotheses x C candidates in one launch).
    lpz (T,V) fp32 CUDA; r_prev (H,T,2); cs (H,C) int32; last (H) int32; out_len (H) int32.
    Returns log_psi (H,C), r_new (H,C,T,2)."""
    L = _lib.lib()
    T, V = lpz.shape
    H, C = cs.shape
    dev = lpz.device
    log_psi = torch.empty(H, C, device=dev, dtype=torch.float32)
    r_new = torch.empty(H, C, T, 2, device=dev, dtype=torch.float32)
    with _lib.on(dev):
        _lib.check(L.re2e_ctc_prefix_score(_lib.ptr(lpz), _lib.ptr(r_prev), _lib.ptr(cs), _lib.ptr(last),
                                           _lib.ptr(out_len), _lib.ptr(log_psi), _lib.ptr(r_new), T, V, H, C,
                                           int(blank), int(eos), _lib.stream_ptr()), "re2e_ctc_prefix_score")
    return log_psi, r_new


class CTCPrefixScore(object):
    """model/e2e_ctc.py:78-155 with the reference's host-side call shape (numpy in / numpy out,
    as Decoder.recognize_beam uses it, model/e2e_decoder.py:217,279), computed on the device."""

    def __init__(self, x, blank, eos, xp=np):
        self.xp = xp
        self.logzero = -10000000000.0
        self.blank = blank
        self.eos = eos
        self.input_length = len(x)
        self.x = x
        _lib.lib()
        self._dev = torch.device('cuda', torch.cuda.current_device())
        self._x_dev = torch.as_tensor(np.asarray(x, dtype=np.float32)).to(self._dev).contiguous()

    def initial_state(self):
        r = np.full((self.input_length, 2), self.logzero, dtype=np.float32)
        r[:, 1] = np.cumsum(np.asarray(self.x)[:, self.blank].astype(np.float32), dtype=np.float32)
        return r

    def __call__(self, y, cs, r_prev):
        cs_np = cs.detach().cpu().numpy() if torch.is_tensor(cs) else np.asarray(cs)
        dev = self._dev
        cs_d = torch.as_tensor(cs_np.astype(np.int32)).to(dev).view(1, -1).contiguous()
        rp = torch.as_tensor(np.ascontiguousarray(r_prev, dtype=np.float32)).to(dev).view(1, -1, 2)
        last = torch.tensor([int(y[-1])], dtype=torch.int32, device=dev)
        olen = torch.tensor([len(y) - 1], dtype=torch.int32, device=dev)
        log_psi, r_new = ctc_prefix_score_batch(self._x_dev, rp, cs_d, last, olen, self.blank, self.eos)
        return log_psi[0].cpu().numpy(), r_new[0].cpu().numpy()
