"""LSTMCell step of the attention decoder on the library's kernels (reference: model/e2e_decoder.py:128,
``z_list[0], c_list[0] = self.decoder[0](ey, (z_list[0], c_list[0]))`` with ``ey = cat(embed(y), att_c)``).

Same arithmetic as ``torch.nn.LSTMCell`` (gate order i, f, g, o) split the way the decoder loop wants it:

* ``embed_gates``: the embedding half of the input product plus both biases, for ALL positions, as one dense product
  on the tcgen05 GEMM before the loop (teacher forcing: the tokens are known);
* ``LSTMLoop.step``: per position ONE launch (``re2e_lstm_step_fwd``: the two batch-sized products that depend on the
  recurrence -- context and previous state -- reduced across a 4-CTA cluster, with the pointwise cell arithmetic as the
  epilogue); its backward is the pointwise kernel plus ONE product launch for d context | d h_prev
  (``re2e_lstm_step_bwd``, 8-CTA clusters).  Dimensions outside that kernel's range compose ``re2e_batch_nt`` products
  with the pointwise kernels;
* the weight gradients of all positions are two dense products after the loop (an anchor node, like AttLoc's).

``LSTMLoop.by_token`` is the same loop with the embedding half looked up by token inside the step kernel from a per-token
table (V, 4Z), for inputs that are chosen while the loop runs (scheduled sampling): the tokens live in a device buffer
the caller may overwrite before each step, and the anchor forms the embedding-half gradients from the final buffer.
"""
import torch

from . import _lib
from .linear import colsum, gemm_tf32x3, linear


def _batch_nt(X, W, out, M, N, K, accumulate=False):
    """out[M,N] (+)= X[M,K] @ W[N,K]^T, M = batch rows (re2e_batch_nt: all SMs stream W once)."""
    L = _lib.lib()
    with _lib.on(out.device):
        _lib.check(L.re2e_batch_nt(_lib.ptr(X), _lib.ptr(W), None, _lib.ptr(out), M, N, K, int(accumulate),
                                   _lib.stream_ptr()), "re2e_batch_nt")


class _State(object):
    def __init__(self):
        self.W_c = self.W_hh = self.W_cT = self.W_hhT = self.Wcat = self.WcatT = self.egates = None
        self.tok = None                  # token-lookup mode: (L, B) int32 rows of `egates` (the per-token table)
        self.dg, self.ctx, self.hprev = {}, {}, {}


class _Anchor(torch.autograd.Function):
    """Owns the two recurrent weight matrices and the embedding-half gates of all positions.  Its backward runs after
    every step's (each step depends on the anchor) and emits, ONCE: the weight gradients as two dense GEMMs over all
    positions, and the gradient of the (L,B,4Z) embedding-half gates as one stacked tensor (41 separate slice
    gradients would each materialise a full-size zero tensor)."""

    @staticmethod
    def forward(ctx, W_c, W_hh, egates, state):
        state.W_c, state.W_hh = _lib.f32c(W_c.detach()), _lib.f32c(W_hh.detach())
        state.W_cT = state.W_hhT = None          # (D,4Z) / (Z,4Z) copies for the backward's products, built on first use
        D, Z = state.W_c.shape[1], state.W_hh.shape[1]
        state.Wcat = state.WcatT = None
        if _lib.lib().re2e_lstm_step_supported(1, D, Z):
            state.Wcat = torch.cat((state.W_c, state.W_hh), 1)                 # (4Z, D+Z): one launch per position
        state.egates = _lib.f32c(egates.detach())
        ctx.state = state
        ctx.set_materialize_grads(False)
        return torch.zeros(1, device=W_c.device, dtype=torch.float32)

    @staticmethod
    def backward(ctx, _g):
        d_eg, dW_c, dW_hh = _recurrent_grads(ctx.state)
        return dW_c, dW_hh, d_eg, None


def _recurrent_grads(st):
    """(d_eg (L,B,4Z), dW_c, dW_hh) from the gate gradients the steps left in ``st``, or Nones when no step had one."""
    dW_c = dW_hh = d_eg = None
    if st.dg:
        L_, B = st.tok.shape if st.tok is not None else st.egates.shape[:2]
        G4 = st.egates.shape[-1]
        zero = None
        rows = []
        for i in range(L_):
            if i in st.dg:
                rows.append(st.dg[i])
            else:
                zero = zero if zero is not None else torch.zeros(B, G4, device=st.egates.device)
                rows.append(zero)
        d_eg = torch.stack(rows, 0)                                           # (L, B, 4Z)
        idx = sorted(st.dg)
        DG = torch.stack([st.dg[i] for i in idx], 0).view(len(idx) * B, G4)
        XC = torch.stack([st.ctx[i] for i in idx], 0).view(len(idx) * B, -1)
        HP = torch.stack([st.hprev[i] for i in idx], 0).view(len(idx) * B, -1)
        dW_c = torch.empty_like(st.W_c)
        dW_hh = torch.empty_like(st.W_hh)
        gemm_tf32x3(DG, True, XC, True, dW_c, G4, XC.shape[1], len(idx) * B)    # sum_s dgates_s^T context_s
        gemm_tf32x3(DG, True, HP, True, dW_hh, G4, HP.shape[1], len(idx) * B)   # sum_s dgates_s^T h_{s-1}
    st.dg, st.ctx, st.hprev = {}, {}, {}
    return d_eg, dW_c, dW_hh


class _TokenAnchor(torch.autograd.Function):
    """``_Anchor`` of the token-lookup loop.  The per-token table is a constant of the forward (it cannot carry gradient
    for tokens chosen inside the loop); the backward forms the gradients of the embedding half itself, once, from the
    stacked gate gradients d_eg (L,B,4Z) and the final token buffer:
        d W_ih[:, :E] = d_eg^T @ embed.weight[tok]   (one tcgen05 GEMM over all positions)
        d b_ih = d b_hh = column sums of d_eg
        d embed.weight = embedding backward of d_eg @ W_ih[:, :E] on tok   (the op behind embed(pad_ys_in)'s backward)"""

    @staticmethod
    def forward(ctx, W_c, W_hh, W_e, b_ih, b_hh, emb, table, tok, state):
        _Anchor.forward(ctx, W_c, W_hh, table, state)
        state.tok = tok
        ctx.W_e, ctx.emb = _lib.f32c(W_e.detach()), emb.detach()
        return torch.zeros(1, device=W_c.device, dtype=torch.float32)

    @staticmethod
    def backward(ctx, _g):
        st = ctx.state
        tok = st.tok
        d_eg, dW_c, dW_hh = _recurrent_grads(st)
        if d_eg is None:
            return (None,) * 9
        L_, B, G4 = d_eg.shape
        E = ctx.W_e.shape[1]
        DG = d_eg.view(L_ * B, G4)
        rows = tok.reshape(-1)
        dW_e = torch.empty(G4, E, device=DG.device, dtype=torch.float32)
        gemm_tf32x3(DG, True, _lib.f32c(ctx.emb.index_select(0, rows)), True, dW_e, G4, E, L_ * B)
        db = colsum(DG)
        d_rows = torch.empty(L_ * B, E, device=DG.device, dtype=torch.float32)
        gemm_tf32x3(DG, False, ctx.W_e, True, d_rows, L_ * B, E, G4)             # d embeddings = d_eg @ W_ih[:, :E]
        d_emb = torch.ops.aten.embedding_dense_backward(d_rows, rows.long(), ctx.emb.shape[0], -1, False)
        return dW_c, dW_hh, dW_e, db, db.clone(), d_emb.to(ctx.emb.dtype), None, None, None


class _Step(torch.autograd.Function):
    @staticmethod
    def forward(ctx, anchor, att_c, h_prev, c_prev, state, i):
        L = _lib.lib()
        dev = att_c.device
        xc, hp, cp = _lib.f32c(att_c.detach()), _lib.f32c(h_prev.detach()), _lib.f32c(c_prev.detach())
        B, Z = hp.shape
        row = state.tok[i] if state.tok is not None else None          # token lookup: egates is the (V, 4Z) table
        eg = state.egates[i] if row is None else state.egates
        D = xc.shape[1]
        gates = torch.empty(B, 4 * Z, device=dev, dtype=torch.float32)
        h, c = torch.empty_like(hp), torch.empty_like(hp)
        with _lib.on(dev):
            if state.Wcat is not None:
                _lib.check(L.re2e_lstm_step_fwd(_lib.ptr(xc), _lib.ptr(hp), _lib.ptr(cp), _lib.ptr(state.Wcat), _lib.ptr(eg),
                                                _lib.ptr(row), _lib.ptr(gates), _lib.ptr(c), _lib.ptr(h), B, D, Z, _lib.stream_ptr()),
                           "re2e_lstm_step_fwd")
            else:
                _batch_nt(xc, state.W_c, gates, B, 4 * Z, D)                     # context @ W_ih[:, Z:]^T
                _batch_nt(hp, state.W_hh, gates, B, 4 * Z, Z, accumulate=True)   # + h_prev @ W_hh^T
                if row is not None:
                    eg = eg.index_select(0, row)
                _lib.check(L.re2e_lstm_pointwise_fwd(_lib.ptr(gates), _lib.ptr(eg), _lib.ptr(cp), _lib.ptr(c),
                                                     _lib.ptr(h), B, Z, _lib.stream_ptr()), "re2e_lstm_pointwise_fwd")
        ctx.state, ctx.i = state, i
        ctx.save_for_backward(gates, cp, c, xc, hp)
        ctx.set_materialize_grads(False)
        return h, c

    @staticmethod
    def backward(ctx, dh, dc):
        L = _lib.lib()
        st = ctx.state
        act, cp, c, xc, hp = ctx.saved_tensors
        B, Z = hp.shape
        D = xc.shape[1]
        dev = hp.device
        if dh is None and dc is None:
            return None, None, None, None, None, None
        dh = _lib.f32c(dh, dev) if dh is not None else None
        dc = _lib.f32c(dc, dev) if dc is not None else None
        dg = torch.empty(B, 4 * Z, device=dev, dtype=torch.float32)
        dcp = torch.empty(B, Z, device=dev, dtype=torch.float32)
        with _lib.on(dev):
            _lib.check(L.re2e_lstm_pointwise_bwd(_lib.ptr(act), _lib.ptr(cp), _lib.ptr(c), _lib.ptr(dh), _lib.ptr(dc),
                                                 _lib.ptr(dg), _lib.ptr(dcp), B, Z, _lib.stream_ptr()),
                       "re2e_lstm_pointwise_bwd")
        d_ctx = torch.empty(B, D, device=dev, dtype=torch.float32)
        d_hp = torch.empty(B, Z, device=dev, dtype=torch.float32)
        if st.Wcat is not None:
            if st.WcatT is None:     # once per loop: the transposed copy makes the backward's product row-streamed as well
                st.WcatT = st.Wcat.t().contiguous()
            with _lib.on(dev):
                _lib.check(L.re2e_lstm_step_bwd(_lib.ptr(dg), _lib.ptr(st.WcatT), _lib.ptr(d_ctx), _lib.ptr(d_hp), B, D, Z,
                                                _lib.stream_ptr()), "re2e_lstm_step_bwd")
        else:
            if st.W_cT is None:
                st.W_cT, st.W_hhT = st.W_c.t().contiguous(), st.W_hh.t().contiguous()
            _batch_nt(dg, st.W_cT, d_ctx, B, D, 4 * Z)                           # d context = dgates @ W_ih[:, Z:]
            _batch_nt(dg, st.W_hhT, d_hp, B, Z, 4 * Z)                           # d h_prev  = dgates @ W_hh
        st.dg[ctx.i], st.ctx[ctx.i], st.hprev[ctx.i] = dg, xc, hp
        return None, d_ctx, d_hp, dcp, None, None


class LSTMLoop(object):
    """One decoder loop's worth of LSTMCell steps for ``cell`` (a torch.nn.LSTMCell whose input is cat(embedding, context)).

        loop = LSTMLoop(cell, eys)          # eys (B, L, dunits): embeddings of all positions
        z, c = loop.step(i, att_c, z, c)    # position i
    """

    def __init__(self, cell, eys):
        E = eys.shape[-1]
        W_ih = cell.weight_ih
        # embedding half + both biases for every position, position-major (L, B, 4Z): one product, contiguous per position
        egates = linear(eys.transpose(0, 1).contiguous(), W_ih[:, :E], cell.bias_ih + cell.bias_hh)
        self.state = _State()
        self.anchor = _Anchor.apply(W_ih[:, E:].contiguous(), cell.weight_hh, egates, self.state)

    @classmethod
    def by_token(cls, cell, embed_weight, tok):
        """The loop with the embedding half looked up by token: ``tok`` (L, B) int32 device buffer, row i = the tokens
        position i feeds (overwritable up to step i).  The table embed_weight @ W_ih[:, :E]^T + b_ih + b_hh (V, 4Z) is
        built here, once, outside autograd."""
        self = cls.__new__(cls)
        E = embed_weight.shape[1]
        W_ih = cell.weight_ih
        with torch.no_grad():
            table = linear(_lib.f32c(embed_weight.detach()), W_ih.detach()[:, :E].contiguous(),
                           (cell.bias_ih + cell.bias_hh).detach()).contiguous()
        self.state = _State()
        self.anchor = _TokenAnchor.apply(W_ih[:, E:].contiguous(), cell.weight_hh, W_ih[:, :E], cell.bias_ih,
                                         cell.bias_hh, embed_weight, table, tok, self.state)
        return self

    def step(self, i, att_c, h_prev, c_prev):
        return _Step.apply(self.anchor, att_c, h_prev, c_prev, self.state, i)
