"""Attention decoder around ``AttLoc`` (reference: model/e2e_decoder.py:25-369), next-row N1/N2 of SURVEY.md 8f.

Same constructor, submodule names (``embed``, ``decoder`` = ModuleList of LSTMCell, ``output``, ``att``) and
state_dict keys as the reference's ``Decoder`` for the configuration the scripts use (no LM fusion,
``model_unit='char'``), so reference ``asr_state_dict`` checkpoints load unchanged.

* ``forward(hpad, hlen, ys, scheduled_sampling_rate)`` -- the training loop of model/e2e_decoder.py:79-167: AttLoc
  step kernel per output position with the alignment fed back un-detached, teacher forcing or scheduled sampling,
  cross-entropy rescaled by ``mean(len(ys_in)) - 1``.  The output layer of all positions is ONE product on the tcgen05
  GEMM after the loop, every LSTMCell is one cluster kernel per position (lstm.py; the upper layers of a multi-layer
  decoder through ``LSTMLoop.stacked``) and the cross-entropy runs on the library's kernels.  The decoder state fed to
  step i depends on the context of step i-1 through the LSTMCell, so this loop calls the per-step AttLoc kernels
  (``AttLoc.forward_loop``, the persistent loop kernels, needs the states of all steps up front).  Scheduled sampling
  (rate > 0) keeps that shape: the reference's one ``random.random()`` per position is drawn before the loop, the
  flags reach the device through a page-locked buffer, and a flagged position's token -- the arg-max of the previous
  position's logits -- is chosen on the device by ``re2e_sample_tokens`` (the logits are never written) into the token
  buffer the LSTM step looks its embedding half up from.  No host round trip, so the forward + backward can be
  captured once and replayed with new draws (``draw_sampling``).  ``fused_lstm = False`` or a CPU module runs the
  reference's own loop.
* ``recognize_beam(h, lpz, recog_args, char_list, rnnlm=None, fstlm=None)`` -- hybrid CTC/attention beam search
  (model/e2e_decoder.py:170-369) re-designed for the GPU: ALL live hypotheses advance together (B = beam instead of
  beam x (B = 1) calls) and the whole output position runs on the device as SIX launches of the library over static
  buffers (csrc/beam.cu), one more per extra decoder layer: AttLoc step, LSTMCell step (one cluster kernel; the
  embedding half of its input product is a per-token table looked up inside the kernel), one LSTMCell step per upper
  layer, output layer, log-softmax + top-``ctc_beam``, batched CTC prefix scores whose forward variables never leave
  the device (the reference copies ``lpz`` to the host and loops over T in numpy per hypothesis,
  model/e2e_ctc.py:143-146), and one kernel for joint score + merge of the beam x beam candidates + gather of the
  chosen rows' states.  Eight positions are one CUDA-graph replay; the winners of every position land in a history
  buffer that the host reads back a chunk at a time (two chunks in flight) to run the reference's own bookkeeping --
  <eos> handling, length penalty, ``end_detect`` -- so there is no host round trip per position.  Scores accumulate in
  fp32 exactly as the reference's 0-dim tensors do.  Decoders the fused position does not take (more than
  FUSED_MAX_LAYERS = 6 LSTM layers, ctc_weight = 1 i.e. all V candidates, V > 8192, dunits or eprojs not a multiple of
  4) use the generic position: library AttLoc / prefix-score kernels + tensor ops, host merge per position.
"""
import random
import time

import numpy as np
import torch
import torch.nn.functional as F

from . import _lib
from .e2e_common import pad_list
from .e2e_ctc import ctc_prefix_score_batch, log_softmax_rows
from .linear import linear
from .lstm import LSTMLoop

CTC_SCORING_RATIO = 1.5   # model/e2e_decoder.py:20
# deepest decoder the fused beam-search position takes: re2e_beam_advance gathers at most 16 state tensors, z and c of
# every layer + the alignment + the two CTC states (include/re2e_b200.h)
FUSED_MAX_LAYERS = 6


def end_detect(ended_hyps, i, M=3, D_end=np.log(1 * np.exp(-10))):
    """model/e2e_common.py:226-254 (Eq. 50 of Watanabe et al., hybrid CTC/attention)."""
    if len(ended_hyps) == 0:
        return False
    count = 0
    best_hyp = sorted(ended_hyps, key=lambda x: x['score'], reverse=True)[0]
    for m in range(M):
        hyp_length = i - m
        same = [x for x in ended_hyps if len(x['yseq']) == hyp_length]
        if len(same) > 0:
            best_same = sorted(same, key=lambda x: x['score'], reverse=True)[0]
            if best_same['score'] - best_hyp['score'] < D_end:
                count += 1
    return count == M


def mask_by_length(xs, length, fill=0):
    """model/e2e_common.py:190-195.  ``length``: list of ints, or a device tensor (then no host round trip: the
    whole decoder forward stays CUDA-graph capturable)."""
    assert xs.size(0) == len(length)
    if torch.is_tensor(length) and length.is_cuda:
        keep = torch.arange(xs.size(1), device=xs.device)[None, :] < length.to(xs.device)[:, None]
        keep = keep.view(keep.shape + (1,) * (xs.dim() - 2))
        return torch.where(keep, xs, xs.new_full((), fill))
    if xs.is_cuda:
        # same values as the reference's per-utterance slice copies, as ONE select (whose backward is one kernel instead
        # of a zero-fill + copy + add of the whole batch tensor per utterance)
        return mask_by_length(xs, torch.as_tensor([int(l) for l in length], dtype=torch.int64).to(xs.device), fill)
    ret = xs.new_full(xs.size(), fill)
    for i, l in enumerate(length):
        ret[i, :l] = xs[i, :l]
    return ret


def _label_batches(ys, sos, eos, ignore_id, keep):
    """pad_ys_in = pad([<sos>, y...], <eos>) and pad_ys_out = pad([y..., <eos>], ignore_id) of model/e2e_decoder.py:88-97
    for label tensors that already live on the device: one concatenation and two gathers through host-built index
    tables (copied from page-locked memory, so the sequence is CUDA-graph capturable; ``keep`` holds the host side)
    instead of two concatenations and two slice copies per utterance."""
    dev, dt = ys[0].device, ys[0].dtype
    lens = [int(y.size(0)) for y in ys]
    n, B, U1 = sum(lens), len(ys), max(lens) + 1
    off = np.concatenate(([0], np.cumsum(lens)[:-1]))
    j = np.arange(U1)[None, :]
    ln, of = np.asarray(lens)[:, None], off[:, None]
    idx = np.stack((np.where(j == 0, n, np.where(j - 1 < ln, of + j - 1, n + 1)),          # n: <sos>, n+1: <eos>
                    np.where(j < ln, of + j, np.where(j == ln, n + 1, n + 2)))).astype(np.int64)   # n+2: ignore_id
    pin, spec = torch.from_numpy(idx).pin_memory(), torch.tensor([sos, eos, ignore_id], dtype=dt).pin_memory()
    keep.append((pin, spec))                        # (alive as long as a captured graph may replay the two copies)
    ext = torch.cat(list(ys) + [spec.to(dev, non_blocking=True)])
    out = ext[pin.to(dev, non_blocking=True).view(-1)].view(2, B, U1)
    return out[0], out[1]


def th_accuracy(y_all, pad_target, ignore_label, pred=None):
    """model/e2e_common.py:198-205.  Returns a Python float like the reference, except while a CUDA graph is being
    captured (no device-to-host read is possible there): then the 0-dim device tensor.  ``pred``: the rows' arg-max
    when the caller already has it."""
    pad_pred = pred if pred is not None else \
        y_all.detach().reshape(pad_target.size(0), pad_target.size(1), y_all.size(1)).max(2)[1]
    mask = pad_target != ignore_label
    num = torch.sum((pad_pred == pad_target) & mask)
    den = torch.sum(mask)
    if y_all.is_cuda and torch.cuda.is_current_stream_capturing():
        return num.float() / den.float()
    return float(num) / float(den)


class _CrossEntropy(torch.autograd.Function):
    """F.cross_entropy(y_all, target, ignore_index, reduction='mean') of model/e2e_decoder.py:155 on the library's
    kernels: no log-softmax tensor, the arg-max of every row (for th_accuracy) from the same pass, the gradient written
    in the row-padded layout the dense layer's backward reads without a copy."""

    @staticmethod
    def forward(ctx, y_all, target, ignore_id):
        L = _lib.lib()
        x = y_all.detach()
        if x.dtype != torch.float32 or x.stride(1) != 1:
            x = x.float().contiguous()
        rows, V = x.shape
        dev = x.device
        tgt = target.contiguous()
        lse = torch.empty(rows, device=dev, dtype=torch.float32)
        nll = torch.empty(rows, device=dev, dtype=torch.float32)
        best = torch.empty(rows, device=dev, dtype=torch.int32)
        with _lib.on(dev):
            _lib.check(L.re2e_cross_entropy_fwd(_lib.ptr(x), x.stride(0), _lib.ptr(tgt), int(ignore_id), rows, V,
                                                _lib.ptr(lse), _lib.ptr(nll), _lib.ptr(best), _lib.stream_ptr()),
                       "re2e_cross_entropy_fwd")
        count = (tgt != ignore_id).sum().to(torch.float32)
        ctx.save_for_backward(x, tgt, lse, count)
        ctx.ignore_id = int(ignore_id)
        ctx.mark_non_differentiable(best)
        return nll.sum() / count, best

    @staticmethod
    def backward(ctx, g, _gbest):
        L = _lib.lib()
        x, tgt, lse, count = ctx.saved_tensors
        rows, V = x.shape
        scale = (g.to(torch.float32) / count).contiguous()
        ldd = (V + 3) // 4 * 4
        dx = torch.empty(rows, ldd, device=x.device, dtype=torch.float32)[:, :V]
        with _lib.on(x.device):
            _lib.check(L.re2e_cross_entropy_bwd(_lib.ptr(x), x.stride(0), _lib.ptr(tgt), ctx.ignore_id, rows, V,
                                                _lib.ptr(lse), _lib.ptr(scale), _lib.ptr(dx), ldd, _lib.stream_ptr()),
                       "re2e_cross_entropy_bwd")
        return dx, None, None


class _FusedSearch(object):
    """One utterance's beam search with the whole position on the device (``Decoder._fused_position``), as a resumable
    object: ``pump()`` keeps two chunks of ``chunk`` positions in flight on ``stream`` (one CUDA-graph replay per chunk,
    then an async copy of the chunk's history rows), ``poll()`` runs the reference's bookkeeping (<eos>, length penalty,
    end_detect; model/e2e_decoder.py:296-333) on the oldest chunk that has arrived.  Positions launched beyond the one
    where the search ends are discarded (past maxlen the merge kernel is a no-op)."""

    def __init__(self, dec, hb, lpz, recog_args, Cb, maxlen, minlen, stream, slot, tables, chunk=8):
        self.dec, self.args, self.maxlen, self.minlen, self.chunk = dec, recog_args, maxlen, minlen, chunk
        self.stream, self.dev = stream, hb.device
        self.beam = hb.size(0)
        self.prof = getattr(recog_args, "profile", None)   # optional dict: host seconds per phase
        t0 = time.perf_counter()
        pins = dec.__dict__.setdefault("_hist_pins", {})
        pin = pins.get(slot)
        if pin is None or pin[0].shape[0] < maxlen or pin[0].shape[2] != self.beam:
            pin = pins[slot] = (torch.empty(max(256, maxlen), 4, self.beam, dtype=torch.float32).pin_memory(),
                                [torch.cuda.Event() for _ in range(3)])
        self.pin, self.events = pin
        self.hist_np = self.pin.numpy()
        with torch.cuda.stream(stream):
            self.position = dec._fused_position(hb, lpz, Cb, self.beam, recog_args.ctc_weight, maxlen, self.pin, tables)
        self.use_graph = bool(getattr(recog_args, "cuda_graph", True)) and maxlen >= 6
        self.graph = None
        self.hyps = [(np.float32(0.0), dec.sos, None, 1)]               # hypothesis k lives in device row k
        self.ended = []
        self.launched = self.processed = 0
        self.flights = []
        self._evi = 0
        self.lazy = True              # no hypothesis has ended yet (see poll)
        self.done = False
        self._t(t0, "setup")

    def _t(self, t0, key):
        if self.prof is not None:
            self.prof[key] = self.prof.get(key, 0.0) + time.perf_counter() - t0

    def _capture(self):
        # raw capture_begin / capture_end on a side stream: the torch.cuda.graph context manager also runs gc.collect()
        # and empty_cache(), tens of milliseconds per utterance.  Nothing is allocated during the capture.
        t0 = time.perf_counter()
        dec, dev = self.dec, self.dev
        if getattr(dec, "_cap_stream", None) is None or dec._cap_stream.device != dev:
            dec._cap_stream = torch.cuda.Stream(dev)
            dec._graph_pool = None        # (the generic position's pool belongs to the previous device)
        dec._cap_stream.wait_stream(self.stream)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.stream(dec._cap_stream):
            self.graph.capture_begin()
            for _ in range(self.chunk):
                self.position()
            self.graph.capture_end()
        self.stream.wait_stream(dec._cap_stream)
        self._t(t0, "capture")

    def pump(self):
        if self.done or self.launched >= self.maxlen or self.launched >= self.processed + 2 * self.chunk:
            return                      # (nothing to launch: do not pay for the stream switch)
        t0 = time.perf_counter()
        with torch.cuda.stream(self.stream):
            while self.launched < self.maxlen and self.launched < self.processed + 2 * self.chunk:
                lo = self.launched
                if lo == 0 or not self.use_graph:
                    hi = 1 if self.use_graph else min(self.maxlen, lo + self.chunk)   # position 0 also warms the kernels up
                    for _ in range(lo, hi):
                        self.position()
                else:
                    if self.graph is None:
                        self._capture()
                    t1 = time.perf_counter()
                    self.graph.replay()
                    self._t(t1, "replay")
                    hi = min(self.maxlen, lo + self.chunk)
                ev = self.events[self._evi]              # (three events, at most two chunks in flight)
                self._evi = (self._evi + 1) % 3
                ev.record(self.stream)
                self.flights.append((lo, hi, ev))
                self.launched = hi
        self._t(t0, "launch")

    def poll(self, block):
        """Book-keep the oldest chunk in flight if it has arrived (or wait for it); True if a chunk was processed."""
        if self.done or not self.flights:
            return False
        lo, hi, ev = self.flights[0]
        if not block and not ev.query():
            return False
        t0 = time.perf_counter()
        ev.synchronize()
        self._t(t0, "wait")
        t0 = time.perf_counter()
        self.flights.pop(0)
        dec, args, beam = self.dec, self.args, self.beam
        blk = self.hist_np[lo:hi]
        if self.lazy:
            # As long as no hypothesis has ended the beam simply extends (every winner survives, its parent index is its
            # position in the previous winners' list), so a chunk in which no <eos> was emitted needs no bookkeeping at
            # all: the history buffer IS the search state.  The first chunk with an <eos> (or the last position)
            # rebuilds the linked hypotheses from the history once and continues position by position.
            if hi < self.maxlen and not (blk[:, 2] == float(dec.eos)).any():
                self.processed = hi
                self._t(t0, "host_merge")
                if self.prof is not None:
                    self.prof["positions"] = self.prof.get("positions", 0.0) + (hi - lo)
                return True
            self.lazy = False
            if lo > 0:
                past = self.hist_np[:lo]
                psc, pidx = past[:, 0].tolist(), past[:, 1:].astype(np.int64).tolist()
                nodes = [self.hyps[0]]
                for i in range(lo):
                    par, tok, cj = pidx[i]
                    nodes = [(np.float32(psc[i][b]), tok[b], nodes[par[b]], i + 2, par[b], cj[b]) for b in range(beam)]
                self.hyps = nodes
        scs, idx = blk[:, 0].tolist(), blk[:, 1:].astype(np.int64).tolist()
        for i in range(lo, hi):
            par, tok, cj = idx[i - lo]
            entries = list(zip(scs[i - lo], par, tok, cj))
            self.hyps = dec._host_merge(self.hyps, self.ended, entries, i, self.maxlen, self.minlen, args.penalty)
            if (end_detect(self.ended, i) and args.maxlenratio == 0.0) or len(self.hyps) == 0:
                self.done = True
                break
        self.processed = hi
        if hi >= self.maxlen:
            self.done = True
        self._t(t0, "host_merge")
        if self.prof is not None:
            self.prof["positions"] = self.prof.get("positions", 0.0) + (hi - lo)
        return True

    def result(self):
        nbest = sorted(self.ended, key=lambda x: x['score'], reverse=True)[:min(len(self.ended), self.args.nbest)]
        return [{'score': float(x['score']), 'yseq': [int(t) for t in x['yseq']]} for x in nbest]


class Decoder(torch.nn.Module):
    def __init__(self, eprojs, odim, dlayers, dunits, sos, eos, att, verbose=0, char_list=None, labeldist=None,
                 lsm_weight=0., fusion=None, rnnlm=None, model_unit='char', space_loss_weight=0.1):
        super(Decoder, self).__init__()
        if fusion is not None and rnnlm is not None:
            raise NotImplementedError("LM fusion decoders are outside the hot path (SURVEY.md section 8)")
        self.dunits = dunits
        self.dlayers = dlayers
        self.embed = torch.nn.Embedding(odim, dunits)
        self.decoder = torch.nn.ModuleList()
        self.fusion = fusion
        self.rnnlm = rnnlm
        self.decoder += [torch.nn.LSTMCell(dunits + eprojs, dunits)]
        for _ in range(1, self.dlayers):
            self.decoder += [torch.nn.LSTMCell(dunits, dunits)]
        self.ignore_id = -1
        self.output = torch.nn.Linear(dunits, odim)
        self.loss = None
        self.att = att
        self.sos = sos
        self.eos = eos
        self.verbose = verbose
        self.char_list = char_list
        self.space_loss_weight = 0
        self.labeldist = labeldist
        self.vlabeldist = None
        self.lsm_weight = lsm_weight
        self.fused_lstm = True     # training loop: every LSTMCell on the library's kernels (lstm.py); False = torch.nn.LSTMCell

    def zero_state(self, hpad):
        return hpad.new_zeros(hpad.size(0), self.dunits)

    # ------------------------------------------------------------------------------------------ training
    def forward(self, hpad, hlen, ys, scheduled_sampling_rate=0.0):
        """model/e2e_decoder.py:79-167.  Returns (loss, acc)."""
        dev = self.embed.weight.device
        if not (torch.is_tensor(hlen) and hlen.is_cuda):      # a device tensor of lengths stays on the device
            hlen = list(map(int, hlen))
        hpad = mask_by_length(hpad.to(dev), hlen, 0)
        self.loss = None
        ys = [y.to(dev) for y in ys]
        if ys[0].is_cuda:
            if not hasattr(self, "_label_tables"):
                import collections
                self._label_tables = collections.deque(maxlen=16)
            pad_ys_in, pad_ys_out = _label_batches(ys, self.sos, self.eos, self.ignore_id, self._label_tables)
            ys_in_lens = [int(y.size(0)) + 1 for y in ys]
        else:
            eos = torch.full((1,), self.eos, dtype=ys[0].dtype, device=ys[0].device)
            sos = torch.full((1,), self.sos, dtype=ys[0].dtype, device=ys[0].device)
            ys_in = [torch.cat([sos, y], dim=0) for y in ys]
            ys_out = [torch.cat([y, eos], dim=0) for y in ys]
            pad_ys_in = pad_list(ys_in, self.eos)
            pad_ys_out = pad_list(ys_out, self.ignore_id)
            ys_in_lens = [len(x) for x in ys_in]
        batch, olength = pad_ys_out.size(0), pad_ys_out.size(1)
        c_list = [self.zero_state(hpad) for _ in range(self.dlayers)]
        z_list = [self.zero_state(hpad) for _ in range(self.dlayers)]
        att_w = None
        y_all = []
        self.att.reset()
        y_i = None
        fused = self.fused_lstm and dev.type == 'cuda'
        sampling = scheduled_sampling_rate > 0.0
        # Teacher forcing (scheduled_sampling_rate == 0, the scripts' default): no step ever looks at its own output
        # distribution, so the output layer of ALL positions is one dense product after the loop (tcgen05 3xTF32 GEMM,
        # (B*olength) x odim x dunits) instead of olength skinny ones inside it -- same values as model/e2e_decoder.py:150.
        # With scheduled sampling the fused loop keeps that product after the loop too: a sampled position only needs
        # the previous position's arg-max, which re2e_sample_tokens takes from the top-layer state on the device.
        batched_output = fused or not sampling
        if fused and sampling:
            # the embedding half is looked up by token from a per-token table; tok (olength, B) starts as the teacher
            # tokens and a flagged position i >= 1 overwrites row i with the previous position's arg-max
            flags = self._sampling_flags(olength, scheduled_sampling_rate, dev)
            tok = pad_ys_in.t().to(torch.int32).contiguous()
            lstm0 = LSTMLoop.by_token(self.decoder[0], self.embed.weight, tok)
            w_out, b_out = _lib.f32c(self.output.weight.detach()), _lib.f32c(self.output.bias.detach())
            ws = self._sampling_ws(batch, dev)
            self._ss_tokens = tok
        else:
            eys = self.embed(pad_ys_in)
            # ... and the embedding half of the first LSTMCell's input product is one dense product before the loop; per
            # position only the context / state products (batch-sized) and one fused pointwise kernel remain (lstm.py)
            lstm0 = LSTMLoop(self.decoder[0], eys) if (fused and not sampling) else None
        # layers 1 .. dlayers-1 (input: the layer below's state) on the same step kernel, one launch per layer and position
        upper = [LSTMLoop.stacked(self.decoder[l]) for l in range(1, self.dlayers)] if fused else None
        z_top = []
        for i in range(olength):
            att_c, att_w = self.att(hpad, hlen, z_list[0], att_w)
            if lstm0 is not None:
                if not sampling:
                    random.random()                              # (the reference draws one number per position)
                elif i > 0:                                      # (the draws were taken up front, see _sampling_flags)
                    zt = _lib.f32c(z_list[-1].detach())
                    with _lib.on(dev):
                        _lib.check(_lib.lib().re2e_sample_tokens(_lib.ptr(zt), _lib.ptr(w_out), _lib.ptr(b_out),
                                                                 _lib.ptr(flags[i]), _lib.ptr(tok[i]), _lib.ptr(ws), batch,
                                                                 w_out.size(0), w_out.size(1), _lib.stream_ptr()),
                                   "re2e_sample_tokens")
                z_list[0], c_list[0] = lstm0.step(i, att_c, z_list[0], c_list[0])
            else:
                if random.random() < scheduled_sampling_rate and i > 0:
                    topi = y_i.topk(1)[1].squeeze(1)
                    ey = torch.cat((self.embed(topi), att_c), dim=1)
                else:
                    ey = torch.cat((eys[:, i, :], att_c), dim=1)
                z_list[0], c_list[0] = self.decoder[0](ey, (z_list[0], c_list[0]))
            for l in range(1, self.dlayers):
                if upper is not None:
                    z_list[l], c_list[l] = upper[l - 1].step(i, z_list[l - 1], z_list[l], c_list[l])
                else:
                    z_list[l], c_list[l] = self.decoder[l](z_list[l - 1], (z_list[l], c_list[l]))
            if batched_output:
                z_top.append(z_list[-1])
            else:
                y_i = self.output(z_list[-1])
                y_all.append(y_i)
        if batched_output:
            z_all = torch.stack(z_top, dim=1)                                   # (B, olength, dunits)
            y_all = linear(z_all, self.output.weight, self.output.bias).reshape(batch * olength, -1)
        else:
            y_all = torch.stack(y_all, dim=0).transpose(0, 1).contiguous().view(batch * olength, -1)
        if y_all.is_cuda and pad_ys_out.dtype == torch.int64:
            # cross-entropy + the arg-max for th_accuracy from one pass over the logits (csrc/ctc.cu)
            self.loss, best = _CrossEntropy.apply(y_all, pad_ys_out.reshape(-1), self.ignore_id)
            self.loss = self.loss * (np.mean(ys_in_lens) - 1)   # quirk 7 of SURVEY.md 8a
            acc = th_accuracy(y_all, pad_ys_out, ignore_label=self.ignore_id, pred=best.view(pad_ys_out.shape))
        else:
            self.loss = F.cross_entropy(y_all, pad_ys_out.view(-1), ignore_index=self.ignore_id, reduction='mean')
            self.loss = self.loss * (np.mean(ys_in_lens) - 1)   # quirk 7 of SURVEY.md 8a
            acc = th_accuracy(y_all, pad_ys_out, ignore_label=self.ignore_id)
        if self.labeldist is not None:
            if self.vlabeldist is None:
                self.vlabeldist = torch.from_numpy(self.labeldist).to(dev)
            loss_reg = -torch.sum((F.log_softmax(y_all, dim=1) * self.vlabeldist).view(-1), dim=0) / len(ys_in_lens)
            self.loss = (1. - self.lsm_weight) * self.loss + self.lsm_weight * loss_reg
        return self.loss, acc

    def _sampling_flags(self, olength, rate, dev):
        """Device int32 (olength,) flags of one scheduled-sampling forward: flag i = (draw_i < rate and i > 0), with the
        olength draws of random.random() taken here, in the reference's order (one per position, position 0 included).
        They travel through a page-locked buffer, so a captured graph re-reads it at every replay (draw_sampling)."""
        pin = torch.empty(olength, dtype=torch.int32).pin_memory()
        self._fill_flags(pin, rate)
        if torch.cuda.is_current_stream_capturing():
            # kept for the module's life: the graph re-reads `pin` at every replay, and freeing the previous buffer
            # inside the capture would record its reuse event into the graph (torch's page-locked allocator then fails
            # on its next allocation)
            self.__dict__.setdefault("_ss_pins", []).extend(p for p in (getattr(self, "_ss_flags", None), pin)
                                                            if p is not None)
        self._ss_flags = pin
        return pin.to(dev, non_blocking=True)

    @staticmethod
    def _fill_flags(pin, rate):
        pin.numpy()[:] = [1 if (random.random() < rate and i > 0) else 0 for i in range(pin.numel())]

    def _sampling_ws(self, batch, dev):
        """Scratch of re2e_sample_tokens: zero when allocated, left zero by every call, so it is kept across forwards."""
        ws = getattr(self, "_ss_ws", None)
        n = (int(_lib.lib().re2e_sample_tokens_ws_bytes(batch)) + 7) // 8
        if ws is None or ws.device != dev or ws.numel() < n:
            ws = self._ss_ws = torch.zeros(n, dtype=torch.int64, device=dev)
        return ws

    def draw_sampling(self, scheduled_sampling_rate):
        """New draws for the most recent scheduled-sampling forward (the one a captured CUDA graph replays): one
        random.random() per position, exactly as an eager forward at this rate would take them.  Waits for the device
        first, so a replay still in flight keeps the flags it started with.  A job that ramps the rate up captures the
        forward + backward once (at a rate > 0) and calls ``draw_sampling(rate_k)`` before each replay."""
        pin = getattr(self, "_ss_flags", None)
        if pin is None:
            raise RuntimeError("draw_sampling: no scheduled-sampling forward has run on this decoder")
        torch.cuda.synchronize(self.embed.weight.device)
        self._fill_flags(pin, scheduled_sampling_rate)

    # ------------------------------------------------------------------------------------------ beam search
    @torch.no_grad()
    def _beam_tables(self):
        """Per-model constants of the fused beam-search position: the embedding half of the LSTMCell input product for
        EVERY token (V, 4Z) = embed.weight @ W_ih[:, :E]^T + b_ih + b_hh (looked up by token in the step kernel), the
        recurrent matrices side by side (4Z, D+Z), the output layer, and per upper layer (decoder[1:]) its matrices side
        by side [W_ih | W_hh] (4Z, 2Z) with its gate row b_ih + b_hh (1, 4Z).  Built once per recognize_beam /
        recognize_beam_batch call, never cached across calls: a write through ``.data`` (checkpoint averaging, a
        training step between decodes) changes a parameter without bumping its version counter, so no cache key can see
        it, and stale tables would make the fused search silently decode with the old weights."""
        cell = self.decoder[0]
        E = self.embed.weight.size(1)
        eg = linear(_lib.f32c(self.embed.weight.detach()), cell.weight_ih.detach()[:, :E].contiguous(),
                    (cell.bias_ih + cell.bias_hh).detach()).contiguous()
        wcat = torch.cat((cell.weight_ih.detach()[:, E:], cell.weight_hh.detach()), 1).float().contiguous()
        upper = [(torch.cat((c.weight_ih.detach(), c.weight_hh.detach()), 1).float().contiguous(),
                  _lib.f32c((c.bias_ih + c.bias_hh).detach()).view(1, -1)) for c in self.decoder[1:]]
        return eg, wcat, _lib.f32c(self.output.weight.detach()), _lib.f32c(self.output.bias.detach()), upper

    def _fused_position(self, hb, lpz, Cb, beam, ctc_weight, maxlen, hist, tables):
        """One output position for all W rows as launches of the library over static buffers (csrc/beam.cu):
        AttLoc step, LSTMCell step (embedding half by token lookup), one LSTMCell step per upper layer (context = the
        new state of the layer below, gate row b_ih + b_hh through the all-zero row index ``zrow``), output layer on the
        top layer, log-softmax + top-Cb, CTC prefix scores, then joint score + merge + gather of the chosen rows' states
        (z and c of every layer, alignment, CTC) for the next position (one launch, ``re2e_beam_advance``).
        ``hist`` (>= maxlen, 4, beam): page-locked host tensor the winners of every position are written to.  ``tables``: ``_beam_tables()`` of this call.  Returns the
        position closure.  The first position needs no special case: the states start as every row's initial state."""
        import ctypes
        lib = _lib.lib()
        dev = hb.device
        W, Th, D = hb.shape
        Z, V = self.dunits, self.output.out_features
        NL = self.dlayers
        eg, wcat, w_out, b_out, upper = tables
        st = self.att.precompute(hb)
        _, _, _, A, _, C, K = st.dims
        W_dec, W_att, W_conv, gvec, gvec_b = st.weights
        # every buffer of the search carved out of two allocations (fp32 / int32); `hist` is page-locked HOST memory that
        # the merge kernel writes directly (160 B per position over the bus: no copy, the host just waits for an event)
        use_ctc = lpz is not None
        # z / c of the layers back to back, (NL, W, Z) per buffer: re2e_beam_init zeroes all layers' inputs at once
        sizes = [("sc", W), ("z_st", NL * W * Z), ("c_st", NL * W * Z), ("z_in", NL * W * Z), ("c_in", NL * W * Z),
                 ("a_st", W * Th), ("a_in", W * Th), ("att_c", W * D), ("act", W * 4 * Z), ("logits", W * V),
                 ("top_v", W * Cb)]
        if use_ctc:
            sizes += [("r_st", W * Cb * Th * 2), ("r_in", W * Th * 2), ("psi_st", W * Cb), ("psi_in", W)]
        flat = torch.empty(sum((n_ + 3) // 4 * 4 for _, n_ in sizes), device=dev, dtype=torch.float32)
        bufs, o = {}, 0
        for name, n_ in sizes:
            bufs[name] = flat[o:o + n_]
            o += (n_ + 3) // 4 * 4
        ints = torch.empty(4 * W + 4 + W * Cb + (W if NL > 1 else 0), device=dev, dtype=torch.int32)
        ctl, state, top_i = ints[:4 * W].view(4, W), ints[4 * W:4 * W + 2], ints[4 * W + 4:4 * W + 4 + W * Cb]
        zrow = ints[4 * W + 4 + W * Cb:].zero_() if NL > 1 else None
        sc = bufs["sc"]
        z_st, c_st, z_in, c_in = (bufs[k_].view(NL, W * Z) for k_ in ("z_st", "c_st", "z_in", "c_in"))
        a_st, a_in, att_c, act, logits, top_v = (bufs[k_] for k_ in ("a_st", "a_in", "att_c", "act", "logits", "top_v"))
        segs = [(z_st[0], z_in[0], Z, 0), (c_st[0], c_in[0], Z, 0), (a_st, a_in, Th, 0)]
        for l in range(1, NL):
            segs += [(z_st[l], z_in[l], Z, 0), (c_st[l], c_in[l], Z, 0)]
        r_st = r_in = psi_st = psi_in = None
        if use_ctc:
            r_st, r_in, psi_st, psi_in = bufs["r_st"], bufs["r_in"], bufs["psi_st"], bufs["psi_in"]
            segs += [(r_st, r_in, 2 * Th, Cb), (psi_st, psi_in, 1, Cb)]
        n = len(segs)
        src = (ctypes.c_void_p * n)(*[s[0].data_ptr() for s in segs])
        dst = (ctypes.c_void_p * n)(*[s[1].data_ptr() for s in segs])
        rowf = (ctypes.c_int * n)(*[s[2] for s in segs])
        subc = (ctypes.c_int * n)(*[s[3] for s in segs])
        w_att, w_ctc = float(1.0 - ctc_weight), float(ctc_weight)
        P = _lib.ptr
        with _lib.on(dev):
            _lib.check(lib.re2e_beam_init(P(z_in), P(c_in), P(a_in), P(r_in), P(psi_in), P(lpz), P(ctl), P(sc), P(state), W,
                                          NL * Z, Th, V, 0, self.sos, _lib.stream_ptr()), "re2e_beam_init")

        def build(sp):
            """The position's launches with their argument tuples, for one stream (everything else is constant)."""
            calls = [
                (lib.re2e_attloc_step_fwd, "re2e_attloc_step_fwd",
                 (P(st.pre), P(st.enc), P(z_in), P(a_in), P(W_dec), P(W_att), P(W_conv), P(gvec), P(gvec_b), 2.0, P(att_c),
                  P(a_st), None, None, None, W, Th, D, A, Z, C, K, sp)),
                (lib.re2e_lstm_step_fwd, "re2e_lstm_step_fwd",
                 (P(att_c), P(z_in[0]), P(c_in[0]), P(wcat), P(eg), P(ctl[2]), P(act), P(c_st[0]), P(z_st[0]), W, D, Z, sp)),
            ] + [
                (lib.re2e_lstm_step_fwd, "re2e_lstm_step_fwd",
                 (P(z_st[l - 1]), P(z_in[l]), P(c_in[l]), P(upper[l - 1][0]), P(upper[l - 1][1]), P(zrow), P(act),
                  P(c_st[l]), P(z_st[l]), W, Z, Z, sp)) for l in range(1, NL)
            ] + [
                (lib.re2e_batch_nt, "re2e_batch_nt", (P(z_st[NL - 1]), P(w_out), P(b_out), P(logits), W, V, Z, 0, sp)),
                (lib.re2e_log_softmax_topk, "re2e_log_softmax_topk", (P(logits), W, V, Cb, None, P(top_v), P(top_i), sp)),
            ]
            if lpz is not None:
                calls.append((lib.re2e_ctc_prefix_score, "re2e_ctc_prefix_score",
                              (P(lpz), P(r_in), P(top_i), P(ctl[2]), P(ctl[3]), P(psi_st), P(r_st), Th, V, W, Cb, 0,
                               self.eos, sp)))
            calls.append((lib.re2e_beam_advance, "re2e_beam_advance",
                          (P(top_v), P(top_i), P(psi_st), P(psi_in), P(sc), w_att, w_ctc, W, Cb, beam, P(state), P(ctl),
                           P(hist), self.eos, maxlen, n, src, dst, rowf, subc, sp)))
            return calls

        built = {}

        def position():
            key = torch.cuda.current_stream(dev).cuda_stream
            calls = built.get(key)
            if calls is None:
                calls = built[key] = build(ctypes.c_void_p(key))
            with _lib.on(dev):
                for fn, name, args in calls:
                    rc = fn(*args)
                    if rc != 0:
                        _lib.check(rc, name)

        position.keep = (flat, ints, eg, wcat, w_out, b_out, upper, lpz, st)   # buffers a captured graph points into
        return position

    def _host_merge(self, hyps, ended_hyps, entries, i, maxlen, minlen, penalty):
        """The reference's bookkeeping for one position (model/e2e_decoder.py:296-333) given the merged candidates, best
        first: ``entries`` = (score, index of the parent in ``hyps``, token, candidate index).  Appends finished
        hypotheses to ``ended_hyps`` (length penalty added) and returns the ones that go on.  Live hypotheses are
        (score, token, parent hypothesis, length) tuples -- the token sequence is only materialised for the ones that
        end (the reference copies ``yseq`` for every candidate at every position)."""
        remained = []
        last = i == maxlen - 1
        for s_, r, t, j in entries:
            parent = hyps[r]
            n = parent[3] + 1
            if last or t == self.eos:
                if n + (1 if last else 0) > minlen:
                    yseq = [self.eos] if last else []
                    yseq.append(t)
                    node = parent
                    while node is not None:
                        yseq.append(node[1])
                        node = node[2]
                    yseq.reverse()
                    ended_hyps.append({'score': np.float32(np.float32(s_) + np.float32((i + 1) * penalty)), 'yseq': yseq})
            else:
                remained.append((np.float32(s_), t, parent, n, r, j))
        return remained

    def _recognize_fused(self, hb, lpz, recog_args, Cb, maxlen, minlen):
        """Beam search with the whole position on the device, one utterance on the current stream (``_FusedSearch``)."""
        search = _FusedSearch(self, hb, lpz, recog_args, Cb, maxlen, minlen, torch.cuda.current_stream(hb.device), 0,
                              self._beam_tables())
        while not search.done:
            search.pump()
            search.poll(block=True)
        return search.result()

    def _fused_plan(self, h, lpz, recog_args):
        """Shapes of one utterance's search and whether the fused position takes it: (hb, lpz, Cb, maxlen, minlen) or None."""
        dev = self.embed.weight.device
        h = _lib.f32c(h.detach(), dev)
        Th = h.size(0)
        beam = int(recog_args.beam_size)
        maxlen = Th if recog_args.maxlenratio == 0 else max(1, int(recog_args.maxlenratio * Th))
        minlen = int(recog_args.minlenratio * Th)
        Cb = beam
        if lpz is not None:
            lpz = _lib.f32c(lpz.detach(), dev)
            V = lpz.size(-1)
            Cb = min(V, int(beam * CTC_SCORING_RATIO)) if recog_args.ctc_weight != 1.0 else V
        lib = _lib.lib()
        if not (self.dlayers <= FUSED_MAX_LAYERS and beam <= Cb <= 32
                and self.output.out_features <= 8192
                and bool(lib.re2e_lstm_step_supported(beam, h.size(1), self.dunits))
                and (self.dlayers == 1 or bool(lib.re2e_lstm_step_supported(beam, self.dunits, self.dunits)))):
            return None
        hb = h.unsqueeze(0).expand(beam, Th, h.size(1)).contiguous()
        return hb, lpz, Cb, maxlen, minlen

    def recognize_beam_batch(self, hs, lpzs, recog_args, char_list=None, rnnlm=None, fstlm=None, concurrency=4):
        """``recognize_beam`` for a list of utterances (``hs[i]`` (Th_i, D), ``lpzs[i]`` (Th_i, V) or None); returns the list
        of n-best lists, identical to calling ``recognize_beam`` per utterance.  An extension of the reference API
        (joint_recog.py:143-149 decodes one utterance at a time): a single search is a strictly serial chain of short
        kernels that leaves most of the GPU idle, so up to ``concurrency`` searches run interleaved, each with its own
        static buffers, CUDA graph and stream; the host pumps them round-robin."""
        if rnnlm is not None or fstlm is not None:
            raise NotImplementedError("LM rescoring is outside the hot path (SURVEY.md section 8)")
        n = len(hs)
        results = [None] * n
        dev = self.embed.weight.device
        cur = torch.cuda.current_stream(dev)
        streams = getattr(self, "_search_streams", None)
        if streams is None or len(streams) < concurrency or streams[0].device != dev:
            streams = self._search_streams = [torch.cuda.Stream(dev) for _ in range(concurrency)]
        active = {}                       # slot -> (utterance index, search)
        tables = None                     # made on the caller's stream, which every search stream waits for below
        nxt = 0
        while nxt < n or active:
            for slot in range(concurrency):
                if slot not in active and nxt < n:
                    i, nxt = nxt, nxt + 1
                    lp = lpzs[i] if lpzs is not None else None
                    plan = self._fused_plan(hs[i], lp, recog_args)
                    if plan is None:      # shapes the fused position does not take: the per-utterance path
                        results[i] = self._recognize_generic(hs[i], lp, recog_args)
                        continue
                    if tables is None:
                        tables = self._beam_tables()
                    for t in plan[:2]:    # made on the caller's stream, consumed on the search's
                        if t is not None:
                            t.record_stream(streams[slot])
                    streams[slot].wait_stream(cur)
                    self.att.reset()
                    active[slot] = (i, _FusedSearch(self, plan[0], plan[1], recog_args, plan[2], plan[3], plan[4],
                                                    streams[slot], slot, tables))
            progressed = False
            for slot, (i, srch) in list(active.items()):
                srch.pump()
                progressed |= srch.poll(block=False)
                if srch.done:
                    results[i] = srch.result()
                    del active[slot]
                    progressed = True
            if not progressed and active:
                slot = next(iter(active))
                i, srch = active[slot]
                srch.poll(block=True)
                if srch.done:
                    results[i] = srch.result()
                    del active[slot]
        for st_ in streams[:concurrency]:
            cur.wait_stream(st_)
        return results

    def recognize_beam(self, h, lpz, recog_args, char_list=None, rnnlm=None, fstlm=None):
        """h (Th, D) encoder output of one utterance, lpz (Th, V) CTC log-probs or None.
        Returns the n-best list of dicts with 'score' (float) and 'yseq' (list of int, <sos> first)."""
        if rnnlm is not None or fstlm is not None:
            raise NotImplementedError("LM rescoring is outside the hot path (SURVEY.md section 8)")
        _lib.lib()
        plan = self._fused_plan(h, lpz, recog_args)
        if plan is None:
            return self._recognize_generic(h, lpz, recog_args)
        self.att.reset()
        return self._recognize_fused(*plan[:2], recog_args, *plan[2:])

    def _recognize_generic(self, h, lpz, recog_args):
        """``recognize_beam`` on the generic position, for the shapes ``_fused_plan`` does not take; tests compare the
        fused position against it."""
        self.att.reset()
        dev = self.embed.weight.device
        h = _lib.f32c(h.detach(), dev)
        Th = h.size(0)
        beam = int(recog_args.beam_size)
        penalty = recog_args.penalty
        ctc_weight = recog_args.ctc_weight
        W = beam                                   # hypothesis rows on the device (constant -> one AttLoc cache shape)
        hb = h.unsqueeze(0).expand(W, Th, h.size(1)).contiguous()
        hlens = [Th] * W
        maxlen = Th if recog_args.maxlenratio == 0 else max(1, int(recog_args.maxlenratio * Th))
        minlen = int(recog_args.minlenratio * Th)
        use_ctc = lpz is not None
        if use_ctc:
            lpz = _lib.f32c(lpz.detach(), dev)
            V = lpz.size(-1)
            ctc_beam = min(V, int(beam * CTC_SCORING_RATIO)) if ctc_weight != 1.0 else V

        # ---- generic position (any layer count / candidate width): tensor ops + the library's AttLoc / CTC kernels
        z = [h.new_zeros(W, self.dunits) for _ in range(self.dlayers)]
        c = [h.new_zeros(W, self.dunits) for _ in range(self.dlayers)]
        if use_ctc:
            # CTCPrefixScore.initial_state (model/e2e_ctc.py:95-107), replicated for every row
            r0 = torch.full((Th, 2), -10000000000.0, device=dev, dtype=torch.float32)
            r0[:, 1] = torch.cumsum(lpz[:, 0], dim=0)
            r_prev = r0.unsqueeze(0).expand(W, Th, 2).contiguous()
            ctc_prev = torch.zeros(W, device=dev, dtype=torch.float32)
        # ---- static device buffers: one output position = one fixed sequence of launches over them, so positions >= 2
        #      are replayed from a CUDA graph (captured once per utterance); the host only exchanges two small packed
        #      arrays per position (control in, candidates out) through pinned memory
        L = self.dlayers
        idt = torch.long
        ctl = torch.zeros(4, W, dtype=idt, device=dev)                 # rows: parent, ctc candidate, token, position
        sc = torch.zeros(W, dtype=torch.float32, device=dev)           # accumulated scores of the rows
        out = torch.empty(3, W, beam, dtype=torch.float32, device=dev)   # candidate scores, token ids, ctc candidate idx
        pins = getattr(self, "_pinned", None)          # page-locked staging is expensive to allocate: keep it per beam
        if pins is None or pins[0].shape[1] != W or pins[2].shape[2] != beam or pins[0].dtype != idt:
            pins = (torch.zeros(4, W, dtype=idt).pin_memory(), torch.zeros(W, dtype=torch.float32).pin_memory(),
                    torch.empty(3, W, beam, dtype=torch.float32).pin_memory())
            self._pinned = pins
        ctl_h, sc_h, out_h = pins
        ctl_h.zero_()
        sc_h.zero_()
        ctl_np, sc_np, out_np = ctl_h.numpy(), sc_h.numpy(), out_h.numpy()      # host views (element access is cheap)
        st_a = torch.empty(W, Th, dtype=torch.float32, device=dev)
        if use_ctc:
            st_r = torch.empty(W, ctc_beam, Th, 2, dtype=torch.float32, device=dev)
            st_psi = torch.empty(W, ctc_beam, dtype=torch.float32, device=dev)

        def dev_step(first):
            vy = ctl[2]
            if first:
                zz, cc, a_prev = z, c, None
                if use_ctc:
                    rp, cp = r_prev, ctc_prev
            else:
                P = ctl[0]
                zz = [t.index_select(0, P) for t in z]
                cc = [t.index_select(0, P) for t in c]
                a_prev = st_a.index_select(0, P)
                if use_ctc:
                    rp = st_r[P, ctl[1]].contiguous()
                    cp = st_psi[P, ctl[1]].contiguous()
            ey = self.embed(vy)
            att_c, att_w = self.att(hb, hlens, zz[0], a_prev)
            ey = torch.cat((ey, att_c), dim=1)
            z_new, c_new = list(zz), list(cc)
            z_new[0], c_new[0] = self.decoder[0](ey, (zz[0], cc[0]))
            for l in range(1, L):
                z_new[l], c_new[l] = self.decoder[l](z_new[l - 1], (zz[l], cc[l]))
            local_att = log_softmax_rows(self.output(z_new[-1]))                    # (W, V)
            if use_ctc:
                _, ids = torch.topk(local_att, ctc_beam, dim=1)                     # attention pre-pruning
                log_psi, r_new = ctc_prefix_score_batch(lpz, rp, ids.to(torch.int32).contiguous(), vy.to(torch.int32),
                                                        ctl[3].to(torch.int32), 0, self.eos)
                local = (1.0 - ctc_weight) * local_att.gather(1, ids) + ctc_weight * (log_psi - cp.unsqueeze(1))
                best_scores, joint = torch.topk(local, beam, dim=1)
                best_ids = ids.gather(1, joint)
                st_r.copy_(r_new)
                st_psi.copy_(log_psi)
            else:
                best_scores, best_ids = torch.topk(local_att, beam, dim=1)
                joint = best_ids
            for l in range(L):
                z[l].copy_(z_new[l])
                c[l].copy_(c_new[l])
            st_a.copy_(att_w)
            cand = sc.unsqueeze(1) + best_scores                                    # fp32, as hyp['score'] + tensor
            out.copy_(torch.stack((cand, best_ids.float(), joint.float()), 0))

        use_graph = bool(getattr(recog_args, "cuda_graph", True)) and maxlen >= 6
        graph = None
        hyps = [(np.float32(0.0), self.sos, None, 1)]               # (score, token, parent, length, row, ctc candidate)
        ended_hyps = []
        for i in range(maxlen):
            n = len(hyps)
            ctl_np[2, :] = [hyps[min(k, n - 1)][1] for k in range(W)]
            ctl_np[3, :] = i
            ctl.copy_(ctl_h, non_blocking=True)
            sc.copy_(sc_h, non_blocking=True)
            if i == 0:
                dev_step(True)
            elif i == 1 or not use_graph:
                dev_step(False)
            else:
                if graph is None:
                    # raw capture_begin / capture_end on a side stream: the torch.cuda.graph context manager also runs
                    # gc.collect() and empty_cache(), tens of milliseconds per utterance
                    cur = torch.cuda.current_stream(dev)
                    if getattr(self, "_cap_stream", None) is None or self._cap_stream.device != dev:
                        self._cap_stream = torch.cuda.Stream(dev)
                        self._graph_pool = None
                    if getattr(self, "_graph_pool", None) is None:     # (a fused search creates the stream only)
                        self._graph_pool = torch.cuda.graph_pool_handle()
                    self._cap_stream.wait_stream(cur)
                    graph = torch.cuda.CUDAGraph()
                    with torch.cuda.stream(self._cap_stream):
                        graph.capture_begin(pool=self._graph_pool)
                        dev_step(False)
                        graph.capture_end()
                    cur.wait_stream(self._cap_stream)
                    # the shared pool lives as long as one graph references it: keep this utterance's graph until the
                    # next one has been captured (then its blocks return to the pool)
                    self._last_graph = graph
                graph.replay()
            out_h.copy_(out, non_blocking=True)
            torch.cuda.current_stream(dev).synchronize()
            cand_h = out_np[0, :n]
            ids_h, joint_h = out_np[1, :n].astype(np.int64), out_np[2, :n].astype(np.int64)
            # the reference merges hypothesis by hypothesis with a stable descending sort truncated to `beam`
            # (model/e2e_decoder.py:296-314) == one stable descending sort over (hypothesis, rank) order
            order = np.argsort(-cand_h.reshape(-1), kind='stable')[:beam]
            entries = []
            for k in order:
                r, j = divmod(int(k), beam)
                entries.append((cand_h[r, j], r, int(ids_h[r, j]), int(joint_h[r, j]) if use_ctc else j))
            remained = self._host_merge(hyps, ended_hyps, entries, i, maxlen, minlen, penalty)
            if end_detect(ended_hyps, i) and recog_args.maxlenratio == 0.0:
                break
            hyps = remained
            if len(hyps) == 0:
                break
            # control block of the next position: parent row, ctc candidate and score of every surviving hypothesis
            # (spare rows repeat the last one)
            rows = [hyps[min(k, len(hyps) - 1)] for k in range(W)]
            ctl_np[0, :] = [hk[4] for hk in rows]
            ctl_np[1, :] = [hk[5] if use_ctc else 0 for hk in rows]
            sc_np[:] = [hk[0] for hk in rows]
        nbest = sorted(ended_hyps, key=lambda x: x['score'], reverse=True)[:min(len(ended_hyps), recog_args.nbest)]
        return [{'score': float(x['score']), 'yseq': [int(t) for t in x['yseq']]} for x in nbest]
