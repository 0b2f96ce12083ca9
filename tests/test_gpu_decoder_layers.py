"""GPU: decoders with more than one LSTMCell layer (``--dlayers N``, model/e2e_decoder.py: LSTMCell(dunits + eprojs,
dunits) followed by N-1 LSTMCell(dunits, dunits)) on the library's kernels:

* ``LSTMLoop.stacked`` (an upper layer on re2e_lstm_step_fwd / _bwd, or the composed path for dunits > 640) against
  torch.nn.LSTMCell, states and every gradient, fp64 as tie-breaker;
* ``Decoder.forward`` + backward with dlayers 2 and 3 (teacher forcing with and without label smoothing, scheduled
  sampling) against the library-free loop and an fp64 CPU restatement, with the upper cells' torch forward disabled;
  the same forward + backward captured into a CUDA graph and replayed on another batch;
* the fused beam-search position for dlayers 2..6 against the generic position, ``recognize_beam_batch`` against
  per-utterance searches, deeper decoders through the generic position;
* the beam kernels' side of it through the C ABI: gathers of 2 * layers + 3 state tensors, and the initial state of
  all layers;
* the reference's own ``E2E`` with dlayers = 2 and the swapped ``Decoder`` (skipped without the reference tree)."""
import copy
import ctypes
import random
import types

import numpy as np
import pytest
import torch

import helpers
from oracle import attloc as oatt
from oracle import beam as obeam
from oracle import refshim
from robust_e2e_gan_b200 import CTC, AttLoc, Decoder, _lib
from robust_e2e_gan_b200.e2e_decoder import FUSED_MAX_LAYERS
from robust_e2e_gan_b200.lstm import LSTMLoop

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _randn(g, *shape, fan):
    return torch.randn(*shape, generator=g) / fan ** 0.5


def _no_torch_cell(dec):
    """Make torch.nn.LSTMCell.forward of the upper cells raise: the fused paths must not call it."""
    def boom(*a, **k):
        raise AssertionError("torch.nn.LSTMCell called on an upper decoder layer")
    for cell in dec.decoder[1:]:
        cell.forward = boom


def _torch_cell_back(dec):
    for cell in dec.decoder[1:]:
        cell.__dict__.pop("forward", None)


# ---------------------------------------------------------------------------------------------- LSTMLoop.stacked
@pytest.mark.parametrize("B,Z,D,L", [(4, 48, 64, 21), (10, 300, 320, 20), (32, 300, 320, 22), (3, 644, 36, 20)])
def test_stacked_loop_matches_torch_lstmcell(B, Z, D, L):
    """LSTMLoop(cell0, eys) followed by LSTMLoop.stacked(cell1) over L positions against two torch.nn.LSTMCell: h of both
    layers at every position and the gradients of the embeddings, the contexts and all eight parameters.  Z = 48 / 300
    run the cluster kernels, Z = 644 the composed batch_nt + pointwise path; the upper layer adds exactly one forward
    launch per position."""
    g = torch.Generator().manual_seed(B * 7 + Z)
    cells = [torch.nn.LSTMCell(Z + D, Z), torch.nn.LSTMCell(Z, Z)]
    with torch.no_grad():
        for cell in cells:
            for p in cell.parameters():
                p.copy_(_randn(g, *p.shape, fan=cell.input_size))
    eys = torch.randn(B, L, Z, generator=g)
    ctxs = torch.randn(L, B, D, generator=g)
    gz = torch.randn(2, L, B, Z, generator=g)

    def run_ref(dt):
        cs = [copy.deepcopy(c).to(dt) for c in cells]
        e = eys.detach().clone().to(dt).requires_grad_(True)
        cx = ctxs.detach().clone().to(dt).requires_grad_(True)
        h = [torch.zeros(B, Z, dtype=dt) for _ in range(2)]
        c = [torch.zeros(B, Z, dtype=dt) for _ in range(2)]
        hs = [[], []]
        for i in range(L):
            h[0], c[0] = cs[0](torch.cat((e[:, i, :], cx[i]), 1), (h[0], c[0]))
            h[1], c[1] = cs[1](h[0], (h[1], c[1]))
            hs[0].append(h[0])
            hs[1].append(h[1])
        hs = torch.stack([torch.stack(x) for x in hs])
        ((hs * gz.to(dt)).sum() + c[1].sum()).backward()
        return [hs.detach(), e.grad, cx.grad] + [p.grad for cc in cs for p in cc.parameters()]

    r32, r64 = run_ref(torch.float32), run_ref(torch.float64)
    cd = [copy.deepcopy(c).to(DEV) for c in cells]
    e = eys.detach().clone().to(DEV).requires_grad_(True)
    cx = ctxs.detach().clone().to(DEV).requires_grad_(True)
    loop0, loop1 = LSTMLoop(cd[0], e), LSTMLoop.stacked(cd[1])
    h = [torch.zeros(B, Z, device=DEV) for _ in range(2)]
    c = [torch.zeros(B, Z, device=DEV) for _ in range(2)]
    hs = [[], []]
    for i in range(L):
        h[0], c[0] = loop0.step(i, cx[i], h[0], c[0])
        n0 = _lib.launch_count()
        h[1], c[1] = loop1.step(i, h[0], h[1], c[1])
        n1 = _lib.launch_count() - n0
        assert n1 == (1 if Z <= 640 else 3), n1         # one cluster launch, or two products + the pointwise kernel
        hs[0].append(h[0])
        hs[1].append(h[1])
    hs = torch.stack([torch.stack(x) for x in hs])
    ((hs * gz.to(DEV)).sum() + c[1].sum()).backward()
    got = [hs.detach(), e.grad, cx.grad] + [p.grad for cc in cd for p in cc.parameters()]
    names = ["h of both layers at every position", "d embeddings", "d contexts"] + \
        ["layer %d: d %s" % (l, n) for l in (0, 1) for n in ("weight_ih", "weight_hh", "bias_ih", "bias_hh")]
    for a, b32, b64, what in zip(got, r32, r64, names):
        helpers.assert_close(a, b32, truth=b64, what=what)


# ---------------------------------------------------------------------------------------------- training
def _flags(seed, rate, L):
    random.seed(seed)
    return [random.random() < rate and i > 0 for i in range(L)]


def ref_forward(sd, hpad, hlen, ys, sos, eos, dlayers, flags, lsm=0.0, ignore_id=-1):
    """model/e2e_decoder.py:79-167 for ``dlayers`` LSTMCell layers on CPU autograd (oracle AttLoc step and LSTMCell
    arithmetic): teacher forcing, or scheduled sampling where ``flags[i]`` (the reference's ``random.random() < rate
    and i > 0``) feeds the arg-max of the previous position's logits; label smoothing with a uniform label distribution
    when ``lsm`` > 0.  Returns (loss, acc, tokens (L, B) fed at every position)."""
    att_p = {k[len("att."):]: v for k, v in sd.items() if k.startswith("att.")}
    hlen = [int(l) for l in hlen]
    mask = torch.zeros_like(hpad)
    for b, l in enumerate(hlen):
        mask[b, :l] = 1.0
    hpad = hpad * mask
    B, Z = hpad.shape[0], sd["embed.weight"].shape[1]
    ys_in = [torch.cat([y.new_tensor([sos]), y]) for y in ys]
    ys_out = [torch.cat([y, y.new_tensor([eos])]) for y in ys]
    L = max(len(y) for y in ys_in)
    pad_in = torch.full((B, L), eos, dtype=torch.long)
    pad_out = torch.full((B, L), ignore_id, dtype=torch.long)
    for b in range(B):
        pad_in[b, :len(ys_in[b])] = ys_in[b]
        pad_out[b, :len(ys_out[b])] = ys_out[b]
    z = [hpad.new_zeros(B, Z) for _ in range(dlayers)]
    c = [hpad.new_zeros(B, Z) for _ in range(dlayers)]
    pre = oatt.precompute(att_p, hpad)
    att_w = None
    y_all, tokens = [], []
    for i in range(L):
        att_c, att_w = oatt.step(att_p, hpad, pre, hlen, z[0], att_w)
        tok = y_all[-1].detach().argmax(1) if flags[i] else pad_in[:, i]
        tokens.append(tok)
        z[0], c[0] = obeam.lstm_cell(sd, "decoder.0.", torch.cat((sd["embed.weight"][tok], att_c), dim=1), (z[0], c[0]))
        for l in range(1, dlayers):
            z[l], c[l] = obeam.lstm_cell(sd, "decoder.%d." % l, z[l - 1], (z[l], c[l]))
        y_all.append(torch.nn.functional.linear(z[-1], sd["output.weight"], sd["output.bias"]))
    y_all = torch.stack(y_all, dim=0).transpose(0, 1).contiguous().view(B * L, -1)
    loss = torch.nn.functional.cross_entropy(y_all, pad_out.view(-1), ignore_index=ignore_id, reduction='mean')
    loss = loss * (np.mean([len(x) for x in ys_in]) - 1)
    if lsm > 0:
        V = y_all.shape[1]
        reg = -torch.sum(torch.log_softmax(y_all, dim=1).view(-1) / V) / len(ys_in)
        loss = (1.0 - lsm) * loss + lsm * reg
    pred = y_all.detach().view(B, L, -1).argmax(2)
    m = pad_out != ignore_id
    acc = float((pred[m] == pad_out[m]).sum()) / float(m.sum())
    return loss, acc, torch.stack(tokens)


def _training_decoder(dlayers, lsm, V=37, D=64, Z=48, A=64, C=4, filts=5, seed=11):
    torch.manual_seed(seed)
    ld = np.full(V, 1.0 / V, dtype=np.float32) if lsm > 0 else None
    dec = Decoder(D, V, dlayers, Z, V - 1, V - 1, AttLoc(D, Z, A, C, filts, "softmax"), labeldist=ld, lsm_weight=lsm)
    return dec.to(DEV).train()


def _batch(D, V, seed=3, B=4, Th=17):
    g = torch.Generator().manual_seed(seed)
    hpad = torch.tanh(torch.randn(B, Th, D, generator=g))
    hlen = [Th, Th - 5, Th - 8, Th][:B]
    ys = [torch.randint(0, V - 1, (n,), generator=g) for n in (5, 3, 4, 6)][:B]
    return hpad, hlen, ys


@pytest.mark.parametrize("dlayers", [2, 3])
@pytest.mark.parametrize("mode", ["teacher", "teacher_lsm", "sampling"])
def test_multilayer_training_matches_library_free_loop_and_fp64(dlayers, mode):
    """Decoder.forward + backward with dlayers layers and fused_lstm on (every layer on the LSTM step kernels, the
    upper cells' torch forward made to raise) against fused_lstm = False (torch.nn.LSTMCell, per-position output layer,
    F.cross_entropy) on the same seeded draws, fp64 CPU restatement as tie-breaker: loss, accuracy, d hpad and every
    parameter gradient.  Scheduled sampling at rate 0.5: the tokens fed equal the fp64 restatement's exactly."""
    lsm = 0.1 if mode == "teacher_lsm" else 0.0
    rate = 0.5 if mode == "sampling" else 0.0
    V, D, Z = 37, 64, 48
    dec = _training_decoder(dlayers, lsm, V=V, D=D, Z=Z)
    hpad, hlen, ys = _batch(D, V)
    L = max(len(y) for y in ys) + 1
    seed = 21 + dlayers
    flags = _flags(seed, rate, L)
    assert any(flags) == (rate > 0)
    res = {}
    for fused in (True, False):
        dec.fused_lstm = fused
        if fused:
            _no_torch_cell(dec)
        dec.zero_grad(set_to_none=True)
        h = hpad.to(DEV).requires_grad_(True)
        random.seed(seed)
        n0 = _lib.launch_count()
        loss, acc = dec(h, hlen, [y.to(DEV) for y in ys], rate)
        loss.backward()
        res[fused] = (loss.detach(), acc, h.grad, {k: p.grad.clone() for k, p in dec.named_parameters()},
                      _lib.launch_count() - n0, random.getstate())
        if fused and rate > 0:
            tok_fused = dec._ss_tokens.cpu().long()
        _torch_cell_back(dec)
    assert res[True][5] == res[False][5], "one draw of random.random() per position on both paths"
    # the upper layers alone launch at least (dlayers - 1) forward steps per position plus their backward
    assert res[True][4] >= res[False][4] + 2 * (dlayers - 1) * L
    sd = {k: v.detach().cpu() for k, v in dec.state_dict().items()}
    sd64 = {k: v.double().requires_grad_(True) for k, v in sd.items()}
    h64 = hpad.double().requires_grad_(True)
    loss64, acc64, tok64 = ref_forward(sd64, h64, hlen, ys, V - 1, V - 1, dlayers, flags, lsm)
    loss64.backward()
    if rate > 0:
        assert torch.equal(tok_fused, tok64), "tokens fed differ from the fp64 restatement's"
    (l1, a1, gh1, g1, _, _), (l0, a0, gh0, g0, _, _) = res[True], res[False]
    helpers.assert_close(l1, l0, truth=loss64.detach(), what="loss")
    assert a1 == pytest.approx(a0) and a1 == pytest.approx(acc64)
    helpers.assert_close(gh1, gh0, truth=h64.grad, what="d hpad")
    for k, p in dec.named_parameters():
        if k == "att.gvec.bias":                  # analytically zero gradient (softmax shift invariance)
            continue
        helpers.assert_close(g1[k], g0[k], truth=sd64[k].grad, what="d " + k)


@pytest.mark.parametrize("rate", [0.0, 0.5])
def test_two_layer_forward_backward_captures_and_replays_on_a_new_batch(rate):
    """dlayers = 2, device lengths: forward + backward captured once (teacher forcing, or scheduled sampling with new
    draws through draw_sampling), then replayed with a batch it was not captured on copied into the static input: loss,
    accuracy, d hpad and every parameter gradient equal an eager run on that batch with the same draws."""
    V, D, Z = 37, 64, 48
    dec = _training_decoder(2, 0.0, V=V, D=D, Z=Z)
    _no_torch_cell(dec)
    hpad, hlen, ys = _batch(D, V)
    hpad2 = torch.tanh(torch.randn(hpad.shape, generator=torch.Generator().manual_seed(9)))
    ys = [y.to(DEV) for y in ys]
    seed2 = 5
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        dec.zero_grad(set_to_none=True)
        h1 = hpad2.to(DEV).requires_grad_(True)
        random.seed(seed2)
        loss1, acc1 = dec(h1, hlen, ys, rate)
        loss1.backward()
        want = (loss1.detach().clone(), acc1, h1.grad.clone(), {k: p.grad.clone() for k, p in dec.named_parameters()})
        dec.zero_grad(set_to_none=True)
        hl_dev = torch.tensor(hlen, device=DEV, dtype=torch.int32)
        h2 = hpad.to(DEV).requires_grad_(True)
        for _ in range(2):                                     # warm-up on the capture stream
            random.seed(1)
            l_, a_ = dec(h2, hl_dev, ys, rate)
            l_.backward()
            dec.zero_grad(set_to_none=True)
            h2.grad = None
    torch.cuda.synchronize()
    del l_, a_
    graph = torch.cuda.CUDAGraph()
    random.seed(1)
    with torch.cuda.graph(graph, stream=st, capture_error_mode="thread_local"):
        loss2, acc2 = dec(h2, hl_dev, ys, rate)
        loss2.backward()
    with torch.no_grad():
        h2.copy_(hpad2.to(DEV))                               # a batch the graph was not captured on
    if rate > 0:
        random.seed(seed2)
        dec.draw_sampling(rate)
    graph.replay()
    torch.cuda.synchronize()
    l1, a1, gh1, g1 = want
    assert float(acc2) == pytest.approx(a1)
    helpers.assert_close(loss2, l1, what="loss (replay)")
    helpers.assert_close(h2.grad, gh1, what="d hpad (replay)")
    for k, p in dec.named_parameters():
        if k != "att.gvec.bias":
            helpers.assert_close(p.grad, g1[k], what="d %s (replay)" % k)


# ---------------------------------------------------------------------------------------------- beam search
def _search_case(dlayers, beam, ctc_weight, Th, nbest, seed, base="beam_eos", **over):
    helpers.BEAM_CASES["_tmp"] = dict(helpers.BEAM_CASES[base], seed=seed, beam=beam, ctc_weight=ctc_weight, nbest=nbest,
                                      Th=Th, **over)
    try:
        c, sd, h, _ = helpers.beam_case("_tmp")
    finally:
        del helpers.BEAM_CASES["_tmp"]
    Z = c["Z"]
    g = torch.Generator().manual_seed(seed + 1000)
    for l in range(1, dlayers):
        sd["decoder.%d.weight_ih" % l] = _randn(g, 4 * Z, Z, fan=Z / 2.0)
        sd["decoder.%d.weight_hh" % l] = _randn(g, 4 * Z, Z, fan=Z)
        sd["decoder.%d.bias_ih" % l] = _randn(g, 4 * Z, fan=4.0)
        sd["decoder.%d.bias_hh" % l] = _randn(g, 4 * Z, fan=4.0)
    att = AttLoc(c["D"], Z, c["A"], c["C"], c["filts"], "softmax")
    dec = Decoder(c["D"], c["V"], dlayers, Z, c["sos"], c["eos"], att)
    ctc = CTC(c["V"], c["D"], 0.0)
    dec.load_state_dict({k: v for k, v in sd.items() if not k.startswith("ctc_lo")}, strict=True)
    ctc.load_state_dict({k: v for k, v in sd.items() if k.startswith("ctc_lo")}, strict=True)
    return c, dec.to(DEV).eval(), ctc.to(DEV).eval(), h


def _recog_args(c, graph=True):
    return types.SimpleNamespace(beam_size=c["beam"], penalty=c["penalty"], ctc_weight=c["ctc_weight"],
                                 maxlenratio=c["maxlenratio"], minlenratio=c["minlenratio"], nbest=c["nbest"],
                                 lm_weight=0.0, cuda_graph=graph)


class _generic_forbidden(object):
    """``with _generic_forbidden(dec):`` -- the generic position raises: what runs inside took the fused position."""

    def __init__(self, dec):
        self.dec = dec

    def __enter__(self):
        def boom(*a, **k):
            raise AssertionError("the generic position was taken")
        self.dec._recognize_generic = boom
        return self

    def __exit__(self, *exc):
        del self.dec._recognize_generic
        return False


def _same_nbest(got, ref, what):
    assert [x["yseq"] for x in got] == [x["yseq"] for x in ref], what
    for a, b in zip(got, ref):
        assert abs(a["score"] - b["score"]) <= 1e-4 * abs(b["score"]), what


@pytest.mark.parametrize("dlayers,ctc_weight,beam,Th", [
    (1, 0.3, 10, 60), (2, 0.3, 10, 60), (2, 0.0, 4, 7), (2, 0.5, 1, 25), (2, 0.3, 12, 3), (2, 0.5, 12, 40),
    (3, 0.3, 12, 33), (3, 0.0, 10, 20), (3, 0.5, 4, 5), (3, 0.3, 1, 9),
    (FUSED_MAX_LAYERS, 0.3, 4, 20), (FUSED_MAX_LAYERS, 0.0, 5, 11)])
def test_multilayer_fused_search_matches_generic_position(dlayers, ctc_weight, beam, Th):
    """recognize_beam of a dlayers-layer decoder takes the fused position (the generic one made to raise, the upper
    cells' torch forward too) and gives the generic position's n-best list -- tokens identical, scores to 1e-4 -- with
    and without CUDA-graph replay (dlayers = 1: the launch count of the one-layer position); beam 12 is the recipe's (Cb = 18), Th = 3 / 5 / 7 are shorter than a graph chunk.
    One position is exactly 4 + dlayers launches, plus one with CTC: one LSTM step per layer."""
    nbest = min(beam, 3)
    c, dec, ctc, h = _search_case(dlayers, beam, ctc_weight, Th, nbest, seed=200 + 10 * dlayers + beam + Th)
    hd = h.to(DEV)
    with torch.no_grad():
        lpz = ctc.log_softmax(hd.unsqueeze(0))[0] if ctc_weight > 0.0 else None
        assert dec._fused_plan(hd, lpz, _recog_args(c)) is not None
        res = {}
        for graph in (True, False):
            res["generic", graph] = dec._recognize_generic(hd, lpz, _recog_args(c, graph))
        _no_torch_cell(dec)
        with _generic_forbidden(dec):
            for graph in (True, False):
                res["fused", graph] = dec.recognize_beam(hd, lpz, _recog_args(c, graph))
            # one position, launched on its own
            plan = dec._fused_plan(hd, lpz, _recog_args(c))
            pin = torch.empty(plan[3], 4, beam, dtype=torch.float32).pin_memory()
            dec.att.reset()
            pos = dec._fused_position(plan[0], plan[1], plan[2], beam, ctc_weight, plan[3], pin, dec._beam_tables())
            n0 = _lib.launch_count()
            pos()
            assert _lib.launch_count() - n0 == 4 + dlayers + (1 if lpz is not None else 0)
            torch.cuda.synchronize()
        _torch_cell_back(dec)
    ref = res["generic", False]
    assert 1 <= len(ref) <= nbest
    for k, got in res.items():
        _same_nbest(got, ref, "%s (dlayers %d)" % (k, dlayers))


@pytest.mark.parametrize("dlayers", [2, 3])
def test_multilayer_recognize_beam_batch_equals_per_utterance(dlayers):
    """recognize_beam_batch of a multi-layer decoder (interleaved fused searches, generic position made to raise) returns
    exactly the per-utterance results of recognize_beam, with CTC and attention-only, for utterances of different
    lengths, some ending through <eos>."""
    c, dec, ctc, _ = _search_case(dlayers, 5, 0.3, 30, 2, seed=300 + dlayers)
    g = torch.Generator().manual_seed(99)
    hs = [torch.tanh(torch.randn(int(t), c["D"], generator=g)).to(DEV) for t in (30, 12, 47, 6, 25, 33)]
    with torch.no_grad():
        lpzs = [ctc.log_softmax(x.unsqueeze(0))[0] for x in hs]
        one = [dec.recognize_beam(x, l, _recog_args(c), None) for x, l in zip(hs, lpzs)]
        att_only = [dec.recognize_beam(x, None, _recog_args(c), None) for x in hs[:3]]
        generic = [dec._recognize_generic(x, l, _recog_args(c)) for x, l in zip(hs, lpzs)]
        with _generic_forbidden(dec):
            for conc in (1, 3):
                got = dec.recognize_beam_batch(hs, lpzs, _recog_args(c), None, concurrency=conc)
                assert got == one, "concurrency %d" % conc
            assert dec.recognize_beam_batch(hs[:3], None, _recog_args(c), None, concurrency=2) == att_only
    for i, (a, b) in enumerate(zip(one, generic)):
        _same_nbest(a, b, "utterance %d" % i)


def test_decoders_deeper_than_the_fused_limit_use_the_generic_position():
    """FUSED_MAX_LAYERS + 1 layers: _fused_plan declines, recognize_beam and recognize_beam_batch give the generic
    position's results; one layer fewer is fused and agrees with it."""
    for dlayers in (FUSED_MAX_LAYERS + 1, FUSED_MAX_LAYERS):
        c, dec, ctc, h = _search_case(dlayers, 4, 0.3, 18, 2, seed=400 + dlayers)
        hd = h.to(DEV)
        with torch.no_grad():
            lpz = ctc.log_softmax(hd.unsqueeze(0))[0]
            fused = dec._fused_plan(hd, lpz, _recog_args(c)) is not None
            assert fused == (dlayers <= FUSED_MAX_LAYERS)
            want = dec._recognize_generic(hd, lpz, _recog_args(c))
            _same_nbest(dec.recognize_beam(hd, lpz, _recog_args(c)), want, "recognize_beam, dlayers %d" % dlayers)
            got = dec.recognize_beam_batch([hd, hd[:9]], [lpz, lpz[:9]], _recog_args(c), None, concurrency=2)
            _same_nbest(got[0], want, "recognize_beam_batch, dlayers %d" % dlayers)
            _same_nbest(got[1], dec._recognize_generic(hd[:9], lpz[:9], _recog_args(c)), "short utterance")


# ---------------------------------------------------------------------------------------------- beam kernels (C ABI)
def _bits(t):
    return t.detach().contiguous().view(torch.int32).cpu()


def test_beam_advance_and_gather_move_every_layer_state():
    """re2e_beam_advance with the 15 segments of a 6-layer search with CTC (z, c of every layer, alignment, r, psi) and
    re2e_beam_gather with 16: every destination holds the rows of the parents (and CTC candidates) the merge chose, bit
    for bit; 17 segments are refused without a launch."""
    W, Cb, beam, Z, Th, V = 10, 15, 10, 24, 37, 4233
    eos = V - 1
    g = torch.Generator().manual_seed(17)
    nl = FUSED_MAX_LAYERS
    layer = torch.randn(2, nl, W, Z, generator=g).to(DEV)              # (z | c, layer, row, unit)
    src = [layer[0, l] for l in range(nl)] + [layer[1, l] for l in range(nl)]
    src += [torch.randn(W, Th, generator=g).to(DEV), torch.randn(W, Cb, Th, 2, generator=g).to(DEV),
            torch.randn(W, Cb, generator=g).to(DEV)]
    rowf = [Z] * (2 * nl) + [Th, 2 * Th, 1]
    subc = [0] * (2 * nl + 1) + [Cb, Cb]
    assert len(src) == 2 * nl + 3 == 15
    dst = [torch.full_like(s[:, 0] if sub else s, -3.0) for s, sub in zip(src, subc)]
    att = torch.log_softmax(torch.randn(W, Cb, generator=g) * 2.0, 1).to(DEV)
    psi = (torch.randn(W, Cb, generator=g) * 3.0 - 20.0).to(DEV)
    prev = (torch.randn(W, generator=g) - 15.0).to(DEV)
    ids = torch.randint(0, V - 1, (W, Cb), generator=g, dtype=torch.int32).to(DEV)
    sc = torch.zeros(W, device=DEV)
    state = torch.tensor([W, 3], dtype=torch.int32, device=DEV)
    ctl = torch.zeros(4, W, dtype=torch.int32, device=DEV)
    hist = torch.zeros(10, 4, beam, device=DEV)
    L, P, sp = _lib.lib(), _lib.ptr, _lib.stream_ptr()
    n = len(src)
    c_src = (ctypes.c_void_p * n)(*[s.data_ptr() for s in src])
    c_dst = (ctypes.c_void_p * n)(*[d.data_ptr() for d in dst])
    c_rowf, c_subc = (ctypes.c_int * n)(*rowf), (ctypes.c_int * n)(*subc)
    _lib.check(L.re2e_beam_advance(P(att), P(ids), P(psi), P(prev), P(sc), 0.7, 0.3, W, Cb, beam, P(state), P(ctl),
                                   P(hist), eos, 200, n, c_src, c_dst, c_rowf, c_subc, sp), "re2e_beam_advance")
    torch.cuda.synchronize()
    assert int(state[0]) > 0
    par, cand = ctl[0].long(), ctl[1].long()
    assert len(set(par.tolist())) > 1, "the merge should pick several parents"
    for s_, (s, d, sub) in enumerate(zip(src, dst, subc)):
        want = s[par, cand] if sub else s[par]
        assert torch.equal(_bits(d), _bits(want)), "segment %d" % s_

    # re2e_beam_gather: 16 segments (one more z), then 17 refused
    src16 = src + [torch.randn(W, Z, generator=g).to(DEV)]
    rowf16, subc16 = rowf + [Z], subc + [0]
    dst16 = [torch.full_like(s[:, 0] if sub else s, -3.0) for s, sub in zip(src16, subc16)]
    parent = torch.randint(0, W, (W,), generator=g, dtype=torch.int32).to(DEV)
    cnd = torch.randint(0, Cb, (W,), generator=g, dtype=torch.int32).to(DEV)

    def gather(k, s_list, d_list, rf, sb):
        return L.re2e_beam_gather(P(parent), P(cnd), W, k, (ctypes.c_void_p * k)(*[t.data_ptr() for t in s_list]),
                                  (ctypes.c_void_p * k)(*[t.data_ptr() for t in d_list]), (ctypes.c_int * k)(*rf),
                                  (ctypes.c_int * k)(*sb), sp)
    _lib.check(gather(16, src16, dst16, rowf16, subc16), "re2e_beam_gather")
    torch.cuda.synchronize()
    pl, cl = parent.long(), cnd.long()
    for s_, (s, d, sub) in enumerate(zip(src16, dst16, subc16)):
        assert torch.equal(_bits(d), _bits(s[pl, cl] if sub else s[pl])), "gather segment %d" % s_
    n0 = _lib.launch_count()
    assert gather(17, src16 + src16[:1], dst16 + dst16[:1], rowf16 + [Z], subc16 + [0]) == -1
    assert L.re2e_beam_advance(P(att), P(ids), P(psi), P(prev), P(sc), 0.7, 0.3, W, Cb, beam, P(state), P(ctl), P(hist),
                               eos, 200, 17, (ctypes.c_void_p * 17)(*([src[0].data_ptr()] * 17)),
                               (ctypes.c_void_p * 17)(*([dst[0].data_ptr()] * 17)), (ctypes.c_int * 17)(*([Z] * 17)),
                               (ctypes.c_int * 17)(*([0] * 17)), sp) == -1
    assert _lib.launch_count() == n0


@pytest.mark.parametrize("layers", [1, 2, 3, FUSED_MAX_LAYERS])
def test_beam_init_zeroes_the_states_of_every_layer(layers):
    """re2e_beam_init with Z = layers * dunits on states laid out (layers, W, dunits): z and c of every layer zero, the
    alignment uniform, the float after the last layer untouched (NaN prefill)."""
    W, Z, Th = 10, 300, 41
    junk = float("nan")
    z = torch.full((layers * W * Z + 4,), junk, device=DEV)
    c = torch.full((layers * W * Z + 4,), junk, device=DEV)
    a = torch.full((W, Th), junk, device=DEV)
    ctl = torch.full((4, W), -5, dtype=torch.int32, device=DEV)
    sc = torch.full((W,), junk, device=DEV)
    state = torch.full((2,), -5, dtype=torch.int32, device=DEV)
    P = _lib.ptr
    _lib.check(_lib.lib().re2e_beam_init(P(z), P(c), P(a), None, None, None, P(ctl), P(sc), P(state), W, layers * Z, Th,
                                         0, 0, 7, _lib.stream_ptr()), "re2e_beam_init")
    torch.cuda.synchronize()
    zero = torch.zeros(layers * W * Z, dtype=torch.int32)
    assert torch.equal(_bits(z[:-4]), zero) and torch.equal(_bits(c[:-4]), zero)
    assert bool(torch.isnan(z[-4:]).all()) and bool(torch.isnan(c[-4:]).all())
    u = np.float32(1.0) / np.float32(Th)
    assert torch.equal(_bits(a), _bits(torch.full((W, Th), float(u))))
    assert ctl.cpu().tolist() == [[0] * W, [0] * W, [7] * W, [0] * W] and state.cpu().tolist() == [1, 0]


# ---------------------------------------------------------------------------------------------- drop-in
needs_reference = pytest.mark.skipif(not refshim.available(), reason="reference tree / oracle/_ref not present")


@pytest.fixture
def strict_fp32_library_math():
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


@needs_reference
def test_reference_e2e_with_two_decoder_layers_and_the_swapped_decoder(strict_fp32_library_math):
    """The reference's own E2E with dlayers = 2, built from its unmodified files with AttLoc, CTC, CTCPrefixScore and
    Decoder bound to ours: loss and every parameter gradient match the unmodified reference on the CPU (fp64 as
    tie-breaker), and recognize (fused beam search) gives its tokens."""
    import robust_e2e_gan_b200 as ours
    args = refshim.e2e_args(dlayers=2, odim=24)
    ref_mod = refshim.load().e2e_model
    torch.manual_seed(5)
    ref = ref_mod.E2E(copy.deepcopy(args))
    with torch.no_grad():
        ref.dec.output.bias[args.odim - 1] += 1.5                 # let hypotheses end
    sd = copy.deepcopy(ref.state_dict())
    g = torch.Generator().manual_seed(11)
    B, T = 3, 40
    x = torch.randn(B, T, args.fbank_dim, generator=g)
    ilens = torch.tensor([T - 3 * i for i in range(B)])
    for b in range(B):
        x[b, int(ilens[b]):] = 0
    tsz = torch.tensor([3, 4, 5])
    targets = torch.randint(1, args.odim - 1, (int(tsz.sum()),), generator=g)

    def run(model, dev, dt=torch.float32):
        model.zero_grad()
        loss_ctc, loss_att, acc = model(x.to(dev, dt), targets.to(dev), ilens, tsz)
        a = model.mtlalpha
        (a * loss_ctc.sum() + (1 - a) * loss_att).backward()
        return float(loss_ctc.sum()), float(loss_att), acc, \
            {k: p.grad.detach().double().cpu() for k, p in model.named_parameters() if p.grad is not None}

    r32 = run(ref, "cpu")
    ref64 = ref_mod.E2E(copy.deepcopy(args)).double()
    ref64.load_state_dict({k: v.double() for k, v in sd.items()})
    r64 = run(ref64, "cpu", torch.float64)
    ra = types.SimpleNamespace(beam_size=4, penalty=0.0, ctc_weight=0.3, maxlenratio=0.0, minlenratio=0.0, nbest=2,
                               lm_weight=0.0)
    xr = torch.randn(1, 60, args.fbank_dim, generator=g)
    with torch.no_grad():
        want = ref.eval().recognize(xr, ra, args.char_list)
    with refshim.swapped(AttLoc=ours.AttLoc, CTC=ours.CTC, CTCPrefixScore=ours.CTCPrefixScore, Decoder=ours.Decoder) as m:
        mine = m.E2E(copy.deepcopy(args))
        assert isinstance(mine.dec, ours.Decoder) and mine.dec.dlayers == 2
        mine.load_state_dict(sd, strict=True)
        mine = mine.to(DEV).train()
        _no_torch_cell(mine.dec)
        got = run(mine, DEV)
        mine.eval()
        with _generic_forbidden(mine.dec), torch.no_grad():
            hyps = mine.recognize(xr, ra, args.char_list)
    helpers.assert_close(np.float64(got[0]), np.float64(r32[0]), truth=np.float64(r64[0]), what="loss_ctc")
    helpers.assert_close(np.float64(got[1]), np.float64(r32[1]), truth=np.float64(r64[1]), what="loss_att")
    assert got[2] == pytest.approx(r32[2])
    assert set(got[3]) == set(r32[3])
    for k in sorted(r32[3]):
        if not k.endswith("att.gvec.bias"):
            helpers.assert_close(got[3][k], r32[3][k], truth=r64[3][k], what="d " + k)
    assert len(hyps) == len(want)
    for a, b in zip(hyps, want):
        assert [int(t) for t in a["yseq"]] == [int(t) for t in b["yseq"]]
        assert abs(float(a["score"]) - float(b["score"])) <= 1e-4 * max(1.0, abs(float(b["score"])))
