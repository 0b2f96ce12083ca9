"""GPU: the decoder around AttLoc -- batched hybrid CTC/attention beam search (BASELINE config 5) and the training
loop -- against (a) tests/golden/beam.npz, produced by the UNMODIFIED reference Decoder.recognize_beam, and (b) the
CPU oracle (oracle/beam.py).  Token sequences must be IDENTICAL; scores within 1e-4 relative."""
import os
import types

import numpy as np
import pytest
import torch

import helpers
from oracle import beam as obeam
from robust_e2e_gan_b200 import CTC, AttLoc, Decoder

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GOLD = np.load(os.path.join(os.path.dirname(__file__), "golden", "beam.npz"))


def build(c, sd):
    att = AttLoc(c["D"], c["Z"], c["A"], c["C"], c["filts"], "softmax")
    dec = Decoder(c["D"], c["V"], 1, c["Z"], c["sos"], c["eos"], att)
    ctc = CTC(c["V"], c["D"], 0.0)
    dec.load_state_dict({k: v for k, v in sd.items() if not k.startswith("ctc_lo")}, strict=True)
    ctc.load_state_dict({k: v for k, v in sd.items() if k.startswith("ctc_lo")}, strict=True)
    return dec.to(DEV).eval(), ctc.to(DEV).eval()


def recog_args(c):
    return types.SimpleNamespace(beam_size=c["beam"], penalty=c["penalty"], ctc_weight=c["ctc_weight"],
                                 maxlenratio=c["maxlenratio"], minlenratio=c["minlenratio"], nbest=c["nbest"],
                                 lm_weight=0.0)


def run_gpu(c, sd, h):
    dec, ctc = build(c, sd)
    hd = h.to(DEV)
    lpz = ctc.log_softmax(hd.unsqueeze(0))[0] if c["ctc_weight"] > 0.0 else None
    return dec.recognize_beam(hd, lpz, recog_args(c), [str(i) for i in range(c["V"])]), ctc, hd


@pytest.mark.parametrize("name", list(helpers.BEAM_CASES))
def test_beam_search_matches_reference_golden(name):
    c, sd, h, checksum = helpers.beam_case(name)
    assert abs(checksum - float(GOLD[name + ".checksum"])) <= 1e-9 * checksum, "fixture weights not reproduced"
    nbest, ctc, hd = run_gpu(c, sd, h)
    n = int(GOLD[name + ".n"])
    assert len(nbest) == n
    for i in range(n):
        assert nbest[i]["yseq"] == [int(t) for t in GOLD["%s.yseq%d" % (name, i)]], "hypothesis %d differs" % i
        ref = float(GOLD["%s.score%d" % (name, i)])
        assert abs(nbest[i]["score"] - ref) <= 1e-4 * abs(ref)
    # CTC best path ("CTC alignment" of the north star) identical
    assert ctc.best_path(hd.unsqueeze(0))[0].cpu().tolist() == [int(t) for t in GOLD[name + ".best_path"]]


def _never_eos(Th):
    # <eos> far below every other token: not even among the CTC candidates, so every search ends through the append at
    # the last position.  maxlen = Th puts that end at every offset within the 8-position graph chunk (5: no graph).
    return pytest.param("beam_eos", dict(seed=50 + Th, beam=5, ctc_weight=0.5, nbest=3, Th=Th, eos_bias=-30.0),
                        id="never_eos-maxlen%d" % Th)


ORACLE_CASES = [
    # greedy (beam 1), hybrid and CTC-only scoring on fresh seeds
    pytest.param("beam_eos", dict(seed=7, beam=1, ctc_weight=0.0, nbest=1, Th=22), id="7-1-0.0"),
    pytest.param("beam_eos", dict(seed=8, beam=6, ctc_weight=0.3, nbest=3, Th=22), id="8-6-0.3"),
    pytest.param("beam_eos", dict(seed=9, beam=4, ctc_weight=1.0, nbest=3, Th=22), id="9-4-1.0"),
] + [_never_eos(Th) for Th in (5, 6, 7, 8, 9, 16, 17, 23)] + [
    # <eos> is the best candidate at position 0: hypotheses end in the first (single-position) flight and end_detect
    # fires inside the first chunk
    pytest.param("beam_eos", dict(seed=60, beam=5, ctc_weight=0.0, nbest=3, Th=22, eos_bias=40.0), id="eos_first-att"),
    pytest.param("beam_eos", dict(seed=61, beam=5, ctc_weight=0.3, nbest=3, Th=22, eos_bias=100.0), id="eos_first-ctc"),
    # the fused position's limits (Cb = int(1.5 beam) <= 32, W <= 32) and the dispatch to the generic position beyond
    pytest.param("beam_default_dims", dict(seed=70, beam=21, nbest=3), id="beam21-Cb31"),
    pytest.param("beam_default_dims", dict(seed=71, beam=22, nbest=3), id="beam22-Cb33-generic"),
    pytest.param("beam_default_dims", dict(seed=72, beam=32, ctc_weight=0.0, nbest=3), id="beam32-att_only"),
    pytest.param("beam_default_dims", dict(seed=73, ctc_weight=1.0, nbest=3), id="ctc_only-generic"),
    # length penalty, minimum and maximum length on a long search (no end_detect with maxlenratio > 0)
    pytest.param("beam_eos", dict(seed=80, beam=5, ctc_weight=0.5, nbest=3, Th=80, eos_bias=0.5, penalty=0.5,
                                  minlenratio=0.3, maxlenratio=0.5), id="nbest3-minlen-maxlen-penalty"),
]


@pytest.mark.parametrize("base,over", ORACLE_CASES)
def test_beam_search_matches_oracle(base, over):
    """GPU tokens == oracle tokens, scores to 1e-4, for search settings beyond the golden cases."""
    helpers.BEAM_CASES["_tmp"] = dict(helpers.BEAM_CASES[base], **over)
    try:
        c, sd, h, _ = helpers.beam_case("_tmp")
    finally:
        del helpers.BEAM_CASES["_tmp"]
    with torch.no_grad():
        ref = obeam.recognize_beam(sd, h, c)
    nbest, _, _ = run_gpu(c, sd, h)
    assert [x["yseq"] for x in nbest] == [x["yseq"] for x in ref]
    for a, b in zip(nbest, ref):
        assert abs(a["score"] - b["score"]) <= 1e-4 * abs(b["score"])
    # the cases do what their names say
    if c["eos_bias"] <= -30.0:
        assert all(len(x["yseq"]) == c["Th"] + 2 and c["eos"] not in x["yseq"][1:-1] for x in ref)
    if c["eos_bias"] >= 40.0:
        assert ref[0]["yseq"] == [c["sos"], c["eos"]]


def training_case(name):
    """(decoder on the GPU in train mode, its CPU state dict, hpad, hlen, ys, sos, eos) of a training-loop input:
    ``beam_small`` dims, or ``bench`` = the workload of bench.py's decoder_forward_bench (must stay equal to it:
    B = 32, Th = 200, U = 40, V = 4233, default AttLoc / decoder dimensions, the same seeds)."""
    if name == "bench":
        from robust_e2e_gan_b200 import synth
        from robust_e2e_gan_b200.hotpath import DEFAULT_CFG
        B, Th, D, A, Z, C, V, U = (DEFAULT_CFG[k] for k in ("B", "Th", "D", "A", "Z", "C", "V", "U"))
        torch.manual_seed(7)
        att = AttLoc(D, Z, A, C, DEFAULT_CFG["filts"], "softmax")
        dec = Decoder(D, V, 1, Z, V - 1, V - 1, att)
        sd = {k: v.detach().clone() for k, v in dec.state_dict().items()}
        hpad, hlen = synth.encoder_batch(B=B, Th=Th, D=D, seed=77)
        ys = synth.targets(B=B, V=V, hlens=hlen, seed=77, fixed_U=U)
        return dec.to(DEV).train(), sd, hpad, hlen, ys, V - 1, V - 1
    c, sd, _, _ = helpers.beam_case(name)
    B, Th = 3, 19
    g = torch.Generator().manual_seed(5)
    hpad = torch.tanh(torch.randn(B, Th, c["D"], generator=g))
    hlen = [19, 15, 11]
    ys = [torch.randint(1, c["V"] - 1, (n,), generator=g) for n in (6, 4, 5)]
    dec, _ = build(c, sd)
    return dec.train(), sd, hpad, hlen, ys, c["sos"], c["eos"]


TRAINING_INPUTS = ("beam_small", "bench")


def test_decoder_training_loop_matches_oracle():
    """Decoder.forward (teacher forcing): loss, accuracy and gradients w.r.t. the encoder output, the attention
    parameters and the decoder's own layers, against the fp32 oracle with the fp64 oracle as tie-breaker, for every
    input of TRAINING_INPUTS."""
    for case in TRAINING_INPUTS:
        _check_training_loop(case)


def _check_training_loop(case):
    dec, sd, hpad, hlen, ys, sos, eos = training_case(case)
    # oracle (CPU autograd), fp32 and fp64
    ref = {}
    for dt in (torch.float32, torch.float64):
        sd_o = {k: v.detach().clone().to(dt).requires_grad_(True) for k, v in sd.items()}
        h_o = hpad.detach().clone().to(dt).requires_grad_(True)
        loss_o, acc_o = obeam.decoder_forward(sd_o, h_o, hlen, ys, sos, eos)
        loss_o.backward()
        ref[dt] = (loss_o.detach(), acc_o, h_o.grad, {k: v.grad for k, v in sd_o.items()})
    (loss_o, acc_o, gh_o, g_o), (loss_t, _, gh_t, g_t) = ref[torch.float32], ref[torch.float64]
    # product
    h_d = hpad.to(DEV).requires_grad_(True)
    loss, acc = dec(h_d, hlen, [y.to(DEV) for y in ys], 0.0)
    loss.backward()
    helpers.assert_close(loss, loss_o, truth=loss_t, what="%s: loss" % case)
    assert acc == pytest.approx(acc_o), case
    helpers.assert_close(h_d.grad, gh_o, truth=gh_t, what="%s: d hpad" % case)
    for k, p in dec.named_parameters():
        if k == "att.gvec.bias":          # analytically zero gradient (softmax shift invariance)
            continue
        helpers.assert_close(p.grad, g_o[k], truth=g_t[k], what="%s: d %s" % (case, k))


def test_decoder_forward_with_device_lengths_is_capturable_and_identical():
    """Lengths given as a CUDA tensor keep Decoder.forward free of host round trips (CUDA-graph capturable); results
    equal the list-of-ints call, and a captured forward + backward replays to the same loss and gradients, for every
    input of TRAINING_INPUTS."""
    for case in TRAINING_INPUTS:
        _check_capturable(case)


def _check_capturable(case):
    dec, _, hpad, hlen, ys, _, _ = training_case(case)
    hpad = hpad.to(DEV)
    ys = [y.to(DEV) for y in ys]
    # everything -- the eager reference run included -- on ONE side stream: a parameter's gradient accumulator stays tied
    # to the stream of its first backward, and a capture may not synchronise with the legacy default stream
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        h1 = hpad.clone().requires_grad_(True)
        loss1, acc1 = dec(h1, hlen, ys, 0.0)
        loss1.backward()
        g1 = {k: p.grad.clone() for k, p in dec.named_parameters()}
        loss1, h1g = loss1.detach().clone(), h1.grad.clone()
        del h1
        dec.zero_grad(set_to_none=True)
        hl_dev = torch.tensor(hlen, device=DEV, dtype=torch.int32)
        h2 = hpad.clone().requires_grad_(True)
    import gc
    gc.collect()
    with torch.cuda.stream(st):
        for _ in range(2):                      # warm-up on the capture stream
            l, a = dec(h2, hl_dev, ys, 0.0)
            l.backward()
            dec.zero_grad(set_to_none=True)
            h2.grad = None
    torch.cuda.synchronize()
    del l, a
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=st, capture_error_mode="thread_local"):
        loss2, acc2 = dec(h2, hl_dev, ys, 0.0)
        loss2.backward()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.is_tensor(acc2) and float(acc2) == pytest.approx(acc1), case
    helpers.assert_close(loss2, loss1, what="%s: loss (graph replay)" % case)
    helpers.assert_close(h2.grad, h1g, what="%s: d hpad (graph replay)" % case)
    for k, p in dec.named_parameters():
        if k == "att.gvec.bias":
            continue
        helpers.assert_close(p.grad, g1[k], what="%s: d %s (graph replay)" % (case, k))


@pytest.mark.parametrize("B,Z,D,L", [(32, 300, 320, 5), (3, 48, 64, 4), (10, 300, 320, 3), (40, 52, 36, 3), (33, 640, 640, 2), (5, 12, 4, 2), (4, 48, 1284, 2)])
def test_lstm_loop_matches_torch_lstmcell(B, Z, D, L):
    """lstm.LSTMLoop (embedding-half gates of all positions in one GEMM + one cluster kernel per position -- or, for
    dimensions that kernel does not take (D or Z > 640), batch-sized products + pointwise kernels; weight gradients in
    two GEMMs after the loop) against torch.nn.LSTMCell on cat(embedding, context), fp64
    as tie-breaker: states of every position and all gradients."""
    from robust_e2e_gan_b200.lstm import LSTMLoop
    g = torch.Generator().manual_seed(B + Z)
    cell = torch.nn.LSTMCell(Z + D, Z)
    with torch.no_grad():
        for p in cell.parameters():
            p.copy_(torch.randn(p.shape, generator=g) / (Z + D) ** 0.5)
    eys = torch.randn(B, L, Z, generator=g)
    ctxs = torch.randn(L, B, D, generator=g)
    gz = torch.randn(L, B, Z, generator=g)

    def run_ref(dt, dev):
        c2 = torch.nn.LSTMCell(Z + D, Z).to(dev, dt)
        c2.load_state_dict({k: v.to(dt) for k, v in cell.state_dict().items()})
        e = eys.detach().clone().to(dev, dt).requires_grad_(True)
        cx = ctxs.detach().clone().to(dev, dt).requires_grad_(True)
        h, c = torch.zeros(B, Z, dtype=dt, device=dev), torch.zeros(B, Z, dtype=dt, device=dev)
        hs = []
        for i in range(L):
            h, c = c2(torch.cat((e[:, i, :], cx[i]), 1), (h, c))
            hs.append(h)
        hs = torch.stack(hs)
        ((hs * gz.to(dev, dt)).sum() + c.sum()).backward()
        return [hs.detach(), e.grad, cx.grad] + [p.grad for p in c2.parameters()]

    r32, r64 = run_ref(torch.float32, "cpu"), run_ref(torch.float64, "cpu")
    cd = torch.nn.LSTMCell(Z + D, Z).to(DEV)
    cd.load_state_dict(cell.state_dict())
    e = eys.detach().clone().to(DEV).requires_grad_(True)
    cx = ctxs.detach().clone().to(DEV).requires_grad_(True)
    n0 = _lib_count()
    loop = LSTMLoop(cd, e)
    h, c = torch.zeros(B, Z, device=DEV), torch.zeros(B, Z, device=DEV)
    hs = []
    for i in range(L):
        h, c = loop.step(i, cx[i], h, c)
        hs.append(h)
    hs = torch.stack(hs)
    ((hs * gz.to(DEV)).sum() + c.sum()).backward()
    assert _lib_count() - n0 >= 3 * L
    got = [hs.detach(), e.grad, cx.grad] + [p.grad for p in cd.parameters()]
    names = ["h of every position", "d embeddings", "d contexts", "d weight_ih", "d weight_hh", "d bias_ih", "d bias_hh"]
    for a, b32, b64, what in zip(got, r32, r64, names):
        helpers.assert_close(a, b32, truth=b64, what=what)


def _lib_count():
    from robust_e2e_gan_b200 import _lib
    return _lib.launch_count()


@pytest.mark.parametrize("M,N,K,acc", [(32, 1200, 320, False), (32, 1200, 300, True), (32, 320, 1200, False),
                                       (40, 50, 44, True), (1, 8, 4, False), (7, 1201, 644, False), (33, 75, 50, False), (5, 9, 323, True)])
def test_batch_nt_product(M, N, K, acc):
    """re2e_batch_nt (the decoder's per-position products, one CTA per 8 output columns) against fp64: rows beyond one
    32-row pass, column counts that are no multiple of 8, reduction lengths that are no multiple of the staged chunk
    or of 4 (scalar staging), and the accumulate form."""
    from robust_e2e_gan_b200 import _lib
    g = torch.Generator().manual_seed(M * N + K)
    X, W, O = torch.randn(M, K, generator=g), torch.randn(N, K, generator=g), torch.randn(M, N, generator=g)
    want64 = X.double() @ W.double().t() + (O.double() if acc else 0.0)
    want32 = X @ W.t() + (O if acc else 0.0)
    Xd, Wd, Od = X.to(DEV), W.to(DEV), O.to(DEV)
    L = _lib.lib()
    _lib.check(L.re2e_batch_nt(_lib.ptr(Xd), _lib.ptr(Wd), None, _lib.ptr(Od), M, N, K, int(acc), _lib.stream_ptr()), "batch_nt")
    helpers.assert_close(Od, want32, truth=want64, what="X @ W^T")


@pytest.mark.parametrize("rows,V,k", [(10, 4233, 15), (1, 52, 1), (3, 8192, 32), (7, 1025, 10)])
def test_log_softmax_topk(rows, V, k):
    """re2e_log_softmax_topk against torch.topk(log_softmax) (model/e2e_decoder.py:262,276): ids identical, values and the
    full log-softmax row to fp32 accuracy; duplicated maxima resolve to the lower index."""
    from robust_e2e_gan_b200 import _lib
    g = torch.Generator().manual_seed(rows * V + k)
    x = torch.randn(rows, V, generator=g) * 3.0
    if V > 60:
        x[0, 50] = x[0, 7] = x[0].max() + 1.0          # a tie at the top
    if rows > 1 and V > 1100:
        x[1, :24] += 40.0                              # the k best all in ONE warp's slice (the selection's slow path)
        x[1, 1024:1030] += 30.0
    xd = x.to(DEV)
    full = torch.empty(rows, V, device=DEV)
    vals, ids = torch.empty(rows, k, device=DEV), torch.empty(rows, k, dtype=torch.int32, device=DEV)
    _lib.check(_lib.lib().re2e_log_softmax_topk(_lib.ptr(xd), rows, V, k, _lib.ptr(full), _lib.ptr(vals), _lib.ptr(ids),
                                                _lib.stream_ptr()), "log_softmax_topk")
    want = torch.log_softmax(x.double(), 1)
    helpers.assert_close(full, want.float(), truth=want, what="log-softmax rows")
    wv, wi = torch.sort(want, dim=1, descending=True, stable=True)
    assert ids.cpu().tolist() == wi[:, :k].tolist()
    helpers.assert_close(vals, wv[:, :k].float(), truth=wv[:, :k], what="top-k values")


def test_beam_gather_and_joint():
    """re2e_beam_gather (parent / (parent, candidate) row gathers of several state tensors in one launch) and
    re2e_beam_joint against the reference's tensor expressions (model/e2e_decoder.py:284-292), bit for bit."""
    import ctypes
    from robust_e2e_gan_b200 import _lib
    L = _lib.lib()
    g = torch.Generator().manual_seed(3)
    W, Cb, beam, Th, Z = 6, 9, 6, 37, 20
    a, r = torch.randn(W, Z, generator=g).to(DEV), torch.randn(W, Cb, Th, 2, generator=g).to(DEV)
    psi = torch.randn(W, Cb, generator=g).to(DEV)
    parent = torch.randint(0, W, (W,), generator=g).int().to(DEV)
    cand = torch.randint(0, Cb, (W,), generator=g).int().to(DEV)
    a2, r2, p2 = torch.empty(W, Z, device=DEV), torch.empty(W, Th, 2, device=DEV), torch.empty(W, device=DEV)
    src = (ctypes.c_void_p * 3)(a.data_ptr(), r.data_ptr(), psi.data_ptr())
    dst = (ctypes.c_void_p * 3)(a2.data_ptr(), r2.data_ptr(), p2.data_ptr())
    rowf, subc = (ctypes.c_int * 3)(Z, 2 * Th, 1), (ctypes.c_int * 3)(0, Cb, Cb)
    _lib.check(L.re2e_beam_gather(_lib.ptr(parent), _lib.ptr(cand), W, 3, src, dst, rowf, subc, _lib.stream_ptr()), "gather")
    pl, cl = parent.long(), cand.long()
    assert torch.equal(a2, a[pl]) and torch.equal(r2, r[pl, cl]) and torch.equal(p2, psi[pl, cl])

    att = torch.randn(W, Cb, generator=g).to(DEV)
    ids = torch.randint(0, 4000, (W, Cb), generator=g).int().to(DEV)
    prev, sc = torch.randn(W, generator=g).to(DEV), torch.randn(W, generator=g).to(DEV)
    out = torch.empty(3, W, beam, device=DEV)
    w = 0.3
    _lib.check(L.re2e_beam_joint(_lib.ptr(att), _lib.ptr(ids), _lib.ptr(psi), _lib.ptr(prev), _lib.ptr(sc), 1.0 - w, w,
                                 W, Cb, beam, _lib.ptr(out), _lib.stream_ptr()), "joint")
    local = (1.0 - w) * att + w * (psi - prev.unsqueeze(1))
    bs, bj = torch.topk(local, beam, dim=1)
    assert torch.equal(out[0], sc.unsqueeze(1) + bs)
    assert torch.equal(out[1], ids.long().gather(1, bj).float()) and torch.equal(out[2], bj.float())
    _lib.check(L.re2e_beam_joint(_lib.ptr(att), _lib.ptr(ids), None, None, _lib.ptr(sc), 1.0, 0.0, W, Cb, beam,
                                 _lib.ptr(out), _lib.stream_ptr()), "joint (attention only)")
    bs, bj = torch.topk(att, beam, dim=1)
    assert torch.equal(out[0], sc.unsqueeze(1) + bs) and torch.equal(out[2], bj.float())


@pytest.mark.parametrize("ctc_weight,beam,Th", [(0.3, 10, 60), (0.0, 5, 40), (0.5, 1, 25), (0.3, 4, 2), (0.3, 6, 7),
                                                 (0.7, 3, 11)])
def test_fused_beam_position_matches_generic_path(ctc_weight, beam, Th):
    """The fused position (csrc/beam.cu; tail as one launch or as joint / merge / gather) and the generic tensor-op
    position of recognize_beam give the same n-best list (tokens identical, scores to 1e-4), with and without CUDA-graph
    replay (fused: 8 positions per replay, history read back in chunks)."""
    helpers.BEAM_CASES["_tmp"] = dict(helpers.BEAM_CASES["beam_eos"], seed=31, beam=beam, ctc_weight=ctc_weight,
                                      nbest=min(beam, 3), Th=Th)
    try:
        c, sd, h, _ = helpers.beam_case("_tmp")
    finally:
        del helpers.BEAM_CASES["_tmp"]
    dec, ctc = build(c, sd)
    hd = h.to(DEV)
    lpz = ctc.log_softmax(hd.unsqueeze(0))[0] if ctc_weight > 0.0 else None
    res = {}
    # (fused first: a generic search with its graph must also work on a decoder that has run fused searches)
    for fused, graph, tail in ((True, True, True), (True, False, True), (True, True, False), (True, False, False),
                               (False, True, True), (False, False, True)):
        ra = recog_args(c)
        ra.fused_position, ra.cuda_graph, ra.fused_tail = fused, graph, tail
        n0 = _lib_count()
        with torch.no_grad():
            res[fused, graph, tail] = dec.recognize_beam(hd, lpz, ra, None)
        if fused and not graph:
            assert _lib_count() - n0 >= 5 * (len(res[fused, graph, tail][0]["yseq"]) - 2)
    ref = res[False, False, True]
    for k, got in res.items():
        assert [x["yseq"] for x in got] == [x["yseq"] for x in ref], "tokens differ for (fused, graph, fused tail) = %s" % (k,)
        for a, b in zip(got, ref):
            assert abs(a["score"] - b["score"]) <= 1e-4 * abs(b["score"])


def test_recognize_beam_batch_equals_per_utterance():
    """recognize_beam_batch (interleaved searches on their own streams and graphs) returns, for every utterance, exactly
    what recognize_beam returns for it alone: lengths differ, some searches end early through <eos> / end_detect
    (eos_bias 2.5) or all run to maxlen (-30).  The last utterance (Th = 300) follows shorter ones on the same slot and
    needs a longer history buffer than the first 256 positions."""
    for eos_bias in (2.5, -30.0):
        helpers.BEAM_CASES["_tmp"] = dict(helpers.BEAM_CASES["beam_eos"], seed=41, beam=5, ctc_weight=0.3, nbest=2, Th=30,
                                          eos_bias=eos_bias)
        try:
            c, sd, h, _ = helpers.beam_case("_tmp")
        finally:
            del helpers.BEAM_CASES["_tmp"]
        dec, ctc = build(c, sd)
        g = torch.Generator().manual_seed(99)
        hs = [torch.tanh(torch.randn(int(t), c["D"], generator=g)).to(DEV) for t in (30, 12, 47, 8, 25, 33, 6, 300)]
        with torch.no_grad():
            lpzs = [ctc.log_softmax(x.unsqueeze(0))[0] for x in hs]
            one = [dec.recognize_beam(x, l, recog_args(c), None) for x, l in zip(hs, lpzs)]
            for conc in (1, 3):
                dec.__dict__.pop("_hist_pins", None)        # every slot's history buffer starts at its first utterance
                got = dec.recognize_beam_batch(hs, lpzs, recog_args(c), None, concurrency=conc)
                assert got == one, "eos_bias %g, concurrency %d" % (eos_bias, conc)
            att_only = [dec.recognize_beam(x, None, recog_args(c), None) for x in hs[:3]]
            assert dec.recognize_beam_batch(hs[:3], None, recog_args(c), None, concurrency=2) == att_only
        if eos_bias < 0:
            assert len(one[-1][0]["yseq"]) == 302, "the long search should run to maxlen"


def test_fused_search_sees_weights_written_through_data():
    """Parameters overwritten through ``.data`` (which does not bump their version counter): the next fused search
    decodes with the new weights, exactly as the oracle with the new state dict and the generic position (run after a
    fused search on the same decoder, with its CUDA graph) do."""
    helpers.BEAM_CASES["_tmp"] = dict(helpers.BEAM_CASES["beam_eos"], seed=45, Th=30)
    try:
        c, sd, h, _ = helpers.beam_case("_tmp")
        helpers.BEAM_CASES["_tmp"]["seed"] = 46
        _, sd2, _, _ = helpers.beam_case("_tmp")
    finally:
        del helpers.BEAM_CASES["_tmp"]
    dec, ctc = build(c, sd)
    hd = h.to(DEV)
    with torch.no_grad():
        lpz = ctc.log_softmax(hd.unsqueeze(0))[0]
        before = dec.recognize_beam(hd, lpz, recog_args(c), None)
        for name, p in (("decoder.0.weight_hh", dec.decoder[0].weight_hh), ("embed.weight", dec.embed.weight)):
            v = p._version
            p.data.copy_(sd2[name].to(DEV))
            assert p._version == v
        fused = dec.recognize_beam(hd, lpz, recog_args(c), None)
        ref = obeam.recognize_beam(dict(sd, **{k: sd2[k] for k in ("decoder.0.weight_hh", "embed.weight")}), h, c)
    assert [x["yseq"] for x in ref] != [x["yseq"] for x in before], "the new weights should change the result"

    def same(got, name):
        assert [x["yseq"] for x in got] == [x["yseq"] for x in ref], name
        for a, b in zip(got, ref):
            assert abs(a["score"] - b["score"]) <= 1e-4 * abs(b["score"]), name

    same(fused, "fused")
    ra = recog_args(c)
    ra.fused_position = False
    with torch.no_grad():
        generic = dec.recognize_beam(hd, lpz, ra, None)
    same(generic, "generic")


def test_label_batches_and_length_mask_match_the_list_formulation():
    """_label_batches (one concatenation + two gathers) == the reference's per-utterance cat / pad_list construction
    (model/e2e_decoder.py:88-97); mask_by_length as one select == the per-utterance slice copies, values and gradient."""
    from robust_e2e_gan_b200.e2e_common import pad_list
    from robust_e2e_gan_b200.e2e_decoder import _label_batches, mask_by_length
    g = torch.Generator().manual_seed(5)
    ys = [torch.randint(0, 50, (int(n),), generator=g).to(DEV) for n in (7, 1, 12, 4, 12)]
    sos, eos, ign = 51, 52, -1
    keep = []
    pin, pout = _label_batches(ys, sos, eos, ign, keep)
    s_, e_ = torch.full((1,), sos, device=DEV), torch.full((1,), eos, device=DEV)
    assert torch.equal(pin, pad_list([torch.cat([s_, y]) for y in ys], eos))
    assert torch.equal(pout, pad_list([torch.cat([y, e_]) for y in ys], ign))
    x = torch.randn(4, 9, 6, generator=g).to(DEV).requires_grad_(True)
    lens = [9, 3, 1, 6]
    got = mask_by_length(x, lens, 0)
    want = x.detach().clone()
    for i, l in enumerate(lens):
        want[i, l:] = 0
    assert torch.equal(got, want)
    w = torch.randn(4, 9, 6, generator=g).to(DEV)
    (got * w).sum().backward()
    gw = w.clone()
    for i, l in enumerate(lens):
        gw[i, l:] = 0
    assert torch.equal(x.grad, gw)


@pytest.mark.parametrize("rows,V,pitched", [(1312, 4233, True), (7, 52, False), (33, 1000, True)])
def test_cross_entropy_kernels_match_torch(rows, V, pitched):
    """_CrossEntropy (re2e_cross_entropy_fwd / _bwd) == F.cross_entropy(ignore_index, mean) in value and gradient (fp64 as
    tie-breaker), arg-max == torch's, on contiguous and row-pitched logits; ignored rows get a zero gradient row."""
    from robust_e2e_gan_b200.e2e_decoder import _CrossEntropy
    g = torch.Generator().manual_seed(rows + V)
    x = torch.randn(rows, V, generator=g) * 2.0
    t = torch.randint(0, V, (rows,), generator=g)
    t[::5] = -1
    ld = (V + 3) // 4 * 4 if pitched else V
    buf = torch.zeros(rows, ld, device=DEV)
    buf[:, :V] = x.to(DEV)
    xd = buf[:, :V].detach().requires_grad_(True)
    loss, best = _CrossEntropy.apply(xd, t.to(DEV), -1)
    (loss * 3.0).backward()
    refs = []
    for dt in (torch.float32, torch.float64):
        xr = x.detach().clone().to(dt).requires_grad_(True)
        lr = torch.nn.functional.cross_entropy(xr, t, ignore_index=-1, reduction='mean')
        (lr * 3.0).backward()
        refs.append((lr.detach(), xr.grad))
    helpers.assert_close(loss.detach(), refs[0][0], truth=refs[1][0], what="cross-entropy")
    helpers.assert_close(xd.grad, refs[0][1], truth=refs[1][1], what="d logits")
    assert torch.equal(best.cpu().long(), x.argmax(1))
    assert float(xd.grad[::5].abs().max()) == 0.0


@pytest.mark.parametrize("dlayers,lsm", [(2, 0.0), (1, 0.1)])
def test_decoder_forward_variants_agree_with_the_library_free_path(dlayers, lsm):
    """Two decoder layers (only the first LSTMCell runs on the cluster kernel) and label smoothing (the extra
    F.log_softmax term of model/e2e_decoder.py:160-164): the fused path (LSTM step kernel, batched output layer,
    cross-entropy kernels) against the same module with torch.nn.LSTMCell + per-position output layer + F.cross_entropy
    (scheduled_sampling_rate just above 0 selects that loop; the draw never fires), loss and all gradients."""
    from robust_e2e_gan_b200 import AttLoc, Decoder
    torch.manual_seed(11)
    V, D, Z, A, C, filts, B, Th = 37, 64, 48, 64, 4, 5, 4, 17
    ld = np.full(V, 1.0 / V, dtype=np.float32) if lsm > 0 else None
    dec = Decoder(D, V, dlayers, Z, V - 1, V - 1, AttLoc(D, Z, A, C, filts, "softmax"), labeldist=ld, lsm_weight=lsm).to(DEV)
    dec.train()
    g = torch.Generator().manual_seed(3)
    hpad = torch.tanh(torch.randn(B, Th, D, generator=g)).to(DEV)
    hlen = [17, 12, 9, 17]
    ys = [torch.randint(0, V - 1, (n,), generator=g).to(DEV) for n in (5, 3, 4, 6)]
    res = []
    for rate in (0.0, 1e-12):
        dec.zero_grad(set_to_none=True)
        h = hpad.clone().requires_grad_(True)
        loss, acc = dec(h, hlen, ys, rate)
        loss.backward()
        res.append((loss.detach(), acc, h.grad, {k: p.grad.clone() for k, p in dec.named_parameters() if p.grad is not None}))
    (l0, a0, h0, g0), (l1, a1, h1, g1) = res
    helpers.assert_close(l0, l1, what="loss")
    assert a0 == pytest.approx(a1)
    helpers.assert_close(h0, h1, what="d hpad")
    assert set(g0) == set(g1)
    for k in g0:
        if k == "att.gvec.bias":
            continue
        helpers.assert_close(g0[k], g1[k], what="d " + k)
