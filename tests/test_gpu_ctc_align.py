"""GPU: forced CTC alignment (ctc_forced_align / CTC.forced_align, csrc/ctc.cu ctc_viterbi_warp_kernel) against the
fp64 Viterbi oracle (oracle.ctc_align.ctc_viterbi), the CTC loss, and itself under CUDA-graph replay."""
import numpy as np
import pytest
import torch

from conftest import golden
from helpers import assert_close
from oracle import ctc as o_ctc
from oracle import ctc_align as o_align
from robust_e2e_gan_b200 import CTC, _lib, ctc_forced_align, ctc_loss, prepare_targets, synth
from robust_e2e_gan_b200.linear import _pad4, linear

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")


def T(a):
    return torch.from_numpy(np.asarray(a))


def lp64(x):
    """fp64 log-softmax of (..., V) logits on the host."""
    return torch.log_softmax(x.detach().double().cpu(), dim=-1).numpy()


def pitched_logits(B, Th, V, seed, scale=2.0):
    """(B,Th,V) logits in the row-padded layout of the tcgen05 ctc_lo GEMM (row pitch _pad4(V) floats)."""
    g = torch.Generator().manual_seed(seed)
    buf = (torch.randn(B, Th, _pad4(V), generator=g) * scale).to(DEV)
    return buf[..., :V]


def check_path(al, b, Th, hlen, y, blank=0):
    """Structure of utterance b's device alignment: a valid lattice path over the first min(hlen, Th) frames, -1 after,
    tokens and spans consistent with the states."""
    st = al.states[b].cpu().numpy().astype(np.int64)
    tk = al.tokens[b].cpu().numpy()
    sp = al.spans[b].cpu().numpy()
    Tb = min(max(hlen, 0), Th)
    U = len(y)
    S = 2 * U + 1
    assert (st[Tb:] == -1).all() and (tk[Tb:] == -1).all()
    s = st[:Tb]
    assert s[0] in (0, 1) and s[-1] in (S - 1, S - 2)
    d = np.diff(s)
    assert ((d >= 0) & (d <= 2)).all()
    for t in np.nonzero(d == 2)[0]:
        tgt = s[t + 1]
        assert tgt & 1 and tgt >= 3 and y[tgt >> 1] != y[(tgt >> 1) - 1], "illegal skip at frame %d" % t
    ext = np.full(S, blank, np.int64)
    ext[1::2] = y
    assert (tk[:Tb] == ext[s]).all()
    collapsed = [v for i, v in enumerate(tk[:Tb]) if v != blank and (i == 0 or v != tk[i - 1])]
    assert collapsed == list(y)
    for u in range(U):
        fr = np.nonzero(s == 2 * u + 1)[0]
        assert sp[u, 0] == fr[0] and sp[u, 1] == fr[-1]
    assert (sp[U:] == -1).all()
    return s


def compare_to_oracle(al, lp, hl, ys, Th, margin_eq=1e-3, rel=1e-4):
    """Every utterance: valid path, fp64 score of the device path within rel of the oracle optimum, device score close
    to the oracle's, states identical where the oracle's decisions are clearer than margin_eq.  Returns the number of
    utterances compared state by state."""
    same = 0
    for b, y in enumerate(ys):
        y = [int(v) for v in y]
        Tb = max(0, min(hl[b], Th))
        ref = o_align.ctc_viterbi(lp[b, :Tb], y)
        if Tb <= 0 or ref["score"] == -np.inf:      # no frames or no path: everything -1
            assert float(al.score[b]) == ref["score"]
            assert (al.states[b] == -1).all() and (al.tokens[b] == -1).all() and (al.spans[b] == -1).all()
            continue
        s = check_path(al, b, Th, hl[b], y)
        ext = np.zeros(2 * len(y) + 1, np.int64)
        ext[1::2] = y
        dev_score = float(lp[b, np.arange(Tb), ext[s]].sum())
        tol = rel * max(1.0, abs(ref["score"]))
        assert dev_score <= ref["score"] + 1e-9 and dev_score >= ref["score"] - tol, (b, dev_score, ref["score"])
        assert abs(float(al.score[b]) - ref["score"]) <= tol, (b, float(al.score[b]), ref["score"])
        if ref["margin"] > margin_eq:
            assert np.array_equal(s, ref["states"]), "utterance %d: margin %.3g" % (b, ref["margin"])
            same += 1
    return same


def test_golden_module():
    g = golden("ctc")
    B, Th, D = g["hs"].shape
    V = g["W"].shape[0]
    ctc = CTC(V, D, 0.0).to(DEV)
    ctc.ctc_lo.weight.data.copy_(T(g["W"]))
    ctc.ctc_lo.bias.data.copy_(T(g["b"]))
    hl = [int(h) for h in g["hlens"]]
    al = ctc.forced_align(T(g["hs"]).to(DEV), hl, T(g["ys_pad"]).to(DEV))
    lp = o_ctc.log_softmax(T(g["W"]).double(), T(g["b"]).double(), T(g["hs"]).double()).numpy()
    ref_scores = []
    for b in range(B):
        y = [int(v) for v in g["ys_pad"][b] if v != -1]
        ref = o_align.ctc_viterbi(lp[b, :hl[b]], y)
        st = al.states[b].cpu().numpy()
        assert np.array_equal(st[:hl[b]], ref["states"]) and (st[hl[b]:] == -1).all()
        check_path(al, b, Th, hl[b], y)
        ref_scores.append(ref["score"])
    assert_close(al.score, np.array(ref_scores), tol=1e-4, what="path score")
    assert not al.score.requires_grad


def test_bench_shape():
    """B = 32, Th = 200, U = 40, V = 4233 with the padded-pitch logits of the ctc_lo GEMM and variable hlens."""
    B, Th, U, V, D = 32, 200, 40, 4233, 320
    hs, hl = synth.encoder_batch(B=B, Th=Th, D=D, seed=11)
    ys = synth.targets(B=B, V=V, hlens=hl, seed=11, fixed_U=U)
    g = torch.Generator().manual_seed(11)
    W = (torch.randn(V, D, generator=g) * 0.25).to(DEV)
    bias = (torch.randn(V, generator=g) * 0.1).to(DEV)
    with torch.no_grad():
        x = linear(hs.to(DEV), W, bias)
    assert x.stride(1) == _pad4(V) > V        # the pitched layout is taken as is
    al = ctc_forced_align(x, hl, ys)
    same = compare_to_oracle(al, lp64(x), hl, ys, Th)
    assert same >= B // 2, same


@pytest.mark.parametrize("Th,Umax,B", [(60, 10, 4), (90, 20, 4), (120, 40, 3), (160, 60, 3), (200, 90, 3),
                                       (260, 120, 2), (400, 150, 3), (800, 255, 2)])
def test_lattice_widths(Th, Umax, B):
    """Every states-per-lane instantiation (1, 2, 3, 4, 6, 8, 12, 16), up to the U = 255 boundary at Th = 800."""
    V = 300
    hl = [Th] + [int(v) for v in np.random.default_rng(Th).integers(2 * Umax + 2, Th + 1, B - 1)]
    ys = synth.targets(B=B, V=V, hlens=hl, seed=Th, umin=Umax // 2, umax=Umax)
    ys[0] = synth.targets(B=1, V=V, hlens=[Th], seed=Th + 1, fixed_U=Umax)[0]
    assert max(len(y) for y in ys) == Umax
    x = pitched_logits(B, Th, V, seed=Th)
    al = ctc_forced_align(x, hl, ys)
    assert al.spans.shape == (B, Umax, 2)
    compare_to_oracle(al, lp64(x), hl, ys, Th)


def test_unsupported_shapes_launch_nothing():
    V = 50
    x = pitched_logits(2, 40, V, seed=1)
    ys = [torch.randint(1, V, (256,)), torch.randint(1, V, (3,))]
    n0 = _lib.launch_count()
    with pytest.raises(RuntimeError, match="not supported"):
        ctc_forced_align(x, [40, 40], ys)
    x = pitched_logits(1, 2000, V, seed=2)
    with pytest.raises(RuntimeError, match="not supported"):
        ctc_forced_align(x, [2000], [torch.tensor([1, 2, 3])])
    torch.cuda.synchronize()
    assert _lib.launch_count() == n0


def test_edge_cases():
    """U = 0, infeasible utterances, hlens beyond Th (clamped), hlens 0, padding frames."""
    Th, V = 30, 20
    x = pitched_logits(6, Th, V, seed=5)
    ys = [torch.tensor([], dtype=torch.long), torch.tensor([3, 3, 3, 3]), torch.tensor([1, 2, 3]),
          torch.tensor([4, 5]), torch.tensor([], dtype=torch.long), torch.tensor([7])]
    hl = [25, 6, 50, 0, 0, 12]      # 1: needs 7 frames; 2: clamped to Th; 3: no frames; 4: no frames and U = 0
    al = ctc_forced_align(x, hl, ys)
    torch.cuda.synchronize()
    st, tk, sp, sc = al.states.cpu(), al.tokens.cpu(), al.spans.cpu(), al.score.cpu()
    lp = lp64(x)
    # U = 0: all blank over the valid frames
    assert (st[0, :25] == 0).all() and (tk[0, :25] == 0).all() and (st[0, 25:] == -1).all()
    assert (sp[0] == -1).all()
    assert float(sc[0]) == pytest.approx(lp[0, :25, 0].sum(), rel=1e-5)
    # infeasible
    assert float(sc[1]) == -np.inf and (st[1] == -1).all() and (tk[1] == -1).all() and (sp[1] == -1).all()
    # hlens > Th: the whole utterance
    check_path(al, 2, Th, 50, [1, 2, 3])
    assert (st[2] >= 0).all()
    # no frames
    assert float(sc[3]) == -np.inf and (st[3] == -1).all() and (sp[3] == -1).all()
    assert float(sc[4]) == 0.0 and (st[4] == -1).all()
    compare_to_oracle(al, lp, [25, 6, 50, 0, 0, 12], ys, Th)
    # the device hlens form gives the same result
    al2 = ctc_forced_align(x, torch.tensor(hl, dtype=torch.int32, device=DEV), ys)
    for a, b in zip(al, al2):
        assert torch.equal(a, b)


def test_consistent_with_the_loss():
    B, Th, V = 8, 120, 500
    hl = [120, 117, 110, 100, 96, 90, 80, 64]
    ys = synth.targets(B=B, V=V, hlens=hl, seed=21, umin=10, umax=40)
    x = pitched_logits(B, Th, V, seed=21)
    al = ctc_forced_align(x, hl, ys)
    _, nll = ctc_loss(x, hl, ys)
    tol = 1e-5 * nll.abs() + 1e-4
    assert (al.score <= -nll + tol).all()
    # exactly one path (T = U, no repeats): Viterbi score == log-likelihood
    hl1 = [12, 12, 7]
    ys1 = [torch.arange(1, 13), torch.arange(20, 32), torch.tensor([5, 4, 3, 2, 1, 2, 3])]
    x1 = pitched_logits(3, 12, 40, seed=22)
    al1 = ctc_forced_align(x1, hl1, ys1)
    _, nll1 = ctc_loss(x1, hl1, ys1)
    assert_close(al1.score, -nll1, tol=1e-5, what="single-path score")
    assert torch.equal(al1.states[0].cpu(), torch.arange(1, 24, 2, dtype=torch.int32))
    # log-probabilities in, the same path out
    D = 64
    ctc = CTC(V, D, 0.0).to(DEV)
    with torch.no_grad():
        ctc.ctc_lo.weight.mul_(20.0)
    hs, hl2 = synth.encoder_batch(B=B, Th=Th, D=D, seed=23)
    ys2 = synth.targets(B=B, V=V, hlens=hl2, seed=23, umin=10, umax=40)
    a_logit = ctc.forced_align(hs.to(DEV), hl2, ys2)
    lsm = ctc.log_softmax(hs.to(DEV))
    a_lp = ctc_forced_align(lsm, hl2, ys2)
    lp = lp64(lsm)
    for b in range(B):
        # a frame shifted by its log-sum-exp rounds differently in fp32: only near-ties may go either way
        if o_align.ctc_viterbi(lp[b, :hl2[b]], ys2[b].tolist())["margin"] > 1e-4:
            assert torch.equal(a_logit.states[b], a_lp.states[b]), b
    assert_close(a_lp.score, a_logit.score, tol=1e-5, what="score from log-probs")


def test_exact_ties_follow_the_rule():
    """One logit per frame is 0 and the rest are -1024 or -2048: the frame's log-sum-exp is exactly 0 in fp32, every
    lattice sum is an exact integer, ties are everywhere, and the path must be the oracle's under the tie rule."""
    B, Th, V = 16, 40, 4
    rng = np.random.default_rng(31)
    x = -1024.0 * rng.integers(1, 3, size=(B, Th, V))
    x[np.arange(B)[:, None], np.arange(Th)[None, :], rng.integers(0, V, size=(B, Th))] = 0.0
    hl = [int(v) for v in rng.integers(20, Th + 1, B)]
    ys = [torch.from_numpy(rng.integers(1, V, size=int(rng.integers(0, 9)))) for _ in range(B)]
    xd = T(x.astype(np.float32)).to(DEV)
    al = ctc_forced_align(xd, hl, ys)
    for b in range(B):
        ref = o_align.ctc_viterbi(x[b, :hl[b]], ys[b].tolist())
        st = al.states[b].cpu().numpy()
        assert np.array_equal(st[:hl[b]], ref["states"]), b
        assert float(al.score[b]) == ref["score"]


def test_two_launches_and_graph_replay():
    B, Th, V = 8, 100, 300
    hl = [100, 99, 90, 85, 70, 66, 60, 51]
    ys = synth.targets(B=B, V=V, hlens=hl, seed=41, umin=5, umax=30)
    tgt = prepare_targets(ys, DEV)
    hl_d = torch.tensor(hl, dtype=torch.int32, device=DEV)
    x = pitched_logits(B, Th, V, seed=41)
    n0 = _lib.launch_count()
    ctc_forced_align(x, hl_d, tgt)
    assert _lib.launch_count() - n0 == 2
    st = torch.cuda.Stream(DEV)
    st.wait_stream(torch.cuda.current_stream(DEV))
    with torch.cuda.stream(st):
        ctc_forced_align(x, hl_d, tgt)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=st):
        out = ctc_forced_align(x, hl_d, tgt)
    for seed in (42, 43):
        x.copy_(pitched_logits(B, Th, V, seed=seed))
        graph.replay()
        torch.cuda.synchronize()
        ref = ctc_forced_align(x, hl_d, tgt)
        for a, b in zip(out, ref):
            assert torch.equal(a, b)
