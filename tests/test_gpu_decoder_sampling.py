"""GPU: scheduled-sampling training on the library's kernels (model/e2e_decoder.py:121-152 with
scheduled_sampling_rate > 0): re2e_sample_tokens through the C ABI against an exact fp64 arg-max, and Decoder.forward
against a CPU restatement of the reference loop (``sampled_forward``, on the oracle's AttLoc step and LSTMCell),
against the library-free loop, as a replayed CUDA graph with new draws before every replay, and its launch profile at
the bench shape."""
import random

import numpy as np
import pytest
import torch

import helpers
from oracle import attloc as oatt
from oracle import beam as obeam
from robust_e2e_gan_b200 import AttLoc, Decoder, _lib
from robust_e2e_gan_b200.e2e_decoder import _label_batches
from test_gpu_decoder import training_case

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _sample(X, W, bias, flag, tok, ws, M=None, N=None, K=None, ptrs=None):
    M = X.shape[0] if M is None else M
    N = W.shape[0] if N is None else N
    K = X.shape[1] if K is None else K
    p = ptrs if ptrs is not None else [_lib.ptr(t) for t in (X, W, bias, flag, tok, ws)]
    return _lib.lib().re2e_sample_tokens(*p, M, N, K, _lib.stream_ptr())


def _ws(M):
    n = _lib.lib().re2e_sample_tokens_ws_bytes(M)
    assert n == 8 * (M + 1)
    return torch.zeros(n // 8, dtype=torch.int64, device=DEV)


def _ints(g, *shape):
    """Integers in [-4, 4]: every product and sum of these shapes is exact in fp32, so the kernel's arg-max must equal the
    fp64 one bit for bit, ties included."""
    return torch.randint(-4, 5, shape, generator=g).float()


def _want(X, W, bias):
    """fp64 arg-max (the first of equal maxima: lowest index) and whether some row's maximum is tied."""
    v = X.double().numpy() @ W.double().numpy().T + (bias.double().numpy() if bias is not None else 0.0)
    return np.argmax(v, axis=1), bool(((v == v.max(1, keepdims=True)).sum(1) > 1).any())


@pytest.mark.parametrize("bias", [True, False])
@pytest.mark.parametrize("K", [48, 300, 301])
@pytest.mark.parametrize("N", [37, 4233, 8192])
def test_sample_tokens_is_the_exact_argmax(N, K, bias):
    """re2e_sample_tokens == fp64 arg-max, lowest index on ties, for M in {1, 10, 32, 33, 70} (one and several 32-row
    passes), 128-bit (K % 4 == 0) and scalar staging (K = 301), one- and 16-column CTAs.  W is drawn once freely and once
    from 12 distinct rows (with their biases), so every arg-max is an exact tie between duplicated rows.  Every call leaves ws zero."""
    g = torch.Generator().manual_seed(N * 7 + K * 3 + int(bias))
    for M in (1, 10, 32, 33, 70):
        for pool in (False, True):
            X = _ints(g, M, K)
            pick = (torch.arange(N) % 12)[torch.randperm(N, generator=g)]          # every pooled row 3+ times
            W = _ints(g, 12, K)[pick] if pool else _ints(g, N, K)
            b = torch.randint(-1, 2, (12 if pool else N,), generator=g).float() if bias else None
            b = b[pick] if (pool and bias) else b
            want, tied = _want(X, W, b)
            assert tied or not pool, "the pooled rows should tie"
            flag = torch.ones(1, dtype=torch.int32, device=DEV)
            tok = torch.full((M,), -7, dtype=torch.int32, device=DEV)
            ws = _ws(M)
            Xd, Wd, bd = X.to(DEV), W.to(DEV), (b.to(DEV) if b is not None else None)
            _lib.check(_sample(Xd, Wd, bd, flag, tok, ws), "re2e_sample_tokens")
            torch.cuda.synchronize()
            assert tok.cpu().numpy().tolist() == want.tolist(), (M, pool)
            assert int(ws.abs().sum()) == 0, "ws must be left zero"


def test_sample_tokens_signed_zero_ties_and_the_flag():
    """A tie between -0 and +0 is a tie (lowest index wins, whichever sign it has); flag = 0 leaves tok untouched and ws
    zero; two calls in a row agree."""
    M, N, K = 33, 300, 64
    g = torch.Generator().manual_seed(1)
    X = torch.randint(1, 4, (M, K), generator=g).float()
    W = -torch.randint(1, 4, (N, K), generator=g).float()
    W[[3, 5, 200]] = 0.0                              # the only rows with a logit >= 0
    Xd, Wd, ws = X.to(DEV), W.to(DEV), _ws(M)
    flag = torch.ones(1, dtype=torch.int32, device=DEV)
    for signs, want in (((-0.0, 0.0, -0.0), 3), ((0.0, -0.0, 0.0), 3)):
        b = torch.full((N,), -0.5)
        b[3], b[5], b[200] = signs
        tok = torch.full((M,), -1, dtype=torch.int32, device=DEV)
        for _ in range(2):
            _lib.check(_sample(Xd, Wd, b.to(DEV), flag, tok, ws), "re2e_sample_tokens")
            torch.cuda.synchronize()
            assert tok.cpu().tolist() == [want] * M, signs
    tok = torch.arange(M, dtype=torch.int32, device=DEV)
    flag.zero_()
    _lib.check(_sample(Xd, Wd, None, flag, tok, ws), "re2e_sample_tokens")
    torch.cuda.synchronize()
    assert tok.cpu().tolist() == list(range(M)) and int(ws.abs().sum()) == 0


def test_sample_tokens_replays_from_a_graph_and_rejects_bad_arguments():
    """A captured call replayed twice gives the eager result both times (ws is left zero, no memset node needed), and
    reads the flag at replay time.  Bad arguments return RE2E_E_ARG without a launch."""
    M, N, K = 40, 4233, 300
    g = torch.Generator().manual_seed(2)
    X, W, b = torch.randn(M, K, generator=g), torch.randn(N, K, generator=g), torch.randn(N, generator=g)
    Xd, Wd, bd, ws = X.to(DEV), W.to(DEV), b.to(DEV), _ws(M)
    flag = torch.ones(1, dtype=torch.int32, device=DEV)
    eager = torch.full((M,), -1, dtype=torch.int32, device=DEV)
    _lib.check(_sample(Xd, Wd, bd, flag, eager, ws), "re2e_sample_tokens")
    tok = torch.full((M,), -1, dtype=torch.int32, device=DEV)
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=st):
        _lib.check(_sample(Xd, Wd, bd, flag, tok, ws), "re2e_sample_tokens")
    for _ in range(2):
        tok.fill_(-1)
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(tok, eager) and int(ws.abs().sum()) == 0
    flag.zero_()
    tok.fill_(-1)
    graph.replay()
    torch.cuda.synchronize()
    assert tok.cpu().tolist() == [-1] * M

    ok = [_lib.ptr(t) for t in (Xd, Wd, bd, flag, tok, ws)]
    n0 = _lib.launch_count()
    for k in (0, 1, 3, 4, 5):                               # X, W, flag, tok, ws NULL
        p = list(ok)
        p[k] = None
        assert _sample(Xd, Wd, bd, flag, tok, ws, ptrs=p) == -1, k
    for dims in ((0, N, K), (M, 0, K), (M, N, 0), (-1, N, K)):
        assert _sample(Xd, Wd, bd, flag, tok, ws, *dims) == -1, dims
    assert _lib.launch_count() == n0
    assert _lib.lib().re2e_sample_tokens_ws_bytes(0) == 0


# ---------------------------------------------------------------------------------------------------- Decoder.forward
def _flags(seed, rate, L):
    random.seed(seed)
    return [random.random() < rate and i > 0 for i in range(L)]


def _state_after(seed, L):
    random.seed(seed)
    for _ in range(L):
        random.random()
    return random.getstate()


def sampled_forward(sd, hpad, hlen, ys, sos, eos, sample, ignore_id=-1):
    """model/e2e_decoder.py:79-167 with scheduled sampling, dlayers = 1, no label smoothing, on CPU autograd (the
    teacher-forced restatement is oracle.beam.decoder_forward; this one adds the sampled positions).  ``sample``: one flag
    per output position (the reference's ``random.random() < rate and i > 0``); a flagged position feeds
    embed(argmax_v y_{i-1}) of these logits (first of equal maxima; the token is not differentiable, the embedding row
    it selects is).  Returns (loss, acc, tokens (L, B) int64 fed at every position, {(i, b): top-1 minus top-2 logit of
    y_{i-1}[b]} at every flagged position)."""
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
    z, c = hpad.new_zeros(B, Z), hpad.new_zeros(B, Z)
    pre = oatt.precompute(att_p, hpad)
    att_w = None
    y_all, tokens, gaps = [], [], {}
    for i in range(L):
        att_c, att_w = oatt.step(att_p, hpad, pre, hlen, z, att_w)
        tok = pad_in[:, i]
        if sample[i]:
            prev = y_all[-1].detach()
            tok = prev.argmax(1)
            top2 = prev.topk(2, dim=1)[0]
            for b in range(B):
                gaps[i, b] = float(top2[b, 0] - top2[b, 1])
        tokens.append(tok)
        z, c = obeam.lstm_cell(sd, "decoder.0.", torch.cat((sd["embed.weight"][tok], att_c), dim=1), (z, c))
        y_all.append(torch.nn.functional.linear(z, sd["output.weight"], sd["output.bias"]))
    y_all = torch.stack(y_all, dim=0).transpose(0, 1).contiguous().view(B * L, -1)
    loss = torch.nn.functional.cross_entropy(y_all, pad_out.view(-1), ignore_index=ignore_id, reduction='mean')
    loss = loss * (np.mean([len(x) for x in ys_in]) - 1)
    pred = y_all.detach().view(B, L, -1).argmax(2)
    m = pad_out != ignore_id
    acc = float((pred[m] == pad_out[m]).sum()) / float(m.sum())
    return loss, acc, torch.stack(tokens), gaps


def test_sampled_forward_without_flags_is_the_teacher_forced_oracle():
    """CPU: with no position flagged, sampled_forward gives oracle.beam.decoder_forward's loss, accuracy and gradients
    exactly (it differs from it only at flagged positions)."""
    c, sd, _, _ = helpers.beam_case("beam_small")
    g = torch.Generator().manual_seed(5)
    hpad = torch.tanh(torch.randn(3, 19, c["D"], generator=g))
    hlen, ys = [19, 15, 11], [torch.randint(1, c["V"] - 1, (n,), generator=g) for n in (6, 4, 5)]
    res = []
    for fn in (lambda *a: obeam.decoder_forward(*a), lambda *a: sampled_forward(*a, [False] * 7)[:2]):
        sd_o = {k: v.detach().clone().double().requires_grad_(True) for k, v in sd.items()}
        loss, acc = fn(sd_o, hpad.double(), hlen, ys, c["sos"], c["eos"])
        loss.backward()
        res.append((float(loss.detach()), acc, {k: v.grad for k, v in sd_o.items()}))
    assert res[0][:2] == res[1][:2]
    for k, g0 in res[0][2].items():                   # (ctc_lo.* get no gradient from either)
        g1 = res[1][2][k]
        assert (g0 is None and g1 is None) or torch.equal(g0, g1), k


# (input, rate, seed of `random`): seeds chosen so that the fp64 top-2 logit gap at every sampled (position, row) is
# at least 1e-5 (asserted below), i.e. fp32 rounding cannot pick another token
ORACLE_CASES = [("beam_small", 0.5, 4), ("beam_small", 1.0, 0), ("bench", 0.5, 6), ("bench", 1.0, 0)]


@pytest.mark.parametrize("case,rate,seed", ORACLE_CASES)
def test_scheduled_sampling_matches_oracle(case, rate, seed):
    """Decoder.forward with scheduled sampling: loss, accuracy, d hpad and every parameter gradient against the fp32
    sampled_forward (fp64 as tie-breaker), the tokens fed on the device == the restatement's exactly, and Python's
    random state afterwards == the library-free loop's (one draw per position)."""
    dec, sd, hpad, hlen, ys, sos, eos = training_case(case)
    L = max(len(y) for y in ys) + 1
    flags = _flags(seed, rate, L)
    assert any(flags)
    ref = {}
    for dt in (torch.float32, torch.float64):
        sd_o = {k: v.detach().clone().to(dt).requires_grad_(True) for k, v in sd.items()}
        h_o = hpad.detach().clone().to(dt).requires_grad_(True)
        loss_o, acc_o, tok_o, gaps = sampled_forward(sd_o, h_o, hlen, ys, sos, eos, flags)
        loss_o.backward()
        ref[dt] = (loss_o.detach(), acc_o, h_o.grad, {k: v.grad for k, v in sd_o.items()}, tok_o, gaps)
    (loss_o, acc_o, gh_o, g_o, tok32, _), (loss_t, _, gh_t, g_t, tok64, gaps) = ref[torch.float32], ref[torch.float64]
    assert len(gaps) == sum(flags) * len(ys) and min(gaps.values()) >= 1e-5, min(gaps.values())
    assert torch.equal(tok32, tok64)

    h_d = hpad.to(DEV).requires_grad_(True)
    random.seed(seed)
    n0 = _lib.launch_count()
    loss, acc = dec(h_d, hlen, [y.to(DEV) for y in ys], rate)
    loss.backward()
    assert random.getstate() == _state_after(seed, L)
    assert _lib.launch_count() > n0
    assert torch.equal(dec._ss_tokens.cpu().long(), tok64), "tokens fed differ from the restatement's"
    helpers.assert_close(loss, loss_o, truth=loss_t, what="%s: loss" % case)
    assert acc == pytest.approx(acc_o), case
    helpers.assert_close(h_d.grad, gh_o, truth=gh_t, what="%s: d hpad" % case)
    for k, p in dec.named_parameters():
        if k == "att.gvec.bias":          # analytically zero gradient (softmax shift invariance)
            continue
        helpers.assert_close(p.grad, g_o[k], truth=g_t[k], what="%s: d %s" % (case, k))


@pytest.mark.parametrize("dlayers,lsm,Z,D", [(2, 0.0, 48, 64), (1, 0.1, 48, 64), (1, 0.0, 644, 64), (2, 0.1, 644, 64)])
def test_scheduled_sampling_matches_the_library_free_loop(dlayers, lsm, Z, D):
    """Two decoder layers (layer 1 stays torch.nn.LSTMCell), label smoothing, and Z = 644 (outside the LSTM cluster
    kernel: batch-sized products + the pointwise kernel on gathered table rows) against fused_lstm = False (LSTMCell,
    per-position output layer and topk, F.cross_entropy) with the same seed: loss, accuracy, all gradients, and the
    random state left behind."""
    torch.manual_seed(11)
    V, A, C, filts, B, Th = 37, 64, 4, 5, 4, 17
    ld = np.full(V, 1.0 / V, dtype=np.float32) if lsm > 0 else None
    dec = Decoder(D, V, dlayers, Z, V - 1, V - 1, AttLoc(D, Z, A, C, filts, "softmax"), labeldist=ld,
                  lsm_weight=lsm).to(DEV).train()
    g = torch.Generator().manual_seed(3)
    hpad = torch.tanh(torch.randn(B, Th, D, generator=g)).to(DEV)
    hlen = [17, 12, 9, 17]
    ys = [torch.randint(0, V - 1, (n,), generator=g).to(DEV) for n in (5, 3, 4, 6)]
    res = []
    for fused in (True, False):
        dec.fused_lstm = fused
        dec.zero_grad(set_to_none=True)
        h = hpad.clone().requires_grad_(True)
        random.seed(21)
        loss, acc = dec(h, hlen, ys, 0.5)
        loss.backward()
        res.append((loss.detach(), acc, h.grad, {k: p.grad.clone() for k, p in dec.named_parameters()},
                    random.getstate()))
    (l0, a0, h0, g0, r0), (l1, a1, h1, g1, r1) = res
    assert any(_flags(21, 0.5, 7)) and r0 == r1
    helpers.assert_close(l0, l1, what="loss")
    assert a0 == pytest.approx(a1)
    helpers.assert_close(h0, h1, what="d hpad")
    for k in g1:
        if k != "att.gvec.bias":
            helpers.assert_close(g0[k], g1[k], what="d " + k)


def test_scheduled_sampling_graph_replays_new_draws():
    """Forward + backward at rate 0.5 captured once; before each replay random.seed(s); dec.draw_sampling(r) with a new
    (s, r), r = 0 included: every replay equals the eager call with that seed and rate (tokens exactly)."""
    dec, _, hpad, hlen, ys, _, _ = training_case("beam_small")
    hpad = hpad.to(DEV)
    ys = [y.to(DEV) for y in ys]
    L = max(len(y) for y in ys) + 1
    draws = [(4, 0.5), (0, 1.0), (5, 0.0), (6, 0.3)]
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    want = []
    with torch.cuda.stream(st):
        for s, r in draws:
            dec.zero_grad(set_to_none=True)
            h = hpad.clone().requires_grad_(True)
            random.seed(s)
            loss, acc = dec(h, hlen, ys, r)
            loss.backward()
            tok = dec._ss_tokens.clone() if r > 0 else None
            want.append((loss.detach().clone(), acc, h.grad.clone(), {k: p.grad.clone() for k, p in dec.named_parameters()},
                         tok))
        dec.zero_grad(set_to_none=True)
        hl_dev = torch.tensor(hlen, device=DEV, dtype=torch.int32)
        h2 = hpad.clone().requires_grad_(True)
        for _ in range(2):
            l_, _a = dec(h2, hl_dev, ys, 0.5)
            l_.backward()
            dec.zero_grad(set_to_none=True)
            h2.grad = None
    torch.cuda.synchronize()
    del l_, _a
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=st, capture_error_mode="thread_local"):
        loss2, acc2 = dec(h2, hl_dev, ys, 0.5)
        loss2.backward()
    tok2 = dec._ss_tokens
    teacher = _label_batches(ys, dec.sos, dec.eos, dec.ignore_id, [])[0].t().to(torch.int32)
    for (s, r), (l1, a1, g_h, g1, t1) in zip(draws, want):
        random.seed(s)
        dec.draw_sampling(r)
        assert random.getstate() == _state_after(s, L)
        graph.replay()
        torch.cuda.synchronize()
        if r > 0:
            assert torch.equal(tok2, t1), (s, r)
        else:
            assert torch.equal(tok2, teacher), "rate 0: every position feeds its teacher token"
        what = "replay (seed %d, rate %g)" % (s, r)
        assert float(acc2) == pytest.approx(a1), what
        helpers.assert_close(loss2, l1, what=what + ": loss")
        helpers.assert_close(h2.grad, g_h, what=what + ": d hpad")
        for k, p in dec.named_parameters():
            if k != "att.gvec.bias":
                helpers.assert_close(p.grad, g1[k], what="%s: d %s" % (what, k))
    # an eager forward after the capture (new page-locked buffers) still works and gives the eager result
    with torch.cuda.stream(st):
        dec.zero_grad(set_to_none=True)
        random.seed(draws[0][0])
        loss3, _ = dec(hpad, hlen, ys, draws[0][1])
    torch.cuda.synchronize()
    helpers.assert_close(loss3, want[0][0], what="eager forward after the capture")


def test_scheduled_sampling_launch_profile_at_the_bench_shape():
    """One forward at the bench shape and rate 0.5 launches re2e_sample_tokens' kernel olength - 1 times and runs no
    torch.nn.LSTMCell, topk, addmm or cuBLAS kernel."""
    dec, _, hpad, hlen, ys, _, _ = training_case("bench")
    hpad = hpad.to(DEV).requires_grad_(True)
    ys = [y.to(DEV) for y in ys]
    L = max(len(y) for y in ys) + 1
    random.seed(6)
    dec(hpad, hlen, ys, 0.5)                                 # (warm-up)
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU,
                                            torch.profiler.ProfilerActivity.CUDA]) as prof:
        random.seed(6)
        loss, _ = dec(hpad, hlen, ys, 0.5)
        torch.cuda.synchronize()
    counts = {}
    for e in prof.key_averages():
        counts[e.key] = counts.get(e.key, 0) + e.count
    n_sample = sum(c for k, c in counts.items() if "sample_tokens_kernel" in k)
    assert n_sample == L - 1, n_sample
    for op in ("aten::lstm_cell", "aten::topk", "aten::addmm"):
        assert counts.get(op, 0) == 0, op
    blas = [k for k in counts if "re2e" not in k and any(s in k.lower() for s in ("gemm", "gemv", "nvjet", "cublas", "cutlass", "xmma"))]
    assert not blas, blas
