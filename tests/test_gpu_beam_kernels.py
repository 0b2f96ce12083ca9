"""GPU: the kernels of one fused beam-search position (csrc/beam.cu, csrc/ctc.cu), each called directly through the C ABI
against a plain restatement of the same operation:

* re2e_ctc_prefix_score against the fp64 prefix-score oracle (fp32 oracle as the reference, fp64 as the truth), at
  V = 4233 and T up to 333, from states reached by running the oracle along a real prefix;
* re2e_beam_merge against a NumPy restatement (stable descending sort of the candidates), bit for bit;
* re2e_beam_advance against re2e_beam_joint + re2e_beam_merge + re2e_beam_gather run separately, bit for bit;
* re2e_beam_init against CTCPrefixScoreOracle.initial_state and the documented initial state, bit for bit."""
import ctypes

import numpy as np
import pytest
import torch

import helpers
from oracle.ctc import CTCPrefixScoreOracle
from robust_e2e_gan_b200 import _lib

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
LOGZERO_CUT = -1e9          # entries at or below this derive from the reference's logzero (-1e10)


def bits(t):
    """Bit pattern of a float32 tensor (so that -0.0 != 0.0 and equality is exact)."""
    return t.detach().contiguous().view(torch.int32).cpu()


def lpz_table(T, V, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.log_softmax(3.0 * torch.randn(T, V, generator=g, dtype=torch.float64), 1).float().numpy()


# ---------------------------------------------------------------------------------------------- CTC prefix scores
@pytest.mark.parametrize("T,H,C", [(1, 3, 8), (2, 5, 15), (75, 32, 32), (200, 12, 15), (333, 8, 32)])
def test_ctc_prefix_score_matches_fp64_oracle(T, H, C):
    """log_psi and r_new of every (hypothesis, candidate) for prefixes of length out_len in {0, 1, T/2, T-1}, candidate
    sets holding blank, <eos>, the prefix's last token (the repeat rule) and duplicates."""
    V, blank = 4233, 0
    eos = V - 1
    lpz = lpz_table(T, V, 1000 + T)
    rng = np.random.RandomState(T * 100 + H)
    # one real prefix of T-1 labels, and the fp64 state after each of its first k labels (r_prev of out_len = k)
    y_full = [eos] + [int(v) for v in rng.randint(1, V - 1, size=max(T - 1, 0))]
    o64 = CTCPrefixScoreOracle(lpz, blank, eos, dtype=np.float64)
    states = [o64.initial_state()]
    for k in range(1, T):
        _, r, _ = o64(y_full[:k], np.array([y_full[k]]), states[-1])
        states.append(r[0])
    out_lens = sorted(set(v for v in (0, 1, T // 2, T - 1) if 0 <= v <= T - 1))
    ol = np.array([out_lens[h % len(out_lens)] for h in range(H)], np.int32)
    last = np.array([y_full[o] for o in ol], np.int32)
    r_prev = np.stack([states[o] for o in ol]).astype(np.float32)      # (H, T, 2): the kernel's input, fp32
    cs = rng.randint(1, V - 1, size=(H, C)).astype(np.int32)
    for h in range(H):
        special = [blank, eos, int(last[h]), int(cs[h, 0])]            # the last one duplicates candidate 0
        for j, v in enumerate(special[:C - 1]):
            cs[h, 1 + (j * 5 + h) % (C - 1)] = v
    if C >= 8:                                                         # and blank / <eos> twice in one row
        cs[0, -1], cs[0, -2] = blank, eos
        cs[0, 1], cs[0, 2] = blank, eos

    psi_d = torch.empty(H, C, device=DEV)
    r_d = torch.full((H, C, T, 2), float("nan"), device=DEV)
    lpz_d, rp_d = torch.from_numpy(lpz).to(DEV), torch.from_numpy(r_prev).to(DEV)
    cs_d, last_d, ol_d = (torch.from_numpy(a).to(DEV) for a in (cs, last, ol))
    L = _lib.lib()
    _lib.check(L.re2e_ctc_prefix_score(_lib.ptr(lpz_d), _lib.ptr(rp_d), _lib.ptr(cs_d), _lib.ptr(last_d), _lib.ptr(ol_d),
                                       _lib.ptr(psi_d), _lib.ptr(r_d), T, V, H, C, blank, eos, _lib.stream_ptr()),
               "re2e_ctc_prefix_score")
    torch.cuda.synchronize()
    psi_k, r_k = psi_d.cpu().double().numpy(), r_d.cpu().double().numpy()

    o32 = CTCPrefixScoreOracle(lpz, blank, eos)
    got_psi, got_r, ref_psi, ref_r, tru_psi, tru_r = ([] for _ in range(6))
    for h in range(H):
        y = y_full[:ol[h] + 1]
        p32, r32, start = o32(y, cs[h], r_prev[h])
        p64, r64, _ = o64(y, cs[h], r_prev[h].astype(np.float64))
        got_psi.append(psi_k[h]), ref_psi.append(p32), tru_psi.append(p64)
        got_r.append(r_k[h, :, start - 1:].ravel()), ref_r.append(r32[:, start - 1:].ravel())
        tru_r.append(r64[:, start - 1:].ravel())
    for what, got, ref, tru in (("log_psi", got_psi, ref_psi, tru_psi), ("r_new", got_r, ref_r, tru_r)):
        got, ref, tru = (np.concatenate(x).astype(np.float64) for x in (got, ref, tru))
        assert np.isfinite(got).all(), what
        # logzero-derived entries on their own: their -1e10 scale would make the element-wise floor accept anything
        zero = tru <= LOGZERO_CUT
        assert np.array_equal(ref <= LOGZERO_CUT, zero), what + ": the fp32 oracle's logzero entries"
        bad = np.flatnonzero((got <= LOGZERO_CUT) != zero)
        assert bad.size == 0, "%s: %d entries on the wrong side of logzero, first at %d: got %r, fp64 %r" % (
            what, bad.size, bad[0], got[bad[0]], tru[bad[0]])
        if (~zero).any():
            helpers.assert_close(got[~zero], ref[~zero], truth=tru[~zero], what=what)


# ---------------------------------------------------------------------------------------------- merge
def merge_ref(out, state, ctl, sc, hist, W, beam, eos, maxlen):
    """NumPy restatement of re2e_beam_merge (include/re2e_b200.h).  Returns the new (state, ctl, sc, hist)."""
    ctl, sc, hist = ctl.copy(), sc.copy(), hist.copy()
    n, pos = int(state[0]), int(state[1])
    if n <= 0 or pos >= maxlen:
        return np.array([n, pos + 1], np.int32), ctl, sc, hist
    win = np.argsort(-out[0, :n].ravel(), kind="stable")[:beam]
    rows = []
    for b, k in enumerate(win):
        r, j = divmod(int(k), beam)
        s, tok, cj = out[0, r, j], out[1, r, j], out[2, r, j]
        hist[pos, :, b] = (s, r, tok, cj)
        if int(tok) != eos and pos != maxlen - 1:
            rows.append((s, r, cj, tok))
    for m in range(W if rows else 0):
        s, r, cj, tok = rows[min(m, len(rows) - 1)]
        ctl[:, m] = (r, cj, tok, pos + 1)
        sc[m] = s
    return np.array([len(rows), pos + 1], np.int32), ctl, sc, hist


def candidates(rng, W, beam, V, eos, eos_top, ties):
    """out (3, W, beam) as re2e_beam_joint writes it: each row's scores sorted descending (equal scores in candidate
    order), token ids, candidate indices.  ``ties``: scores on a coarse grid, so exact ties within and across rows."""
    s = rng.randn(W, beam).astype(np.float32) * 2.0 - 5.0
    if ties:
        s = (np.round(s * 2.0) / 2.0).astype(np.float32)
    if eos_top:
        s[0, 0] = s.max() + 0.5      # row 0's best is the best of all, and it is <eos> (below)
    s = -np.sort(-s, axis=1, kind="stable")
    tok = rng.randint(0, V, size=(W, beam)).astype(np.float32)
    tok[tok == eos] = 1.0
    if eos_top:                      # <eos> among the winners (row 0's best, and one more further down)
        tok[0, 0] = eos
        tok[min(1, W - 1), min(1, beam - 1)] = eos
    cj = np.stack([rng.permutation(max(beam, 15))[:beam] for _ in range(W)]).astype(np.float32)
    return np.stack((s, tok, cj))


def run_merge(out, state, ctl, sc, hist, W, beam, eos, maxlen):
    d = [torch.from_numpy(np.ascontiguousarray(a)).to(DEV) for a in (out, state, ctl, sc, hist)]
    _lib.check(_lib.lib().re2e_beam_merge(*(_lib.ptr(t) for t in d), W, beam, eos, maxlen, _lib.stream_ptr()),
               "re2e_beam_merge")
    torch.cuda.synchronize()
    return [t.cpu().numpy() for t in d[1:]]


MERGE_CASES = [
    # W, beam, n_live, pos, maxlen, eos among winners, ties
    (10, 10, 10, 3, 40, False, False),
    (10, 10, 10, 3, 40, False, True),      # exact ties within and across rows
    (10, 10, 4, 7, 40, False, True),       # n_live < W
    (10, 10, 10, 0, 40, True, True),       # <eos> winners: fewer rows go on
    (6, 6, 1, 0, 9, True, False),          # position 0: one live row, its best candidate is <eos>
    (10, 10, 7, 39, 40, False, True),      # pos = maxlen - 1: every winner ends, nothing survives
    (10, 10, 10, 40, 40, False, False),    # pos >= maxlen: a no-op that only advances pos
    (10, 10, 0, 12, 40, False, False),     # n_live = 0: the same
    (1, 1, 1, 5, 20, False, False),        # greedy
    (1, 1, 1, 5, 20, True, False),         # greedy, <eos>
    (32, 32, 32, 11, 50, True, True),      # the kernel's limit, 1024 candidates
    (32, 32, 17, 11, 50, False, True),
]


@pytest.mark.parametrize("W,beam,n,pos,maxlen,eos_top,ties", MERGE_CASES)
def test_beam_merge_matches_numpy_restatement(W, beam, n, pos, maxlen, eos_top, ties):
    V = 4233
    eos = V - 1
    rng = np.random.RandomState(W * 1000 + n * 10 + pos)
    out = candidates(rng, W, beam, V, eos, eos_top, ties)
    if ties and W > 1 and beam > 1:                           # a tie at the very top, across rows and within row 1
        top = out[0, :2, 0].max()
        out[0, 0, 0] = out[0, 1, 0] = out[0, 1, 1] = top
    state = np.array([n, pos], np.int32)
    ctl = rng.randint(0, 9, size=(4, W)).astype(np.int32)     # what the previous position left there
    sc = rng.randn(W).astype(np.float32)
    hist = np.full((maxlen + 2, 4, beam), -7.0, np.float32)
    want = merge_ref(out, state, ctl, sc, hist, W, beam, eos, maxlen)
    got = run_merge(out, state, ctl, sc, hist, W, beam, eos, maxlen)
    for name, a, b in zip(("state", "ctl", "sc", "hist"), got, want):
        assert a.dtype == b.dtype and np.array_equal(a.view(np.int32), b.view(np.int32)), name
    if eos_top and pos < maxlen - 1 and n > 0:
        assert want[0][0] < beam, "the case was meant to end a hypothesis"


# ---------------------------------------------------------------------------------------------- advance
def _segs(W, Z, Th, Cb, g):
    """State tensors of a search as the fused position lays them out: z (W, Z), r (W, Cb, Th, 2), psi (W, Cb)."""
    src = [torch.randn(W, Z, generator=g), torch.randn(W, Cb, Th, 2, generator=g), torch.randn(W, Cb, generator=g)]
    src = [s.to(DEV) for s in src]
    rowf, subc = [Z, 2 * Th, 1], [0, Cb, Cb]
    return src, rowf, subc


@pytest.mark.parametrize("W,Cb,n,pos,maxlen,ctc,ties", [
    (10, 15, 10, 4, 200, True, False), (10, 15, 10, 4, 200, True, True), (10, 15, 3, 4, 200, True, True),
    (10, 15, 10, 199, 200, True, False), (10, 15, 10, 200, 200, True, False), (10, 15, 0, 9, 200, True, False),
    (21, 31, 21, 2, 30, True, True), (32, 32, 32, 6, 30, False, True), (1, 1, 1, 0, 5, True, False),
    (4, 6, 1, 0, 8, True, True), (7, 7, 7, 3, 9, False, False)])
def test_beam_advance_equals_joint_merge_gather(W, Cb, n, pos, maxlen, ctc, ties):
    """re2e_beam_advance == re2e_beam_joint, re2e_beam_merge, re2e_beam_gather launched one after the other on the same
    inputs, bit for bit in every output (scores, control block, history, state and the gathered rows).  When no
    hypothesis goes on (none survives, or the merge is a no-op past maxlen / without live rows) there is no next
    position, and the advance does not gather: the working copies stay untouched."""
    beam, V, Z, Th = W, 4233, 24, 37
    eos = V - 1
    g = torch.Generator().manual_seed(W * 100 + Cb + n + pos)
    att = torch.log_softmax(torch.randn(W, Cb, generator=g) * 2.0, 1)
    psi = torch.randn(W, Cb, generator=g) * 3.0 - 20.0
    prev = torch.randn(W, generator=g) - 15.0
    if ties:                    # coarse grid: equal joint scores within a row and across rows
        att, psi, prev = (torch.round(t * 2.0) / 2.0 for t in (att, psi, prev))
        att[:, 1] = att[:, 0]
    ids = torch.randint(0, V - 1, (W, Cb), generator=g, dtype=torch.int32)
    ids[0, 0] = eos
    if Cb > 3:
        ids[min(2, W - 1), 3] = eos
    sc = torch.round(torch.randn(W, generator=g) * 4.0) / 4.0 - 30.0
    if ties and W > 1:
        att[1], psi[1], prev[1], sc[1] = att[0], psi[0], prev[0], sc[0]
    att, psi, prev, ids, sc = (t.to(DEV).contiguous() for t in (att, psi, prev, ids, sc))
    w_ctc = 0.3 if ctc else 0.0
    w_att = 1.0 - w_ctc
    lp, pp = (psi, prev) if ctc else (None, None)
    src, rowf, subc = _segs(W, Z, Th, Cb, g)
    ctl0 = torch.randint(0, min(W, Cb), (4, W), generator=g, dtype=torch.int32).to(DEV)
    state0 = torch.tensor([n, pos], dtype=torch.int32, device=DEV)
    hist0 = torch.full((maxlen + 2, 4, beam), -7.0, device=DEV)
    L, P, sp = _lib.lib(), _lib.ptr, _lib.stream_ptr()
    nseg = len(src)
    c_src = (ctypes.c_void_p * nseg)(*[s.data_ptr() for s in src])
    c_rowf, c_subc = (ctypes.c_int * nseg)(*rowf), (ctypes.c_int * nseg)(*subc)

    def fresh():
        dst = [torch.full_like(s[:, 0] if sub else s, -3.0) for s, sub in zip(src, subc)]
        return dict(sc=sc.clone(), state=state0.clone(), ctl=ctl0.clone(), hist=hist0.clone(), dst=dst)

    a = fresh()
    c_dst = (ctypes.c_void_p * nseg)(*[d.data_ptr() for d in a["dst"]])
    _lib.check(L.re2e_beam_advance(P(att), P(ids), P(lp), P(pp), P(a["sc"]), w_att, w_ctc, W, Cb, beam, P(a["state"]),
                                   P(a["ctl"]), P(a["hist"]), eos, maxlen, nseg, c_src, c_dst, c_rowf, c_subc, sp),
               "re2e_beam_advance")
    b = fresh()
    out = torch.empty(3, W, beam, device=DEV)
    _lib.check(L.re2e_beam_joint(P(att), P(ids), P(lp), P(pp), P(b["sc"]), w_att, w_ctc, W, Cb, beam, P(out), sp),
               "re2e_beam_joint")
    _lib.check(L.re2e_beam_merge(P(out), P(b["state"]), P(b["ctl"]), P(b["sc"]), P(b["hist"]), W, beam, eos, maxlen, sp),
               "re2e_beam_merge")
    torch.cuda.synchronize()
    n2 = int(b["state"][0]) if n > 0 and pos < maxlen else 0      # hypotheses that go on to a next position
    if n2 > 0:
        c_dst = (ctypes.c_void_p * nseg)(*[d.data_ptr() for d in b["dst"]])
        _lib.check(L.re2e_beam_gather(P(b["ctl"][0]), P(b["ctl"][1]), W, nseg, c_src, c_dst, c_rowf, c_subc, sp),
                   "re2e_beam_gather")
    torch.cuda.synchronize()
    for k in ("sc", "state", "ctl", "hist"):
        assert torch.equal(bits(a[k]), bits(b[k])), k
    for i, (x, y) in enumerate(zip(a["dst"], b["dst"])):
        assert torch.equal(bits(x), bits(y)), "gathered segment %d" % i
    if n2 == 0:
        assert all(bool((d == -3.0).all()) for d in a["dst"]), "gathered without a next position"
    else:                       # and the gather took the rows the merge chose
        par, cand = b["ctl"][0].long(), b["ctl"][1].long()
        assert torch.equal(a["dst"][0], src[0][par]) and torch.equal(a["dst"][1], src[1][par, cand])
    # the joint scores themselves against the reference's tensor expression (model/e2e_decoder.py:284-292)
    local = w_att * att + w_ctc * (psi - prev.unsqueeze(1)) if ctc else att
    bs, _ = torch.topk(local, beam, dim=1)
    assert torch.equal(out[0], sc.unsqueeze(1) + bs)


# ---------------------------------------------------------------------------------------------- init
@pytest.mark.parametrize("Th,ctc", [(1, True), (75, True), (200, True), (333, True), (50, False)])
def test_beam_init_state(Th, ctc):
    """re2e_beam_init: r_in of every row == CTCPrefixScoreOracle.initial_state (sequential fp32 sum of the blank
    column), alignment uniform 1/Th, z = c = 0, psi = 0, ctl = {parent 0, candidate 0, <sos>, position 0}, sc = 0,
    state = {1 live hypothesis, position 0} -- every buffer pre-filled with garbage first."""
    W, Z, V = 10, 300, 4233
    sos = V - 1
    lpz = lpz_table(Th, V, 77 + Th)
    junk = float("nan")
    z, c, a = (torch.full((W, n_), junk, device=DEV) for n_ in (Z, Z, Th))
    r = torch.full((W, Th, 2), junk, device=DEV) if ctc else None
    psi = torch.full((W,), junk, device=DEV) if ctc else None
    lpz_d = torch.from_numpy(lpz).to(DEV) if ctc else None
    ctl = torch.full((4, W), -5, dtype=torch.int32, device=DEV)
    sc = torch.full((W,), junk, device=DEV)
    state = torch.full((2,), -5, dtype=torch.int32, device=DEV)
    P = _lib.ptr
    _lib.check(_lib.lib().re2e_beam_init(P(z), P(c), P(a), P(r), P(psi), P(lpz_d), P(ctl), P(sc), P(state), W, Z, Th, V,
                                         0, sos, _lib.stream_ptr()), "re2e_beam_init")
    torch.cuda.synchronize()
    zero = torch.zeros(W, Z, dtype=torch.int32)
    assert torch.equal(bits(z), zero) and torch.equal(bits(c), zero)
    u = np.float32(1.0) / np.float32(Th)
    assert torch.equal(bits(a), bits(torch.full((W, Th), float(u))))
    assert torch.equal(bits(sc), torch.zeros(W, dtype=torch.int32))
    assert ctl.cpu().tolist() == [[0] * W, [0] * W, [sos] * W, [0] * W]
    assert state.cpu().tolist() == [1, 0]
    if ctc:
        want = torch.from_numpy(CTCPrefixScoreOracle(lpz, 0, sos).initial_state())
        for w in range(W):
            assert torch.equal(bits(r[w]), bits(want)), "row %d" % w
        assert torch.equal(bits(psi), torch.zeros(W, dtype=torch.int32))
