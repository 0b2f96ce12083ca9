"""CPU: the fp64 forced-alignment oracle (oracle.ctc_align.ctc_viterbi) against brute-force enumeration of every frame
labelling that collapses to the transcript."""
import itertools

import numpy as np
import pytest

from oracle import ctc as o_ctc
from oracle import ctc_align as o_align


def collapse(y, blank=0):
    out, prev = [], None
    for v in y:
        if v != blank and v != prev:
            out.append(v)
        prev = v
    return out


def labelling_states(y, blank=0):
    """Lattice state of every frame of a labelling that collapses to the transcript (unique)."""
    st, u, prev = [], 0, None
    for v in y:
        if v == blank:
            st.append(2 * u)
        elif v == prev:
            st.append(st[-1])
        else:
            u += 1
            st.append(2 * u - 1)
        prev = v
    return st


def brute_force(lp, labels, blank=0):
    """(best score, [(score, states)] of every labelling collapsing to labels)."""
    T, V = lp.shape
    paths = []
    for y in itertools.product(range(V), repeat=T):
        if collapse(y, blank) == list(labels):
            paths.append((float(sum(lp[t, y[t]] for t in range(T))), labelling_states(y, blank)))
    best = max((p[0] for p in paths), default=-np.inf)
    return best, paths


def tie_rule_pick(paths, best, tol=0.0):
    """The tie rule (stay before s-1 before s-2 at every step, final blank before the last label) picks, among the
    maximisers, the path whose states read from the last frame backwards are lexicographically largest."""
    cands = [tuple(reversed(s)) for sc, s in paths if sc >= best - tol]
    return list(reversed(max(cands)))


def check_spans(res, labels):
    st = res["states"]
    for u in range(len(labels)):
        frames = np.nonzero(st == 2 * u + 1)[0]
        assert len(frames) > 0
        assert res["spans"][u, 0] == frames[0] and res["spans"][u, 1] == frames[-1]
        assert frames[-1] - frames[0] + 1 == len(frames)      # one run of frames per label


CASES = [
    # (T, V, labels)
    (1, 3, []), (4, 3, []), (1, 3, [2]), (3, 3, [1]), (5, 3, [1, 1]), (5, 4, [1, 2, 3]), (6, 3, [1, 1, 2]),
    (7, 4, [3, 3, 3]), (7, 4, [1, 2, 1, 2]), (6, 2, [1]), (7, 3, [2, 1, 2]), (4, 4, [1, 2, 3, 1]),
    # infeasible: T < U + adjacent repeats
    (2, 3, [1, 1]), (3, 4, [1, 2, 3, 2]), (4, 3, [2, 2, 2]),
]


@pytest.mark.parametrize("T,V,labels", CASES)
@pytest.mark.parametrize("seed", [0, 1])
def test_viterbi_matches_enumeration(T, V, labels, seed):
    rng = np.random.default_rng(1000 * seed + 7 * T + V + len(labels))
    x = rng.normal(size=(T, V)) * 2
    lp = x - np.log(np.exp(x).sum(1, keepdims=True))
    res = o_align.ctc_viterbi(lp, labels)
    best, paths = brute_force(lp, labels)
    if not paths:
        assert res["score"] == -np.inf
        assert (res["states"] == -1).all() and (res["tokens"] == -1).all() and (res["spans"] == -1).all()
        return
    assert res["score"] == pytest.approx(best, abs=1e-12)
    maximisers = [list(s) for sc, s in paths if sc >= best - 1e-12]
    assert list(res["states"]) in maximisers
    ext = np.zeros(2 * len(labels) + 1, np.int64)
    ext[1::2] = labels
    assert (res["tokens"] == ext[res["states"]]).all()
    assert collapse(res["tokens"]) == list(labels)
    check_spans(res, labels)
    assert res["margin"] >= 0


@pytest.mark.parametrize("T,V,labels", [c for c in CASES if c[0] >= 3])
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_viterbi_integer_ties_follow_the_rule(T, V, labels, seed):
    """Integer log-probabilities in fp64: every sum is exact and ties are everywhere."""
    rng = np.random.default_rng(seed + 17 * T)
    lp = -rng.integers(0, 3, size=(T, V)).astype(np.float64)
    res = o_align.ctc_viterbi(lp, labels)
    best, paths = brute_force(lp, labels)
    if not paths:
        assert res["score"] == -np.inf
        return
    assert res["score"] == best
    assert list(res["states"]) == tie_rule_pick(paths, best)


def test_hand_built_ties():
    # uniform frames, one label: (1,1,1) (1,1,b) (1,b,b) (b,1,1) (b,1,b) (b,b,1) all tie; the rule ends in the final
    # blank and then stays as long as it can
    lp = np.zeros((3, 2))
    res = o_align.ctc_viterbi(lp, [1])
    assert list(res["states"]) == [1, 2, 2] and res["margin"] == 0.0
    # stay in the label state rather than come from the blank before it
    lp = np.array([[0., 0., -5.], [-5., 0., -5.], [-5., -5., 0.]])
    res = o_align.ctc_viterbi(lp, [1, 2])
    # (1,1,2) and (b,1,2) tie: at frame 1 state 1 stays (from 1) rather than coming from 0
    assert list(res["states"]) == [1, 1, 3] and res["score"] == 0.0
    # s-1 before s-2: (1,b,2) and (1,1,2) tie at state 3 of frame 2 -> comes from state 2 (the blank)
    lp = np.array([[-5., 0., -5.], [0., 0., -5.], [-5., -5., 0.]])
    res = o_align.ctc_viterbi(lp, [1, 2])
    assert list(res["states"]) == [1, 2, 3]
    assert list(res["spans"].ravel()) == [0, 0, 2, 2]


def test_edges():
    r = o_align.ctc_viterbi(np.zeros((0, 3)), [])
    assert r["score"] == 0.0 and r["states"].shape == (0,)
    r = o_align.ctc_viterbi(np.zeros((0, 3)), [1])
    assert r["score"] == -np.inf and (r["spans"] == -1).all()
    lp = np.log(np.full((4, 3), 1 / 3))
    r = o_align.ctc_viterbi(lp, [])
    assert list(r["states"]) == [0] * 4 and r["score"] == pytest.approx(4 * np.log(1 / 3))
    # exactly one path: T = U, no repeats
    rng = np.random.default_rng(5)
    x = rng.normal(size=(4, 6))
    lp = x - np.log(np.exp(x).sum(1, keepdims=True))
    r = o_align.ctc_viterbi(lp, [1, 2, 3, 4])
    assert list(r["states"]) == [1, 3, 5, 7] and r["margin"] == np.inf
    assert r["score"] == pytest.approx(-o_ctc.ctc_alpha_beta(x, [1, 2, 3, 4])["nll"], abs=1e-12)
