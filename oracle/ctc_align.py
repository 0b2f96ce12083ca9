"""Oracle of the forced CTC alignment (csrc/ctc.cu ctc_viterbi_warp_kernel, re2e_ctc_align).  TEST INFRASTRUCTURE ONLY.

The reference has no alignment function (SURVEY.md section 8a-4); this is the textbook Viterbi recursion over the
blank-interleaved CTC lattice of Graves et al. 2006 (the lattice and transitions of oracle/ctc.py ctc_alpha_beta, with
log-sum-exp replaced by max), in float64 numpy, with the device kernel's tie rule.
"""
import numpy as np


def ctc_viterbi(lp_tv, labels, blank=0):
    """Forced alignment of one utterance: the most likely path through the blank-interleaved lattice of ``labels``
    (Viterbi, fp64).  lp_tv (T,V) per-frame log-probabilities (any per-frame constant shift gives the same path).
    Tie rule (the device kernel's): on equal values a state stays in s, else comes from s-1, else from s-2; at the
    end S-1 (final blank) is taken over S-2.
    Returns dict(states (T,) int, tokens (T,) int, spans (U,2) int first/last frame of each label, score float,
    margin float = the smallest gap between the chosen and the runner-up predecessor along the path, and between
    the two end states; inf where there was no alternative).  Infeasible (T < U + adjacent repeats): states, tokens
    and spans -1, score -inf.  T = 0: score 0 for U = 0, else -inf."""
    lp = np.asarray(lp_tv, dtype=np.float64)
    T = lp.shape[0]
    lab = [int(v) for v in labels]
    U = len(lab)
    S = 2 * U + 1
    ext = np.full(S, blank, dtype=np.int64)
    ext[1::2] = lab
    NEG = -np.inf
    skip = np.zeros(S, dtype=bool)
    for s in range(3, S, 2):
        skip[s] = ext[s] != ext[s - 2]
    fail = dict(states=np.full(T, -1, np.int64), tokens=np.full(T, -1, np.int64), spans=np.full((U, 2), -1, np.int64),
                score=(0.0 if U == 0 else NEG) if T == 0 else NEG, margin=np.inf)
    if T == 0:
        return fail
    cand = np.full((T, 3, S), NEG)          # predecessor values: stay, from s-1, from s-2
    bp = np.zeros((T, S), dtype=np.int64)
    v = np.full(S, NEG)
    v[0] = lp[0, ext[0]]
    if S > 1:
        v[1] = lp[0, ext[1]]
    for t in range(1, T):
        c = cand[t]
        c[0] = v
        c[1, 1:] = v[:-1]
        c[2, 2:] = np.where(skip[2:], v[:-2], NEG)
        d = np.zeros(S, dtype=np.int64)
        best = c[0].copy()
        for k in (1, 2):                    # strict: an equal value keeps the earlier choice
            better = c[k] > best
            d[better] = k
            best[better] = c[k][better]
        bp[t] = d
        v = best + lp[t, ext]
    x, y = v[S - 1], (v[S - 2] if S > 1 else NEG)
    if max(x, y) == NEG:
        return fail
    s = S - 2 if y > x else S - 1
    margin = abs(x - y) if S > 1 and y > NEG and x > NEG else np.inf
    states = np.zeros(T, dtype=np.int64)
    for t in range(T - 1, -1, -1):
        states[t] = s
        if t > 0:
            c = cand[t][:, s]
            k = bp[t, s]
            others = [c[j] for j in range(3) if j != k and c[j] > NEG]
            if others:
                margin = min(margin, c[k] - max(others))
            s -= k
    tokens = ext[states]
    spans = np.full((U, 2), -1, np.int64)
    for t in range(T - 1, -1, -1):
        if states[t] & 1:
            spans[states[t] >> 1, 0] = t
    for t in range(T):
        if states[t] & 1:
            spans[states[t] >> 1, 1] = t
    score = float(sum(lp[t, tokens[t]] for t in range(T)))
    return dict(states=states, tokens=tokens, spans=spans, score=score, margin=float(margin))
