"""GPU: hybrid CTC/attention beam search at the shape bench.py times (its ``recog`` record), against the fp32 CPU oracle
(oracle/beam.py).  Token sequences must be IDENTICAL; scores within 1e-4 relative.

These searches are unlike the small ones of test_gpu_decoder.py: V = 4233, D = A = 320, Z = 300, beam 10, and most
of them run for well over a hundred positions without any <eos>, so they end through the append at the last position.
That is the lazy-history path of ``_FusedSearch.poll``: no host bookkeeping until the first <eos>, then the hypotheses
are rebuilt from the history buffer."""
import types

import numpy as np
import pytest
import torch

import helpers
from oracle import beam as obeam
from robust_e2e_gan_b200 import CTC, AttLoc, Decoder

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
N_UTTS = 8

# Must stay equal to bench.py's recog_bench workload (its BEAM_CASES["_recog"], utterance generator and lengths).
RECOG_CASE = dict(V=4233, D=320, Z=300, A=320, C=10, filts=100, Th=200, beam=10, ctc_weight=0.3, nbest=1, penalty=0.0,
                  maxlenratio=0.0, minlenratio=0.0, eos_bias=2.0, seed=5000)


@pytest.fixture(scope="module")
def recog():
    """(case, decoder, CTC module, encoder outputs, oracle n-best lists) of the first N_UTTS utterances of the bench."""
    helpers.BEAM_CASES["_recog"] = dict(RECOG_CASE)
    try:
        c, sd, _, _ = helpers.beam_case("_recog")
    finally:
        del helpers.BEAM_CASES["_recog"]
    g = torch.Generator().manual_seed(5001)
    lens = torch.randint(75, 201, (1000,), generator=g).tolist()
    hs = [torch.tanh(torch.randn(lens[i], c["D"], generator=g)) for i in range(N_UTTS)]
    with torch.no_grad():
        refs = [obeam.recognize_beam(sd, h, c) for h in hs]
    att = AttLoc(c["D"], c["Z"], c["A"], c["C"], c["filts"], "softmax")
    dec = Decoder(c["D"], c["V"], 1, c["Z"], c["sos"], c["eos"], att)
    ctc = CTC(c["V"], c["D"], 0.0)
    dec.load_state_dict({k: v for k, v in sd.items() if not k.startswith("ctc_lo")}, strict=True)
    ctc.load_state_dict({k: v for k, v in sd.items() if k.startswith("ctc_lo")}, strict=True)
    return c, dec.to(DEV).eval(), ctc.to(DEV).eval(), hs, refs


def recog_args(c):
    return types.SimpleNamespace(beam_size=c["beam"], penalty=c["penalty"], ctc_weight=c["ctc_weight"],
                                 maxlenratio=c["maxlenratio"], minlenratio=c["minlenratio"], nbest=c["nbest"],
                                 lm_weight=0.0)


def check_against_oracle(got, refs):
    for u, (nb, ref) in enumerate(zip(got, refs)):
        assert len(nb) == len(ref), "utterance %d: %d hypotheses, oracle %d" % (u, len(nb), len(ref))
        for k, (a, b) in enumerate(zip(nb, ref)):
            if a["yseq"] != b["yseq"]:
                n = next((i for i, (x, y) in enumerate(zip(a["yseq"], b["yseq"])) if x != y),
                         min(len(a["yseq"]), len(b["yseq"])))
                raise AssertionError("utterance %d, hypothesis %d: tokens differ from position %d on (%s vs oracle %s), "
                                     "lengths %d / %d" % (u, k, n, a["yseq"][n:n + 3], b["yseq"][n:n + 3],
                                                         len(a["yseq"]), len(b["yseq"])))
            assert abs(a["score"] - b["score"]) <= 1e-4 * abs(b["score"]), (u, k, a["score"], b["score"])


@pytest.mark.parametrize("batched", [True, False], ids=["recognize_beam_batch", "recognize_beam"])
def test_beam_search_matches_oracle_at_bench_shape(recog, batched):
    """The bench's decode (recognize_beam_batch, 4 searches interleaved) and one recognize_beam per utterance both give
    the oracle's n-best, for utterances of 75 to 200 frames."""
    c, dec, ctc, hs, refs = recog
    ra = recog_args(c)
    with torch.no_grad():
        hd = [h.to(DEV) for h in hs]
        lpz = [ctc.log_softmax(h.unsqueeze(0))[0] for h in hd]
        if batched:
            got = dec.recognize_beam_batch(hd, lpz, ra, None, concurrency=4)
        else:
            got = [dec.recognize_beam(h, l, ra, None) for h, l in zip(hd, lpz)]
    check_against_oracle(got, refs)
    # the workload is what the module docstring says: most searches run to maxlen = Th without an <eos>
    long_ones = sum(len(r[0]["yseq"]) == h.size(0) + 2 for r, h in zip(refs, hs))
    assert long_ones >= N_UTTS // 2, long_ones
