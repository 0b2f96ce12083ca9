"""Time one- and two-layer decoders (``--dlayers`` 1 and 2) on the paths the library offers them, in one run:

Beam search at beam 10, ctc_weight 0.3, Th = 137, V = 4233, D = A = 320, Z = 300 (the recipe's dimensions), with the
<eos> logit lowered by 30 so that no hypothesis ends and every search runs its full maxlen = Th positions:
  position   the fused position (csrc/beam.cu launches, dlayers + 5 per position) as a warm CUDA-graph replay of 8
             positions, 16 replays = 128 positions after position 0, CUDA events; us per position.  The working set
             (weights and search state, a few MB) is L2-resident, as it is between the positions of a real search.
  utterance  wall time of recognize_beam (fused) and of Decoder._recognize_generic (tensor ops + CUDA graph, host merge
             after every position) for the whole utterance, ended by a device synchronise; also per position.
Training: Decoder.forward + backward at B = 32, Th = 200, 40 labels (41 positions), V = 4233, captured once per
variant (fused_lstm on / off) and replayed; L2 is overwritten (256 MB write) before every timed replay.
Variants alternate round by round; medians and min / max over the rounds.  The GPU name and power limit are read in the
same run and written beside the numbers.

    python tools/decoder_layers_time.py [--rounds 15] [--out FILE.json]
"""
import argparse
import gc
import json
import os
import random
import subprocess
import sys
import time
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from robust_e2e_gan_b200 import CTC, AttLoc, Decoder, synth  # noqa: E402
from robust_e2e_gan_b200.hotpath import DEFAULT_CFG  # noqa: E402

D = A = 320
Z, V, C, FILTS = 300, 4233, 10, 100


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out or "unknown"
    except Exception:
        return "unknown"


def stats(v):
    s = sorted(v)
    return {"median": round(s[len(s) // 2], 3), "min": round(s[0], 3), "max": round(s[-1], 3)}


def make_decoder(dlayers, dev, seed=7):
    torch.manual_seed(seed)
    dec = Decoder(D, V, dlayers, Z, V - 1, V - 1, AttLoc(D, Z, A, C, FILTS, "softmax"))
    return dec.to(dev)


class L2Flush(object):
    """Overwrites 256 MB (twice the B200's 126 MB L2) on the given stream."""

    def __init__(self, dev):
        self.buf = torch.empty(64 << 20, dtype=torch.float32, device=dev)

    def __call__(self):
        self.buf.fill_(1.0)


def beam_part(dev, rounds, out):
    Th, beam = 137, 10
    ra = types.SimpleNamespace(beam_size=beam, penalty=0.0, ctc_weight=0.3, maxlenratio=0.0, minlenratio=0.0, nbest=1,
                               lm_weight=0.0, cuda_graph=True)
    g = torch.Generator().manual_seed(5)
    h = torch.tanh(torch.randn(Th, D, generator=g)).to(dev)
    torch.manual_seed(3)
    ctc = CTC(V, D, 0.0).to(dev).eval()
    decs = {}
    with torch.no_grad():
        lpz = ctc.log_softmax(h.unsqueeze(0))[0]
        for nl in (1, 2):
            dec = make_decoder(nl, dev).eval()
            dec.output.bias[V - 1] -= 30.0                       # no hypothesis ends: every search runs Th positions
            decs[nl] = dec
    stream = torch.cuda.current_stream(dev)

    def position_us(dec):
        """us per position: 16 graph replays of 8 positions after position 0 of a fresh search."""
        plan = dec._fused_plan(h, lpz, ra)
        assert plan is not None, "the fused position should take this decoder"
        hb, lp, Cb, maxlen, _ = plan
        pin = torch.empty(maxlen, 4, beam, dtype=torch.float32).pin_memory()
        dec.att.reset()
        pos = dec._fused_position(hb, lp, Cb, beam, ra.ctc_weight, maxlen, pin, dec._beam_tables())
        pos()                                                    # position 0 (also loads every kernel)
        side = torch.cuda.Stream(dev)
        side.wait_stream(stream)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.stream(side):
            graph.capture_begin()
            for _ in range(8):
                pos()
            graph.capture_end()
        stream.wait_stream(side)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(16):
            graph.replay()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1000.0 / 128

    def wall_ms(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1000.0, res

    times = {}
    results = {}
    with torch.no_grad():
        for rnd in range(rounds + 2):
            for nl, dec in decs.items():
                t = {"position_us fused": position_us(dec)}
                t["utterance_ms fused"], r_f = wall_ms(lambda: dec.recognize_beam(h, lpz, ra))
                t["utterance_ms generic"], r_g = wall_ms(lambda: dec._recognize_generic(h, lpz, ra))
                results[nl] = (r_f, r_g)
                if rnd >= 2:                                     # (two warm-up rounds)
                    for k, v in t.items():
                        times.setdefault("dlayers %d: %s" % (nl, k), []).append(v)
    out["beam_search"] = {
        "workload": "recognize_beam, beam %d, ctc_weight 0.3, Th %d (= positions), V %d, D = A = %d, Z %d"
                    % (beam, Th, V, D, Z),
        "note": "position_us: warm graph replay, L2-resident working set; utterance_ms: wall time of one search ended "
                "by a device synchronise (generic position: host merge after every position)",
        "times": {k: stats(v) for k, v in sorted(times.items())},
        "same_tokens_fused_generic": {"dlayers %d" % nl: [x["yseq"] for x in r_f] == [x["yseq"] for x in r_g]
                                      for nl, (r_f, r_g) in results.items()},
        "positions_run": {"dlayers %d" % nl: len(r_f[0]["yseq"]) - 2 for nl, (r_f, _) in results.items()}}
    for nl in (1, 2):
        for k in ("fused", "generic"):
            out["beam_search"]["times"]["dlayers %d: utterance_us_per_position %s" % (nl, k)] = round(
                stats(times["dlayers %d: utterance_ms %s" % (nl, k)])["median"] * 1000.0 / Th, 1)


def training_part(dev, rounds, out):
    B, Th, U = DEFAULT_CFG["B"], DEFAULT_CFG["Th"], DEFAULT_CFG["U"]
    hpad, hl = synth.encoder_batch(B=B, Th=Th, D=D, seed=77)
    ys = [y.to(dev) for y in synth.targets(B=B, V=V, hlens=hl, seed=77, fixed_U=U)]
    hpad = hpad.to(dev).requires_grad_(True)
    hl_dev = torch.tensor(hl, device=dev, dtype=torch.int32)
    st = torch.cuda.Stream(dev)
    st.wait_stream(torch.cuda.current_stream(dev))
    flush = L2Flush(dev)
    graphs = {}
    for nl in (1, 2):
        dec = make_decoder(nl, dev).train()
        for fused in (True, False):
            dec.fused_lstm = fused
            with torch.cuda.stream(st):
                for _ in range(2):
                    loss, _ = dec(hpad, hl_dev, ys, 0.0)
                    loss.backward()
                    dec.zero_grad(set_to_none=True)
                    hpad.grad = None
            torch.cuda.synchronize()
            del loss
            gc.collect()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=st, capture_error_mode="thread_local"):
                loss, _ = dec(hpad, hl_dev, ys, 0.0)
                loss.backward()
            dec.zero_grad(set_to_none=True)
            hpad.grad = None
            graphs["dlayers %d: fused_lstm %s" % (nl, "on" if fused else "off")] = (graph, dec, loss)

    def timed(graph):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(st):
            flush()
            e0.record(st)
            graph.replay()
            e1.record(st)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    times = {k: [] for k in graphs}
    for rnd in range(rounds + 2):
        for k, (graph, _, _) in graphs.items():
            t = timed(graph)
            if rnd >= 2:
                times[k].append(t)
    out["training"] = {
        "workload": "Decoder.forward + backward (teacher forcing), B %d, Th %d, %d labels (%d positions), V %d, D = A "
                    "= %d, Z %d, CUDA-graph replay, L2 overwritten before every replay" % (B, Th, U, U + 1, V, D, Z),
        "times_ms": {k: stats(v) for k, v in times.items()}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=15)
    ap.add_argument("--out", default=None, help="also write the JSON result here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("decoder_layers_time: needs a CUDA device")
    dev = torch.device("cuda:0")
    random.seed(0)
    out = {"device": torch.cuda.get_device_name(dev), "power_limit": power_limit(), "rounds": args.rounds}
    beam_part(dev, args.rounds, out)
    training_part(dev, args.rounds, out)
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
