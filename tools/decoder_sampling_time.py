"""Time Decoder.forward + backward with scheduled sampling at the bench shape (B = 32, Th = 200, U = 40, V = 4233: the
workload of bench.py's decoder_forward_bench).

Variants, alternated round by round, medians of CUDA-event times:
  teacher   the teacher-forced path (rate 0) as a graph replay -- what bench.py reports as decoder_forward;
  ss r      the scheduled-sampling path captured once at rate 0.5 and replayed after draw_sampling(r), r = 0, 0.5, 1.0;
  free 0.5  the library-free loop (fused_lstm = False: torch.nn.LSTMCell, per-position output layer and topk), eager.
Prints the device name and power limit next to the numbers.

    python tools/decoder_sampling_time.py [--rounds 15]
"""
import argparse
import gc
import json
import os
import random
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from robust_e2e_gan_b200 import AttLoc, Decoder, synth  # noqa: E402
from robust_e2e_gan_b200.hotpath import DEFAULT_CFG  # noqa: E402


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out or "unknown"
    except Exception:
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=15)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("decoder_sampling_time: needs a CUDA device")
    dev = torch.device("cuda:0")
    B, Th, D, A, Z, C, V, U = (DEFAULT_CFG[k] for k in ("B", "Th", "D", "A", "Z", "C", "V", "U"))
    torch.manual_seed(7)
    dec = Decoder(D, V, 1, Z, V - 1, V - 1, AttLoc(D, Z, A, C, DEFAULT_CFG["filts"], "softmax")).to(dev).train()
    hpad, hl = synth.encoder_batch(B=B, Th=Th, D=D, seed=77)
    ys = [y.to(dev) for y in synth.targets(B=B, V=V, hlens=hl, seed=77, fixed_U=U)]
    hpad = hpad.to(dev).requires_grad_(True)
    hl_dev = torch.tensor(hl, device=dev, dtype=torch.int32)
    st = torch.cuda.Stream(dev)
    st.wait_stream(torch.cuda.current_stream(dev))

    def fwd_bwd(rate, lengths):
        loss, _ = dec(hpad, lengths, ys, rate)
        loss.backward()

    def capture(rate):
        with torch.cuda.stream(st):
            for _ in range(2):
                fwd_bwd(rate, hl_dev)
                dec.zero_grad(set_to_none=True)
                hpad.grad = None
        torch.cuda.synchronize()
        gc.collect()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=st, capture_error_mode="thread_local"):
            fwd_bwd(rate, hl_dev)
        dec.zero_grad(set_to_none=True)
        hpad.grad = None
        return g

    teacher = capture(0.0)
    ss = capture(0.5)                       # captured last: draw_sampling refills this graph's flags

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(st):
            e0.record(st)
            fn()
            e1.record(st)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    def free():
        dec.fused_lstm = False
        try:
            fwd_bwd(0.5, hl)
        finally:
            dec.fused_lstm = True

    times = {k: [] for k in ("teacher graph", "ss 0.0 graph", "ss 0.5 graph", "ss 1.0 graph", "free 0.5 eager")}
    for rnd in range(args.rounds + 2):
        random.seed(rnd)
        t = {"teacher graph": timed(teacher.replay)}
        for r in (0.0, 0.5, 1.0):
            dec.draw_sampling(r)
            t["ss %.1f graph" % r] = timed(ss.replay)
        t["free 0.5 eager"] = timed(free)
        if rnd >= 2:                         # (two warm-up rounds)
            for k, v in t.items():
                times[k].append(v)
    med = {k: round(sorted(v)[len(v) // 2], 3) for k, v in times.items()}
    spread = {k: [round(min(v), 3), round(max(v), 3)] for k, v in times.items()}
    print(json.dumps({"device": torch.cuda.get_device_name(dev), "power_limit": power_limit(),
                      "workload": "Decoder.forward + backward, B=%d Th=%d U=%d V=%d" % (B, Th, U, V),
                      "rounds": args.rounds, "median_ms": med, "min_max_ms": spread}))


if __name__ == "__main__":
    main()
