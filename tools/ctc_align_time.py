"""Time the forced CTC alignment (re2e_ctc_align) next to the CTC loss forward (re2e_ctc_loss_fwd) at the bench shape:
B = 32, Th = 200, U = 40, V = 4233, logits in the row-padded layout of the tcgen05 ctc_lo GEMM, hlens ~ U(0.6 Th, Th).

  1. whole calls: CUDA events around each call, the two entry points alternated call by call, median over --iters
     calls of each after --warmup calls of each;
  2. kernels: a separate torch.profiler pass over the same alternation gives the mean time of ctc_lse_kernel (shared by
     both calls), ctc_viterbi_warp_kernel and ctc_ab_warp_kernel (alpha / beta).
The (B,Th,V) logits are 108 MB, close to the 126 MB L2, so a 256 MB buffer is overwritten before every timed call: the
numbers are for logits read from HBM.  Prints the device name and power limit next to the numbers.

    python tools/ctc_align_time.py [--iters 300] [--warmup 30] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from robust_e2e_gan_b200 import _lib, prepare_targets, synth  # noqa: E402
from robust_e2e_gan_b200.linear import _pad4, linear  # noqa: E402


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out or "unknown"
    except Exception:
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=30)
    ap.add_argument("--out", default=None, help="also write the report to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ctc_align_time: needs a CUDA device")
    dev = torch.device("cuda:0")
    B, Th, U, V, D = 32, 200, 40, 4233, 320
    hs, hl = synth.encoder_batch(B=B, Th=Th, D=D, seed=11)
    ys = synth.targets(B=B, V=V, hlens=hl, seed=11, fixed_U=U)
    g = torch.Generator().manual_seed(11)
    W = (torch.randn(V, D, generator=g) * 0.25).to(dev)
    bias = (torch.randn(V, generator=g) * 0.1).to(dev)
    with torch.no_grad():
        x = linear(hs.to(dev), W, bias)
    assert x.stride(1) == _pad4(V)
    tg = prepare_targets(ys, dev)
    hl_d = torch.tensor(hl, dtype=torch.int32, device=dev)
    L = _lib.lib()
    P = _lib.ptr
    nb = int(L.re2e_ctc_ws_bytes(B, Th, V, tg.umax))
    ws = torch.empty(nb, device=dev, dtype=torch.uint8)
    i32 = dict(device=dev, dtype=torch.int32)
    states, tokens, spans = torch.empty(B, Th, **i32), torch.empty(B, Th, **i32), torch.empty(B, tg.umax, 2, **i32)
    score, nll, loss = (torch.empty(n, device=dev) for n in (B, B, 1))
    flush = torch.empty(256 << 20, device=dev, dtype=torch.uint8)
    sb, st = x.stride(0), x.stride(1)

    def align():
        _lib.check(L.re2e_ctc_align(P(x), sb, st, P(tg.labels), P(tg.offs), P(tg.lens), P(hl_d), 0, P(states), P(tokens),
                                    P(spans), P(score), P(ws), nb, B, Th, V, tg.umax, _lib.stream_ptr()), "re2e_ctc_align")

    def loss_fwd():
        _lib.check(L.re2e_ctc_loss_fwd(P(x), sb, st, P(tg.labels), P(tg.offs), P(tg.lens), P(hl_d), 0, P(nll), P(loss),
                                       P(ws), nb, B, Th, V, tg.umax, _lib.stream_ptr()), "re2e_ctc_loss_fwd")

    calls = (("ctc_align", align), ("ctc_loss_fwd", loss_fwd))
    times = {n: [] for n, _ in calls}
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(2)]
    for it in range(args.warmup + args.iters):
        for k, (name, fn) in enumerate(calls):
            flush.fill_(it & 0xff)
            e0, e1 = ev[k]
            e0.record()
            fn()
            e1.record()
        torch.cuda.synchronize()
        if it >= args.warmup:
            for k, (name, _) in enumerate(calls):
                times[name].append(ev[k][0].elapsed_time(ev[k][1]) * 1e3)
    med = {n: round(sorted(v)[len(v) // 2], 2) for n, v in times.items()}
    spread = {n: [round(sorted(v)[len(v) // 10], 2), round(sorted(v)[(9 * len(v)) // 10], 2)] for n, v in times.items()}

    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for it in range(args.iters):
            for name, fn in calls:
                flush.fill_(it & 0xff)
                fn()
        torch.cuda.synchronize()
    kern = {}
    for e in prof.key_averages():
        for key in ("ctc_lse_kernel", "ctc_viterbi_warp_kernel", "ctc_ab_warp_kernel"):
            if key in e.key:
                t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0)
                k = kern.setdefault(key, [0.0, 0])
                k[0] += t
                k[1] += e.count
    kern_us = {k: round(v[0] / max(v[1], 1), 2) for k, v in kern.items()}
    res = {"device": torch.cuda.get_device_name(dev), "power_limit": power_limit(),
           "shape": "B=%d Th=%d U=%d V=%d, logits row pitch %d floats, valid frames %d" % (B, Th, U, V, st, sum(hl)),
           "iters": args.iters, "l2": "256 MB buffer overwritten before every call (logits read from HBM)",
           "call_median_us": med, "call_p10_p90_us": spread, "kernel_mean_us": kern_us,
           "kernel_calls": {k: v[1] for k, v in kern.items()}}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
