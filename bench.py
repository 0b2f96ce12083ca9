#!/usr/bin/env python
"""Benchmark of the joint-step hot path (fused front-end x3 + CTC + 41-step AttLoc loop, fwd + bwd).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (config.workload): BASELINE.json configs[2]/[3] per-GPU shape -- B=32 utterances, T=800 STFT
frames x 257 bins -> 40 mel, encoder length Th=200, U=40 labels (41 decoder steps), vocab 4233,
D=A=320, Z=300, C=10, K=201, mtlalpha=0.5; synthetic seeded tensors (robust_e2e_gan_b200/synth.py).
Metric: utterances/sec = (N * 32) / step time.  One process per GPU (torchrun for N > 1): every rank
runs its own 32 utterances and the hot-path parameter gradients are all-reduced (NCCL) -> weak scaling.

JSON keys beyond the base contract: ``roofline`` (dominant kernel, CUDA-event timed), ``kernels``
(every kernel of ours with achieved GB/s), ``cpu_baseline`` (the oracle port timed on the host cores),
``e2e`` (public nn.Module API, pinned host inputs copied in and the loss read back every step),
``gpu_launches``, ``clocks``.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# stdout carries exactly ONE JSON line (the contract).  NCCL prints its version banner / debug lines to the process's
# stdout from C, so file descriptor 1 is pointed at stderr for the whole run and the JSON line is written to a private
# duplicate of the original stdout.
_JSON_OUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)
sys.stdout = sys.stderr


def emit(line):
    _JSON_OUT.write(json.dumps(line) + "\n")
    _JSON_OUT.flush()


import torch  # noqa: E402

METRIC = "utterances/sec (joint step fwd/bwd)"
UNIT = "utt/s"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def tensor_peak_tf32():
    """Dense TF32 tensor peak used for the GEMM entries: half the MEASURED bf16 cuBLAS throughput
    (MEASURED_PEAKS.json; tf32 runs at half the bf16 rate on tcgen05), else half the recipe's fallback."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return round(float(json.load(f)["bf16_tflops"]) / 2.0, 1)
    return 1125.0


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons through NVML while the timed region runs."""

    def __init__(self, index=0, period=0.02):
        super().__init__(daemon=True)
        self.period, self.index = period, index
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if mask & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def cpu_arm():
    """(step function, kind) of the CPU arm: the reference's OWN modules (oracle/_ref copy or /root/reference, imported
    unmodified through oracle/refshim.py) when they are present -- kind "reference" -- else the oracle port."""
    from oracle import refshim
    if refshim.available():
        from oracle.reference_step import reference_step
        return reference_step, "reference"
    from oracle.hotpath_oracle import oracle_step
    return oracle_step, "port"


def cpu_step_time(cfg, batch, sd, reps, warm):
    """The reference's CPU path fwd+bwd on the host cores (median of reps); returns (seconds, kind)."""
    step, kind = cpu_arm()
    for _ in range(warm):
        step(cfg, batch, sd)
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        step(cfg, batch, sd)
        ts.append(time.perf_counter() - t0)
    ts.sort()
    return ts[len(ts) // 2], kind


def sub_batch(batch, cfg, nb):
    """First nb utterances of a host batch (bounded CPU sample of the same workload)."""
    from robust_e2e_gan_b200.hotpath import Batch
    d = {}
    for k in Batch.FIELDS:
        v = getattr(batch, k)
        if k in ("dec_z", "g_c"):
            d[k] = v[:, :nb].contiguous()
        elif k == "cmvn":
            d[k] = v
        else:
            d[k] = v[:nb].contiguous()
    c2 = dict(cfg)
    c2["B"] = nb
    return Batch(ys=batch.ys[:nb], hlens_list=batch.hlens_list[:nb], targets=None, **d), c2


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path -- its unmodified FbankModel / CTC /
    AttLoc modules (oracle/_ref) driven through the same step as our arm, all host threads.  A step covers the same
    global batch as our arm's: --gpus N -> the N per-GPU batches of 32 utterances (seeds 4000+r, as our ranks use),
    one after the other in ONE process (rank 0; the CPU arm has nothing to shard onto)."""
    if rank != 0:
        return
    from robust_e2e_gan_b200.hotpath import DEFAULT_CFG, HotPath, make_batch
    cfg = dict(DEFAULT_CFG)
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    nrep = max(1, args.gpus)
    batches = [make_batch(cfg, seed=4000 + r) for r in range(nrep)]
    sd = HotPath(cfg, seed=4000).state_dict_cpu()
    step, kind = cpu_arm()
    nb = cfg["B"]
    t0 = time.perf_counter()
    step(cfg, batches[0], sd)                  # untimed probe
    if (time.perf_counter() - t0) * nrep * (args.steps + args.warmup) > 600.0:
        nb = 8                                 # very slow host: bound the sample, and say so in the line
    scfg = cfg
    if nb != cfg["B"]:
        batches = [sub_batch(b, cfg, nb)[0] for b in batches]
        scfg = dict(cfg, B=nb)
    for _ in range(args.warmup):
        for b in batches:
            step(scfg, b, sd)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        for b in batches:
            step(scfg, b, sd)
    dt = (time.perf_counter() - t0) / args.steps
    val = nb * nrep / dt
    sample = ("the full step: %d x %d utterances, all %d decoder steps" % (nrep, nb, cfg["steps"]) if nb == cfg["B"] else
              "%d of the %d utterances of each of the %d per-GPU batches, all %d decoder steps, per step"
              % (nb, cfg["B"], nrep, cfg["steps"]))
    conf = workload_config(cfg, nrep)
    if nb != cfg["B"]:
        conf["workload"] += " -- CPU arm sampled: " + sample
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
            "config": conf,
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


def workload_config(cfg, world):
    return {"workload": "joint hot path, BASELINE configs[2]/[3] per-GPU shape: B=%d/GPU T=%d F=%d M=%d Th=%d U=%d "
                        "(%d AttLoc steps) V=%d D=A=%d Z=%d" % (cfg["B"], cfg["T"], cfg["F"], cfg["M"], cfg["Th"],
                                                                  cfg["U"], cfg["steps"], cfg["V"], cfg["D"], cfg["Z"]),
            "global_batch": cfg["B"] * world, "parallelism": "dp%d (utterance-sharded, grad all-reduce)" % world,
            "l2": "256 MiB scratch write between timed steps (excluded from step time)"}


def kernel_specs(hp, db, cfg, dev):
    """(name, callable, algorithmic bytes per launch, repetitions) for each of OUR kernels, on the bench
    tensors and through the same C-ABI calls the step makes."""
    from robust_e2e_gan_b200 import _lib
    L = _lib.lib()
    B, T, F, M, Th, D, A, Z, C, V, U = (cfg[k] for k in ("B", "T", "F", "M", "Th", "D", "A", "Z", "C", "V", "U"))
    K = 2 * cfg["filts"] + 1
    N = B * T
    sp = _lib.stream_ptr
    P = _lib.ptr
    res = {}
    f32 = dict(device=dev, dtype=torch.float32)
    fc = hp.feat.fc.detach()
    Y, G, dY, din = (torch.empty(B, T, M, **f32), torch.empty(B, T, M, **f32), torch.randn(B, T, M).to(dev),
                     torch.empty(B, T, F, **f32))
    lens = db.lens.to(torch.int32)
    att = hp.att
    W_dec, W_att = att.mlp_dec.weight.detach().contiguous(), att.mlp_att.weight.detach().contiguous()
    W_conv = att.loc_conv.weight.detach().view(C, K).contiguous()
    W_decT = W_dec.t().contiguous()
    gv, gb = att.gvec.weight.detach().view(A).contiguous(), att.gvec.bias.detach().contiguous()
    enc = db.hpad.contiguous()
    pre = torch.addmm(att.mlp_enc.bias.detach(), enc.view(B * Th, D), att.mlp_enc.weight.detach().t()).view(B, Th, A)
    ap = torch.softmax(torch.randn(B, Th), 1).to(dev)
    c, w, dproj, conv = torch.empty(B, D, **f32), torch.empty(B, Th, **f32), torch.empty(B, A, **f32), torch.empty(B, Th, C, **f32)
    xsave = torch.empty(B, Th, A, **f32)
    dz = db.dec_z[0].contiguous()
    dc, dw = torch.randn(B, D).to(dev), torch.randn(B, Th).to(dev)
    d_pre, ddp, dprev = torch.zeros(B, Th, A, **f32), torch.empty(B, A, **f32), torch.empty(B, Th, **f32)
    nslots = int(L.re2e_attloc_acc_slots(B, Th, D, A, Z, C, K))
    acc = torch.zeros(nslots, int(L.re2e_attloc_acc_floats(A, C, K)), **f32)
    d_dz = torch.empty(B, Z, **f32)
    logits = torch.randn(B, Th, V).to(dev)
    grad = torch.empty_like(logits)
    tg = db.targets
    hl = db.hlens.to(torch.int32)
    nb = int(L.re2e_ctc_ws_bytes(B, Th, V, tg.umax))
    ws = torch.empty(nb, device=dev, dtype=torch.uint8)
    nll, loss = torch.empty(B, **f32), torch.empty(1, **f32)
    valid_frames = int(hl.sum())

    # the front-end kernels the step really runs: banded (streaming) for the mel bank, dense tcgen05 otherwise
    from robust_e2e_gan_b200.feat_model import _band_for
    band = _band_for(hp.feat.fc, B, T)
    Y1, Y2 = torch.empty(B, T, M, **f32), torch.empty(B, T, M, **f32)

    def k_fb_fwd():
        if band is not None:
            _lib.check(L.re2e_fbank_band_fwd(P(db.mask_logits), 1, P(db.mix), None, P(band[0]), P(band[1]), P(db.cmvn),
                                             P(lens), P(Y), P(G), None, None, B, T, F, M, sp()))
        else:
            _lib.check(L.re2e_fbank_fwd(P(db.mask_logits), 1, P(db.mix), P(fc), P(db.cmvn), P(lens), P(Y), P(G), None,
                                        B, T, F, M, sp()))

    def k_fb_fwd_plain():
        if band is not None:
            _lib.check(L.re2e_fbank_band_fwd(None, 0, P(db.clean), None, P(band[0]), P(band[1]), P(db.cmvn), None, P(Y),
                                             None, None, None, B, T, F, M, sp()))
        else:
            _lib.check(L.re2e_fbank_fwd(None, 0, P(db.clean), P(fc), P(db.cmvn), None, P(Y), None, None, B, T, F, M, sp()))

    def k_fb_joint():
        _lib.check(L.re2e_fbank_band_fwd(P(db.mask_logits), 1, P(db.mix), P(db.clean), P(band[0]), P(band[1]), P(db.cmvn),
                                         P(lens), P(Y), P(G), P(Y1), P(Y2), B, T, F, M, sp()))

    def k_fb_bwd():
        if band is not None:
            _lib.check(L.re2e_fbank_band_bwd(P(dY), P(G), P(db.mask_logits), 1, P(db.mix), P(band[2]), P(band[3]), P(lens),
                                             P(din), B, T, F, M, sp()))
        else:
            _lib.check(L.re2e_fbank_bwd(P(dY), P(G), P(db.mask_logits), 1, P(db.mix), P(fc), P(lens), P(din), None,
                                        B, T, F, M, sp()))

    def k_att_fwd():
        _lib.check(L.re2e_attloc_step_fwd(P(pre), P(enc), P(dz), P(ap), P(W_dec), P(W_att), P(W_conv), P(gv), P(gb),
                                          2.0, P(c), P(w), P(dproj), P(conv), P(xsave), B, Th, D, A, Z, C, K, sp()))

    def k_att_bwd():
        _lib.check(L.re2e_attloc_step_bwd(P(dc), P(dw), P(xsave), P(enc), P(ap), P(w), P(conv), P(W_dec), P(W_decT),
                                          P(W_att), P(W_conv), P(gv), 2.0, P(d_pre), 1, P(ddp), P(d_dz), P(dprev), P(acc),
                                          nslots, B, Th, D, A, Z, C, K, sp()))

    # the whole decoder loop (all `steps` attention steps) in one persistent cluster kernel per direction
    NS = cfg["steps"]
    dec_proj_all = torch.randn(NS, B, A, **f32) * 0.3
    dec_proj_all[0].zero_()
    c_all, w_all = torch.empty(NS, B, D, **f32), torch.empty(NS, B, Th, **f32)
    conv_all = torch.empty(NS, B, Th, C, **f32)
    dc_all = torch.randn(NS, B, D, **f32) / (B * D) ** 0.5
    dw_all = torch.zeros(NS, B, Th, **f32)
    dw_all[-1] = torch.randn(B, Th, **f32) / B ** 0.5
    att0 = torch.full((B, Th), 1.0 / Th, **f32)
    d_pre_l, d_dproj_l = torch.empty(B, Th, A, **f32), torch.empty(NS, B, A, **f32)
    lslots = int(L.re2e_attloc_loop_slots(NS, B, Th, D, A, C, K))
    have_loop = lslots > 0 and bool(L.re2e_attloc_loop_supported(NS, B, Th, D, A, C, K))
    acc_l = torch.empty(max(lslots, 1), int(L.re2e_attloc_acc_floats(A, C, K)), **f32)

    def k_loop_fwd():
        _lib.check(L.re2e_attloc_loop_fwd(P(pre), P(enc), P(dec_proj_all), P(att0), P(W_att), P(W_conv), P(gv), P(gb), 2.0,
                                          P(c_all), P(w_all), P(conv_all), NS, B, Th, D, A, C, K, sp()))

    def k_loop_bwd():
        _lib.check(L.re2e_attloc_loop_bwd(P(pre), P(enc), P(dec_proj_all), P(att0), P(w_all), P(conv_all), P(dc_all),
                                          P(dw_all), P(W_att), P(W_conv), P(gv), 2.0, P(d_pre_l), P(d_dproj_l), P(acc_l),
                                          lslots, NS, B, Th, D, A, C, K, sp()))

    def k_ctc_fwd():
        _lib.check(L.re2e_ctc_loss_fwd(P(logits), Th * V, V, P(tg.labels), P(tg.offs), P(tg.lens), P(hl), 0, P(nll),
                                       P(loss), P(ws), nb, B, Th, V, tg.umax, sp()))

    def k_ctc_bwd():
        _lib.check(L.re2e_ctc_loss_bwd(P(logits), Th * V, V, P(tg.labels), P(tg.offs), P(tg.lens), P(hl), 0, P(nll),
                                       None, P(ws), nb, P(grad), B, Th, V, tg.umax, sp()))

    # dense layers on the tcgen05 3xTF32 GEMM (ctc_lo fwd / dX / dW, mlp_enc fwd): (flops, "tensor") entries
    from robust_e2e_gan_b200.linear import gemm_tf32x3, _pad4
    Wlo, blo = hp.ctc.ctc_lo.weight.detach().contiguous(), hp.ctc.ctc_lo.bias.detach().contiguous()
    Wenc, benc = att.mlp_enc.weight.detach().contiguous(), att.mlp_enc.bias.detach().contiguous()
    R = B * Th
    x2 = enc.view(R, D)
    lg = torch.empty(R, _pad4(V), **f32)[:, :V]
    gl = (torch.randn(R, _pad4(V), **f32) * 1e-3)[:, :V]
    dx, dWlo, pre2 = torch.empty(R, D, **f32), torch.empty(V, D, **f32), torch.empty(R, A, **f32)

    def k_lo_fwd():
        gemm_tf32x3(x2, False, Wlo, False, lg, R, V, D, bias=blo)

    def k_lo_dx():
        gemm_tf32x3(gl, False, Wlo, True, dx, R, D, V)

    def k_lo_dw():
        gemm_tf32x3(gl, True, x2, True, dWlo, V, D, R)

    def k_enc_fwd():
        gemm_tf32x3(x2, False, Wenc, False, pre2, R, A, D, bias=benc)

    if have_loop:
        k_loop_fwd()          # w_all / conv_all of a real forward feed the backward timing
        torch.cuda.synchronize()
    S = 2 * tg.umax + 1
    nst = cfg["steps"]
    # Decoder-loop kernels: "algorithmic" = SURVEY 8(d)'s per-step figure x the steps one launch processes (the bytes
    # a step-at-a-time formulation has to move: pre + enc_h read per step; + the d pre accumulation in the backward);
    # "resident" = what the persistent kernel really moves (pre / enc_h once, the small per-step tensors, and in the
    # backward the L2-resident d pre reduce-add per step).
    loop_fwd_alg = nst * (4.0 * B * Th * (A + D) + 4.0 * B * (A + Th * (2 + C) + D))
    loop_bwd_alg = nst * (4.0 * B * Th * (A + D) + 4.0 * B * Th * A + 4.0 * B * Th * (4 + C))
    loop_fwd_res = 4.0 * B * Th * (A + D) + nst * 4.0 * B * (A + D + Th + Th * C)
    loop_bwd_res = 4.0 * B * Th * (A + D) + nst * (4.0 * B * Th * A + 4.0 * B * (2 * A + D + 3 * Th + Th * C))
    specs = ([("fbank_joint_fwd(mask,mix,clean->3Y,G)", k_fb_joint, 4.0 * N * (3 * F + 4 * M), 4)] if band is not None else []) + [
        ("fbank_fwd(mask,mag->Y,G)", k_fb_fwd, 4.0 * N * (2 * F + 2 * M), 4),
        ("fbank_fwd(mag->Y)", k_fb_fwd_plain, 4.0 * N * (F + M), 4),
        ("fbank_bwd(->d mask)", k_fb_bwd, 4.0 * N * (2 * M + 3 * F), 4),
        ("attloc_step_fwd", k_att_fwd, 4.0 * B * Th * (2 * A + D) + 4.0 * B * (Z + Th * (2 + C) + D + A), 20),
        ("attloc_step_bwd", k_att_bwd, 4.0 * B * Th * (A + D) + 4.0 * B * Th * A + 4.0 * B * Th * (4 + C), 20),
    ] + ([
        ("attloc_loop_fwd(%d steps)" % nst, k_loop_fwd, loop_fwd_alg, 2, {"steps": nst, "resident_MB": round(loop_fwd_res / 1e6, 2)}),
        ("attloc_loop_bwd(%d steps)" % nst, k_loop_bwd, loop_bwd_alg, 2, {"steps": nst, "resident_MB": round(loop_bwd_res / 1e6, 2)}),
    ] if have_loop else []) + [
        ("ctc_fwd(lse+alpha/beta)", k_ctc_fwd, 4.0 * valid_frames * V + 4.0 * 3 * valid_frames * S, 4),
        ("ctc_bwd(grad)", k_ctc_bwd, 4.0 * valid_frames * V + 4.0 * B * Th * V, 4),
        ("gemm ctc_lo fwd (%dx%dx%d)" % (R, V, D), k_lo_fwd, ("flop", 2.0 * R * V * D), 4),
        ("gemm ctc_lo dX (%dx%dx%d)" % (R, D, V), k_lo_dx, ("flop", 2.0 * R * V * D), 4),
        ("gemm ctc_lo dW (%dx%dx%d)" % (V, D, R), k_lo_dw, ("flop", 2.0 * R * V * D), 4),
        ("gemm mlp_enc fwd (%dx%dx%d)" % (R, A, D), k_enc_fwd, ("flop", 2.0 * R * A * D), 8),
    ]
    return specs


RECOG_CONCURRENCY = 4


def recog_bench(rank, world, dev, total_utts=1000, per_rank_cap=125):
    """BASELINE configs[4] (joint_recog.py:143-149, run.sh:199-226): hybrid CTC/attention beam search, beam 10,
    ctc_weight 0.3, maxlenratio = minlenratio = 0 (end_detect), nbest 1, over a seeded set of 1000 synthetic utterances
    (encoder outputs Th ~ U(75, 200) = T/4 of 300..800 frames; default AttLoc / decoder / CTC dimensions, V = 4233),
    utterance-sharded across the ranks with no collective.  Every rank decodes at most ``per_rank_cap`` utterances of
    its shard (8 ranks x 125 = the full set; fewer ranks = a bounded sample of the same set, stated in the record) so
    that the default run stays short.  Returns (utterances decoded by this rank, seconds, tokens emitted)."""
    import types
    from robust_e2e_gan_b200 import CTC, AttLoc, Decoder, synth
    from robust_e2e_gan_b200.parallel import shard_range
    synth.BEAM_CASES["_recog"] = dict(V=4233, D=320, Z=300, A=320, C=10, filts=100, Th=200, beam=10, ctc_weight=0.3,
                                      nbest=1, penalty=0.0, maxlenratio=0.0, minlenratio=0.0, eos_bias=2.0, seed=5000)
    c, sd, _, _ = synth.beam_case("_recog")
    att = AttLoc(c["D"], c["Z"], c["A"], c["C"], c["filts"], "softmax")
    dec = Decoder(c["D"], c["V"], 1, c["Z"], c["sos"], c["eos"], att)
    ctc = CTC(c["V"], c["D"], 0.0)
    dec.load_state_dict({k: v for k, v in sd.items() if not k.startswith("ctc_lo")})
    ctc.load_state_dict({k: v for k, v in sd.items() if k.startswith("ctc_lo")})
    dec, ctc = dec.to(dev).eval(), ctc.to(dev).eval()
    g = torch.Generator().manual_seed(5001)
    lens = torch.randint(75, 201, (total_utts,), generator=g).tolist()
    lo, hi = shard_range(total_utts, rank, world)
    hi = min(hi, lo + per_rank_cap)
    hs = {}
    for i in range(total_utts):                    # one generator stream: utterance i is the same at every world size
        h = torch.tanh(torch.randn(lens[i], c["D"], generator=g))
        if lo <= i < hi:
            hs[i] = h.pin_memory()
    ra = types.SimpleNamespace(beam_size=c["beam"], penalty=c["penalty"], ctc_weight=c["ctc_weight"],
                               maxlenratio=c["maxlenratio"], minlenratio=c["minlenratio"], nbest=c["nbest"], lm_weight=0.0)

    def decode(idx):
        """A group of utterances through Decoder.recognize_beam_batch (4 searches interleaved on their own streams)."""
        with torch.no_grad():
            hd = [hs[i].to(dev, non_blocking=True) for i in idx]
            lp = [ctc.log_softmax(h.unsqueeze(0))[0] for h in hd]
            return dec.recognize_beam_batch(hd, lp, ra, None, concurrency=RECOG_CONCURRENCY)

    decode(list(range(lo, min(hi, lo + RECOG_CONCURRENCY))))      # warm-up (allocator, shared-memory attributes, streams)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    toks = 0
    for nb in decode(list(range(lo, hi))):
        toks += len(nb[0]["yseq"]) - 1
    torch.cuda.synchronize()
    return hi - lo, time.perf_counter() - t0, toks


def decoder_forward_bench(cfg, dev, reps=5):
    """Next-row N1 (model/e2e_decoder.py:79-167): the REAL training loop of the attention decoder -- AttLoc step kernel,
    LSTMCell step on the library's kernels, teacher forcing, output layer batched on the tcgen05 GEMM, cross-entropy -- forward + backward at
    the bench shape (B=32, Th=200, U=40 labels -> 41 positions, V=4233).  Eager launches (median of `reps`)."""
    from robust_e2e_gan_b200 import AttLoc, Decoder, synth
    B, Th, D, A, Z, C, V, U = (cfg[k] for k in ("B", "Th", "D", "A", "Z", "C", "V", "U"))
    torch.manual_seed(7)
    att = AttLoc(D, Z, A, C, cfg["filts"], "softmax")
    dec = Decoder(D, V, 1, Z, V - 1, V - 1, att).to(dev).train()
    hpad, hl = synth.encoder_batch(B=B, Th=Th, D=D, seed=77)
    ys = [y.to(dev) for y in synth.targets(B=B, V=V, hlens=hl, seed=77, fixed_U=U)]
    hpad = hpad.to(dev).requires_grad_(True)
    from robust_e2e_gan_b200 import _lib
    ts, launches = [], 0
    st = torch.cuda.Stream(dev)      # everything on one side stream: the later capture must not meet autograd state
    st.wait_stream(torch.cuda.current_stream(dev))      # (gradient accumulators) tied to the default stream
    with torch.cuda.stream(st):
        for it in range(reps + 2):
            dec.zero_grad()
            hpad.grad = None
            torch.cuda.synchronize()
            n0 = _lib.launch_count()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            loss, acc = dec(hpad, hl, ys, 0.0)
            loss.backward()
            e1.record(st)
            torch.cuda.synchronize()
            launches = _lib.launch_count() - n0
            if it >= 2:
                ts.append(e0.elapsed_time(e1))
    ts.sort()
    ms = ts[len(ts) // 2]
    rec = {"workload": "Decoder.forward + backward (teacher forcing), B=%d Th=%d U=%d V=%d" % (B, Th, U, V),
           "ms_eager": round(ms, 3), "utt_per_s_eager": round(B / (ms * 1e-3), 1), "our_kernel_launches": int(launches),
           "mode": "AttLoc per-step cluster kernels; LSTMCell = embedding-half gates of all positions in one tcgen05 GEMM + "
                   "ONE cluster kernel per position (both recurrent products, split-K over a 4-CTA cluster, pointwise cell as "
                   "epilogue; backward: pointwise kernel + one 8-CTA-cluster product launch); one tcgen05 output-layer GEMM"}
    # the same forward + backward captured once into a CUDA graph (lengths as a device tensor: no host round trip
    # inside the loop) and replayed: what the loop costs on the GPU once the Python / launch overhead is gone
    try:
        import gc
        hl_dev = torch.tensor(hl, device=dev, dtype=torch.int32)
        dec.zero_grad(set_to_none=True)
        hpad.grad = None
        loss = acc = None
        gc.collect()
        with torch.cuda.stream(st):
            for _ in range(2):
                loss, acc = dec(hpad, hl_dev, ys, 0.0)
                loss.backward()
                dec.zero_grad(set_to_none=True)
                hpad.grad = None
        torch.cuda.synchronize()
        loss = acc = None
        gc.collect()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=st, capture_error_mode="thread_local"):
            loss, acc = dec(hpad, hl_dev, ys, 0.0)
            loss.backward()
        ts = []
        for _ in range(reps + 2):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(st):
                e0.record(st)
                g.replay()
                e1.record(st)
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        ts = sorted(ts[2:])
        msg = ts[len(ts) // 2]
        rec.update(ms_graph_replay=round(msg, 3), utt_per_s_graph_replay=round(B / (msg * 1e-3), 1))
        del g
    except Exception as ex:      # a capture failure must not take the headline line down
        rec["graph_replay_error"] = str(ex)[:200]
    return rec


def kernel_rooflines(hp, db, cfg, peak, dev):
    """Per-kernel CUDA-event timings: each kernel is captured R times into a CUDA graph and replayed, so
    the events see back-to-back launches without Python gaps.  achieved = algorithmic bytes / avg launch."""
    res = {}
    f32 = dict(device=dev, dtype=torch.float32)
    flush = torch.empty(64 * 1024 * 1024, **f32)
    flush_mode = os.environ.get("RE2E_FLUSH", "write")     # A/B: "write+read" leaves CLEAN lines in L2
    for spec in kernel_specs(hp, db, cfg, dev):
        name, fn, nbytes, reps = spec[:4]
        extra = spec[4] if len(spec) > 4 else {}
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(3):
                fn()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for _ in range(reps):
                fn()
        ts = []
        for _ in range(5):
            if not name.startswith("attloc"):      # AttLoc's working set is L2-resident in the real loop too
                flush.fill_(1.0)
                if flush_mode == "write+read":
                    flush.sum()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            g.replay()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e3 / reps)
        ts.sort()
        us = ts[len(ts) // 2]
        if isinstance(nbytes, tuple):       # tensor-bound entry: fp32-equivalent flops; 3 TF32 MMAs per product
            fl = nbytes[1]
            tf = fl / (us * 1e-6) / 1e12
            tf32_peak = tensor_peak_tf32()
            res[name] = {"us_per_launch": round(us, 2), "algorithmic_GFLOP": round(fl / 1e9, 2),
                         "achieved_TFLOPs_fp32_equiv": round(tf, 1), "executed_TFLOPs_tf32": round(3 * tf, 1),
                         "frac_of_tf32_peak": round(3 * tf / tf32_peak, 3), "bound": "tensor",
                         "tf32_peak_TFLOPs": tf32_peak}
            continue
        ach = nbytes / (us * 1e-6) / 1e9
        res[name] = {"us_per_launch": round(us, 2), "algorithmic_MB": round(nbytes / 1e6, 2),
                     "achieved_GBps": round(ach, 1), "frac_of_hbm_peak": round(ach / peak, 3)}
        if "steps" in extra:
            res[name]["us_per_step"] = round(us / extra["steps"], 2)
        res[name].update(extra)
    return res


DUMP_LIMIT_BYTES = 64 * 1000 * 1000


def dump_items(out):
    """(name, tensor) of what a step returns to its caller (``HotPath.step``: features, losses, attention, gradients).
    Keys starting with '_' are buffers a data-parallel job adds after the replay (the all-reduced gradients)."""
    for k, v in out.items():
        if not k.startswith("_"):
            yield k, (torch.stack(list(v)) if isinstance(v, (list, tuple)) else v)   # per-step loop: d_dec_z is a list


def check_dump_size(out):
    total = sum(4 * v.numel() for _, v in dump_items(out))
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit("--dump-outputs: %d bytes exceed the %d-byte limit" % (total, DUMP_LIMIT_BYTES))


def dump_outputs(out, path):
    """Every tensor of ``dump_items(out)`` as ``path/<name>.npy`` in float32, so that two builds can be compared output
    for output on the same seeded inputs.  At the bench shape that is the whole output, about 56 MB."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for k, v in dump_items(out):
        np.save(os.path.join(path, k + ".npy"), v.detach().float().cpu().numpy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-kernels", action="store_true")
    ap.add_argument("--no-overlap", action="store_true", help="run the three branches of the step on ONE stream (A/B)")
    ap.add_argument("--no-recog", action="store_true", help="skip the beam-search (configs[4]) record")
    ap.add_argument("--per-step-loop", action="store_true",
                    help="one AttLoc launch per decoder step instead of the persistent loop kernels (A/B)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs and gradients of the last timed step of --impl ours as DIR/<name>.npy "
                         "(rank 0); choose a DIR outside the source tree")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    from robust_e2e_gan_b200.parallel import init_distributed
    world_env = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, int(os.environ.get("RANK", "0")), world_env)
        return

    import torch.distributed as dist
    rank, world = init_distributed()
    local = int(os.environ.get("LOCAL_RANK", "0"))
    from robust_e2e_gan_b200.parallel import bind_host_to_gpu
    bound_cpus = bind_host_to_gpu(local)                 # before any pinned allocation (first touch decides the node)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    from robust_e2e_gan_b200 import _lib
    from robust_e2e_gan_b200.hotpath import DEFAULT_CFG, HotPath, make_batch
    cfg = dict(DEFAULT_CFG)
    peak, peak_src = load_peaks()

    from robust_e2e_gan_b200.hotpath import StepRunner
    hp = HotPath(cfg, seed=4000, overlap=not args.no_overlap, fused_loop=not args.per_step_loop).to(dev)   # identical init on every rank
    hb = make_batch(cfg, seed=4000 + rank).pin()         # distinct utterances per rank
    db = hb.to(dev)
    torch.cuda.synchronize()
    flush = torch.empty(64 * 1024 * 1024, device=dev, dtype=torch.float32)   # 256 MiB > 126 MB L2

    def barrier():
        # device first: the replayed graphs carry their own NCCL kernels, and collectives of one job must not be
        # enqueued eagerly while a replay that contains others is still in flight (their order could differ per rank)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # Gradient exchange of the data-parallel job (DESIGN.md section 5).  Default: ONE flat NCCL all-reduce (6.2 MB) on the
    # step's stream right after each replay.  RE2E_GRAD_REDUCE=graph captures the exchange INSIDE the step graph instead:
    # ctc_lo.weight (5.4 MB) is reduced from its post-accumulate-grad hook on the CTC branch's stream while the decoder
    # loop is still running, the small gradients (0.83 MB) as one flat message at the end, on their own communicator.
    # Measured: N=2 1.84 ms (default: 1.83), N=8 1.98 ms (default: 1.87) (the NCCL CTAs then hold SMs the latency-bound decoder chain
    # is waiting for, and eight ranks reach the hook with more skew) -- hence opt-in.
    grad_keys = ["d_" + k for k, p in hp.named_parameters() if p.requires_grad]
    reduce_in_graph = world > 1 and os.environ.get("RE2E_GRAD_REDUCE", "post") == "graph"
    if reduce_in_graph:
        big = [p for _, p in hp.named_parameters() if p.requires_grad and p.numel() * p.element_size() >= (1 << 20)]
        small_keys = ["d_" + k for k, p in hp.named_parameters()
                      if p.requires_grad and p.numel() * p.element_size() < (1 << 20)]
        inflight = []
        gg = dist.new_group(list(range(world)))     # own communicator: never interleaves with the eager barrier / MAX

        def reduce_when_ready(p):
            inflight.append(dist.all_reduce(p.grad, op=dist.ReduceOp.AVG, group=gg, async_op=True))

        for p in big:
            p.register_post_accumulate_grad_hook(reduce_when_ready)

        def join_grad_reduce(out):
            flat = torch.cat([out[k].reshape(-1) for k in small_keys if k in out])
            dist.all_reduce(flat, op=dist.ReduceOp.AVG, group=gg)
            out["_small_grads_mean"] = flat
            while inflight:
                inflight.pop().wait()

        hp.after_backward = join_grad_reduce

    # ---- warm-up (eager public modules), launch count of one step
    n0 = _lib.launch_count()
    hp.step(db, hlens_for_att=db.hlens)
    torch.cuda.synchronize()
    launches_per_step = _lib.launch_count() - n0
    for _ in range(max(0, args.warmup - 1)):
        for p in hp.parameters():
            p.grad = None
        hp.step(db, hlens_for_att=db.hlens)
    torch.cuda.synchronize()

    # ---- the step as a user runs it: StepRunner = CUDA-graph replay over static buffers, H2D on a copy stream
    # only what is host-resident in the reference flow crosses PCIe per step (mix, clean, lengths, labels); the
    # stand-ins for tensors that upstream networks produce on the device stay resident (declared in the e2e record)
    runner = StepRunner(hp, hb, slots=3, upstream="device")
    if args.dump_outputs:
        check_dump_size(runner.slots[0]["out"])     # every rank, before any collective: all of them stop together
    mode = "cuda_graph" + ("" if args.no_overlap else " (front-end | CTC | decoder-loop branches on 3 streams)")
    if reduce_in_graph:
        mode += "; gradient all-reduce captured in the graph (ctc_lo.weight from its grad hook, the rest as one flat message)"
    elif world > 1:
        def allreduce_grads(out):
            flat = torch.cat([out[k].reshape(-1) for k in grad_keys if k in out])
            dist.all_reduce(flat, op=dist.ReduceOp.AVG)
            out["_grads_flat_mean"] = flat
        runner.post = allreduce_grads
        mode += "; one flat gradient all-reduce after each replay"
    if rank == 0:
        sys.stderr.write("[bench] timing mode: %s; launches/step %d\n" % (mode, launches_per_step))

    rs = runner.run_stream
    for _ in range(3):
        runner.replay_resident(0)
    sampler = ClockSampler(local)
    barrier()
    sampler.start()
    evs = []
    for _ in range(args.steps):
        with torch.cuda.stream(rs):
            flush.fill_(0.0)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(rs)
        out = runner.replay_resident(0)
        e1.record(rs)
        evs.append((e0, e1))
    barrier()
    total_ms = sum(a.elapsed_time(b) for a, b in evs)
    clocks = sampler.stop()
    t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_per_step = float(t.item()) / args.steps
    value = cfg["B"] * world / (ms_per_step * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(out, args.dump_outputs)

    # ---- end to end through StepRunner: every step copies its pinned host batch in and reads the loss back.
    #      Two steps of look-ahead over three input slots: while step i computes, batch i+1 is already resident and
    #      batch i+2 is being copied (copy stream), so neither the PCIe transfer (52.7 MB, ~1.0 ms at 55 GB/s) nor the
    #      host-side staging sits on the critical path of the loop.
    # The loop is timed in steady state: the pipeline is primed first (untimed), then every timed iteration submits one
    # host batch (its H2D copy happens inside the window) and reads one finished step's loss back (D2H, synchronises).
    # (t0 is taken right after a result read, with `ahead` steps in flight -- exactly the state the loop is in at t1;
    # a device synchronize here would let the first `ahead` timed reads return steps finished before the window.)
    ahead = 2
    barrier()
    for _ in range(ahead):
        runner.submit(hb)
    for _ in range(3):
        runner.submit(hb)
        float(runner.result()["loss_ctc"].detach().cpu())
    t0 = time.perf_counter()
    d2h = 0
    for i in range(args.steps):
        runner.submit(hb)
        lv = runner.result()["loss_ctc"].detach().cpu()      # D2H read of the step's result (synchronises)
        d2h = lv.numel() * 4
    t1 = time.perf_counter()
    for _ in range(ahead):                                   # drain (untimed)
        runner.result()
    barrier()
    e2e_s = torch.tensor([(t1 - t0) / args.steps], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e = {"value": cfg["B"] * world / float(e2e_s.item()), "unit": UNIT, "h2d_bytes_per_step": runner.h2d_bytes(hb),
           "d2h_bytes_per_step": d2h, "ms_per_step": float(e2e_s.item()) * 1e3,
           "h2d_tensors": runner.h2d_tensors(hb),
           "device_resident_stand_ins": runner.resident_tensors(hb),
           "h2d_note": "copied per step = what the reference's collated batch holds on the host "
                       "(data/mix_data_loader.py:264-302: spectra, lengths, labels); mask logits, encoder output, decoder "
                       "states, incoming gradients and CMVN constants are produced on the device by the networks around "
                       "the path in the reference flow (model/enhance_model.py:131-156, model/e2e_encoder.py, "
                       "model/e2e_decoder.py:128) and stay device-resident here",
           "api": "robust_e2e_gan_b200.hotpath.StepRunner (graph replay; 3 input slots, H2D of batches i+1 / i+2 overlaps step i)"}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "fp32", "data": "synthetic", "config": workload_config(cfg, world),
            "mode": mode, "host_affinity": ("%d CPUs local to the GPU" % bound_cpus) if bound_cpus else "inherited",
            "e2e": e2e, "gpu_launches": int(launches_per_step * args.steps), "clocks": clocks}

    # ---- BASELINE configs[4]: beam search, utterance-sharded, no collective (a secondary record on the same line)
    if not args.no_recog:
        barrier()
        try:
            n_dec, sec, toks = recog_bench(rank, world, dev)
        except Exception as ex:       # a secondary record must never take the headline line down
            sys.stderr.write("[bench] recog record failed: %s\n" % str(ex)[:300])
            n_dec, sec, toks = 0, 1.0, 0
        rt = torch.tensor([sec, float(n_dec), float(toks)], device=dev, dtype=torch.float64)
        if world > 1:
            mx = rt.clone()
            dist.all_reduce(mx, op=dist.ReduceOp.MAX)
            dist.all_reduce(rt, op=dist.ReduceOp.SUM)
            sec = float(mx[0].item())
        total_dec, total_tok = int(rt[1].item()), int(rt[2].item())
        line["recog"] = {"error": "beam-search record failed on at least one rank"} if total_dec == 0 else {
                         "metric": "utterances/sec (beam search, beam=10, ctc_weight=0.3, maxlenratio=0)",
                         "value": total_dec / sec, "unit": "utt/s", "n_gpus": world, "utterances": total_dec,
                         "of_set": 1000, "tokens_per_utt": total_tok / max(1, total_dec),
                         "ms_per_utt_per_gpu": sec / max(1, total_dec / world) * 1e3,
                         "sample": "%d of the 1000 seeded utterances (each rank decodes <= 125 of its shard; 8 ranks "
                                   "cover the set); seeded untrained weights never emit <eos>, so every search runs "
                                   "to maxlen = Th -- the longest case" % total_dec,
                         "workload": "BASELINE configs[4]: joint_recog beam search, Th~U(75,200), V=4233, D=A=320, "
                                     "Z=300, sharded by utterance, no collective",
                         "mode": "whole output position on the device: 6 library launches (AttLoc step, LSTM step, output "
                                 "layer, log-softmax+top-k, CTC prefix scores, joint+merge+gather), 8 positions per graph "
                                 "replay, winners written to a page-locked history buffer that the host book-keeps in chunks; "
                                 "%d utterances' searches interleaved on their own streams "
                                 "(Decoder.recognize_beam_batch)" % RECOG_CONCURRENCY}
    if rank == 0:
        if not args.no_kernels:
            ks = kernel_rooflines(hp, db, cfg, peak, dev)
            line["kernels"] = ks
            # launches of each kernel in ONE step of the timed workload (the per-step AttLoc kernels are only launched
            # when the loop kernels cannot take the shape)
            fused = hp.fused_loop and any(k.startswith("attloc_loop") for k in ks)
            joint = hp.joint_frontend and any(k.startswith("fbank_joint") for k in ks)
            per_step = {"attloc_step_fwd": 0 if fused else cfg["steps"], "attloc_step_bwd": 0 if fused else cfg["steps"],
                        "fbank_fwd(mag->Y)": 0 if joint else 2, "fbank_fwd(mask,mag->Y,G)": 0 if joint else 1}
            dom = max((k for k in ks if "frac_of_hbm_peak" in ks[k]),
                      key=lambda k: ks[k]["us_per_launch"] * per_step.get(k, 1))
            line["roofline"] = {"kernel": dom, "bound": "hbm", "achieved": ks[dom]["achieved_GBps"], "peak": peak,
                                "unit": "GB/s", "frac": ks[dom]["frac_of_hbm_peak"], "peak_source": peak_src,
                                "launches_per_step": per_step.get(dom, 1), "us_per_launch": ks[dom]["us_per_launch"],
                                "traffic": None}
            # DRAM bytes per launch of that kernel from the committed `ncu --set full` capture (profiles/traffic.json,
            # written by tools/summarize_profiles.py); null when no capture of this kernel is committed
            tpath = os.path.join(ROOT, "profiles", "traffic.json")
            if os.path.exists(tpath):
                with open(tpath) as f:
                    tj = json.load(f)
                tk = next((k for k in tj.get("kernels", {}) if dom.startswith(k)), None)
                if tk is not None:
                    line["roofline"]["traffic"] = tj["kernels"][tk]["bytes"]
                    line["roofline"]["traffic_source"] = tj.get("source")
            line["roofline"]["algorithmic_bytes"] = int(ks[dom]["algorithmic_MB"] * 1e6)
        if not args.no_kernels:
            try:
                line["decoder_forward"] = decoder_forward_bench(cfg, dev)
            except Exception as ex:
                line["decoder_forward"] = {"error": str(ex)[:200]}
        if world == 1 and not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            torch.set_num_threads(cores)
            dt, kind = cpu_step_time(cfg, hb, hp.state_dict_cpu(), reps=5, warm=2)
            line["cpu_baseline"] = {"value": cfg["B"] / dt, "unit": UNIT, "cores": cores, "kind": kind,
                                    "sample": "the full step on the same batch: %d utterances, all %d decoder steps; "
                                              "2 warm-ups + median of 5" % (cfg["B"], cfg["steps"]),
                                    "ms_per_step": dt * 1e3}
        emit(line)
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()
        # teardown: graphs first (they hold the captured collectives' communicator), then the process groups; a timer
        # bounds it -- the result line is already out, a stuck communicator teardown must not hang the launcher
        import threading
        killer = threading.Timer(30.0, lambda: os._exit(0))
        killer.daemon = True
        killer.start()
        hp.after_backward = None
        runner.close()
        dist.destroy_process_group()
        killer.cancel()


if __name__ == "__main__":
    main()
