"""Device time of the decoder's per-position products: re2e_batch_nt against the dense GEMM."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
from robust_e2e_gan_b200 import _lib
from robust_e2e_gan_b200.linear import gemm_tf32x3
dev = torch.device("cuda:0")
L = _lib.lib()
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)


def timeit(fn, n=20):
    for _ in range(3):
        fn()
    ts = []
    for _ in range(n):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    ts.sort()
    return ts[len(ts) // 2]


def timeit_warm(fn, n=50):
    for _ in range(3):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / n



def graph_time(fn, n=40):
    """Per-launch device time from a replayed CUDA graph of n back-to-back launches (no host launch cost)."""
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=st, capture_error_mode="thread_local"):
            for _ in range(n):
                fn()
        g.replay(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); g.replay(); e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / n


sp = lambda: _lib.stream_ptr()
for M, N, K in [(32, 1200, 320), (32, 1200, 300), (32, 320, 1200), (32, 300, 1200)]:
    X, W, O = torch.randn(M, K, device=dev), torch.randn(N, K, device=dev), torch.zeros(M, N, device=dev)
    WT = W.t().contiguous()
    row = {"shape": (M, N, K),
           "batch_nt": graph_time(lambda: L.re2e_batch_nt(_lib.ptr(X), _lib.ptr(W), None, _lib.ptr(O), M, N, K, 0, sp())),
           "gemm": graph_time(lambda: gemm_tf32x3(X, False, WT, True, O, M, N, K))}
    print({k: (round(v, 2) if isinstance(v, float) else v) for k, v in row.items()}, flush=True)

B, D, Z = 32, 320, 300
xc, hp, cp = torch.randn(B, D, device=dev), torch.randn(B, Z, device=dev), torch.randn(B, Z, device=dev)
Wcat = torch.randn(4 * Z, D + Z, device=dev) * 0.05
WcatT = Wcat.t().contiguous()
eg, act = torch.randn(B, 4 * Z, device=dev), torch.empty(B, 4 * Z, device=dev)
c, h = torch.empty(B, Z, device=dev), torch.empty(B, Z, device=dev)
dg, dctx, dhp, dcp = torch.randn(B, 4 * Z, device=dev), torch.empty(B, D, device=dev), torch.empty(B, Z, device=dev), torch.empty(B, Z, device=dev)
print({"lstm_step_fwd": round(graph_time(lambda: L.re2e_lstm_step_fwd(
    _lib.ptr(xc), _lib.ptr(hp), _lib.ptr(cp), _lib.ptr(Wcat), _lib.ptr(eg), None, _lib.ptr(act), _lib.ptr(c), _lib.ptr(h), B, D, Z, sp())), 2),
    "lstm_step_bwd": round(graph_time(lambda: L.re2e_lstm_step_bwd(
        _lib.ptr(dg), _lib.ptr(WcatT), _lib.ptr(dctx), _lib.ptr(dhp), B, D, Z, sp())), 2),
    "pointwise_fwd": round(graph_time(lambda: L.re2e_lstm_pointwise_fwd(
        _lib.ptr(act), _lib.ptr(eg), _lib.ptr(cp), _lib.ptr(c), _lib.ptr(h), B, Z, sp())), 2),
    "pointwise_bwd": round(graph_time(lambda: L.re2e_lstm_pointwise_bwd(
        _lib.ptr(act), _lib.ptr(cp), _lib.ptr(c), _lib.ptr(h), _lib.ptr(c), _lib.ptr(dg), _lib.ptr(dcp), B, Z, sp())), 2)})

# ---- the beam-search position (W = 10 rows, V = 4233, Th = 137), kernel by kernel
import ctypes
from robust_e2e_gan_b200 import AttLoc
W, V, Th, Cb, beam, A, C, K = 10, 4233, 137, 15, 10, 320, 10, 201
torch.manual_seed(0)
att = AttLoc(D, Z, A, C, 100, "softmax").to(dev)
hb = torch.tanh(torch.randn(1, Th, D, device=dev)).expand(W, Th, D).contiguous()
with torch.no_grad():
    st = att.precompute(hb)
W_dec, W_att, W_conv, gvec, gvec_b = st.weights
K = st.dims[6]
P = _lib.ptr
z_in, c_in, a_in = torch.randn(W, Z, device=dev), torch.randn(W, Z, device=dev), torch.softmax(torch.randn(W, Th, device=dev), 1)
z_st, c_st, a_st, att_c = torch.empty(W, Z, device=dev), torch.empty(W, Z, device=dev), torch.empty(W, Th, device=dev), torch.empty(W, D, device=dev)
EG = torch.randn(V, 4 * Z, device=dev) * 0.1
tok = torch.randint(0, V, (W,), device=dev).int()
pos = torch.full((W,), 20, device=dev).int()
w_out, b_out, logits = torch.randn(V, Z, device=dev) * 0.05, torch.randn(V, device=dev), torch.empty(W, V, device=dev)
top_v, top_i = torch.empty(W, Cb, device=dev), torch.empty(W, Cb, dtype=torch.int32, device=dev)
lpz = torch.log_softmax(torch.randn(Th, V, device=dev), 1)
r_st, r_in = torch.randn(W, Cb, Th, 2, device=dev) - 30, torch.randn(W, Th, 2, device=dev) - 30
psi_st, psi_in, scr, outb = torch.randn(W, Cb, device=dev), torch.randn(W, device=dev), torch.randn(W, device=dev), torch.empty(3, W, beam, device=dev)
parent, cand = torch.randint(0, W, (W,), device=dev).int(), torch.randint(0, Cb, (W,), device=dev).int()
segs = [(z_in, z_st, Z, 0), (c_in, c_st, Z, 0), (a_in, a_st, Th, 0), (r_st, r_in, 2 * Th, Cb), (psi_st, psi_in, 1, Cb)]
n = len(segs)
src = (ctypes.c_void_p * n)(*[s[0].data_ptr() for s in segs]); dst = (ctypes.c_void_p * n)(*[s[1].data_ptr() for s in segs])
rowf = (ctypes.c_int * n)(*[s[2] for s in segs]); subc = (ctypes.c_int * n)(*[s[3] for s in segs])
steps = {
    "beam_gather": lambda: L.re2e_beam_gather(P(parent), P(cand), W, n, src, dst, rowf, subc, sp()),
    "attloc_step_fwd": lambda: L.re2e_attloc_step_fwd(P(st.pre), P(st.enc), P(z_in), P(a_in), P(W_dec), P(W_att), P(W_conv), P(gvec), P(gvec_b), 2.0, P(att_c), P(a_st), None, None, None, W, Th, D, A, Z, C, K, sp()),
    "lstm_step_fwd": lambda: L.re2e_lstm_step_fwd(P(att_c), P(z_in), P(c_in), P(Wcat), P(EG), P(tok), P(act[:W]), P(c_st), P(z_st), W, D, Z, sp()),
    "batch_nt(out)": lambda: L.re2e_batch_nt(P(z_st), P(w_out), P(b_out), P(logits), W, V, Z, 0, sp()),
    "log_softmax_topk": lambda: L.re2e_log_softmax_topk(P(logits), W, V, Cb, None, P(top_v), P(top_i), sp()),
    "ctc_prefix": lambda: L.re2e_ctc_prefix_score(P(lpz), P(r_in), P(top_i), P(tok), P(pos), P(psi_st), P(r_st), Th, V, W, Cb, 0, V - 1, sp()),
    "beam_joint": lambda: L.re2e_beam_joint(P(top_v), P(top_i), P(psi_st), P(psi_in), P(scr), 0.7, 0.3, W, Cb, beam, P(outb), sp()),
}
state = torch.tensor([10, 20], dtype=torch.int32, device=dev)
ctlb = torch.zeros(4, W, dtype=torch.int32, device=dev)
histb = torch.empty(256, 4, beam, device=dev)


def advance():
    state.fill_(10)      # (keeps the search alive; one tiny fill kernel inside the timed graph)
    L.re2e_beam_advance(P(top_v), P(top_i), P(psi_st), P(psi_in), P(scr), 0.7, 0.3, W, Cb, beam, P(state), P(ctlb), P(histb),
                        V - 1, 100000, n, src, dst, rowf, subc, sp())


res = {k: round(graph_time(f), 2) for k, f in steps.items()}
res["beam_advance(+fill)"] = round(graph_time(advance), 2)


def whole():
    for f in steps.values():
        f()


res["position (7 launches)"] = round(graph_time(whole, n=20), 2)
print(res)
