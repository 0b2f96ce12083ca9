"""The per-step AttLoc kernels (re2e_attloc_step_fwd / re2e_attloc_step_bwd) and the helpers the per-step backward
calls (re2e_attloc_acc_reduce, re2e_attloc_enc_grad, re2e_attloc_init_att), called through the C ABI against an fp64
restatement of one step (fp32 of the same restatement as the reference, fp64 as the truth):

* every cluster size the launch geometry picks (1, 2, 4, 8, 16 per direction), grids that run in waves, a forward
  ring shorter than the frame range, one-CTA utterances and short last CTAs;
* every kernel instantiation (A / 64 x C == 10 or not x D == A or not);
* the forward's optional inputs and outputs and the mlp_dec paths, the backward's optional inputs and outputs, the
  d_pre store / accumulate modes and the accumulator-slot contract;
* AttLoc at batch sizes and lengths training produces, through the module and through forward_loop's per-step fallback.

The CPU test at the end checks the shapes the step kernels accept, without a device."""
import ctypes
import os
import sys

import pytest
import torch
import torch.nn.functional as F

from helpers import assert_close
from oracle import attloc as o_att
from oracle.gen_golden import make_attloc_inputs
from robust_e2e_gan_b200 import AttLoc, _lib
from test_gpu_attloc import run_loop, run_module, run_oracle, run_oracle_loop

gpu = pytest.mark.gpu
DEV = "cuda:0"
DEFAULT = (320, 320, 300, 10, 201)          # D, A, Z, C, K of the benchmarked model
E_WORKSPACE = -3


def step_geometry(B, Th, D, A, Z, C, K):
    """(forward cluster size, backward cluster size), 0 where a direction does not take the shape."""
    f, b = ctypes.c_int(-1), ctypes.c_int(-1)
    ok = _lib.load().re2e_attloc_step_supported(B, Th, D, A, Z, C, K, ctypes.byref(f), ctypes.byref(b))
    assert ok == (f.value > 0 and b.value > 0)
    return f.value, b.value


# ---------------------------------------------------------------------------------------------- fp64 restatement
def make_step(B, Th, D, A, Z, C, K, seed, with_dec_z=True):
    """fp64 inputs of one step on the device: a peaked previous alignment, parameters at the module's scale."""
    g = torch.Generator().manual_seed(seed)

    def r(*shape, scale=1.0):
        return torch.randn(*shape, generator=g, dtype=torch.float64) * scale

    t = dict(pre=r(B, Th, A, scale=0.7), enc=torch.tanh(r(B, Th, D)),
             dec_z=r(B, Z, scale=0.5) if with_dec_z else None,
             att_prev=torch.softmax(3.0 * r(B, Th), 1),
             W_dec=r(A, Z, scale=1.5 / Z ** 0.5), W_att=r(A, C, scale=1.5 / C ** 0.5),
             W_conv=r(C, K, scale=3.0 / K ** 0.5), gvec=r(A, scale=1.5 / A ** 0.5), gvec_b=r(1, scale=0.5),
             dc=r(B, D), dw=r(B, Th))
    return {k: None if v is None else v.to(DEV) for k, v in t.items()}


def reference(t, scaling, dt, use_dc=True, use_dw=True):
    """One AttLoc step (oracle/attloc.py:step) from its parts, with pre, dec_proj and att_prev as autograd leaves."""
    p = {k: None if v is None else v.detach().to(dt) for k, v in t.items()}
    B, Th, A = p["pre"].shape
    C, K = p["W_conv"].shape
    filts = (K - 1) // 2
    for k in ("pre", "att_prev", "W_att", "W_conv", "gvec", "gvec_b"):
        p[k].requires_grad_(True)
    dp = (p["dec_z"] @ p["W_dec"].t() if p["dec_z"] is not None else p["pre"].new_zeros(B, A)).requires_grad_(True)
    conv = F.pad(p["att_prev"], (filts, filts)).unfold(1, K, 1) @ p["W_conv"].t()      # (B,Th,C) = loc_conv
    x = torch.tanh(conv @ p["W_att"].t() + p["pre"] + dp[:, None, :])
    e = x @ p["gvec"] + p["gvec_b"]
    w = torch.softmax(scaling * e, 1)
    c = (p["enc"] * w[..., None]).sum(1)
    loss = 0.0
    if use_dc:
        loss = loss + (c * p["dc"]).sum()
    if use_dw:
        loss = loss + (w * p["dw"]).sum()
    loss.backward()
    return dict(c=c.detach(), w=w.detach(), conv=conv.detach(), xsave=x.detach(), dec_proj=dp.detach(),
                d_pre=p["pre"].grad, d_decproj=dp.grad, d_att_prev=p["att_prev"].grad, dW_att=p["W_att"].grad,
                dW_conv=p["W_conv"].grad, dgvec=p["gvec"].grad, dgvec_b=p["gvec_b"].grad,
                d_dec_z=dp.grad @ p["W_dec"])


def f32(x):
    return None if x is None else x.detach().float().contiguous()


def f32_all(t):
    """fp32 copies of every input, held by the caller until the kernel has read them (a temporary passed straight to
    _lib.ptr would be freed, and its memory reused, before the launch)."""
    return {k: f32(v) for k, v in t.items()}


def kernel_fwd(t, dims, scaling, dec_z=True, w_dec=None, outputs=True):
    """re2e_attloc_step_fwd; outputs=False passes NULL for every optional output."""
    B, Th, D, A, Z, C, K = dims
    c = torch.full((B, D), float("nan"), device=DEV)
    w = torch.full((B, Th), float("nan"), device=DEV)
    dec_proj = torch.full((B, A), float("nan"), device=DEV) if outputs else None
    conv = torch.full((B, Th, C), float("nan"), device=DEV) if outputs else None
    xsave = torch.full((B, Th, A), float("nan"), device=DEV) if outputs else None
    a = f32_all(t)
    W_dec = a["W_dec"] if w_dec is None else w_dec
    rc = _lib.lib().re2e_attloc_step_fwd(
        _lib.ptr(a["pre"]), _lib.ptr(a["enc"]), _lib.ptr(a["dec_z"] if dec_z else None),
        _lib.ptr(a["att_prev"]), _lib.ptr(W_dec), _lib.ptr(a["W_att"]), _lib.ptr(a["W_conv"]),
        _lib.ptr(a["gvec"]), _lib.ptr(a["gvec_b"]), float(scaling), _lib.ptr(c), _lib.ptr(w),
        _lib.ptr(dec_proj), _lib.ptr(conv), _lib.ptr(xsave), B, Th, D, A, Z, C, K, _lib.stream_ptr())
    assert rc == 0, _lib.load().re2e_error_string(rc)
    return dict(c=c, w=w, dec_proj=dec_proj, conv=conv, xsave=xsave)


def kernel_bwd(t, saved, dims, scaling, use_dc=True, use_dw=True, want_dec_z=True, want_att_prev=True,
               accumulate_pre=0, d_pre_init=None, extra_slots=0):
    """re2e_attloc_step_bwd from the fp64 forward's saved tensors (so the backward is checked on its own), then
    re2e_attloc_acc_reduce over every slot."""
    B, Th, D, A, Z, C, K = dims
    L = _lib.lib()
    n_min = L.re2e_attloc_acc_slots(B, Th, D, A, Z, C, K)
    assert n_min > 0, "acc_slots refused the shape (%d)" % n_min
    stride = int(L.re2e_attloc_acc_floats(A, C, K))
    acc = torch.zeros(n_min + extra_slots, stride, device=DEV)
    d_pre = d_pre_init.clone() if d_pre_init is not None else torch.full((B, Th, A), float("nan"), device=DEV)
    d_decproj = torch.full((B, A), float("nan"), device=DEV)
    d_dec_z = torch.full((B, Z), float("nan"), device=DEV) if want_dec_z else None
    d_prev = torch.full((B, Th), float("nan"), device=DEV) if want_att_prev else None
    a, sv = f32_all(t), f32_all({k: saved[k] for k in ("xsave", "w", "conv")})
    W_decT = a["W_dec"].t().contiguous()
    rc = L.re2e_attloc_step_bwd(
        _lib.ptr(a["dc"] if use_dc else None), _lib.ptr(a["dw"] if use_dw else None),
        _lib.ptr(sv["xsave"]), _lib.ptr(a["enc"]), _lib.ptr(a["att_prev"]), _lib.ptr(sv["w"]),
        _lib.ptr(sv["conv"]), _lib.ptr(a["W_dec"]), _lib.ptr(W_decT), _lib.ptr(a["W_att"]),
        _lib.ptr(a["W_conv"]), _lib.ptr(a["gvec"]), float(scaling), _lib.ptr(d_pre), accumulate_pre,
        _lib.ptr(d_decproj), _lib.ptr(d_dec_z), _lib.ptr(d_prev), _lib.ptr(acc), n_min + extra_slots,
        B, Th, D, A, Z, C, K, _lib.stream_ptr())
    assert rc == 0, L.re2e_error_string(rc)
    tot = torch.full((A * C + C * K + A + 1,), float("nan"), device=DEV)
    _lib.check(L.re2e_attloc_acc_reduce(_lib.ptr(acc), n_min + extra_slots, _lib.ptr(tot), A, C, K, _lib.stream_ptr()),
               "re2e_attloc_acc_reduce")
    return dict(d_pre=d_pre, d_decproj=d_decproj, d_dec_z=d_dec_z, d_att_prev=d_prev, dW_att=tot[:A * C].view(A, C),
                dW_conv=tot[A * C:A * C + C * K].view(C, K), dgvec=tot[A * C + C * K:A * C + C * K + A],
                dgvec_b=tot[A * C + C * K + A:], acc=acc, n_min=n_min)


def compare(got, r32, r64, keys, tag):
    for k in keys:
        assert_close(got[k], r32[k], truth=r64[k], what="%s %s" % (tag, k))


BWD_KEYS = ("d_pre", "d_decproj", "d_dec_z", "d_att_prev", "dW_att", "dW_conv", "dgvec")


def check_step(dims, seed, scaling=2.0, fwd=True, bwd=True):
    """Forward and backward of one step against the fp64 restatement; returns the kernel results."""
    t = make_step(*dims, seed)
    r32, r64 = reference(t, scaling, torch.float32), reference(t, scaling, torch.float64)
    out = {}
    if fwd:
        out = kernel_fwd(t, dims, scaling)
        compare(out, r32, r64, ("c", "w", "dec_proj", "conv", "xsave"), "fwd")
        assert torch.allclose(out["w"].sum(1), torch.ones(dims[0], device=DEV), atol=1e-5)
    if bwd:
        g = kernel_bwd(t, r64, dims, scaling)
        compare(g, r32, r64, BWD_KEYS, "bwd")
        # d gvec.bias is analytically zero (softmax is shift invariant): no scale of its own to compare to
        assert float(g["dgvec_b"].abs().max()) < 1e-4 * float(r64["dgvec"].abs().max())
        out.update(g)
    return out


# ---------------------------------------------------------------------------------------------- a. cluster geometry
GEOMETRY = [
    # B, Th, forward CL, backward CL
    (1, 5, 1, 1),          # Th < 8: one CTA per utterance, B = 1
    (96, 50, 1, 1),        # clusters of 1; mlp_dec slice of 320 channels (several kCPW passes)
    (74, 100, 2, 2),
    (75, 100, 1, 2),       # refused by the backward before clusters could run in waves
    (38, 200, 2, 4),       # refused before: 38 utterances at the bench's Th
    (32, 200, 4, 4),       # the bench shape
    (8, 100, 8, 8),
    (1, 163, 8, 8),        # Th % 8 != 0: the last CTA's range is short
    (32, 357, 4, 8),       # refused before; 256 backward CTAs run in waves
    (96, 600, 2, 8),       # refused before; 768 backward CTAs
    (2, 700, 8, 16),
    (16, 641, 8, 16),      # refused before; 256 CTAs in clusters of 16, short last CTA
    (128, 1000, 2, 16),    # corner of the supported envelope
]


@gpu
@pytest.mark.parametrize("B,Th,cl_fwd,cl_bwd", GEOMETRY)
def test_step_cluster_geometry(B, Th, cl_fwd, cl_bwd):
    dims = (B, Th) + DEFAULT
    check_step(dims, seed=B * 1000 + Th)
    assert _lib.lib().re2e_attloc_acc_slots(*dims) // B == cl_bwd
    assert step_geometry(*dims) == (cl_fwd, cl_bwd)


@gpu
def test_step_forward_cluster_of_16_with_wrapping_ring():
    """Beyond the backward's range (Th > 1032) the forward alone still runs: clusters of 16, 263 frames per CTA, i.e.
    33 eight-frame chunks through a ring of at most 30 stages."""
    dims = (2, 4200) + DEFAULT
    assert step_geometry(*dims) == (16, 0)
    check_step(dims, seed=4200, bwd=False)


# ---------------------------------------------------------------------------------------------- b. instantiations
D_OTHER = {64: 132, 128: 100, 256: 500, 320: 36, 512: 260}
C_OTHER = {1: 3, 2: 7, 4: 16, 5: 3, 8: 7}
INSTANTIATIONS = [(apl, c10, same_d) for apl in (1, 2, 4, 5, 8) for c10 in (True, False) for same_d in (True, False)]


@gpu
@pytest.mark.parametrize("apl,c10,same_d", INSTANTIATIONS)
def test_step_every_instantiation(apl, c10, same_d):
    A = 64 * apl
    D = A if same_d else D_OTHER[A]
    C = 10 if c10 else C_OTHER[apl]
    K = 31 if apl % 2 else 201
    Z = 96 + 52 * apl
    B, Th = (3, 45) if apl < 8 else (2, 37)
    check_step((B, Th, D, A, Z, C, K), seed=apl * 10 + 2 * c10 + same_d)


# ---------------------------------------------------------------------------------------------- c. forward options
@gpu
@pytest.mark.parametrize("Z,offset,dec_z,scaling", [
    (301, False, True, 2.0),      # Z % 4 != 0: scalar mlp_dec
    (300, True, True, 2.0),       # W_dec one float off 16 B alignment: scalar mlp_dec
    (700, False, True, 2.0),      # Z > 384: several kZQ passes of the vector mlp_dec
    (700, True, True, 1.3),       # the same on the scalar path, scaling != 2
    (300, False, False, 0.5),     # dec_z = NULL (zeros)
])
def test_step_forward_options(Z, offset, dec_z, scaling):
    B, Th, D, A, C, K = 5, 70, 320, 320, 10, 201
    dims = (B, Th, D, A, Z, C, K)
    t = make_step(*dims, seed=Z + 7 * offset + 3 * dec_z, with_dec_z=dec_z)
    r32, r64 = reference(t, scaling, torch.float32), reference(t, scaling, torch.float64)
    w_dec = None
    if offset:
        buf = torch.empty(A * Z + 1, device=DEV)
        buf[1:] = t["W_dec"].float().reshape(-1)
        w_dec = buf[1:]
    got = kernel_fwd(t, dims, scaling, dec_z=dec_z, w_dec=w_dec)
    compare(got, r32, r64, ("c", "w", "conv", "xsave"), "fwd")
    if dec_z:
        compare(got, r32, r64, ("dec_proj",), "fwd")
    # the outputs do not depend on the optional ones being requested
    lean = kernel_fwd(t, dims, scaling, dec_z=dec_z, w_dec=w_dec, outputs=False)
    assert torch.equal(lean["c"], got["c"]) and torch.equal(lean["w"], got["w"])
    g = kernel_bwd(t, r64, dims, scaling)
    compare(g, r32, r64, BWD_KEYS, "bwd")


@gpu
def test_step_forward_mlp_dec_slices_over_a_cluster():
    """A / CL > 80 (several kCPW passes per CTA) together with the DSMEM exchange of the slices (CL = 2)."""
    dims = (74, 60, 512, 512, 300, 10, 201)
    assert step_geometry(*dims)[0] == 2
    check_step(dims, seed=74)


# ---------------------------------------------------------------------------------------------- d. backward options
BWD_CASES = dict(
    no_dc=dict(use_dc=False),
    no_dw=dict(use_dw=False),
    no_dec_z_no_att_prev=dict(want_dec_z=False, want_att_prev=False),
    extra_slots=dict(extra_slots=37),
)


@gpu
@pytest.mark.parametrize("case", sorted(BWD_CASES))
@pytest.mark.parametrize("B,Th", [(4, 90), (40, 200)])
def test_step_backward_options(case, B, Th):
    opt = BWD_CASES[case]
    dims = (B, Th) + DEFAULT
    t = make_step(*dims, seed=len(case) + B)
    use_dc, use_dw = opt.get("use_dc", True), opt.get("use_dw", True)
    r32 = reference(t, 2.0, torch.float32, use_dc, use_dw)
    r64 = reference(t, 2.0, torch.float64, use_dc, use_dw)
    g = kernel_bwd(t, r64, dims, 2.0, **opt)
    keys = [k for k in BWD_KEYS if g[k] is not None]
    compare(g, r32, r64, keys, "bwd " + case)
    assert g["d_dec_z"] is None or torch.isfinite(g["d_dec_z"]).all()
    if opt.get("extra_slots"):
        assert torch.count_nonzero(g["acc"][g["n_min"]:]) == 0, "slots beyond one per CTA must stay untouched"


@gpu
@pytest.mark.parametrize("B,Th", [(4, 90), (40, 200), (16, 641)])
def test_step_backward_d_pre_store_and_accumulate(B, Th):
    """accumulate_pre = 0 stores over a NaN-filled d_pre; accumulate_pre = 1 adds onto what is there."""
    dims = (B, Th) + DEFAULT
    t = make_step(*dims, seed=B + Th)
    r32, r64 = reference(t, 2.0, torch.float32), reference(t, 2.0, torch.float64)
    stored = kernel_bwd(t, r64, dims, 2.0, accumulate_pre=0)
    assert torch.isfinite(stored["d_pre"]).all()
    assert_close(stored["d_pre"], r32["d_pre"], truth=r64["d_pre"], what="d_pre (store)")
    base = torch.randn(B, Th, dims[3], device=DEV, dtype=torch.float64,
                       generator=torch.Generator(device=DEV).manual_seed(Th))
    added = kernel_bwd(t, r64, dims, 2.0, accumulate_pre=1, d_pre_init=base.float())
    assert_close(added["d_pre"], base.float() + r32["d_pre"], truth=base + r64["d_pre"], what="d_pre (accumulate)")


@gpu
def test_step_backward_too_few_slots_is_refused_before_launch():
    dims = (40, 200) + DEFAULT
    B, Th, D, A, Z, C, K = dims
    L = _lib.lib()
    t = make_step(*dims, seed=5)
    n_min = L.re2e_attloc_acc_slots(*dims)
    stride = int(L.re2e_attloc_acc_floats(A, C, K))
    acc = torch.zeros(n_min, stride, device=DEV)
    d_pre = torch.zeros(B, Th, A, device=DEV)
    d_decproj = torch.zeros(B, A, device=DEV)
    a = f32_all(t)
    conv = torch.zeros(B, Th, C, device=DEV)
    W_decT = a["W_dec"].t().contiguous()
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    rc = L.re2e_attloc_step_bwd(
        _lib.ptr(a["dc"]), _lib.ptr(a["dw"]), _lib.ptr(a["pre"]), _lib.ptr(a["enc"]),
        _lib.ptr(a["att_prev"]), _lib.ptr(a["att_prev"]), _lib.ptr(conv),
        _lib.ptr(a["W_dec"]), _lib.ptr(W_decT), _lib.ptr(a["W_att"]), _lib.ptr(a["W_conv"]),
        _lib.ptr(a["gvec"]), 2.0, _lib.ptr(d_pre), 0, _lib.ptr(d_decproj), None, None, _lib.ptr(acc), n_min - 1,
        B, Th, D, A, Z, C, K, _lib.stream_ptr())
    torch.cuda.synchronize()
    assert rc == E_WORKSPACE
    assert _lib.launch_count() == n0
    assert torch.count_nonzero(d_pre) == 0 and torch.count_nonzero(acc) == 0 and torch.count_nonzero(d_decproj) == 0


# ---------------------------------------------------------------------------------------------- e. helpers
@gpu
@pytest.mark.parametrize("accumulate", [0, 1])
@pytest.mark.parametrize("D", [320, 512, 38])
@pytest.mark.parametrize("steps", [1, 41, 145, 146, 300])
def test_enc_grad_matches_fp64(steps, D, accumulate):
    """d_enc[b,t,:] (+)= sum_i w_all[i,b,t] dc_all[i,b,:]; D = 38 stages dc with scalar loads, Th = 77 leaves a short
    last tile of frames, and more steps than fit in shared memory at once (146 at D = 320, 95 at D = 512) run as
    several launches."""
    B, Th = 3, 77
    g = torch.Generator(device=DEV).manual_seed(steps * 7 + D + accumulate)
    w_all = torch.softmax(2.0 * torch.randn(steps, B, Th, device=DEV, dtype=torch.float64, generator=g), -1)
    dc_all = torch.randn(steps, B, D, device=DEV, dtype=torch.float64, generator=g)
    base = torch.randn(B, Th, D, device=DEV, dtype=torch.float64, generator=g)
    out = base.float() if accumulate else torch.full((B, Th, D), float("nan"), device=DEV)
    w32, dc32 = f32(w_all), f32(dc_all)
    _lib.check(_lib.lib().re2e_attloc_enc_grad(_lib.ptr(w32), _lib.ptr(dc32), _lib.ptr(out), steps, B, Th, D,
                                               accumulate, _lib.stream_ptr()), "re2e_attloc_enc_grad")
    ref32 = torch.einsum("sbt,sbd->btd", w32, dc32) + (base.float() if accumulate else 0.0)
    ref64 = torch.einsum("sbt,sbd->btd", w32.double(), dc32.double()) + (base.float().double() if accumulate else 0.0)
    assert_close(out, ref32, truth=ref64, what="d enc (steps %d, D %d)" % (steps, D))


@gpu
@pytest.mark.parametrize("B,slots_per_utt", [(1, 1), (3, 16), (40, 16)])
def test_acc_reduce_matches_fp64(B, slots_per_utt):
    A, C, K = 320, 10, 201
    L = _lib.lib()
    stride = int(L.re2e_attloc_acc_floats(A, C, K))
    n = B * slots_per_utt
    n_out = A * C + C * K + A + 1
    slots = torch.randn(n, stride, device=DEV, dtype=torch.float64, generator=torch.Generator(device=DEV).manual_seed(n))
    out = torch.full((n_out,), float("nan"), device=DEV)
    s32 = f32(slots)
    _lib.check(L.re2e_attloc_acc_reduce(_lib.ptr(s32), n, _lib.ptr(out), A, C, K, _lib.stream_ptr()),
               "re2e_attloc_acc_reduce")
    s32 = s32[:, :n_out]
    assert_close(out, s32.sum(0), truth=s32.double().sum(0), what="acc_reduce (%d slots)" % n)


@gpu
@pytest.mark.parametrize("B,Th,short", [(1, 1, False), (5, 37, False), (5, 37, True), (96, 600, True)])
def test_init_att_matches_uniform_att_prev(B, Th, short):
    hl = [Th] * B if not short else [max(1, Th - 3 * b) for b in range(B)]
    hl_d = torch.tensor(hl, dtype=torch.int32, device=DEV)
    out = torch.full((B, Th), float("nan"), device=DEV)
    _lib.check(_lib.lib().re2e_attloc_init_att(_lib.ptr(hl_d), _lib.ptr(out), B, Th, _lib.stream_ptr()),
               "re2e_attloc_init_att")
    ref = o_att.uniform_att_prev(torch.zeros(B, Th, 1, dtype=torch.float64), hl)
    assert torch.equal(out.cpu(), ref.float())


# ---------------------------------------------------------------------------------------------- f. module level
MODULE_DIMS = (320, 300, 320, 10, 100)      # eprojs, dunits, att_dim, aconv_chans, aconv_filts


@gpu
@pytest.mark.parametrize("B,Th,steps", [(40, 200, 5), (32, 400, 3), (96, 600, 2), (2, 60, 160)])
def test_module_at_training_shapes(B, Th, steps):
    """AttLoc through several steps with the alignment fed back, backward into every parameter and enc_h, at shapes
    the step kernels refused before (B = 2 x 160 steps: d enc_h over more decoder steps than one enc_grad launch takes)."""
    params, enc, hlens, zs, gc, gw = make_attloc_inputs(*MODULE_DIMS, B, Th, steps, B + Th)
    got = run_module(MODULE_DIMS, params, enc, hlens, zs, gc, gw)
    r32 = run_oracle(params, enc, hlens, zs, gc, gw, torch.float32)
    r64 = run_oracle(params, enc, hlens, zs, gc, gw, torch.float64)
    assert_close(torch.stack(got[0]), torch.stack(r32[0]), truth=torch.stack(r64[0]), what="c")
    assert_close(torch.stack(got[1]), torch.stack(r32[1]), truth=torch.stack(r64[1]), what="w")
    assert_close(got[2], r32[2], truth=r64[2], what="d enc")
    assert_close(torch.stack(got[3]), torch.stack(r32[3]), truth=torch.stack(r64[3]), what="d dec_z")
    for k in r32[4]:
        if k == "gvec.bias":
            assert float(got[4][k].abs().max()) < 1e-4 * float(r32[4]["gvec.weight"].abs().max())
            continue
        assert_close(got[4][k], r32[4][k], truth=r64[4][k], what="d " + k)


@gpu
def test_forward_loop_falls_back_per_step_at_large_batch():
    B, Th, steps = 40, 200, 5
    params, enc, hlens, zs, gc, gw = make_attloc_inputs(*MODULE_DIMS, B, Th, steps, 41)
    g = torch.Generator().manual_seed(42)
    gw_all = torch.randn(steps, B, Th, generator=g) / B ** 0.5
    gw_all[-1] = gw
    assert not AttLoc(*MODULE_DIMS, "softmax").loop_supported(steps, B, Th)
    got = run_loop(MODULE_DIMS, params, enc, hlens, zs, gc, gw_all)
    r32 = run_oracle_loop(params, enc, hlens, zs, gc, gw_all, torch.float32)
    r64 = run_oracle_loop(params, enc, hlens, zs, gc, gw_all, torch.float64)
    for i, what in enumerate(("c_all", "w_all", "d enc", "d dec_z")):
        assert_close(got[i], r32[i], truth=r64[i], what=what + " (fallback)")
    for k in r32[4]:
        if k != "gvec.bias":
            assert_close(got[4][k], r32[4][k], truth=r64[4][k], what="d " + k + " (fallback)")


# ---------------------------------------------------------------------------------------------- g. determinism
@gpu
def test_replays_identically_when_the_grid_runs_in_waves():
    """B = 96, Th = 600: 768 backward CTAs in clusters of 8, more than the GPU holds at once.  Two runs of the step
    kernels are bit-identical, and so are two runs of the module -- but for d mlp_enc.weight, a product over
    B*Th = 57600 rows that the dense GEMM splits along K and sums with atomics."""
    B, Th, steps = 96, 600, 2
    dims = (B, Th) + DEFAULT
    assert _lib.lib().re2e_attloc_acc_slots(*dims) > torch.cuda.get_device_properties(0).multi_processor_count
    t = make_step(*dims, seed=96)
    saved = reference(t, 2.0, torch.float64)
    runs = [dict(kernel_fwd(t, dims, 2.0), **kernel_bwd(t, saved, dims, 2.0)) for _ in range(2)]
    for k, v in runs[0].items():
        if torch.is_tensor(v):
            assert torch.equal(v, runs[1][k]), k
    params, enc, hlens, zs, gc, gw = make_attloc_inputs(*MODULE_DIMS, B, Th, steps, 96)
    a = run_module(MODULE_DIMS, params, enc, hlens, zs, gc, gw)
    b = run_module(MODULE_DIMS, params, enc, hlens, zs, gc, gw)
    for i in (0, 1, 3):
        for x, y in zip(a[i], b[i]):
            assert torch.equal(x, y)
    assert torch.equal(a[2], b[2])
    for k in a[4]:
        if k != "mlp_enc.weight":
            assert torch.equal(a[4][k], b[4][k]), k


# ---------------------------------------------------------------------------------------------- 3. envelope (CPU)
@pytest.fixture(scope="module")
def built():
    if not os.path.exists(_lib.LIB_PATH):
        sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
        import __graft_entry__
        __graft_entry__.build()
    return _lib.load()


def test_step_kernels_accept_the_supported_envelope(built):
    """Every B in 1..128 with Th in 1..1000 at the default dims, Th <= 512 at D = A = 512, in both directions; the
    shapes training produces that were refused before; and unchanged launch geometry for the shapes accepted before
    (the bench shape among them).  Without a device the SM count is taken as the B200's 148."""
    refused = [(B, Th) for B in range(1, 129) for Th in range(1, 1001) if 0 in step_geometry(B, Th, *DEFAULT)]
    assert not refused, refused[:10]
    for Z in (300, 1024):
        refused = [(B, Th) for B in range(1, 129) for Th in range(1, 513)
                   if 0 in step_geometry(B, Th, 512, 512, Z, 10, 201)]
        assert not refused, (Z, refused[:10])
    for B, Th in [(32, 200), (32, 356), (32, 357), (37, 200), (38, 200), (74, 100), (75, 100), (16, 641)]:
        assert built.re2e_attloc_acc_slots(B, Th, *DEFAULT) >= 0, (B, Th)
    for B, Th, slots in [(32, 200, 128), (8, 100, 64), (1, 163, 8), (2, 700, 32), (64, 100, 128), (74, 100, 148),
                         (96, 50, 96)]:
        assert built.re2e_attloc_acc_slots(B, Th, *DEFAULT) == slots, (B, Th)
    assert built.re2e_attloc_acc_slots(5, 19, 64, 128, 40, 7, 7) == 10
    assert step_geometry(32, 200, *DEFAULT) == (4, 4)            # the bench shape
    assert step_geometry(96, 50, *DEFAULT) == (1, 1)
    # outside the envelope: refused by both the query and the backward's slot count (the backward's frame range no
    # longer fits on chip at clusters of 16)
    for Th in (1033, 1200):
        assert step_geometry(8, Th, *DEFAULT)[1] == 0
        assert built.re2e_attloc_acc_slots(8, Th, *DEFAULT) == -2
    assert step_geometry(4, 100, 320, 320, 300, 17, 201) == (0, 0)      # C > 16
