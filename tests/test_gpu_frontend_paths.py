"""GPU: every front-end kernel path against the oracle (oracle/frontend.py), forward and backward.

Each case is built to reach one path of the host dispatch -- banded streaming kernels (csrc/fbank_band.cu), tcgen05
kernels (csrc/fbank_tc.cu), SIMT fallbacks and the trainable-bank gradient (csrc/fbank.cu), picked by
re2e_fbank_fwd / _bwd and by feat_model.py -- and checks from a torch.profiler trace that the kernels it was built for
are the ones that ran, so that a change in the dispatch cannot quietly move a case onto another path.

Outputs are compared with the fp32 oracle at the project tolerance (1e-4, max-norm and element-wise), the fp64 oracle
breaking ties (helpers.assert_close).  The bank gradient dfc is summed with atomics, so it is compared within that
tolerance, never bit for bit.  Inputs keep P = x^2 @ fc either exactly 0 (all-zero or padded frames) or far above the
1e-7 clamp, where two correct fp32 evaluations cannot disagree on the clamp.

The SIMT forward for M <= 48 (fbank_fwd_kernel<2>) has no case: for every F its shared-memory tile is larger than the
tcgen05 forward's, so whenever the tcgen05 forward does not fit, neither does it.
"""
import re

import numpy as np
import pytest
import torch

from helpers import assert_close
from oracle import frontend as o_fe
from robust_e2e_gan_b200 import FbankModel, _lib, apply_mask, fbank, masked_fbank, synth
from robust_e2e_gan_b200 import feat_model as fm

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
E_UNSUPPORTED = -2
FAMILIES = ("fbank_band_fwd_kernel", "fbank_band_bwd_kernel", "fbank_tc_fwd_kernel", "fbank_tc_bwd_kernel",
            "fbank_fwd_kernel", "fbank_bwd_kernel", "fbank_dfc_kernel", "mask_apply_kernel", "cmvn_stats_kernel")
BAND_FWD, BAND_BWD = "fbank_band_fwd_kernel", "fbank_band_bwd_kernel"
TC_FWD, TC_BWD = "fbank_tc_fwd_kernel", "fbank_tc_bwd_kernel"
SIMT_FWD, SIMT_BWD, DFC = "fbank_fwd_kernel", "fbank_bwd_kernel", "fbank_dfc_kernel"


class Args:
    def __init__(self, **kw):
        self.__dict__.update(dict(idim=257, fbank_dim=80, enhance_type="blstm", fbank_opti_type="frozen",
                                  train_dataset_len=1000, num_utt_cmvn=100))
        self.__dict__.update(kw)


# ---- which kernels ran -----------------------------------------------------------------------------------------------
def _template_args(name, family):
    """Template arguments of a kernel name, demangled ('<true, 2, 257, false>', '<(bool)1, (int)2, ...>') or mangled
    ('ILb1ELi2E...E'), as strings: 'true' / 'false' / decimal."""
    m = re.search(re.escape(family) + r"<([^>]*)>", name)
    if m:
        out = []
        for a in m.group(1).split(","):
            a = a.strip().replace("(int)", "")
            out.append({"(bool)1": "true", "(bool)0": "false"}.get(a, a))
        return out
    m = re.search(re.escape(family) + r"I((?:L[bi]\d+E)+)E", name)
    if m:
        return [("true" if v == "1" else "false") if t == "b" else v for t, v in re.findall(r"L([bi])(\d+)E", m.group(1))]
    return []


class Kernels(object):
    """``with Kernels() as k:`` records the kernels that ran inside the block (torch.profiler, CUDA activities).
    ``k.families``: the front-end kernel families among them; ``k.variants(family)``: their template arguments."""

    def __enter__(self):
        torch.cuda.synchronize()
        self._prof = torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA])
        self._prof.__enter__()
        return self

    def __exit__(self, *exc):
        torch.cuda.synchronize()
        self._prof.__exit__(*exc)
        if exc[0] is not None:
            return False
        names = []
        for e in self._prof.events():
            names.append(e.name)
            names.extend(k.name for k in getattr(e, "kernels", []))
        self.names = [n for n in names if any(f in n for f in FAMILIES)]
        self.families = {f for n in self.names for f in FAMILIES if f in n}
        return False

    def variants(self, family):
        return {tuple(_template_args(n, family)) for n in self.names if family in n}

    def expect(self, *families):
        assert self.families == set(families), "expected kernels %s, ran %s" % (sorted(families), sorted(self.families))


def tc_fwd_kind(k):
    """'pair' (F = 257, 8 B aligned inputs), '257' (F = 257 otherwise) or '0' (any other F) per tcgen05 forward."""
    return {("pair" if a[3] == "true" else a[2]) for a in k.variants(TC_FWD)}


# ---- inputs ------------------------------------------------------------------------------------------------------------
def dense_bank(F, M, seed):
    """A bank with every entry > 0: no banded structure, so the dense kernels run it."""
    g = torch.Generator().manual_seed(seed)
    return 0.05 + torch.rand(F, M, generator=g)


def ref_bank80():
    return torch.from_numpy(fm.reference_fbank80().T.astype(np.float32)).contiguous()


def batch(B, T, F=257, seed=1, lens=None, zeros=16):
    d = synth.frontend_batch(B=B, T=T, F=F, seed=seed, zeros=min(zeros, B * T))
    if lens is not None:
        d["lens"] = torch.tensor(lens, dtype=torch.int32)
        for b, n in enumerate(lens):
            d["mix"][b, n:] = 0
            d["clean"][b, n:] = 0
    return d


def on_dev(t, offset=0):
    """``t`` on the GPU, its storage starting ``offset`` floats past a 16 B aligned address (a contiguous view)."""
    if not offset:
        return t.to(DEV)
    buf = torch.zeros(t.numel() + offset, device=DEV, dtype=t.dtype)
    v = buf[offset:].view(t.shape)
    v.copy_(t)
    assert v.data_ptr() % 16 == 4 * offset
    return v


def oracle(x, fc, dY, mix=None, lens=None, cm=None, mask_is_logit=True, want_dfc=False):
    """fp32 and fp64 oracle: {dtype: (Y, dY/dx, dfc)}.  ``mix`` given: x is the mask (masked form), else the input."""
    outs = {}
    for dt in (torch.float32, torch.float64):
        xx = x.detach().clone().to(dt).requires_grad_(True)
        f = fc.detach().cpu().to(dt).requires_grad_(want_dfc)
        c = None if cm is None else cm.cpu().to(dt)
        if mix is None:
            y = o_fe.fbank_forward(xx, f, c)
        else:
            y = o_fe.masked_fbank_forward(xx, mix.to(dt), lens, f, c, mask_is_logit)
        y.backward(dY.to(dt))
        outs[dt] = (y.detach(), xx.grad, f.grad)
    return outs


def compare(ref, y, dx, dfc=None, what=""):
    r32, r64 = ref[torch.float32], ref[torch.float64]
    assert_close(y, r32[0], truth=r64[0], what="Y " + what)
    assert_close(dx, r32[1], truth=r64[1], what="d in " + what)
    if dfc is not None:
        assert_close(dfc, r32[2], truth=r64[2], what="dfc " + what)


def run(x, fc, dY, mix=None, lens=None, cm=None, mask_is_logit=True, want_dfc=False, offset=0):
    """The library's front-end forward + backward on the GPU.  Returns (Y, dx, dfc, forward kernels, backward kernels).
    ``offset``: x and mix are placed ``offset`` floats off 16 B alignment."""
    f = fc.detach().to(DEV).clone().requires_grad_(want_dfc)
    xd = on_dev(x, offset).requires_grad_(True)
    c = None if cm is None else cm.to(DEV)
    with Kernels() as kf:
        if mix is None:
            y = fbank(xd, f, c)
        else:
            y = masked_fbank(xd, on_dev(mix, offset), lens, f, c, mask_is_logit=mask_is_logit)
    with Kernels() as kb:
        y.backward(dY.to(DEV))
    return y, xd.grad, f.grad, kf, kb


def check_case(d, fc, masked=True, cm=None, mask_is_logit=True, want_dfc=False, offset=0, seed=0, what=""):
    B, T = d["mix"].shape[:2]
    dY = torch.randn(B, T, fc.shape[1], generator=torch.Generator().manual_seed(100 + seed))
    if masked:
        x = d["mask_logits"] if mask_is_logit else torch.sigmoid(d["mask_logits"])
        kw = dict(mix=d["mix"], lens=d["lens"], cm=cm, mask_is_logit=mask_is_logit, want_dfc=want_dfc)
    else:
        x = d["mix"]
        kw = dict(cm=cm, want_dfc=want_dfc)
    y, dx, dfc, kf, kb = run(x, fc, dY, offset=offset, **kw)
    compare(oracle(x, fc, dY, **kw), y, dx, dfc, what)
    return y, dx, kf, kb


# ---- tcgen05 kernels ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("masked", [True, False])
@pytest.mark.parametrize("offset", [0, 1, 2])
def test_tc_dense_bank_f257(masked, offset):
    """Dense 40-filter bank at the bench size: tcgen05 forward and backward.  The F = 257 forward pairs rows when the
    inputs are 8 B aligned (offset 0 and 2 floats); a 1-float offset takes its unpaired variant."""
    d = batch(32, 800, seed=11)
    fc = dense_bank(257, 40, 1)
    _, _, kf, kb = check_case(d, fc, masked=masked, cm=synth.cmvn(40, 3), want_dfc=not masked, offset=offset,
                              what="dense F=257 masked=%s offset=%d" % (masked, offset))
    kf.expect(TC_FWD)
    assert tc_fwd_kind(kf) == {"257" if offset == 1 else "pair"}
    assert {a[0] for a in kf.variants(TC_FWD)} == {"true" if masked else "false"}
    kb.expect(TC_BWD, *([] if masked else [DFC]))


@pytest.mark.parametrize("M", [40, 80])
def test_tc_forward_f256(M):
    """F = 256, the idim of the unet_128/256 enhancers: the generic (FC = 0) tcgen05 forward; the backward is the
    tcgen05 one over two 128-bin tiles for M = 40 and the SIMT one for M = 80."""
    d = batch(8, 400, F=256, seed=12)
    fc = dense_bank(256, M, 2)
    _, _, kf, kb = check_case(d, fc, cm=synth.cmvn(M, 4), want_dfc=True, what="F=256 M=%d" % M)
    kf.expect(TC_FWD)
    assert tc_fwd_kind(kf) == {"0"}
    kb.expect(TC_BWD if M == 40 else SIMT_BWD, DFC)


@pytest.mark.parametrize("F", [129, 100])
def test_tc_k_tails(F):
    """F = 129: a 1-bin tail after the last 32-bin chunk (forward) and after the 128-bin tile (backward); F = 100: a
    4-bin tail and a partial last chunk in the forward, one partial 128-bin tile in the backward."""
    d = batch(8, 400, F=F, seed=13)
    fc = dense_bank(F, 40, 3)
    _, _, kf, kb = check_case(d, fc, what="F=%d" % F)
    kf.expect(TC_FWD)
    assert tc_fwd_kind(kf) == {"0"}
    kb.expect(TC_BWD)
    _, _, kf, kb = check_case(d, fc, masked=False, seed=1, what="F=%d single input" % F)
    kf.expect(TC_FWD)
    kb.expect(TC_BWD)


@pytest.mark.parametrize("M", [80, 30])
def test_tc_forward_simt_backward(M):
    """The tcgen05 backward takes M <= 64 with M % 4 == 0: M = 80 and M = 30 run the SIMT backward.  At M = 80 only one
    pipeline stage fits shared memory, too few for the paired F = 257 forward."""
    d = batch(8, 400, seed=14)
    fc = dense_bank(257, M, 4)
    _, _, kf, kb = check_case(d, fc, cm=synth.cmvn(M, 5), what="M=%d" % M)
    kf.expect(TC_FWD)
    assert tc_fwd_kind(kf) == {"257" if M == 80 else "pair"}
    kb.expect(SIMT_BWD)


# ---- SIMT kernels and the M limit --------------------------------------------------------------------------------------
@pytest.mark.parametrize("M", [96, 128])
def test_simt_forward_and_backward(M):
    """Above 80 filters the tcgen05 forward's accumulators do not fit tensor memory: the SIMT kernels both ways."""
    d = batch(8, 400, seed=15)
    fc = dense_bank(257, M, 5)
    _, _, kf, kb = check_case(d, fc, cm=synth.cmvn(M, 6), what="M=%d" % M)
    kf.expect(SIMT_FWD)
    assert kf.variants(SIMT_FWD) == {("4",)}
    kb.expect(SIMT_BWD)
    _, _, kf, kb = check_case(d, fc, masked=False, want_dfc=True, seed=1, what="M=%d single input" % M)
    kf.expect(SIMT_FWD)
    kb.expect(SIMT_BWD, DFC)


def test_m_limit_is_the_same_both_ways():
    """At F = 257 the SIMT forward's shared-memory tile fits up to M = 176: both directions run there, and both entry
    points reject M = 177 before launching anything."""
    d = batch(2, 64, seed=16)
    fc = dense_bank(257, 176, 6)
    _, _, kf, kb = check_case(d, fc, want_dfc=True, what="M=176")
    kf.expect(SIMT_FWD)
    kb.expect(SIMT_BWD, DFC)

    M = 177
    L = _lib.lib()
    B, T, F = 2, 64, 257
    z = lambda *s: torch.zeros(*s, device=DEV)
    mag, mask, fcd, dY, G, d_in, dfc = z(B, T, F), z(B, T, F), z(F, M), z(B, T, M), z(B, T, M), z(B, T, F), z(F, M)
    Y = z(B, T, M)
    lens = torch.full((B,), T, device=DEV, dtype=torch.int32)
    P, s = _lib.ptr, _lib.stream_ptr()
    n0 = _lib.launch_count()
    assert L.re2e_fbank_fwd(P(mask), 1, P(mag), P(fcd), None, P(lens), P(Y), P(G), None, B, T, F, M, s) == E_UNSUPPORTED
    assert L.re2e_fbank_bwd(P(dY), P(G), P(mask), 1, P(mag), P(fcd), P(lens), P(d_in), P(dfc),
                            B, T, F, M, s) == E_UNSUPPORTED
    assert L.re2e_fbank_bwd(P(dY), P(G), P(mask), 1, P(mag), P(fcd), P(lens), None, P(dfc),
                            B, T, F, M, s) == E_UNSUPPORTED
    assert _lib.launch_count() == n0
    with pytest.raises(RuntimeError, match="not supported"):
        masked_fbank(mask, mag, lens.cpu(), dense_bank(F, M, 7).to(DEV))


# ---- trainable bank ----------------------------------------------------------------------------------------------------
def test_trainable_bank_banded_then_dense():
    """FbankModel(fbank_opti_type="train") starts from the reference's banded 80-filter bank: banded forward and
    backward, dense dfc.  After an update that fills every entry the bank is dense: tcgen05 forward, SIMT backward
    (M = 80), dfc."""
    d = batch(32, 800, seed=17)
    cm = synth.cmvn(80, 7)
    m = FbankModel(Args(fbank_opti_type="train")).to(DEV)
    assert m.fc.requires_grad
    dY = torch.randn(32, 800, 80, generator=torch.Generator().manual_seed(5))
    for step in ("banded", "dense"):
        if step == "dense":
            with torch.no_grad():
                m.fc.add_(1e-3 + 1e-3 * torch.rand(m.fc.shape, generator=torch.Generator().manual_seed(6)).to(DEV))
        fc = m.fc.detach().cpu().clone()
        ref = oracle(d["mask_logits"], fc, dY, mix=d["mix"], lens=d["lens"], cm=cm, want_dfc=True)
        m.fc.grad = None
        lo = d["mask_logits"].to(DEV).requires_grad_(True)
        with Kernels() as kf:
            y = m.forward_masked(lo, d["mix"].to(DEV), d["lens"], cm)
        with Kernels() as kb:
            y.backward(dY.to(DEV))
        compare(ref, y, lo.grad, m.fc.grad, what="trainable bank, " + step)
        if step == "banded":
            kf.expect(BAND_FWD)
            kb.expect(BAND_BWD, DFC)
        else:
            kf.expect(TC_FWD)
            kb.expect(SIMT_BWD, DFC)
        # the single-input form on the same bank
        ref = oracle(d["clean"], fc, dY, want_dfc=True)
        m.fc.grad = None
        x = d["clean"].to(DEV).requires_grad_(True)
        with Kernels() as kf:
            y = m(x)
        with Kernels() as kb:
            y.backward(dY.to(DEV))
        compare(ref, y, x.grad, m.fc.grad, what="trainable bank single input, " + step)
        kf.expect(BAND_FWD if step == "banded" else TC_FWD)
        kb.expect(BAND_BWD if step == "banded" else SIMT_BWD, DFC)


def test_forward_joint_with_trainable_bank():
    """forward_joint with a trainable bank makes three calls (no joint kernel): all three outputs, d logits and dfc
    (summed over the three outputs) against the oracle."""
    B, T, M = 8, 400, 80
    d = batch(B, T, seed=18)
    cm = synth.cmvn(M, 8)
    m = FbankModel(Args(fbank_opti_type="train")).to(DEV)
    g = torch.Generator().manual_seed(7)
    dYs = [torch.randn(B, T, M, generator=g) for _ in range(3)]
    refs = {}
    for dt in (torch.float32, torch.float64):
        f = m.fc.detach().cpu().to(dt).requires_grad_(True)
        lo = d["mask_logits"].clone().to(dt).requires_grad_(True)
        c = cm.to(dt)
        outs = (o_fe.masked_fbank_forward(lo, d["mix"].to(dt), d["lens"], f, c), o_fe.fbank_forward(d["mix"].to(dt), f, c),
                o_fe.fbank_forward(d["clean"].to(dt), f, c))
        torch.autograd.backward(outs, [y.to(dt) for y in dYs])
        refs[dt] = [o.detach() for o in outs] + [lo.grad, f.grad]
    lo = d["mask_logits"].to(DEV).requires_grad_(True)
    with Kernels() as kf:
        outs = m.forward_joint(lo, d["mix"].to(DEV), d["clean"].to(DEV), d["lens"], cm)
    with Kernels() as kb:
        torch.autograd.backward(outs, [y.to(DEV) for y in dYs])
    kf.expect(BAND_FWD)
    kb.expect(BAND_BWD, DFC)
    for got, i, what in ((outs[0], 0, "enhance_feat"), (outs[1], 1, "mix_feat"), (outs[2], 2, "clean_feat"),
                         (lo.grad, 3, "d logits"), (m.fc.grad, 4, "dfc")):
        assert_close(got, refs[torch.float32][i], truth=refs[torch.float64][i], what=what + " (joint, trainable)")


# ---- mask forms, return_enhanced, edge rows ----------------------------------------------------------------------------
@pytest.mark.parametrize("path", ["banded", "tcgen05", "simt"])
def test_plain_mask(path):
    """mask_is_logit=False (the mask is used as given) on each path."""
    d = batch(8, 400, seed=19)
    fc = {"banded": synth.mel_fc(257, 40), "tcgen05": dense_bank(257, 40, 8), "simt": dense_bank(257, 96, 9)}[path]
    _, _, kf, kb = check_case(d, fc, cm=synth.cmvn(fc.shape[1], 9), mask_is_logit=False, what="plain mask, " + path)
    kf.expect({"banded": BAND_FWD, "tcgen05": TC_FWD, "simt": SIMT_FWD}[path])
    kb.expect({"banded": BAND_BWD, "tcgen05": TC_BWD, "simt": SIMT_BWD}[path])


def test_return_enhanced():
    """return_enhanced=True writes enhance_out from the dense forward (the banded kernels do not write it)."""
    B, T, M = 32, 800, 40
    d = batch(B, T, seed=20)
    fc, cm = synth.mel_fc(257, M), synth.cmvn(M, 10)
    dY = torch.randn(B, T, M, generator=torch.Generator().manual_seed(8))
    ref = oracle(d["mask_logits"], fc, dY, mix=d["mix"], lens=d["lens"], cm=cm)
    enh64 = o_fe.mask_tail(d["mask_logits"].double(), d["mix"].double(), d["lens"])
    enh32 = o_fe.mask_tail(d["mask_logits"], d["mix"], d["lens"])
    lo = d["mask_logits"].to(DEV).requires_grad_(True)
    with Kernels() as kf:
        y, enh = masked_fbank(lo, d["mix"].to(DEV), d["lens"], fc.to(DEV), cm.to(DEV), return_enhanced=True)
    with Kernels() as kb:
        y.backward(dY.to(DEV))
    kf.expect(TC_FWD)
    kb.expect(TC_BWD)
    assert_close(enh, enh32, truth=enh64, what="enhance_out")
    compare(ref, y, lo.grad, what="return_enhanced")


@pytest.mark.parametrize("B,T,lens,path", [(1, 1, None, "tcgen05"), (3, 101, [101, 50, 0], "tcgen05"),
                                           (4, 50, [50, 37, 12, 0], "banded")])
def test_edge_rows(B, T, lens, path):
    """One frame; N = 303 (not a multiple of 8 or 64: no banded path); utterances of length 0."""
    d = batch(B, T, seed=21, lens=lens, zeros=0 if B * T == 1 else 4)
    M = 40
    y, dx, kf, kb = check_case(d, synth.mel_fc(257, M), cm=synth.cmvn(M, 11), what="B=%d T=%d" % (B, T))
    kf.expect(BAND_FWD if path == "banded" else TC_FWD)
    kb.expect(BAND_BWD if path == "banded" else TC_BWD)
    for b in range(B):
        n = int(d["lens"][b])
        assert torch.all(dx[b, n:] == 0)          # padded frames: exactly zero gradient
    _, _, kf, kb = check_case(d, synth.mel_fc(257, M), masked=False, seed=1, what="single input B=%d T=%d" % (B, T))
    kf.expect(BAND_FWD if path == "banded" else TC_FWD)


# ---- stand-alone mask tail and CMVN statistics -------------------------------------------------------------------------
@pytest.mark.parametrize("offset", [0, 1])
def test_apply_mask(offset):
    """The stand-alone mask tail, forward and backward: 16 B aligned buffers take the vector loop, a 1-float offset
    the scalar one."""
    B, T = 32, 800
    d = batch(B, T, seed=22)
    dE = torch.randn(B, T, 257, generator=torch.Generator().manual_seed(9))
    ref = {}
    for dt in (torch.float32, torch.float64):
        lo = d["mask_logits"].clone().to(dt).requires_grad_(True)
        e = o_fe.mask_tail(lo, d["mix"].to(dt), d["lens"])
        e.backward(dE.to(dt))
        ref[dt] = (e.detach(), lo.grad)
    lo = on_dev(d["mask_logits"], offset).requires_grad_(True)
    with Kernels() as kf:
        e = apply_mask(lo, on_dev(d["mix"], offset), d["lens"])
    with Kernels() as kb:
        e.backward(on_dev(dE, offset))
    kf.expect("mask_apply_kernel")
    kb.expect("mask_apply_kernel")
    assert_close(e, ref[torch.float32][0], truth=ref[torch.float64][0], what="apply_mask")
    assert_close(lo.grad, ref[torch.float32][1], truth=ref[torch.float64][1], what="apply_mask d logits")
    assert torch.all(e[B - 1, int(d["lens"][B - 1]):] == 0)


def test_compute_cmvn_statistics():
    """compute_cmvn (re2e_cmvn_stats) at the bench size against fp64 NumPy sums over the valid frames, lengths 0 and
    T included."""
    B, T, M = 32, 800, 80
    lens = [T] + sorted(np.random.RandomState(3).randint(1, T, B - 2).tolist(), reverse=True) + [0]
    d = batch(B, T, seed=23, lens=lens)
    m = FbankModel(Args(train_dataset_len=B, num_utt_cmvn=B)).to(DEV)
    mag = d["mix"].to(DEV)
    with Kernels() as k:
        assert m.compute_cmvn(mag, d["lens"]) is None
    k.expect(BAND_FWD, "cmvn_stats_kernel")
    est = m.compute_cmvn(mag, d["lens"])
    assert m.frame_count == sum(lens) and int(m._dev_frames) == sum(lens) and m.cmvn_processed_num == B
    feats = m(mag).detach().cpu().double().numpy()
    valid = np.concatenate([feats[b, :n] for b, n in enumerate(lens)])
    mean = valid.sum(0) / len(valid)
    var = np.square(valid).sum(0) / len(valid) - np.square(mean)
    assert_close(m.sum[0], valid.sum(0), what="sum")
    assert_close(m.sum_sq[0], np.square(valid).sum(0), what="sum of squares")
    assert_close(est[0], -mean, what="-mean")
    assert_close(est[1], 1 / np.sqrt(var), what="1/std")


# ---- band-table cache and alignment ------------------------------------------------------------------------------------
def test_band_tables_follow_writes_through_data():
    """A bank written through ``fc.data`` (which does not bump ``fc._version``) is what the next call computes with:
    a different banded bank on the banded kernels, a dense one on the dense kernels."""
    d = batch(8, 400, seed=24)
    m = FbankModel(Args()).to(DEV)
    x = d["mix"].to(DEV)
    with Kernels() as k:
        m(x)
    k.expect(BAND_FWD)
    for new, path in ((2.0 * ref_bank80(), BAND_FWD), (dense_bank(257, 80, 10), TC_FWD)):
        m.fc.data.copy_(new)
        with Kernels() as k:
            y = m(x)
        k.expect(path)
        assert_close(y, o_fe.fbank_forward(d["mix"], new), truth=o_fe.fbank_forward(d["mix"].double(), new.double()),
                     what="after fc.data.copy_ (%s)" % path)


def test_band_tables_of_a_freed_bank_do_not_alias():
    """A new bank allocated where a freed one was, with an equal ``_version``, gets its own tables."""
    d = batch(8, 400, seed=25)
    x = d["mix"].to(DEV)
    bank_a, bank_b = ref_bank80(), 0.5 * ref_bank80()
    pool = torch.cuda.MemPool()
    with torch.cuda.use_mem_pool(pool):
        fa = bank_a.to(DEV)
    where = (fa.data_ptr(), fa._version)
    assert_close(fbank(x, fa), o_fe.fbank_forward(d["mix"], bank_a), what="first bank")
    del fa
    with torch.cuda.use_mem_pool(pool):
        fb = bank_b.to(DEV)
    assert (fb.data_ptr(), fb._version) == where, "the allocator did not reuse the freed bank's block"
    with Kernels() as k:
        y = fbank(x, fb)
    k.expect(BAND_FWD)
    assert_close(y, o_fe.fbank_forward(d["mix"], bank_b), truth=o_fe.fbank_forward(d["mix"].double(), bank_b.double()),
                 what="second bank at the first one's address")
    del fb


def test_unaligned_inputs_take_the_dense_kernels():
    """Contiguous views that are not 16 B aligned (``x[1:]`` with T % 4 != 0, a 1-float offset for dY) run on the dense
    kernels instead of failing in the banded ones -- masked, single-input and joint forms, forward and backward."""
    B, T, M = 8, 401, 40
    big = batch(B + 1, T, seed=26)
    d = {k: v[1:] for k, v in big.items() if k != "lens"}
    d["lens"] = big["lens"][1:]
    fc, cm = synth.mel_fc(257, M), synth.cmvn(M, 12)
    assert fm._band_for(fc.to(DEV), B, T) is not None
    dY = torch.randn(B, T, M, generator=torch.Generator().manual_seed(11))
    ref = oracle(d["mask_logits"], fc, dY, mix=d["mix"], lens=d["lens"], cm=cm)
    lo_all, mix_all, clean_all = (big[k].to(DEV) for k in ("mask_logits", "mix", "clean"))
    lo, mix, clean = lo_all[1:], mix_all[1:], clean_all[1:]
    assert lo.data_ptr() % 16 and mix.data_ptr() % 16 and clean.data_ptr() % 16
    fcd = fc.to(DEV)

    # unaligned inputs: dense forward (the unpaired F = 257 variant) and backward
    lo.requires_grad_(True)
    with Kernels() as kf:
        y = masked_fbank(lo, mix, d["lens"], fcd, cm.to(DEV))
    with Kernels() as kb:
        y.backward(dY.to(DEV))
    kf.expect(TC_FWD)
    assert tc_fwd_kind(kf) == {"257"}
    kb.expect(TC_BWD)
    compare(ref, y, lo.grad, what="unaligned mask and mix")

    # aligned inputs, unaligned dY: banded forward, dense backward
    lo2 = d["mask_logits"].to(DEV).requires_grad_(True)
    with Kernels() as kf:
        y = masked_fbank(lo2, d["mix"].to(DEV), d["lens"], fcd, cm.to(DEV))
    with Kernels() as kb:
        y.backward(on_dev(dY, 1))
    kf.expect(BAND_FWD)
    kb.expect(SIMT_BWD)
    compare(ref, y, lo2.grad, what="unaligned dY")

    # single input
    ref1 = oracle(d["clean"], fc, dY, cm=cm)
    x = clean_all[1:].detach().requires_grad_(True)
    with Kernels() as kf:
        y = fbank(x, fcd, cm.to(DEV))
    with Kernels() as kb:
        y.backward(dY.to(DEV))
    kf.expect(TC_FWD)
    kb.expect(TC_BWD)
    compare(ref1, y, x.grad, what="unaligned single input")

    # forward_joint of a frozen banded bank: three dense calls instead of the joint kernel
    m = FbankModel(Args(fbank_dim=M)).to(DEV)
    m.fc.data.copy_(fc)
    lo3 = lo_all[1:].detach().requires_grad_(True)
    with Kernels() as kf:
        enh, mixf, cleanf = m.forward_joint(lo3, mix, clean, d["lens"], cm)
    with Kernels() as kb:
        enh.backward(dY.to(DEV))
    kf.expect(TC_FWD)
    kb.expect(TC_BWD)
    compare(ref, enh, lo3.grad, what="unaligned joint")
    assert_close(mixf, o_fe.fbank_forward(d["mix"], fc, cm), what="mix_feat (unaligned joint)")
    assert_close(cleanf, ref1[torch.float32][0], truth=ref1[torch.float64][0], what="clean_feat (unaligned joint)")

    # forward_joint on aligned inputs with an unaligned dY: the joint kernel, then the dense backward
    lo4 = d["mask_logits"].to(DEV).requires_grad_(True)
    with Kernels() as kf:
        enh, _, _ = m.forward_joint(lo4, d["mix"].to(DEV), d["clean"].to(DEV), d["lens"], cm)
    with Kernels() as kb:
        enh.backward(on_dev(dY, 1))
    kf.expect(BAND_FWD)
    kb.expect(SIMT_BWD)
    compare(ref, enh, lo4.grad, what="joint, unaligned dY")
