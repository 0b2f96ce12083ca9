"""GPU: the drop-in claim of INTEGRATION.md, SHOWN -- the reference's own ``E2E`` (model/e2e_model.py:20-137) is
built from the UNMODIFIED reference files with only the import bindings swapped (``AttLoc``, ``CTC`` in
model/e2e_model.py:14-16; ``CTCPrefixScore`` in model/e2e_decoder.py:14; optionally ``Decoder``), runs
``forward`` + ``backward`` and ``recognize`` on the GPU, and is compared with the unmodified reference on the CPU
(fp32, with the reference in fp64 as tie-breaker): losses and EVERY parameter gradient within 1e-4, beam-search
tokens identical.  Plus ``FbankModel.load_model`` on a reference-format checkpoint (model/e2e_common.py:22-38).

The swapped-import tests import the reference's unmodified modules through ``oracle/refshim.py`` and skip when they
are not present; the checkpoint test needs only tests/golden.
"""
import copy
import types

import numpy as np
import pytest
import torch

import helpers
from conftest import golden
from oracle import frontend as o_fe
from oracle import refshim
import robust_e2e_gan_b200 as ours
from robust_e2e_gan_b200 import synth

pytestmark = pytest.mark.gpu
needs_reference = pytest.mark.skipif(not refshim.available(), reason="reference tree / oracle/_ref not present")
DEV = "cuda:0"


@pytest.fixture(autouse=True)
def strict_fp32_library_math():
    """The parts of the swapped model that are NOT ours -- the reference's BLSTM encoder and LSTMCell decoder -- run
    in cuDNN / cuBLAS on the GPU; cuDNN's default TF32 RNN math alone moves every gradient by ~5e-4 against the
    CPU reference.  Pin the library code to fp32 so the comparison isolates the swapped modules."""
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _batch(args, B=3, T=40, seed=0):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, T, args.fbank_dim, generator=g)
    ilens = torch.tensor(sorted([T - 3 * i for i in range(B)], reverse=True))
    for b in range(B):
        x[b, int(ilens[b]):] = 0
    tsz = torch.tensor([3 + (i % 3) for i in range(B)])
    targets = torch.randint(1, args.odim - 1, (int(tsz.sum()),), generator=g)
    return x, targets, ilens, tsz


def _run(model, batch, dev):
    x, targets, ilens, tsz = batch
    model.zero_grad()
    loss_ctc, loss_att, acc = model(x.to(dev), targets.to(dev), ilens, tsz)
    a = model.mtlalpha
    (a * loss_ctc.sum() + (1 - a) * loss_att).backward()          # asr_train.py:123
    grads = {k: p.grad.detach().double().cpu() for k, p in model.named_parameters() if p.grad is not None}
    return float(loss_ctc.sum()), float(loss_att), acc, grads


@needs_reference
@pytest.mark.parametrize("dims", [dict(), dict(eprojs=320, adim=320, dunits=300, aconv_chans=10, aconv_filts=100,
                                               eunits=64, odim=52)])
@pytest.mark.parametrize("swap_decoder", [False, True])
def test_reference_e2e_with_swapped_imports_matches_reference(dims, swap_decoder):
    args = refshim.e2e_args(**dims)
    ref_mod = refshim.load().e2e_model
    torch.manual_seed(5)
    ref = ref_mod.E2E(copy.deepcopy(args))                       # unmodified reference, CPU
    sd = copy.deepcopy(ref.state_dict())
    batch = _batch(args, seed=11)
    r32 = _run(ref, batch, "cpu")
    ref64 = ref_mod.E2E(copy.deepcopy(args)).double()
    ref64.load_state_dict({k: v.double() for k, v in sd.items()})
    x, targets, ilens, tsz = batch
    r64 = _run(ref64, (x.double(), targets, ilens, tsz), "cpu")

    n0 = ours._lib.launch_count()
    with refshim.swapped(AttLoc=ours.AttLoc, CTC=ours.CTC, CTCPrefixScore=ours.CTCPrefixScore,
                         Decoder=ours.Decoder if swap_decoder else None) as m:
        mine = m.E2E(copy.deepcopy(args))
        assert type(mine.att) is ours.AttLoc and type(mine.ctc) is ours.CTC and mine.dec.att is mine.att
        assert isinstance(mine.dec, ours.Decoder) == swap_decoder
        mine.load_state_dict(sd, strict=True)                                # reference checkpoint loads unchanged
        mine = mine.to(DEV)
        g = _run(mine, batch, DEV)
    assert ours._lib.launch_count() - n0 > 0, "the swapped model launched none of our kernels"
    helpers.assert_close(np.float64(g[0]), np.float64(r32[0]), truth=np.float64(r64[0]), what="loss_ctc")
    helpers.assert_close(np.float64(g[1]), np.float64(r32[1]), truth=np.float64(r64[1]), what="loss_att")
    assert g[2] == pytest.approx(r32[2])
    assert set(g[3]) == set(r32[3])
    bad = []
    for k in sorted(r32[3]):
        if k.endswith("att.gvec.bias"):        # analytically zero (softmax shift invariance): no scale to compare to
            continue
        try:
            helpers.assert_close(g[3][k], r32[3][k], truth=r64[3][k], what="d " + k)
        except AssertionError as e:
            bad.append(str(e))
    assert not bad, "\n".join(bad)


@needs_reference
@pytest.mark.parametrize("swap_decoder", [False, True])
@pytest.mark.parametrize("ctc_weight,beam", [(0.3, 4), (0.0, 3), (1.0, 2)])
def test_reference_recognize_with_swapped_imports_gives_identical_tokens(swap_decoder, ctc_weight, beam):
    args = refshim.e2e_args(odim=24)
    ref_mod = refshim.load().e2e_model
    torch.manual_seed(17)
    ref = ref_mod.E2E(copy.deepcopy(args))
    with torch.no_grad():
        ref.dec.output.bias[args.odim - 1] += 1.5                 # let hypotheses end (random-init models rarely emit <eos>)
    sd = copy.deepcopy(ref.state_dict())
    g = torch.Generator().manual_seed(3)
    x = torch.randn(1, 60, args.fbank_dim, generator=g)
    ra = types.SimpleNamespace(beam_size=beam, penalty=0.0, ctc_weight=ctc_weight, maxlenratio=0.0, minlenratio=0.0,
                               nbest=min(2, beam), lm_weight=0.0)
    want = ref.recognize(x, ra, args.char_list)
    with refshim.swapped(AttLoc=ours.AttLoc, CTC=ours.CTC, CTCPrefixScore=ours.CTCPrefixScore,
                         Decoder=ours.Decoder if swap_decoder else None) as m:
        mine = m.E2E(copy.deepcopy(args))
        mine.load_state_dict(sd, strict=True)
        mine = mine.to(DEV)
        got = mine.recognize(x, ra, args.char_list)
    assert len(got) == len(want)
    for a, b in zip(got, want):
        assert [int(t) for t in a["yseq"]] == [int(t) for t in b["yseq"]]
        assert abs(float(a["score"]) - float(b["score"])) <= 1e-4 * max(1.0, abs(float(b["score"])))


def test_fbank_load_model_from_reference_checkpoint(tmp_path):
    """ModelBase.load_model (model/e2e_common.py:22-38) on a checkpoint written the way the reference's scripts do
    (enhance_fbank_train.py: {'opt': ..., 'fbank_state_dict': feat_model.state_dict()}), trained-bank case.  The
    reference FbankModel's state is its 80-filter bank alone, stored as ``fc`` in tests/golden/fbank.npz; its forward
    is the oracle restatement, which tests/test_oracle.py pins to the reference's own outputs."""
    opt = refshim.fbank_args(fbank_dim=80, fbank_opti_type="train")
    ref_fc = torch.from_numpy(golden("fbank")["fc"])
    fc = ref_fc * (1.0 + 0.01 * torch.randn(ref_fc.shape, generator=torch.Generator().manual_seed(1)))   # "trained"
    path = str(tmp_path / "fbank.pth")
    torch.save({"opt": opt, "fbank_state_dict": {"fc": fc}}, path)
    opt_run = copy.deepcopy(opt)
    opt_run.gpu_ids = [0]
    mine = ours.FbankModel.load_model(path, "fbank_state_dict", opt_run)
    assert mine.fc.is_cuda and torch.equal(mine.fc.detach().cpu(), fc)
    g = torch.Generator().manual_seed(2)
    x = (torch.randn(2, 30, 257, generator=g).abs() * 300).requires_grad_(True)
    cm = synth.cmvn(80, 4)
    fc_ref = fc.clone().requires_grad_(True)
    y_ref = o_fe.fbank_forward(x, fc_ref, cm)
    dY = torch.randn(y_ref.shape, generator=g)
    y_ref.backward(dY)
    xg = x.detach().clone().requires_grad_(True)                 # CPU leaf: moved like the reference's to_cuda does
    y = mine(xg, cm)
    y.backward(dY.to(DEV))
    helpers.assert_close(y, y_ref, what="Y (loaded checkpoint)")
    helpers.assert_close(xg.grad, x.grad, what="d mag (loaded checkpoint)")
    helpers.assert_close(mine.fc.grad, fc_ref.grad, what="d fc (loaded checkpoint)")
    # no path: cls(opt) -- the freshly constructed model is the reference's fresh model
    fresh = ours.FbankModel.load_model(None, "fbank_state_dict", opt_run)
    assert torch.equal(fresh.fc.detach().cpu(), ref_fc)
