"""Drop-in ``FbankModel`` (reference: model/feat_model.py:93-135) on the fused sm_100a front-end.

Same constructor (``FbankModel(args)``), same parameter (``fc`` (idim, fbank_dim)), same
``forward(xs, fbank_cmvn=None)`` and ``compute_cmvn(inputs, input_sizes)``; the arithmetic runs in
``re2e_fbank_fwd`` / ``re2e_fbank_bwd`` (csrc/fbank.cu).  In addition ``forward_masked`` exposes the
fully fused stage named by the north star -- mask tail of EnhanceModel.forward
(model/enhance_model.py:157-164) + power + mel + log + CMVN in one kernel -- so that the
(B,T,257) ``enhance_out`` never round-trips through HBM.
"""
import weakref

import numpy as np
import torch

from . import _lib
from .e2e_common import ModelBase


# ------------------------------------------------------------------------------------------ banks
def kaldi_mel_banks(num_bins=80, nfft=512, samplerate=16000, low_freq=20.0):
    """Kaldi-style triangular bank in the mel domain (mel = 1127 ln(1 + f/700)), (num_bins, nfft/2+1).

    Used for every size EXCEPT 80: the reference has a table only for 80 filters (its constructor crashes for any
    other size, SURVEY.md 0.5), and for 80 ``reference_fbank80`` returns that table's exact constants (this
    formula lands within 1.4e-5 of them, which is not the same model).
    """
    f32 = np.float32

    def mel(f):
        return f32(1127.0) * np.log(f32(1.0) + f32(f) / f32(700.0), dtype=f32)

    fbw = f32(samplerate) / f32(nfft)
    ml, mh = mel(low_freq), mel(samplerate / 2.0)
    delta = (mh - ml) / f32(num_bins + 1)
    out = np.zeros((num_bins, nfft // 2 + 1), dtype=np.float64)
    mels = np.array([mel(fbw * f32(i)) for i in range(nfft // 2)], dtype=f32)
    for b in range(num_bins):
        left, center, right = ml + f32(b) * delta, ml + f32(b + 1) * delta, ml + f32(b + 2) * delta
        for i in range(nfft // 2):
            m = mels[i]
            if m > left and m < right:
                w = (m - left) / (center - left) if m <= center else (right - m) / (right - center)
                out[b, i] = float('%g' % w)
    return out


def reference_fbank80():
    """The reference's hard-coded 80-filter bank (model/feat_model.py:15-33) as a dense (80, 257) float64
    matrix, bit-identical to what its ``get_filterbanks(80)`` builds (constants in fbank80_table.py)."""
    from . import fbank80_table as tb
    out = np.zeros((tb.NUM_FILTERS, tb.NUM_BINS), dtype=np.float64)
    pos = 0
    for j, (lo, n) in enumerate(zip(tb.FIRST_BIN, tb.RUN)):
        out[j, lo:lo + n] = tb.WEIGHTS[pos:pos + n]
        pos += n
    assert pos == len(tb.WEIGHTS)
    return out


def generic_mel_banks(nfilt=40, nfft=512, samplerate=16000, lowfreq=0, highfreq=None):
    """Triangular bank on fft-bin edges (formula of model/e2e_common.py:104-132)."""
    highfreq = highfreq or samplerate / 2
    lowmel = 2595 * np.log10(1 + lowfreq / 700.)
    highmel = 2595 * np.log10(1 + highfreq / 700.)
    melpoints = np.linspace(lowmel, highmel, nfilt + 2)
    edges = np.floor((nfft + 1) * (700 * (10 ** (melpoints / 2595.0) - 1)) / samplerate)
    fbank = np.zeros([nfilt, nfft // 2 + 1])
    for j in range(nfilt):
        lo, mid, hi = int(edges[j]), int(edges[j + 1]), int(edges[j + 2])
        for i in range(lo, mid):
            fbank[j, i] = (i - edges[j]) / (edges[j + 1] - edges[j])
        for i in range(mid, hi):
            fbank[j, i] = (edges[j + 2] - i) / (edges[j + 2] - edges[j + 1])
    return fbank


# ------------------------------------------------------------------------------------ band tables
BAND_W, BIN_W = 32, 4          # csrc/fbank_band.cu: bins per filter window, filters per bin window
_BAND_CACHE = {}               # id(fc) -> (weak reference to fc, copy of fc the tables were built from, tables or None)


def band_tables(fc):
    """Structure tables of a BANDED bank for re2e_fbank_band_* (see include/re2e_b200.h), or None when ``fc`` (F, M)
    numpy is not banded (some filter's support wider than 32 bins, or some bin feeding filters more than 4 apart --
    e.g. a trained, dense bank).  Returns (flo int32 (M,), fw float32 (M,32), mlo int32 (F,), bw float32 (F,4))."""
    F, M = fc.shape
    if F < BAND_W or M < BIN_W:
        return None
    nz = fc != 0
    flo, fw = np.zeros(M, np.int32), np.zeros((M, BAND_W), np.float32)
    for m in range(M):
        idx = np.flatnonzero(nz[:, m])
        if idx.size:
            if idx[-1] - idx[0] + 1 > BAND_W:
                return None
            flo[m] = min(int(idx[0]), F - BAND_W)
        fw[m] = fc[flo[m]:flo[m] + BAND_W, m]
    mlo, bw = np.zeros(F, np.int32), np.zeros((F, BIN_W), np.float32)
    for f in range(F):
        idx = np.flatnonzero(nz[f])
        if idx.size:
            if idx[-1] - idx[0] + 1 > BIN_W:
                return None
            mlo[f] = min(int(idx[0]), M - BIN_W)
        bw[f] = fc[f, mlo[f]:mlo[f] + BIN_W]
    return flo, fw, mlo, bw


def _band_for(fc, B, T):
    """Device band tables of ``fc`` when the banded kernels apply to this call, else None.

    Entries are keyed on the tensor object through a weak reference, so a freed bank's entry goes with it and a new bank
    allocated at the same address never finds it.  Each entry keeps a copy of the values its tables were built from.
    Outside a CUDA-graph capture every call compares ``fc`` with that copy on the device (one small compare and a sync)
    and rebuilds on a mismatch: a write through ``fc.data`` does not bump ``fc._version``, so nothing cheaper sees it.
    Building the tables is a device-to-host read, so a capture never builds or checks them: it uses the entry of this
    ``fc`` that its eager warm-up left, or the dense kernels when there is none.  A captured graph replays the tables
    it was captured with, so a bank is frozen for the life of a captured StepRunner."""
    F, M = fc.shape
    if not _lib.load().re2e_fbank_band_supported(B, T, F, M):
        return None
    ent = _BAND_CACHE.get(id(fc))
    if ent is not None and (ent[0]() is not fc or (ent[1].device, ent[1].dtype) != (fc.device, fc.dtype)):
        ent = None
    if torch.cuda.is_current_stream_capturing():
        return None if ent is None else ent[2]
    if ent is not None and torch.equal(ent[1], fc.detach()):
        return ent[2]
    snap = fc.detach().clone()
    tabs = band_tables(snap.float().cpu().numpy())
    tabs = None if tabs is None else tuple(torch.from_numpy(t).to(fc.device) for t in tabs)
    key = id(fc)

    def forget(ref):
        if _BAND_CACHE.get(key, (None,))[0] is ref:
            del _BAND_CACHE[key]

    _BAND_CACHE[key] = (weakref.ref(fc, forget), snap, tabs)
    return tabs


def _aligned16(*ts):
    """The banded kernels move rows with 16 B bulk copies: every buffer they read or write must be 16 B aligned."""
    return all(t is None or t.data_ptr() % 16 == 0 for t in ts)


# --------------------------------------------------------------------------------------- autograd
class _FbankFunction(torch.autograd.Function):
    """Y = CMVN(log(clamp((act(mask)*valid*mag)^2 @ fc))) ; mask may be None (single-input form)."""

    @staticmethod
    def forward(ctx, mask, mag, fc, cmvn, lens, mask_is_logit, want_enh):
        L = _lib.lib()
        dev = fc.device
        mag = _lib.f32c(mag, dev)
        mask = _lib.f32c(mask, dev) if mask is not None else None
        fcc = _lib.f32c(fc.detach(), dev)
        cm = _lib.f32c(cmvn, dev) if cmvn is not None else None
        ln = lens.to(dev, torch.int32, non_blocking=True).contiguous() if lens is not None else None
        B, T, F = mag.shape
        M = fcc.shape[1]
        assert fcc.shape[0] == F, "fc must be (idim=%d, odim), got %s" % (F, tuple(fcc.shape))
        need_grad = any(ctx.needs_input_grad[:3])
        Y = torch.empty(B, T, M, device=dev, dtype=torch.float32)
        G = torch.empty(B, T, M, device=dev, dtype=torch.float32) if need_grad else None
        enh = torch.empty(B, T, F, device=dev, dtype=torch.float32) if (want_enh and mask is not None) else None
        band = _band_for(fc, B, T) if enh is None and _aligned16(mag, mask) else None
        with _lib.on(dev):
            if band is not None:      # banded (mel) bank: the streaming kernels
                _lib.check(L.re2e_fbank_band_fwd(_lib.ptr(mask), int(mask_is_logit), _lib.ptr(mag), None,
                                                 _lib.ptr(band[0]), _lib.ptr(band[1]), _lib.ptr(cm), _lib.ptr(ln),
                                                 _lib.ptr(Y), _lib.ptr(G), None, None, B, T, F, M, _lib.stream_ptr()),
                           "re2e_fbank_band_fwd")
            else:
                _lib.check(L.re2e_fbank_fwd(_lib.ptr(mask), int(mask_is_logit), _lib.ptr(mag), _lib.ptr(fcc),
                                            _lib.ptr(cm), _lib.ptr(ln), _lib.ptr(Y), _lib.ptr(G), _lib.ptr(enh),
                                            B, T, F, M, _lib.stream_ptr()), "re2e_fbank_fwd")
        if need_grad:
            ctx.save_for_backward(mask, mag, fcc, ln, G)
            ctx.mask_is_logit = int(mask_is_logit)
            ctx.band = band
        if enh is not None:
            ctx.mark_non_differentiable(enh)
            return Y, enh
        return Y, None

    @staticmethod
    def backward(ctx, dY, _d_enh):
        L = _lib.lib()
        mask, mag, fcc, ln, G = ctx.saved_tensors
        dev = mag.device
        B, T, F = mag.shape
        M = fcc.shape[1]
        dY = _lib.f32c(dY, dev)
        want_in = ctx.needs_input_grad[0] if mask is not None else ctx.needs_input_grad[1]
        d_in = torch.empty(B, T, F, device=dev, dtype=torch.float32) if want_in else None
        dfc = torch.zeros(F, M, device=dev, dtype=torch.float32) if ctx.needs_input_grad[2] else None
        band = ctx.band if _aligned16(dY) else None      # mask, mag: checked in forward; G, d_in: fresh
        with _lib.on(dev):
            if band is not None and d_in is not None:      # banded bank: d_in from the streaming kernel
                _lib.check(L.re2e_fbank_band_bwd(_lib.ptr(dY), _lib.ptr(G), _lib.ptr(mask), ctx.mask_is_logit,
                                                 _lib.ptr(mag), _lib.ptr(band[2]), _lib.ptr(band[3]), _lib.ptr(ln),
                                                 _lib.ptr(d_in), B, T, F, M, _lib.stream_ptr()), "re2e_fbank_band_bwd")
                if dfc is not None:                        # a trainable bank that is (still) banded: dfc is dense
                    _lib.check(L.re2e_fbank_bwd(_lib.ptr(dY), _lib.ptr(G), _lib.ptr(mask), ctx.mask_is_logit,
                                                _lib.ptr(mag), _lib.ptr(fcc), _lib.ptr(ln), None, _lib.ptr(dfc),
                                                B, T, F, M, _lib.stream_ptr()), "re2e_fbank_bwd")
            else:
                _lib.check(L.re2e_fbank_bwd(_lib.ptr(dY), _lib.ptr(G), _lib.ptr(mask), ctx.mask_is_logit,
                                            _lib.ptr(mag), _lib.ptr(fcc), _lib.ptr(ln), _lib.ptr(d_in),
                                            _lib.ptr(dfc), B, T, F, M, _lib.stream_ptr()), "re2e_fbank_bwd")
        if mask is not None:
            return d_in, None, dfc, None, None, None, None
        return None, d_in, dfc, None, None, None, None


class _FbankJoint(torch.autograd.Function):
    """The three front-end calls of one joint_train.py iteration (:158-161) in ONE launch when the bank is banded:
    enhance_feat (mask tail x mix, differentiable w.r.t. the mask), mix_feat and clean_feat (plain, no gradient: the
    bank is frozen and the inputs are data).  ``mix`` is read once for two outputs."""

    @staticmethod
    def forward(ctx, mask, mix, clean, fc, cmvn, lens, band):
        L = _lib.lib()
        dev = fc.device
        mix, clean, mask = _lib.f32c(mix, dev), _lib.f32c(clean, dev), _lib.f32c(mask, dev)
        cm = _lib.f32c(cmvn, dev) if cmvn is not None else None
        ln = lens.to(dev, torch.int32, non_blocking=True).contiguous() if lens is not None else None
        B, T, F = mix.shape
        M = fc.shape[1]
        need_grad = ctx.needs_input_grad[0]
        Y, Ym, Yc = (torch.empty(B, T, M, device=dev, dtype=torch.float32) for _ in range(3))
        G = torch.empty(B, T, M, device=dev, dtype=torch.float32) if need_grad else None
        with _lib.on(dev):
            _lib.check(L.re2e_fbank_band_fwd(_lib.ptr(mask), 1, _lib.ptr(mix), _lib.ptr(clean), _lib.ptr(band[0]),
                                             _lib.ptr(band[1]), _lib.ptr(cm), _lib.ptr(ln), _lib.ptr(Y), _lib.ptr(G),
                                             _lib.ptr(Ym), _lib.ptr(Yc), B, T, F, M, _lib.stream_ptr()),
                       "re2e_fbank_band_fwd")
        if need_grad:
            ctx.save_for_backward(mask, mix, _lib.f32c(fc.detach(), dev), ln, G, band[2], band[3])
        ctx.mark_non_differentiable(Ym, Yc)
        return Y, Ym, Yc

    @staticmethod
    def backward(ctx, dY, _dYm, _dYc):
        L = _lib.lib()
        mask, mix, fcc, ln, G, mlo, bw = ctx.saved_tensors
        B, T, F = mix.shape
        M = G.shape[2]
        dY = _lib.f32c(dY, mix.device)
        d_mask = torch.empty(B, T, F, device=mix.device, dtype=torch.float32)
        with _lib.on(mix.device):
            if _aligned16(dY):
                _lib.check(L.re2e_fbank_band_bwd(_lib.ptr(dY), _lib.ptr(G), _lib.ptr(mask), 1, _lib.ptr(mix),
                                                 _lib.ptr(mlo), _lib.ptr(bw), _lib.ptr(ln), _lib.ptr(d_mask),
                                                 B, T, F, M, _lib.stream_ptr()), "re2e_fbank_band_bwd")
            else:                 # the banded kernel needs 16 B aligned rows: the dense kernels take any dY
                _lib.check(L.re2e_fbank_bwd(_lib.ptr(dY), _lib.ptr(G), _lib.ptr(mask), 1, _lib.ptr(mix), _lib.ptr(fcc),
                                            _lib.ptr(ln), _lib.ptr(d_mask), None, B, T, F, M, _lib.stream_ptr()),
                           "re2e_fbank_bwd")
        return d_mask, None, None, None, None, None, None


def fbank(xs, fc, fbank_cmvn=None):
    """Functional single-input front-end: (B,T,F) magnitudes -> (B,T,M) log-mel (+CMVN)."""
    return _FbankFunction.apply(None, xs, fc, fbank_cmvn, None, 0, False)[0]


def masked_fbank(linear_out, mix_inputs, input_sizes, fc, fbank_cmvn=None, mask_is_logit=True,
                 return_enhanced=False):
    """Fused mask tail + front-end.  ``linear_out`` is the enhancement net's pre-sigmoid output
    (model/enhance_model.py:156); frames t >= input_sizes[b] are zeroed as at :158-163."""
    if not torch.is_tensor(input_sizes):
        input_sizes = torch.as_tensor(np.asarray(input_sizes))
    Y, enh = _FbankFunction.apply(linear_out, mix_inputs, fc, fbank_cmvn, input_sizes,
                                  1 if mask_is_logit else 0, bool(return_enhanced))
    return (Y, enh) if return_enhanced else Y


def global_mean_var(stats, frames):
    """(mean, var) per mel bin from running sums ``stats`` = [sum; sum of squares] (2, M) float64 (any device) over
    ``frames`` frames.  Under utterance-sharded data parallelism (torch.distributed initialised, world > 1) every rank
    accumulated its own utterances: the statistics of the whole set are the sums over the ranks (SURVEY.md 8e) -- ONE
    all-reduce of 2M + 1 doubles -- so every rank returns the same CMVN.  Returns float64 numpy arrays."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        packed = torch.cat([stats.reshape(-1), stats.new_tensor([float(frames)])])
        dist.all_reduce(packed, op=dist.ReduceOp.SUM)
        stats, frames = packed[:-1].view_as(stats), float(packed[-1].item())
    s = stats.cpu().numpy()
    mean = s[0] / frames
    var = s[1] / frames - np.square(mean)
    return mean, var


# ----------------------------------------------------------------------------------------- module
class FFTModel(ModelBase):
    """Base of FbankModel in the reference (model/feat_model.py:36-90).  Only ``compute_cmvn`` is
    inherited by the hot path; the statistics are reduced on the device (re2e_cmvn_stats)."""

    def _init_cmvn_state(self, dim, args):
        self.fbank_cmvn = np.zeros(shape=[2, dim], dtype=np.float32)
        self.cmvn_num = min(args.train_dataset_len, args.num_utt_cmvn)
        self.cmvn_processed_num = 0
        self.frame_count = 0
        self._dev_sum = None
        self._dim = dim

    # reference attributes `sum` / `sum_sq` ([1, dim] float32 numpy): read back on demand
    @property
    def sum(self):
        if self._dev_sum is None:
            return np.zeros([1, self._dim], dtype=np.float32)
        return self._dev_sum[0].cpu().numpy().astype(np.float32)[None, :]

    @property
    def sum_sq(self):
        if self._dev_sum is None:
            return np.zeros([1, self._dim], dtype=np.float32)
        return self._dev_sum[1].cpu().numpy().astype(np.float32)[None, :]

    def compute_cmvn(self, inputs, input_sizes):
        """model/feat_model.py:62-90: accumulate until cmvn_num utterances were seen (returns None),
        then return [[-mean], [1/sqrt(var)]] float32 (2, dim)."""
        if self.cmvn_processed_num < self.cmvn_num:
            features = self.forward(inputs)
            L = _lib.lib()
            dev = features.device
            B, T, M = features.shape
            if self._dev_sum is None:
                self._dev_sum = torch.zeros(2, M, device=dev, dtype=torch.float64)
                self._dev_frames = torch.zeros(1, device=dev, dtype=torch.int64)
            sizes = torch.as_tensor(np.asarray(input_sizes)).to(torch.int32)
            ln = sizes.to(dev, non_blocking=True).contiguous()
            with _lib.on(dev):
                _lib.check(L.re2e_cmvn_stats(_lib.ptr(features.detach()), _lib.ptr(ln),
                                             _lib.ptr(self._dev_sum[0]), _lib.ptr(self._dev_sum[1]),
                                             _lib.ptr(self._dev_frames), B, T, M, _lib.stream_ptr()),
                           "re2e_cmvn_stats")
            self.frame_count += int(sizes.clamp(max=T).sum())
            self.cmvn_processed_num += int(sizes.numel())
            return None
        mean, var = global_mean_var(self._dev_sum, self.frame_count)
        self.fbank_cmvn[0, :] = (-mean).astype(np.float32)
        self.fbank_cmvn[1, :] = (1 / np.sqrt(var)).astype(np.float32)
        return self.fbank_cmvn


class FbankModel(FFTModel):
    """model/feat_model.py:93-135.  ``args`` needs: idim, fbank_dim, enhance_type,
    fbank_opti_type, train_dataset_len, num_utt_cmvn."""

    def __init__(self, args):
        super(FFTModel, self).__init__()
        self.opt = args
        idim = args.idim
        odim = args.fbank_dim
        # 80 filters: the reference's own constants; any other size: Kaldi-style bank by formula (reference: crash)
        filterbanks = reference_fbank80() if odim == 80 else kaldi_mel_banks(num_bins=odim)
        if args.enhance_type == 'unet_128' or args.enhance_type == 'unet_256':
            idim = 256
            filterbanks = filterbanks[:, :256]
        else:
            filterbanks = filterbanks[:, :idim]
        self.fc = torch.nn.Parameter(torch.Tensor(idim, odim))
        self.fc.data.copy_(torch.from_numpy(np.ascontiguousarray(filterbanks.T)))
        if args.fbank_opti_type == 'frozen':
            self.fc.requires_grad_(False)
        self._init_cmvn_state(args.fbank_dim, args)

    def forward(self, xs, fbank_cmvn=None):
        """xs (B,T,idim) non-negative magnitudes (CPU or CUDA; moved like to_cuda does) ->
        (B,T,fbank_dim).  fbank_cmvn: (2,fbank_dim) tensor/ndarray, row 0 = -mean, row 1 = 1/std."""
        if fbank_cmvn is not None and not torch.is_tensor(fbank_cmvn):
            fbank_cmvn = torch.from_numpy(np.asarray(fbank_cmvn, dtype=np.float32))
        if torch.is_tensor(xs) and xs.device != self.fc.device:
            xs = xs.to(self.fc.device)        # to_cuda (model/feat_model.py:124), differentiable: a CPU leaf gets a CPU grad
        return _FbankFunction.apply(None, xs, self.fc, fbank_cmvn, None, 0, False)[0]

    def forward_masked(self, linear_out, mix_inputs, input_sizes, fbank_cmvn=None, return_enhanced=False):
        """Fused EnhanceModel tail + forward (see masked_fbank)."""
        if fbank_cmvn is not None and not torch.is_tensor(fbank_cmvn):
            fbank_cmvn = torch.from_numpy(np.asarray(fbank_cmvn, dtype=np.float32))
        return masked_fbank(linear_out, mix_inputs, input_sizes, self.fc, fbank_cmvn,
                            mask_is_logit=True, return_enhanced=return_enhanced)


def _joint_features(self, linear_out, mix_inputs, clean_inputs, input_sizes, fbank_cmvn=None):
    """enhance_feat, mix_feat, clean_feat of one joint_train.py iteration (:158-161):

        enhance_feat = feat_model(mask-tail(linear_out, mix_inputs, input_sizes), cmvn)     (grad -> linear_out)
        mix_feat     = feat_model(mix_inputs, cmvn)          clean_feat = feat_model(clean_inputs, cmvn)

    One launch reading mask, mix and clean once when the bank is frozen and banded; three calls otherwise."""
    if fbank_cmvn is not None and not torch.is_tensor(fbank_cmvn):
        fbank_cmvn = torch.from_numpy(np.asarray(fbank_cmvn, dtype=np.float32))
    if not torch.is_tensor(input_sizes):
        input_sizes = torch.as_tensor(np.asarray(input_sizes))
    B, T = mix_inputs.shape[0], mix_inputs.shape[1]
    joint = not (self.fc.requires_grad or mix_inputs.requires_grad or clean_inputs.requires_grad)
    # an aligned input stays aligned through f32c (the same buffer, or a fresh copy)
    band = _band_for(self.fc, B, T) if joint and _aligned16(linear_out, mix_inputs, clean_inputs) else None
    if band is not None:
        return _FbankJoint.apply(linear_out, mix_inputs, clean_inputs, self.fc, fbank_cmvn, input_sizes, band)
    enh = masked_fbank(linear_out, mix_inputs, input_sizes, self.fc, fbank_cmvn)
    return enh, self.forward(mix_inputs, fbank_cmvn), self.forward(clean_inputs, fbank_cmvn)


FbankModel.forward_joint = _joint_features


class _MaskApply(torch.autograd.Function):
    @staticmethod
    def forward(ctx, linear_out, mix_inputs, lens):
        L = _lib.lib()
        dev = linear_out.device
        lo = _lib.f32c(linear_out, dev)
        mx = _lib.f32c(mix_inputs, dev)
        ln = lens.to(dev, torch.int32, non_blocking=True).contiguous()
        B, T, F = lo.shape
        out = torch.empty_like(lo)
        with _lib.on(dev):
            _lib.check(L.re2e_mask_apply_fwd(_lib.ptr(lo), _lib.ptr(mx), _lib.ptr(ln), _lib.ptr(out), B, T, F,
                                             _lib.stream_ptr()), "re2e_mask_apply_fwd")
        ctx.save_for_backward(lo, mx, ln)
        return out

    @staticmethod
    def backward(ctx, d_enh):
        L = _lib.lib()
        lo, mx, ln = ctx.saved_tensors
        B, T, F = lo.shape
        d = torch.empty_like(lo)
        with _lib.on(lo.device):
            _lib.check(L.re2e_mask_apply_bwd(_lib.ptr(_lib.f32c(d_enh, lo.device)), _lib.ptr(lo), _lib.ptr(mx),
                                             _lib.ptr(ln), _lib.ptr(d), B, T, F, _lib.stream_ptr()),
                       "re2e_mask_apply_bwd")
        return d, None, None


def apply_mask(linear_out, mix_inputs, input_sizes):
    """Stand-alone tail of EnhanceModel.forward (model/enhance_model.py:157-164):
    sigmoid(linear_out), frames t >= input_sizes[b] zeroed, times mix_inputs -> enhance_out."""
    if not torch.is_tensor(input_sizes):
        input_sizes = torch.as_tensor(np.asarray(input_sizes))
    return _MaskApply.apply(linear_out, mix_inputs, input_sizes)
