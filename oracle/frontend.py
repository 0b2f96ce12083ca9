"""Oracle (CPU restatement) of the differentiable front-end.  TEST INFRASTRUCTURE ONLY.

Follows, line by line:
  * mask tail ............ /root/reference/model/enhance_model.py:157-164
  * FbankModel.forward ... /root/reference/model/feat_model.py:118-135
  * compute_cmvn ......... /root/reference/model/feat_model.py:62-90
  * mel table (generic) .. /root/reference/model/e2e_common.py:104-132
Gradients come from torch autograd over this restatement, exactly as the
reference gets them.  ``dtype=torch.float64`` gives a high-precision arm used
to attribute error between the fp32 reference and the fp32 CUDA kernels.
"""
import numpy as np
import torch


def mask_tail(linear_out, mix_inputs, ilens, mask_is_logit=True):
    """enhance_model.py:157-164 -- sigmoid, zero the frames t >= ilens[b], times mix.  ``mask_is_logit=False``: the
    mask is used as given, without the sigmoid (the kernels' identity activation)."""
    out = torch.sigmoid(linear_out) if mask_is_logit else linear_out
    B, T = out.shape[0], out.shape[1]
    pad = torch.zeros(B, T, 1, dtype=torch.bool)
    for i, length in enumerate(ilens):
        length = int(length)
        if T - length > 0:
            pad[i, length:] = True
    out = out.masked_fill(pad, 0)
    return out * mix_inputs


def fbank_forward(xs, fc, fbank_cmvn=None):
    """feat_model.py:118-135 -- power, (B*T,F)@(F,M), clamp<=1e-7 (zero grad), log, CMVN."""
    xs = xs ** 2
    n, t = xs.size(0), xs.size(1)
    xs = xs.view(n * t, -1)
    xs = torch.mm(xs, fc)
    out = xs.view(n, t, -1)
    # reference does the in-place ``out[out <= 1e-7] = 1e-7`` on a view of the mm
    # result; clone keeps autograd legal on modern torch with the same values/grads.
    out = out.clone()
    out[out <= 1e-7] = 1e-7
    out = torch.log(out)
    if fbank_cmvn is not None:
        out = (out + fbank_cmvn[0, :]) * fbank_cmvn[1, :]
    return out


def masked_fbank_forward(linear_out, mix_inputs, ilens, fc, fbank_cmvn=None, mask_is_logit=True):
    """The fused stage named by north_star: mask tail followed by FbankModel.forward."""
    return fbank_forward(mask_tail(linear_out, mix_inputs, ilens, mask_is_logit), fc, fbank_cmvn)


class CmvnAccumulator(object):
    """feat_model.py:62-90 running sums; returns [[-mean],[1/sqrt(var)]] float32 (2,M)."""

    def __init__(self, odim, cmvn_num):
        self.sum = np.zeros([1, odim], dtype=np.float32)
        self.sum_sq = np.zeros([1, odim], dtype=np.float32)
        self.fbank_cmvn = np.zeros([2, odim], dtype=np.float32)
        self.cmvn_num = cmvn_num
        self.cmvn_processed_num = 0
        self.frame_count = 0

    def update(self, features, input_sizes):
        """features: (B,T,M) output of fbank_forward without cmvn."""
        if self.cmvn_processed_num < self.cmvn_num:
            for x in range(len(input_sizes)):
                input_size = int(input_sizes[x])
                feature_mat = features[x].detach().cpu().numpy()[:input_size, :]
                self.sum = np.add(self.sum, np.sum(feature_mat, axis=0))
                self.sum_sq = np.add(self.sum_sq, np.sum(np.square(feature_mat), axis=0))
                self.frame_count += feature_mat.shape[0]
                self.cmvn_processed_num += 1
            return None
        mean = self.sum / self.frame_count
        var = self.sum_sq / self.frame_count - np.square(mean)
        self.fbank_cmvn[0, :] = -mean
        self.fbank_cmvn[1, :] = 1 / np.sqrt(var)
        return self.fbank_cmvn


def mel_filterbank_generic(nfilt=40, nfft=512, samplerate=16000, lowfreq=0, highfreq=None):
    """e2e_common.py:104-132 triangular mel bank (nfilt, nfft/2+1), float64."""
    def hz2mel(hz):
        return 2595 * np.log10(1 + hz / 700.)

    def mel2hz(mel):
        return 700 * (10 ** (mel / 2595.0) - 1)

    highfreq = highfreq or samplerate / 2
    melpoints = np.linspace(hz2mel(lowfreq), hz2mel(highfreq), nfilt + 2)
    bins = np.floor((nfft + 1) * mel2hz(melpoints) / samplerate)
    fbank = np.zeros([nfilt, nfft // 2 + 1])
    for j in range(nfilt):
        for i in range(int(bins[j]), int(bins[j + 1])):
            fbank[j, i] = (i - bins[j]) / (bins[j + 1] - bins[j])
        for i in range(int(bins[j + 1]), int(bins[j + 2])):
            fbank[j, i] = (bins[j + 2] - i) / (bins[j + 2] - bins[j + 1])
    return fbank
