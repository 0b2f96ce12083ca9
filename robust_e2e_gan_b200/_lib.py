"""ctypes binding of the C-ABI in include/re2e_b200.h.

There is NO fallback: if ``libre2e_b200.so`` is missing, or a call is made
without a CUDA device, this module raises.  Build the library with
``python -c "import __graft_entry__ as g; g.build()"`` (or ``make -C
robust_e2e_gan_b200/csrc``).
"""
import ctypes
import os
import re
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libre2e_b200.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "re2e_b200.h")

_c = ctypes
_P = _c.c_void_p
_I = _c.c_int
_LL = _c.c_longlong
_F = _c.c_float
_SZ = _c.c_size_t

# name -> (restype, argtypes); kept in the order of the header
SIGNATURES = {
    "re2e_abi_version": (_I, []),
    "re2e_build_info": (_c.c_char_p, []),
    "re2e_error_string": (_c.c_char_p, [_I]),
    "re2e_launch_count": (_c.c_ulonglong, []),
    "re2e_fbank_fwd": (_I, [_P, _I, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "re2e_fbank_bwd": (_I, [_P, _P, _P, _I, _P, _P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "re2e_fbank_band_supported": (_I, [_I] * 4),
    "re2e_fbank_band_fwd": (_I, [_P, _I] + [_P] * 10 + [_I] * 4 + [_P]),
    "re2e_fbank_band_bwd": (_I, [_P, _P, _P, _I] + [_P] * 5 + [_I] * 4 + [_P]),
    "re2e_mask_apply_fwd": (_I, [_P, _P, _P, _P, _I, _I, _I, _P]),
    "re2e_mask_apply_bwd": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _P]),
    "re2e_cmvn_stats": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _P]),
    "re2e_attloc_init_att": (_I, [_P, _P, _I, _I, _P]),
    "re2e_attloc_step_supported": (_I, [_I] * 7 + [_P, _P]),
    "re2e_attloc_step_fwd": (_I, [_P] * 9 + [_F] + [_P] * 5 + [_I] * 7 + [_P]),
    "re2e_attloc_acc_floats": (_SZ, [_I, _I, _I]),
    "re2e_attloc_acc_slots": (_I, [_I] * 7),
    "re2e_attloc_step_bwd": (_I, [_P] * 12 + [_F, _P, _I] + [_P] * 4 + [_I] * 8 + [_P]),
    "re2e_attloc_acc_reduce": (_I, [_P, _I, _P, _I, _I, _I, _P]),
    "re2e_attloc_enc_grad": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "re2e_attloc_loop_supported": (_I, [_I] * 7),
    "re2e_attloc_loop_slots": (_I, [_I] * 7),
    "re2e_attloc_loop_fwd": (_I, [_P] * 8 + [_F] + [_P] * 3 + [_I] * 7 + [_P]),
    "re2e_attloc_loop_bwd": (_I, [_P] * 11 + [_F] + [_P] * 3 + [_I] * 8 + [_P]),
    "re2e_batch_nt": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "re2e_sample_tokens_ws_bytes": (_I, [_I]),
    "re2e_sample_tokens": (_I, [_P] * 6 + [_I, _I, _I, _P]),
    "re2e_beam_gather": (_I, [_P, _P, _I, _I, _P, _P, _P, _P, _P]),
    "re2e_log_softmax_topk": (_I, [_P, _LL, _I, _I, _P, _P, _P, _P]),
    "re2e_beam_advance": (_I, [_P, _P, _P, _P, _P, _F, _F, _I, _I, _I, _P, _P, _P, _I, _I, _I, _P, _P, _P, _P, _P]),
    "re2e_cross_entropy_fwd": (_I, [_P, _LL, _P, _LL, _LL, _I, _P, _P, _P, _P]),
    "re2e_cross_entropy_bwd": (_I, [_P, _LL, _P, _LL, _LL, _I, _P, _P, _P, _LL, _P]),
    "re2e_beam_init": (_I, [_P] * 9 + [_I] * 6 + [_P]),
    "re2e_beam_merge": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "re2e_beam_joint": (_I, [_P, _P, _P, _P, _P, _F, _F, _I, _I, _I, _P, _P]),
    "re2e_lstm_step_supported": (_I, [_I, _I, _I]),
    "re2e_lstm_step_fwd": (_I, [_P] * 9 + [_I, _I, _I, _P]),
    "re2e_lstm_step_bwd": (_I, [_P] * 4 + [_I, _I, _I, _P]),
    "re2e_lstm_pointwise_fwd": (_I, [_P] * 5 + [_I, _I, _P]),
    "re2e_lstm_pointwise_bwd": (_I, [_P] * 7 + [_I, _I, _P]),
    "re2e_gemm_tf32x3": (_I, [_P, _I, _I, _P, _I, _I, _P, _I, _P, _I, _I, _I, _I, _P]),
    "re2e_colsum_blocks": (_I, [_I]),
    "re2e_colsum": (_I, [_P, _LL, _I, _I, _P, _P, _P]),
    "re2e_ctc_ws_bytes": (_SZ, [_I, _I, _I, _I]),
    "re2e_ctc_loss_fwd": (_I, [_P, _LL, _LL, _P, _P, _P, _P, _I, _P, _P, _P, _SZ, _I, _I, _I, _I, _P]),
    "re2e_ctc_loss_bwd": (_I, [_P, _LL, _LL, _P, _P, _P, _P, _I, _P, _P, _P, _SZ, _P, _I, _I, _I, _I, _P]),
    "re2e_ctc_align": (_I, [_P, _LL, _LL, _P, _P, _P, _P, _I, _P, _P, _P, _P, _P, _SZ, _I, _I, _I, _I, _P]),
    "re2e_log_softmax": (_I, [_P, _P, _P, _LL, _I, _P]),
    "re2e_ctc_prefix_score": (_I, [_P] * 7 + [_I] * 6 + [_P]),
}

_lock = threading.Lock()
_handle = None


def header_symbols():
    """Every function name declared in include/re2e_b200.h (used by the CPU export test)."""
    with open(HEADER_PATH) as f:
        text = f.read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(re2e_[a-z0-9_]+)\s*\(", text)))


def load():
    """dlopen the library and attach prototypes.  Does not need a GPU."""
    global _handle
    with _lock:
        if _handle is None:
            if not os.path.exists(LIB_PATH):
                raise RuntimeError(
                    "robust_e2e_gan_b200: %s not found -- the sm_100a extension is not built "
                    "(run __graft_entry__.build()); there is no CPU or PyTorch fallback." % LIB_PATH)
            h = ctypes.CDLL(LIB_PATH)
            for name, (res, args) in SIGNATURES.items():
                fn = getattr(h, name)
                fn.restype = res
                fn.argtypes = args
            _handle = h
    return _handle


def lib():
    """The loaded library, for compute calls: additionally requires a CUDA device."""
    if not torch.cuda.is_available():
        raise RuntimeError("robust_e2e_gan_b200: no CUDA device -- the hot path has no CPU fallback")
    return load()


def check(rc, what=""):
    if rc != 0:
        msg = load().re2e_error_string(int(rc)).decode()
        raise RuntimeError("%s failed: %s (code %d)" % (what or "re2e call", msg, rc))


_get_device = getattr(torch._C, "_cuda_getDevice", None)
_set_device = getattr(torch._C, "_cuda_setDevice", None)
_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def stream_ptr():
    """Handle of torch's current stream on the current device.  The raw query is ~40x cheaper than
    torch.cuda.current_stream() (which builds a Stream object and resolves the device index in Python); a decoder loop
    makes several hundred of these calls per step."""
    if _raw_stream is not None and _get_device is not None:
        return ctypes.c_void_p(_raw_stream(_get_device()))
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


class on(object):
    """``with on(device):`` -- make ``device`` current for the calls inside, like torch.cuda.device(device) but free when
    it already is (the usual case: one process per GPU)."""
    __slots__ = ("idx", "prev")

    def __init__(self, device):
        self.idx = device.index if isinstance(device, torch.device) else int(device)
        self.prev = -1

    def __enter__(self):
        if self.idx is None or _get_device is None:
            return self
        cur = _get_device()
        if cur != self.idx:
            self.prev = cur
            _set_device(self.idx)
        return self

    def __exit__(self, *exc):
        if self.prev >= 0:
            _set_device(self.prev)
            self.prev = -1
        return False


def ptr(t):
    """Raw device pointer of a tensor (None -> NULL) as a plain int (ctypes converts it for the declared void* argument).
    Tensors must be CUDA fp32/int32 contiguous."""
    return None if t is None else t.data_ptr()


def launch_count():
    return int(load().re2e_launch_count())


def f32c(t, device=None):
    """Contiguous fp32 CUDA view/copy of ``t`` (moves CPU tensors like the reference's to_cuda)."""
    if device is not None and t.device != device:
        t = t.to(device, non_blocking=True)
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()
