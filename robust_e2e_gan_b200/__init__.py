"""B200-native (sm_100a) hot path of Robust_e2e_gan's joint enhancement + ASR training step.

Drop-in classes (same constructors / forward signatures / state_dict keys as the reference's
model/feat_model.py, model/e2e_attention.py, model/e2e_ctc.py):

    FbankModel, AttLoc, CTC, CTCPrefixScore, Decoder (training loop + batched beam search around AttLoc)

plus the fused functional entry points ``masked_fbank`` / ``apply_mask`` for the tail of
EnhanceModel.forward (model/enhance_model.py:157-164).  All arithmetic runs in hand-written CUDA
kernels behind the C ABI of include/re2e_b200.h (robust_e2e_gan_b200/libre2e_b200.so); there is no
CPU, Triton or PyTorch fallback -- calls raise if the library or the GPU is missing.
"""
from .feat_model import FbankModel, FFTModel, fbank, masked_fbank, apply_mask  # noqa: F401
from .e2e_attention import AttLoc  # noqa: F401
from .e2e_ctc import (CTC, CTCPrefixScore, PreparedTargets, prepare_targets, ctc_loss,  # noqa: F401
                      log_softmax_rows, ctc_prefix_score_batch, ctc_forced_align, CTCAlignment)
from .e2e_decoder import Decoder  # noqa: F401
from .parallel import GradBuckets, init_distributed, shard_range  # noqa: F401

__version__ = "0.1.0"
