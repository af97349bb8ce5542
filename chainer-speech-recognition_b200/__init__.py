"""chainer-speech-recognition_b200 -- B200-native CTC / Gram-CTC loss (forward + backward).

The directory name is not a Python identifier; import it with
``importlib.import_module("chainer-speech-recognition_b200")`` or through the alias module
``b200ctc`` at the repository root.  Layout mirrors the reference for the one path it replaces:

    asr/loss/gram_ctc.py   gram_ctc(...)                                (reference: asr/loss/gram_ctc.py)
    asr/loss/ctc.py        connectionist_temporal_classification(...)   (reference: Chainer's, via run/ctc/*)
    asr/loss/layernorm_loss.py  layernorm_ctc(...), layernorm_gram_ctc(...), layernorm_greedy_argmax(...)   (reference: asr/nn/layernorm.py + asr/model/cnn.py:41-44 + the loss)
    asr/data/processing.py labels_to_minibatch(...)   (reference: asr/data/processing.py, label half of features_to_minibatch)
    asr/align.py           ctc_forced_align(...), gram_ctc_forced_align(...)   (Viterbi path of the same lattices; no reference counterpart)
    asr/error.py           compute_minibatch_error(...), compute_character_error_rate(...)   (reference: asr/error.py)
    csrc/                  sm_100a kernels + the C ABI (include/b200ctc.h)
"""
from . import _lib, distributed, synth
from ._build import build
from .asr.loss import (gram_ctc, joint_gram_ctc, GramCTC, connectionist_temporal_classification, ctc,
                       ConnectionistTemporalClassification, greedy_argmax, ctc_host, gram_ctc_host,
                       layernorm_ctc, layernorm_gram_ctc, layernorm_greedy_argmax, GraphedStep)

from .asr.align import Alignment, ctc_forced_align, gram_ctc_forced_align
from .asr.data import labels_to_minibatch
from .asr.error import (compute_minibatch_error, compute_character_error_rate, build_expansion_table,
                        minibatch_error_details)

__all__ = ["Alignment", "ctc_forced_align", "gram_ctc_forced_align", "GraphedStep", "layernorm_ctc", "layernorm_gram_ctc", "layernorm_greedy_argmax", "labels_to_minibatch", "joint_gram_ctc", "compute_minibatch_error", "compute_character_error_rate", "build_expansion_table", "minibatch_error_details",
           "gram_ctc", "GramCTC", "connectionist_temporal_classification", "ctc",
           "ConnectionistTemporalClassification", "greedy_argmax", "ctc_host", "gram_ctc_host", "build", "distributed", "synth"]
