"""``asr.loss`` -- drop-in for the reference's ``asr/loss/__init__.py:1`` (which exports ``gram_ctc``)
plus plain CTC, which the reference takes from Chainer (``F.connectionist_temporal_classification``)."""
from .gram_ctc import gram_ctc, joint_gram_ctc, GramCTC                                      # noqa: F401
from .ctc import connectionist_temporal_classification, ctc, ConnectionistTemporalClassification   # noqa: F401
from ._function import greedy_argmax                                         # noqa: F401
from .host import ctc_host, gram_ctc_host                                   # noqa: F401
from .layernorm_loss import layernorm_ctc, layernorm_gram_ctc, layernorm_greedy_argmax   # noqa: F401
from .graphed import GraphedStep                                             # noqa: F401
