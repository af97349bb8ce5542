"""Forced alignment: the best path through the CTC / Gram-CTC lattice of a transcription (Viterbi), on the device.

The loss gives the total probability of a transcription over every path through its lattice; the alignment gives
the single most probable path -- where in the audio each label sits, and for Gram-CTC whether the model emits a
bigram or its two unigrams.  Same lattice, same length clamping and the same input forms as the losses
(``connectionist_temporal_classification`` / ``gram_ctc``); nothing here is differentiable.

    a = ctc_forced_align(x, t, blank, input_length, label_length)
    a.score       (B,) float32  -ln P(best path); >= the loss; 1e10 when no alignment exists, NaN on a NaN frame
    a.path        (B,T) int32   lattice node per frame (-1 beyond the input length / without an alignment)
    a.ids         (B,T) int64   vocabulary id per frame (blank where path is -1): minibatch_error_details input
    a.frame_logp  (B,T) float32 ln softmax(x_t)[ids[t]] (0 where path is -1), or None
    a.spans       (B,Lmax,2) int32 [first, last + 1) frame of the node emitting label i ((-1, -1) if none), or None

Lattice nodes: CTC 2i+1 = label i, even = blank; Gram-CTC 3i = blank, 3i+1 = unigram i, 3i+2 = bigram i (labels i-1
and i).  Ties between exactly equal scores are broken deterministically (include/b200ctc.h, b200ctc_align).
"""
import collections

import torch

from .. import _lib
from .loss._function import lattice_inputs, _workspace_bytes, _on_device, _stream_ptr

Alignment = collections.namedtuple("Alignment", "score path ids frame_logp spans")


def _detach(xs):
    if isinstance(xs, torch.Tensor):
        return xs.detach()
    if isinstance(xs, (list, tuple)):
        return [x.detach() if isinstance(x, torch.Tensor) else x for x in xs]
    return xs


def _forced_align(kind, xs, labels, bigrams, blank_symbol, input_length, label_length, batch_first, spans, frame_logp):
    with torch.no_grad():
        acts, labels, bigrams, input_length, label_length, blank = lattice_inputs(
            kind, _detach(xs), labels, bigrams, blank_symbol, input_length, label_length, batch_first)
        lib = _lib.load()
        T, B, V = acts.shape
        Lmax = labels.shape[1]
        dev = acts.device
        score = torch.empty(B, dtype=torch.float32, device=dev)
        path = torch.empty((B, T), dtype=torch.int32, device=dev)
        ids = torch.empty((B, T), dtype=torch.int64, device=dev)
        fl = torch.empty((B, T), dtype=torch.float32, device=dev) if frame_logp else None
        sp = torch.empty((B, Lmax, 2), dtype=torch.int32, device=dev) if spans else None
        ptr = lambda t: t.data_ptr() if t is not None else None
        workspace = torch.empty(max(_workspace_bytes(kind, B, T, V, Lmax), 16), dtype=torch.uint8, device=dev)
        with _on_device(dev):
            _lib.check(lib.b200ctc_align(
                kind, acts.data_ptr(), acts.stride(0), acts.stride(1), labels.data_ptr(), ptr(bigrams),
                ptr(input_length), ptr(label_length), blank, B, T, V, Lmax, score.data_ptr(), path.data_ptr(),
                ids.data_ptr(), ptr(fl), ptr(sp), workspace.data_ptr(), workspace.numel(), _stream_ptr(dev)))
    return Alignment(score, path, ids, fl, sp)


def ctc_forced_align(x, t, blank_symbol, input_length=None, label_length=None, batch_first=False, spans=True,
                     frame_logp=True):
    """Best path of the plain CTC lattice.  Arguments as ``connectionist_temporal_classification``; ``spans`` /
    ``frame_logp`` = False leave those fields None (and unwritten)."""
    return _forced_align(_lib.KIND_CTC, x, t, None, blank_symbol, input_length, label_length, batch_first, spans,
                         frame_logp)


def gram_ctc_forced_align(xs, label_unigram, label_bigram, blank_symbol, input_length=None, length_unigram=None,
                          batch_first=False, spans=True, frame_logp=True):
    """Best path of the Gram-CTC lattice.  Arguments as ``gram_ctc``."""
    return _forced_align(_lib.KIND_GRAM, xs, label_unigram, label_bigram, blank_symbol, input_length, length_unigram,
                         batch_first, spans, frame_logp)
