"""torch.autograd bridge to the C ABI -- the counterpart of the reference's ``chainer.Function``
protocol (asr/loss/gram_ctc.py:219-297): ``forward`` stashes a workspace, ``backward`` consumes it.

Everything that touches numbers happens in libb200ctc.so; this file only validates arguments the way
the reference does (gram_ctc.py:224-227, :230-244, :300-308), moves pointers, and allocates buffers
with torch so that CUDA OOM surfaces as ``torch.cuda.OutOfMemoryError`` (the call sites catch the
CuPy equivalent to shrink the batch, run/ctc/cnn/train.py:204-211).
"""
import collections.abc
import os

import numpy as np
import torch

from ... import _lib


def _flags():
    """B200CTC_NO_CONCURRENT=1: run the lattice kernel behind the softmax/gather kernel instead of next to it
    (include/b200ctc.h, B200CTC_FLAG_SERIAL); read per call so that tests can toggle it."""
    return _lib.FLAG_SERIAL if os.environ.get("B200CTC_NO_CONCURRENT") else _lib.FLAG_NONE


def as_device_tensor(a, name="array"):
    """Any CUDA array -> torch tensor WITHOUT a copy: torch tensors pass through; CuPy arrays and anything else that
    exposes ``__cuda_array_interface__`` are wrapped in place; a Chainer ``Variable`` contributes its ``.array`` /
    ``.data`` (gram_ctc.py:312-313 builds Variables around the same arrays).  This is what lets the reference's own
    training scripts hand their CuPy activations to this library (INTEGRATION.md).  Anything else (NumPy arrays,
    lists) is returned unchanged for the caller to convert."""
    if isinstance(a, torch.Tensor):
        return a
    if hasattr(a, "__cuda_array_interface__"):
        return torch.as_tensor(a, device=torch.device("cuda", torch.cuda.current_device()))
    for attr in ("array", "data"):
        inner = getattr(a, attr, None)
        if isinstance(inner, torch.Tensor) or hasattr(inner, "__cuda_array_interface__"):
            return as_device_tensor(inner, name)
    return a


def _stream_ptr(device):
    return torch.cuda.current_stream(device).cuda_stream


_ws_bytes = {}


def _workspace_bytes(kind, B, T, V, Lmax):
    """b200ctc_workspace_bytes, remembered per shape (a training loop asks for the same few shapes over and over)."""
    key = (kind, B, T, V, Lmax)
    n = _ws_bytes.get(key)
    if n is None:
        n = _ws_bytes[key] = _lib.workspace_bytes(kind, B, T, V, Lmax)
    return n


class _on_device(object):
    """``with torch.cuda.device(dev)`` only when dev is not already the current device (the context manager costs
    several microseconds per use, and a step has two)."""

    def __init__(self, dev):
        self.ctx = None if dev.index is None or dev.index == torch.cuda.current_device() else torch.cuda.device(dev)

    def __enter__(self):
        if self.ctx is not None:
            self.ctx.__enter__()

    def __exit__(self, *exc):
        if self.ctx is not None:
            self.ctx.__exit__(*exc)


class _CaiBlock(object):
    """A (T,B,V) float32 block of device memory described for torch.as_tensor; keeps the frame owners alive."""

    def __init__(self, ptr, shape, strides_bytes, owners):
        self.owners = owners
        self.__cuda_array_interface__ = {"data": (int(ptr), False), "shape": tuple(int(v) for v in shape),
                                         "strides": tuple(int(v) for v in strides_bytes), "typestr": "<f4", "version": 2}


def stack_frames(xs):
    """Sequence of T (B,V) tensors -> one (T,B,V) tensor (gram_ctc.py:272-273).

    If the frames are equally spaced views of one storage (the usual result of splitting a model
    output) the stacked view is recovered without a copy; otherwise torch.stack copies once, as the
    reference's xp.vstack does.
    """
    x0 = xs[0]
    T = len(xs)
    if T == 1:
        return x0.unsqueeze(0)
    try:
        same = all(x.untyped_storage().data_ptr() == x0.untyped_storage().data_ptr() and
                   x.shape == x0.shape and x.stride() == x0.stride() for x in xs)
        if same and not any(x.requires_grad and x.grad_fn is not None for x in xs):
            step = xs[1].storage_offset() - x0.storage_offset()
            if step > 0 and all(xs[t].storage_offset() == x0.storage_offset() + t * step for t in range(T)):
                return torch.as_strided(x0, (T,) + tuple(x0.shape), (step,) + tuple(x0.stride()),
                                        x0.storage_offset())
        if not any(x.requires_grad for x in xs) and x0.is_cuda and x0.dtype == torch.float32:
            # frames wrapped one by one from foreign arrays (CuPy views of one model output): separate storage
            # objects over equally spaced addresses -- describe the whole block through __cuda_array_interface__
            step_b = xs[1].data_ptr() - x0.data_ptr()
            if step_b > 0 and step_b % 4 == 0 and all(
                    x.shape == x0.shape and x.stride() == x0.stride() and x.data_ptr() == x0.data_ptr() + t * step_b
                    for t, x in enumerate(xs)):
                holder = _CaiBlock(x0.data_ptr(), (T,) + tuple(x0.shape),
                                   (step_b,) + tuple(4 * st for st in x0.stride()), xs)
                return torch.as_tensor(holder, device=x0.device)
    except (RuntimeError, AttributeError, TypeError, ValueError):
        pass
    return torch.stack(tuple(xs), dim=0)


def _as_int32(a, device, name):
    if a is None:
        return None
    if isinstance(a, torch.Tensor) and a.dtype == torch.int32 and a.device == device and a.is_contiguous():
        return a                                               # the usual case: nothing to convert
    a = as_device_tensor(a, name)
    if isinstance(a, torch.Tensor):
        if a.dtype.is_floating_point or a.dtype == torch.bool:
            raise TypeError("%s must be an integer array (int32 in the reference), got %s" % (name, a.dtype))
        return a.to(device=device, dtype=torch.int32).contiguous()
    arr = np.asarray(a)
    if arr.dtype.kind not in "iu":
        raise TypeError("%s must be an integer array (int32 in the reference), got %s" % (name, arr.dtype))
    return torch.as_tensor(arr.astype(np.int32), device=device).contiguous()


class LatticeLossFunction(torch.autograd.Function):
    """forward(acts_tbv) -> loss; backward -> d loss / d acts.  acts_tbv is a (T,B,V) *view*: any
    strides over T and B are passed through to the kernels, the vocabulary axis must be dense."""

    @staticmethod
    def forward(ctx, acts, kind, labels, bigrams, input_length, label_length, blank, reduce, batch_global,
                group, want_argmax):
        lib = _lib.load()
        T, B, V = acts.shape
        Lmax = labels.shape[1]
        dev = acts.device
        losses = torch.empty(B + 1, dtype=torch.float32, device=dev)          # [per-utterance losses | reduced loss]
        loss_b, loss_red = losses[:B], losses[B]
        loss_scale = 1.0 / float(batch_global) if reduce == "mean" else 1.0     # gram_ctc.py:280-281
        argmax = torch.empty((B, T), dtype=torch.int64, device=dev) if want_argmax else None
        ptr = lambda t: t.data_ptr() if t is not None else None
        nbytes = _workspace_bytes(kind, B, T, V, Lmax)
        workspace = torch.empty(max(nbytes, 16), dtype=torch.uint8, device=dev)
        with _on_device(dev):
            _lib.check(lib.b200ctc_forward(
                kind, acts.data_ptr(), acts.stride(0), acts.stride(1), labels.data_ptr(), ptr(bigrams),
                ptr(input_length), ptr(label_length), blank, B, T, V, Lmax, loss_b.data_ptr(), loss_red.data_ptr(),
                loss_scale, ptr(argmax), workspace.data_ptr(), workspace.numel(), _flags(), _stream_ptr(dev)))
        ctx.kind, ctx.blank, ctx.reduce, ctx.dims = kind, blank, reduce, (B, T, V, Lmax)
        ctx.batch_global = batch_global
        ctx.save_for_backward(acts, labels, bigrams if bigrams is not None else labels, workspace)
        ctx.has_bigrams = bigrams is not None
        ctx.argmax = argmax
        if reduce == "mean":                                     # gram_ctc.py:280-281 (scaled in-kernel)
            loss = loss_red
            if group is not None:
                import torch.distributed as dist
                dist.all_reduce(loss, op=dist.ReduceOp.SUM, group=group)
            out = loss
        else:                                                    # 'no': per-utterance vector (:279)
            out = loss_b
        if want_argmax:
            ctx.mark_non_differentiable(argmax)
            return out, argmax
        return out

    @staticmethod
    def backward(ctx, gy, *unused):
        lib = _lib.load()
        acts, labels, bigrams, workspace = ctx.saved_tensors
        B, T, V, Lmax = ctx.dims
        dev = acts.device
        if not (gy.dtype == torch.float32 and gy.device == dev and gy.is_contiguous()):
            gy = gy.to(device=dev, dtype=torch.float32).contiguous()
        per_utt = 0 if ctx.reduce == "mean" else 1
        scale = 1.0 / float(ctx.batch_global) if ctx.reduce == "mean" else 1.0     # :291-294
        big_ptr = bigrams.data_ptr() if ctx.has_bigrams else None
        grad = torch.empty_like(acts)
        if grad.stride(2) != 1:
            grad = torch.empty(acts.shape, dtype=acts.dtype, device=dev)
        with _on_device(dev):
            _lib.check(lib.b200ctc_backward(
                ctx.kind, acts.data_ptr(), acts.stride(0), acts.stride(1), labels.data_ptr(), big_ptr,
                ctx.blank, B, T, V, Lmax, gy.data_ptr(), per_utt, scale, grad.data_ptr(), grad.stride(0),
                grad.stride(1), workspace.data_ptr(), workspace.numel(), _stream_ptr(dev)))
        return (grad,) + (None,) * 10


def check_reduce(reduce):
    if reduce not in ("mean", "no"):                             # gram_ctc.py:224-227
        raise ValueError("only 'mean' and 'no' are valid for 'reduce', but '%s' is given" % reduce)


def check_blank(blank_symbol):
    if isinstance(blank_symbol, bool) or not isinstance(blank_symbol, (int, np.integer)):   # gram_ctc.py:303-304
        raise TypeError("blank_symbol must be non-negative integer.")
    return int(blank_symbol)


def label_inputs(kind, B, V, dev, labels, bigrams, blank_symbol, input_length, label_length):
    """Reference-style checks and normalisation of everything but the activations, shared by every loss path and the
    forced alignment: returns the int32 device tensors (labels, bigrams, input_length, label_length) and the blank id."""
    blank_symbol = check_blank(blank_symbol)
    assert blank_symbol >= 0                                     # gram_ctc.py:305
    assert blank_symbol < V                                      # :306
    labels = _as_int32(labels, dev, "labels")                    # :234
    if labels.dim() != 2 or labels.shape[0] != B:
        raise ValueError("labels must have shape (B, Lmax)")
    if kind != _lib.KIND_CTC:
        bigrams = _as_int32(bigrams, dev, "label_bigram")        # :235
        assert labels.shape[1] == bigrams.shape[1]               # :308
        if bigrams.shape != labels.shape:
            raise ValueError("label_bigram must have the shape of label_unigram")
    else:
        bigrams = None
    if input_length is None:
        # gram_ctc.py:310-313 (and Chainer's CTC, which it derives from): when input_length is omitted BOTH lengths
        # default to the full padded widths -- a label_length passed without an input_length is ignored there, so it
        # is ignored here
        label_length = None
    input_length = _as_int32(input_length, dev, "input_length")
    label_length = _as_int32(label_length, dev, "label_length")
    for name, v in (("input_length", input_length), ("label_length", label_length)):
        if v is not None and v.shape != (B,):
            raise ValueError("%s must have shape (B,)" % name)
    return labels, bigrams, input_length, label_length, blank_symbol


def resolve_batch_global(B, batch_global, group, reduce, dev):
    """The denominator of the 'mean' loss: the local batch size, or the sum over `group` of the local batch sizes."""
    if batch_global is None:
        batch_global = B
        if group is not None and reduce == "mean":
            # shards may differ in size (distributed.shard_range): the mean's denominator is the sum of the local
            # batch sizes, agreed on with one small all-reduce (a host sync -- pass batch_global to avoid it)
            import torch.distributed as dist
            n = torch.tensor([B], dtype=torch.int64, device=dev)
            dist.all_reduce(n, op=dist.ReduceOp.SUM, group=group)
            batch_global = int(n.item())
    return batch_global


def lattice_inputs(kind, xs, labels, bigrams, blank_symbol, input_length, label_length, batch_first=False):
    """Reference-style argument checks and normalisation of the losses on activations and of the forced alignment:
    returns the (T,B,V) activation view and the int32 device tensors (acts, labels, bigrams, input_length, label_length,
    blank)."""
    check_blank(blank_symbol)
    if not isinstance(xs, (torch.Tensor, collections.abc.Sequence)):
        xs = as_device_tensor(xs, "xs")                          # CuPy array / Chainer Variable / DLPack capsule owner
    elif not isinstance(xs, torch.Tensor) and len(xs) > 0 and not isinstance(xs[0], torch.Tensor):
        xs = [as_device_tensor(x, "xs[t]") for x in xs]
    if isinstance(xs, torch.Tensor):
        if xs.dim() != 3:
            raise TypeError("xs must be a sequence of (B,V) tensors or one 3-D tensor")
        acts = xs.transpose(0, 1) if batch_first else xs         # -> (T,B,V) view
    elif isinstance(xs, collections.abc.Sequence):               # :301-302
        if len(xs) == 0:
            raise ValueError("xs is empty")
        assert xs[0].dim() == 2                                  # :307
        acts = stack_frames(xs)
    else:
        raise TypeError("xs must be a list of Variables")
    if acts.dtype != torch.float32:                              # :241-242
        raise TypeError("activations must be float32, got %s" % acts.dtype)
    if not acts.is_cuda:
        raise RuntimeError("b200ctc has no CPU path: activations must live on a CUDA device")
    if acts.stride(2) != 1 and acts.shape[2] > 1:
        acts = acts.contiguous()
    T, B, V = acts.shape
    return (acts,) + label_inputs(kind, B, V, acts.device, labels, bigrams, blank_symbol, input_length, label_length)


def lattice_loss(kind, xs, labels, bigrams, blank_symbol, input_length, label_length, reduce,
                 batch_first=False, batch_global=None, group=None, return_argmax=False):
    """Shared front end of ``ctc`` and ``gram_ctc``: reference-style argument checks, then the kernels."""
    check_reduce(reduce)
    acts, labels, bigrams, input_length, label_length, blank_symbol = lattice_inputs(
        kind, xs, labels, bigrams, blank_symbol, input_length, label_length, batch_first)
    batch_global = resolve_batch_global(acts.shape[1], batch_global, group, reduce, acts.device)
    return LatticeLossFunction.apply(acts, kind, labels, bigrams, input_length, label_length, blank_symbol,
                                     reduce, batch_global, group, return_argmax)


def greedy_argmax(y, batch_first=True):
    """``xp.argmax(y.data, axis=2)`` of the evaluation path (run/ctc/cnn/train.py:232): y is (B,T,V)
    (asr/model/cnn.py:45-47) -> (B,T) int64, first maximum wins, NaN is maximal."""
    if not isinstance(y, torch.Tensor) or y.dim() != 3:
        raise TypeError("y must be a 3-D tensor")
    if not y.is_cuda:
        raise RuntimeError("b200ctc has no CPU path: activations must live on a CUDA device")
    if y.dtype != torch.float32:
        raise TypeError("activations must be float32, got %s" % y.dtype)
    y = y.detach()
    v = y if batch_first else y.transpose(0, 1)                  # (B,T,V) view
    if v.stride(2) != 1 and v.shape[2] > 1:
        v = v.contiguous()
    B, T, V = v.shape
    out = torch.empty((B, T), dtype=torch.int64, device=y.device)
    with torch.cuda.device(y.device):
        _lib.check(_lib.load().b200ctc_greedy_argmax(v.data_ptr(), v.stride(1), v.stride(0), B, T, V,
                                                     out.data_ptr(), _stream_ptr(y.device)))
    return out if batch_first else out.transpose(0, 1)
