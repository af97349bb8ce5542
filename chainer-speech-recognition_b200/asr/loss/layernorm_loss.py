"""LayerNormalization fused into the loss (SURVEY.md 8f rank 3).

In the reference the last layer of every CTC / Gram-CTC model is
``Convolution2D(ndim_dense, vocab_size, ksize=1)`` followed by ``LayerNormalization(None)``
(run/ctc/cnn/model.py:85-88; asr/nn/nn.py:240-265; asr/nn/layernorm.py:29-61), and ``AcousticModel.__call__`` then makes
a transposed copy of the whole output -- ``swapaxes(1, 3)``, ``reshape``, ``split_axis`` into T arrays of (B, V)
(asr/model/cnn.py:41-44) -- for the loss.  The functions below take the convolution output ``z`` of shape
(B, V, 1, T) (or (B, V, T)) and LayerNormalization's ``gamma`` / ``beta`` and return the loss of
``gamma * normalize_layer(z) + beta``; backward returns ``dz`` in z's own layout plus ``dgamma`` / ``dbeta``.  The
normalised tensor, its transpose and their gradients are never materialised (csrc/layernorm_loss.cu).

    loss = layernorm_ctc(z, ln.gamma, ln.beta, t_batch, ID_BLANK, x_length_batch, t_length_batch)
    # instead of:  y_batch = model(x_batch)  [..., LayerNormalization, swapaxes/reshape/split_axis]
    #              loss = F.connectionist_temporal_classification(y_batch, t_batch, ID_BLANK, x_length_batch, t_length_batch)

    loss = layernorm_gram_ctc(z, ln.gamma, ln.beta, t_batch, bigram_batch, ID_BLANK, x_length_batch, t_length_batch,
                              joint_ctc=args.joint_training)     # Gram-CTC, optionally + CTC (joint training)

    y = layernorm_greedy_argmax(z, ln.gamma, ln.beta)              # the development loop's greedy ids, (B, T)
    # instead of:  y = xp.argmax(model(x, split_into_variables=False).data, axis=2)
"""
import torch

from ... import _lib
from ._function import _flags, _stream_ptr, as_device_tensor, check_blank, check_reduce, label_inputs, resolve_batch_global


class LayerNormLossFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, z, gamma, beta, kind, labels, bigrams, input_length, label_length, blank, reduce, batch_global, group):
        lib = _lib.load()
        B, V, T = z.shape
        Lmax = labels.shape[1]
        dev = z.device
        loss_b = torch.empty(B, dtype=torch.float32, device=dev)
        loss_red = torch.empty((), dtype=torch.float32, device=dev)
        loss_scale = 1.0 / float(batch_global) if reduce == "mean" else 1.0
        nbytes = _lib.ln_workspace_bytes(kind, B, T, V, Lmax)
        workspace = torch.empty(max(nbytes, 16), dtype=torch.uint8, device=dev)
        ptr = lambda t: t.data_ptr() if t is not None else None
        with torch.cuda.device(dev):
            _lib.check(lib.b200ctc_ln_forward(
                kind, z.data_ptr(), z.stride(0), z.stride(1), gamma.data_ptr(), beta.data_ptr(), labels.data_ptr(),
                ptr(bigrams), ptr(input_length), ptr(label_length), blank, B, T, V, Lmax, loss_b.data_ptr(),
                loss_red.data_ptr(), loss_scale, workspace.data_ptr(), workspace.numel(), _flags(), _stream_ptr(dev)))
        ctx.kind, ctx.blank, ctx.reduce, ctx.dims, ctx.batch_global = kind, blank, reduce, (B, T, V, Lmax), batch_global
        ctx.has_bigrams = bigrams is not None
        ctx.save_for_backward(z, gamma, beta, labels, bigrams if bigrams is not None else labels, workspace)
        if reduce == "mean":
            if group is not None:
                import torch.distributed as dist
                dist.all_reduce(loss_red, op=dist.ReduceOp.SUM, group=group)
            return loss_red
        return loss_b

    @staticmethod
    def backward(ctx, gy):
        lib = _lib.load()
        z, gamma, beta, labels, bigrams, workspace = ctx.saved_tensors
        B, T, V, Lmax = ctx.dims
        dev = z.device
        gy = gy.to(device=dev, dtype=torch.float32).contiguous()
        per_utt = 0 if ctx.reduce == "mean" else 1
        scale = 1.0 / float(ctx.batch_global) if ctx.reduce == "mean" else 1.0
        # dz in z's layout; rows must be 16-byte aligned for the kernel's 128-bit stores, so a T that is not a multiple
        # of 4 gets rows with a padded pitch (z itself came in with such a pitch, or the forward call would have refused)
        Tp = (T + 3) & ~3
        dz = torch.empty((B, V, Tp), dtype=z.dtype, device=dev)[:, :, :T]
        dgamma = torch.empty_like(gamma) if ctx.needs_input_grad[1] or ctx.needs_input_grad[2] else None
        dbeta = torch.empty_like(beta) if dgamma is not None else None
        with torch.cuda.device(dev):
            _lib.check(lib.b200ctc_ln_backward(
                ctx.kind, z.data_ptr(), z.stride(0), z.stride(1), gamma.data_ptr(), beta.data_ptr(), labels.data_ptr(),
                bigrams.data_ptr() if ctx.has_bigrams else None, ctx.blank, B, T, V, Lmax, gy.data_ptr(), per_utt, scale,
                dz.data_ptr(), dz.stride(0), dz.stride(1), dgamma.data_ptr() if dgamma is not None else None,
                dbeta.data_ptr() if dbeta is not None else None, workspace.data_ptr(), workspace.numel(), _stream_ptr(dev)))
        return (dz, dgamma if ctx.needs_input_grad[1] else None, dbeta if ctx.needs_input_grad[2] else None) + (None,) * 9


def _layernorm_inputs(z, gamma, beta):
    """z (B, V, 1, T) or (B, V, T) -> a (B, V, T) view with time stride 1; gamma, beta -> float32 (V,) on z's device."""
    z, gamma, beta = as_device_tensor(z), as_device_tensor(gamma), as_device_tensor(beta)
    if not isinstance(z, torch.Tensor) or z.dim() not in (3, 4):
        raise TypeError("z must be the (B, V, 1, T) output of the model's last convolution")
    if z.dtype != torch.float32:
        raise TypeError("activations must be float32, got %s" % z.dtype)
    if not z.is_cuda:
        raise RuntimeError("b200ctc has no CPU path: activations must live on a CUDA device")
    if z.dim() == 4:
        if z.shape[2] != 1:
            raise ValueError("z must have height 1 (B, V, 1, T); got %r" % (tuple(z.shape),))
        z3 = z.squeeze(2)
    else:
        z3 = z
    if z3.stride(2) != 1 and z3.shape[2] > 1:
        z3 = z3.contiguous()
    V = z3.shape[1]
    dev = z3.device
    gamma = gamma.to(device=dev, dtype=torch.float32).reshape(-1).contiguous() if not (
        gamma.device == dev and gamma.dtype == torch.float32 and gamma.dim() == 1 and gamma.is_contiguous()) else gamma
    beta = beta.to(device=dev, dtype=torch.float32).reshape(-1).contiguous() if not (
        beta.device == dev and beta.dtype == torch.float32 and beta.dim() == 1 and beta.is_contiguous()) else beta
    if gamma.numel() != V or beta.numel() != V:
        raise ValueError("gamma and beta must have one entry per vocabulary id (V = %d)" % V)
    return z3, gamma, beta


def _layernorm_loss(kind, z, gamma, beta, labels, bigrams, blank_symbol, input_length, label_length, reduce,
                    batch_global=None, group=None):
    check_reduce(reduce)
    check_blank(blank_symbol)
    z3, gamma, beta = _layernorm_inputs(z, gamma, beta)
    B, V, T = z3.shape
    labels, bigrams, input_length, label_length, blank_symbol = label_inputs(
        kind, B, V, z3.device, labels, bigrams, blank_symbol, input_length, label_length)
    batch_global = resolve_batch_global(B, batch_global, group, reduce, z3.device)
    out = LayerNormLossFunction.apply(z3, gamma, beta, kind, labels, bigrams, input_length, label_length, blank_symbol,
                                      reduce, batch_global, group)
    return out


def layernorm_ctc(z, gamma, beta, t, blank_symbol, input_length=None, label_length=None, reduce="mean", **kw):
    """``connectionist_temporal_classification(split(swapaxes(LayerNormalization(z))), t, ...)`` without the
    normalised tensor or its transpose ever existing.  z: (B, V, 1, T) float32 CUDA tensor (T-contiguous rows that are
    16-byte aligned); gamma, beta: (V,)."""
    return _layernorm_loss(_lib.KIND_CTC, z, gamma, beta, t, None, blank_symbol, input_length, label_length, reduce, **kw)


def layernorm_gram_ctc(z, gamma, beta, label_unigram, label_bigram, blank_symbol, input_length=None, length_unigram=None,
                       reduce="mean", joint_ctc=False, **kw):
    """The same in front of ``gram_ctc`` (asr/loss/gram_ctc.py:300).

    ``joint_ctc=True`` is the joint-training objective of run/gram_ctc/cnn/train.py:196-198 (``args.joint_training``):
    ``gram_ctc(...) + connectionist_temporal_classification(..., label_unigram, ...)`` on the same normalised activations,
    as ``gram_ctc(..., joint_ctc=True)`` computes it.  Per-utterance losses are the sums of the two losses, the reduced
    loss is ``scale * sum_b (gram_b + ctc_b)``, and dz / dgamma / dbeta are the gradients of the sum."""
    kind = _lib.KIND_JOINT if joint_ctc else _lib.KIND_GRAM
    return _layernorm_loss(kind, z, gamma, beta, label_unigram, label_bigram, blank_symbol, input_length,
                           length_unigram, reduce, **kw)


def layernorm_greedy_argmax(z, gamma, beta):
    """The development loop's ``xp.argmax(model(x, split_into_variables=False).data, axis=2)`` (run/ctc/cnn/train.py:232)
    for a model built without its final LayerNormalization: the (B, T) int64 greedy ids of
    ``gamma * normalize_layer(z) + beta`` for every frame, from one read of z.  Takes z, gamma and beta as
    ``layernorm_ctc`` does and raises what it raises; the result goes straight into ``compute_minibatch_error``.
    numpy.argmax rules: the first of equal maxima wins, NaN counts as maximal.  Builds no autograd edge."""
    z3, gamma, beta = _layernorm_inputs(z, gamma, beta)
    z3, gamma, beta = z3.detach(), gamma.detach(), beta.detach()
    B, V, T = z3.shape
    dev = z3.device
    out = torch.empty((B, T), dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.load().b200ctc_ln_greedy_argmax(
            z3.data_ptr(), z3.stride(0), z3.stride(1), gamma.data_ptr(), beta.data_ptr(), B, T, V, out.data_ptr(),
            _stream_ptr(dev)))
    return out
