"""Host-buffer entry points: the counterpart of calling the reference loss with NumPy (CPU) arrays.

The reference's functions accept host arrays and compute on the CPU (`xp = numpy`,
asr/loss/gram_ctc.py:247,285); a user of that path hands over host activations and reads host
gradients.  Here the arithmetic still runs on the GPU: the batch is cut into utterance groups and the
three stages of a group -- activations host->device, loss forward + gradient, gradient device->host --
run on three CUDA streams, so the PCIe transfers in both directions overlap each other and the kernels.
Only valid frames cross PCIe, in both directions: padded frames are never read by the kernels, and their gradient rows
are exactly zero (gram_ctc.py:296), so the host clears those itself -- libc memset (streaming stores) on two helper
threads while the copies are in flight (a NumPy slice assignment needed eight threads for the same work).
Utterances are independent, so grouping changes no result bit-for-bit per utterance.

Layout: host activations are (B,T,V) ("batch first", the decoder layout of asr/model/cnn.py:45-47), which makes
a group a contiguous slab of host memory; pass pinned tensors (``torch.Tensor.pin_memory()``) for the
copies to be asynchronous.
"""
import concurrent.futures
import ctypes
import os

import numpy as np
import torch

from ... import _lib
from ._function import check_blank, check_reduce, label_inputs

_streams = {}
_pool = None


def _zero_pool():
    """Threads that zero the padded gradient rows on the host (NumPy slice assignment releases the GIL)."""
    global _pool
    if _pool is None:
        try:
            n = len(os.sched_getaffinity(0))
        except Exception:
            n = os.cpu_count() or 2
        # two threads keep up with the DMA now that the rows are cleared by libc memset (one does, measured); more only
        # fight the other ranks of a multi-GPU job for the memory system.  B200CTC_HOST_THREADS overrides.
        want = os.environ.get("B200CTC_HOST_THREADS")
        n = int(want) if want else min(2, n)
        _pool = concurrent.futures.ThreadPoolExecutor(max_workers=max(1, n), thread_name_prefix="b200ctc-zero")
    return _pool


def _get_streams(dev):
    key = (dev.type, dev.index)
    if key not in _streams:
        _streams[key] = tuple(torch.cuda.Stream(device=dev) for _ in range(3))
    return _streams[key]


def _raw_forward_backward(kind, acts_tbv, labels, bigrams, in_len, lab_len, blank, loss_scale, grad_scale, grad_tbv,
                          gy_one, stream):
    """One group through the C ABI on `stream`: per-utterance losses + gradient (unit upstream gradient)."""
    lib = _lib.load()
    T, B, V = acts_tbv.shape
    Lmax = labels.shape[1]
    dev = acts_tbv.device
    ws = torch.empty(max(_lib.workspace_bytes(kind, B, T, V, Lmax), 16), dtype=torch.uint8, device=dev)
    loss_b = torch.empty(B, dtype=torch.float32, device=dev)
    loss_red = torch.empty((), dtype=torch.float32, device=dev)
    sp = stream.cuda_stream
    _lib.check(lib.b200ctc_forward(kind, acts_tbv.data_ptr(), acts_tbv.stride(0), acts_tbv.stride(1), labels.data_ptr(),
                                   bigrams.data_ptr() if bigrams is not None else None,
                                   in_len.data_ptr() if in_len is not None else None,
                                   lab_len.data_ptr() if lab_len is not None else None,
                                   blank, B, T, V, Lmax, loss_b.data_ptr(), loss_red.data_ptr(), loss_scale, None,
                                   ws.data_ptr(), ws.numel(), 0, sp))
    _lib.check(lib.b200ctc_backward(kind, acts_tbv.data_ptr(), acts_tbv.stride(0), acts_tbv.stride(1), labels.data_ptr(),
                                    bigrams.data_ptr() if bigrams is not None else None, blank, B, T, V, Lmax,
                                    gy_one.data_ptr(), 0, grad_scale, grad_tbv.data_ptr(), grad_tbv.stride(0),
                                    grad_tbv.stride(1), ws.data_ptr(), ws.numel(), sp))
    for t_ in (ws, loss_b, loss_red):
        t_.record_stream(stream)
    return loss_b, loss_red


def lattice_loss_host(kind, x_host, labels, bigrams, blank_symbol, input_length, label_length, reduce="mean",
                      grad_out=None, groups=16, device=None, gy=1.0):
    """x_host: (B,T,V) float32 host tensor / ndarray.  Returns (loss, grad_host): loss a Python float ('mean') or a
    (B,) ndarray ('no'); grad_host a (B,T,V) host tensor = d loss / d x (times gy)."""
    check_reduce(reduce)
    check_blank(blank_symbol)
    if not torch.cuda.is_available():
        raise RuntimeError("b200ctc has no CPU path: a CUDA device is required")
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    x_host = torch.as_tensor(x_host)
    if x_host.dtype != torch.float32 or x_host.dim() != 3:
        raise TypeError("activations must be a float32 (B,T,V) array")
    x_host = x_host.contiguous()
    B, T, V = x_host.shape
    if grad_out is None:
        grad_out = torch.empty((B, T, V), dtype=torch.float32, pin_memory=True)
    elif not (isinstance(grad_out, torch.Tensor) and grad_out.dtype == torch.float32 and not grad_out.is_cuda and
              tuple(grad_out.shape) == (B, T, V) and grad_out.is_contiguous()):
        raise ValueError("grad_out must be a contiguous float32 host tensor of shape (B,T,V)")
    il_host = None
    if input_length is not None:
        il_host = (input_length.detach().cpu().numpy() if isinstance(input_length, torch.Tensor)
                   else np.asarray(input_length)).astype(np.int64)
    labels, bigrams, input_length, label_length, blank_symbol = label_inputs(
        kind, B, V, dev, labels, bigrams, blank_symbol, input_length, label_length)
    s_in, s_run, s_out = _get_streams(dev)
    cur = torch.cuda.current_stream(dev)
    for s in (s_in, s_run, s_out):
        s.wait_stream(cur)
    x_dev = torch.empty((B, T, V), dtype=torch.float32, device=dev)
    g_dev = torch.empty((B, T, V), dtype=torch.float32, device=dev)
    gy_one = torch.full((), float(gy), dtype=torch.float32, device=dev)
    loss_scale = 1.0 / B if reduce == "mean" else 1.0
    groups = max(1, min(int(groups), B))
    bounds = [B * g // groups for g in range(groups + 1)]
    parts = []
    zero_jobs = []
    if il_host is not None:
        # padded rows of the host gradient: zeroed by the pool while the DMA engines move the valid rows
        g_base, row_bytes = grad_out.data_ptr(), V * 4

        def zero_rows(b, n):               # libc memset: streaming stores, and ctypes drops the GIL for the call
            ctypes.memset(g_base + (b * T + n) * row_bytes, 0, (T - n) * row_bytes)
        pool = _zero_pool()
        for b in range(B):
            n = int(min(max(il_host[b], 0), T))
            if n < T:
                zero_jobs.append(pool.submit(zero_rows, b, n))
    for g in range(groups):
        b0, b1 = bounds[g], bounds[g + 1]
        if b1 == b0:
            continue
        with torch.cuda.stream(s_in):
            if il_host is None:
                x_dev[b0:b1].copy_(x_host[b0:b1], non_blocking=True)
            else:                              # padded frames are never read by the kernels: do not ship them
                for b in range(b0, b1):
                    n = int(min(max(il_host[b], 0), T))
                    if n > 0:
                        x_dev[b, :n].copy_(x_host[b, :n], non_blocking=True)
            e_in = torch.cuda.Event(); e_in.record(s_in)
        with torch.cuda.stream(s_run):
            s_run.wait_event(e_in)
            loss_b, loss_red = _raw_forward_backward(
                kind, x_dev[b0:b1].transpose(0, 1), labels[b0:b1], None if bigrams is None else bigrams[b0:b1],
                None if input_length is None else input_length[b0:b1],
                None if label_length is None else label_length[b0:b1], blank_symbol, loss_scale,
                loss_scale, g_dev[b0:b1].transpose(0, 1), gy_one, s_run)
            parts.append((loss_b, loss_red))
            e_run = torch.cuda.Event(); e_run.record(s_run)
        with torch.cuda.stream(s_out):
            s_out.wait_event(e_run)
            if il_host is None:
                grad_out[b0:b1].copy_(g_dev[b0:b1], non_blocking=True)
            else:
                for b in range(b0, b1):
                    n = int(min(max(il_host[b], 0), T))
                    if n > 0:
                        grad_out[b, :n].copy_(g_dev[b, :n], non_blocking=True)
    with torch.cuda.stream(s_out):
        s_out.wait_stream(s_run)
        if reduce == "mean":
            total = torch.stack([p[1] for p in parts]).sum()
        else:
            total = torch.cat([p[0] for p in parts])
        total_host = total.cpu()
    for t_ in (x_dev, g_dev, gy_one, labels):
        t_.record_stream(s_run); t_.record_stream(s_out)
    s_out.synchronize()
    for j in zero_jobs:
        j.result()
    cur.wait_stream(s_out)
    return (float(total_host) if reduce == "mean" else total_host.numpy()), grad_out


def ctc_host(x, t, blank_symbol, input_length=None, label_length=None, reduce="mean", **kw):
    """Host-array form of ``connectionist_temporal_classification`` (+ its gradient): see module docstring."""
    return lattice_loss_host(_lib.KIND_CTC, x, t, None, blank_symbol, input_length, label_length, reduce, **kw)


def gram_ctc_host(xs, label_unigram, label_bigram, blank_symbol, input_length=None, length_unigram=None,
                  reduce="mean", **kw):
    """Host-array form of ``gram_ctc`` (+ its gradient)."""
    return lattice_loss_host(_lib.KIND_GRAM, xs, label_unigram, label_bigram, blank_symbol, input_length,
                             length_unigram, reduce, **kw)
