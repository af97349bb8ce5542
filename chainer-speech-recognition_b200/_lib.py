"""ctypes binding of libb200ctc.so (the C ABI in include/b200ctc.h).

There is deliberately no fallback: if the CUDA library cannot be found (or built), importing the
loss functions raises.  Nothing in this package imports ``oracle/``.
"""
import ctypes
import os

from . import _build

OK, INVALID_ARGUMENT, UNSUPPORTED, CUDA_ERROR, WORKSPACE_TOO_SMALL, OUT_OF_MEMORY = range(6)
KIND_CTC, KIND_GRAM, KIND_JOINT = 0, 1, 2
FLAG_NONE, FLAG_SERIAL = 0, 1

_lib = None


class B200CTCError(RuntimeError):
    pass


def _bind(lib):
    c = ctypes
    lib.b200ctc_version.restype = c.c_int
    lib.b200ctc_last_error.restype = c.c_char_p
    lib.b200ctc_workspace_bytes.restype = c.c_int
    lib.b200ctc_workspace_bytes.argtypes = [c.c_int] * 5 + [c.POINTER(c.c_size_t)]
    lib.b200ctc_forward.restype = c.c_int
    lib.b200ctc_forward.argtypes = [
        c.c_int, c.c_void_p, c.c_int64, c.c_int64, c.c_void_p, c.c_void_p, c.c_void_p, c.c_void_p,
        c.c_int, c.c_int, c.c_int, c.c_int, c.c_int, c.c_void_p, c.c_void_p, c.c_float, c.c_void_p,
        c.c_void_p, c.c_size_t, c.c_uint, c.c_void_p]
    lib.b200ctc_backward.restype = c.c_int
    lib.b200ctc_backward.argtypes = [
        c.c_int, c.c_void_p, c.c_int64, c.c_int64, c.c_void_p, c.c_void_p,
        c.c_int, c.c_int, c.c_int, c.c_int, c.c_int, c.c_void_p, c.c_int, c.c_float,
        c.c_void_p, c.c_int64, c.c_int64, c.c_void_p, c.c_size_t, c.c_void_p]
    lib.b200ctc_ln_workspace_bytes.restype = c.c_int
    lib.b200ctc_ln_workspace_bytes.argtypes = [c.c_int] * 5 + [c.POINTER(c.c_size_t)]
    lib.b200ctc_ln_forward.restype = c.c_int
    lib.b200ctc_ln_forward.argtypes = [
        c.c_int, c.c_void_p, c.c_int64, c.c_int64, c.c_void_p, c.c_void_p, c.c_void_p, c.c_void_p, c.c_void_p, c.c_void_p,
        c.c_int, c.c_int, c.c_int, c.c_int, c.c_int, c.c_void_p, c.c_void_p, c.c_float, c.c_void_p, c.c_size_t, c.c_uint,
        c.c_void_p]
    lib.b200ctc_ln_backward.restype = c.c_int
    lib.b200ctc_ln_backward.argtypes = [
        c.c_int, c.c_void_p, c.c_int64, c.c_int64, c.c_void_p, c.c_void_p, c.c_void_p, c.c_void_p,
        c.c_int, c.c_int, c.c_int, c.c_int, c.c_int, c.c_void_p, c.c_int, c.c_float,
        c.c_void_p, c.c_int64, c.c_int64, c.c_void_p, c.c_void_p, c.c_void_p, c.c_size_t, c.c_void_p]
    lib.b200ctc_align.restype = c.c_int
    lib.b200ctc_align.argtypes = [
        c.c_int, c.c_void_p, c.c_int64, c.c_int64, c.c_void_p, c.c_void_p, c.c_void_p, c.c_void_p,
        c.c_int, c.c_int, c.c_int, c.c_int, c.c_int, c.c_void_p, c.c_void_p, c.c_void_p, c.c_void_p, c.c_void_p,
        c.c_void_p, c.c_size_t, c.c_void_p]
    lib.b200ctc_greedy_argmax.restype = c.c_int
    lib.b200ctc_greedy_argmax.argtypes = [c.c_void_p, c.c_int64, c.c_int64, c.c_int, c.c_int, c.c_int,
                                          c.c_void_p, c.c_void_p]
    lib.b200ctc_ln_greedy_argmax.restype = c.c_int
    lib.b200ctc_ln_greedy_argmax.argtypes = [c.c_void_p, c.c_int64, c.c_int64, c.c_void_p, c.c_void_p, c.c_int, c.c_int,
                                             c.c_int, c.c_void_p, c.c_void_p]
    lib.b200ctc_greedy_error.restype = c.c_int
    lib.b200ctc_greedy_error.argtypes = [c.c_void_p, c.c_void_p, c.c_int, c.c_int, c.c_void_p, c.c_int, c.c_int,
                                         c.c_void_p, c.c_int, c.c_int, c.c_int, c.c_void_p, c.c_void_p, c.c_void_p,
                                         c.c_void_p, c.c_void_p, c.c_void_p, c.c_void_p, c.c_size_t, c.c_void_p]
    lib.b200ctc_edit_distance.restype = c.c_int
    lib.b200ctc_edit_distance.argtypes = [c.c_void_p, c.c_void_p, c.c_int, c.c_void_p, c.c_void_p, c.c_int, c.c_int,
                                          c.c_int, c.c_void_p, c.c_void_p, c.c_void_p, c.c_void_p, c.c_size_t,
                                          c.c_void_p]
    return lib


ERROR_WORKSPACE_BYTES = 256


def library_path():
    return _build.SO_PATH


def load():
    """Load the in-tree library, building it first if it is missing or stale and nvcc exists.

    Several processes may get here at once (one rank per GPU under torchrun): the build goes to a temporary file
    under an exclusive file lock and is moved into place atomically (``_build.build``).  A stale library that
    cannot be rebuilt (no nvcc on this machine) is refused rather than loaded silently -- unless
    ``B200CTC_ALLOW_STALE=1`` says the caller knows."""
    global _lib
    if _lib is not None:
        return _lib
    override = os.environ.get("B200CTC_LIB")                 # development: load a specific build of the library
    if override:
        _lib = _bind(ctypes.CDLL(override))
        return _lib
    path = _build.SO_PATH
    if not _build.is_current():
        if _build.find_nvcc() is not None:
            _build.build()
        elif not os.path.exists(path):
            raise B200CTCError("libb200ctc.so is missing and nvcc is unavailable; run __graft_entry__.build() "
                               "-- there is no CPU fallback")
        elif os.environ.get("B200CTC_ALLOW_STALE") != "1":
            raise B200CTCError("libb200ctc.so does not match csrc/ (stale build stamp) and nvcc is unavailable to "
                               "rebuild it; run __graft_entry__.build() where nvcc exists, or set "
                               "B200CTC_ALLOW_STALE=1 to load it anyway")
    _lib = _bind(ctypes.CDLL(path))
    return _lib


def last_error():
    return load().b200ctc_last_error().decode("utf-8", "replace")


def check(status):
    """Map a status code to the Python exception the reference would have raised (SURVEY.md 8b)."""
    if status == OK:
        return
    msg = last_error()
    if status == INVALID_ARGUMENT:
        raise ValueError(msg)
    if status == UNSUPPORTED:
        raise NotImplementedError(msg)
    if status in (WORKSPACE_TOO_SMALL, OUT_OF_MEMORY):
        import torch
        raise torch.cuda.OutOfMemoryError(msg)
    raise B200CTCError(msg)


def ln_workspace_bytes(kind, B, T, V, Lmax):
    out = ctypes.c_size_t(0)
    check(load().b200ctc_ln_workspace_bytes(kind, B, T, V, Lmax, ctypes.byref(out)))
    return int(out.value)


def workspace_bytes(kind, B, T, V, Lmax):
    out = ctypes.c_size_t(0)
    check(load().b200ctc_workspace_bytes(kind, B, T, V, Lmax, ctypes.byref(out)))
    return int(out.value)
