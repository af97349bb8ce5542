"""Run the reference's own ``asr/loss/gram_ctc.py`` UNMODIFIED on its NumPy path.

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).  Needs the reference's files: ``/root/reference``
in the build container, or the unmodified copies staged under ``oracle/_ref/`` by ``__graft_entry__.build()``
(git-ignored) on the GPU box.  Nothing under ``-m gpu`` tests or ``smoke()`` calls this; ``bench.py`` uses it only
as the timed CPU baseline (``--impl reference`` and the ``cpu_baseline`` leg).  It exists to (1) pin
oracle/lattice.py and oracle/ctc_oracle.c, (2) generate the committed golden vectors
(tests/golden/generate_golden.py) and (3) be that baseline.

The reference file needs only a handful of Chainer symbols (SURVEY.md section 8c):
``chainer.is_debug`` (gram_ctc.py:255), ``chainer.cuda.get_array_module`` (:247,285,311),
``chainer.function.Function`` (:219), ``chainer.utils.force_array`` (:281),
``chainer.utils.type_check`` (import only) and ``chainer.variable.Variable`` (:312-313).
Chainer and CuPy are not installable here (no network), so a tiny stand-in for exactly those
symbols is registered in ``sys.modules`` before the file is loaded with importlib.
"""
import collections
import collections.abc
import importlib.util
import os
import sys
import types

import numpy as np

# Where the reference lives: the mounted checkout in the build container; on the GPU box (no /root/reference) the
# unmodified copies of the few files of the path that __graft_entry__.build() staged under oracle/_ref/ (git-ignored,
# never part of the repository; it travels with the snapshot like the built .so files) -- bench.py's reference arm
# times the reference's own NumPy path from there.
_STAGED = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")
REFERENCE_ROOT = os.environ.get("B200CTC_REFERENCE_ROOT") or (
    "/root/reference" if os.path.isfile("/root/reference/asr/loss/gram_ctc.py") else _STAGED)
STAGED_FILES = ("asr/loss/gram_ctc.py", "asr/error.py", "asr/vocab.py", "asr/utils.py", "asr/nn/layernorm.py",
                "asr/data/processing.py")


def stage(src_root=None):
    """Copy the reference files of the path, unmodified, from src_root (default: the checkout REFERENCE_ROOT names)
    into oracle/_ref/."""
    import shutil
    src_root = src_root or REFERENCE_ROOT
    if os.path.abspath(src_root) == _STAGED or not os.path.isfile(os.path.join(src_root, "asr", "loss", "gram_ctc.py")):
        return False
    for rel in STAGED_FILES:
        dst = os.path.join(_STAGED, rel)
        os.makedirs(os.path.dirname(dst), exist_ok=True)
        shutil.copyfile(os.path.join(src_root, rel), dst)
    return True
_REF_FILE = os.path.join(REFERENCE_ROOT, "asr", "loss", "gram_ctc.py")
_module = None


def available():
    return os.path.isfile(_REF_FILE)


def _install_chainer_stub():
    if "chainer" in sys.modules and getattr(sys.modules["chainer"], "_b200ctc_stub", False):
        return
    if not hasattr(collections, "Sequence"):          # gram_ctc.py:301 (removed in Python 3.10)
        collections.Sequence = collections.abc.Sequence

    class Variable(object):
        def __init__(self, data):
            self.data = data

        @property
        def shape(self):
            return self.data.shape

    class Function(object):
        def __call__(self, *inputs):
            arrays = tuple(i.data if isinstance(i, Variable) else np.asarray(i) for i in inputs)
            return Variable(self.forward(arrays)[0])

    chainer = types.ModuleType("chainer")
    chainer._b200ctc_stub = True
    chainer.is_debug = lambda: False
    cuda = types.ModuleType("chainer.cuda")
    cuda.get_array_module = lambda *a: np
    cuda.cupy = None
    function = types.ModuleType("chainer.function")
    function.Function = Function
    utils = types.ModuleType("chainer.utils")
    utils.force_array = lambda x, dtype=None: np.asarray(x)
    type_check = types.ModuleType("chainer.utils.type_check")
    utils.type_check = type_check
    variable = types.ModuleType("chainer.variable")
    variable.Variable = Variable
    chainer.cuda, chainer.function, chainer.utils, chainer.variable = cuda, function, utils, variable
    for name, mod in (("chainer", chainer), ("chainer.cuda", cuda), ("chainer.function", function),
                      ("chainer.utils", utils), ("chainer.utils.type_check", type_check),
                      ("chainer.variable", variable)):
        sys.modules[name] = mod


def load():
    """Return the reference module object (cached)."""
    global _module
    if _module is None:
        if not available():
            raise RuntimeError("reference not mounted at %s" % REFERENCE_ROOT)
        _install_chainer_stub()
        spec = importlib.util.spec_from_file_location("_ref_gram_ctc", _REF_FILE)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        _module = mod
    return _module


def run_gram_ctc(x_tbv, unigram, bigram, input_length, label_length, blank=0, reduce="no", gy=None):
    """Reference forward+backward.  x_tbv: (T,B,V) float32.  Returns (loss, grad (T,B,V), prob_trans).

    Inputs are passed in the Function's own order (gram_ctc.py:248-253).  A fresh GramCTC object is
    used per call because backward mutates the saved softmax in place (gram_ctc.py:290-296).
    """
    ref = load()
    x_tbv = np.ascontiguousarray(x_tbv, dtype=np.float32)
    T, B, V = x_tbv.shape
    xs = tuple(x_tbv[t].copy() for t in range(T))
    f = ref.GramCTC(int(blank), reduce)
    inputs = (np.asarray(input_length, np.int32), np.asarray(label_length, np.int32),
              np.asarray(unigram, np.int32), np.asarray(bigram, np.int32)) + xs
    loss = np.array(f.forward(inputs)[0], copy=True)
    prob_trans = np.array(f.prob_trans, copy=True)
    if gy is None:
        gy = np.ones((B,), np.float32) if reduce == "no" else np.float32(1.0)
    grads = f.backward(inputs, (gy,))
    assert all(g is None for g in grads[:4])          # gram_ctc.py:297
    grad = np.stack(grads[4:]).astype(np.float32)
    return loss, grad, prob_trans


def run_ctc(x_tbv, labels, input_length, label_length, blank=0, reduce="no", gy=None):
    """Plain CTC through the reference: every bigram node dead (gram_ctc.py:95-98)."""
    labels = np.asarray(labels, np.int32)
    return run_gram_ctc(x_tbv, labels, np.full_like(labels, -1), input_length, label_length,
                        blank=blank, reduce=reduce, gy=gy)


_error_modules = None


def load_error_module():
    """The reference's asr/error.py and asr/vocab.py, UNMODIFIED, loaded as the synthetic package ``_refasr``
    (asr/error.py:4-5 uses relative imports of .utils and .vocab; both are pure Python).  Returns (error, vocab)."""
    global _error_modules
    if _error_modules is None:
        if not available():
            raise RuntimeError("reference not mounted at %s" % REFERENCE_ROOT)
        pkg = types.ModuleType("_refasr")
        pkg.__path__ = [os.path.join(REFERENCE_ROOT, "asr")]
        sys.modules["_refasr"] = pkg
        mods = {}
        for name in ("utils", "vocab", "error"):
            spec = importlib.util.spec_from_file_location("_refasr." + name, os.path.join(REFERENCE_ROOT, "asr", name + ".py"))
            mod = importlib.util.module_from_spec(spec)
            sys.modules["_refasr." + name] = mod
            spec.loader.exec_module(mod)
            mods[name] = mod
        _error_modules = (mods["error"], mods["vocab"])
    return _error_modules


_processing_module = None


def load_processing_module():
    """The reference's asr/data/processing.py, UNMODIFIED.  It imports chainer (stubbed above), jaconv, acoustics and
    asr/fft.py (python_speech_features): none of them is needed by ``Processor.features_to_minibatch``, so empty
    stand-ins are registered.  Returns the module."""
    global _processing_module
    if _processing_module is None:
        _install_chainer_stub()
        load_error_module()                                   # registers _refasr, _refasr.utils, _refasr.vocab
        for name in ("jaconv", "acoustics"):
            sys.modules.setdefault(name, types.ModuleType(name))
        fft = types.ModuleType("_refasr.fft")
        fft.get_filterbanks = lambda **kw: None                # Processor.__init__ (:65) builds a mel filterbank: unused here
        sys.modules.setdefault("_refasr.fft", fft)
        sys.modules["_refasr"].fft = sys.modules["_refasr.fft"]
        data = types.ModuleType("_refasr.data")
        data.__path__ = [os.path.join(REFERENCE_ROOT, "asr", "data")]
        sys.modules["_refasr.data"] = data
        spec = importlib.util.spec_from_file_location("_refasr.data.processing",
                                                      os.path.join(REFERENCE_ROOT, "asr", "data", "processing.py"))
        mod = importlib.util.module_from_spec(spec)
        sys.modules["_refasr.data.processing"] = mod
        spec.loader.exec_module(mod)
        _processing_module = mod
    return _processing_module


_layernorm_module = None


def _backward_one(xp, shape, dtype, g):
    """``chainer.functions.array.broadcast._backward_one`` (third-party: Chainer, version unpinned "Chainer 2+",
    README.md:14; imported by asr/nn/layernorm.py:6).  Its published behaviour -- the backward of ``broadcast_to``:
    sum the gradient over the leading axes the broadcast added and over every axis whose input extent was 1,
    keeping those axes -- restated here because Chainer is not installable offline."""
    g = xp.asarray(g)
    ndim = len(shape)
    if g.ndim != ndim:
        g = g.sum(axis=tuple(range(g.ndim - ndim)))
    axis = tuple(i for i, sx in enumerate(shape) if sx == 1)
    if axis:
        g = g.sum(keepdims=True, axis=axis)
    return g.astype(dtype, copy=False)


def load_layernorm_module():
    """The reference's asr/nn/layernorm.py, UNMODIFIED (NumPy path).  Needs ``chainer.function.Function`` (with
    ``retain_inputs``), ``chainer.cuda.get_array_module`` and ``_backward_one`` (above)."""
    global _layernorm_module
    if _layernorm_module is None:
        if not os.path.isfile(os.path.join(REFERENCE_ROOT, "asr", "nn", "layernorm.py")):
            raise RuntimeError("reference not available at %s" % REFERENCE_ROOT)
        _install_chainer_stub()
        chainer = sys.modules["chainer"]
        if not hasattr(chainer.function.Function, "retain_inputs"):
            chainer.function.Function.retain_inputs = lambda self, idx: None          # layernorm.py:34
        chainer.function.cuda = chainer.cuda                                           # "from chainer import function, cuda"
        functions = types.ModuleType("chainer.functions")
        array = types.ModuleType("chainer.functions.array")
        broadcast = types.ModuleType("chainer.functions.array.broadcast")
        broadcast._backward_one = _backward_one
        array.broadcast = broadcast
        functions.array = array
        chainer.functions = functions
        sys.modules.setdefault("chainer.functions", functions)
        sys.modules.setdefault("chainer.functions.array", array)
        sys.modules.setdefault("chainer.functions.array.broadcast", broadcast)
        spec = importlib.util.spec_from_file_location("_ref_layernorm", os.path.join(REFERENCE_ROOT, "asr", "nn", "layernorm.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        _layernorm_module = mod
    return _layernorm_module


def run_layernorm_ctc(z_bv1t, gamma, beta, unigram, bigram, input_length, label_length, blank=0, reduce="no", gy=None):
    """The reference's model tail + loss, forward and backward, every piece the reference's own code:
    NormalizeLayer (asr/nn/layernorm.py) -> scale/bias by gamma/beta (asr/nn/nn.py:265; Chainer's scale/bias are
    broadcast multiplies/adds along axis 1) -> swapaxes/reshape/split (asr/model/cnn.py:41-44) -> GramCTC
    (asr/loss/gram_ctc.py).  z_bv1t: (B, V, 1, T) float32.  Returns loss, dz (B,V,1,T), dgamma, dbeta, activations."""
    ln = load_layernorm_module()
    z = np.ascontiguousarray(z_bv1t, np.float32)
    gamma = np.asarray(gamma, np.float32)
    beta = np.asarray(beta, np.float32)
    B, V, H, T = z.shape
    f = ln.NormalizeLayer()
    n = f.forward((z,))[0]                                             # (B, V, 1, T)
    y = n * gamma[None, :, None, None] + beta[None, :, None, None]     # nn.py:265
    out = np.swapaxes(y, 1, 3).reshape(B, -1)                          # cnn.py:42-43
    xs = np.split(out, T, axis=1)                                      # cnn.py:44: T arrays (B, V)
    x_tbv = np.stack(xs).astype(np.float32)
    loss, grad_tbv, _ = run_gram_ctc(x_tbv, unigram, bigram, input_length, label_length, blank=blank, reduce=reduce, gy=gy)
    g_out = np.concatenate([grad_tbv[t] for t in range(T)], axis=1)    # backward of split_axis
    g_y = np.swapaxes(g_out.reshape(B, T, H, V), 1, 3)                  # backward of reshape / swapaxes: (B, V, 1, T)
    dbeta = g_y.sum(axis=(0, 2, 3))                                    # bias backward
    dgamma = (g_y * n).sum(axis=(0, 2, 3))                             # scale backward
    dn = np.ascontiguousarray(g_y * gamma[None, :, None, None], np.float32)
    dz = f.backward((z,), (dn,))[0]
    return loss, np.asarray(dz, np.float32), dgamma.astype(np.float32), dbeta.astype(np.float32), x_tbv
