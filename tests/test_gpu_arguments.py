"""-m gpu: every loss entry point and both forced alignments check their labels, bigrams, lengths and blank id the way
``ctc`` / ``gram_ctc`` do (asr/loss/_function.py, label_inputs): the same malformed argument raises the same exception
type whichever path it is handed to, before anything is launched."""
import importlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

B, T, V, L = 3, 12, 16, 3


def pkg_():
    return importlib.import_module("chainer-speech-recognition_b200")


def problem():
    rs = np.random.RandomState(3)
    return dict(x=rs.randn(B, T, V).astype(np.float32),                     # (B,T,V)
                gamma=(1.0 + 0.1 * rs.randn(V)).astype(np.float32), beta=(0.1 * rs.randn(V)).astype(np.float32),
                labels=rs.randint(1, V, size=(B, L)).astype(np.int32),
                bigrams=rs.randint(1, V, size=(B, L)).astype(np.int32),
                input_length=np.array([T, T - 2, T - 4], np.int32), label_length=np.array([L, L - 1, 1], np.int32))


def call(entry, labels, bigrams, blank, input_length, label_length, p):
    """One call of `entry` on the activations of `p` and the given label-side arguments."""
    import torch
    pkg = pkg_()
    dev = torch.device("cuda:0")
    x = torch.tensor(p["x"], device=dev).transpose(0, 1)                   # (T,B,V) view
    z = torch.tensor(p["x"].transpose(0, 2, 1).copy(), device=dev).unsqueeze(2)      # (B,V,1,T)
    g, b = torch.tensor(p["gamma"], device=dev), torch.tensor(p["beta"], device=dev)
    host = torch.from_numpy(p["x"])
    if entry == "ctc":
        return pkg.ctc(x, labels, blank, input_length, label_length, reduce="no")
    if entry == "gram_ctc":
        return pkg.gram_ctc(x, labels, bigrams, blank, input_length, label_length, reduce="no")
    if entry == "joint_gram_ctc":
        return pkg.gram_ctc(x, labels, bigrams, blank, input_length, label_length, reduce="no", joint_ctc=True)
    if entry == "layernorm_ctc":
        return pkg.layernorm_ctc(z, g, b, labels, blank, input_length, label_length, reduce="no")
    if entry == "layernorm_gram_ctc":
        return pkg.layernorm_gram_ctc(z, g, b, labels, bigrams, blank, input_length, label_length, reduce="no")
    if entry == "layernorm_joint_gram_ctc":
        return pkg.layernorm_gram_ctc(z, g, b, labels, bigrams, blank, input_length, label_length, reduce="no",
                                      joint_ctc=True)
    if entry == "ctc_host":
        return pkg.ctc_host(host, labels, blank, input_length, label_length, reduce="no")
    if entry == "gram_ctc_host":
        return pkg.gram_ctc_host(host, labels, bigrams, blank, input_length, label_length, reduce="no")
    if entry == "ctc_forced_align":
        return pkg.ctc_forced_align(x, labels, blank, input_length, label_length)
    if entry == "gram_ctc_forced_align":
        return pkg.gram_ctc_forced_align(x, labels, bigrams, blank, input_length, label_length)
    raise AssertionError(entry)


ENTRIES = ["ctc", "gram_ctc", "joint_gram_ctc", "layernorm_ctc", "layernorm_gram_ctc", "layernorm_joint_gram_ctc",
           "ctc_host", "gram_ctc_host", "ctc_forced_align", "gram_ctc_forced_align"]
GRAM_ENTRIES = [e for e in ENTRIES if "gram" in e]

# (name, what to change, exception ctc / gram_ctc raise)
MALFORMED = [
    ("short_input_length", lambda a: dict(a, input_length=a["input_length"][:B - 1]), ValueError),
    ("short_label_length", lambda a: dict(a, label_length=a["label_length"][:B - 1]), ValueError),
    ("long_label_length", lambda a: dict(a, label_length=np.full(B + 1, L, np.int32)), ValueError),
    ("labels_of_fewer_utterances", lambda a: dict(a, labels=a["labels"][:B - 1]), ValueError),
    ("one_dimensional_labels", lambda a: dict(a, labels=a["labels"][0]), ValueError),
    ("float_labels", lambda a: dict(a, labels=a["labels"].astype(np.float32)), TypeError),
    ("float_input_length", lambda a: dict(a, input_length=a["input_length"].astype(np.float32)), TypeError),
    ("blank_out_of_range", lambda a: dict(a, blank=V), AssertionError),
    ("negative_blank", lambda a: dict(a, blank=-1), AssertionError),
    ("bool_blank", lambda a: dict(a, blank=True), TypeError),
]
MALFORMED_BIGRAMS = [
    ("bigrams_of_another_width", lambda a: dict(a, bigrams=np.zeros((B, L + 1), np.int32)), AssertionError),
    ("bigrams_of_fewer_utterances", lambda a: dict(a, bigrams=a["bigrams"][:B - 1]), ValueError),
    ("float_bigrams", lambda a: dict(a, bigrams=a["bigrams"].astype(np.float32)), TypeError),
]


def good_args(p):
    return dict(labels=p["labels"], bigrams=p["bigrams"], blank=0, input_length=p["input_length"],
                label_length=p["label_length"])


@pytest.mark.parametrize("entry", ENTRIES)
def test_well_formed_arguments_run(entry):
    """The baseline the refusals below are measured against: the same call with nothing malformed goes through."""
    import torch
    p = problem()
    call(entry, p=p, **good_args(p))
    torch.cuda.synchronize()


@pytest.mark.parametrize("case", MALFORMED, ids=[c[0] for c in MALFORMED])
@pytest.mark.parametrize("entry", ENTRIES)
def test_malformed_argument_raises_what_ctc_raises(entry, case):
    _, change, exc = case
    p = problem()
    with pytest.raises(exc):
        call(entry, p=p, **change(good_args(p)))


@pytest.mark.parametrize("case", MALFORMED_BIGRAMS, ids=[c[0] for c in MALFORMED_BIGRAMS])
@pytest.mark.parametrize("entry", GRAM_ENTRIES)
def test_malformed_bigrams_raise_what_gram_ctc_raises(entry, case):
    _, change, exc = case
    p = problem()
    with pytest.raises(exc):
        call(entry, p=p, **change(good_args(p)))


@pytest.mark.parametrize("entry", ["ctc_host", "gram_ctc_host"])
def test_host_ignores_label_length_without_input_length(entry):
    """gram_ctc.py:310-313: with input_length omitted both lengths default to the full widths, as in ``ctc``."""
    p = problem()
    args = good_args(p)
    loss_a, grad_a = call(entry, p=p, **dict(args, input_length=None, label_length=None))
    grad_a = grad_a.clone()
    loss_b, grad_b = call(entry, p=p, **dict(args, input_length=None, label_length=p["label_length"]))
    assert np.array_equal(loss_a, loss_b)
    assert np.array_equal(grad_a.numpy(), grad_b.numpy())
