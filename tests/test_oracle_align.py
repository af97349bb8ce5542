"""CPU: the forced-alignment oracle (tests/align_oracle.py) against a brute-force maximum over frame labellings and
against torchaudio's CTC forced alignment; the C entry point is declared, bound, and refuses bad arguments before it
touches a device."""
import ctypes
import importlib
import os
import re

import numpy as np
import pytest

import align_oracle as ao
from oracle import lattice

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INVENTORY = {1: (1,), 2: (2,), 3: (3,), 4: (1, 2), 5: (2, 3), 6: (1, 1), 7: (2, 1)}
PAIR = {v: k for k, v in INVENTORY.items() if len(v) == 2}


@pytest.mark.parametrize("target", [(1, 2), (1, 2, 3), (1, 1), (1, 1, 1), (2, 1, 2), (1, 1, 1, 1), (1, 2, 1, 2), (3,), ()])
def test_viterbi_matches_brute_force_maximum(target):
    """The targets of test_oracle.py's enumeration (T=5, V=8): CTC and Gram-CTC with bigrams."""
    rs = np.random.RandomState(len(target) * 7 + 1)
    T, V = 5, 8
    x = rs.randn(T, V)
    L = len(target)
    uni = np.array(target, np.int64)
    big = np.full(L, -1, np.int64)
    for i in range(1, L):
        big[i] = PAIR.get((target[i - 1], target[i]), -1)
    logp = lattice.log_softmax(x)
    for lat, gram_to_chars in ((ao.gram_ctc_lattice(uni, big, 0), INVENTORY),
                               (ao.ctc_lattice(uni, 0), {k: (k,) for k in range(1, V)})):
        bf = ao.max_log_likelihood(logp, target, gram_to_chars, 0)
        score, path, spans = ao.viterbi(logp, lat)
        if not np.isfinite(bf):
            assert score == np.inf and path is None
            continue
        assert np.isclose(score, -bf, rtol=1e-10, atol=0)
        assert np.isclose(ao.rescore(logp, lat, path), bf, rtol=1e-10, atol=0)
        covered = [q for j in path[np.r_[True, path[1:] != path[:-1]]] for q in ao.node_positions(int(j), ao.lattice_kind(lat))]
        assert covered == list(range(L))
        assert np.all(spans[:, 0] < spans[:, 1])


def test_viterbi_tie_rule():
    """Uniform log-probabilities: every path ties, so the rule decides -- the final blank ends it, and walking back
    every node takes its self-loop while that is a path, so the labels come as early as the lattice allows."""
    logp = np.full((5, 4), np.log(0.25))
    _, path, spans = ao.viterbi(logp, ao.ctc_lattice([1, 2], 0))
    assert path.tolist() == [1, 3, 4, 4, 4]
    assert spans.tolist() == [[0, 1], [1, 2]]


def _ctc_cases():
    synth = importlib.import_module("chainer-speech-recognition_b200.synth")
    yield "random", synth.ctc_problem(6, 50, 23, 8, seed=3)
    yield "trained", synth.ctc_problem(6, 60, 40, 10, seed=4, trained=True)


@pytest.mark.parametrize("case", ["random", "trained"])
def test_viterbi_matches_torchaudio_forced_align(case):
    torch = pytest.importorskip("torch")
    F = pytest.importorskip("torchaudio.functional")
    prob = dict(_ctc_cases())[case]
    x = prob["x"].astype(np.float64)
    for b in range(x.shape[1]):
        Tb, Lb = int(prob["input_length"][b]), int(prob["label_length"][b])
        lab = prob["labels"][b, :Lb]
        logp = lattice.log_softmax(x[:Tb, b])
        score, path, _ = ao.viterbi(logp, ao.ctc_lattice(lab, 0))
        ids = ao.ctc_lattice(lab, 0).symbols[path]
        a, s = F.forced_align(torch.tensor(logp)[None], torch.tensor(lab, dtype=torch.int32)[None],
                              torch.tensor([Tb]), torch.tensor([Lb]), blank=0)
        assert a[0].numpy().tolist() == ids.tolist()
        assert np.isclose(-score, float(s.sum()), rtol=1e-9, atol=0)


def test_align_is_declared_and_bound(pkg):
    header = open(os.path.join(ROOT, "include", "b200ctc.h")).read()
    assert re.search(r"\bint b200ctc_align\s*\(", header)
    assert int(re.search(r"#define B200CTC_VERSION (\d+)", header).group(1)) >= 203
    lib = pkg._lib.load()
    assert lib.b200ctc_align.restype == ctypes.c_int and len(lib.b200ctc_align.argtypes) == 21


def test_align_status_codes_without_a_device(pkg):
    L = pkg._lib
    fn = L.load().b200ctc_align
    fake = 1 << 20                            # 16-byte aligned, never dereferenced: every call below returns first
    ws = 1 << 40

    def call(kind=L.KIND_CTC, acts=fake, labels=fake, bigrams=fake, blank=0, B=2, T=10, V=8, Lmax=3, score=fake,
             path=fake, ids=fake, workspace=fake, wsbytes=ws):
        return fn(kind, acts, 2 * V, V, labels, bigrams, None, None, blank, B, T, V, Lmax, score, path, ids, None, None,
                  workspace, wsbytes, None)

    assert call(kind=L.KIND_JOINT) == L.INVALID_ARGUMENT
    assert call(kind=7) == L.INVALID_ARGUMENT
    assert call(V=0) == L.INVALID_ARGUMENT
    assert call(blank=8) == L.INVALID_ARGUMENT
    assert call(acts=None) == L.INVALID_ARGUMENT
    assert call(labels=None) == L.INVALID_ARGUMENT
    assert call(kind=L.KIND_GRAM, bigrams=None) == L.INVALID_ARGUMENT
    assert call(score=None) == L.INVALID_ARGUMENT
    assert call(path=None) == L.INVALID_ARGUMENT
    assert call(ids=None) == L.INVALID_ARGUMENT
    assert call(workspace=None) == L.INVALID_ARGUMENT
    assert call(workspace=fake + 4) == L.INVALID_ARGUMENT
    assert call(acts=fake + 2) == L.INVALID_ARGUMENT
    assert call(wsbytes=16) == L.WORKSPACE_TOO_SMALL
    assert call(Lmax=1023) == L.UNSUPPORTED                   # 2047 CTC nodes: above the loss's limit
    assert call(kind=L.KIND_GRAM, Lmax=1025) == L.UNSUPPORTED
    assert call(B=0) == L.OK                                   # nothing to do


def test_python_front_end_refusals(pkg):
    torch = pytest.importorskip("torch")
    x = torch.zeros(4, 2, 5)                                   # CPU tensor: no CPU path
    t = torch.ones(2, 2, dtype=torch.int32)
    with pytest.raises(TypeError):
        pkg.ctc_forced_align(x, t, True)                       # bool blank
    with pytest.raises(TypeError):
        pkg.ctc_forced_align(x.double(), t, 0)
    with pytest.raises(RuntimeError):
        pkg.ctc_forced_align(x, t, 0)
    with pytest.raises(ValueError):
        pkg.ctc_forced_align([], t, 0)
    with pytest.raises(TypeError):
        pkg.gram_ctc_forced_align(x[0], t, t, 0)               # 2-D tensor
