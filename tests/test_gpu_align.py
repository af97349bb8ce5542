"""GPU: forced alignment (ctc_forced_align / gram_ctc_forced_align) against the float64 Viterbi oracle
(tests/align_oracle.py), the planted alignment of trained-like inputs, the loss, and torchaudio.

Random inputs can hold paths whose scores tie to within fp32 rounding, so a returned path is checked for being a path
of the lattice whose float64 probability equals the oracle's best, not for being the oracle's path; on trained-like
inputs the best path is unique and must be the planted one exactly."""
import importlib

import numpy as np
import pytest

import align_oracle as ao
from oracle import lattice

pytestmark = pytest.mark.gpu
RTOL = 1e-5


def synth():
    return importlib.import_module("chainer-speech-recognition_b200.synth")


CTC_SHAPES = [
    # B, T, V, L
    (3, 12, 9, 3),
    (4, 50, 40, 8),
    (2, 33, 37, 5),        # V not a multiple of 4
    (2, 7, 5, 1),          # Lmax = 1
    (8, 200, 3500, 40),    # BASELINE configs[0]
    (2, 300, 64, 100),
    (1, 800, 50, 380),     # N = 761
    (1, 2100, 40, 1022),   # N = 2045, the loss's largest CTC lattice: two nodes per thread
]
GRAM_SHAPES = [
    (3, 12, 9, 3),
    (4, 50, 40, 8),
    (2, 33, 37, 5),
    (2, 9, 11, 1),
    (4, 120, 300, 30),
    (2, 400, 200, 100),
    (1, 900, 150, 250),    # N = 751
    (2, 200, 8000, 60),    # V = 8000
    (1, 3100, 150, 1020),  # N = 3061: three nodes per thread
]


def run(pkg, prob, kind, form="tbv", blank=None, **kw):
    import torch
    dev = torch.device("cuda:0")
    x = torch.tensor(prob["x"], device=dev)
    if form == "bf":
        xin, kw = x.transpose(0, 1).contiguous(), dict(kw, batch_first=True)
    elif form == "list":
        xin = [x[t] for t in range(x.shape[0])]
    else:
        xin = x
    blank = prob["blank"] if blank is None else blank
    lab = torch.tensor(prob["labels"], device=dev)
    il = None if prob.get("input_length") is None else torch.tensor(prob["input_length"], device=dev)
    ll = None if prob.get("label_length") is None else torch.tensor(prob["label_length"], device=dev)
    if kind == "ctc":
        a = pkg.ctc_forced_align(xin, lab, blank, il, ll, **kw)
    else:
        a = pkg.gram_ctc_forced_align(xin, lab, torch.tensor(prob["bigrams"], device=dev), blank, il, ll, **kw)
    torch.cuda.synchronize()
    return {k: (None if v is None else v.cpu().numpy()) for k, v in a._asdict().items()}


def lattice_of(prob, kind, b, Lb, blank):
    lab = np.asarray(prob["labels"][b, :Lb], np.int64)
    if kind == "ctc":
        return ao.ctc_lattice(lab, blank)
    return ao.gram_ctc_lattice(lab, np.asarray(prob["bigrams"][b, :Lb], np.int64), blank)


def lengths(prob, b):
    T, _, _ = prob["x"].shape
    Lmax = prob["labels"].shape[1]
    Tb = T if prob.get("input_length") is None else int(np.clip(prob["input_length"][b], 0, T))
    Lb = Lmax if prob.get("label_length") is None else int(np.clip(prob["label_length"][b], 0, Lmax))
    return Tb, Lb


def close(a, b):
    return abs(a - b) <= RTOL * max(abs(b), 1.0)


def check_against_oracle(prob, kind, out, blank=None):
    """Checks 1, 2, 5 and the Gram-CTC half of 4 for every utterance; returns the oracle scores."""
    blank = prob["blank"] if blank is None else blank
    x = prob["x"].astype(np.float64)
    T, B, _ = x.shape
    per = 2 if kind == "ctc" else 3
    scores = []
    for b in range(B):
        Tb, Lb = lengths(prob, b)
        lat = lattice_of(prob, kind, b, Lb, blank)
        logp = lattice.log_softmax(x[:Tb, b])
        ref, _, _ = ao.viterbi(logp, lat)
        scores.append(ref)
        s, path, ids = float(out["score"][b]), out["path"][b], out["ids"][b]
        assert np.all(path[Tb:] == -1) and np.all(ids[Tb:] == blank)
        if not np.isfinite(ref):
            assert s == 1e10 and np.all(path == -1) and np.all(ids == blank)
            if out["spans"] is not None:
                assert np.all(out["spans"][b] == -1)
            continue
        assert close(s, ref), (b, s, ref)
        p = path[:Tb].astype(np.int64)
        rescored = ao.rescore(logp, lat, p)
        assert rescored is not None, "utterance %d: not a path of the lattice" % b
        assert close(-rescored, ref), (b, -rescored, ref)
        assert np.array_equal(ids[:Tb], lat.symbols[p])
        runs = p[np.r_[True, p[1:] != p[:-1]]] if Tb else p
        assert [q for j in runs for q in ao.node_positions(int(j), per)] == list(range(Lb))
        if out["spans"] is not None:
            sp = out["spans"][b]
            assert np.array_equal(sp[:Lb], ao.path_spans(p, per, Lb)) and np.all(sp[Lb:] == -1)
        if out["frame_logp"] is not None:
            fl = out["frame_logp"][b]
            assert np.all(fl[Tb:] == 0)
            assert close(-float(np.sum(fl[:Tb].astype(np.float64))), s)
            assert np.allclose(fl[:Tb], logp[np.arange(Tb), ids[:Tb]], rtol=1e-5, atol=1e-5)
    return np.array(scores)


def planted_nodes(prob, kind, b):
    """Node path of synth.add_alignment_bump: an even spread of blank, l0, blank, l1, ..., blank."""
    Tb, Lb = lengths(prob, b)
    S = 2 * Lb + 1
    s = np.minimum(S - 1, np.arange(Tb) * S // max(Tb, 1))
    return s if kind == "ctc" else (s // 2) * 3 + (s % 2)


def check_loss_and_planted(pkg, prob, kind, out, trained):
    import torch
    dev = torch.device("cuda:0")
    x = torch.tensor(prob["x"], device=dev)
    lab = torch.tensor(prob["labels"], device=dev)
    il, ll = torch.tensor(prob["input_length"], device=dev), torch.tensor(prob["label_length"], device=dev)
    if kind == "ctc":
        loss = pkg.ctc(x, lab, prob["blank"], il, ll, reduce="no")
    else:
        loss = pkg.gram_ctc(x, lab, torch.tensor(prob["bigrams"], device=dev), prob["blank"], il, ll, reduce="no")
    loss = loss.detach().cpu().numpy().astype(np.float64)
    s = out["score"].astype(np.float64)
    assert np.all(s >= loss - 1e-5 * np.abs(loss)), (s, loss)
    if kind == "ctc":
        _, B, V = prob["x"].shape
        det = pkg.minibatch_error_details(out["ids"], lab, prob["blank"], np.arange(V, dtype=np.int32)[:, None],
                                          input_length=il)
        feas = s < 1e10
        assert np.all(det["distance"].cpu().numpy()[feas] == 0)
    if trained:
        for b in range(prob["x"].shape[1]):
            Tb, Lb = lengths(prob, b)
            if Tb < 2 * Lb + 1:
                continue
            want = planted_nodes(prob, kind, b)
            assert np.array_equal(out["path"][b, :Tb], want), b
            lat = lattice_of(prob, kind, b, Lb, prob["blank"])
            assert np.array_equal(out["ids"][b, :Tb], lat.symbols[want])
            assert np.array_equal(out["spans"][b, :Lb], ao.path_spans(want, 2 if kind == "ctc" else 3, Lb))


@pytest.mark.parametrize("shape", CTC_SHAPES)
@pytest.mark.parametrize("trained", [False, True])
def test_ctc_alignment(pkg, shape, trained):
    B, T, V, L = shape
    prob = synth().ctc_problem(B, T, V, L, seed=1, trained=trained)
    out = run(pkg, prob, "ctc")
    check_against_oracle(prob, "ctc", out)
    check_loss_and_planted(pkg, prob, "ctc", out, trained)


@pytest.mark.parametrize("shape", GRAM_SHAPES)
@pytest.mark.parametrize("trained", [False, True])
def test_gram_ctc_alignment(pkg, shape, trained):
    B, T, V, L = shape
    prob = synth().gram_problem(B, T, V, L, seed=2, trained=trained, n_unigram=max(3, min(119, V // 3)))
    out = run(pkg, prob, "gram")
    check_against_oracle(prob, "gram", out)
    check_loss_and_planted(pkg, prob, "gram", out, trained)


@pytest.mark.parametrize("kind", ["ctc", "gram"])
def test_edge_cases(pkg, kind):
    s = synth()
    mk = (lambda **k: s.ctc_problem(**k)) if kind == "ctc" else (lambda **k: s.gram_problem(n_unigram=6, **k))
    prob = mk(B=5, T=20, V=12, L=4, seed=7)
    prob["labels"][1, :2] = [3, 3]                      # repeated label: needs 3 frames for CTC
    if kind == "gram":
        prob["bigrams"][1, :2] = -1                     # no bigram to cover the pair, so Gram-CTC needs 3 frames too
    prob["label_length"][1] = 2
    prob["input_length"][1] = 2                         # infeasible
    prob["input_length"][2] = 0
    prob["label_length"][2] = 0                         # Tb = Lb = 0
    prob["input_length"][3] = 99                        # out of range: clamped to T
    prob["label_length"][3] = -3                        # clamped to 0
    prob["input_length"][4] = -1                        # clamped to 0, Lb > 0: infeasible
    out = run(pkg, prob, kind)
    assert out["score"][1] == 1e10 and np.all(out["path"][1] == -1) and np.all(out["spans"][1] == -1)
    assert out["score"][2] == 0.0 and np.all(out["path"][2] == -1)
    assert out["score"][4] == 1e10
    assert np.all(out["frame_logp"][1] == 0)
    check_against_oracle(prob, kind, out)
    # a non-zero blank id
    prob = mk(B=3, T=30, V=12, L=5, seed=8)
    blank = 11
    prob["labels"][prob["labels"] == blank] = 1
    if kind == "gram":
        prob["bigrams"][prob["bigrams"] == blank] = -1
    out = run(pkg, prob, kind, blank=blank)
    check_against_oracle(prob, kind, out, blank=blank)
    # optional outputs left out
    out2 = run(pkg, prob, kind, blank=blank, spans=False, frame_logp=False)
    assert out2["spans"] is None and out2["frame_logp"] is None
    assert np.array_equal(out2["path"], out["path"]) and np.array_equal(out2["score"], out["score"])


def test_many_utterances_and_nan(pkg):
    prob = synth().ctc_problem(200, 60, 33, 10, seed=9)
    prob["x"][5, 17, 4] = np.nan                        # inside utterance 17's valid frames
    assert prob["input_length"][17] > 5
    out = run(pkg, prob, "ctc")
    assert np.isnan(out["score"][17])
    assert np.all(np.isfinite(out["score"][np.arange(200) != 17]))
    prob["x"][5, 17, 4] = 0.0
    good = run(pkg, prob, "ctc")
    keep = np.arange(200) != 17
    assert np.array_equal(good["score"][keep], out["score"][keep])
    assert np.array_equal(good["path"][keep], out["path"][keep])
    check_against_oracle(prob, "ctc", good)


@pytest.mark.parametrize("kind", ["ctc", "gram"])
def test_bit_identical(pkg, kind):
    """Two calls, batched against solo utterances, and the three input forms give the same bits (V % 4 == 0, so every
    activation row sits at the same 16-byte phase in every form)."""
    s = synth()
    prob = (s.ctc_problem(6, 120, 64, 20, seed=11) if kind == "ctc"
            else s.gram_problem(6, 120, 64, 20, seed=11, n_unigram=20))
    ref = run(pkg, prob, kind)
    for k, v in run(pkg, prob, kind).items():
        assert np.array_equal(v, ref[k]), k
    for form in ("list", "bf"):
        for k, v in run(pkg, prob, kind, form=form).items():
            assert np.array_equal(v, ref[k]), (form, k)
    for b in range(6):
        solo = {k: (v[:, b:b + 1] if k == "x" else (v[b:b + 1] if isinstance(v, np.ndarray) else v))
                for k, v in prob.items()}
        one = run(pkg, solo, kind)
        for k, v in one.items():
            assert np.array_equal(v[0], ref[k][b]), (b, k)


def test_matches_torchaudio_on_the_gpu(pkg):
    torch = pytest.importorskip("torch")
    F = pytest.importorskip("torchaudio.functional")
    prob = synth().ctc_problem(8, 200, 500, 30, seed=12, trained=True)
    out = run(pkg, prob, "ctc")
    x = torch.tensor(prob["x"], device="cuda")
    for b in range(8):
        Tb, Lb = lengths(prob, b)
        lp = torch.log_softmax(x[:Tb, b], dim=-1)[None]
        tg = torch.tensor(prob["labels"][b:b + 1, :Lb], device="cuda", dtype=torch.int32)
        a, _ = F.forced_align(lp, tg, blank=0)
        assert np.array_equal(a[0].cpu().numpy(), out["ids"][b, :Tb]), b
