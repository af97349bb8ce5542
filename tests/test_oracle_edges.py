"""CPU: both oracles (oracle/lattice.py and oracle/ctc_oracle.c) against brute-force enumeration in the corners the
synthetic generator never reaches -- a blank id other than 0 (label id 0 then an ordinary symbol), tight and infeasible
alignments, Gram-CTC utterances shorter than their character count, closed k=6 edges, all-dead and all-alive bigrams --
and against each other on labels equal to the blank and on degenerate lengths.  The device edge tests
(test_gpu_edges.py) judge the kernels by these oracles, so the oracles are pinned here first."""
import numpy as np
import pytest

from oracle import lattice, c_oracle, brute_force


def _x(T, V, seed, B=1):
    return np.random.RandomState(seed).randn(T, B, V).astype(np.float32)


def _both(kind, x, labels, bigrams, il, ll, blank):
    """(loss, grad) of the NumPy and of the C oracle."""
    labels = np.asarray(labels, np.int32).reshape(x.shape[1], -1)
    if kind == "ctc":
        ln, gn = lattice.ctc(x, labels, il, ll, blank)
        r = c_oracle.run(0, x, labels, None, il, ll, blank)
    else:
        bigrams = np.asarray(bigrams, np.int32).reshape(labels.shape)
        ln, gn = lattice.gram_ctc(x, labels, bigrams, il, ll, blank)
        r = c_oracle.run(1, x, labels, bigrams, il, ll, blank)
    return (ln, gn), (r["loss"], r["grad"])


def _agree(a, b):
    assert np.array_equal(a[0] == 1e10, b[0] == 1e10), (a[0], b[0])
    assert np.allclose(a[0], b[0], rtol=1e-10, atol=1e-10), (a[0], b[0])
    assert np.abs(a[1] - b[1]).max(initial=0.0) <= 1e-6


def _check_ctc(labels, T, V, blank, seed):
    x = _x(T, V, seed)
    L = len(labels)
    a, b = _both("ctc", x, [labels], None, [T], [L], blank)
    _agree(a, b)
    bf = brute_force.ctc_log_likelihood(lattice.log_softmax(x[:, 0]), labels, blank)
    for loss, _ in (a, b):
        if np.isfinite(bf):
            assert np.isclose(loss[0], -bf, rtol=1e-10), (loss[0], -bf)
        else:
            assert loss[0] == 1e10
    return bf


def _check_gram(uni, pairs, T, V, blank, seed):
    """uni: the characters; pairs: {(a, b): bigram id} of the inventory (ids of V that are neither a character nor blank)."""
    L = len(uni)
    big = [-1] + [pairs.get((uni[i - 1], uni[i]), -1) for i in range(1, L)]
    x = _x(T, V, seed)
    a, b = _both("gram", x, [uni], [big], [T], [L], blank)
    _agree(a, b)
    inventory = {c: (c,) for c in set(uni)}
    inventory.update({k: p for p, k in pairs.items()})
    assert blank not in inventory
    bf = brute_force.log_likelihood(lattice.log_softmax(x[:, 0]), uni, inventory, blank)
    for loss, _ in (a, b):
        if np.isfinite(bf):
            assert np.isclose(loss[0], -bf, rtol=1e-10), (loss[0], -bf)
        else:
            assert loss[0] == 1e10
    return bf


# ---- blank != 0, label 0 an ordinary symbol ----

@pytest.mark.parametrize("blank,V", [(2, 3), (3, 4), (5, 6), (2, 4)])
@pytest.mark.parametrize("labels", [(0, 0, 1), (0, 1), (1, 0, 1), (0,)])
def test_ctc_blank_not_zero(blank, V, labels):
    bf = _check_ctc(list(labels), 4, V, blank, seed=blank * 31 + len(labels))
    assert np.isfinite(bf)


# ---- tight alignments: T = L + #adjacent repeats is the least feasible length ----

@pytest.mark.parametrize("blank", [0, 3])
@pytest.mark.parametrize("labels", [(1, 1, 1), (1, 2, 2), (2, 1, 2), (1, 1), (2,)])
def test_ctc_tight_and_one_short(blank, labels):
    labels = [l if l != blank else 0 for l in labels]
    need = len(labels) + sum(labels[i] == labels[i - 1] for i in range(1, len(labels)))
    assert np.isfinite(_check_ctc(labels, need, 4, blank, seed=need))
    assert _check_ctc(labels, need - 1, 4, blank, seed=need) == -np.inf


def test_ctc_tight_alignment_has_one_path():
    """At the tight length the only path is the labels with one blank between each repeat: loss = -sum log p."""
    labels, blank, V = [0, 0, 1], 2, 3
    x = _x(4, V, 7)
    logp = lattice.log_softmax(x[:, 0])
    want = -(logp[0, 0] + logp[1, 2] + logp[2, 0] + logp[3, 1])
    a, b = _both("ctc", x, [labels], None, [4], [3], blank)
    assert np.isclose(a[0][0], want, rtol=1e-12) and np.isclose(b[0][0], want, rtol=1e-12)
    # one path: the posterior is 1 on it, so the gradient is softmax - one-hot of the path
    onehot = np.zeros((4, V))
    onehot[[0, 1, 2, 3], [0, 2, 0, 1]] = 1.0
    assert np.abs(a[1][:, 0] - (np.exp(logp) - onehot)).max() <= 1e-12
    assert np.abs(b[1][:, 0] - (np.exp(logp) - onehot)).max() <= 1e-6


# ---- Gram-CTC: blank = V - 1, fewer frames than characters, closed k=6 edges, dead / alive bigrams ----

# characters 0..3, bigram ids 4..6, blank 7
PAIRS = {(0, 1): 4, (2, 3): 5, (1, 2): 6}


@pytest.mark.parametrize("T", [2, 3, 4, 5])
def test_gram_fewer_frames_than_characters(T):
    """Four characters, bigrams at positions 1 and 3: at T = 2 only (01)(23) aligns, at T = 3 the k=5/7 edges and
    the final bigram node carry most paths."""
    bf = _check_gram([0, 1, 2, 3], {(0, 1): 4, (2, 3): 5}, T, 8, 7, seed=40 + T)
    assert np.isfinite(bf)


def test_gram_one_frame_short_of_the_bigram_path_is_infeasible():
    assert _check_gram([0, 1, 2, 3], {(0, 1): 4, (2, 3): 5}, 1, 8, 7, seed=3) == -np.inf


@pytest.mark.parametrize("T", [2, 3, 4, 5])
def test_gram_equal_consecutive_bigrams(T):
    """(0,1,0,1): bigram 4 at positions 1 and 3, so the k=6 edge between them is closed (its two nodes would merge)."""
    _check_gram([0, 1, 0, 1], {(0, 1): 4}, T, 8, 7, seed=50 + T)


@pytest.mark.parametrize("T", [3, 4, 5])
def test_gram_every_bigram_alive(T):
    _check_gram([0, 1, 2, 3], PAIRS, T, 8, 7, seed=60 + T)


@pytest.mark.parametrize("T", [4, 5])
def test_gram_every_bigram_dead(T):
    _check_gram([0, 1, 2, 1], {}, T, 8, 7, seed=70 + T)


@pytest.mark.parametrize("T", [3, 4])
def test_gram_repeated_characters_blank_in_the_middle(T):
    """blank = 3 sits between the characters 0..2 and the bigram ids 4..6."""
    _check_gram([1, 1, 2], {(1, 1): 4, (1, 2): 5}, T, 7, 3, seed=80 + T)


# ---- labels equal to the blank: not expressible by brute force, the two oracles must agree ----

@pytest.mark.parametrize("blank", [0, 2, 4])
@pytest.mark.parametrize("kind", ["ctc", "gram"])
def test_label_equal_to_blank(kind, blank):
    V, T = 5, 6
    labels = [[blank, 1 if blank != 1 else 3, blank], [1, blank, blank]]
    big = [[-1, blank, 4 if blank != 4 else 0], [-1, 3, blank]]
    x = _x(T, V, 90 + blank, B=2)
    a, b = _both(kind, x, labels, big, [T, 5], [3, 3], blank)
    _agree(a, b)
    assert np.all(a[0] < 1e10)


# ---- degenerate lengths ----

DEGENERATE = [  # (input_length, label_length) per utterance of one batch
    ([0, 0, 3, 1, 1, 4], [0, 2, 0, 0, 1, 2]),
    ([0], [0]),
    ([0], [1]),
    ([1, 2], [1, 1]),
]


@pytest.mark.parametrize("kind", ["ctc", "gram"])
@pytest.mark.parametrize("case", range(len(DEGENERATE)))
@pytest.mark.parametrize("blank", [0, 4])
def test_degenerate_lengths_oracles_agree(kind, case, blank):
    il, ll = DEGENERATE[case]
    B, T, V, L = len(il), 4, 5, 2
    rs = np.random.RandomState(case)
    labels = rs.randint(0, V, size=(B, L)).astype(np.int32)
    big = np.where(rs.rand(B, L) < 0.5, -1, rs.randint(0, V, size=(B, L))).astype(np.int32)
    x = _x(T, V, 100 + case, B=B)
    a, b = _both(kind, x, labels, big, il, ll, blank)
    _agree(a, b)
    for i in range(B):
        if il[i] == 0:
            assert a[0][i] == (0.0 if ll[i] == 0 else 1e10)
        assert not np.any(a[1][il[i]:, i]) and not np.any(b[1][il[i]:, i])


@pytest.mark.parametrize("kind", ["ctc", "gram"])
def test_no_labels_at_all(kind):
    """Lmax = 0: every utterance is all blank; loss = -sum_t log p(blank), gradient = softmax - one-hot(blank)."""
    B, T, V, blank = 3, 4, 5, 2
    x = _x(T, V, 5, B=B)
    il = [4, 2, 0]
    labels = np.zeros((B, 0), np.int32)
    a, b = _both(kind, x, labels, labels, il, [0, 0, 0], blank)
    _agree(a, b)
    for i in range(B):
        logp = lattice.log_softmax(x[:il[i], i])
        assert np.isclose(a[0][i], -logp[:, blank].sum(), rtol=1e-12, atol=1e-12)
        want = np.exp(logp)
        want[:, blank] -= 1.0
        assert np.abs(a[1][:il[i], i] - want).max(initial=0.0) <= 1e-12


def test_no_frames_no_labels_is_certain():
    """T_b = 0 and L_b = 0: nothing to emit in no frames, P = 1 (loss 0) in both oracles."""
    x = _x(3, 4, 0, B=1)
    for kind in ("ctc", "gram"):
        a, b = _both(kind, x, [[1]], [[-1]], [0], [0], 0)
        assert a[0][0] == 0.0 and b[0][0] == 0.0
