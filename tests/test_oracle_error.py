"""CPU: the error-rate oracle (oracle/error.py) against the committed golden vectors -- outputs of the
reference's own asr/error.py (tests/golden/generate_golden_cer.py) -- and, where the reference is mounted,
against the reference itself on fresh seeds."""
import glob
import os
import warnings

import numpy as np
import pytest

from oracle import error as oerr
from oracle import ref_stub

GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "cer", "*.npz")))


def load(path):
    z = np.load(path)
    return {k: z[k] for k in z.files}


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
@pytest.mark.parametrize("wrap", [False, True])
def test_oracle_matches_reference_golden(path, wrap):
    g = load(path)
    mean, errs, _ = oerr.minibatch_error(g["y"], g["t"], int(g["blank"]), g["expansion"], uint8_wrap=wrap)
    assert mean == float(g["ref_mean"])                      # bit-exact: same float64 operations in the same order
    assert np.array_equal(errs, g["ref_each"])


def test_golden_set_is_present():
    assert len(GOLDEN) >= 5


@pytest.mark.skipif(not ref_stub.available(), reason="reference not mounted")
def test_oracle_matches_reference_live():
    err, vocab = ref_stub.load_error_module()
    ids, inv = vocab.get_unigram_ids()
    table = np.array([vocab.convert_sentence_to_unigram_ids(inv[i], ids) for i in range(len(ids))], np.int32)
    rng = np.random.RandomState(7)
    for _ in range(5):
        B, T, L = 3, int(rng.randint(1, 50)), int(rng.randint(1, 12))
        y = rng.randint(0, len(ids), size=(B, T))
        y[rng.rand(B, T) < 0.4] = 0
        t = rng.randint(0, len(ids), size=(B, L))
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            ref = err.compute_minibatch_error(y, t, 0, ids, inv)
        assert oerr.minibatch_error(y, t, 0, table)[0] == ref
    assert err.compute_character_error_rate([], [1, 2, 3]) == oerr.character_error_rate([], [1, 2, 3]) == 3
    assert err.compute_character_error_rate([1, 2], []) == oerr.character_error_rate([1, 2], []) == 1.0


def test_character_error_rate_of_empty_sequences_is_the_references():
    # the reference's compute_character_error_rate returns these (asr/error.py:8-9 and :24; checked against it live above)
    assert oerr.character_error_rate([], [1, 2, 3]) == 3
    assert oerr.character_error_rate([1, 2], []) == 1.0


def test_collapse_is_the_prev_token_state_machine():
    # asr/error.py:38-47: a blank resets prev_token, repeats are dropped, a repeat after a blank counts again
    assert oerr.collapse([0, 3, 3, 0, 3, 4, 4, 4, 0, 0, 5], 0) == [3, 3, 4, 5]
    assert oerr.collapse([], 0) == []
    assert oerr.collapse([2, 2, 2], 0) == [2]
    # equivalent closed form used by the kernel: keep[t] = tok[t] != blank and tok[t] != tok[t-1]
    rng = np.random.RandomState(0)
    for _ in range(50):
        y = rng.randint(0, 4, size=30)
        keep = [int(v) for i, v in enumerate(y) if v != 0 and (i == 0 or v != y[i - 1])]
        assert oerr.collapse(y, 0) == keep


def test_edit_distance_known_answers():
    assert oerr.edit_distance([1, 2, 3], [1, 2, 3]) == 0
    assert oerr.edit_distance([1, 2, 3], [1, 3]) == 1
    assert oerr.edit_distance([1, 2, 3], [4, 5, 6, 7]) == 4
    assert oerr.edit_distance(list("kitten"), list("sitting")) == 3
    assert oerr.edit_distance([], [1] * 7) == 7


def test_uint8_wrap_is_modulo_256_arithmetic():
    # restate asr/error.py:10-23 with an explicit numpy.uint8 table (array arithmetic wraps silently)
    rng = np.random.RandomState(3)
    r = list(rng.randint(0, 3, size=300))
    h = list(rng.randint(3, 6, size=280))                    # nothing matches: true distance 300 -> wraps
    R, H = len(r), len(h)
    d = np.zeros((R + 1, H + 1), dtype=np.uint8)
    d[0, :] = (np.arange(H + 1) % 256).astype(np.uint8)
    d[:, 0] = (np.arange(R + 1) % 256).astype(np.uint8)
    one = np.uint8(1)
    with np.errstate(over="ignore"):
        for i in range(1, R + 1):
            for j in range(1, H + 1):
                if r[i - 1] == h[j - 1]:
                    d[i, j] = d[i - 1, j - 1]
                else:
                    d[i, j] = min(np.add(d[i - 1, j - 1], one, dtype=np.uint8), np.add(d[i, j - 1], one, dtype=np.uint8),
                                  np.add(d[i - 1, j], one, dtype=np.uint8))
    assert oerr.edit_distance(r, h, uint8_wrap=True) == int(d[R, H])
    assert oerr.edit_distance(r, h) == 300
