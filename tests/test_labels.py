"""CPU: the label half of minibatch assembly (asr/data/processing.py of this package) against golden vectors
produced by the reference's own Processor.features_to_minibatch (tests/golden/generate_golden_labels.py) and, where
the reference is mounted, against the reference itself on fresh seeds."""
import glob
import importlib
import os

import numpy as np
import pytest

from oracle import ref_stub

GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "labels", "*.npz")))


def mine():
    return importlib.import_module("chainer-speech-recognition_b200.asr.data.processing")


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_labels_match_reference_golden(path):
    g = np.load(path)
    ids = {str(t): i for i, t in enumerate(g["inventory"])}
    offs = g["offsets"]
    sentences = [[str(t) for t in g["tokens"][offs[b]:offs[b + 1]]] for b in range(len(offs) - 1)]
    t, big, xl, tl = mine().labels_to_minibatch(sentences, g["x_length"], int(g["Lmax"]), ids, 0)
    assert t.dtype.is_floating_point is False and str(t.dtype) == "torch.int32"
    assert np.array_equal(t.numpy(), g["ref_t"])
    assert np.array_equal(big.numpy(), g["ref_bigram"])
    assert np.array_equal(tl.numpy(), g["ref_t_length"])
    assert np.array_equal(xl.numpy(), g["ref_x_length"])
    # one host block behind all four views (one copy moves everything to the device)
    assert t.untyped_storage().data_ptr() == big.untyped_storage().data_ptr() == tl.untyped_storage().data_ptr()
    # the transcriptions as strings through tokenizer=: the golden tokens are the reference tokeniser's output for them
    # (tests/golden/generate_golden_labels.py), so a lookup of that output stands in for the reference's tokeniser
    reference_tokens = {"".join(s): s for s in sentences}
    t, big, xl, tl = mine().labels_to_minibatch(["".join(s) for s in sentences], g["x_length"], int(g["Lmax"]), ids, 0,
                                                tokenizer=lambda s: list(reference_tokens[s]))
    assert np.array_equal(t.numpy(), g["ref_t"]) and np.array_equal(big.numpy(), g["ref_bigram"])
    assert np.array_equal(tl.numpy(), g["ref_t_length"]) and np.array_equal(xl.numpy(), g["ref_x_length"])


def test_golden_set_is_present():
    assert len(GOLDEN) >= 3


@pytest.mark.skipif(not ref_stub.available(), reason="reference not mounted")
def test_labels_match_reference_live():
    proc = ref_stub.load_processing_module()
    _, vocab = ref_stub.load_error_module()
    toks = vocab.UNIGRAM_TOKENS
    rng = np.random.RandomState(11)
    for _ in range(4):
        ids, _ = vocab.get_unigram_ids()
        B = 5
        sentences = ["".join(toks[rng.randint(len(toks))] for _ in range(rng.randint(1, 10))) for _ in range(B)]
        tokenised = [vocab.convert_sentence_to_unigram_tokens(s) for s in sentences]
        for tk in tokenised:
            for a, c in zip(tk[:-1], tk[1:]):
                if rng.rand() < 0.5:
                    ids.setdefault(a + c, len(ids))
        x_len = [int(rng.randint(1, 25)) for _ in range(B)]
        Lmax = max(len(tk) for tk in tokenised)
        P = proc.Processor(using_delta=False, using_delta_delta=False)
        feats = [(np.zeros((40, x), np.float32), None, None) for x in x_len]
        _, xlb, tb, tlb, bb = P.features_to_minibatch(feats, sentences, max(x_len), Lmax, ids, 0)
        t, big, xl, tl = mine().labels_to_minibatch(sentences, x_len, Lmax, ids, 0,
                                                    tokenizer=vocab.convert_sentence_to_unigram_tokens)
        assert np.array_equal(t.numpy(), tb) and np.array_equal(big.numpy(), bb)
        assert tl.tolist() == list(tlb) and xl.tolist() == list(xlb)


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_length_sorted_layout_is_a_row_permutation_of_the_reference(path):
    """sort_by_length=True: longest utterance first (stable), every row still the reference's row for that sentence."""
    g = np.load(path)
    ids = {str(t): i for i, t in enumerate(g["inventory"])}
    offs = g["offsets"]
    sentences = [[str(t) for t in g["tokens"][offs[b]:offs[b + 1]]] for b in range(len(offs) - 1)]
    t, big, xl, tl, order = mine().labels_to_minibatch(sentences, g["x_length"], int(g["Lmax"]), ids, 0,
                                                       sort_by_length=True)
    order = order.numpy()
    assert sorted(order.tolist()) == list(range(len(sentences)))
    assert np.all(np.diff(xl.numpy()) <= 0)
    assert np.array_equal(order, np.argsort(-g["ref_x_length"].astype(np.int64), kind="stable"))
    assert np.array_equal(t.numpy(), g["ref_t"][order])
    assert np.array_equal(big.numpy(), g["ref_bigram"][order])
    assert np.array_equal(tl.numpy(), g["ref_t_length"][order])
    assert np.array_equal(xl.numpy(), g["ref_x_length"][order])


@pytest.mark.gpu
@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_device_block_feeds_the_loss(path):
    """device=: the four arrays arrive on the GPU as views of ONE device block, equal to the reference's arrays, and go
    into gram_ctc as they are; the length-sorted layout gives the same per-utterance losses, permuted."""
    import torch
    import b200ctc
    g = np.load(path)
    ids = {str(t): i for i, t in enumerate(g["inventory"])}
    offs = g["offsets"]
    sentences = [[str(t) for t in g["tokens"][offs[b]:offs[b + 1]]] for b in range(len(offs) - 1)]
    dev = torch.device("cuda:0")
    Lmax, B = int(g["Lmax"]), len(sentences)
    t, big, xl, tl = mine().labels_to_minibatch(sentences, g["x_length"], Lmax, ids, 0, device=dev)
    assert t.is_cuda and t.untyped_storage().data_ptr() == tl.untyped_storage().data_ptr()
    assert np.array_equal(t.cpu().numpy(), g["ref_t"]) and np.array_equal(big.cpu().numpy(), g["ref_bigram"])
    assert np.array_equal(tl.cpu().numpy(), g["ref_t_length"]) and np.array_equal(xl.cpu().numpy(), g["ref_x_length"])
    T, V = int(g["x_length"].max()), len(ids)
    x = torch.randn((T, B, V), device=dev, generator=torch.Generator(device=dev).manual_seed(3))
    loss = b200ctc.gram_ctc(x, t, big, 0, xl, tl, reduce="no")
    ts, bs, xls, tls, order = mine().labels_to_minibatch(sentences, g["x_length"], Lmax, ids, 0, device=dev,
                                                         sort_by_length=True)
    loss_sorted = b200ctc.gram_ctc(x[:, order.to(dev)], ts, bs, 0, xls, tls, reduce="no")
    assert torch.equal(loss_sorted, loss[order.to(dev)])
    assert torch.isfinite(loss).all()
