"""The development loop's greedy argmax with LayerNormalization fused in (b200ctc.layernorm_greedy_argmax,
csrc/layernorm_loss.cu ln_argmax_kernel) against numpy.argmax of the float64 oracle (oracle/layernorm.py).  The device
tests are marked gpu one by one; the argument checks that need no device, and the C-ABI status codes, are not."""
import ctypes
import importlib

import numpy as np
import pytest

from oracle import error as oerr, layernorm as oln


def synth():
    return importlib.import_module("chainer-speech-recognition_b200.synth")


def make_z(B, T, V, seed, bumped=True, bump=6.0, full_length=False):
    """z ~ N(0.3, 1.7^2) as (B, V, T) float32 (a convolution output is neither centred nor unit-variance), optionally
    +bump on a plausible alignment of random labels (the trained-like case: most frames have a clear winner);
    gamma ~ 1 +- 0.2, beta ~ +-0.1.  Drawn one utterance at a time so that the largest case stays small in host memory."""
    s = synth()
    rs = np.random.RandomState(seed)
    L = max(1, min(40, (T - 1) // 2))
    in_len, lab_len = s.make_lengths(rs, B, T, L)
    if full_length:
        in_len[:] = T
    labels = s.make_ctc_labels(rs, B, L, V, lab_len)
    z = np.empty((B, V, T), np.float32)
    for b in range(B):
        z[b] = (rs.standard_normal((V, T)) * 1.7 + 0.3).astype(np.float32)
        if bumped:
            path = [0]
            for i in range(int(lab_len[b])):
                path += [int(labels[b, i]), 0]
            Tb = int(in_len[b])
            for t in range(Tb):
                z[b, path[min(len(path) - 1, t * len(path) // Tb)], t] += bump
    gamma = (1.0 + 0.2 * rs.randn(V)).astype(np.float32)
    beta = (0.1 * rs.randn(V)).astype(np.float32)
    return z, gamma, beta, labels


def oracle_values(z, gamma, beta):
    """(B, T, V) float64 normalised activations, one utterance at a time."""
    B, V, T = z.shape
    out = np.empty((B, T, V), np.float64)
    with np.errstate(invalid="ignore", divide="ignore"):
        for b in range(B):
            acts, _ = oln.forward(z[b:b + 1], gamma, beta)            # (T, 1, V)
            out[b] = acts[:, 0, :]
    return out


def run(pkg, z, gamma, beta, z4d=True, pitch=None):
    import torch
    dev = torch.device("cuda:0")
    B, V, T = z.shape
    if pitch is None:
        zt = torch.tensor(z, device=dev)
    else:
        buf = torch.zeros((B, V, pitch), device=dev)
        buf[:, :, :T] = torch.tensor(z, device=dev)
        zt = buf[:, :, :T]
    out = pkg.layernorm_greedy_argmax(zt.unsqueeze(2) if z4d else zt, torch.tensor(gamma, device=dev),
                                      torch.tensor(beta, device=dev))
    assert out.dtype == torch.int64 and tuple(out.shape) == (B, T) and out.is_cuda
    return out.cpu().numpy()


def assert_picks_a_maximum(pick, y64):
    """Every pick is a maximum of its frame up to float32 rounding: exact agreement wherever the winner is clear."""
    assert pick.min() >= 0 and pick.max() < y64.shape[2]
    mx = y64.max(axis=2)
    got = np.take_along_axis(y64, pick[:, :, None], axis=2)[:, :, 0]
    bad = got < mx - 1e-4 * np.maximum(1.0, np.abs(mx))
    assert not bad.any(), (np.argwhere(bad)[:5], got[bad][:5], mx[bad][:5])


SHAPES = [
    # B, T, V
    (3, 40, 37),          # V below one box, odd V
    (2, 64, 241),         # one box + 1 row
    (5, 100, 1213),       # a real vocabulary size, T % 8 != 0
    (8, 200, 3500),       # BASELINE configs[0]
    (2, 48, 3601),        # 16 boxes
    (2, 48, 4080),        # the largest supported vocabulary (17 boxes)
    (64, 800, 3500),      # the bench shape
]


@pytest.mark.gpu
@pytest.mark.parametrize("bumped", [True, False], ids=["bumped", "plain"])
@pytest.mark.parametrize("shape", SHAPES, ids=["B%d-T%d-V%d" % s for s in SHAPES])
def test_matches_float64_oracle(pkg, shape, bumped):
    B, T, V = shape
    z, gamma, beta, _ = make_z(B, T, V, seed=71 + V, bumped=bumped)
    pick = run(pkg, z, gamma, beta)
    y64 = oracle_values(z, gamma, beta)
    assert_picks_a_maximum(pick, y64)
    if bumped:                               # the bumped frames have clear winners: most picks agree exactly
        assert (pick == y64.argmax(axis=2)).mean() > 0.99


@pytest.mark.gpu
def test_layouts_give_the_same_bits(pkg):
    z, gamma, beta, _ = make_z(3, 40, 300, seed=72)
    a = run(pkg, z, gamma, beta)
    assert np.array_equal(a, run(pkg, z, gamma, beta, z4d=False))
    assert np.array_equal(a, run(pkg, z, gamma, beta, pitch=44))
    assert np.array_equal(a, run(pkg, z, gamma, beta, pitch=64))
    z, gamma, beta, _ = make_z(3, 42, 300, seed=73)             # T = 42 (not a multiple of 4) needs a padded pitch
    assert_picks_a_maximum(run(pkg, z, gamma, beta, pitch=44), oracle_values(z, gamma, beta))


@pytest.mark.gpu
@pytest.mark.parametrize("rows,want", [
    ([3000, 250, 17, 5], 5),             # different threads of one warp, different warps, different boxes
    ([3499, 240, 239], 239),             # the last thread of box 0 against the first row of box 1
    ([1200, 480, 721], 480),
])
def test_equal_maxima_give_the_smallest_row(pkg, rows, want):
    """gamma = 0: every value of a frame is its beta exactly, so the tied rows are exactly equal in float32."""
    B, T, V = 3, 37, 3500
    z, _, _, _ = make_z(B, T, V, seed=74, bumped=False)
    gamma = np.zeros(V, np.float32)
    beta = np.random.RandomState(5).uniform(-1.0, 1.0, V).astype(np.float32)
    beta[rows] = 2.5
    assert np.array_equal(run(pkg, z, gamma, beta, pitch=40), np.full((B, T), want))


@pytest.mark.gpu
def test_nan_counts_as_maximal_and_the_first_nan_wins(pkg):
    B, T, V = 2, 24, 3500
    z, _, _, _ = make_z(B, T, V, seed=75, bumped=False)
    gamma = np.zeros(V, np.float32)
    beta = np.random.RandomState(6).uniform(-1.0, 1.0, V).astype(np.float32)
    beta[3] = 100.0
    beta[[2900, 700, 1900]] = np.nan
    assert np.array_equal(run(pkg, z, gamma, beta), np.full((B, T), 700))


@pytest.mark.gpu
def test_degenerate_frames(pkg):
    """One 8-frame tile (frames 8..15 of utterance 1) holds a NaN in a late box, a +inf, a -inf and a frame of zeros:
    every normalised value of those frames is NaN in the reference, so each gives 0; the other frames of the tile and
    of the batch keep their answers."""
    B, T, V = 2, 24, 3500
    z, gamma, beta, _ = make_z(B, T, V, seed=76, bump=20.0, full_length=True)
    z[1, 3400, 9] = np.nan
    z[1, 1000, 10] = np.inf
    z[1, 17, 11] = -np.inf
    z[1, :, 12] = 0.0
    pick = run(pkg, z, gamma, beta)
    assert list(pick[1, 9:13]) == [0, 0, 0, 0]
    y64 = oracle_values(z, gamma, beta)
    with np.errstate(invalid="ignore"):
        want = y64.argmax(axis=2)
    assert list(want[1, 9:13]) == [0, 0, 0, 0]                 # numpy on the float64 reference says the same
    assert np.array_equal(pick, want)


@pytest.mark.gpu
def test_dev_loop_pipeline(pkg):
    """run/ctc/cnn/train.py:224-234 with the fused tail: greedy ids of z straight into compute_minibatch_error, with the
    toy vocabulary whose bigram tokens are two characters."""
    import torch
    ids = {"_": 0}
    for ch in "abcdefg":
        ids[ch] = len(ids)
    for a in "abc":
        for b in "defg":
            ids[a + b] = len(ids)
    inv = {v: k for k, v in ids.items()}
    V = len(ids)
    B, T = 6, 50
    z, gamma, beta, labels = make_z(B, T, V, seed=77, bump=20.0, full_length=True)
    tb = labels.copy()
    dev = torch.device("cuda:0")
    buf = torch.zeros((B, V, 52), device=dev)                   # T = 50: rows need a pitch that is a multiple of 4
    buf[:, :, :T] = torch.tensor(z, device=dev)
    y = pkg.layernorm_greedy_argmax(buf[:, :, :T].unsqueeze(2), torch.tensor(gamma, device=dev),
                                    torch.tensor(beta, device=dev))
    got = pkg.compute_minibatch_error(y, torch.tensor(tb, device=dev), 0, ids, inv)
    y64 = oracle_values(z, gamma, beta)
    table = pkg.build_expansion_table(ids, inv).numpy()
    want, _, _ = oerr.minibatch_error(y64.argmax(axis=2), tb, 0, table)
    assert got == want


class _Cai(object):
    def __init__(self, t):
        self.t = t
        self.__cuda_array_interface__ = t.__cuda_array_interface__


class _Variable(object):                     # what a Chainer Variable offers: the array under .array
    def __init__(self, a):
        self.array = a


@pytest.mark.gpu
def test_foreign_inputs_and_graph_capture(pkg):
    import torch
    dev = torch.device("cuda:0")
    z, gamma, beta, _ = make_z(4, 64, 500, seed=78)
    zt = torch.tensor(z, device=dev).unsqueeze(2)
    gt, bt = torch.tensor(gamma, device=dev), torch.tensor(beta, device=dev)
    want = pkg.layernorm_greedy_argmax(zt, gt, bt)
    for args in ((_Cai(zt), _Cai(gt), _Cai(bt)), (_Variable(_Cai(zt)), _Variable(gt), _Variable(bt))):
        assert torch.equal(pkg.layernorm_greedy_argmax(*args), want)
    # gamma/beta that require grad, in float64 and (V, 1) shape: converted, no autograd edge
    g64 = torch.tensor(gamma, device=dev, dtype=torch.float64).reshape(-1, 1).requires_grad_(True)
    out = pkg.layernorm_greedy_argmax(zt.clone().requires_grad_(True), g64, bt.double())
    assert torch.equal(out, want) and out.grad_fn is None and not out.requires_grad
    # one call captured in a CUDA graph, replayed on new data copied into the captured z
    static_z = zt.clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        pkg.layernorm_greedy_argmax(static_z, gt, bt)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static_out = pkg.layernorm_greedy_argmax(static_z, gt, bt)
    z2, _, _, _ = make_z(4, 64, 500, seed=79)
    z2t = torch.tensor(z2, device=dev).unsqueeze(2)
    static_z.copy_(z2t)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(static_out, pkg.layernorm_greedy_argmax(z2t, gt, bt))
    assert not torch.equal(static_out, want)


@pytest.mark.gpu
def test_refusals_and_empty_shapes(pkg):
    import torch
    dev = torch.device("cuda:0")
    with pytest.raises(NotImplementedError):                  # V above 17 boxes of 240 rows
        pkg.layernorm_greedy_argmax(torch.zeros((1, 5000, 1, 16), device=dev), torch.ones(5000), torch.zeros(5000))
    with pytest.raises(NotImplementedError):                  # rows of 18 floats are not 16-byte aligned
        pkg.layernorm_greedy_argmax(torch.zeros((2, 40, 1, 18), device=dev), torch.ones(40), torch.zeros(40))
    with pytest.raises(ValueError):
        pkg.layernorm_greedy_argmax(torch.zeros((2, 40, 1, 16), device=dev), torch.ones(39), torch.zeros(40))
    with pytest.raises(ValueError):
        pkg.layernorm_greedy_argmax(torch.zeros((2, 40, 2, 16), device=dev), torch.ones(40), torch.zeros(40))
    for B, T in ((0, 16), (3, 0)):
        out = pkg.layernorm_greedy_argmax(torch.zeros((B, 40, 1, T), device=dev), torch.ones(40), torch.zeros(40))
        assert tuple(out.shape) == (B, T) and out.dtype == torch.int64 and out.is_cuda


def test_host_side_refusals(pkg):
    import torch
    with pytest.raises(RuntimeError):
        pkg.layernorm_greedy_argmax(torch.zeros((2, 40, 1, 16)), torch.ones(40), torch.zeros(40))
    with pytest.raises(TypeError):
        pkg.layernorm_greedy_argmax(torch.zeros((2, 40, 1, 16), dtype=torch.float64), torch.ones(40), torch.zeros(40))
    with pytest.raises(TypeError):
        pkg.layernorm_greedy_argmax(np.zeros((2, 40, 1, 16), np.float32), np.ones(40), np.zeros(40))


def test_c_abi_status_codes_without_a_device(pkg):
    L = pkg._lib
    fn = L.load().b200ctc_ln_greedy_argmax
    fake = 1 << 20                           # 16-byte aligned, never dereferenced: every call below returns before
    assert fn(None, 0, 0, None, None, 0, 8, 10, None, None) == L.OK                 # B*T == 0: nothing to do
    assert fn(None, 0, 0, None, None, 4, 0, 10, None, None) == L.OK
    assert fn(fake, 80, 8, fake, fake, 1, 8, 0, fake, None) == L.INVALID_ARGUMENT  # V = 0
    assert fn(fake, 80, 8, fake, fake, -1, 8, 10, fake, None) == L.INVALID_ARGUMENT
    assert fn(None, 80, 8, fake, fake, 1, 8, 10, fake, None) == L.INVALID_ARGUMENT  # NULL z
    assert fn(fake, 80, 8, fake, fake, 1, 8, 10, None, None) == L.INVALID_ARGUMENT  # NULL output
    assert fn(fake, 5000 * 16, 16, fake, fake, 1, 16, 5000, fake, None) == L.UNSUPPORTED   # V > 4080
    assert fn(fake, 40 * 18, 18, fake, fake, 1, 18, 40, fake, None) == L.UNSUPPORTED       # pitch % 4 != 0
    assert fn(fake + 4, 40 * 16, 16, fake, fake, 1, 16, 40, fake, None) == L.UNSUPPORTED   # unaligned base
    assert "4080" in L.last_error()
