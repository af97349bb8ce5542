"""NumPy restatement of the reference CTC / Gram-CTC loss on the banded lattice.

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).  float64 by default, so it doubles as the
noise-free ground truth SURVEY.md section 7.3 asks for.

What it follows in the reference (``/root/reference/asr/loss/gram_ctc.py``):
  * node symbols            -- ``_label_to_path``                         :24-32
  * forward edges           -- ``_create_forward_connection_matrix``      :66-99
  * backward edges          -- ``_create_backward_connection_matrix``     :103-140  (here: the
                               transpose of the forward edge set, which is what that matrix is
                               once un-reversed)
  * alpha / beta convention -- ``_compute_transition_probability``        :142-178  (beta at frame
                               t EXCLUDES the emission at t, so alpha_t + beta_t sums to log P)
  * loss                    -- ``GramCTC.forward``                        :279-281
  * gradient, scale, mask   -- ``GramCTC.backward``                       :284-297
  * per-symbol merge        -- ``_compute_label_probability``             :180-217

The reference evaluates each frame as a dense (B,N,N) log-matmul; the adjacency it builds has at
most four non-zeros per row, so this file evaluates the same recurrence edge by edge.  Where the
reference represents log(0) by -1e10 (:222) this file uses -inf; the only observable difference
is on infeasible alignments, which ``loss_and_grad`` maps back to the reference's 1e10.
"""
import numpy as np

NEG_INF = -np.inf
REF_ZERO_PADDING = -10000000000.0     # gram_ctc.py:222


class Lattice(object):
    """One utterance's lattice: node symbols + banded predecessor structure.

    ``edges`` is a list of (k, allowed) with ``allowed`` a bool array over nodes: node j has the
    predecessor j-k iff allowed[j] (and j-k >= 0).  Dead nodes have no edges at all.
    """

    def __init__(self, symbols, dead, edges, final_nodes):
        self.symbols = np.asarray(symbols, np.int64)
        self.dead = np.asarray(dead, bool)
        self.edges = edges
        self.final_nodes = list(final_nodes)
        self.N = len(self.symbols)


def ctc_lattice(labels, blank):
    """Classic blank-interleaved lattice, N = 2L+1 (SURVEY.md section 3.2 / 8a row a16)."""
    labels = np.asarray(labels, np.int64)
    L = len(labels)
    N = 2 * L + 1
    sym = np.full(N, blank, np.int64)
    sym[1::2] = labels
    idx = np.arange(N)
    is_label = (idx % 2) == 1
    skip = np.zeros(N, bool)
    for j in range(3, N, 2):
        i = j // 2
        skip[j] = labels[i] != labels[i - 1]
    edges = [(0, np.ones(N, bool)), (1, idx >= 1), (2, is_label & skip)]
    return Lattice(sym, np.zeros(N, bool), edges, [n for n in (N - 1, N - 2) if n >= 0])


def gram_ctc_lattice(unigram, bigram, blank):
    """Unigram+bigram lattice, N = 3L+1 (gram_ctc.py:24-32, :66-99; SURVEY.md 'banded lattice spec').

    node j: i = j // 3, type = j % 3: 0 blank, 1 unigram_i, 2 bigram_i (covers chars i-1,i; id -1 = dead).
    """
    unigram = np.asarray(unigram, np.int64)
    bigram = np.asarray(bigram, np.int64)
    L = len(unigram)
    N = 3 * L + 1
    sym = np.full(N, blank, np.int64)
    sym[1::3] = unigram
    sym[2::3] = bigram
    idx = np.arange(N)
    typ = idx % 3
    dead = np.zeros(N, bool)
    dead[2::3] = bigram == -1                          # :94-98
    uni_differs = np.zeros(N, bool)                    # k=3, :70-73,84
    bi_differs = np.zeros(N, bool)                     # k=6, :75-78,85
    for i in range(1, L):
        uni_differs[3 * i + 1] = unigram[i] != unigram[i - 1]
    for i in range(2, L):
        bi_differs[3 * i + 2] = bigram[i] != bigram[i - 2]
    edges = [
        (0, np.ones(N, bool)),                         # :82
        (1, typ != 2), (2, typ != 2),                  # :83
        (3, (typ == 1) & uni_differs),                 # :84
        (6, (typ == 2) & bi_differs),                  # :85
        (5, typ == 2), (7, typ == 2),                  # :86
    ]
    # a dead node neither receives nor sends (:95-98)
    alive = ~dead
    pruned = []
    for k, allowed in edges:
        a = allowed & alive & (idx - k >= 0)
        src_alive = np.zeros(N, bool)
        if k < N:
            src_alive[k:] = alive[:N - k]
        pruned.append((k, a & src_alive))
    finals = [n for n in (N - 1, N - 2, N - 3) if n >= 0 and not dead[n]]
    return Lattice(sym, dead, pruned, finals)


def _lse(values, axis=None):
    values = np.asarray(values)
    m = np.max(values, axis=axis, keepdims=True)
    m = np.where(np.isfinite(m), m, 0.0)
    with np.errstate(divide="ignore"):
        out = m + np.log(np.sum(np.exp(values - m), axis=axis, keepdims=True))
    return np.squeeze(out, axis=axis) if axis is not None else out.reshape(())


def log_softmax(x, dtype=np.float64):
    """gram_ctc.py:18-21 + :274 as one numerically exact step."""
    x = np.asarray(x, dtype)
    m = np.max(x, axis=-1, keepdims=True)
    e = np.exp(x - m)
    s = np.sum(e, axis=-1, keepdims=True)
    return (x - m) - np.log(s)


def alpha_beta(logp_tv, lat, dtype=np.float64):
    """alpha[t,j] (includes emission at t) and beta[t,j] (EXCLUDES emission at t); gram_ctc.py:142-178."""
    T = logp_tv.shape[0]
    N = lat.N
    emit = np.where(lat.dead, NEG_INF, logp_tv[:, np.where(lat.dead, 0, lat.symbols)]).astype(dtype)  # (T,N)
    alpha = np.full((T, N), NEG_INF, dtype)
    prev = np.full(N, NEG_INF, dtype)
    prev[0] = 0.0                                       # :144 virtual state before frame 0
    for t in range(T):
        terms = np.full((len(lat.edges), N), NEG_INF, dtype)
        for e, (k, allowed) in enumerate(lat.edges):
            shifted = np.full(N, NEG_INF, dtype)
            if k < N:
                shifted[k:] = prev[:N - k]
            terms[e] = np.where(allowed, shifted, NEG_INF)
        prev = emit[t] + _lse(terms, axis=0)
        prev = np.where(lat.dead, NEG_INF, prev)
        alpha[t] = prev
    beta = np.full((T, N), NEG_INF, dtype)
    nxt = np.full(N, NEG_INF, dtype)                    # virtual state after the last frame:
    end_node = N - 1                                    # all mass on the final blank, emission prob 1
    nxt[end_node] = 0.0
    for t in range(T - 1, -1, -1):
        # beta_t[j'] = LSE over successors j of (beta_{t+1}[j] + emit_{t+1}[j]); nxt already holds that sum
        terms = np.full((len(lat.edges), N), NEG_INF, dtype)
        for e, (k, allowed) in enumerate(lat.edges):
            contrib = np.where(allowed, nxt, NEG_INF)   # value at destination j, sent back to j-k
            shifted = np.full(N, NEG_INF, dtype)
            if k < N:
                shifted[:N - k] = contrib[k:]
            terms[e] = shifted
        b = _lse(terms, axis=0)
        b = np.where(lat.dead, NEG_INF, b)
        beta[t] = b
        nxt = b + emit[t]
    return alpha, beta


def utterance(logp_tv, lat, dtype=np.float64):
    """Returns (logP, gamma[t,j] = alpha+beta-logP, posterior[t,V])."""
    T, V = logp_tv.shape
    alpha, beta = alpha_beta(logp_tv, lat, dtype)
    finals = lat.final_nodes
    if T > 0:
        logP = _lse(alpha[T - 1, finals]) if finals else np.array(NEG_INF)
    else:                                               # no frames: P = 1 iff there is nothing to emit (DESIGN.md quirks)
        logP = np.array(0.0 if lat.N == 1 else NEG_INF)
    logP = float(logP)
    post = np.zeros((T, V), dtype)
    if np.isfinite(logP):
        with np.errstate(invalid="ignore"):
            gamma = alpha + beta - logP
        gamma = np.where(np.isnan(gamma), NEG_INF, gamma)
        w = np.exp(gamma)
        for j in range(lat.N):
            if not lat.dead[j]:
                post[:, lat.symbols[j]] += w[:, j]      # :180-217 merged in linear space
    else:
        gamma = np.full((T, lat.N), NEG_INF, dtype)
    return logP, gamma, post


def loss_and_grad(x_tbv, lattices, input_length, dtype=np.float64, gy=None, reduce="no", batch_global=None):
    """Loss (B,) or scalar and d loss / d x (T,B,V).  gram_ctc.py:279-297.

    infeasible alignment => loss = 1e10 (what the reference returns, SURVEY.md 8a quirks) and a
    zero posterior (gradient = softmax on the valid frames).
    """
    x = np.asarray(x_tbv, dtype)
    T, B, V = x.shape
    loss = np.zeros(B, dtype)
    grad = np.zeros((T, B, V), dtype)
    for b in range(B):
        Tb = int(input_length[b])
        logp = log_softmax(x[:Tb, b], dtype)
        logP, _, post = utterance(logp, lattices[b], dtype)
        loss[b] = -logP if np.isfinite(logP) else -REF_ZERO_PADDING
        grad[:Tb, b] = np.exp(logp) - post
    if reduce == "mean":
        n = B if batch_global is None else batch_global
        g = 1.0 if gy is None else float(gy)
        return np.asarray(loss.sum() / n, dtype), grad * (g / n)
    if gy is not None:
        grad = grad * np.asarray(gy, dtype)[None, :, None]
    return loss, grad


def ctc(x_tbv, labels, input_length, label_length, blank=0, dtype=np.float64, **kw):
    lats = [ctc_lattice(np.asarray(labels[b])[:int(label_length[b])], blank) for b in range(len(labels))]
    return loss_and_grad(x_tbv, lats, input_length, dtype, **kw)


def gram_ctc(x_tbv, unigram, bigram, input_length, label_length, blank=0, dtype=np.float64, **kw):
    lats = [gram_ctc_lattice(np.asarray(unigram[b])[:int(label_length[b])],
                             np.asarray(bigram[b])[:int(label_length[b])], blank)
            for b in range(len(unigram))]
    return loss_and_grad(x_tbv, lats, input_length, dtype, **kw)


def greedy_argmax(x):
    """run/ctc/cnn/train.py:232 -- first maximal index, NaN counts as maximal (NumPy semantics)."""
    return np.argmax(np.asarray(x), axis=-1).astype(np.int64)
