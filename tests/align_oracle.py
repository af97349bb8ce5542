"""Float64 restatement of the forced alignment (the Viterbi path through the loss's lattice), for the tests.

It runs over the edge sets of ``oracle.lattice`` (the loss's lattice) with the tie rule of ``b200ctc_align``: among a
node's predecessors the smallest back-offset wins, among the end nodes the final blank, then N-2, then N-3.  The
brute-force twin below is independent of any lattice: the maximum over every frame labelling whose collapse and
gram expansion is the target.
"""
import itertools

import numpy as np

from oracle import brute_force
from oracle.lattice import ctc_lattice, gram_ctc_lattice, log_softmax   # noqa: F401  (re-exported for the tests)

NEG_INF = -np.inf


def lattice_kind(lat):
    """Nodes per label: 2 (CTC) or 3 (Gram-CTC)."""
    return 3 if len(lat.edges) > 3 else 2


def viterbi(logp_tv, lat):
    """Best path of ``lat`` on log-probabilities (T,V).  Returns (score, path, spans): score = -ln P(best path)
    (inf when no path exists), path = node per frame (None without a path), spans = (L,2) [first, last+1) frame of
    the node that emits each label position (None without a path)."""
    logp = np.asarray(logp_tv, np.float64)
    T = logp.shape[0]
    N = lat.N
    per = lattice_kind(lat)
    L = (N - 1) // per
    if T == 0:
        ok = N == 1
        return (0.0 if ok else np.inf), (np.zeros(0, np.int64) if ok else None), (np.zeros((0, 2), np.int64) if ok else None)
    emit = np.where(lat.dead, NEG_INF, logp[:, np.where(lat.dead, 0, lat.symbols)])
    edges = sorted(lat.edges, key=lambda e: e[0])
    prev = np.full(N, NEG_INF)
    prev[0] = 0.0
    bp = np.zeros((T, N), np.int64)
    for t in range(T):
        best = np.full(N, NEG_INF)
        arg = np.zeros(N, np.int64)
        for k, allowed in edges:
            shifted = np.full(N, NEG_INF)
            if k < N:
                shifted[k:] = prev[:N - k]
            cand = np.where(allowed, shifted, NEG_INF)
            upd = cand > best
            best = np.where(upd, cand, best)
            arg = np.where(upd, k, arg)
        prev = np.where(lat.dead, NEG_INF, best + emit[t])
        bp[t] = arg
    jend, best = -1, NEG_INF
    for j in lat.final_nodes:                  # N-1, N-2, N-3 in that order
        if prev[j] > best:
            jend, best = j, prev[j]
    if jend < 0:
        return np.inf, None, None
    path = np.zeros(T, np.int64)
    j = jend
    for t in range(T - 1, -1, -1):
        path[t] = j
        j -= bp[t, j]
    return -float(best), path, path_spans(path, per, L)


def node_positions(j, per):
    """Label positions node j emits (empty for a blank)."""
    i, typ = divmod(j, per) if per == 3 else (j // 2, j % 2)
    if typ == 0:
        return []
    return [i - 1, i] if (per == 3 and typ == 2) else [i]


def path_spans(path, per, L):
    spans = np.full((L, 2), -1, np.int64)
    T = len(path)
    for t, j in enumerate(path):
        for q in node_positions(int(j), per):
            if t == 0 or path[t - 1] != j:
                spans[q, 0] = t
            if t == T - 1 or path[t + 1] != j:
                spans[q, 1] = t + 1
    return spans


def rescore(logp_tv, lat, path):
    """ln P of a given node path, or None when it is not a path of the lattice (start, edges, end)."""
    logp = np.asarray(logp_tv, np.float64)
    T = len(path)
    edge_ok = {k: allowed for k, allowed in lat.edges}
    prev = 0                                  # virtual start node
    total = 0.0
    for t in range(T):
        j = int(path[t])
        if j < 0 or j >= lat.N or lat.dead[j]:
            return None
        k = j - prev
        if k not in edge_ok or not edge_ok[k][j]:
            return None
        total += logp[t, lat.symbols[j]]
        prev = j
    if T > 0 and int(path[-1]) not in lat.final_nodes:
        return None
    return total


def max_log_likelihood(logp_tv, target_chars, gram_to_chars, blank=0):
    """Max-over-labellings twin of ``oracle.brute_force.log_likelihood`` (tiny T and V only)."""
    logp = np.asarray(logp_tv, np.float64)
    T, V = logp.shape
    target = tuple(target_chars)
    best = NEG_INF
    usable = [k for k in range(V) if k == blank or k in gram_to_chars]
    for ids in itertools.product(usable, repeat=T):
        chars = []
        for k in brute_force.collapse(ids, blank):
            chars.extend(gram_to_chars[k])
        if tuple(chars) == target:
            best = max(best, float(sum(logp[t, k] for t, k in enumerate(ids))))
    return best
