"""Numpy fp64 reference for structure learning -- TEST INFRASTRUCTURE ONLY, like ``oracle/bayescard_oracle.py``.

The checker of ``bc_pair_counts`` / ``bc_chow_liu`` (``tests/test_structure.py``) and the CPU timing of
``tools/structure_bench.py``: all-pairs counts by ``np.bincount``, mutual information, and Prim's algorithm written as
pomegranate's ``discrete_chow_liu_tree`` loops (reference ``Models/BN_single_model.py:141-202`` calls
``BayesianNetwork.from_samples(algorithm='chow-liu', root=0)``).  The product package never imports it.
"""
from __future__ import annotations

import numpy as np

def pair_counts(card, table):
    """Marginal counts of every column, then for every pair i < j (row-major pair order) the card_i x card_j joint
    counts, row-major, as one flat uint64 vector (the layout of ``bc_pair_counts``).  Rows holding an id >= card are
    skipped, as in ``fit_counts``.  Returns ``(counts, skipped)``."""
    table = np.asarray(table).astype(np.int64)
    card = np.asarray(card, dtype=np.int64)
    ok = (table < card[None, :]).all(axis=1) if table.size else np.zeros(len(table), dtype=bool)
    t = table[ok]
    n = len(card)
    out = [np.bincount(t[:, i], minlength=int(card[i])) for i in range(n)]
    for i in range(n):
        for j in range(i + 1, n):
            out.append(np.bincount(t[:, i] * card[j] + t[:, j], minlength=int(card[i] * card[j])))
    return np.concatenate(out).astype(np.uint64), int((~ok).sum())


def mutual_information(card, counts, n_kept):
    """MI[i][j] = sum_ab (n_ab/N) log(N n_ab / (n_a n_b)) over n_ab > 0 (fp64, symmetric, zero diagonal): pomegranate's
    mutual information with its default pseudocount 0, times N."""
    card = [int(c) for c in card]
    n = len(card)
    first = np.concatenate([[0], np.cumsum(card)]).astype(np.int64)
    N = float(n_kept)
    mi = np.zeros((n, n))
    off = int(first[-1])
    for i in range(n):
        for j in range(i + 1, n):
            blk = counts[off: off + card[i] * card[j]].astype(np.float64).reshape(card[i], card[j])
            off += card[i] * card[j]
            na = counts[first[i]: first[i + 1]].astype(np.float64)
            nb = counts[first[j]: first[j + 1]].astype(np.float64)
            a, b = np.nonzero(blk)
            f = blk[a, b]
            mi[i, j] = mi[j, i] = float(np.sum((f / N) * np.log((N * f) / (na[a] * nb[b]))))
    return mi


def chow_liu(mi, root=0):
    """Prim's maximum spanning tree as pomegranate's ``discrete_chow_liu_tree`` loops: per step the (in-tree x, outside y)
    pair of largest MI, x in the order the nodes joined, y ascending, only a strictly larger MI replacing the best.
    Returns parent[n] (-1 for the root)."""
    n = len(mi)
    parent = np.full(n, -1, dtype=np.int32)
    visited, unvisited = [root], [y for y in range(n) if y != root]
    for _ in range(n - 1):
        best, bx, by = -np.inf, -1, -1
        for x in visited:
            for y in unvisited:
                if mi[x][y] > best:
                    best, bx, by = mi[x][y], x, y
        parent[by] = bx
        visited.append(by)
        unvisited.remove(by)
    return parent
