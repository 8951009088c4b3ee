"""fp64 helpers for GROUP BY two columns -- TEST INFRASTRUCTURE ONLY, like ``groupby_oracle.py``.

``joint(m, W, a, b)`` is the checker of ``bc_joint_marginal_batch``: ``groupby_oracle.marginal(b)`` with a's weights masked
to each state of a in turn, i.e. ``out[i][j] = sum_{x : x_a = i, x_b = j} prod_v w_v[x_v] T_v[x_v, x_pa(v)]``.
``brute_force`` enumerates every joint state of a tiny tree.  ``joint_ffma`` counts the CPT-carrying FMAs of a generated
joint module from the CPTs with the generator's rules (the number its header reports as BC_SPEC_FFMA).  The generated
bodies run on the host through ``join_groupby_oracle.interpret_masked``: their per-state stores are plain ``[%rtmp+off]``
stores.
"""
from __future__ import annotations

import itertools

import numpy as np

import groupby_oracle as GO


def joint(m, W, a, b):
    """``W``: per node ``[card_v]`` or ``[B, card_v]`` weights.  Returns ``[card_a, card_b]`` or ``[B, card_a, card_b]``."""
    cols = []
    for i in range(int(m.card[a])):
        Wi = list(W)
        onehot = np.zeros(int(m.card[a]))
        onehot[i] = 1.0
        Wi[a] = np.asarray(W[a], dtype=np.float64) * onehot
        cols.append(GO.marginal(m, Wi, b))
    return np.stack(cols, axis=-2)


def brute_force(m, W, a, b):
    """Sum over every joint assignment of a tiny tree: ``[card_a, card_b]`` for per-node ``[card_v]`` W."""
    n = len(m.infer_names)
    out = np.zeros((int(m.card[a]), int(m.card[b])))
    for x in itertools.product(*[range(int(c)) for c in m.card]):
        p = 1.0
        for v in range(n):
            T = np.asarray(m.cpts[v], dtype=np.float64)
            p *= W[v][x[v]] * (T.reshape(-1)[x[v]] if v == 0 else T[x[v], x[int(m.parent[v])]])
        out[x[a], x[b]] += p
    return out


def _root_path(m, v):
    p = [v]
    while v > 0:
        v = int(m.parent[v])
        p.append(v)
    return p[::-1]


def joint_ffma(m, a, b, X):
    """FMA-pipe instructions carrying a CPT entry in the joint module of (a, b) with loop node X: one per non-zero entry of
    every node off the X - c - Y path and of the chain root -> c, plus, per state i of X, one per non-zero entry that meets
    a structurally non-zero input on the way from row i of T_X (or column i of the first CPT below c when X == c) to Y."""
    Y = b if X == a else a
    nz = [np.asarray(c, dtype=np.float32).reshape(int(m.card[v]), -1) != 0 for v, c in enumerate(m.cpts)]
    px, py = _root_path(m, X), _root_path(m, Y)
    d = 0
    while d + 1 < len(px) and d + 1 < len(py) and px[d + 1] == py[d + 1]:
        d += 1
    c, up, down = px[d], px[d + 1:], py[d + 1:]
    count = sum(int(nz[v].sum()) for v in range(m.n_nodes) if v not in up and v not in down)
    pz = ~nz[c].any(axis=1)   # all-zero CPT rows of c
    for i in range(int(m.card[X])):
        if up:
            vec = nz[X][i]
            count += int(vec.sum())
            for w in reversed(up[:-1]):
                count += int(nz[w][vec].sum())
                vec = nz[w][vec].any(axis=0)
            r = vec & ~pz
            rest = down
        else:
            col = nz[down[0]][:, i] if not pz[i] else np.zeros(int(m.card[down[0]]), dtype=bool)
            count += int(col.sum())
            r, rest = col, down[1:]
        for v in rest:
            count += int(nz[v][:, r].sum())
            r = nz[v][:, r].any(axis=1)
    return count
