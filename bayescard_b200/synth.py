"""Synthetic tree BNs and range-query workloads (BASELINE.json config 4, SURVEY.md section 8d).

Trees are built directly, not through the reference's discretiser (which caps domains at ~100-140 bins,
``Testing/stability_experiment.ipynb`` cell 2, ``Models/tools.py:69``): a random recursive tree (the parent of node i
is uniform over 0..i-1, one root) and CPT columns drawn from Dirichlet(alpha), seeded per node.  Queries follow
config 2: k ~ U{1..kmax} columns without replacement, ``lo ~ U{0..card-1}``, ``hi ~ U{lo..card-1}``.
"""
from __future__ import annotations

import numpy as np

from .loader import TreeModel


def make_tree_model(n_cols: int, card, seed: int = 0, alpha: float = 0.5, dtype=np.float64, parent=None) -> TreeModel:
    """``card`` is an int (every column) or a sequence of n_cols ints; ``parent``: the tree (parent[0] = -1, parent[i] < i),
    random when omitted."""
    rng = np.random.default_rng(seed)
    cards = np.full(n_cols, card, dtype=np.int32) if np.isscalar(card) else np.asarray(card, dtype=np.int32)
    if parent is None:
        parent = np.full(n_cols, -1, dtype=np.int32)
        for i in range(1, n_cols):
            parent[i] = rng.integers(0, i)
    else:
        parent = np.asarray(parent, dtype=np.int32)
        assert parent.shape == (n_cols,) and parent[0] == -1 and all(0 <= parent[i] < i for i in range(1, n_cols))
    cpts = []
    for v in range(n_cols):
        node_rng = np.random.default_rng([seed, v])
        cols = 1 if parent[v] < 0 else int(cards[parent[v]])
        g = node_rng.standard_gamma(alpha, size=(int(cards[v]), cols), dtype=np.float32 if dtype == np.float32 else np.float64)
        g = np.maximum(g, np.finfo(g.dtype).tiny)
        g /= g.sum(axis=0, keepdims=True)
        cpts.append(g.reshape(-1) if parent[v] < 0 else g)
    names = [f"c{v}" for v in range(n_cols)]
    return TreeModel(
        table_name="synthetic", nrows=1_000_000, node_names=names,
        structure=tuple(() if parent[v] < 0 else (int(parent[v]),) for v in range(n_cols)),
        attr_type={k: "categorical" for k in names}, algorithm="chow-liu", topo_names=names, infer_names=names,
        parent=parent, card=cards, cpts=cpts, dropped_names=[])


def random_range_queries(tm: TreeModel, nq: int, seed: int = 0, kmax: int = 10):
    """``(lo, hi)`` int32 arrays ``[nq, n_nodes]``; unconstrained columns are ``[0, card-1]``."""
    rng = np.random.default_rng(seed)
    n = tm.n_nodes
    card = tm.card.astype(np.int64)
    kmax = min(kmax, n)
    k = rng.integers(1, kmax + 1, size=nq)
    # k distinct columns per query: rank random keys
    order = np.argsort(rng.random((nq, n)), axis=1)
    chosen = np.zeros((nq, n), dtype=bool)
    np.put_along_axis(chosen, order, np.arange(n)[None, :] < k[:, None], axis=1)
    lo_r = (rng.random((nq, n)) * card[None, :]).astype(np.int64)
    hi_r = lo_r + (rng.random((nq, n)) * (card[None, :] - lo_r)).astype(np.int64)
    lo = np.where(chosen, lo_r, 0).astype(np.int32)
    hi = np.where(chosen, hi_r, card[None, :] - 1).astype(np.int32)
    return lo, hi


def pack_ranges_u16(lo: np.ndarray, hi: np.ndarray) -> np.ndarray:
    """RANGE_U16 rows: uint16 lo_0, hi_0, lo_1, hi_1, ... (row stride 4*n bytes)."""
    nq, n = lo.shape
    out = np.empty((nq, 2 * n), dtype=np.uint16)
    out[:, 0::2] = lo
    out[:, 1::2] = hi
    return out


def sample_table_device(tm: TreeModel, n: int, seed: int = 0, device: int = 0):
    """Ancestral sample of ``n`` rows of ``tm`` on the device: a ``[n, n_nodes]`` uint8 (uint16 when a card exceeds
    256) torch tensor, columns in the model's topological order.  torch is plumbing here (seeded ``torch.rand``)."""
    import torch

    dev = torch.device("cuda", device)
    dtype = torch.uint8 if int(np.max(tm.card)) <= 256 else torch.int16
    g = torch.Generator(device=dev).manual_seed(seed)
    cols = []
    for v in range(tm.n_nodes):
        pa = int(tm.parent[v])
        t = torch.tensor(np.asarray(tm.cpts[v], dtype=np.float64).reshape(int(tm.card[v]), -1), device=dev)
        cdf = torch.cumsum(t / t.sum(dim=0, keepdim=True), dim=0).T.contiguous()   # [card_pa, card]
        u = torch.rand(n, generator=g, device=dev, dtype=torch.float64)
        idx = cols[pa].long() if pa >= 0 else torch.zeros(n, dtype=torch.long, device=dev)
        out = torch.empty(n, dtype=torch.long, device=dev)
        for s in range(0, n, 1 << 22):   # bounded [rows, card] temporaries
            out[s:s + (1 << 22)] = (cdf[idx[s:s + (1 << 22)]] < u[s:s + (1 << 22), None]).sum(dim=1)
        cols.append(torch.clamp(out, max=int(tm.card[v]) - 1).to(dtype))
    return torch.stack(cols, dim=1).contiguous()
