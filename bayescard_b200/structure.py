"""Structure learning on the GPU: the Chow-Liu tree of a discretised table, and a model learned from it.

Stands in for pomegranate's ``BayesianNetwork.from_samples(algorithm='chow-liu', root=0)`` of the reference
(``Models/BN_single_model.py:141-202``).  The joint counts of every pair of columns are one int8 tensor-core GEMM
(``bc_pair_counts``, ``csrc/bc_structure.cu``); mutual information is computed from them on the device and Prim's
algorithm runs inside the library (``bc_chow_liu``).  :func:`learn_tree_model` then takes the CPTs from the same
counts -- no second pass over the table -- normalised exactly as :mod:`.fit` normalises them.  torch only moves
buffers.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence, Tuple

import numpy as np

from . import _lib as L
from .fit import count_layout, counts_to_cpts
from .loader import TreeModel, topological_order


def pair_count_layout(card: Sequence[int]) -> Tuple[np.ndarray, np.ndarray, int]:
    """``(marg_off[n], pair_off[n, n], total)`` of the flat counter vector of ``bc_pair_counts``: the marginal counts of
    column i at ``marg_off[i]``; the card_i x card_j block of a pair i < j (row-major) at ``pair_off[i, j]``
    (-1 where i >= j); ``total`` counters (the skipped-row counter follows them)."""
    card = np.asarray(card, dtype=np.int64)
    n = len(card)
    marg_off = np.concatenate([[0], np.cumsum(card)[:-1]]).astype(np.int64)
    pair_off = np.full((n, n), -1, dtype=np.int64)
    total = int(card.sum())
    for i in range(n):
        for j in range(i + 1, n):
            pair_off[i, j] = total
            total += int(card[i] * card[j])
    return marg_off, pair_off, total


def _check_table(table: np.ndarray, card) -> Tuple[np.ndarray, np.ndarray]:
    table = np.ascontiguousarray(table)
    card = np.ascontiguousarray(card, dtype=np.int32)
    if table.dtype not in (np.uint8, np.uint16) or table.ndim != 2 or table.shape[1] != len(card):
        raise ValueError("table must be [n_rows, n_cols] uint8 or uint16 with one card per column")
    return table, card


def pair_counts_device(card: Sequence[int], table_ptr: int, n_rows: int, elem_bytes: int, row_stride_elems: int,
                       counts_ptr: int, device: int = 0, stream: int = 0, want_bad_rows: bool = False) -> Optional[int]:
    """One stream-ordered counting pass on DEVICE buffers (raw addresses).  ``counts_ptr`` must have room for
    ``pair_count_layout(card)[2] + 1`` 64-bit counters (the last one receives the number of skipped rows)."""
    card = np.ascontiguousarray(card, dtype=np.int32)
    total = pair_count_layout(card)[2]
    bad = C.c_uint32(0)
    L.check(L.lib().bc_pair_counts(device, len(card), card.ctypes.data, table_ptr or None, elem_bytes, n_rows,
                                   row_stride_elems, counts_ptr, total, C.byref(bad) if want_bad_rows else None,
                                   stream or None))
    return int(bad.value) if want_bad_rows else None


def pair_counts(table: np.ndarray, card: Sequence[int], device: int = 0) -> Tuple[np.ndarray, int]:
    """Host table -> ``(counts uint64[total], skipped rows)`` in the layout of :func:`pair_count_layout`."""
    import torch

    table, card = _check_table(table, card)
    total = pair_count_layout(card)[2]
    dev = torch.device("cuda", device)
    with torch.cuda.device(dev):
        d_table = torch.from_numpy(table.view(np.uint8)).to(dev)
        d_counts = torch.empty(total + 1, dtype=torch.int64, device=dev)
        bad = pair_counts_device(card, d_table.data_ptr() if table.shape[0] else 0, table.shape[0], table.dtype.itemsize,
                                 table.shape[1], d_counts.data_ptr(), device, torch.cuda.current_stream().cuda_stream, True)
        counts = d_counts[:total].cpu().numpy().astype(np.uint64)
    return counts, bad


def _chow_liu(table: np.ndarray, card, root: int, device: int, want_counts: bool):
    import torch

    table, card = _check_table(table, card)
    n = len(card)
    total = pair_count_layout(card)[2] if want_counts else 0
    parent = np.zeros(n, dtype=np.int32)
    mi = np.zeros((n, n), dtype=np.float64)
    bad = C.c_uint32(0)
    dev = torch.device("cuda", device)
    with torch.cuda.device(dev):
        d_table = torch.from_numpy(table.view(np.uint8)).to(dev)
        d_counts = torch.empty(total + 1, dtype=torch.int64, device=dev) if want_counts else None
        L.check(L.lib().bc_chow_liu(device, n, card.ctypes.data, d_table.data_ptr() if table.shape[0] else None,
                                    table.dtype.itemsize, table.shape[0], table.shape[1], root,
                                    d_counts.data_ptr() if want_counts else None, total, parent.ctypes.data, mi.ctypes.data,
                                    C.byref(bad), torch.cuda.current_stream().cuda_stream or None))
        counts = d_counts[:total].cpu().numpy().astype(np.uint64) if want_counts else None
    return parent, mi, int(bad.value), counts


def mutual_information(table: np.ndarray, card: Sequence[int], device: int = 0) -> Tuple[np.ndarray, int]:
    """``(MI [n, n] fp64, skipped rows)``: MI[i][j] = sum_ab (n_ab/N) log(N n_ab / (n_a n_b)) over n_ab > 0, N = rows
    kept (pomegranate's mutual information with pseudocount 0, times N).  Symmetric, zero diagonal."""
    _, mi, bad, _ = _chow_liu(table, card, 0, device, False)
    return mi, bad


def chow_liu(table: np.ndarray, card: Sequence[int], root: int = 0, device: int = 0) -> Tuple[np.ndarray, np.ndarray, int]:
    """``(parent[n], MI, skipped rows)``: the Chow-Liu tree in table column order (parent -1 for ``root``), with
    pomegranate's tie rule (see ``bc_chow_liu`` in include/bayescard_b200.h)."""
    parent, mi, bad, _ = _chow_liu(table, card, root, device, False)
    return parent, mi, bad


def learn_tree_model(table: np.ndarray, card: Sequence[int], names: Optional[Sequence[str]] = None, root: int = 0,
                     device: int = 0, table_name: str = "table") -> TreeModel:
    """Table of bin ids in, model out: the Chow-Liu tree rooted at column ``root``, numbered like the reference's
    ``align_cpds_in_topological`` (:func:`.loader.topological_order`), with maximum-likelihood CPTs (pgmpy's MLE, as
    :func:`.fit.counts_to_cpts`) gathered from the pair counts the tree was learned from.  Every column is categorical
    with bin id b encoded as the value b.  Rows holding a bin id outside their column's domain raise."""
    table, card = _check_table(table, card)
    names = [f"c{i}" for i in range(len(card))] if names is None else [str(x) for x in names]
    if len(names) != len(card) or len(set(names)) != len(names):
        raise ValueError("one distinct name per column")
    parent, _, bad, counts = _chow_liu(table, card, root, device, True)
    if bad:
        raise ValueError(f"{bad} rows hold a bin id outside the columns' domains")
    return model_from_counts(parent, card, counts, names, root, table_name, int(table.shape[0]))


def model_from_counts(parent: Sequence[int], card: Sequence[int], counts: np.ndarray, names: Sequence[str], root: int = 0,
                      table_name: str = "table", nrows: int = 0) -> TreeModel:
    """The TreeModel of a tree given in table column order (``parent[root] = -1``), its CPTs gathered from pair counts
    in the layout of :func:`pair_count_layout`."""
    card = np.asarray(card, dtype=np.int64)
    n = len(card)
    names = list(names)
    structure = tuple(() if parent[i] < 0 else (int(parent[i]),) for i in range(n))
    order = topological_order(structure)
    pos = {c: v for v, c in enumerate(order)}
    t_parent = np.asarray([-1 if parent[c] < 0 else pos[int(parent[c])] for c in order], dtype=np.int32)
    t_card = card[order].astype(np.int32)
    # counts of every node in fit.count_layout order: [own bin][parent bin]
    marg_off, pair_off, _ = pair_count_layout(card)
    off, total = count_layout(t_parent, t_card)
    flat = np.empty(total, dtype=np.uint64)
    for v, c in enumerate(order):
        p = int(parent[c])
        if p < 0:
            blk = counts[marg_off[c]: marg_off[c] + card[c]]
        elif c < p:
            blk = counts[pair_off[c, p]: pair_off[c, p] + card[c] * card[p]]
        else:  # block (p, c) is [parent bin][own bin]
            blk = counts[pair_off[p, c]: pair_off[p, c] + card[p] * card[c]].reshape(card[p], card[c]).T
        flat[off[v]: off[v] + blk.size] = np.asarray(blk).reshape(-1)
    cpts = counts_to_cpts(t_parent, t_card, flat)
    topo_names = [names[c] for c in order]
    return TreeModel(
        table_name=table_name, nrows=nrows, node_names=names, structure=structure,
        attr_type={k: "categorical" for k in names}, algorithm="chow-liu", topo_names=topo_names, infer_names=topo_names,
        parent=t_parent, card=t_card, cpts=cpts, dropped_names=[],
        encoding={names[i]: {b: b for b in range(int(card[i]))} for i in range(n)},
        domain={names[i]: list(range(int(card[i]))) for i in range(n)}, root=root,
        counts=flat, fit_rows=int(flat[: int(t_card[0])].sum()))
