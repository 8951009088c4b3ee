"""CPT fitting for a fixed tree on the GPU: the step right before the inference path.

Stands in for ``self.model.fit(discrete_table)`` of ``Bayescard_BN.build_from_data`` (reference
``Models/Bayescard_BN.py:108-110``): pgmpy's maximum-likelihood estimate (``Pgmpy/estimators/MLE.py:61-104``) -- per
node the 2-D histogram of (own bin, parent bin), an all-zero column replaced by ones, columns normalised.  The
histogram pass is one CUDA kernel over the discretised table (``bc_fit_counts``, ``csrc/bc_fit.cu``); the few thousand
fp64 divisions happen here, written the way the reference writes them so that the CPTs are bit-identical.

The tree is an input here; :mod:`.structure` learns it (pomegranate's Chow-Liu) from the same kind of table.

A served model follows inserted and deleted rows without a refit (``DeviceModel.update``, DESIGN.md section 9e): it needs
the counts behind its CPTs, which a model fitted here carries and :func:`counts_from_cpts` recovers exactly from any
other model's CPTs and the number of rows they were fitted on (:func:`infer_fit_rows`).
"""
from __future__ import annotations

import copy
import ctypes as C
from fractions import Fraction
from math import lcm
from typing import List, Optional, Sequence, Tuple

import numpy as np

from . import _lib as L
from .loader import TreeModel


def count_layout(parent: Sequence[int], card: Sequence[int]) -> Tuple[np.ndarray, int]:
    """Offsets of the per-node count tables in the flat counter array (node v: card_v x card_pa, [c][p] row-major)."""
    off, total = [], 0
    for v in range(len(card)):
        off.append(total)
        total += int(card[v]) * (int(card[parent[v]]) if parent[v] >= 0 else 1)
    return np.asarray(off, dtype=np.int64), total


def counts_to_cpts(parent: Sequence[int], card: Sequence[int], counts: np.ndarray) -> List[np.ndarray]:
    """``estimate_cpd`` after the counting: zero columns -> ones (MLE.py:77-79), ``values / values.sum(axis=0)``
    (``TabularCPD.normalize``, Pgmpy/factors/discrete/CPD.py).  fp64; the root comes back as a vector."""
    off, total = count_layout(parent, card)
    counts = np.asarray(counts).reshape(-1)
    if counts.size != total:
        raise ValueError(f"{counts.size} counters for a tree that needs {total}")
    return [node_cpt(parent, card, v, counts[off[v]: off[v] + int(card[v]) * (int(card[parent[v]]) if parent[v] >= 0 else 1)])
            for v in range(len(card))]


def node_cpt(parent: Sequence[int], card: Sequence[int], v: int, counts_v: np.ndarray) -> np.ndarray:
    """:func:`counts_to_cpts` of one node from its own counters (``card_v x card_pa``, [c][p] row-major)."""
    cols = int(card[parent[v]]) if parent[v] >= 0 else 1
    t = np.asarray(counts_v).astype(np.float64).reshape(int(card[v]), cols)
    t[:, (t == 0).all(axis=0)] = 1.0
    t = t / t.sum(axis=0)
    return t.reshape(-1) if parent[v] < 0 else t


def counts_from_cpts(parent: Sequence[int], card: Sequence[int], cpts: Sequence[np.ndarray], fit_rows: int) -> np.ndarray:
    """The counts (uint64, :func:`count_layout` order) that CPTs fitted on ``fit_rows`` rows came from, top-down: the
    root's are ``T_root * fit_rows``, node v's are ``T_v[c, p] * n(parent = p)``, each rounded once to the nearest
    integer.  Raises ``ValueError`` naming the node when a product is more than 1e-6 from an integer, when a node's column
    sums differ from its parent's state counts, or when :func:`counts_to_cpts` of the result does not give back ``cpts``
    bit for bit -- i.e. when ``fit_rows`` is not a row count these CPTs were fitted on."""
    fit_rows = int(fit_rows)
    if fit_rows < 0:
        raise ValueError(f"fit_rows = {fit_rows} is negative")
    off, total = count_layout(parent, card)
    out = np.zeros(total, dtype=np.uint64)
    marg: List[np.ndarray] = []      # per node: rows in each of its states
    for v in range(len(card)):
        n_pa = np.asarray([float(fit_rows)]) if parent[v] < 0 else marg[parent[v]]
        t = np.asarray(cpts[v], dtype=np.float64).reshape(int(card[v]), n_pa.size)
        x = t * n_pa[None, :]
        r = np.rint(x)
        err = float(np.abs(x - r).max()) if x.size else 0.0
        if not err <= 1e-6 or (r < 0).any():
            raise ValueError(f"node {v}: T * n(parent state) is {err:.3g} from an integer with fit_rows = {fit_rows}")
        if not np.array_equal(r.sum(axis=0), n_pa):
            raise ValueError(f"node {v}: column sums of the recovered counts differ from the parent's state counts "
                             f"with fit_rows = {fit_rows}")
        out[off[v]: off[v] + r.size] = r.astype(np.uint64).reshape(-1)
        marg.append(r.sum(axis=1))
    for v, t in enumerate(counts_to_cpts(parent, card, out)):
        if not np.array_equal(t.reshape(-1), np.asarray(cpts[v], dtype=np.float64).reshape(-1)):
            raise ValueError(f"node {v}: the recovered counts do not reproduce the CPT bit for bit with fit_rows = {fit_rows}")
    return out


def infer_fit_rows(tm: TreeModel, max_tries: int = 100000) -> int:
    """The smallest row count the CPTs of ``tm`` can have been fitted on: a multiple of the lcm of the denominators of
    the root's probabilities (read as fractions with denominators up to ``nrows``) for which :func:`counts_from_cpts`
    succeeds.  It is ``nrows`` for a model fitted on the whole table and smaller for one fitted on a sample.  Raises
    ``ValueError`` when no multiple up to ``max_tries`` works."""
    root = np.asarray(tm.cpts[0], dtype=np.float64).reshape(-1)
    bound = max(int(tm.nrows), 1)
    step = 1
    for x in root:
        if x > 0:
            step = lcm(step, Fraction(float(x)).limit_denominator(bound).denominator)
    for k in range(1, max_tries + 1):
        try:
            counts_from_cpts(tm.parent, tm.card, tm.cpts, k * step)
            return k * step
        except ValueError:
            continue
    raise ValueError(f"no multiple of {step} up to {max_tries * step} rows reconstructs the counts of every node")


def fit_counts_device(parent: Sequence[int], card: Sequence[int], table_ptr: int, n_rows: int, elem_bytes: int,
                      row_stride_elems: int, counts_ptr: int, device: int = 0, stream: int = 0,
                      want_bad_rows: bool = False) -> Optional[int]:
    """One stream-ordered histogram pass on DEVICE buffers (raw addresses).  ``counts_ptr`` must have room for
    ``count_layout(...)[1] + 1`` 64-bit counters (the last one receives the number of skipped rows)."""
    parent = np.ascontiguousarray(parent, dtype=np.int32)
    card = np.ascontiguousarray(card, dtype=np.int32)
    _, total = count_layout(parent, card)
    bad = C.c_uint32(0)
    L.check(L.lib().bc_fit_counts(device, len(card), parent.ctypes.data, card.ctypes.data, table_ptr or None, elem_bytes,
                                  n_rows, row_stride_elems, counts_ptr, total, C.byref(bad) if want_bad_rows else None,
                                  stream or None))
    return int(bad.value) if want_bad_rows else None


def fit_cpts(parent: Sequence[int], card: Sequence[int], table: np.ndarray, device: int = 0):
    """Host table (``[n_rows, n_cols]`` uint8 / uint16 bin ids, columns in topological order) -> ``(cpts, counts,
    bad_rows)``.  torch moves the buffers; the counting is the CUDA kernel."""
    import torch

    table = np.ascontiguousarray(table)
    if table.dtype not in (np.uint8, np.uint16) or table.ndim != 2 or table.shape[1] != len(card):
        raise ValueError("table must be [n_rows, n_nodes] uint8 or uint16")
    _, total = count_layout(parent, card)
    dev = torch.device("cuda", device)
    with torch.cuda.device(dev):
        d_table = torch.from_numpy(table.view(np.uint8)).to(dev)
        d_counts = torch.empty(total + 1, dtype=torch.int64, device=dev)  # + the skipped-row counter
        bad = fit_counts_device(parent, card, d_table.data_ptr() if table.shape[0] else 0, table.shape[0], table.dtype.itemsize,
                                table.shape[1], d_counts.data_ptr(), device, torch.cuda.current_stream().cuda_stream, True)
        counts = d_counts[:total].cpu().numpy().astype(np.uint64)
    return counts_to_cpts(parent, card, counts), counts, bad


def refit(tm: TreeModel, table: np.ndarray, device: int = 0, nrows: Optional[int] = None) -> TreeModel:
    """A copy of ``tm`` whose CPTs are re-estimated from ``table`` (same tree, same discretisation)."""
    cpts, counts, bad = fit_cpts(tm.parent, tm.card, table, device)
    if bad:
        raise ValueError(f"{bad} rows hold a bin id outside the model's domains")
    out = copy.copy(tm)
    out.cpts = cpts
    out.nrows = int(table.shape[0]) if nrows is None else nrows
    out.counts = counts
    out.fit_rows = int(table.shape[0])
    return out
