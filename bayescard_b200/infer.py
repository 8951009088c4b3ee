"""``VariableEliminationB200``: the ``infer_machine`` plug-in that runs on the GPU.

It fills the slot the reference fills with ``VariableEliminationJIT`` (reference
``Models/Bayescard_BN.py:141``): any object with ``.query(query, n_distinct)`` and
``.expectation(query, fanout_attrs, n_distinct)`` (``Pgmpy/inference/ExactInference.py:112,199``).
The scalar methods keep the reference's return conventions -- numpy fp64 scalar, a shape-(1,) array
when the root is the only node involved (``:140-142``), int ``0`` when no queried column is reachable
(``:197``), ``AssertionError`` for a lone fan-out root (``:225``) -- and run a batch of one through the
same CUDA path as the batch methods.  There is no CPU path.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence

import numpy as np

from . import _lib as L
from .decode import dense_to_wsparse, PredicateCompiler
from .engine import DeviceModel, ShardedModel
from .loader import TreeModel


class VariableEliminationB200:
    def __init__(self, tm: TreeModel, device=0, specialize: bool = True, kernel: int = L.KERNEL_AUTO):
        self.tm = tm
        self.compiler = PredicateCompiler(tm)
        if isinstance(device, (list, tuple)):
            self.dev = ShardedModel(tm, list(device), specialize=specialize)
            self._single = self.dev.replicas[0]
        else:
            self.dev = DeviceModel(tm, int(device), specialize=specialize)
            self._single = self.dev
        self.kernel = kernel
        self.specialize = specialize
        self.root = tm.infer_names[0]
        self.fanouts = tm.fanouts

    # ------------------------------------------------------------------ batch
    def run_decoded(self, decoded, fanouts: Optional[Sequence[Sequence[str]]] = None) -> np.ndarray:
        """fp32 device results (as fp64) for already decoded queries; no return-shape quirks."""
        nq = len(decoded)
        out = np.zeros(nq, dtype=np.float64)
        if nq == 0:
            return out
        b_idx, b_desc, d_idx, d_desc, mask = self.compiler.pack(decoded, fanouts)
        if len(b_idx):
            out[b_idx] = self.dev.run_host(b_desc, L.DESC_BITS, None if mask is None else mask[b_idx], self.kernel)
        if len(d_idx):
            # fractional weights cross PCIe as weighted runs (WSPARSE, ~20x smaller) and become DENSE rows on the device
            dmask = None if mask is None else mask[d_idx]
            row_off, words = dense_to_wsparse(self.tm, d_desc)   # (one device or several: ShardedModel slices the CSR)
            out[d_idx] = self.dev.run_wsparse_host(row_off, words, dmask, self.kernel)
        return out

    def query_batch(self, queries: Sequence[Dict[str, Sequence[int]]],
                    n_distincts: Sequence[Dict[str, np.ndarray]]) -> np.ndarray:
        decoded = [(q, self._unit(q) if nd is None else nd) for q, nd in zip(queries, n_distincts)]
        out = self.run_decoded(decoded)
        for i, q in enumerate(queries):  # no reachable column -> 0 (ExactInference.py:197)
            if not any(k in self.tm._index for k in q):
                out[i] = 0.0
        return out

    def expectation_batch(self, queries, fanout_attrs, n_distincts) -> np.ndarray:
        decoded = [(q, self._unit(q) if nd is None else nd) for q, nd in zip(queries, n_distincts)]
        out = self.run_decoded(decoded, fanout_attrs)
        for i, (q, f) in enumerate(zip(queries, fanout_attrs)):
            if not any(k in self.tm._index for k in list(q) + list(f)):
                out[i] = 0.0
        return out

    def marginal_batch(self, decoded, name: str, kernel: Optional[int] = None,
                       fanouts: Optional[Sequence[Sequence[str]]] = None) -> np.ndarray:
        """GROUP BY ``name``: ``[len(decoded), card]`` fp64, row i = the per-state mass of column ``name`` under the
        already decoded query i, weighted by the fan-out columns ``fanouts[i]`` when given (``bc_expectation_marginal_batch``;
        its row sums are what ``run_decoded(decoded, fanouts)`` returns).  The first call for a column attaches its
        specialised marginal kernel; a sharded machine answers on its first replica."""
        v = self.tm._index[name]
        kernel = self.kernel if kernel is None else kernel
        dm = self._single
        if self.specialize and kernel in (L.KERNEL_AUTO, L.KERNEL_SPEC) and dm.device >= 0:
            dm.specialize_marginal(v)
        out = np.zeros((len(decoded), int(self.tm.card[v])), dtype=np.float64)
        if len(decoded) == 0:
            return out
        b_idx, b_desc, d_idx, d_desc, mask = self.compiler.pack(decoded, fanouts)
        if len(b_idx):
            out[b_idx] = dm.run_marginal_host(b_desc, L.DESC_BITS, v, kernel, None if mask is None else mask[b_idx])
        if len(d_idx):
            out[d_idx] = dm.run_marginal_host(d_desc, L.DESC_DENSE_F32, v, kernel, None if mask is None else mask[d_idx])
        return out

    def joint_batch(self, decoded, names, kernel: Optional[int] = None,
                    fanouts: Optional[Sequence[Sequence[str]]] = None) -> np.ndarray:
        """GROUP BY two columns ``names = (name_a, name_b)``: ``[len(decoded), card_a, card_b]`` fp64, the mass of every pair
        of states under the already decoded query i, weighted by the fan-out columns ``fanouts[i]`` when given
        (``bc_joint_marginal_batch``).  The first call for a pair attaches its joint module; a sharded machine answers on
        its first replica."""
        a, b = (self.tm._index[n] for n in names)
        kernel = self.kernel if kernel is None else kernel
        dm = self._single
        if self.specialize and kernel in (L.KERNEL_AUTO, L.KERNEL_SPEC) and dm.device >= 0:
            dm.specialize_joint(a, b)
        out = np.zeros((len(decoded), int(self.tm.card[a]), int(self.tm.card[b])), dtype=np.float64)
        if len(decoded) == 0:
            return out
        b_idx, b_desc, d_idx, d_desc, mask = self.compiler.pack(decoded, fanouts)
        if len(b_idx):
            out[b_idx] = dm.run_joint_host(b_desc, L.DESC_BITS, a, b, kernel, None if mask is None else mask[b_idx])
        if len(d_idx):
            out[d_idx] = dm.run_joint_host(d_desc, L.DESC_DENSE_F32, a, b, kernel, None if mask is None else mask[d_idx])
        return out

    @staticmethod
    def _unit(q):
        """``n_distinct`` falsy: the reference sums the selected rows (ExactInference.py:138-139)."""
        return {k: np.ones(len(v) if isinstance(v, (list, tuple, np.ndarray)) else 1) for k, v in q.items()}

    # ------------------------------------------------------------------ scalar drop-in
    def _touched(self, names) -> List[int]:
        return [self.tm._index[k] for k in names if k in self.tm._index]

    def query(self, query, n_distinct=None):
        touched = self._touched(query.keys())
        if not touched:
            return 0
        nd = n_distinct if n_distinct else self._unit(query)
        val = np.float64(self.run_decoded([(query, nd)])[0])
        if all(v == 0 for v in touched):
            return np.asarray([val])
        return val

    def expectation(self, query, fanout_attrs, n_distinct=None):
        touched = self._touched(list(query.keys()) + list(fanout_attrs))
        if not touched:
            return 0
        if all(v == 0 for v in touched) and self.root not in query:
            raise AssertionError("no querying variables")
        nd = n_distinct if n_distinct else self._unit(query)
        val = np.float64(self.run_decoded([(query, nd)], [list(fanout_attrs)])[0])
        if all(v == 0 for v in touched):
            return np.asarray([val])
        return val

    def close(self):
        self.dev.close()
