"""``Bayescard_BN`` drop-in: same pickle, same ``query(...)`` / ``expectation(...)`` API, GPU underneath.

Mirrors the public surface of the reference class for the exact-jit path
(``Models/Bayescard_BN.py``): ``init_inference_method`` (``:122-178``), ``query_decoding`` (``:279-325``),
``query`` (``:496-556``), ``expectation`` (``:559-621``), ``align_cpds_in_topological`` (``:340-358``) and the
metadata attributes drivers read (``nrows``, ``attr_type``, ``domain``, ``encoding``, ``fanouts``, ...).
Only ``infer_algo='exact-jit'`` exists here; the other algorithms of the reference are out of scope.

New next to the scalar methods: ``query_batch`` / ``expectation_batch`` (one CUDA launch per batch), the GROUP BY
forms ``groupby_batch`` / ``expectation_groupby_batch`` (one pass per query for every group) and ``update_rows``
(inserted / deleted rows move the CPTs on the GPU without a refit).
"""
from __future__ import annotations

import copy
import itertools
from typing import Any, Dict, List, Optional, Sequence

import numpy as np

from . import _lib as L
from .infer import VariableEliminationB200
from .loader import TreeModel, load_model


class Bayescard_BN:
    def __init__(self, tree: TreeModel, device=0, infer_algo: Optional[str] = None, specialize: bool = True,
                 kernel: int = L.KERNEL_AUTO):
        self.tree = tree
        self.device = device
        self.specialize = specialize
        self.kernel = kernel
        # reference attributes (Models/BN_single_model.py:18-41, Models/Bayescard_BN.py:43-51)
        self.table_name = tree.table_name
        self.nrows = tree.nrows
        self.node_names = tree.node_names
        self.structure = tree.structure
        self.attr_type = tree.attr_type
        self.algorithm = tree.algorithm
        self.max_parents = tree.max_parents
        self.n_mcv = tree.n_mcv
        self.n_bins = tree.n_bins
        self.root = tree.root
        self.encoding = tree.encoding
        self.n_in_bin = tree.n_in_bin
        self.mapping = tree.mapping
        self.domain = tree.domain
        self.null_values = tree.null_values
        self.n_distinct_mapping = tree.n_distinct_mapping
        self.fanouts = tree.fanouts
        self.fanout_attr = tree.fanout_attr
        self.fanout_attr_inverse = tree.fanout_attr_inverse
        self.fanout_attr_positive = tree.fanout_attr_positive
        self.infer_algo = infer_algo
        self.infer_machine = None
        self.cpds = None

    # ------------------------------------------------------------------ construction
    @classmethod
    def load(cls, path: str, device=0, **kw) -> "Bayescard_BN":
        """Load a reference pickle (``pickle.dump(Bayescard_BN)``) or the flat ``.npz`` form."""
        return cls(load_model(path), device=device, **kw)

    @classmethod
    def build_from_table(cls, table, card, names=None, root=0, device=0, table_name="table", **kw) -> "Bayescard_BN":
        """Table-level counterpart of the reference's ``build_from_data`` (without its discretisation): learn the Chow-Liu
        tree of a table of bin ids (``[n_rows, n_cols]`` uint8 / uint16) and fit its CPTs on the GPU
        (:func:`.structure.learn_tree_model`).  The result is ready for ``init_inference_method()``."""
        from .structure import learn_tree_model

        return cls(learn_tree_model(table, card, names=names, root=root, device=device, table_name=table_name),
                   device=device, **kw)

    def __str__(self):
        return f"bn{self.table_name}.{self.algorithm}-{self.max_parents}-{self.root}-{self.n_mcv}-{self.n_bins}"

    # ------------------------------------------------------------------ init
    def align_cpds_in_topological(self):
        t = self.tree
        order = [t.node_names.index(n) for n in t.topo_names]
        return list(t.cpts), order, list(t.topo_names)

    def init_inference_method(self, algorithm: Optional[str] = None):
        if algorithm:
            self.infer_algo = algorithm
        if self.infer_algo is None:
            self.infer_algo = "exact-jit"
        if self.infer_algo != "exact-jit":
            raise NotImplementedError(
                f"infer_algo={self.infer_algo!r}: bayescard_b200 implements the exact-jit path only")
        assert self.algorithm == "chow-liu", "Currently JIT only supports CLT"
        self.cpds, self.topological_order, self.topological_order_node = self.align_cpds_in_topological()
        self.infer_machine = VariableEliminationB200(self.tree, device=self.device, specialize=self.specialize,
                                                     kernel=self.kernel)

    def _machine(self) -> VariableEliminationB200:
        assert self.infer_algo is not None and self.infer_machine is not None, \
            "must call .init_inference_method() first"
        return self.infer_machine

    # ------------------------------------------------------------------ decode
    def query_decoding(self, query, coverage=None, epsilon=0.5):
        return self._machine().compiler.decode(query, coverage, epsilon)

    # ------------------------------------------------------------------ scalar API
    def query(self, query, num_samples=1, n_distinct=None, coverage=None, return_prob=False, sample_size=1000,
              hard_sample=False):
        m = self._machine()
        nrows = self.nrows
        if n_distinct is None:
            query, n_distinct = m.compiler.decode(query, coverage)
        if query is None:
            return (0, nrows) if return_prob else 0
        p = m.query(query, n_distinct)
        return (p, nrows) if return_prob else p * nrows

    def expectation(self, query, fanout_attrs, num_samples=1, n_distinct=None, coverage=None, return_prob=False,
                    sample_size=1000, hard_sample=False):
        if fanout_attrs is None or len(fanout_attrs) == 0:
            return self.query(query, num_samples, n_distinct, coverage, return_prob, sample_size)
        m = self._machine()
        if n_distinct is None:
            query, n_distinct = m.compiler.decode(query, coverage)
        if query is None:
            # the reference does not test for an undecodable predicate here and fails inside
            # VariableEliminationJIT.expectation on None.keys() (Models/Bayescard_BN.py:581-583)
            raise AttributeError("'NoneType' object has no attribute 'keys'")
        e = m.expectation(query, fanout_attrs, n_distinct)
        return (e, self.nrows) if return_prob else e * self.nrows

    # ------------------------------------------------------------------ batch API
    def query_batch(self, queries: Sequence[dict], return_prob: bool = False) -> np.ndarray:
        """Raw predicate dicts -> cardinalities (or probabilities); undecodable queries give 0."""
        return self.expectation_batch(queries, None, return_prob)

    def expectation_batch(self, queries: Sequence[dict], fanout_attrs: Optional[Sequence[Sequence[str]]],
                          return_prob: bool = False) -> np.ndarray:
        m = self._machine()
        decoded, keep = [], []
        for i, q in enumerate(queries):
            b, w = m.compiler.decode(q)
            if b is not None:
                decoded.append((b, w))
                keep.append(i)
        out = np.zeros(len(queries), dtype=np.float64)
        if decoded:
            if fanout_attrs is None:
                res = m.query_batch([d[0] for d in decoded], [d[1] for d in decoded])
            else:
                fans = [list(fanout_attrs[i] or []) for i in keep]
                res = m.expectation_batch([d[0] for d in decoded], fans, [d[1] for d in decoded])
                for j, i in enumerate(keep):  # expectation with no fan-out column is query (:568-569)
                    if not fans[j] and not any(k in self.tree._index for k in decoded[j][0]):
                        res[j] = 0.0
            out[np.asarray(keep)] = res
        return out if return_prob else out * self.nrows

    def query_sql_batch(self, sqls: Sequence[str], return_prob: bool = False) -> np.ndarray:
        """SQL texts (``SELECT COUNT(*) FROM t WHERE ...``, the language of ``parse_query_single_table``) ->
        cardinalities.  Parsing, decoding and descriptor packing of the whole batch happen in one native call
        (``bayescard_b200.sqlc``); the results equal ``[self.query(parse_query_single_table(s, self)) for s in sqls]``."""
        m = self._machine()
        if getattr(self, "_sqlc", None) is None:
            from .sqlc import SqlBatchCompiler

            self._sqlc = SqlBatchCompiler(self.tree, m.compiler)
        bits_idx, bits_rows, dense_idx, dense_rows, _zero = self._sqlc.compile(sqls)
        out = np.zeros(len(sqls), dtype=np.float64)
        if len(bits_idx):
            out[bits_idx] = m.dev.run_host(bits_rows, L.DESC_BITS, None, m.kernel)
        if len(dense_idx):
            out[dense_idx] = m.dev.run_host(dense_rows, L.DESC_DENSE_F32, None, m.kernel)
        return out if return_prob else out * self.nrows

    # ------------------------------------------------------------------ GROUP BY one or two columns
    def groupby_batch(self, queries: Sequence[dict], column, return_prob: bool = False):
        """``SELECT column, COUNT(*) ... WHERE P GROUP BY column`` for a batch of predicate dicts ``P``: returns ``(keys,
        est)`` with ``est[i, j]`` the estimate of group ``keys[j]`` under query i -- one pass per query on the GPU
        (``bc_marginal_batch``) instead of one query per group value.

        * A categorical column with an encoding: the keys are its original values in encoding order and
          ``est(v) = nrows * M[bin(v)] * weight(v)``, which is ``self.query({**P_without_column, column: v})``.  M is the
          per-bin mass without the predicate on ``column``; values that predicate does not select get 0.
        * A continuous column, or one without an encoding: the keys are the bins (continuous: the bin's interval from
          ``mapping``); the predicate on ``column`` stays, with its coverage weights, and ``est(b) = nrows * M[b]``.

        ``column`` may also be a pair ``(a, b)`` of distinct columns, ``GROUP BY a, b`` (``bc_joint_marginal_batch``, one
        pass per query for all ``card(a) * card(b)`` groups): the keys are the row-major pairs ``(ka, kb)`` of each column's
        keys under the rules above, and for two categorical columns ``est(va, vb) = nrows * J[bin(va)][bin(vb)] * weight(va)
        * weight(vb)``, which is ``self.query({**P_without_a_b, a: va, b: vb})``; ``est`` is ``[n, Ka * Kb]``.

        Undecodable queries give a zero row; a query without predicates gives the column's marginal."""
        return self._groupby(queries, None, column, return_prob)

    def expectation_groupby_batch(self, queries: Sequence[dict], fanout_attrs: Sequence[Sequence[str]], column,
                                  return_prob: bool = False):
        """:meth:`groupby_batch` of an expectation: query i is weighted by its fan-out columns ``fanout_attrs[i]``, so that
        ``est[i, j]`` is ``self.expectation({**P_without_column, column: keys[j]}, fanout_attrs[i])`` for the values the
        predicate on ``column`` selects (0 for the others) -- the factor of a join estimate for every group at once, one
        pass per query (``bc_expectation_marginal_batch``, or ``bc_joint_marginal_batch`` for a pair of columns).  Keys and
        value selection are those of :meth:`groupby_batch`.  Undecodable queries give a zero row (where ``expectation``
        raises ``AttributeError``).  Grouping by a fan-out column raises ``ValueError``."""
        if len(fanout_attrs) != len(queries):
            raise ValueError("one list of fan-out columns per query")
        return self._groupby(queries, [list(f or []) for f in fanout_attrs], column, return_prob)

    def _group_keys(self, m, column):
        """``(node, categorical, keys, key_bin, key_wt)`` of one grouping column (``key_bin`` / ``key_wt``: categorical only)."""
        v = self.tree._index.get(column)
        if v is None:
            raise ValueError(f"column {column!r} is not a node of this model")
        col = m.compiler.cols[column]
        categorical = col.kind != "continuous" and col.enc is not None
        key_bin = key_wt = None
        if categorical:
            keys = list(col.pair)
            key_bin = np.asarray([col.pair[k][0] for k in keys], dtype=np.int64)
            key_wt = np.asarray([col.pair[k][1] for k in keys], dtype=np.float64)
        elif col.kind == "continuous" and col.edges is not None:
            keys = [tuple(col.edges[b]) for b in range(int(self.tree.card[v]))]
        else:
            keys = list(range(int(self.tree.card[v])))
        return v, categorical, keys, key_bin, key_wt

    def _groupby(self, queries, fanout_attrs, column, return_prob):
        cols = (column,) if isinstance(column, str) else tuple(column)
        if len(cols) not in (1, 2) or len(set(cols)) != len(cols):
            raise ValueError(f"GROUP BY takes one column or a pair of distinct columns, got {column!r}")
        if fanout_attrs is not None or len(cols) == 2:
            for c in cols:
                v = self.tree._index.get(c)
                if c in self.fanout_attr or (v is not None and self.tree.fan_vector(v) is not None):
                    raise ValueError(f"column {c!r} is a fan-out column; GROUP BY needs a column of the table")
        m = self._machine()
        info = [self._group_keys(m, c) for c in cols]
        keys = info[0][2] if len(cols) == 1 else list(itertools.product(info[0][2], info[1][2]))
        est = np.zeros((len(queries), len(keys)), dtype=np.float64)
        decoded, keep, sel = [], [], []
        for i, q in enumerate(queries):
            s_q = []
            for c, (_, categorical, ck, _, _) in zip(cols, info):
                if categorical:
                    s = np.ones(len(ck), dtype=bool)
                    if c in q:
                        s = m.compiler.select_values(c, q[c])
                        if s is None:
                            break
                    q = {k: x for k, x in q.items() if k != c}
                s_q.append(s if categorical else None)
            else:
                b, w = m.compiler.decode(q)
                if b is not None:
                    decoded.append((b, w))
                    keep.append(i)
                    sel.append(s_q)
        if decoded:
            fans = None if fanout_attrs is None else [fanout_attrs[i] for i in keep]
            if len(cols) == 1:
                M = m.marginal_batch(decoded, cols[0], fanouts=fans)
            else:
                M = m.joint_batch(decoded, cols, fanouts=fans)
            for k, (_, categorical, _, key_bin, key_wt) in enumerate(info):
                if categorical:
                    shape = [1] * M.ndim
                    shape[1 + k] = -1
                    S = np.asarray([s[k] for s in sel]).reshape([len(sel)] + shape[1:])
                    M = np.take(M, key_bin, axis=1 + k) * key_wt.reshape(shape) * S
            est[keep] = M.reshape(len(keep), -1)
        return keys, (est if return_prob else est * self.nrows)

    def groupby(self, query: dict, column, return_prob: bool = False) -> Dict[Any, float]:
        """One query of :meth:`groupby_batch` (one column or a pair): ``{key: estimate}``."""
        keys, est = self.groupby_batch([query], column, return_prob)
        return {k: float(e) for k, e in zip(keys, est[0])}

    def groupby_sql_batch(self, sqls: Sequence[str], return_prob: bool = False) -> List[Dict[Any, float]]:
        """``SELECT a, COUNT(*) FROM t [WHERE ...] GROUP BY a`` and ``SELECT a, b, COUNT(*) ... GROUP BY a, b`` texts -> one
        ``{key: estimate}`` per text (two columns: keys ``(ka, kb)``); the texts that group by the same columns are answered
        in one batch."""
        from .sql_front import parse_groupby_single_table

        parsed = [parse_groupby_single_table(s, self) for s in sqls]
        out: List[Dict[Any, float]] = [{} for _ in sqls]
        for column in dict.fromkeys(c for _, c in parsed):
            idx = [i for i, (_, c) in enumerate(parsed) if c == column]
            keys, est = self.groupby_batch([parsed[i][0] for i in idx], column, return_prob)
            for j, i in enumerate(idx):
                out[i] = {k: float(e) for k, e in zip(keys, est[j])}
        return out

    # ------------------------------------------------------------------ table changes
    def update_rows(self, inserted=None, deleted=None, fit_rows: Optional[int] = None) -> List[str]:
        """Follow rows inserted into / deleted from the table without a refit: the CPTs become those of ``fit.refit`` on
        the rows the model was fitted on plus ``inserted`` minus ``deleted`` (same tree), on the GPU, and ``nrows`` moves by
        the difference.  Returns the names of the columns whose CPTs changed.

        Rows are bin ids (``[n, len(node_names)]``, uint8 / uint16) with columns in ``node_names`` order -- for
        ``build_from_table`` the table's own column order; columns in ``dropped_names`` are ignored.  Only the CPTs move:
        the tree, the discretisation (``encoding``, ``n_in_bin``, ``mapping``, ``domain``) and the fan-out vectors stay as
        they are.  A model fitted on a sample (``fit_rows < nrows``) counts inserted rows with weight 1 against the
        sample's counts.  A batch holding an out-of-domain bin id, or deleting more rows of some (column, parent) bin pair
        than were counted, raises and changes nothing; deleting rows that were never in the data cannot be detected
        otherwise.

        The first call attaches the counts behind the CPTs: the tree model's own when it has them, otherwise
        ``fit.counts_from_cpts`` with ``fit_rows`` (default: ``tree.fit_rows``, else ``fit.infer_fit_rows``)."""
        from .fit import count_layout, counts_from_cpts, infer_fit_rows, node_cpt

        m = self._machine()
        t = self.tree
        if not getattr(self, "_counts_attached", False):
            if t.counts is None:
                rows = fit_rows if fit_rows is not None else (t.fit_rows if t.fit_rows is not None else infer_fit_rows(t))
                t.counts = counts_from_cpts(t.parent, t.card, t.cpts, rows)
                t.fit_rows = int(rows)
            elif t.fit_rows is None:
                t.fit_rows = int(np.asarray(t.counts[: int(t.card[0])], dtype=np.uint64).sum())
            t.counts = np.array(t.counts, dtype=np.uint64)   # (a private, writable copy: refreshed below)
            m.dev.attach_counts(t.counts)
            self._counts_attached = True
        tabs = [None if rows is None else rows_to_topological(t, rows) for rows in (inserted, deleted)]
        touched = m.dev.update(tabs[0], tabs[1])
        off, total = count_layout(t.parent, t.card)
        off = np.append(off, total)
        for v in touched:   # the host mirror of the touched nodes: counts and fp64 CPTs
            c = m.dev.get_counts(int(v), 1)
            t.counts[off[v]: off[v + 1]] = c
            t.cpts[v] = node_cpt(t.parent, t.card, int(v), c)
        delta = (0 if tabs[0] is None else tabs[0].shape[0]) - (0 if tabs[1] is None else tabs[1].shape[0])
        t.fit_rows += delta
        t.nrows = t.nrows + delta
        self.nrows = t.nrows
        if self.cpds is not None:
            self.cpds = list(t.cpts)
        return [t.infer_names[int(v)] for v in touched]

    def close(self):
        if getattr(self, "_sqlc", None) is not None:
            self._sqlc.close()
            self._sqlc = None
        if self.infer_machine is not None:
            self.infer_machine.close()
            self.infer_machine = None


def rows_to_topological(tm: TreeModel, rows) -> np.ndarray:
    """Rows of bin ids with columns in ``node_names`` order -> the same rows with columns in topological order (the
    convention of ``bc_fit_counts`` / ``bc_model_update``); columns outside the root component (``dropped_names``) are
    dropped.  uint8 / uint16 rows keep their type unless a domain needs uint16; other integer types are range-checked and
    narrowed."""
    rows = np.asarray(rows)
    if rows.ndim != 2 or rows.shape[1] != len(tm.node_names):
        raise ValueError(f"rows must be [n, {len(tm.node_names)}] bin ids in node_names order")
    wide = int(np.max(tm.card)) > 256
    if rows.dtype not in (np.uint8, np.uint16):
        if rows.size and (rows.min() < 0 or rows.max() > 65535):
            raise ValueError("bin ids must lie in [0, 65535]")
        rows = rows.astype(np.uint16 if wide or (rows.size and rows.max() > 255) else np.uint8)
    elif wide:
        rows = rows.astype(np.uint16)
    cols = [tm.node_names.index(name) for name in tm.infer_names]
    return np.ascontiguousarray(rows[:, cols])


def load_BN_single(path: str, device=0, **kw) -> Bayescard_BN:
    """Name-compatible with reference ``Models/BN_single_model.py:219-223``."""
    return Bayescard_BN.load(path, device=device, **kw)
