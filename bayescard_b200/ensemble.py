"""``BN_ensemble``: the IMDB join-cardinality glue around per-table-join BNs.

Follows reference ``Models/BN_ensemble_model.py``: ``parse_query_all`` (``:192-225``) resolves
``bn_index``, drops a factor that repeats its neighbour and pre-decodes the predicates;
``cardinality`` (``:228-252``) multiplies ``join_size`` by ``p`` (or ``1/p`` for ``inverse`` factors),
returns 1 as soon as a factor is 0 and clamps the result to >= 1.

``cardinality_batch`` is new: it gathers the factors of MANY join queries per BN, evaluates each
BN's factors in one CUDA batch, and combines on the host with the same rules.  ``groupby_batch`` does the
same for GROUP BY plans (``joblight.plan_star_groupby``): every group of a query in one pass per factor.
"""
from __future__ import annotations

from typing import Dict, List, Sequence

import numpy as np

from .model import Bayescard_BN


class BN_ensemble:
    def __init__(self, schema_graph=None, bns: Dict[int, Bayescard_BN] = None):
        self.schema_graph = schema_graph
        self.bns = dict() if bns is None else bns
        self.join_size = dict()

    def add_BN(self, bn: Bayescard_BN):
        self.bns[bn.table_name] = bn

    # ------------------------------------------------------------------ parse_query_all
    def parse_query_all(self, table_queries: Sequence[list]) -> List[list]:
        parsed_all = []
        for tq in table_queries:
            factors = tq[1:]
            for f in factors:
                if type(f["bn_index"]) != int:
                    for j, bn in self.bns.items():
                        if set(bn.table_name) == f["bn_index"]:
                            f["bn_index"] = j
                            break
                assert type(f["bn_index"]) == int, f["bn_index"]

            def same(a, b):
                return (a["bn_index"] == b["bn_index"] and a["query"] == b["query"]
                        and a["expectation"] == b["expectation"])

            parsed = [tq[0]]
            for i, f in enumerate(factors):
                if i + 1 < len(factors) and same(f, factors[i + 1]):
                    continue
                if i > 0 and same(f, factors[i - 1]):
                    continue
                bins, wts = self.bns[f["bn_index"]].query_decoding(f["query"])
                parsed.append({"bn_index": f["bn_index"], "inverse": f["inverse"], "expectation": f["expectation"],
                               "query": bins, "n_distinct": wts})
            parsed_all.append(parsed)
        return parsed_all

    # ------------------------------------------------------------------ cardinality
    _UNDECODABLE = object()  # factor the reference would crash on IF its loop reaches it

    @staticmethod
    def _combine(join_size, factors, probs):
        card = join_size
        for f, p in zip(factors, probs):
            if p is BN_ensemble._UNDECODABLE:
                # Bayescard_BN.expectation has no `query is None` guard (Models/Bayescard_BN.py:581-583);
                # the reference only fails if no earlier factor already returned 1 (:244-245)
                raise AttributeError("'NoneType' object has no attribute 'keys'")
            if p == 0:
                return 1
            card = card * (1 / p) if f["inverse"] else card * p
        return 1 if card <= 1 else card

    def cardinality(self, table_query, sample_size=1000, hard_sample=False):
        probs = []
        for f in table_query[1:]:
            bn = self.bns[f["bn_index"]]
            if len(f["expectation"]) == 0:
                p, _ = bn.query(f["query"], n_distinct=f["n_distinct"], return_prob=True)
            else:
                p, _ = bn.expectation(f["query"], f["expectation"], n_distinct=f["n_distinct"], return_prob=True)
            p = float(np.asarray(p).reshape(-1)[0]) if not isinstance(p, int) else p
            probs.append(p)
            if p == 0:
                return 1
        return self._combine(table_query[0], table_query[1:], probs)

    def cardinality_batch(self, table_queries: Sequence[list]) -> np.ndarray:
        """Cardinalities of many parsed join queries with one device batch per BN."""
        per_bn: Dict[int, list] = {}
        for qi, tq in enumerate(table_queries):
            for fi, f in enumerate(tq[1:]):
                per_bn.setdefault(f["bn_index"], []).append((qi, fi, f))
        probs = [[None] * (len(tq) - 1) for tq in table_queries]
        self._factor_probs(per_bn, probs)
        return np.asarray([self._combine(tq[0], tq[1:], probs[qi]) for qi, tq in enumerate(table_queries)],
                          dtype=np.float64)

    def _factor_probs(self, per_bn: Dict[int, list], probs) -> None:
        """``probs[qi][fi]`` of parsed factors ``(qi, fi, f)`` grouped by BN: one ``expectation_batch`` per BN; an undecodable
        factor is 0 (a query) or ``_UNDECODABLE`` (an expectation)."""
        for j, items in per_bn.items():
            m = self.bns[j]._machine()
            ok = [(qi, fi, f) for qi, fi, f in items if f["query"] is not None]
            for qi, fi, f in items:
                if f["query"] is None:
                    probs[qi][fi] = 0 if len(f["expectation"]) == 0 else self._UNDECODABLE
            if ok:
                res = m.expectation_batch([f["query"] for _, _, f in ok], [list(f["expectation"]) for _, _, f in ok],
                                          [f["n_distinct"] for _, _, f in ok])
                for (qi, fi, _), p in zip(ok, res):
                    probs[qi][fi] = float(p)

    # ------------------------------------------------------------------ GROUP BY over a join
    @staticmethod
    def _dedupe(factors: Sequence[dict]) -> List[dict]:
        """``parse_query_all``'s rule without the decoding: drop a factor equal to a neighbour."""
        def same(a, b):
            return a["bn_index"] == b["bn_index"] and a["query"] == b["query"] and a["expectation"] == b["expectation"]

        return [f for i, f in enumerate(factors)
                if not (i + 1 < len(factors) and same(f, factors[i + 1])) and not (i > 0 and same(f, factors[i - 1]))]

    def groupby_batch(self, planned: Sequence[dict], column: str):
        """``SELECT column, COUNT(*) FROM <star join> WHERE ... GROUP BY column`` for many planned queries
        (``joblight.plan_star_groupby``, all grouping by ``column``): returns ``(keys, est)``, ``est[i, j]`` the estimate of
        group ``keys[j]`` under query i.

        A factor whose query holds ``column`` gives a vector over the keys (``Bayescard_BN.expectation_groupby_batch``: every
        group in one pass; a factor without fan-out columns is a plain query); the other factors give one number each
        (``cardinality_batch``'s machinery).  Each BN serves its factors of the whole batch in one device batch per kind.
        The keys are the union of the column's original values over the BNs of those factors.  Per group v:

        * 0 where the WHERE clause does not select v, or where a factor is 0 -- among them a v missing from a factor's BN
          (the per-value estimate ``cardinality`` instead returns 1 as soon as a factor is 0);
        * otherwise ``join_size * prod p^(+-1)``, at least 1, as in ``cardinality``;
        * 0 where the per-value ``cardinality`` would raise the reference's ``AttributeError`` for an undecodable
          expectation factor (a deliberate deviation: one undecodable group does not fail the whole GROUP BY).

        Only categorical columns with an encoding can be grouped by (``ValueError`` otherwise)."""
        plans = []
        for p in planned:
            if p["column"] != column:
                raise ValueError(f"planned query groups by {p['column']!r}, not {column!r}")
            plans.append((p["plan"][0], self._dedupe(p["plan"][1:]), p["where"]))
        holders = sorted({f["bn_index"] for _, fs, _ in plans for f in fs if column in f["query"]})
        key_pos: Dict = {}
        for j in holders:
            col = self.bns[j]._machine().compiler.cols[column]
            if col.kind == "continuous" or col.enc is None:
                raise ValueError(f"GROUP BY {column!r}: only categorical columns with an encoding are supported")
            for k in col.pair:
                key_pos.setdefault(k, len(key_pos))
        keys = list(key_pos)
        nk = len(keys)
        # factors: per-key vectors (grouping factors) and scalars, each gathered per BN
        vec_items: Dict[int, list] = {}
        per_bn: Dict[int, list] = {}
        probs = []
        for qi, (_, fs, where) in enumerate(plans):
            probs.append([None] * len(fs))
            for fi, f in enumerate(fs):
                j = f["bn_index"]
                if column in f["query"]:
                    q = {k: x for k, x in f["query"].items() if k != column}
                    if where is not None:
                        q[column] = where   # selects the groups (Bayescard_BN.groupby_batch's value selection)
                    vec_items.setdefault(j, []).append((qi, fi, q, list(f["expectation"])))
                else:
                    bins, wts = self.bns[j].query_decoding(f["query"])
                    per_bn.setdefault(j, []).append((qi, fi, {"bn_index": j, "inverse": f["inverse"],
                                                              "expectation": f["expectation"], "query": bins, "n_distinct": wts}))
        self._factor_probs(per_bn, probs)
        for j, items in vec_items.items():
            bkeys, est = self.bns[j].expectation_groupby_batch([q for _, _, q, _ in items], [e for _, _, _, e in items], column,
                                                              return_prob=True)
            pos = np.asarray([key_pos[k] for k in bkeys], dtype=np.int64)
            for (qi, fi, _, _), row in zip(items, est):
                vec = np.zeros(nk, dtype=np.float64)   # a key missing from this BN: factor 0
                vec[pos] = row
                probs[qi][fi] = vec
        est = np.zeros((len(plans), nk), dtype=np.float64)
        for qi, (join_size, fs, _) in enumerate(plans):
            card = np.full(nk, float(join_size))
            zero = np.zeros(nk, dtype=bool)
            for f, p in zip(fs, probs[qi]):
                if p is self._UNDECODABLE:
                    zero[:] = True
                    continue
                p = np.broadcast_to(np.asarray(p, dtype=np.float64), (nk,))
                zero |= p == 0
                with np.errstate(divide="ignore", invalid="ignore"):
                    card = card * (1 / p) if f["inverse"] else card * p
            est[qi] = np.where(zero, 0.0, np.where(card <= 1, 1.0, card))
        return keys, est
