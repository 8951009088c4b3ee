"""job-light star-join planner for the shipped IMDB ensemble (SURVEY.md section 8f item 2).

The reference plans join queries with DeepDB's ensemble machinery (``Evaluation/parse_query_imdb.py:54-325`` over
``DeepDBUtils/ensemble_compilation``), which cannot run here (``ensemble_loader.pkl`` is missing, spflow / sqlparse are
not installed).  This module restates what that machinery produces for the ONLY shape job-light has -- a star on
``title.id`` over the five two-table models ``title x X`` (``Schemas/imdb/schema.py:59-63``; BN index = relationship
order) -- and emits factor lists in the reference's own format, ``[full_join_size, {"bn_index", "inverse", "query",
"expectation"}, ...]`` (``parse_query_imdb.py:301-323``), so that ``BN_ensemble.parse_query_all`` / ``.cardinality``
consume them unchanged.

For a query over ``title`` and the tables ``a, b, ...`` with conditions ``C_t, C_a, C_b, ...`` ``generate_factors``
(``:54-240``) yields, with two-table models:

    card = |J_a| * E_a[ 1{C_t, C_a, a not null} * prod_{b != a} F_b ]                    (first model, ``:81-88``; the
                                                                                          outgoing fan-outs F_b =
                                                                                          title.mul_b.movie_id are
                                                                                          merged into it, ``:124-130``)
           * prod_{b != a}  P_b(C_b, C_t, b not null) / P_b(C_t, b not null)             (``:187-223``: overlap = title)

``relevant_conditions`` adds the NOT NULL condition of every merged table (``spn_ensemble.py:96-101``);
``factor_refine`` (``:243-254``) drops a nominator / denominator pair that cancels (no condition on b).  Strict
comparisons get ``epsilon = 0.1`` (``prepare_single_query``, ``:19-44``).

NOT PINNED against the reference (it cannot run); validated against the 70 true cardinalities shipped in
``Benchmark/IMDB/job-light.sql`` and the paper's q-error row (Table 9: 1.30 / 3.534 / 4.836 / 19.13 at 50 / 90 / 95 / 100 %;
this planner over the shipped models gives 1.301 / 3.535 / 4.837 / 19.14).
The first model is chosen as ``_greedily_select_first_cardinality_spn`` does with ``rdc_spn_selection=True``
(``DeepDBUtils/ensemble_compilation/spn_ensemble.py:1312-1350``): the candidate vector (sum of the pairwise RDC values of
the conditioned columns the model covers, number of covered tables with conditions, ...) is maximised, the models are
visited in BN-index order and a later one must be strictly better.  The RDC values are the twelve title-x-X entries of the
shipped ``Benchmark/IMDB/pairwise_rdc.pkl`` (data, copied below).
"""
from __future__ import annotations

import math
import re
from typing import Dict, List, Sequence, Tuple

ALIASES = {"t": "title", "mc": "movie_companies", "mi": "movie_info", "mi_idx": "movie_info_idx", "mk": "movie_keyword",
           "ci": "cast_info"}
# BN index = order of the relationships in Schemas/imdb/schema.py:59-63 (== the shipped {i}_chow-liu_1.pkl files)
BN_INDEX = {"movie_info_idx": 0, "movie_info": 1, "cast_info": 2, "movie_keyword": 3, "movie_companies": 4}
EPSILON = 0.1

# Benchmark/IMDB/pairwise_rdc.pkl, the pairs inside one two-table model (no entry exists for two columns of one table)
PAIRWISE_RDC = {
    ("movie_info_idx.info_type_id", "title.kind_id"): 0.39070659303540217,
    ("movie_info_idx.info_type_id", "title.production_year"): 0.14469894415051307,
    ("movie_info.info_type_id", "title.kind_id"): 0.5492260005642482,
    ("movie_info.info_type_id", "title.production_year"): 0.2902598439357767,
    ("cast_info.role_id", "title.kind_id"): 0.1293990618864897,
    ("cast_info.role_id", "title.production_year"): 0.16279968513002951,
    ("movie_keyword.keyword_id", "title.kind_id"): 0.5536931277256608,
    ("movie_keyword.keyword_id", "title.production_year"): 0.19072312253292326,
    ("movie_companies.company_id", "title.kind_id"): 0.6260741802831398,
    ("movie_companies.company_type_id", "title.kind_id"): 0.553063881600441,
    ("movie_companies.company_id", "title.production_year"): 0.34941105786412013,
    ("movie_companies.company_type_id", "title.production_year"): 0.257376245147359,
}

_COND = re.compile(r"^\s*(\w+)\.(\w+)\s*(<=|>=|=|<|>)\s*(-?\d+(?:\.\d+)?)\s*$")
_JOIN = re.compile(r"^\s*(\w+)\.(\w+)\s*=\s*(\w+)\.(\w+)\s*$")


def parse_job_light(sql: str) -> Tuple[List[str], Dict[str, List[Tuple[str, str, float]]]]:
    """``SELECT COUNT(*) FROM a x, b y WHERE ...`` -> (joined tables in FROM order without title, {table: [(column, op, value)]})."""
    sql = sql.strip().rstrip(";")
    m = re.match(r"(?is)^select\s+count\(\*\)\s+from\s+(.*?)\s+where\s+(.*)$", sql)
    if not m:
        raise ValueError("not a job-light query: " + sql[:80])
    alias_of = {}
    order = []
    for part in m.group(1).split(","):
        toks = part.split()
        table, alias = toks[0], toks[-1]
        alias_of[alias] = table
        if table != "title":
            if table not in BN_INDEX:
                raise ValueError("table outside the job-light star: " + table)
            order.append(table)
    if "title" not in alias_of.values():
        raise ValueError("job-light queries join through title")
    conds: Dict[str, List[Tuple[str, str, float]]] = {}
    for c in re.split(r"(?i)\s+and\s+", m.group(2)):
        if _JOIN.match(c):
            continue
        mc = _COND.match(c)
        if not mc:
            raise ValueError("unsupported condition: " + c)
        alias, col, op, val = mc.groups()
        conds.setdefault(alias_of[alias], []).append((col, op, float(val)))
    return order, conds


def _table_query(table: str, conds: Sequence[Tuple[str, str, float]]) -> dict:
    """Conditions of one table -> the ``{column: scalar | (lo, hi)}`` dict of ``prepare_single_query``."""
    per_col: Dict[str, List[Tuple[str, float]]] = {}
    for col, op, val in conds:
        per_col.setdefault(col, []).append((op, val))
    q = {}
    for col, ops in per_col.items():
        lo, hi, eq = -math.inf, math.inf, None
        for op, val in ops:
            if op == "=":
                eq = val
            elif op == ">":
                lo = max(lo, val + EPSILON)
            elif op == ">=":
                lo = max(lo, val)
            elif op == "<":
                hi = min(hi, val - EPSILON)
            elif op == "<=":
                hi = min(hi, val)
        q[f"{table}.{col}"] = eq if eq is not None else (lo, hi)
    return q


def _first_table(order: Sequence[str], conds: Dict[str, list]) -> str:
    """``_greedily_select_first_cardinality_spn`` over the five two-table models (start table title or X: same vector)."""
    best, best_vec = None, None
    for table in sorted(order, key=lambda t: BN_INDEX[t]):   # self.spns order
        cols = {f"{t}.{c}" for t in ("title", table) for c, _, _ in conds.get(t, [])}
        rdc = 0.0
        for x in cols:
            for y in cols:
                if x < y:
                    rdc += PAIRWISE_RDC.get((x, y), PAIRWISE_RDC.get((y, x), 0.0))
        n_where = sum(1 for t in ("title", table) if conds.get(t))
        vec = (rdc, n_where, 2, 0)
        if best_vec is None or vec > best_vec:
            best, best_vec = table, vec
    return best


def plan_star_query(sql: str, join_sizes: Dict[int, float]) -> list:
    """One job-light SQL text -> ``[full_join_size, factor, ...]`` in the reference's format."""
    order, conds = parse_job_light(sql)
    return _plan(order, conds, join_sizes)


def _plan(order: Sequence[str], conds: Dict[str, list], join_sizes: Dict[int, float]) -> list:
    if not order:
        raise ValueError("no joined table")
    c_t = _table_query("title", conds.get("title", []))
    first = _first_table(order, conds)
    a = BN_INDEX[first]

    def nn(table):   # the NOT NULL condition of relevant_conditions: the null marker of <table>_nn is 0
        return {f"{table}.{table}_nn": 1}

    q_first = dict(c_t)
    q_first.update(_table_query(first, conds.get(first, [])))
    q_first.update(nn(first))
    others = [t for t in order if t != first]
    factors = [{"bn_index": a, "inverse": False, "query": q_first,
                "expectation": [f"title.mul_{b}.movie_id" for b in others]}]
    for b in others:
        c_b = _table_query(b, conds.get(b, []))
        if not c_b:
            continue   # factor_refine: nominator and denominator cancel
        nom = dict(c_t)
        nom.update(c_b)
        nom.update(nn(b))
        den = dict(c_t)
        den.update(nn(b))
        factors.append({"bn_index": BN_INDEX[b], "inverse": False, "query": nom, "expectation": []})
        factors.append({"bn_index": BN_INDEX[b], "inverse": True, "query": den, "expectation": []})
    return [join_sizes[a]] + factors


def plan_workload(sqls: Sequence[str], join_sizes: Dict[int, float]) -> List[list]:
    return [plan_star_query(s, join_sizes) for s in sqls]


# ------------------------------------------------------------------------------------ GROUP BY over the star
class _GroupValue:
    """The placeholder of the grouping column's value in a planned GROUP BY (kept as one object through deep copies)."""

    def __repr__(self):
        return "GROUP_VALUE"

    def __copy__(self):
        return self

    def __deepcopy__(self, memo):
        return self


GROUP_VALUE = _GroupValue()


def parse_job_light_groupby(sql: str) -> Tuple[List[str], Dict[str, List[Tuple[str, str, float]]], str, str]:
    """``SELECT x.col, COUNT(*) FROM ... WHERE ... GROUP BY x.col`` (job-light's grammar otherwise) -> (joined tables, conditions
    as :func:`parse_job_light` returns them, grouping table, grouping column)."""
    sql = sql.strip().rstrip(";").strip()
    m = re.match(r"(?is)^select\s+(.*?)\s+from\s+(.*?)\s+group\s+by\s+(\w+)\.(\w+)$", sql)
    if not m:
        raise ValueError("not a job-light GROUP BY query: " + sql[:80])
    items = [x.strip() for x in m.group(1).split(",")]
    galias, gcol = m.group(3), m.group(4)
    if sorted(x.lower().replace(" ", "") for x in items) != sorted(["count(*)", f"{galias}.{gcol}".lower()]):
        raise ValueError("the select list of a GROUP BY must be the grouping column and COUNT(*): " + m.group(1))
    rest = m.group(2)
    order, conds = parse_job_light("SELECT COUNT(*) FROM " + rest)
    alias_of = {part.split()[-1]: part.split()[0] for part in re.split(r"(?i)\s+where\s+", rest)[0].split(",")}
    if galias not in alias_of:
        raise ValueError(f"grouping column {galias}.{gcol}: unknown alias")
    return order, conds, alias_of[galias], gcol


def plan_star_groupby(sql: str, join_sizes: Dict[int, float]) -> dict:
    """One job-light GROUP BY text -> ``{"column", "where", "plan"}``, the plan of every group at once.

    ``plan`` is :func:`plan_star_query`'s factor list for the query with the grouping column counted as a conditioned column:
    an equality with the placeholder :data:`GROUP_VALUE`, which is what the per-value query ``... AND x.col = v`` sees (``=``
    wins over the column's other conditions in ``_table_query``).  ``_first_table``, ``factor_refine`` and the title conditions
    therefore do not depend on v: :func:`groupby_value_plan` with v is ``plan_star_query`` of the per-value text.  ``where`` is
    the ``_table_query`` value of the grouping column's own WHERE conditions (``None`` without any): they select the groups."""
    order, conds, table, col = parse_job_light_groupby(sql)
    where = _table_query(table, [c for c in conds.get(table, []) if c[0] == col]).get(f"{table}.{col}")
    conds = {t: list(c) for t, c in conds.items()}
    conds.setdefault(table, []).append((col, "=", GROUP_VALUE))
    return {"column": f"{table}.{col}", "where": where, "plan": _plan(order, conds, join_sizes)}


def groupby_value_plan(planned: dict, value) -> list:
    """The plan of one group: ``planned["plan"]`` with the placeholder replaced by ``value``."""
    out = [planned["plan"][0]]
    for f in planned["plan"][1:]:
        q = {k: (value if x is GROUP_VALUE else x) for k, x in f["query"].items()}
        out.append({"bn_index": f["bn_index"], "inverse": f["inverse"], "query": q, "expectation": list(f["expectation"])})
    return out


def groupby_sql_batch(ensemble, sqls: Sequence[str], join_sizes: Dict[int, float] = None) -> List[dict]:
    """job-light GROUP BY texts -> one ``{key: estimate}`` per text (:meth:`BN_ensemble.groupby_batch`; the texts that group
    by the same column are answered together).  ``join_sizes``: ``{bn_index: full join size}``, by default each BN's
    ``nrows``."""
    if join_sizes is None:
        join_sizes = {i: float(ensemble.bns[i].nrows) for i in range(len(BN_INDEX))}
    planned = [plan_star_groupby(s, join_sizes) for s in sqls]
    out: List[dict] = [{} for _ in sqls]
    for column in dict.fromkeys(p["column"] for p in planned):
        idx = [i for i, p in enumerate(planned) if p["column"] == column]
        keys, est = ensemble.groupby_batch([planned[i] for i in idx], column)
        for j, i in enumerate(idx):
            out[i] = {k: float(e) for k, e in zip(keys, est[j])}
    return out


class NativeJobLight:
    """The whole job-light path off the Python hot loop: ``cardinality_sql_batch(sqls)`` plans a batch of SQL texts
    (``bc_joblight_plan``, C++), decodes and packs every factor (``bc_sqlc_compile_factors``, C++, the column tables of each
    BN), runs one device batch per BN and descriptor kind, and combines (``bc_joblight_combine``).  Queries the native planner
    declines (not a job-light star) and factors the native decoder declines go through :func:`plan_star_query` and the Python
    mirror, so the results equal ``BN_ensemble.cardinality(parse_query_all(plan_workload(sqls)))`` either way."""

    def __init__(self, ensemble):
        import ctypes as C

        import numpy as np

        from . import _lib as L
        from .sqlc import SqlBatchCompiler

        self.ens = ensemble
        self.n_bn = len(BN_INDEX)
        tables = [t for t, _ in sorted(BN_INDEX.items(), key=lambda kv: kv[1])]
        self.tables = tables
        self.machines = [ensemble.bns[i]._machine() for i in range(self.n_bn)]
        self.sqlc = [SqlBatchCompiler(ensemble.bns[i].tree, self.machines[i].compiler) for i in range(self.n_bn)]
        fan = np.full((self.n_bn, self.n_bn), -1, dtype=np.int32)
        for a in range(self.n_bn):
            tm = ensemble.bns[a].tree
            for b in range(self.n_bn):
                name = f"title.mul_{tables[b]}.movie_id"
                if name in tm._index and tm.fan_vector(tm._index[name]) is not None:
                    fan[a, b] = tm._index[name]
        joins = np.asarray([float(ensemble.bns[i].nrows) for i in range(self.n_bn)], dtype=np.float64)
        pairs = list(PAIRWISE_RDC.items())
        enc = lambda xs: (C.c_char_p * max(1, len(xs)))(*[x.encode() for x in xs])
        ra, rb = enc([k[0] for k, _ in pairs]), enc([k[1] for k, _ in pairs])
        rv = np.asarray([v for _, v in pairs], dtype=np.float64)
        hs = (C.c_void_p * self.n_bn)(*[c._h for c in self.sqlc])
        tb = enc(tables)
        h = C.c_void_p()
        L.check(L.lib().bc_joblight_create(self.n_bn, C.cast(hs, C.c_void_p), C.cast(tb, C.c_void_p), joins.ctypes.data, fan.ctypes.data,
                                           len(pairs), C.cast(ra, C.c_void_p), C.cast(rb, C.c_void_p), rv.ctypes.data, EPSILON, C.byref(h)))
        self._h = h
        self.join_sizes = {i: joins[i] for i in range(self.n_bn)}

    def close(self):
        from . import _lib as L

        if getattr(self, "_h", None):
            L.lib().bc_joblight_destroy(self._h)
            self._h = None
        if getattr(self, "_dev_pool", None) is not None:
            self._dev_pool.shutdown(wait=True)
            self._dev_pool = None
        for c in getattr(self, "sqlc", []):
            c.close()

    @staticmethod
    def join_texts(sqls: Sequence[str]):
        """A batch of SQL strings as ONE buffer + offsets (what ``bc_joblight_plan_text`` reads): ``(bytes, uint64[n + 1])``."""
        import numpy as np

        n = len(sqls)
        blob = "\n".join(sqls).encode("utf-8")
        lens = np.fromiter(map(len, sqls), dtype=np.uint64, count=n)
        if n and int(lens.sum()) + n - 1 != len(blob):   # non-ASCII text: byte lengths differ from character counts
            lens = np.fromiter((len(s.encode("utf-8")) for s in sqls), dtype=np.uint64, count=n)
        off = np.zeros(n + 1, dtype=np.uint64)
        if n:
            np.cumsum(lens + np.uint64(1), out=off[1:])
            off[n] -= np.uint64(1)
        return blob, off

    def plan(self, sqls, text_off=None):
        """The factor table of a batch: dict of numpy arrays (``status, join_size, first_factor, factor_bn, factor_inverse,
        factor_fan_mask, pred_off, pred_col, pred_kind, pred_a, pred_b``).  ``sqls``: a sequence of SQL strings, or one
        ``bytes`` buffer with ``text_off`` (``uint64[n + 1]``: query q is ``sqls[text_off[q]:text_off[q + 1]]``)."""
        import ctypes as C

        import numpy as np

        from . import _lib as L

        if isinstance(sqls, (bytes, bytearray, memoryview)):
            blob, off = bytes(sqls) if not isinstance(sqls, bytes) else sqls, np.ascontiguousarray(text_off, dtype=np.uint64)
        else:
            blob, off = self.join_texts(sqls)
        n = int(off.size) - 1
        if n > 0 and int(off[n]) > len(blob):
            raise ValueError("text_off runs past the text buffer")
        # (a query ends one byte before the next one's offset when the buffer was joined with a separator: the parser strips it)
        text = C.c_char_p(blob)
        status = np.zeros(n, dtype=np.uint8)
        join = np.zeros(n, dtype=np.float64)
        first = np.zeros(n + 1, dtype=np.uint32)
        cap_f, cap_p = max(16, 3 * n), max(64, 10 * n)
        while True:
            f_bn = np.empty(cap_f, dtype=np.int32)
            f_inv = np.empty(cap_f, dtype=np.uint8)
            f_fan = np.empty(cap_f, dtype=np.uint32)
            p_off = np.empty(cap_f + 1, dtype=np.uint32)
            p_col = np.empty(cap_p, dtype=np.int32)
            p_kind = np.empty(cap_p, dtype=np.uint8)
            p_a = np.empty(cap_p, dtype=np.float64)
            p_b = np.empty(cap_p, dtype=np.float64)
            nf, npred = C.c_size_t(), C.c_size_t()
            rc = L.lib().bc_joblight_plan_text(self._h, n, text, off.ctypes.data, status.ctypes.data, join.ctypes.data, first.ctypes.data,
                                               cap_f, f_bn.ctypes.data, f_inv.ctypes.data, f_fan.ctypes.data, p_off.ctypes.data, cap_p,
                                               p_col.ctypes.data, p_kind.ctypes.data, p_a.ctypes.data, p_b.ctypes.data, C.byref(nf), C.byref(npred))
            if rc == L.ELIMIT and (nf.value > cap_f or npred.value > cap_p):
                cap_f, cap_p = max(cap_f, nf.value), max(cap_p, npred.value)
                continue
            L.check(rc)
            break
        nf, npred = nf.value, npred.value
        return {"status": status, "join_size": join, "first_factor": first, "factor_bn": f_bn[:nf], "factor_inverse": f_inv[:nf],
                "factor_fan_mask": f_fan[:nf], "pred_off": p_off[:nf + 1], "pred_col": p_col[:npred], "pred_kind": p_kind[:npred],
                "pred_a": p_a[:npred], "pred_b": p_b[:npred], "n_queries": n}

    def factor_rows(self, plan, wsparse: bool = False):
        """Per BN: ``(factor ids, kind, BITS rows, DENSE rows | WSPARSE (row_off, words), dense index)`` of the planned factors."""
        import numpy as np

        out = {}
        for b in range(self.n_bn):
            ids = np.nonzero(plan["factor_bn"] == b)[0].astype(np.uint32)
            if ids.size == 0:
                continue
            out[b] = (ids,) + self.sqlc[b].compile_factors(ids, plan["pred_off"], plan["pred_col"], plan["pred_kind"], plan["pred_a"],
                                                           plan["pred_b"], plan["factor_fan_mask"], wsparse)
        return out

    def cardinality_sql_batch(self, sqls, text_off=None, timing=None):
        """Cardinalities of a batch of job-light SQL texts (a sequence of strings, or one ``bytes`` buffer + ``text_off``).
        ``timing``: optional dict that receives the seconds spent per phase."""
        import time

        import numpy as np

        from . import _lib as L

        t0 = time.perf_counter()
        plan = self.plan(sqls, text_off)
        nq = plan["n_queries"]
        t1 = time.perf_counter()
        nf = plan["factor_bn"].size
        prob = np.zeros(nf, dtype=np.float64)
        python_factors = []

        def device_part(b, ids, kind, bits, ws, didx):
            """One BN's factors through the device (disjoint slots of ``prob``); returns the factors the mirror has to redo."""
            m = self.machines[b]
            mask = plan["factor_fan_mask"][ids].reshape(-1, 1)
            if np.count_nonzero(kind == L.SQLC_BITS):
                # every row of the BN goes through the kernel (rows of the other kinds hold arbitrary selection bits: finite
                # results that are not used) -- cheaper than gathering the BITS rows on the host
                p_all = m.dev.run_host(bits, L.DESC_BITS, mask, m.kernel)
                sel = np.nonzero(kind == L.SQLC_BITS)[0]
                prob[ids[sel]] = p_all[sel]
            if didx.size:   # fractional weights: weighted runs over PCIe (~100 B per factor), DENSE rows built on the device
                prob[ids[didx]] = m.dev.run_wsparse_host(ws[0], ws[1], np.ascontiguousarray(mask[didx]), m.kernel)
            # SQLC_ZERO: probability 0 (already) -- except on an EXPECTATION factor: Bayescard_BN.expectation has no guard for an
            # undecodable predicate and the reference fails there (Models/Bayescard_BN.py:581-583); the mirror raises the same
            bad = (kind == L.SQLC_PYTHON) | ((kind == L.SQLC_ZERO) & (mask[:, 0] != 0))
            return ids[np.nonzero(bad)[0]].tolist() if bad.any() else []

        # decode + pack of model b + 1 (host threads inside the library) runs while model b is on the device (one worker thread:
        # the device calls block in CUDA with the GIL released)
        if getattr(self, "_dev_pool", None) is None:
            from concurrent.futures import ThreadPoolExecutor

            self._dev_pool = ThreadPoolExecutor(max_workers=1)
        t_dec = 0.0
        futs = []
        for b in range(self.n_bn):
            td = time.perf_counter()
            ids = np.nonzero(plan["factor_bn"] == b)[0].astype(np.uint32)
            if ids.size == 0:
                continue
            rows_b = self.sqlc[b].compile_factors(ids, plan["pred_off"], plan["pred_col"], plan["pred_kind"], plan["pred_a"],
                                                  plan["pred_b"], plan["factor_fan_mask"], True)
            t_dec += time.perf_counter() - td
            futs.append(self._dev_pool.submit(device_part, b, ids, *rows_b))
        t2 = time.perf_counter()
        for f in futs:
            python_factors.extend(f.result())
        t3 = time.perf_counter()
        out = np.zeros(nq, dtype=np.float64)
        redo = set(np.nonzero(plan["status"])[0].tolist())
        if python_factors:   # a factor the native decoder declined: its whole query goes through the mirror
            owner = np.searchsorted(plan["first_factor"], np.asarray(python_factors), side="right") - 1
            redo.update(int(q) for q in owner)
        L.check(L.lib().bc_joblight_combine(nq, plan["status"].ctypes.data, plan["join_size"].ctypes.data,
                                            plan["first_factor"].ctypes.data, plan["factor_inverse"].ctypes.data, prob.ctypes.data,
                                            out.ctypes.data))
        if redo:
            if isinstance(sqls, (bytes, bytearray, memoryview)):
                off = np.asarray(text_off, dtype=np.uint64)
                text_of = lambda q: bytes(sqls[int(off[q]):int(off[q + 1])]).decode("utf-8")
            else:
                text_of = lambda q: sqls[q]
            for q in sorted(redo):
                tq = self.ens.parse_query_all([plan_star_query(text_of(q), self.join_sizes)])[0]
                out[q] = float(np.asarray(self.ens.cardinality(tq)).reshape(-1)[0])
        if timing is not None:
            timing.update(plan=t1 - t0, decode_pack=t_dec, decode_pack_with_device_overlapped=t2 - t1, device_tail=t3 - t2,
                          combine=time.perf_counter() - t3, factors=int(nf))
        return out
