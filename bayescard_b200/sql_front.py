"""Single-table SQL front end: ``SELECT COUNT(*) FROM t WHERE a OP v AND ...`` -> predicate dict, and
``SELECT a, COUNT(*) FROM t [WHERE ...] GROUP BY a`` -> (predicate dict, grouping column), and the same with two grouping
columns.

Same input language and output as the reference's ``parse_query_single_table``
(``Evaluation/cardinality_estimation.py:22-119``), which feeds ``Bayescard_BN.query``:

* ``col IN [a, b, ...]``: a Python literal list if it parses as one, otherwise the bracket body
  split on commas and stripped (bare words; an empty item from a trailing comma is kept, ``:28-35``);
* ``< > <= >= = ==`` with an int, float or bare-word operand (tried in that order, ``:48-57``);
* continuous columns collect a ``(lo, hi)`` interval, strict bounds moved by ``1e-6`` (``:63-83``),
  repeated predicates intersect (``:87-91``);
* categorical columns collect the list of ORIGINAL values that satisfy the predicate, inequality
  operators being evaluated against ``BN.domain[attr]`` (``:97-103``); repeated predicates intersect
  keeping the order of the newest list (``:105-109``).
"""
from __future__ import annotations

import ast
import operator
import re
from typing import Any, Dict, Tuple

import numpy as np

_CMP = {">": np.greater, "<": np.less, ">=": np.greater_equal, "<=": np.less_equal, "=": np.equal, "==": np.equal}
_OP_CHARS = set("<>=")
EPSILON = 1e-6


def _scalar(text: str) -> Any:
    for conv in (int, float):
        try:
            return conv(text)
        except Exception:  # noqa: BLE001
            pass
    return text


def split_predicate(pred: str) -> Tuple[str, str, Any]:
    """``'a >= 3'`` -> ``('a', '>=', 3)``; ``'a IN [x, y]'`` -> ``('a', 'in', ['x', 'y'])``."""
    parts = pred.split(" IN ")
    if len(parts) != 1:
        body = parts[1].strip()
        try:
            values = list(ast.literal_eval(body))
        except Exception:  # noqa: BLE001 - bare words are not Python literals
            values = [item.strip() for item in body[1:-1].split(",")]
        return parts[0].strip(), "in", values
    first = next((i for i, ch in enumerate(pred) if ch in _OP_CHARS), None)
    if first is None:
        # the reference falls through with op_start = 0 and an unbound op_end (NameError)
        raise NameError("predicate has no comparison operator: " + pred)
    last = first + 1 if first + 1 < len(pred) and pred[first + 1] in _OP_CHARS else first
    return pred[:first].strip(), pred[first:last + 1].strip(), _scalar(pred[last + 1:].strip())


def add_predicate(bn, table_query: Dict[str, Any], attr: str, op: str, val: Any, epsilon: float = EPSILON):
    """Fold one predicate into ``table_query`` (in place) and return it; None for unknown columns."""
    if bn is None or attr not in bn.attr_type:
        return None
    if bn.attr_type[attr] == "continuous":
        if op == ">=":
            dom = (val, np.inf)
        elif op == ">":
            dom = (val + epsilon, np.inf)
        elif op == "<=":
            dom = (-np.inf, val)
        elif op == "<":
            dom = (-np.inf, val - epsilon)
        elif op in ("=", "=="):
            dom = val
        else:
            raise AssertionError(f"operation {op} is invalid for continous domain")
        if attr in table_query:
            old = table_query[attr]
            dom = (max(old[0], dom[0]), min(old[1], dom[1]))
        table_query[attr] = dom
        return table_query
    domain = bn.domain[attr]
    if type(domain[0]) != str:
        domain = np.asarray(domain)
    if op == "in":
        if type(val) != list:
            raise AssertionError("use list for in query")
        dom = val
    elif op in ("=", "=="):
        dom = val if type(val) == list else [val]
    else:
        if type(val) == list:
            assert len(val) == 1
            val = val[0]
            assert type(val) == int or type(val) == float
        dom = list(domain[_CMP[op](domain, val)])
    if attr in table_query:
        earlier = table_query[attr]
        dom = [x for x in dom if x in earlier]
    table_query[attr] = dom
    return table_query


def parse_query_single_table(sql: str, bn) -> Dict[str, Any]:
    where = sql.split(" WHERE ")[-1].strip()
    out: Dict[str, Any] = {}
    for pred in where.split(" AND "):
        attr, op, val = split_predicate(pred.strip())
        add_predicate(bn, out, attr, op, val)
    return out


_GROUPBY = re.compile(r"^\s*SELECT\s+(?P<sel>.+?)\s+FROM\s+(?P<table>\S+?)(?:\s+WHERE\s+(?P<where>.+?))?"
                      r"\s+GROUP\s+BY\s+(?P<group>.+?)\s*;?\s*$", re.S | re.I)


def parse_groupby_single_table(sql: str, bn):
    """``SELECT a, COUNT(*) FROM t [WHERE ...] GROUP BY a`` -> ``(query, "a")`` and ``SELECT a, b, COUNT(*) FROM t [WHERE ...]
    GROUP BY a, b`` -> ``(query, ("a", "b"))``.  The WHERE clause is read as by :func:`parse_query_single_table`
    (``split_predicate`` / ``add_predicate``).  One or two distinct grouping columns, which the model must hold, and a
    select list of exactly those columns and ``COUNT(*)``; anything else raises ``ValueError``."""
    mt = _GROUPBY.match(sql)
    if mt is None:
        raise ValueError("not a single-table GROUP BY query: " + sql)
    group = [g.strip() for g in mt.group("group").split(",")]
    if len(group) not in (1, 2) or not all(group):
        raise ValueError("GROUP BY takes one or two columns here, got " + mt.group("group"))
    if len(set(group)) != len(group):
        raise ValueError("GROUP BY names a column twice: " + mt.group("group"))
    for column in group:
        if column not in bn.attr_type or column not in bn.tree._index:
            raise ValueError(f"GROUP BY column {column!r} is not a column of the model")
    sel = sorted(x.strip().replace(" ", "").upper() for x in mt.group("sel").split(","))
    if sel != sorted(["COUNT(*)"] + [c.upper() for c in group]):
        raise ValueError("the select list must be the grouping columns and COUNT(*): " + mt.group("sel"))
    out: Dict[str, Any] = {}
    if mt.group("where"):
        for pred in mt.group("where").split(" AND "):
            attr, op, val = split_predicate(pred.strip())
            add_predicate(bn, out, attr, op, val)
    return out, (group[0] if len(group) == 1 else tuple(group))
