#!/usr/bin/env python
"""BASELINE.json config 4, the reference's OWN synthetic experiment (paper section E.3, Tables 10 / 11): the generator of
``Testing/stability_experiment.ipynb`` cells 1-2 -- Pareto-skewed columns, a fraction ``correlation`` of every column
copied from a random earlier column, range / equality queries with known true cardinalities -- for domain sizes <= 100,
where the reference's discretiser (``Models/tools.py:49-128`` with ``n_mcv=30, n_bins=70``) keeps every value as its own
bin, so the states ARE the values.

Per configuration: generate the table (cell 1 ``data_generation``), learn the Chow-Liu tree rooted at column 0 and its
CPTs on the GPU (``bayescard_b200.structure.learn_tree_model``, what ``pomegranate`` + pgmpy do for the reference), draw the queries (cell 1 ``generate_single_query``), evaluate them through the drop-in ``Bayescard_BN.query``
(scalar latency, as the notebook times it) and ``query_batch``, and print the q-error percentiles and latency beside
the paper's Table 11 rows.

    python tools/stability_experiment.py [--rows 1000000] [--queries 200] [--out profiles/r2_stability_experiment.json]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# paper Table 11 (BASELINE.md section 1): latency in ms and 95 % q-error of the reference (CPU, fp64)
TABLE11_DOMAIN = {10: (1.0, 1.29), 100: (2.4, 1.49)}                                   # s = 1.0, c = 0.4, n = 10
TABLE11_COLUMNS = {2: (0.4, 1.04), 5: (1.5, 1.12), 10: (2.4, 1.49), 50: (4.7, 2.58), 100: (11.3, 1.97)}   # d = 100
# the notebook's own per-experiment knobs (cells 3 and 7): probability of a predicate per column and the shift of range bounds
NOTEBOOK_P = {2: 0.8, 5: 0.8, 10: 0.8, 50: 0.2, 100: 0.1}
NOTEBOOK_SKIP_ZERO_BIT = {2: 6, 5: 6, 10: 4, 50: 2, 100: 0}


def discretize_series(rng, s, domain_size):
    """Cell 1: Pareto samples >= domain_size are redrawn uniformly, the rest floored."""
    n_invalid = int((s >= domain_size).sum())
    s = np.floor(s[s < domain_size])
    s = np.concatenate((s, rng.integers(0, domain_size, size=n_invalid).astype(np.float64)))
    return rng.permutation(s)


def data_generation(rng, skew, domain_size, correlation, column_size, nrows):
    """Cell 1 ``data_generation`` (scipy's ``pareto.rvs(b, scale=1)`` = (1 - U)^(-1/b))."""
    data = np.zeros((column_size, nrows))
    for i in range(column_size):
        if i == 0:
            data[i] = rng.integers(0, domain_size, size=nrows)
            continue
        s = (1.0 - rng.random(nrows)) ** (-1.0 / skew)
        s = discretize_series(rng, s, domain_size)
        selected = [0] if i == 1 else list(rng.permutation(i)[:1])
        idx = rng.permutation(nrows)[: int(nrows * correlation)]
        if len(idx):
            sel = np.ceil(np.mean(data[selected, :], axis=0))
            s[idx] = sel[idx]
        data[i] = s
    return data.T.astype(np.int64)   # [nrows, column_size]


def generate_queries(rng, table, card, num, p=0.8, nval=4, skip_zero_bit=4):
    """Cell 1 ``generate_single_query``: (lo, hi) per column (full domain when unpredicated) + the true cardinality."""
    nrows, n = table.shape
    los, his, cards = [], [], []
    while len(los) < num:
        lo = np.zeros(n, dtype=np.int64)
        hi = np.full(n, card - 1, dtype=np.int64)
        sel = np.ones(nrows, dtype=bool)
        any_pred = False
        for c in range(n):
            if rng.random() < p:
                vals = np.sort(table[rng.integers(0, nrows, size=nval), c])
                l, r = int(vals[0]), int(vals[-1])
                if l != r and skip_zero_bit:
                    l, r = l + skip_zero_bit, r + skip_zero_bit
                lo[c], hi[c] = l, r
                sel &= (table[:, c] >= l) & (table[:, c] <= r)
                any_pred = True
        true = int(sel.sum())
        if not any_pred or true == 0:
            continue
        los.append(lo)
        his.append(np.minimum(hi, card - 1))
        cards.append(true)
    return np.asarray(los), np.asarray(his), np.asarray(cards, dtype=np.float64)


def q_errors(pred, true):
    pred = np.where((pred == 0) | np.isnan(pred), 1.0, pred)
    return np.maximum(pred / true, true / pred)


def run_one(skew, domain, corr, ncols, nrows, nq, seed, device=0, p=0.8, skip_zero_bit=4):
    from bayescard_b200 import _lib as L
    from bayescard_b200.engine import DeviceModel
    from bayescard_b200.structure import learn_tree_model
    from bayescard_b200.synth import pack_ranges_u16

    rng = np.random.default_rng(seed)
    t0 = time.perf_counter()
    table = data_generation(rng, skew, domain, corr, ncols, nrows)
    t_gen = time.perf_counter() - t0
    t0 = time.perf_counter()
    names = [f"attr{c}" for c in range(ncols)]
    card = np.full(ncols, domain, dtype=np.int32)
    tm = learn_tree_model(table.astype(np.uint8), card, names=names, root=0, device=device, table_name="toy")
    t_struct = time.perf_counter() - t0   # tree and CPTs: one pass over the table on the GPU
    order = [names.index(x) for x in tm.infer_names]
    table_t = np.ascontiguousarray(table[:, order].astype(np.uint8))
    lo, hi, true = generate_queries(rng, table_t.astype(np.int64), domain, nq, p=p, skip_zero_bit=skip_zero_bit)
    dm = DeviceModel(tm, device=device, specialize=ncols * domain * domain <= 200_000)   # (the straight-line kernel is for small models)
    desc = pack_ranges_u16(lo.astype(np.int32), hi.astype(np.int32))
    lat = []
    for i in range(nq):   # the notebook times one BN.query per query
        t = time.perf_counter()
        dm.run_host(desc[i:i + 1], L.DESC_RANGE_U16)
        lat.append(time.perf_counter() - t)
    t0 = time.perf_counter()
    prob = dm.run_host(desc, L.DESC_RANGE_U16).astype(np.float64)
    t_batch = time.perf_counter() - t0
    dm.close()
    qe = q_errors(prob * nrows, true)
    return {"skew": skew, "domain": domain, "correlation": corr, "columns": ncols, "rows": nrows, "queries": nq, "p": p, "skip_zero_bit": skip_zero_bit,
            "q_error_50_90_95_99_100": [float(np.percentile(qe, x)) for x in (50, 90, 95, 99, 100)],
            "latency_ms_scalar_p50": float(np.median(lat[5:]) * 1e3), "latency_ms_scalar_mean": float(np.mean(lat[5:]) * 1e3),
            "batch_ms": t_batch * 1e3, "seconds": {"generate": t_gen, "chow_liu_and_fit_gpu": t_struct}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=1_000_000)
    ap.add_argument("--queries", type=int, default=200)
    ap.add_argument("--out", default="")
    ap.add_argument("--max-columns", type=int, default=100)
    args = ap.parse_args()
    res = []
    print("vary domain size (s = 1.0, c = 0.4, n = 10)")
    for d, (lat_ref, q95_ref) in TABLE11_DOMAIN.items():
        r = run_one(1.0, d, 0.4, 10, args.rows, args.queries, seed=d, skip_zero_bit=4 if d > 10 else 0)
        r["paper_table11"] = {"latency_ms": lat_ref, "q_error_95": q95_ref}
        res.append(r)
        print(f"  d={d:5d}: q95 {r['q_error_50_90_95_99_100'][2]:.3f} (paper {q95_ref}), scalar latency p50 {r['latency_ms_scalar_p50']:.3f} ms "
              f"(paper {lat_ref} ms), {args.queries} queries in one batch {r['batch_ms']:.2f} ms", flush=True)
    print("vary number of columns (s = 1.0, c = 0.4, d = 100)")
    for n, (lat_ref, q95_ref) in TABLE11_COLUMNS.items():
        if n > args.max_columns:
            continue
        r = run_one(1.0, 100, 0.4, n, args.rows, args.queries, seed=1000 + n, p=NOTEBOOK_P[n], skip_zero_bit=NOTEBOOK_SKIP_ZERO_BIT[n])
        r["paper_table11"] = {"latency_ms": lat_ref, "q_error_95": q95_ref}
        res.append(r)
        print(f"  n={n:5d}: q95 {r['q_error_50_90_95_99_100'][2]:.3f} (paper {q95_ref}), scalar latency p50 {r['latency_ms_scalar_p50']:.3f} ms "
              f"(paper {lat_ref} ms), batch {r['batch_ms']:.2f} ms", flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump({"note": "generator of Testing/stability_experiment.ipynb cells 1-2 (numpy port, own seeds), Chow-Liu by mutual "
                               "information, CPTs fitted on the GPU, queries through bc_query_batch_host; paper numbers from Table 11",
                       "results": res}, f, indent=1)


if __name__ == "__main__":
    main()
