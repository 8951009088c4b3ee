#!/usr/bin/env python
"""GROUP BY over fan-out expectations (bc_expectation_marginal_batch) and job-light GROUP BY end to end.

Marginals: IMDB model 1 (movie_info x title), targets title.kind_id, title.production_year and movie_info.info_type_id.
`--rows` (1 M) BITS rows and as many DENSE_F32 rows, tiled from the model's decoded infer_cases, each with a seeded random
set of the model's fan-out columns (mask rows).  Per target and format, CUDA events after a warm-up, `--reps` repetitions
(median / min / max):
  spec            bc_expectation_marginal_batch with BC_KERNEL_SPEC (the marginal module of the target attached)
  expansion_auto  the same call with BC_KERNEL_AUTO on a model without that module: card(t) rows (and mask rows) per query
                  through bc_query_batch's AUTO dispatch (K3 on this model)
  query_auto      bc_query_batch with the same rows and masks (one scalar per query)
plus the largest relative difference of spec vs expansion on a 10 k sample.  The rows are read from HBM (BITS 1 M x 80 B,
DENSE 1 M x 2 KB); the outputs are 4 * card(t) B per query.

job-light: the 70 shipped queries grouped by title.kind_id, title.production_year and a joined table's categorical column
(210 texts): joblight.groupby_sql_batch against the per-value loop (the plan of every group, parse_query_all and
BN_ensemble.cardinality_batch of the plans without an undecodable expectation factor), host clock around calls that return
host results; the largest relative difference of the non-zero groups.  One JSON record with the card name, power limit and
max SM clock read in the same run.

    python tools/join_groupby_bench.py [--reps 10] [--out profiles/r5_join_groupby_bench.json]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def timed(fn, reps):
    import torch

    fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return {"median_ms": float(np.median(ms)), "min_ms": float(np.min(ms)), "max_ms": float(np.max(ms))}


def wall(fn, reps):
    fn()
    s = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        s.append(time.perf_counter() - t0)
    return {"median_s": float(np.median(s)), "min_s": float(np.min(s)), "max_s": float(np.max(s))}


def marginals(args, res):
    import torch

    import golden_util as G
    import groupby_oracle as GO
    from bayescard_b200 import _lib as L
    from bayescard_b200.decode import PredicateCompiler
    from bayescard_b200.engine import DeviceModel

    tm = G.model("imdb1")
    targets = [tm._index[c] for c in ("title.kind_id", "title.production_year", "movie_info.info_type_id")]
    cache = tempfile.mkdtemp(prefix="bc_marg_")
    GO.assemble_marginals(tm, targets, cache)
    spec = DeviceModel(tm, device=0, specialize=False)
    for t in targets:
        assert spec.specialize_marginal(t, cache), spec.marginal_error.get(t)
    plain = DeviceModel(tm, device=0, specialize=False)   # no marginal module: AUTO expands
    pc = PredicateCompiler(tm)
    cases = [r for r in G.load("infer_cases.json.gz")["imdb1"] if "error" not in r]
    decoded = [({k: list(v) for k, v in r["bins"].items()}, {k: np.asarray(v) for k, v in r["weights"].items()}) for r in cases]
    decoded.append(({}, {}))
    rng = np.random.default_rng(0)
    fan = [tm.infer_names[v] for v in range(tm.n_nodes) if tm.fan_vector(v) is not None]
    fans = [[f for f in fan if rng.random() < 0.6] for _ in decoded]
    st = torch.cuda.current_stream().cuda_stream
    n = args.rows
    for force_dense, fmt, label in ((False, L.DESC_BITS, "BITS"), (True, L.DESC_DENSE_F32, "DENSE_F32")):
        b_idx, b_desc, d_idx, d_desc, mask = pc.pack(decoded, fans, force_dense=force_dense)
        idx, desc = (d_idx, d_desc) if force_dense else (b_idx, b_desc)
        pick = rng.integers(0, len(idx), size=n)
        d_rows = torch.from_numpy(np.ascontiguousarray(desc[pick]).reshape(-1).view(np.uint8)).to("cuda")
        d_mask = torch.from_numpy(np.ascontiguousarray(mask[idx][pick]).reshape(-1)).to("cuda")
        prob = torch.empty(n, dtype=torch.float32, device="cuda")
        q = timed(lambda: plain.run_device(d_rows.data_ptr(), n, fmt, prob.data_ptr(), d_mask.data_ptr(), L.KERNEL_AUTO, st), args.reps)
        for t in targets:
            card = int(tm.card[t])
            out = torch.empty((n, card), dtype=torch.float32, device="cuda")
            rec = {"model": "imdb1", "column": tm.infer_names[t], "target": t, "card": card, "format": label, "rows": n,
                   "row_bytes": int(d_rows.numel() // n), "query_auto": q}
            rec["spec"] = timed(lambda: spec.run_marginal_device(d_rows.data_ptr(), n, fmt, t, out.data_ptr(), L.KERNEL_SPEC, st,
                                                                 d_mask.data_ptr()), args.reps)
            sample = min(n, 10000)
            s_spec = out[:sample].cpu().numpy().astype(np.float64)
            rec["expansion_auto"] = timed(lambda: plain.run_marginal_device(d_rows.data_ptr(), n, fmt, t, out.data_ptr(), L.KERNEL_AUTO,
                                                                            st, d_mask.data_ptr()), args.reps)
            s_exp = out[:sample].cpu().numpy().astype(np.float64)
            err = np.abs(s_spec - s_exp) / np.maximum(np.abs(s_exp), 1e-300)
            err[(s_spec == 0) & (s_exp == 0)] = 0
            rec["spec_vs_expansion_max_rel"] = float(err.max())
            rec["spec_queries_per_s"] = n / (rec["spec"]["median_ms"] * 1e-3)
            rec["speedup_vs_expansion"] = rec["expansion_auto"]["median_ms"] / rec["spec"]["median_ms"]
            res.append(rec)
            print(json.dumps(rec), flush=True)
            del out
    spec.close()
    plain.close()


def joblight(args):
    import golden_util as G
    from bayescard_b200.ensemble import BN_ensemble
    from bayescard_b200.joblight import groupby_sql_batch, groupby_value_plan, plan_star_groupby
    from bayescard_b200.model import Bayescard_BN
    from test_join_groupby import _groupby_texts, _per_value_cardinalities

    bns = {}
    for i in range(5):
        bns[i] = Bayescard_BN(G.model(f"imdb{i}"), device=0, infer_algo="exact-jit")
        bns[i].init_inference_method()
    ens = BN_ensemble(bns=bns)
    js = {i: float(bns[i].nrows) for i in range(5)}
    texts = _groupby_texts()
    box = {}

    def grouped():
        box["g"] = groupby_sql_batch(ens, texts, js)

    def per_value():
        plans, owner = [], []
        for i, sql in enumerate(texts):
            planned = plan_star_groupby(sql, js)
            for k in box["g"][i]:
                plans.append(groupby_value_plan(planned, k))
                owner.append((i, k))
        box["p"] = (owner, _per_value_cardinalities(ens, plans))

    rec = {"texts": len(texts), "groupby_sql_batch": wall(grouped, args.reps_e2e), "per_value_loop": wall(per_value, args.reps_e2e)}
    owner, ref = box["p"]
    got = np.asarray([box["g"][i][k] for i, k in owner])
    nz = (got != 0) & ~np.isnan(ref)
    rec["per_value_undecodable"] = int(np.isnan(ref).sum())
    rec["groups"] = int(len(got))
    rec["nonzero_groups"] = int(nz.sum())
    rec["nonzero_max_rel_vs_per_value"] = float(np.max(np.abs(got[nz] - ref[nz]) / ref[nz]))
    rec["speedup"] = rec["per_value_loop"]["median_s"] / rec["groupby_sql_batch"]["median_s"]
    print(json.dumps(rec), flush=True)
    for bn in bns.values():
        bn.close()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--reps-e2e", type=int, default=3)
    ap.add_argument("--rows", type=int, default=1 << 20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r5_join_groupby_bench.json"))
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("join_groupby_bench needs a CUDA device")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    res = []
    marginals(args, res)
    e2e = joblight(args)
    rec = {"tool": "tools/join_groupby_bench.py", "gpu": smi, "reps": args.reps, "marginals": res, "job_light_groupby": e2e}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
