#!/usr/bin/env python
"""GROUP BY one column (bc_marginal_batch): the specialised marginal kernel against the expansion and a plain query.

DMV and Census: 1 M BITS rows from the device generator (bc_gen_range_queries + bc_convert_desc, seeded), three targets
each (the root, the deepest node, the widest column).  Per target, with CUDA events after a warm-up, `--reps` repetitions
(median / min / max):
  spec       bc_marginal_batch with BC_KERNEL_SPEC (the marginal module of the target attached)
  expansion  bc_marginal_batch with BC_KERNEL_AUTO on a model without that module (card(t) rows per query through the
             model's own AUTO dispatch, here its specialised query kernel)
  query      bc_query_batch with BC_KERNEL_AUTO on the same rows (one scalar per query)
plus output bytes and FFMA per query, and the largest relative difference of spec vs expansion on a 10 k sample.  A
synthetic tree with a 257-state column and no specialised module measures the expansion through AUTO on 100 k rows.
The 1 M rows (DMV 48 MB, Census 32 MB) fit in the 126 MB L2; the outputs (4 * card(t) MB) mostly do not.  One JSON record.

    python tools/groupby_bench.py [--reps 20] [--out profiles/r4_groupby_bench.json]
"""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys
import tempfile

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


def main():
    import torch

    from bayescard_b200 import _lib as L
    from bayescard_b200.engine import DeviceModel
    from bayescard_b200.loader import TreeModel
    from bayescard_b200.synth import make_tree_model
    import groupby_oracle as GO

    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rows", type=int, default=1 << 20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4_groupby_bench.json"))
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    models = os.path.join(ROOT, "tests", "golden", "models")
    st = torch.cuda.current_stream().cuda_stream
    cache = tempfile.mkdtemp(prefix="bc_marg_")
    res = []

    def measure(name, tm, spec_dm, plain_dm, targets, n):
        desc = torch.empty((n, plain_dm.desc_stride(L.DESC_RANGE_U8)), dtype=torch.uint8, device="cuda")
        bits = torch.empty((n, plain_dm.desc_stride(L.DESC_BITS)), dtype=torch.uint8, device="cuda")
        plain_dm.gen_range_queries_device(7, 0, n, 1, min(tm.n_nodes, 8), desc.data_ptr(), st)
        plain_dm.convert_device(desc.data_ptr(), L.DESC_RANGE_U8, bits.data_ptr(), L.DESC_BITS, n, st)
        del desc
        prob = torch.empty(n, dtype=torch.float32, device="cuda")
        q = timed(lambda: plain_dm.run_device(bits.data_ptr(), n, L.DESC_BITS, prob.data_ptr(), L.KERNEL_AUTO, st), args.reps)
        for role, t in targets:
            card = int(tm.card[t])
            out = torch.empty((n, card), dtype=torch.float32, device="cuda")
            rec = {"model": name, "target": t, "role": role, "card": card, "rows": n, "query_auto": q,
                   "out_bytes_per_query": 4 * card}
            if spec_dm is not None:
                rec["ffma_per_query"] = int(re.search(r"BC_SPEC_FFMA=(\d+)", spec_dm.marginal_source(t)).group(1))
                rec["spec"] = timed(lambda: spec_dm.run_marginal_device(bits.data_ptr(), n, L.DESC_BITS, t, out.data_ptr(),
                                                                        L.KERNEL_SPEC, st), args.reps)
                sample = min(n, 10000)
                spec_s = out[:sample].cpu().numpy().astype(np.float64)
            rec["expansion_auto"] = timed(lambda: plain_dm.run_marginal_device(bits.data_ptr(), n, L.DESC_BITS, t, out.data_ptr(),
                                                                               L.KERNEL_AUTO, st), args.reps)
            if spec_dm is not None:
                exp_s = out[:sample].cpu().numpy().astype(np.float64)
                err = np.abs(spec_s - exp_s) / np.maximum(np.abs(exp_s), 1e-300)
                err[(spec_s == 0) & (exp_s == 0)] = 0
                rec["spec_vs_expansion_max_rel"] = float(err.max())
                rec["speedup_vs_expansion"] = rec["expansion_auto"]["median_ms"] / rec["spec"]["median_ms"]
                rec["spec_over_query"] = rec["spec"]["median_ms"] / q["median_ms"]
            res.append(rec)
            print(json.dumps(rec), flush=True)
            del out

    for name in ("dmv", "census"):
        tm = TreeModel.load(os.path.join(models, name + ".npz"))
        tg = GO.tree_targets(tm)
        targets = list(dict.fromkeys((r, tg[r]) for r in ("root", "deepest", "widest")))
        GO.assemble_marginals(tm, [t for _, t in targets], cache)
        spec_dm = DeviceModel(tm, device=0, specialize=True)
        plain_dm = DeviceModel(tm, device=0, specialize=True)   # same query kernels, no marginal module
        assert spec_dm.has_spec and plain_dm.has_spec, spec_dm.spec_error
        for _, t in targets:
            assert spec_dm.specialize_marginal(t, cache), spec_dm.marginal_error.get(t)
        measure(name, tm, spec_dm, plain_dm, targets, args.rows)
        spec_dm.close()
        plain_dm.close()
    cards = [7, 130, 33, 257, 64, 5, 90, 200, 17, 128, 40, 3]
    syn = make_tree_model(len(cards), cards, seed=12, dtype=np.float32)
    plain = DeviceModel(syn, device=0, specialize=False)
    measure("synthetic_12col_257", syn, None, plain, [("small", 5), ("widest", 3)], 100_000)
    plain.close()
    rec = {"tool": "tools/groupby_bench.py", "gpu": smi, "reps": args.reps, "results": res}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
