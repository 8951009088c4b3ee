#!/usr/bin/env python
"""Incremental update of a served model (bc_model_update) against a full refit of the changed table.

Base tables, sampled on the device from the shipped models (synth.sample_table_device, seeded): DMV-shaped 11 575 467 x 10
and Census-shaped 2 458 285 x 68 (uint8, topological column order).  The base model is fitted on the base table
(bc_fit_counts).  Changes: inserts of 0.1 %, 1 % and 10 % of the base rows, drawn from a model of the same shape with
reversed CPT rows (so that the CPTs really move), and a delete of the first 1 % of the base rows.  Per change, on a fresh
DeviceModel with the counts attached and the specialised kernel of the base CPTs attached:
  update_ms          bc_model_update on device rows, CUDA events around the call (delta counts, validation, apply,
                     normalisation, host mirror, dropping the modules and plans)
  first_auto_ms      the first 1 M-row BITS batch through BC_KERNEL_AUTO after it (no specialised image: includes the
                     K3 / K2 plan rebuild), CUDA events; steady_auto_ms: the same batch again
  respec_cold_ms     bc_model_specialize with no cubin of the new CPTs in the cache (the driver JIT), host clock
  respec_warm_ms     bc_model_specialize with the cubin already assembled (ptxas, not timed), host clock
  update_rows_ms     Bayescard_BN.update_rows with host rows in node_names order (H2D, update, CPT refresh of the
                     touched nodes), host clock; the model is built with specialize=False, so no re-specialisation
  refit_ms           fit.refit of the whole changed table from the host (H2D, counting, normalisation), host clock
  refit_count_ms     bc_fit_counts over the whole changed table already on the device, CUDA events
and a check that the updated counts equal bc_fit_counts of the changed table.  The card name, power limit and max SM clock
are read in the same run.  One JSON record.

    python tools/update_bench.py [--out profiles/r6_update_bench.json]
"""
from __future__ import annotations

import argparse
import copy
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

BASES = {"dmv": 11_575_467, "census": 2_458_285}
CHANGES = [("insert", 0.001), ("insert", 0.01), ("insert", 0.10), ("delete", 0.01)]


def events_ms(fn):
    import torch

    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b), out


def host_ms(fn):
    import torch

    torch.cuda.synchronize()
    t = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t) * 1e3, out


def main():
    import torch

    from bayescard_b200 import _lib as L
    from bayescard_b200 import aot
    from bayescard_b200 import fit as F
    from bayescard_b200.engine import DeviceModel
    from bayescard_b200.loader import TreeModel
    from bayescard_b200.model import Bayescard_BN
    from bayescard_b200.synth import sample_table_device

    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r6_update_bench.json"))
    ap.add_argument("--queries", type=int, default=1 << 20)
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    st = torch.cuda.current_stream().cuda_stream
    rec = {"gpu": smi, "queries_per_batch": args.queries, "bases": {}}
    for name, n_rows in BASES.items():
        gen = TreeModel.load(os.path.join(ROOT, "tests", "golden", "models", name + ".npz"))
        other = copy.copy(gen)
        other.cpts = [np.asarray(c)[::-1].copy() if v == 0 else np.asarray(c)[::-1, :].copy() for v, c in enumerate(gen.cpts)]
        table = sample_table_device(gen, n_rows, seed=1)
        extra = sample_table_device(other, int(round(0.10 * n_rows)), seed=2)
        n = gen.n_nodes
        off, total = F.count_layout(gen.parent, gen.card)

        def count(t, rows):
            c = torch.empty(total + 1, dtype=torch.int64, device="cuda")
            F.fit_counts_device(gen.parent, gen.card, t.data_ptr(), rows, 1, n, c.data_ptr(), 0, st)
            return c

        base_counts = count(table, n_rows)[:total].cpu().numpy().astype(np.uint64)
        base = copy.copy(gen)
        base.cpts = F.counts_to_cpts(gen.parent, gen.card, base_counts)
        base.counts, base.fit_rows, base.nrows, base.fanouts = base_counts, n_rows, n_rows, {}
        # the query batch: 1 M BITS rows from the device generator
        probe = DeviceModel(base, device=0, specialize=False)
        desc = torch.empty((args.queries, probe.desc_stride(L.DESC_RANGE_U8)), dtype=torch.uint8, device="cuda")
        bits = torch.empty((args.queries, probe.desc_stride(L.DESC_BITS)), dtype=torch.uint8, device="cuda")
        out = torch.empty(args.queries, dtype=torch.float32, device="cuda")
        probe.gen_range_queries_device(3, 0, args.queries, 1, min(n, 8), desc.data_ptr(), st)
        probe.convert_device(desc.data_ptr(), L.DESC_RANGE_U8, bits.data_ptr(), L.DESC_BITS, args.queries, st)
        probe.close()
        del desc
        base_cache = tempfile.mkdtemp(prefix="bc_upd_base_")
        aot.build_cubin(base, base_cache)
        # warm-up: the first update of the process loads the update kernels (not timed)
        dm = DeviceModel(base, device=0, specialize=False)
        dm.attach_counts(base_counts)
        dm.update(extra[:1000].data_ptr(), table[:1000].data_ptr(), n_inserted=1000, n_deleted=1000, elem_bytes=1, stream=st)
        dm.close()
        rows = []
        for kind, frac in CHANGES:
            k = int(round(frac * n_rows))
            ins = extra[:k] if kind == "insert" else None
            dele = table[:k] if kind == "delete" else None
            assert (ins if ins is not None else dele).shape[0] == k
            dm = DeviceModel(base, device=0, specialize=True, cache_dir=base_cache)
            assert dm.has_spec, dm.spec_error
            dm.attach_counts(base_counts)
            dm._specialize = False   # re-specialisation is timed separately below
            dm.run_device(bits.data_ptr(), args.queries, L.DESC_BITS, out.data_ptr(), L.KERNEL_AUTO, st)   # warm
            upd_ms, _ = events_ms(lambda: dm.update(ins.data_ptr() if ins is not None else None,
                                                    dele.data_ptr() if dele is not None else None,
                                                    n_inserted=k if ins is not None else 0, n_deleted=k if dele is not None else 0,
                                                    elem_bytes=1, stream=st))
            assert not dm.has_spec
            first_ms, _ = events_ms(lambda: dm.run_device(bits.data_ptr(), args.queries, L.DESC_BITS, out.data_ptr(),
                                                          L.KERNEL_AUTO, st))
            steady_ms, _ = events_ms(lambda: dm.run_device(bits.data_ptr(), args.queries, L.DESC_BITS, out.data_ptr(),
                                                           L.KERNEL_AUTO, st))
            # the changed table on the device, counted from scratch: the reference point for the counts and the refit
            changed = torch.cat([table, ins]) if ins is not None else table[k:]
            want = count(changed, changed.shape[0])[:total].cpu().numpy().astype(np.uint64)
            counts_ok = bool(np.array_equal(dm.get_counts(), want))
            new = copy.copy(base)
            new.cpts = F.counts_to_cpts(base.parent, base.card, want)
            cold = tempfile.mkdtemp(prefix="bc_upd_cold_")
            cold_ms, _ = host_ms(lambda: dm.specialize(cold))
            assert dm.has_spec
            warm = tempfile.mkdtemp(prefix="bc_upd_warm_")
            aot.build_cubin(new, warm)
            warm_ms, _ = host_ms(lambda: dm.specialize(warm))
            spec_ms, _ = events_ms(lambda: dm.run_device(bits.data_ptr(), args.queries, L.DESC_BITS, out.data_ptr(),
                                                         L.KERNEL_AUTO, st))
            dm.close()
            shutil.rmtree(cold, ignore_errors=True)
            shutil.rmtree(warm, ignore_errors=True)
            refit_count_ms, _ = events_ms(lambda: count(changed, changed.shape[0]))
            host_changed = changed.cpu().numpy()
            refit_ms, _ = host_ms(lambda: F.refit(base, host_changed))
            del host_changed, changed
            # the Python entry point with host rows in node_names order
            bn = Bayescard_BN(copy.copy(base), device=0, specialize=False)
            bn.tree.counts = base_counts.copy()
            bn.tree.cpts = list(base.cpts)
            bn.init_inference_method()
            bn.update_rows()   # attaches the counts
            perm = [bn.tree.infer_names.index(c) for c in bn.tree.node_names]
            h_ins = None if ins is None else np.ascontiguousarray(ins.cpu().numpy()[:, perm])
            h_del = None if dele is None else np.ascontiguousarray(dele.cpu().numpy()[:, perm])
            rows_ms, _ = host_ms(lambda: bn.update_rows(h_ins, h_del))
            rows_ok = bool(np.array_equal(bn.tree.counts, want))
            bn.close()
            row = {"change": kind, "fraction": frac, "rows": k, "row_bytes": k * n, "update_ms": upd_ms,
                   "first_auto_ms": first_ms, "steady_auto_ms": steady_ms, "respec_cold_ms": cold_ms, "respec_warm_ms": warm_ms,
                   "spec_auto_ms": spec_ms, "update_rows_ms": rows_ms, "refit_ms": refit_ms, "refit_count_ms": refit_count_ms,
                   "counts_equal_refit": counts_ok, "update_rows_counts_equal_refit": rows_ok}
            print(name, json.dumps(row), flush=True)
            rows.append(row)
        shutil.rmtree(base_cache, ignore_errors=True)
        rec["bases"][name] = {"rows": n_rows, "cols": n, "counters": int(total), "changes": rows}
        del table, extra
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps({"gpu": smi, "out": args.out}))


if __name__ == "__main__":
    main()
