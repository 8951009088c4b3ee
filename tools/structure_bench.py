#!/usr/bin/env python
"""Structure learning throughput: all-pairs counts (bc_pair_counts) and the whole Chow-Liu call (bc_chow_liu).

Tables are sampled on the device from seeds: Census-shaped (2 458 285 x 68) and DMV-shaped (11 591 877 x 10) by
ancestral sampling of the shipped models, and a wide synthetic one (1 M rows x 100 columns x 100 bins, S = 10 000).
Per table: kernel time of the counts with CUDA events (warmed up, repeated, median and spread), the bc_chow_liu call
time, algorithmic pair counters per row, the int8 MACs the tensor cores execute (whole 256 x 256 window pairs, minus the
skipped diagonal quarter) as a fraction of the data-sheet dense INT8 rate, table bytes / HBM bandwidth, and the host
time of the numpy oracle's counting on the same table.  One JSON record.

    python tools/structure_bench.py [--reps 20] [--out profiles/r3_structure_bench.json]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

INT8_DENSE_OPS = 4.5e15      # NVIDIA HGX B200 data sheet, per GPU, dense INT8 (ops = 2 x MAC), 1 000 W card
HBM_BYTES_PER_S = 7.7e12     # same data sheet


def tensor_macs(card, rows):
    """MACs issued: per window pair (I, J >= I) and 128-row tile 2 x M128 x N256 x K128, N128 for the diagonal's second
    accumulator."""
    w = -(-int(np.sum(card)) // 256)
    pairs = w * (w + 1) // 2
    tiles = -(-rows // 128)
    return tiles * 128 * (pairs * 2 * 128 * 256 - w * 128 * 128)


def main():
    import torch

    from bayescard_b200 import structure as S
    from bayescard_b200.loader import TreeModel
    from bayescard_b200.synth import make_tree_model, sample_table_device
    import structure_oracle as SO

    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_structure_bench.json"))
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    models = os.path.join(ROOT, "tests", "golden", "models")
    cases = [("census", TreeModel.load(os.path.join(models, "census.npz")), 2_458_285),
             ("dmv", TreeModel.load(os.path.join(models, "dmv.npz")), 11_591_877),
             ("wide_100x100", make_tree_model(100, 100, seed=1), 1_000_000)]
    stream = torch.cuda.current_stream()
    res = []
    for name, tm, rows in cases:
        t = sample_table_device(tm, rows, seed=1)
        card = np.ascontiguousarray(tm.card, dtype=np.int32)
        n = len(card)
        total = S.pair_count_layout(card)[2]
        counts = torch.empty(total + 1, dtype=torch.int64, device="cuda")

        def run():
            S.pair_counts_device(card, t.data_ptr(), rows, t.element_size(), n, counts.data_ptr(), 0, stream.cuda_stream)

        for _ in range(3):
            run()
        torch.cuda.synchronize()
        times = []
        for _ in range(args.reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            run()
            b.record()
            b.synchronize()
            times.append(a.elapsed_time(b) * 1e-3)
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for _ in range(5):
                run()
            torch.cuda.synchronize()
        per_kernel = {e.key: e.device_time_total * 1e-6 / 5 for e in prof.key_averages()
                      if e.device_time_total > 0 and "pair_" in e.key}
        host = t.cpu().numpy()
        host = host.view(np.uint16) if t.element_size() == 2 else host
        cl = []
        for _ in range(3):
            t0 = time.perf_counter()
            parent, _, bad = S.chow_liu(host, card)
            cl.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        want, want_bad = SO.pair_counts(card, host)
        t_oracle = time.perf_counter() - t0
        got = counts[:total].cpu().numpy().astype(np.uint64)
        med = float(np.median(times))
        macs = tensor_macs(card, rows)
        pairs = int(sum(int(card[i]) * int(card[j]) for i in range(n) for j in range(i + 1, n)))
        r = {"table": name, "rows": rows, "columns": n, "S": int(card.sum()), "elem_bytes": t.element_size(),
             "counts_equal_oracle": bool(np.array_equal(got, want)) and bad == want_bad,
             "counts_kernel_s": {"median": med, "min": float(np.min(times)), "max": float(np.max(times)), "reps": args.reps},
             "chow_liu_call_s_incl_host_to_device_copy": {"median": float(np.median(cl)), "min": float(np.min(cl))},
             "kernel_s_per_call_profiler": per_kernel,
             "pair_counters_per_row": pairs,
             "tensor_int8_macs": macs,
             "fraction_of_datasheet_int8_dense": 2 * macs / med / INT8_DENSE_OPS,
             "table_bytes": rows * n * t.element_size(),
             "table_read_at_datasheet_hbm_s": rows * n * t.element_size() / HBM_BYTES_PER_S,
             "oracle_numpy_counting_s": t_oracle,
             "tree_equals_model": bool(np.array_equal(parent, tm.parent))}
        res.append(r)
        print(json.dumps(r), flush=True)
        del t, counts
        torch.cuda.empty_cache()
    rec = {"gpu": smi, "note": "counts: one bc_pair_counts call (pre-pass + tensor-core kernel), CUDA events; chow_liu: "
           "host clock around structure.chow_liu (host table -> device copy, counts, MI, Prim, MI back)", "results": res}
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print("gpu:", smi)


if __name__ == "__main__":
    main()
