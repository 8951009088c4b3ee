#!/usr/bin/env python
"""GROUP BY two columns (bc_joint_marginal_batch): the joint module against the expansions and the scalar floor.

Pairs: DMV -- a small sibling pair, an ancestor/descendant pair, the largest pair under the cap (BC_JOINT_MAX_FFMA) and one
pair over it; Census -- the widest-product pair, a deep pair whose lowest common ancestor is the root, and an
ancestor/descendant pair.  Rows: n = min(--rows, 1 GB / (4 card(a) card(b))) random BITS range queries per pair, generated
on the device, so the output is at most 1 GB.  BITS rows are 48-96 B: n rows are at most 25 MB and stay L2-resident (126 MB)
across repetitions; the output is written to HBM.  Per path, CUDA events after a warm-up, median of `--reps`:
  joint          BC_KERNEL_SPEC with the joint module of (a, b) attached (absent above the cap)
  expand_marg    BC_KERNEL_AUTO on a model with only b's marginal module: card(a) rows per query through that module
  expand_query   BC_KERNEL_AUTO on a model with only the spec module: card(a) * card(b) rows per query through bc_query_batch
  query          bc_query_batch on the same rows (one scalar per query): the floor
Reported: output bytes/s against 7.7 TB/s of HBM, executed FFMA/s (the module header's BC_SPEC_FFMA per query) against the
FP32 peak measured in the same run, and the largest relative difference of the module against the expansion on 4 k rows.
One JSON record with the card name, power limit and max SM clock read in the same run.

    python tools/joint_groupby_bench.py [--reps 10] [--rows 262144] [--out profiles/r7_joint_groupby_bench.json]
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

HBM_BYTES_PER_S = 7.7e12


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


def pick_pairs(name, m, dm):
    from bayescard_b200 import _lib as L
    from test_joint_groupby import census_pairs

    lib = L.lib()
    n = m.n_nodes
    ok = {}
    for a in range(n):
        for b in range(n):
            if a != b:
                ok[(a, b)] = lib.bc_model_joint_source(dm._h, a, b, None, 0) > 0
    prod = lambda p: int(m.card[p[0]]) * int(m.card[p[1]])  # noqa: E731
    if name == "dmv":
        kids = {}
        for v in range(1, n):
            kids.setdefault(int(m.parent[v]), []).append(v)
        sib = min(((k[i], k[j]) for k in kids.values() for i in range(len(k)) for j in range(i + 1, len(k))), key=prod)
        anc = max(((int(m.parent[v]), v) for v in range(1, n) if ok[(int(m.parent[v]), v)]), key=prod)
        largest = max((p for p in ok if ok[p] and p[0] < p[1]), key=prod)
        over = min((p for p in ok if not ok[p] and p[0] < p[1]), key=prod)
        return {"small_sibling": sib, "ancestor_descendant": anc, "largest_under_cap": largest, "over_cap": over}
    cp = census_pairs(m)
    widest = max((p for p in ok if ok[p] and p[0] < p[1]), key=prod)
    return {"widest_product": widest, "deep_lca_root": cp[3], "ancestor_descendant": cp[1]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--rows", type=int, default=262144)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r7_joint_groupby_bench.json"))
    args = ap.parse_args()

    import torch

    import golden_util as G
    from bayescard_b200 import _lib as L
    from bayescard_b200.engine import DeviceModel, measure_fp32_peak

    assert torch.cuda.is_available(), "the benchmark needs a GPU"
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    peak_tflops, _ = measure_fp32_peak(0)
    cache = tempfile.mkdtemp(prefix="bc_joint_bench_")
    st = torch.cuda.current_stream().cuda_stream
    record = {"hardware": smi, "fp32_peak_tflops_measured": peak_tflops, "hbm_bytes_per_s_datasheet": HBM_BYTES_PER_S,
              "reps": args.reps, "pairs": []}
    for name in ("dmv", "census"):
        m = G.model(name)
        host = DeviceModel(m, device=-1, specialize=False)
        pairs = pick_pairs(name, m, host)
        spec_only = DeviceModel(m, device=0, specialize=True, cache_dir=cache)
        for label, (a, b) in pairs.items():
            ca, cb = int(m.card[a]), int(m.card[b])
            n = int(min(args.rows, (1 << 30) // (4 * ca * cb)))
            desc = torch.empty((n, spec_only.desc_stride(L.DESC_RANGE_U8)), dtype=torch.uint8, device="cuda:0")
            bits = torch.empty((n, spec_only.desc_stride(L.DESC_BITS)), dtype=torch.uint8, device="cuda:0")
            spec_only.gen_range_queries_device(11, 0, n, 1, 5, desc.data_ptr(), st)
            spec_only.convert_device(desc.data_ptr(), L.DESC_RANGE_U8, bits.data_ptr(), L.DESC_BITS, n, st)
            del desc
            out = torch.empty(n * ca * cb, dtype=torch.float32, device="cuda:0")
            out2 = torch.empty_like(out)
            q = torch.empty(n, dtype=torch.float32, device="cuda:0")
            rec = {"model": name, "pair": label, "a": a, "b": b, "card_a": ca, "card_b": cb, "rows": n,
                   "out_bytes": 4 * n * ca * cb, "bits_row_bytes": spec_only.desc_stride(L.DESC_BITS)}
            jm = DeviceModel(m, device=0, specialize=False)
            has_joint = jm.specialize_joint(a, b, cache)
            if has_joint:
                src = jm.joint_source(a, b)
                ffma = int(re.search(r"BC_SPEC_FFMA=(\d+)", src).group(1))
                rec.update(loop_node=int(re.search(r"  X: (\d+)", src).group(1)), ffma_per_query=ffma,
                           fma_pipe_per_query=int(re.search(r"FMA-pipe=(\d+)", src).group(1)))
                rec["joint"] = timed(lambda: jm.run_joint_device(bits.data_ptr(), n, L.DESC_BITS, a, b, out.data_ptr(),
                                                                 L.KERNEL_SPEC, st), args.reps)
                t = rec["joint"]["median_ms"] * 1e-3
                rec["joint"]["queries_per_s"] = n / t
                rec["joint"]["out_bytes_per_s"] = rec["out_bytes"] / t
                rec["joint"]["out_bw_share_of_hbm"] = rec["out_bytes"] / t / HBM_BYTES_PER_S
                rec["joint"]["ffma_per_s"] = ffma * n / t
                rec["joint"]["ffma_share_of_fp32_peak"] = 2 * ffma * n / t / (peak_tflops * 1e12)
            else:
                rec["joint_refused"] = jm.joint_error[(a, b)]
            mm = DeviceModel(m, device=0, specialize=False)
            if mm.specialize_marginal(b, cache):
                rec["expand_marg"] = timed(lambda: mm.run_joint_device(bits.data_ptr(), n, L.DESC_BITS, a, b, out2.data_ptr(),
                                                                       L.KERNEL_AUTO, st), args.reps)
            rec["expand_query"] = timed(lambda: spec_only.run_joint_device(bits.data_ptr(), n, L.DESC_BITS, a, b, out2.data_ptr(),
                                                                           L.KERNEL_AUTO, st), min(args.reps, 3))
            rec["query"] = timed(lambda: spec_only.run_device(bits.data_ptr(), n, L.DESC_BITS, q.data_ptr(), 0, L.KERNEL_AUTO, st),
                                 args.reps)
            for k in ("expand_marg", "expand_query"):
                if has_joint and k in rec:
                    rec[f"joint_speedup_over_{k}"] = rec[k]["median_ms"] / rec["joint"]["median_ms"]
            if has_joint:
                s = min(n, 4096)
                jm.run_joint_device(bits.data_ptr(), s, L.DESC_BITS, a, b, out.data_ptr(), L.KERNEL_SPEC, st)
                mm.run_joint_device(bits.data_ptr(), s, L.DESC_BITS, a, b, out2.data_ptr(), L.KERNEL_GENERIC, st)
                torch.cuda.synchronize()
                x = out[: s * ca * cb].double().cpu().numpy()
                y = out2[: s * ca * cb].double().cpu().numpy()
                err = np.abs(x - y) / np.maximum(np.abs(y), 1e-30)
                err[(x == 0) & (y == 0)] = 0
                rec["max_rel_diff_joint_vs_expansion_k1"] = float(err.max())
            jm.close()
            mm.close()
            del out, out2, bits, q
            torch.cuda.empty_cache()
            record["pairs"].append(rec)
            print(json.dumps(rec), flush=True)
        spec_only.close()
        host.close()
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(record, f, indent=1)
    print(json.dumps({"hardware": smi, "fp32_peak_tflops_measured": peak_tflops}))


if __name__ == "__main__":
    main()
