#!/usr/bin/env python
"""bench.py -- queries/sec of exact tree inference (BASELINE.json metric) on N B200s.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the hot path over one batch of synthetic range-predicate queries:
BASELINE.json configs[1], "Census Chow-Liu BN, batch of 1M synthetic multi-column range queries"
(seeded counter-based generator, k ~ U{1..14} constrained columns, SURVEY.md section 8d).  With N > 1
every rank runs the same per-GPU batch on its own replica of the CPT arena (weak scaling; the path
has no exchange step, so no collective runs inside the timed region -- NCCL is used for the barrier
and the max-over-ranks reduction only).

  value        whole-job q/s, BITS descriptors (one bit per column state) already resident in HBM,
               CUDA events around K steps; the steps are independent batches and are launched on two
               streams in turn (--streams), so a launch's first CTAs fill the SMs the previous launch's
               last round leaves idle; the one-stream figure is printed in roofline.single_stream
  sustained    the same launch repeated back to back for >= 2 s (clocks settle below the burst clock)
  e2e          same metric through the host-buffer C-ABI: pinned host queries -> H2D -> expand to BITS ->
               kernel -> D2H of the fp32 results, every step, all inside the timed region, two batches
               in flight (submit step i, wait for step i - 1); the one-synchronous-call-per-step figure
               beside it; `h2d_peak` is a plain pinned cudaMemcpy of the same byte count measured in
               the same run on every rank
  roofline     dominant kernel: FMA-pipe issue slots against the FFMA rate measured in this same run
               (the kernel keeps the CPTs in the instruction stream; HBM view in roofline_hbm)
  dmv_large_batch   BASELINE configs[4]: --dmv-queries device-generated DMV range queries, sharded over
               the N ranks (strong scaling inside this leg), generator + conversion + inference timed
  secondary    BASELINE configs[2]: fan-out weighted expectation factors on the shipped IMDB-1 BN through
               the fused tcgen05 tree kernel (K3), against the 3xTF32 tensor ceiling; every rank runs it
  cpu_baseline the UNMODIFIED reference (baseline/_ref, staged by baseline/stage_reference.py) driven
               as Testing/BN_testing.py:9-46 drives it, single thread (the reference has no parallelism),
               on the first queries of this very batch -- and its probabilities compared with the GPU's
  --impl reference   the same reference in one worker process per host core on the same query stream
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "queries/sec exact tree inference"
UNIT = "queries/s"
KMIN, KMAX = 1, 14
DMV_KMIN, DMV_KMAX = 1, 5
SEED = 0


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="census")
    ap.add_argument("--batch", type=int, default=1_000_000)
    ap.add_argument("--kernel", default="auto", choices=["auto", "generic", "spec"])
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline leg")
    ap.add_argument("--sustained-seconds", type=float, default=2.0)
    ap.add_argument("--dmv-queries", type=float, default=1e9, help="total queries of the DMV large-batch leg (0 = skip)")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--streams", type=int, default=2, help="launch consecutive (independent) steps on this many streams in turn")
    ap.add_argument("--inproc", action="store_true", help="add the in-process multi-GPU leg (one process, all visible GPUs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the probabilities of the last timed step (rank 0) to DIR/probabilities.npy, float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs is available for --impl ours only")
    return args


DUMP_MAX_VALUES = 15_000_000   # 60 MB of float32: larger batches are dumped as a fixed, seeded sample


def dump_outputs(out_dir, probs):
    """Write the results a caller of the timed path receives, so that two builds can be compared value for value."""
    probs = np.asarray(probs, dtype=np.float32)
    if probs.size > DUMP_MAX_VALUES:
        probs = probs[np.sort(np.random.default_rng(SEED).choice(probs.size, DUMP_MAX_VALUES, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "probabilities.npy"), probs)


def load_tree(name):
    from bayescard_b200.loader import TreeModel

    return TreeModel.load(os.path.join(ROOT, "tests", "golden", "models", name + ".npz"))


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1590.0}, "fallback (B200_PROFILING.md)"


def workload_config(model, n_cols, batch, world):
    """The `config` object of BOTH arms (the reference arm runs a bounded sample of this workload per step)."""
    return {"workload": f"{model} Chow-Liu BN ({n_cols} columns), {batch} synthetic range queries per GPU per step, "
                        f"k~U{{{KMIN}..{KMAX}}} constrained columns, seed {SEED}",
            "model": f"Benchmark/{'Census' if model == 'census' else model.upper()}/chow-liu_1.pkl (shipped)",
            "queries_per_gpu_per_step": batch, "n_gpus": world}


# ------------------------------------------------------------------------------------ CPU legs
def queries_as_dicts(tm, desc):
    """RANGE_U8 rows -> the (bins, n_distinct) dicts VariableEliminationJIT.query takes."""
    from bayescard_b200.decode import unpack_ranges

    lo, hi = unpack_ranges(tm, desc)
    out = []
    for i in range(lo.shape[0]):
        q = {}
        for v in range(tm.n_nodes):
            if lo[i, v] > 0 or hi[i, v] < tm.card[v] - 1:
                q[tm.infer_names[v]] = list(range(int(lo[i, v]), int(hi[i, v]) + 1))
        out.append(q)
    return out


def cpu_baseline_port(tm, name, seconds):
    """Oracle port (numpy fp64 restatement without the reference's per-query deepcopy), one core."""
    from bayescard_b200.engine import gen_range_queries_host
    from oracle import bayescard_oracle as O

    n = 2000
    qs = queries_as_dicts(tm, gen_range_queries_host(tm, SEED, 0, n, KMIN, KMAX))
    t = time.perf_counter()
    done = 0
    for q in qs:
        O.ve_query(tm, q, {k: np.ones(len(b)) for k, b in q.items()})
        done += 1
        if time.perf_counter() - t > seconds:
            break
    dt = time.perf_counter() - t
    return {"value": done / dt, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": f"first {done} queries of the {name} bench batch, oracle/bayescard_oracle.py ve_query"}


def cpu_baseline_reference(tm, name, seconds, gpu_probs):
    """The unmodified reference (baseline/_ref), single thread, on the first queries of the bench batch; its
    probabilities are compared with the GPU's for the same queries (``gpu_probs`` = results of batch 0)."""
    from baseline import ref_runner as RR

    if not RR.available():
        return None
    card = [int(c) for c in tm.card]
    names = list(tm.infer_names)
    RR.load_bn(name)
    t_in, res, nq = 0.0, [], 0
    chunk = 250
    t_wall = time.perf_counter()
    while t_in < seconds and nq < len(gpu_probs) and time.perf_counter() - t_wall < 4 * seconds:
        dt, r = RR.run_chunk((name, names, card, SEED, nq, chunk, KMIN, KMAX))
        t_in += dt
        res.append(r)
        nq += chunk
    res = np.concatenate(res)
    lo, hi = RR.gen_ranges(card, SEED, 0, nq, KMIN, KMAX)
    nonempty = ((lo > 0) | (hi < np.asarray(card)[None, :] - 1)).any(axis=1)   # BN.query({}) returns 0 (ExactInference.py:197)
    got = np.asarray(gpu_probs[:nq], dtype=np.float64)
    # fp32 results below the smallest normal number (1.2e-38) are outside the fp32 result format
    chk = nonempty & ((res == 0) | (res > 1e-37))
    rel = np.abs(got[chk] - res[chk]) / np.maximum(np.abs(res[chk]), 1e-300)
    return {"value": nq / t_in, "unit": UNIT, "cores": 1, "kind": "reference",
            "sample": f"first {nq} queries of the {name} bench batch through the unmodified reference staged in baseline/_ref: "
                      f"pickle.load -> init_inference_method('exact-jit') -> BN.query(bins, n_distinct=ones, return_prob=True), "
                      f"time inside BN.query only (Testing/BN_testing.py:27-32), numpy fp64, one thread",
            "rel_err_max_gpu_vs_reference": float(rel.max()) if rel.size else None,
            "queries_compared": int(chk.sum()), "empty_predicate_queries_skipped": int((~nonempty).sum())}


def _ref_worker(conn, model, names, card):
    from baseline import ref_runner as RR

    RR.load_bn(model)
    conn.send("ready")
    prepared = {}
    while True:
        msg = conn.recv()
        if msg[0] == "stop":
            return
        if msg[0] == "prepare":   # untimed: regenerate this worker's slice of the seeded stream
            _, key, first, n = msg
            lo, hi = RR.gen_ranges(card, SEED, first, n, KMIN, KMAX)
            prepared[key] = RR.queries_as_dicts(names, card, lo, hi)
            conn.send("ok")
        elif msg[0] == "run":
            bn = RR.load_bn(model)
            qs = prepared.pop(msg[1])
            t = time.perf_counter()
            for q, nd in qs:
                bn.query(q, n_distinct=nd, return_prob=True)
            conn.send(time.perf_counter() - t)


def run_reference_arm(args):
    """--impl reference: the unmodified reference (baseline/_ref) through its own public API, one worker process per
    host core (the reference itself is single threaded; N independent processes is the most a user can do with it)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp

    from baseline import ref_runner as RR

    tm = load_tree(args.model)
    card, names = [int(c) for c in tm.card], list(tm.infer_names)
    cfg = workload_config(args.model, tm.n_nodes, args.batch, args.gpus)
    if not RR.available():
        print(json.dumps({"impl": "reference", "unavailable": "baseline/_ref not staged (run __graft_entry__.build() where "
                                                              "/root/reference is mounted)"}))
        return
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    per_core = 60
    # single thread first (what the reference is), on a bounded sample
    t1, _ = RR.run_chunk((args.model, names, card, SEED, 0, 400, KMIN, KMAX))
    single = 400 / t1
    ctx = mp.get_context("fork")
    workers = []
    for _ in range(cores):
        a, b = ctx.Pipe()
        p = ctx.Process(target=_ref_worker, args=(b, args.model, names, card), daemon=True)
        p.start()
        workers.append((p, a))
    for _, c in workers:
        c.recv()

    def step(k):
        for w, (_, c) in enumerate(workers):
            c.send(("prepare", k, (k * cores + w) * per_core, per_core))
        for _, c in workers:
            c.recv()
        t = time.perf_counter()
        for _, c in workers:
            c.send(("run", k))
        for _, c in workers:
            c.recv()
        return time.perf_counter() - t

    for k in range(args.warmup):
        step(k)
    t_total = sum(step(args.warmup + k) for k in range(args.steps))
    for p, c in workers:
        c.send(("stop",))
    for p, _ in workers:
        p.join(timeout=5)
    nq = args.steps * cores * per_core
    value = nq / t_total
    sample = (f"{cores * per_core} queries of the workload per step ({per_core} per worker), unmodified reference from baseline/_ref "
              f"(pickle.load -> init_inference_method('exact-jit') -> BN.query(bins, n_distinct=ones, return_prob=True)) in "
              f"{cores} worker processes, wall clock around each step; query dicts prepared outside the timed region")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_total / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": cfg,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "reference", "sample": sample},
            "single_thread": {"value": single, "unit": UNIT, "cores": 1, "sample": "first 400 queries, time inside BN.query"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(index)], stdout=subprocess.PIPE, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def window(self, t0, t1):
        sm, smax, reasons, power = [], None, set(), []
        for t, line in self.rows:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8:
                continue
            try:
                smax = float(f[2])
                if t0 - 0.05 <= t <= t1 + 0.05:
                    sm.append(float(f[1]))
                    power.append(float(f[3]))
                    for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                                         f[4:8]):
                        if val.lower().startswith("active"):
                            reasons.add(name)
            except ValueError:
                continue
        return sm, smax, reasons, power

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons, power = self.window(t0, t1)
        if not sm:  # timed region shorter than the sampling period: use every sample we have
            sm, smax, reasons, power = self.window(-1e30, 1e30)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power) if power else None}


# ------------------------------------------------------------------------------------ our arm: legs
def imdb_expectation_leg(device, peaks, world, barrier, max_over_ranks, n=262144, reps=5):
    """BASELINE.json configs[2] in short (not the headline): fan-out weighted expectation factors on the shipped IMDB-1 BN
    (fractional n_distinct weights on random ranges + fan-out mask) through the fused tensor-core kernel (K3), next to the
    per-model straight-line kernel, and end to end from pinned host memory as WSPARSE runs.  Every rank runs it (weak)."""
    import torch

    from bayescard_b200 import _lib as L
    from bayescard_b200.decode import dense_to_wsparse, unpack_ranges
    from bayescard_b200.engine import DeviceModel
    from oracle import bayescard_oracle as O

    rank = int(os.environ.get("RANK", "0"))
    tm = load_tree("imdb1")
    dm = DeviceModel(tm, device=device, specialize=True)
    stream = torch.cuda.current_stream()
    st = stream.cuda_stream
    ranges = dm.gen_range_queries_host(SEED + 1, rank * n, n, 1, 4)
    lo, hi = unpack_ranges(tm, ranges)
    rng = np.random.default_rng(SEED + 2 + rank)
    W = np.zeros((n, dm.dense_width), dtype=np.float32)
    for v in range(tm.n_nodes):
        c = np.arange(int(tm.card[v]))[None, :]
        sel = (c >= lo[:, v:v + 1]) & (c <= hi[:, v:v + 1])
        con = (lo[:, v] > 0) | (hi[:, v] < int(tm.card[v]) - 1)
        w = np.where(con[:, None], rng.uniform(0.2, 1.0, sel.shape), 1.0)
        o = int(dm.dense_offset[v])
        W[:, o:o + int(tm.card[v])] = sel * w
    fan_nodes = [v for v in range(tm.n_nodes) if tm.infer_names[v] in tm.fanouts and tm.fan_vector(v) is not None]
    mask = np.zeros((n, 1), dtype=np.uint32)
    for v in fan_nodes:
        mask[:, 0] |= (rng.random(n) < 0.4).astype(np.uint32) << np.uint32(v)
    d_w, d_m = torch.from_numpy(W).cuda(device), torch.from_numpy(mask.view(np.int32)).cuda(device)
    out = torch.empty(n, dtype=torch.float32, device=f"cuda:{device}")
    res = {}
    for kname, kernel in (("k_spec", L.KERNEL_SPEC), ("k3_fused_tcgen05", L.KERNEL_FUSED)):
        ts = []
        for r in range(reps + 2):
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            dm.run_device(d_w.data_ptr(), n, L.DESC_DENSE_F32, out.data_ptr(), mask_ptr=d_m.data_ptr(), kernel=kernel, stream=st)
            e1.record(stream)
            torch.cuda.synchronize()
            if r >= 2:
                ts.append(max_over_ranks(e0.elapsed_time(e1)))
        res[kname] = world * n / (float(np.median(ts)) * 1e-3)
    got = out.cpu().numpy().astype(np.float64)
    sub = np.arange(0, n, n // 2048)[:2048]
    Wl = []
    for v in range(tm.n_nodes):
        o = int(dm.dense_offset[v])
        w = W[sub, o:o + int(tm.card[v])].astype(np.float64)
        f = tm.fan_vector(v)
        if f is not None:
            on = ((mask[sub, 0] >> np.uint32(v)) & 1).astype(bool)
            w = np.where(on[:, None], w * f[None, :], w)
        Wl.append(w)
    ref = O.dense_tree(tm, Wl)
    rel = max_over_ranks(float(np.max(np.abs(got[sub] - ref) / np.maximum(np.abs(ref), 1e-300))))
    row_off, words = dense_to_wsparse(tm, W)
    p_off = torch.from_numpy(row_off.view(np.int32)).pin_memory().numpy().view(np.uint32)
    p_words = torch.from_numpy(words.view(np.int32)).pin_memory().numpy().view(np.uint32)
    p_mask = torch.from_numpy(mask.view(np.int32)).pin_memory().numpy().view(np.uint32)
    p_out = torch.empty(n, dtype=torch.float32).pin_memory().numpy()
    dm.run_wsparse_host(p_off, p_words, p_mask, out=p_out)
    barrier()
    t = time.perf_counter()
    for _ in range(3):
        dm.run_wsparse_host(p_off, p_words, p_mask, out=p_out)
    e2e = world * 3 * n / max_over_ranks(time.perf_counter() - t)
    flops = dm.flops_dense
    dm.close()
    k3 = res["k3_fused_tcgen05"]
    # ceiling of an error-compensated 3xTF32 product on the tensor pipe: TF32 dense = bf16 dense / 2, three products
    tf32x3 = peaks["bf16_tflops"] / 2 / 3
    ach = k3 / world * flops / 1e12
    return {"workload": f"shipped IMDB BN #1 (Benchmark/IMDB/1_chow-liu_1.pkl), {n} fan-out weighted expectation factors per GPU "
                        "(DENSE_F32 rows + fan-out mask), device resident",
            "factors_per_s": k3, "factors_per_s_k_spec": res["k_spec"], "kernel": "k3_kernel (tcgen05 3xTF32, messages in TMEM)",
            "flop_per_factor_dense": flops,
            "roofline": {"bound": "tensor", "achieved": ach, "peak": tf32x3, "unit": "TFLOP/s", "frac": ach / tf32x3,
                         "traffic": None, "kernel": "k3_kernel",
                         "peak_source": "MEASURED_PEAKS.json bf16_tflops / 2 (TF32) / 3 (error-compensated 3xTF32 product)",
                         "note": "algorithmic flops = 2 x non-root CPT entries per factor (dense tree); per GPU"},
            "e2e_factors_per_s_wsparse_host": e2e, "e2e_bytes_per_factor": (row_off.nbytes + words.nbytes + mask.nbytes) / n + 4,
            "rel_err_max_vs_fp64_oracle": rel}


def dmv_large_batch_leg(device, world, rank, total, barrier, max_over_ranks, chunk=1 << 22, check=10000):
    """BASELINE.json configs[4] / north_star target: ``total`` device-generated DMV range queries sharded over the ranks
    (contiguous index ranges, no collective): generator -> RANGE_U8 -> BITS -> specialised kernel, fp32 results kept in HBM;
    spot-checked against the fp64 oracle on sampled indices regenerated on the host."""
    import torch

    from bayescard_b200 import _lib as L
    from bayescard_b200.decode import unpack_ranges
    from bayescard_b200.engine import DeviceModel, gen_range_queries_host
    from bayescard_b200.sharding import rank_range
    from oracle import bayescard_oracle as O

    tm = load_tree("dmv")
    dm = DeviceModel(tm, device=device, specialize=True)
    if not dm.has_spec:
        raise SystemExit("specialised DMV kernel unavailable: " + str(dm.spec_error))
    dev = f"cuda:{device}"
    stream = torch.cuda.current_stream()
    st = stream.cuda_stream
    rstride, bstride = dm.desc_stride(L.DESC_RANGE_U8), dm.desc_stride(L.DESC_BITS)
    a, b = rank_range(total, rank, world)
    mine = b - a
    NROT = 8
    ranges = torch.empty((chunk, rstride), dtype=torch.uint8, device=dev)
    bits = [torch.empty((chunk, bstride), dtype=torch.uint8, device=dev) for _ in range(NROT)]
    out = torch.empty(max(mine, 1), dtype=torch.float32, device=dev)

    def full_pass():
        for k, q0 in enumerate(range(a, b, chunk)):
            n = min(chunk, b - q0)
            dm.gen_range_queries_device(SEED, q0, n, DMV_KMIN, DMV_KMAX, ranges.data_ptr(), st)
            dm.convert_device(ranges.data_ptr(), L.DESC_RANGE_U8, bits[k % NROT].data_ptr(), L.DESC_BITS, n, st)
            dm.run_device(bits[k % NROT].data_ptr(), n, L.DESC_BITS, out.data_ptr() + 4 * (q0 - a), kernel=L.KERNEL_SPEC, stream=st)

    def infer_pass():
        for k, q0 in enumerate(range(a, b, chunk)):
            n = min(chunk, b - q0)
            dm.run_device(bits[k % NROT].data_ptr(), n, L.DESC_BITS, out.data_ptr() + 4 * (q0 - a), kernel=L.KERNEL_SPEC, stream=st)

    full_pass()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    full_pass()
    e1.record(stream)
    barrier()
    total_ms = max_over_ranks(e0.elapsed_time(e1))
    checked = out.clone()
    infer_pass()
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record(stream)
    infer_pass()
    e3.record(stream)
    barrier()
    infer_ms = max_over_ranks(e2.elapsed_time(e3))
    rel = 0.0
    if check and mine:
        rng = np.random.default_rng(total + rank)
        idx = np.unique(rng.integers(a, b, size=min(check // world + 1, mine)))
        rows = np.concatenate([gen_range_queries_host(tm, SEED, int(i), 1, DMV_KMIN, DMV_KMAX) for i in idx])
        lo, hi = unpack_ranges(tm, rows)
        ref = O.dense_tree(tm, O.range_weights(tm, lo, hi))
        got = checked[torch.from_numpy(idx - a).to(dev)].cpu().numpy().astype(np.float64)
        rel = float(np.max(np.abs(got - ref) / np.maximum(np.abs(ref), 1e-300)))
    rel = max_over_ranks(rel)
    flop_q = 2 * dm.spec_ffma()
    dm.close()
    del ranges, bits, out, checked
    torch.cuda.empty_cache()
    return {"workload": f"DMV Chow-Liu BN (10 columns), {total} device-generated range queries in total, k~U{{{DMV_KMIN}..{DMV_KMAX}}}, "
                        f"seed {SEED}, sharded over {world} GPU(s) in contiguous index ranges (strong scaling inside this leg)",
            "queries_per_s": total / (total_ms * 1e-3), "seconds": total_ms * 1e-3,
            "includes": "on-device generation (RANGE_U8) + conversion to BITS + inference, chunks of %d" % chunk,
            "queries_per_s_inference_only": total / (infer_ms * 1e-3), "kernel": "bc_spec_bits (DMV image)",
            "fma_issue_slots_per_query": flop_q // 2,
            "checked_indices": int(check), "rel_err_max_vs_fp64_oracle": rel,
            "north_star_target_8gpu_queries_per_s": 1e8}


def h2d_peak_leg(nbytes, device, barrier, max_over_ranks, reps=5):
    """Plain cudaMemcpyAsync of ``nbytes`` from pinned host memory, all ranks at the same time: what the box's PCIe /
    host memory system gives THIS rank while the other ranks copy too -- the ceiling of the e2e number's H2D part."""
    import torch

    h = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    d = torch.empty(nbytes, dtype=torch.uint8, device=f"cuda:{device}")
    d.copy_(h, non_blocking=True)
    torch.cuda.synchronize()
    barrier()
    t = time.perf_counter()
    for _ in range(reps):
        d.copy_(h, non_blocking=True)
    torch.cuda.synchronize()
    dt = max_over_ranks(time.perf_counter() - t)
    return nbytes * reps / dt / 1e9


def inproc_leg(ngpu, B, kernel, reps=5):
    """north_star item 4 as written: ONE process, one host thread + stream set per device (engine.ShardedModel), the PACKED
    batch of ngpu x B queries in one pinned host array, results gathered in one pinned host array.  Same metric and workload
    as `e2e`, beside the one-process-per-GPU (torchrun) number."""
    import torch

    from bayescard_b200.engine import ShardedModel

    tm = load_tree("census")
    sm = ShardedModel(tm, list(range(ngpu)), specialize=True)
    n = ngpu * B
    row_off, entries = sm.replicas[0].gen_sparse_queries_host(SEED, 0, n, KMIN, KMAX)
    klen, blk, pay = sm.replicas[0].pack_sparse(row_off, entries)
    pin = lambda a: torch.from_numpy(a).pin_memory()
    hk, hb, hp = pin(klen), pin(blk.view(np.int32)), pin(pay)
    ho = torch.empty(n, dtype=torch.float32).pin_memory()
    k_np, b_np, p_np, o_np = hk.numpy(), hb.numpy().view(np.uint32), hp.numpy(), ho.numpy()
    for _ in range(2):
        sm.run_packed_host(k_np, b_np, p_np, None, kernel, out=o_np)
    t = time.perf_counter()
    for _ in range(reps):
        sm.run_packed_host(k_np, b_np, p_np, None, kernel, out=o_np)
    dt_sync = time.perf_counter() - t
    first = o_np[:B].copy()
    # two batches in flight per device (double-buffered pinned memory), like the e2e leg
    h2 = [pin(klen), pin(blk.view(np.int32)), pin(pay), torch.empty(n, dtype=torch.float32).pin_memory()]
    bufs = [(k_np, b_np, p_np, o_np), (h2[0].numpy(), h2[1].numpy().view(np.uint32), h2[2].numpy(), h2[3].numpy())]
    for i in range(2):
        sm.wait(sm.submit_packed_host(*bufs[i][:3], out=bufs[i][3], kernel=kernel))
    t = time.perf_counter()
    prev = None
    for i in range(reps):
        tk = sm.submit_packed_host(*bufs[i % 2][:3], out=bufs[i % 2][3], kernel=kernel)
        if prev is not None:
            sm.wait(prev)
        prev = tk
    sm.wait(prev)
    dt = time.perf_counter() - t
    if not (np.array_equal(bufs[1][3][:B], first) and np.array_equal(bufs[0][3][:B], first)):
        raise SystemExit("in-process in-flight results differ from the synchronous call")
    sm.close()
    return {"value": n * reps / dt, "unit": UNIT, "n_gpus": ngpu, "queries_per_call": n,
            "api": "engine.ShardedModel.submit_packed_host / wait: one process, one host thread + stream set per device, two batches in "
                   "flight per device, no collective",
            "one_synchronous_call_per_step": n * reps / dt_sync,
            "h2d_bytes_per_call": int(k_np.nbytes + b_np.nbytes + p_np.nbytes)}, first


def run_ours(args):
    import torch

    from bayescard_b200 import _lib as L
    from bayescard_b200.decode import unpack_ranges
    from bayescard_b200.engine import DeviceModel, launch_count, measure_fp32_peak
    from bayescard_b200.model import Bayescard_BN
    from bayescard_b200.sharding import max_over_ranks as _mor
    from oracle import bayescard_oracle as O  # checker + cpu_baseline leg only

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: bayescard_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        # a CPU-side group for the one wait that must not occupy the GPUs (the in-process multi-GPU leg of rank 0)
        gloo_group = dist.new_group(backend="gloo")
    dev = f"cuda:{local}"
    kernel = {"auto": L.KERNEL_AUTO, "generic": L.KERNEL_GENERIC, "spec": L.KERNEL_SPEC}[args.kernel]

    def max_over_ranks(x):
        return _mor(x, device=dev)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    tm = load_tree(args.model)
    dm = DeviceModel(tm, device=local, specialize=True)
    if kernel != L.KERNEL_GENERIC and not dm.has_spec:
        raise SystemExit("specialised kernel unavailable: " + str(dm.spec_error))
    B = args.batch
    rstride = dm.desc_stride(L.DESC_RANGE_U8)
    spec = kernel != L.KERNEL_GENERIC
    fmt = L.DESC_BITS
    stride = dm.desc_stride(fmt)
    NBUF = 4  # rotate over 4 resident batches: the working set (4 x B x stride) is larger than L2
    stream = torch.cuda.current_stream()
    st = stream.cuda_stream
    # seeded queries are generated on the device as RANGE_U8 rows (the form the host twin of the generator
    # and the oracle read) and converted once, outside the timed region, to the resident BITS rows
    ranges0 = torch.empty((B, rstride), dtype=torch.uint8, device=dev)
    tmp = torch.empty((B, rstride), dtype=torch.uint8, device=dev)
    descs = [torch.empty((B, stride), dtype=torch.uint8, device=dev) for _ in range(NBUF)]
    out = torch.empty(B, dtype=torch.float32, device=dev)
    for b, d in enumerate(descs):
        r = ranges0 if b == 0 else tmp
        dm.gen_range_queries_device(SEED, (rank * NBUF + b) * B, B, KMIN, KMAX, r.data_ptr(), st)
        dm.convert_device(r.data_ptr(), L.DESC_RANGE_U8, d.data_ptr(), fmt, B, st)
    torch.cuda.synchronize()
    del tmp

    # Consecutive steps are independent batches: with --streams 2 they are launched on two streams in turn, so the first CTAs of
    # step k + 1 fill the SMs that the last round of step k leaves idle (a launch of 90 us spends ~8 % of it ramping up and
    # draining: ncu, FMA pipe 80.6 % of active but 72 % of elapsed cycles).  Each stream has its own result buffer.
    n_streams = max(1, int(args.streams))
    side = [torch.cuda.Stream(device=dev) for _ in range(n_streams - 1)]
    lanes = [stream] + side
    outs = [out] + [torch.empty(B, dtype=torch.float32, device=dev) for _ in side]
    join_ev = [torch.cuda.Event() for _ in side]

    def step(k):
        lane = k % n_streams
        dm.run_device(descs[k % NBUF].data_ptr(), B, fmt, outs[lane].data_ptr(), kernel=kernel, stream=lanes[lane].cuda_stream)

    def fork():   # the side streams start after everything recorded on the main stream so far
        if side:
            ev = torch.cuda.Event()
            ev.record(stream)
            for s_ in side:
                s_.wait_event(ev)

    def join():   # ... and the main stream continues after their last launch
        for s_, ev in zip(side, join_ev):
            ev.record(s_)
            stream.wait_event(ev)

    # ---- FP32 peak of this device, measured before the timed region ---------------------------
    fp32_peak, _ = measure_fp32_peak(local)

    # ---- device-resident throughput --------------------------------------------------------
    for k in range(max(args.warmup, 3)):
        step(k)
    torch.cuda.synchronize()
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    time.sleep(0.25 if sampler else 0)
    launches0 = launch_count()
    single_ms = None
    if n_streams > 1:   # the same steps on ONE stream, for the record (every launch waits for the one before to drain)
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        a0.record(stream)
        for k in range(args.steps):
            dm.run_device(descs[k % NBUF].data_ptr(), B, fmt, out.data_ptr(), kernel=kernel, stream=st)
        a1.record(stream)
        barrier()
        single_ms = max_over_ranks(a0.elapsed_time(a1))
        launches0 = launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t0 = time.perf_counter()
    e0.record(stream)
    fork()
    for k in range(args.steps):
        step(k)
    join()
    e1.record(stream)
    barrier()
    t1 = time.perf_counter()
    launches = launch_count() - launches0
    ms = max_over_ranks(e0.elapsed_time(e1))
    value = world * B * args.steps / (ms * 1e-3)
    if args.dump_outputs and rank == 0:   # copied now: the legs below reuse the result buffers
        dump_outputs(args.dump_outputs, outs[(args.steps - 1) % n_streams].cpu().numpy())

    # ---- sustained: the same launch back to back for >= sustained_seconds ----------------------------
    sustained = None
    if args.sustained_seconds > 0:
        n_sus = max(args.steps, int(args.sustained_seconds / (ms * 1e-3 / args.steps)) + 1)
        barrier()
        ts0 = time.perf_counter()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record(stream)
        fork()
        for k in range(n_sus):
            step(k)
        join()
        s1.record(stream)
        barrier()
        ts1 = time.perf_counter()
        sus_ms = max_over_ranks(s0.elapsed_time(s1))
        sm, _, reasons, power = sampler.window(ts0 + 0.3, ts1) if sampler else ([], None, set(), [])
        sustained = {"value": world * B * n_sus / (sus_ms * 1e-3), "unit": UNIT, "steps": n_sus, "seconds": sus_ms * 1e-3,
                     "sm_mhz_median": float(np.median(sm)) if sm else None, "power_w_max": max(power) if power else None,
                     "reasons": sorted(reasons)}

    # ---- end to end through the host-buffer C-ABI call ---------------------------------------------
    # the same B queries as SPARSE (CSR) entries in pinned host memory -- what a caller holding the
    # reference's sparse {column: bins} dicts would hand over
    # -- as PACKED entries (bit-packed {column, lo, hi}: the densest wire form, 17 B per Census query; the link is PCIe)
    row_off_np, entries_np = dm.gen_sparse_queries_host(SEED, rank * NBUF * B, B, KMIN, KMAX)
    klen_np, blk_np, pay_np = dm.pack_sparse(row_off_np, entries_np)   # host-side packing: outside the timed region, like the CSR
    pin = lambda a: torch.from_numpy(a).pin_memory()
    h_klen, h_blk, h_pay = pin(klen_np), pin(blk_np.view(np.int32)), pin(pay_np)
    h_out = torch.empty(B, dtype=torch.float32).pin_memory()
    hk, hb, hp, ho = h_klen.numpy(), h_blk.numpy().view(np.uint32), h_pay.numpy(), h_out.numpy()
    h2d_bytes = int(hk.nbytes + hb.nbytes + hp.nbytes)
    e2e_steps = max(3, min(args.steps, 10))
    for _ in range(2):
        dm.run_packed_host(hk, hb, hp, None, kernel, out=ho)
    e2e_first = ho.copy()
    # (a) one synchronous call per step: copy in, expand, infer, copy out, return
    barrier()
    te = time.perf_counter()
    for _ in range(e2e_steps):
        dm.run_packed_host(hk, hb, hp, None, kernel, out=ho)
    torch.cuda.synchronize()
    e2e_sync_s = max_over_ranks(time.perf_counter() - te)
    e2e_sync_value = world * B * e2e_steps / e2e_sync_s
    # (b) the serving loop: two batches in flight (submit step i, then wait for step i - 1 and read its results), double-buffered
    # pinned host memory.  Every step still copies its own inputs host -> device and its own results device -> host inside the
    # timed region; the copy of step i runs under the kernels and the read-back of step i - 1.
    bufs = [(hk, hb, hp, ho)]
    h2 = [pin(klen_np), pin(blk_np.view(np.int32)), pin(pay_np), torch.empty(B, dtype=torch.float32).pin_memory()]
    bufs.append((h2[0].numpy(), h2[1].numpy().view(np.uint32), h2[2].numpy(), h2[3].numpy()))
    for o in (bufs[0][3], bufs[1][3]):
        o[:] = -1.0
    checksum = 0.0
    for it in range(2):   # warm-up of the second buffer set
        dm.wait(dm.submit_packed_host(*bufs[it % 2][:3], out=bufs[it % 2][3], kernel=kernel))
    barrier()
    te = time.perf_counter()
    prev = None
    for it in range(e2e_steps):
        k_, b_, p_, o_ = bufs[it % 2]
        t_ = dm.submit_packed_host(k_, b_, p_, out=o_, kernel=kernel)
        if prev is not None:
            dm.wait(prev[0])
            checksum += float(prev[1][0]) + float(prev[1][-1])   # the step's results are read on the host
        prev = (t_, o_)
    dm.wait(prev[0])
    checksum += float(prev[1][0]) + float(prev[1][-1])
    e2e_s = max_over_ranks(time.perf_counter() - te)
    e2e_value = world * B * e2e_steps / e2e_s
    if not (np.array_equal(bufs[0][3], e2e_first) and np.array_equal(bufs[1][3], e2e_first)):
        raise SystemExit("results of the in-flight submissions differ from the synchronous call")
    # the round-1 wire format (SPARSE CSR, 4 B row offset + 4 B per entry) through its own entry point, for reference
    h_off, h_ent = pin(row_off_np.view(np.int32)), pin(entries_np.view(np.int32))
    ho_np, he_np = h_off.numpy().view(np.uint32), h_ent.numpy().view(np.uint32)
    dm.run_sparse_host(ho_np, he_np, None, kernel, out=ho)
    if not np.array_equal(ho, e2e_first):
        raise SystemExit("PACKED and SPARSE host paths disagree")
    barrier()
    te = time.perf_counter()
    for _ in range(3):
        dm.run_sparse_host(ho_np, he_np, None, kernel, out=ho)
    torch.cuda.synchronize()
    e2e_csr_value = world * B * 3 / max_over_ranks(time.perf_counter() - te)
    csr_bytes = int(ho_np.nbytes + he_np.nbytes)
    h2d_peak = h2d_peak_leg(h2d_bytes, local, barrier, max_over_ranks)
    clocks = sampler.stop(t0, t1) if sampler else None

    # ---- the other BASELINE configs, at every N ------------------------------------------------------------
    peaks, peak_src = measured_peaks()
    dmv_leg = None
    if args.dmv_queries > 0:
        dmv_leg = dmv_large_batch_leg(local, world, rank, int(args.dmv_queries), barrier, max_over_ranks)
    secondary = None if args.no_secondary else imdb_expectation_leg(local, peaks, world, barrier, max_over_ranks)

    if rank != 0:
        if dist is not None:
            dist.barrier(group=gloo_group)   # rank 0 runs the in-process multi-GPU leg on all N devices meanwhile: wait on the CPU
            dist.barrier()
            dist.destroy_process_group()
        return
    inproc = None
    n_inproc = world if world > 1 else (torch.cuda.device_count() if args.inproc else 0)
    if n_inproc > 1:
        inproc, inproc_first = inproc_leg(n_inproc, B, kernel)
        if not np.array_equal(inproc_first, e2e_first) and world == 1:
            raise SystemExit("in-process multi-GPU results differ from the single-GPU results")
    if dist is not None:
        dist.barrier(group=gloo_group)

    # ---- parity of this very batch against the fp64 oracle (sub-sample) ------------------------
    rng = np.random.default_rng(0)
    idx = np.sort(rng.choice(B, size=min(B, 10000), replace=False))
    dm.run_device(descs[0].data_ptr(), B, fmt, out.data_ptr(), kernel=kernel, stream=st)
    torch.cuda.synchronize()
    full = out.cpu().numpy()
    if not np.array_equal(full, e2e_first):
        raise SystemExit("end-to-end (PACKED host) results differ from the device-resident (BITS) results")
    got = full[idx].astype(np.float64)
    lo, hi = unpack_ranges(tm, ranges0.cpu().numpy()[idx])
    ref = O.dense_tree(tm, O.range_weights(tm, lo, hi))
    ok = (ref == 0) | (ref > 1e-37)   # below the fp32 normal range the fp32 result format itself ends
    rel_err = float(np.max(np.abs(got[ok] - ref[ok]) / np.maximum(np.abs(ref[ok]), 1e-300)))

    # ---- p50 latency of the scalar drop-in call (B = 1, decode included) ----------------------
    bn = Bayescard_BN(tm, device=local, infer_algo="exact-jit")
    bn.init_inference_method()
    qd = queries_as_dicts(tm, dm.gen_range_queries_host(SEED, 0, 300, KMIN, KMAX))
    raw = []
    inv = {n: {b: v for v, b in tm.encoding[n].items()} for n in tm.infer_names if tm.encoding.get(n)}
    for q in qd:
        raw.append({k: [inv[k][b] for b in bins] for k, bins in q.items()})
    lat = []
    for q in raw:
        if not q:
            continue
        tq = time.perf_counter()
        bn.query(q)
        lat.append(time.perf_counter() - tq)
    p50_us = float(np.median(lat[20:]) * 1e6)
    bn.close()

    # ---- roofline of the dominant kernel ------------------------------------------------------
    slots_q = dm.spec_ffma() if spec else dm.flops_dense // 2
    flop_q = 2 * slots_q
    kernel_s = ms * 1e-3 / args.steps
    achieved_tf = flop_q * B / kernel_s / 1e12
    bytes_q = stride + 4
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    kname = "bc_spec_bits" if spec else "k1_kernel"
    if os.path.exists(tpath):  # dram__bytes_read+write per query of this kernel, from the committed ncu capture
        with open(tpath) as f:
            per_q = json.load(f).get(f"{args.model}:{kname}")
        traffic = per_q * B if per_q is not None else None
    roof = {"bound": "fp32", "achieved": achieved_tf, "peak": fp32_peak, "unit": "TFLOP/s",
            "frac": achieved_tf / fp32_peak if fp32_peak else None, "traffic": traffic,
            "kernel": kname, "what": "FMA-pipe issue-slot fraction",
            "fma_issue_slots_per_query": slots_q, "flop_per_query_counted": flop_q, "flop_per_query_dense": dm.flops_dense,
            "peak_source": "FFMA micro-benchmark (bc_measure_fp32_peak) in this run",
            "launch_overlap": (f"consecutive steps (independent batches) are launched on {n_streams} streams in turn: the first CTAs of a launch fill the "
                               "SMs the last round of the launch before leaves idle; achieved = flops of the K steps / time of the timed region"
                               if n_streams > 1 else "one stream"),
            "single_stream": ({"value": world * B * args.steps / (single_ms * 1e-3), "ms_per_step": single_ms / args.steps,
                               "frac": (flop_q * B / (single_ms * 1e-3 / args.steps) / 1e12 / fp32_peak) if fp32_peak else None}
                              if single_ms else None),
            "note": "achieved = FMA-pipe instructions the generated kernel contains per query (one per non-zero CPT entry: "
                    "FFMA, or a predicated FADD / seed FMUL that occupies the same pipe slot) x 2 flop x q/s; predicated-off "
                    "instructions still occupy their issue slot, so this is pipe utilisation, not useful flops; exact zeros "
                    "of the CPTs emit nothing"}
    roof_hbm = {"bound": "hbm", "achieved": bytes_q * B / kernel_s / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": bytes_q * B / kernel_s / 1e9 / peaks["hbm_gbs"], "bytes_per_query": bytes_q,
                "peak_source": f"MEASURED_PEAKS.json ({peak_src})"}

    cpu_ref = cpu_baseline_reference(tm, args.model, args.cpu_seconds, full) if args.model in ("census", "dmv") else None
    cpu_port = cpu_baseline_port(tm, args.model, min(args.cpu_seconds, 6.0))
    cpu = cpu_ref if cpu_ref is not None else cpu_port

    cfg = workload_config(args.model, tm.n_nodes, B, world)
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg,
            "path": {"descriptor": "BITS (resident) / PACKED bit-packed entries (e2e)", "bytes_per_query": bytes_q, "streams": n_streams,
                     "l2": f"inputs rotate over {NBUF} resident batches = {NBUF * B * stride / 1e6:.0f} MB > 126 MB L2",
                     "kernel": roof["kernel"], "parallelism": f"replica x{world}, batch sharded, no collective"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": B * 4,
                    "steps": e2e_steps,
                    "api": "bc_query_batch_packed_host_submit + bc_pipe_wait: two batches in flight (pinned host PACKED entries -> H2D -> expand -> "
                           "infer -> D2H per step, the copy of step i under the kernels and the read-back of step i - 1)",
                    "one_synchronous_call_per_step": {"value": e2e_sync_value, "api": "bc_query_batch_packed_host"},
                    "bytes_per_query_h2d": h2d_bytes / B,
                    "sparse_csr": {"value": e2e_csr_value, "h2d_bytes_per_step": csr_bytes,
                                   "api": "bc_query_batch_sparse_host (round-1 wire format)"},
                    "h2d_gbs_per_rank": h2d_bytes * e2e_steps / e2e_s / 1e9,
                    "h2d_peak_gbs_per_rank": h2d_peak,
                    "h2d_peak_note": "plain pinned cudaMemcpy of the same byte count, all ranks copying at once, same run"},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "roofline_hbm": roof_hbm,
            "cpu_baseline": cpu, "cpu_baseline_port": cpu_port,
            "rel_err_max_vs_fp64_oracle": rel_err, "p50_latency_us_scalar_query": p50_us,
            "fp32_peak_tflops_measured": fp32_peak}
    if inproc is not None:
        line["e2e_inproc"] = inproc
    if sustained is not None:
        line["sustained"] = sustained
    if dmv_leg is not None:
        line["dmv_large_batch"] = dmv_leg
    if secondary is not None:
        line["secondary"] = secondary
    print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.gpus > 1 and "RANK" not in os.environ:
        # launched by hand: re-exec under torchrun, one rank per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29517", os.path.abspath(__file__)] + sys.argv[1:]
        os.execv(sys.executable, cmd)
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
