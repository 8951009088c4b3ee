"""Numpy fp64 reference for GROUP BY one column -- TEST INFRASTRUCTURE ONLY, like ``oracle/bayescard_oracle.py``.

``marginal(m, W, t)`` is the checker of ``bc_marginal_batch``: ``oracle.dense_tree`` evaluated once per state b of the
target node t with ``W[t]`` masked to the one-hot of b, i.e. ``out[b] = sum_{x : x_t = b} prod_v w_v[x_v] T_v[x_v, x_pa(v)]``.
``brute_force`` enumerates every joint state of a tiny tree, the independent check of ``marginal`` itself.
The product package never imports this module.
"""
from __future__ import annotations

import itertools

import numpy as np

from oracle import bayescard_oracle as O


def marginal(m, W, t):
    """``W``: per node ``[card_v]`` or ``[B, card_v]`` weights.  Returns ``[card_t]`` or ``[B, card_t]`` (fp64)."""
    card = int(m.card[t])
    cols = []
    for b in range(card):
        Wb = list(W)
        onehot = np.zeros(card)
        onehot[b] = 1.0
        Wb[t] = np.asarray(W[t], dtype=np.float64) * onehot
        cols.append(O.dense_tree(m, Wb))
    return np.stack(cols, axis=-1)


def brute_force(m, W, t):
    """Sum over every joint assignment of a tiny tree (no message passing): ``[card_t]`` for per-node ``[card_v]`` W."""
    n = len(m.infer_names)
    out = np.zeros(int(m.card[t]))
    for x in itertools.product(*[range(int(c)) for c in m.card]):
        p = 1.0
        for v in range(n):
            T = np.asarray(m.cpts[v], dtype=np.float64)
            p *= W[v][x[v]] * (T.reshape(-1)[x[v]] if v == 0 else T[x[v], x[int(m.parent[v])]])
        out[x[t]] += p
    return out


def tree_targets(m):
    """The targets the GROUP BY tests and the benchmark use on a model: root, deepest node, widest column, first leaf."""
    n = len(m.infer_names)
    depth = [0] * n
    for v in range(1, n):
        depth[v] = depth[int(m.parent[v])] + 1
    inner = set(int(p) for p in m.parent[1:])
    leaf = next(v for v in range(n) if v not in inner)
    return {"root": 0, "deepest": int(np.argmax(depth)), "widest": int(np.argmax(m.card)), "leaf": leaf}


def assemble_marginals(tm, nodes, cache_dir, workers=None):
    """``ptxas -arch=sm_100a`` the marginal modules of ``nodes`` into ``cache_dir/marg_<hash>.cubin`` in parallel (the
    files ``bc_model_specialize_marginal`` loads before it falls back to the driver JIT, which compiles one at a time)."""
    import os
    import subprocess
    import tempfile
    from concurrent.futures import ThreadPoolExecutor

    from bayescard_b200 import _lib as L
    from bayescard_b200.engine import DeviceModel

    dm = DeviceModel(tm, device=-1, specialize=False)
    jobs = [(os.path.join(cache_dir, "marg_%016x.cubin" % dm.marginal_hash(v)), dm.marginal_source(v)) for v in nodes]
    dm.close()
    os.makedirs(cache_dir, exist_ok=True)

    def one(job):
        out, src = job
        if os.path.exists(out):
            return
        with tempfile.TemporaryDirectory() as td:
            ptx = os.path.join(td, "marg.ptx")
            with open(ptx, "w") as f:
                f.write(src)
            res = subprocess.run([os.environ.get("PTXAS", "/usr/local/cuda/bin/ptxas"), "-arch=sm_100a", "-O3", "-o", out + ".tmp", ptx],
                                 capture_output=True, text=True)
            if res.returncode != 0:
                raise L.BayesCardError("ptxas failed for a marginal module:\n" + res.stderr[-2000:])
            os.replace(out + ".tmp", out)

    with ThreadPoolExecutor(max_workers=workers or os.cpu_count() or 4) as ex:
        list(ex.map(one, jobs))


def interpret(src, entry, row):
    """Run one thread of a generated marginal / spec entry point on ONE descriptor row (bytes) on the host: the
    straight-line body and the stores, in fp32 (FMA with one rounding).  Checks the code generator's arithmetic without a
    GPU; it knows only the instructions the generator emits inside the loop body."""
    import re
    import struct

    body = src.split(".visible .entry " + entry + "(")[1].split(".visible .entry")[0]
    lines = [ln.strip() for ln in body.split("\n")]
    start = next(i for i, ln in enumerate(lines) if ln.startswith("mad.lo.u64 %rrow"))
    row = np.frombuffer(bytes(row), dtype=np.uint8)
    regs, out = {}, {}

    def val(x):
        if x.startswith("0f"):
            return np.frombuffer(struct.pack("<I", int(x[2:], 16)), dtype=np.float32)[0]
        return int(x) if re.fullmatch(r"-?\d+", x) else regs[x]

    for ln in lines[start + 1:]:
        if not ln or ln.startswith("//"):
            continue
        if ln.startswith("bra LOOP"):
            break
        if ln.startswith("@"):
            pred, ln = ln.split(" ", 1)
            if pred != "@%pvalid" and not regs[pred[1:]]:
                continue
        op, rest = ln.rstrip(";").split(" ", 1)
        if op.startswith("ld.global.nc.v4"):
            dst, off = re.match(r"\{(.*)\}, \[%rrow\+(\d+)\]", rest).groups()
            vals = np.frombuffer(row[int(off):int(off) + 16].tobytes(), dtype=np.float32 if op.endswith("f32") else np.uint32)
            for r, v in zip(dst.split(","), vals):
                regs[r.strip()] = v
        elif op == "st.global.f32":
            off, r = re.match(r"\[%rtmp(?:\+(\d+))?\], (\S+)", rest).groups()
            out[int(off or 0) // 4] = regs[r]
        elif op in ("shl.b64", "add.u64", "mul.lo.u64"):
            continue   # output address arithmetic
        else:
            a = [x.strip() for x in rest.split(",")]
            if op == "and.b32":
                regs[a[0]] = int(val(a[1])) & int(val(a[2]))
            elif op == "setp.ne.u32":
                regs[a[0]] = int(val(a[1])) != int(val(a[2]))
            elif op == "selp.f32":
                regs[a[0]] = np.float32(val(a[1]) if regs[a[3]] else val(a[2]))
            elif op == "mul.f32":
                regs[a[0]] = np.float32(np.float32(val(a[1])) * np.float32(val(a[2])))
            elif op == "add.f32":
                regs[a[0]] = np.float32(np.float32(val(a[1])) + np.float32(val(a[2])))
            elif op == "fma.rn.f32":
                regs[a[0]] = np.float32(np.float64(val(a[1])) * np.float64(val(a[2])) + np.float64(val(a[3])))
            elif op == "mov.f32":
                regs[a[0]] = np.float32(val(a[1]))
            else:
                raise ValueError("instruction outside the generator's body: " + ln)
    return np.asarray([out[i] for i in range(len(out))], dtype=np.float64)
