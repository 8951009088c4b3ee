"""fp64 helpers for GROUP BY over fan-out expectations -- TEST INFRASTRUCTURE ONLY, like ``groupby_oracle.py``.

The reference of ``bc_expectation_marginal_batch`` is ``groupby_oracle.marginal`` with the fan-out vectors multiplied into W:
``oracle.dense_weights(m, query, n_distinct, fanout_attrs)`` (a predicate on a column wins over its fan-out vector, as
``PredicateCompiler.pack`` clears the mask bit of a predicated column), or ``oracle.range_weights(m, lo, hi, fan_mask)`` for
raw mask rows (bit v multiplies w_v by fanouts[v] whatever the predicate).  ``interpret_masked`` runs one thread of a
generated entry point on the host with a mask row supplied.
"""
from __future__ import annotations

import re
import struct

import numpy as np

import groupby_oracle as GO
from oracle import bayescard_oracle as O


def fan_nodes(m):
    """Nodes with a fan-out vector (the bits a mask can set)."""
    return [v for v in range(m.n_nodes) if m.fan_vector(v) is not None]


def masked_marginal(m, decoded, fanouts, t):
    """``[len(decoded), card_t]`` fp64: the per-state mass of node t under each decoded query weighted by its fan-outs."""
    per = [O.dense_weights(m, b, w, f) for (b, w), f in zip(decoded, fanouts)]
    W = [np.stack([p[v] for p in per]) for v in range(m.n_nodes)]
    return GO.marginal(m, W, t)


def interpret_masked(src, entry, row, mask=None):
    """``groupby_oracle.interpret`` with the fan-out mask row ``mask`` (uint32 words, or ``None`` for a NULL pointer): the
    mask loads of the entry's prologue read it, and ``@%pfm`` is whether it is non-NULL."""
    body = src.split(".visible .entry " + entry + "(")[1].split(".visible .entry")[0]
    lines = [ln.strip() for ln in body.split("\n")]
    start = next(i for i, ln in enumerate(lines) if ln.startswith("mad.lo.u64 %rrow"))
    row = np.frombuffer(bytes(row), dtype=np.uint8)
    words = np.zeros(0, dtype=np.uint32) if mask is None else np.asarray(mask, dtype=np.uint32).reshape(-1)
    regs, out = {"%pfm": mask is not None}, {}

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
        elif op == "ld.global.nc.u32":   # a mask word
            dst, off = re.match(r"(\S+), \[%rtmp\+(\d+)\]", rest).groups()
            regs[dst] = int(words[int(off) // 4])
        elif op == "mov.u32":
            dst, src_ = [x.strip() for x in rest.split(",")]
            regs[dst] = int(val(src_))
        elif op == "st.global.f32":
            off, r = re.match(r"\[%rtmp(?:\+(\d+))?\], (\S+)", rest).groups()
            out[int(off or 0) // 4] = regs[r]
        elif op in ("shl.b64", "add.u64", "mul.lo.u64", "mad.lo.u64"):
            continue   # address arithmetic
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


def per_value_sql(sql, value):
    """The job-light text of one group: ``SELECT x.col, COUNT(*) ... GROUP BY x.col`` -> ``SELECT COUNT(*) ... AND x.col=v``
    (``None`` for a value the grammar cannot write)."""
    m = re.match(r"(?is)^\s*select\s+.*?\s+from\s+(.*?)\s+group\s+by\s+(\w+\.\w+)\s*;?\s*$", sql)
    v = float(value)
    if not v.is_integer():
        # job-light's grammar reads "x.col=1992.78" as a join condition: such a value (the null marker of a column) has no text
        return None
    return f"SELECT COUNT(*) FROM {m.group(1)} AND {m.group(2)}={int(v)}"
