"""Predicate compiler: raw predicates -> (bins, weights) -> packed per-query descriptors.

Stage 1 (:meth:`PredicateCompiler.decode`) has the semantics of ``Bayescard_BN.query_decoding``
(reference ``Models/Bayescard_BN.py:279-325``) with its helpers ``realign`` (``:53-72``),
``continuous_range_map`` (``:180-239``), ``apply_encoding_to_value`` / ``apply_ndistinct_to_value``
(``Models/BN_single_model.py:98-139``), quirks included (SURVEY.md section 8a rows 4-6):

* an unknown scalar, a column without an encoding or an empty value list make the whole query
  undecodable (``(None, None)``, estimate 0); unknown members of a value LIST are silently dropped;
* several values falling into one bin add their ``n_in_bin`` fractions, capped at 1;
* a ``(lo, hi)`` tuple on a categorical column enumerates the ORIGINAL values inside the range, minus
  the column's null value;
* continuous ranges are clamped to the column domain, a point ``x`` becomes ``[x-eps, x+eps]`` (times the
  hard-coded ``n_distinct_mapping`` multiplier), and the bin walk stops expanding on one side as soon
  as the other side reaches the edge of the domain.

Unlike the reference nothing is mutated: ``decode`` returns fresh dicts.

Stage 2 (:meth:`PredicateCompiler.pack`) writes descriptors for the CUDA kernels: a ``BITS`` row (one
bit per column state) when every weight of a query is 1 -- ranges, equality and IN lists, 96 % of the
shipped DMV predicates -- and the dense fp32 weight row otherwise; fan-out columns of ``expectation``
become a bitmask (a predicate on the same column clears the bit, because the reference tests the
predicate first: ``Pgmpy/inference/ExactInference.py:209,:238``).  :meth:`pack_sparse` writes the
compact CSR form the host-buffer entry point ships over PCIe.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

from . import _lib as L
from .loader import TreeModel

Decoded = Tuple[Optional[Dict[str, List[int]]], Optional[Dict[str, np.ndarray]]]


class _Column:
    """Per-column lookup tables built once per model."""

    __slots__ = ("name", "kind", "enc", "pair", "num_vals", "num_bins", "num_wts", "null", "has_null",
                 "edges", "domain", "nd_map", "card")

    def __init__(self, tm: TreeModel, name: str):
        self.name = name
        self.kind = tm.attr_type.get(name)
        self.enc = tm.encoding.get(name) if name in tm.encoding else None
        self.card = int(tm.card[tm.index_of(name)]) if name in tm._index else None
        nib = tm.n_in_bin.get(name) if name in tm.n_in_bin else None
        has_nib = name in tm.n_in_bin
        # value -> (bin, weight)
        self.pair = {}
        if self.enc is not None:
            for val, b in self.enc.items():
                w = 1
                if has_nib and nib is not None and b in nib:
                    t = nib[b]
                    if isinstance(t, int):
                        w = 1 / t
                    elif val in t:
                        w = t[val]
                self.pair[val] = (b, w)
        nv = tm.null_values
        self.has_null = not (nv is None or len(nv) == 0 or name not in nv)
        self.null = nv[name] if self.has_null else None
        # numeric categorical columns: arrays in encoding (dict) order for vectorised range lookups
        self.num_vals = self.num_bins = self.num_wts = None
        if self.enc is not None and len(self.enc) and all(
                isinstance(k, (int, float)) and not isinstance(k, bool) for k in self.enc):
            keys = list(self.enc.keys())
            self.num_vals = np.asarray(keys, dtype=np.float64)
            self.num_bins = np.asarray([self.pair[k][0] for k in keys], dtype=np.int64)
            self.num_wts = np.asarray([self.pair[k][1] for k in keys], dtype=np.float64)
        self.edges = tm.mapping.get(name) if name in tm.mapping else None
        self.domain = tm.domain.get(name)
        self.nd_map = tm.n_distinct_mapping.get(name) if name in tm.n_distinct_mapping else None


def _merge(bins: Sequence, wts: Sequence) -> Tuple[List[int], np.ndarray]:
    """realign: drop None, first-occurrence order, duplicate bins add up capped at 1."""
    pos: Dict[int, int] = {}
    out_b: List[int] = []
    out_w: List[float] = []
    for b, w in zip(bins, wts):
        if b is None:
            continue
        j = pos.get(b)
        if j is None:
            pos[b] = len(out_b)
            out_b.append(int(b))
            out_w.append(w)
        else:
            out_w[j] = min(out_w[j] + w, 1)
    return out_b, np.asarray(out_w, dtype=np.float64)


class PredicateCompiler:
    def __init__(self, tm: TreeModel):
        self.tm = tm
        self.cols: Dict[str, _Column] = {n: _Column(tm, n) for n in tm.node_names}

    # ------------------------------------------------------------------ stage 1
    def _continuous(self, col: _Column, lo: float, hi: float) -> Tuple[List[int], np.ndarray]:
        edges = col.edges
        n = len(edges)

        def cover(k: int) -> float:
            tl, tr = edges[k]
            if lo >= tr or hi <= tl:
                return 0
            if hi > tr:
                return 1 if lo < tl else (tr - lo) / (tr - tl)
            return (hi - lo) / (tr - tl) if lo > tl else (hi - tl) / (tr - tl)

        # bisection for any bin overlapping [lo, hi]; same probe sequence as the reference
        i, j = 0, n
        while i != j:
            mid = int(i + (j - i) / 2)
            tl, tr = edges[mid]
            if lo >= tr:
                if i == mid:  # the reference recurses forever here; cannot happen for lo inside the domain
                    break
                i = mid
            elif hi <= tl:
                j = mid
            else:
                i = j = mid
        down, up = i, i + 1
        more_down = more_up = True
        bins: List[int] = []
        cov: List[float] = []
        while down >= 0 and up < n and (more_down or more_up):
            if more_down:
                c = cover(down)
                if c != 0:
                    bins.append(down)
                    cov.append(c)
                    down -= 1
                else:
                    more_down = False
            if more_up:
                c = cover(up)
                if c != 0:
                    bins.append(up)
                    cov.append(c)
                    up += 1
                else:
                    more_up = False
        return bins, np.asarray(cov, dtype=np.float64)

    _MEMO_MAX = 1 << 16

    def decode(self, query: dict, coverage: Optional[dict] = None, epsilon: float = 0.5) -> Decoded:
        """``query_decoding`` (Models/Bayescard_BN.py:279-325).  Every column decodes independently of the others, so the
        result per (column, predicate value) is memoised: serving workloads repeat the same few hundred predicates.  The
        cached weight arrays are read-only and shared between results; the bin lists are copied."""
        bins_out: Dict[str, List[int]] = {}
        wts_out: Dict[str, np.ndarray] = {}
        memo = self.__dict__.setdefault("_memo", {})
        for attr, val in query.items():
            key = None
            if coverage is None:
                try:
                    key = (attr, tuple(val) if type(val) == list else val, type(val) == list, epsilon)
                    hit = memo.get(key)
                except TypeError:   # unhashable value (an ndarray, ...): decode without the memo
                    key, hit = None, None
                if hit is not None:
                    if hit is False:
                        return None, None
                    bins_out[attr], wts_out[attr] = list(hit[0]), hit[1]
                    continue
            one_b, one_w = self._decode_one({attr: val}, coverage, epsilon)
            if key is not None and len(memo) < self._MEMO_MAX:
                if one_b is None:
                    memo[key] = False
                else:
                    w = np.asarray(one_w[attr])
                    w.setflags(write=False)
                    memo[key] = (tuple(one_b[attr]), w)
            if one_b is None:
                return None, None
            bins_out[attr], wts_out[attr] = one_b[attr], one_w[attr]
        return bins_out, wts_out

    def _decode_one(self, query: dict, coverage: Optional[dict] = None, epsilon: float = 0.5) -> Decoded:
        bins_out: Dict[str, List[int]] = {}
        wts_out: Dict[str, np.ndarray] = {}
        for attr, val in query.items():
            col = self.cols.get(attr)
            if col is None or col.kind is None:
                raise KeyError(attr)
            if col.kind == "continuous":
                if coverage is not None:
                    bins_out[attr] = list(val) if isinstance(val, (list, tuple, np.ndarray)) else [val]
                    wts_out[attr] = np.asarray(coverage[attr], dtype=np.float64)
                    continue
                mult = None
                if type(val) == tuple:
                    lo = max(col.domain[0], val[0])
                    hi = min(col.domain[1], val[1])
                else:
                    lo, hi = val - epsilon, val + epsilon
                    if col.nd_map is not None and val in col.nd_map:
                        mult = col.nd_map[val]
                if lo > hi:
                    return None, None
                b, w = self._continuous(col, lo, hi)
                if mult is not None:
                    w = w * mult
                bins_out[attr], wts_out[attr] = b, w
            elif type(val) == tuple:
                lo, hi = val[0], val[1]
                if col.num_vals is not None and isinstance(lo, (int, float)) and isinstance(hi, (int, float)):
                    keep = (col.num_vals >= lo) & (col.num_vals <= hi)
                    if col.has_null:
                        keep &= col.num_vals != col.null
                    sel_b, sel_w = col.num_bins[keep], col.num_wts[keep]
                else:
                    sel_b, sel_w = [], []
                    for v, (b, w) in col.pair.items():
                        if col.has_null and v == col.null:
                            continue
                        if lo <= v <= hi:
                            sel_b.append(b)
                            sel_w.append(w)
                if len(sel_b) == 0:
                    return None, None
                bins_out[attr], wts_out[attr] = _merge(sel_b, sel_w)
            else:
                if col.enc is None:
                    return None, None
                if type(val) == list:
                    if len(val) == 0:
                        return None, None
                    pairs = [col.pair.get(v, (None, 1)) for v in val]
                    bins_out[attr], wts_out[attr] = _merge([p[0] for p in pairs], [p[1] for p in pairs])
                else:
                    p = col.pair.get(val)
                    if p is None:
                        return None, None
                    bins_out[attr], wts_out[attr] = [int(p[0])], np.asarray([p[1]], dtype=np.float64)
        return bins_out, wts_out

    def select_values(self, attr: str, val) -> Optional[np.ndarray]:
        """Which original values of categorical column ``attr`` a predicate value selects, by ``decode``'s rules: a bool
        mask over the encoding's keys in encoding order, or ``None`` where ``decode`` finds the predicate undecodable.
        A scalar selects itself; a list its known members (unknown ones are dropped); a ``(lo, hi)`` tuple every value
        inside the range except the column's null value."""
        col = self.cols[attr]
        if col.enc is None:
            return None
        keys = list(col.pair)
        if type(val) == tuple:
            lo, hi = val[0], val[1]
            if col.num_vals is not None and isinstance(lo, (int, float)) and isinstance(hi, (int, float)):
                keep = (col.num_vals >= lo) & (col.num_vals <= hi)
                if col.has_null:
                    keep &= col.num_vals != col.null
            else:
                keep = np.asarray([not (col.has_null and k == col.null) and lo <= k <= hi for k in keys], dtype=bool)
            return keep if keep.any() else None
        if type(val) == list:
            if len(val) == 0:
                return None
            chosen = set(v for v in val if v in col.pair)
        else:
            if val not in col.pair:
                return None
            chosen = {val}
        return np.asarray([k in chosen for k in keys], dtype=bool)

    # ------------------------------------------------------------------ stage 2
    @staticmethod
    def _unit_bins(b: Sequence[int], w) -> bool:
        """True when the selected bins all carry weight exactly 1 and none repeats."""
        if len(b) > 1 and len(set(b)) != len(b):
            return False
        if type(w) is np.ndarray:
            w = w.ravel().tolist()
        elif not isinstance(w, (list, tuple)):
            w = np.asarray(w, dtype=np.float64).reshape(-1).tolist()
        for x in w:
            if x != 1:
                return False
        return True

    def geometry(self):
        """(bit offsets int64[n], BITS row bytes, dense offsets int64[n], dense width) -- same rules as the C ABI."""
        card = self.tm.card.astype(np.int64)
        bit_off = np.concatenate([[0], np.cumsum(card)[:-1]]).astype(np.int64)
        row_bytes = -(-int(card.sum()) // 128) * 16
        pad = -(-card // 4) * 4
        dense_off = np.concatenate([[0], np.cumsum(pad)[:-1]]).astype(np.int64)
        return bit_off, row_bytes, dense_off, int(pad.sum())

    def _pack_cache(self) -> dict:
        """Per-model constants of ``pack`` (row geometry, per-column bit masks, the unconstrained DENSE row), built once."""
        g = getattr(self, "_pack_g", None)
        if g is None:
            tm = self.tm
            n = tm.n_nodes
            bit_off, row_bytes, off, width = self.geometry()
            card = [int(c) for c in tm.card]
            boff = [int(b) for b in bit_off]
            dense_default = np.zeros(width, dtype=np.float32)
            for v in range(n):
                dense_default[off[v]: off[v] + card[v]] = 1.0
            g = {"row_bytes": row_bytes, "off": off, "width": width, "card": card, "boff": boff,
                 "full_mask": (1 << int(tm.card.sum())) - 1,
                 "col_mask": [((1 << card[v]) - 1) << boff[v] for v in range(n)], "dense_default": dense_default}
            self._pack_g = g
        return g

    def pack(self, decoded: Sequence[Tuple[Dict[str, Sequence[int]], Dict[str, np.ndarray]]],
             fanouts: Optional[Sequence[Sequence[str]]] = None, force_dense: bool = False):
        """Pack already decoded queries.

        Returns ``(bits_idx, bits_desc, dense_idx, dense_desc, mask)``: indices of the queries that
        went to the ``BITS`` / ``DENSE_F32`` batch, the two descriptor arrays (uint8 rows / fp32 rows)
        and the fan-out bitmask rows (``None`` when no query has fan-out columns), all in input order
        within a batch.  Columns outside the root component are ignored, as the reference's Steiner
        walk never sees them.
        """
        tm = self.tm
        n = tm.n_nodes
        nq = len(decoded)
        g = self._pack_cache()
        row_bytes, off, width = g["row_bytes"], g["off"], g["width"]
        card, boff, full_mask, col_mask, dense_default = g["card"], g["boff"], g["full_mask"], g["col_mask"], g["dense_default"]
        words = (n + 31) // 32
        mask = np.zeros((nq, words), dtype=np.uint32) if fanouts is not None else None
        kinds = np.zeros(nq, dtype=np.int8)  # 0 = bits, 1 = dense
        bit_rows: List[bytes] = []     # BITS rows as little-endian byte strings built from Python integers
        dense_rows: List[np.ndarray] = []
        index = tm._index
        for qi, (bins, wts) in enumerate(decoded):
            cols = []
            ok = not force_dense
            for attr, b in bins.items():
                v = index.get(attr)
                if v is None:
                    continue
                bl = list(b) if isinstance(b, (list, tuple, np.ndarray)) else [b]
                cols.append((v, bl, wts[attr]))
                if ok and not self._unit_bins(bl, wts[attr]):
                    ok = False
            if fanouts is not None:
                for attr in fanouts[qi]:
                    v = index.get(attr)
                    if v is None or attr in bins or tm.fan_vector(v) is None:
                        continue
                    mask[qi, v >> 5] |= np.uint32(1 << (v & 31))
            if ok:
                row = full_mask
                for v, bl, _ in cols:
                    row &= ~col_mask[v]
                    o = boff[v]
                    for b in bl:
                        b = int(b)
                        if not 0 <= b < card[v]:
                            raise IndexError(f"bin {b} outside the domain of column {v}")
                        row |= 1 << (o + b)
                bit_rows.append(row.to_bytes(row_bytes, "little"))
            else:
                kinds[qi] = 1
                row = dense_default.copy()
                for v, bl, w in cols:
                    w = np.asarray(w, dtype=np.float64).reshape(-1)
                    seg = np.zeros(card[v], dtype=np.float64)
                    if len(bl):
                        if w.size == 1 and len(bl) > 1:
                            w = np.full(len(bl), w[0])
                        np.add.at(seg, np.asarray(bl, dtype=np.int64), w)
                    row[off[v]: off[v] + card[v]] = seg
                dense_rows.append(row)
        bits_idx = np.nonzero(kinds == 0)[0]
        dense_idx = np.nonzero(kinds == 1)[0]
        bits_desc = (np.frombuffer(b"".join(bit_rows), dtype=np.uint8).reshape(len(bit_rows), row_bytes).copy()
                     if bit_rows else np.zeros((0, row_bytes), dtype=np.uint8))
        dense_desc = np.stack(dense_rows) if dense_rows else np.zeros((0, width), dtype=np.float32)
        return bits_idx, bits_desc, dense_idx, dense_desc, mask

    def pack_sparse(self, lo: np.ndarray, hi: np.ndarray):
        """SPARSE (CSR) form of ``[B, n_nodes]`` bin bounds: ``(row_off uint32[B+1], entries uint32[...])``.

        One entry ``col | lo<<16 | hi<<24`` per column whose bounds are narrower than its domain,
        ascending column order.  Vectorised; needs every domain <= 256 states."""
        card = self.tm.card.astype(np.int64)
        if int(card.max()) > 256:
            raise ValueError("SPARSE entries hold 8-bit state bounds")
        lo = np.asarray(lo, dtype=np.int64)
        hi = np.asarray(hi, dtype=np.int64)
        con = (lo > 0) | (hi < card[None, :] - 1)
        row_off = np.zeros(lo.shape[0] + 1, dtype=np.uint32)
        np.cumsum(con.sum(axis=1), out=row_off[1:])
        qi, vi = np.nonzero(con)  # row-major: ascending query, then ascending column
        entries = (vi.astype(np.uint32) | (lo[qi, vi].astype(np.uint32) << 16) | (hi[qi, vi].astype(np.uint32) << 24))
        return row_off, entries.astype(np.uint32)

    def pack_bits(self, lo: np.ndarray, hi: np.ndarray) -> np.ndarray:
        """Vectorised BITS packing of ``[B, n_nodes]`` bin bounds (uint8 rows)."""
        bit_off, row_bytes, _, _ = self.geometry()
        card = self.tm.card.astype(np.int64)
        cols = []
        for v in range(self.tm.n_nodes):
            c = np.arange(int(card[v]))[None, :]
            cols.append((c >= np.asarray(lo)[:, v:v + 1]) & (c <= np.asarray(hi)[:, v:v + 1]))
        packed = np.packbits(np.concatenate(cols, axis=1), axis=1, bitorder="little")
        out = np.zeros((packed.shape[0], row_bytes), dtype=np.uint8)
        out[:, : packed.shape[1]] = packed
        return out

    def pack_ranges(self, lo: np.ndarray, hi: np.ndarray) -> np.ndarray:
        """Vectorised RANGE_U8 packing of ``[B, n_nodes]`` bin bounds (topological node order)."""
        n = self.tm.n_nodes
        stride = -(-2 * n // 4) * 4
        out = np.zeros((lo.shape[0], stride), dtype=np.uint8)
        out[:, 0:2 * n:2] = lo
        out[:, 1:2 * n:2] = hi
        return out


def dense_to_wsparse(tm: TreeModel, dense: np.ndarray):
    """DENSE_F32 rows -> WSPARSE (``include/bayescard_b200.h``): per row and constrained column ONE run covering the
    states from the first to the last non-zero weight (zeros inside the run are sent as weights).  A column is
    constrained when its segment differs from all-ones.  Vectorised over the batch; returns ``(row_off, words)`` uint32.
    The expansion on the device reproduces ``dense`` bit for bit (row padding excepted, which no kernel reads)."""
    dense = np.ascontiguousarray(dense, dtype=np.float32)
    nq = dense.shape[0]
    n = tm.n_nodes
    off = np.zeros(n, dtype=np.int64)
    acc = 0
    for v in range(n):
        off[v] = acc
        acc += -(-int(tm.card[v]) // 4) * 4
    if dense.shape[1] != acc:
        raise ValueError(f"dense rows have {dense.shape[1]} floats, the model needs {acc}")
    if int(tm.card.max()) > 256:
        raise ValueError("WSPARSE runs hold 8-bit state indices")
    first = np.zeros((nq, n), dtype=np.int64)
    count = np.full((nq, n), -1, dtype=np.int64)  # -1: unconstrained (no run)
    for v in range(n):
        card = int(tm.card[v])
        seg = dense[:, off[v]: off[v] + card]
        con = np.any(seg != 1.0, axis=1)
        nz = seg != 0.0
        anynz = nz.any(axis=1)
        f = np.where(anynz, nz.argmax(axis=1), 0)
        l = np.where(anynz, card - 1 - nz[:, ::-1].argmax(axis=1), -1)
        first[:, v] = f
        count[:, v] = np.where(con, l - f + 1, -1)
    # the run length is an 8-bit field: a run of 256 states (a 256-state column whose first and last weights are
    # non-zero) is sent as a run of 255 plus a one-state continuation run (bit 15)
    tail = np.where(count > 255, count - 255, 0)
    head = count - tail
    run_words = np.where(count >= 0, head + 1, 0) + np.where(tail > 0, tail + 1, 0)   # headers + weights per (row, column)
    row_len = run_words.sum(axis=1)
    row_off = np.zeros(nq + 1, dtype=np.int64)
    np.cumsum(row_len, out=row_off[1:])
    if row_off[-1] >= 1 << 32:
        raise ValueError("batch too large for 32-bit offsets: split it")
    words = np.zeros(int(row_off[-1]), dtype=np.uint32)
    col_start = row_off[:-1, None] + np.cumsum(run_words, axis=1) - run_words   # word index of each run's header
    for v in range(n):
        rows = np.nonzero(count[:, v] >= 0)[0]
        if rows.size == 0:
            continue
        c, f, st, t = head[rows, v], first[rows, v], col_start[rows, v], tail[rows, v]
        words[st] = (np.uint32(v) | (f.astype(np.uint32) << np.uint32(16)) | (c.astype(np.uint32) << np.uint32(24)))
        seg = dense[:, off[v]: off[v] + int(tm.card[v])].view(np.uint32)
        for j in range(int(c.max()) if c.size else 0):   # at most card(v) vectorised passes
            m = c > j
            words[st[m] + 1 + j] = seg[rows[m], f[m] + j]
        if t.any():
            m = t > 0
            st2, f2 = st[m] + 1 + c[m], f[m] + c[m]
            words[st2] = (np.uint32(v) | np.uint32(1 << 15) | (f2.astype(np.uint32) << np.uint32(16))
                          | (t[m].astype(np.uint32) << np.uint32(24)))
            for j in range(int(t.max())):
                mm = t[m] > j
                words[st2[mm] + 1 + j] = seg[rows[m][mm], f2[mm] + j]
    return row_off.astype(np.uint32), words


def unpack_ranges(tm: TreeModel, desc: np.ndarray):
    """Inverse of :meth:`PredicateCompiler.pack_ranges`: ``(lo, hi)`` int arrays ``[B, n_nodes]``."""
    n = tm.n_nodes
    d = np.asarray(desc, dtype=np.uint8).reshape(-1, -(-2 * n // 4) * 4)
    return d[:, 0:2 * n:2].astype(np.int64), d[:, 1:2 * n:2].astype(np.int64)
