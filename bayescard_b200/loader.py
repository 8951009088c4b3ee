"""Model loader: reference pickle -> :class:`TreeModel` -> packed fp32 CPT arena.

The reference persists a model as a plain ``pickle`` of its ``Bayescard_BN`` object
(reference ``Models/BN_single_model.py:207-223``, ``Testing/BN_training.py:20``).  This module reads
that pickle WITHOUT the reference sources on ``sys.path``: a restricted ``Unpickler`` maps the three
reference classes to attribute bags and lets only numpy / networkx-view / pandas-Interval /
builtin containers through.  Everything the exact-jit path needs is then copied into a
:class:`TreeModel`:

* the topological order of ``align_cpds_in_topological`` (reference ``Models/Bayescard_BN.py:340-358``),
* ``parent[]``/``card[]`` and the fp64 CPTs ``T_v[x_v, x_pa]`` (reference
  ``Pgmpy/factors/discrete/CPD.py:137-139``: ``values`` is ``[card(child), card(parent)]``),
* the root component seen by ``get_root`` + ``steiner_tree`` (reference
  ``Pgmpy/inference/ExactInference.py:42-75``: only the component of ``list(model.nodes)[0]`` is
  ever walked, predicates elsewhere are silently dropped),
* the decode metadata (``encoding``, ``n_in_bin``, ``mapping``, ``domain``, ``null_values``,
  ``n_distinct_mapping``, ``attr_type``, ``fanouts``, ``nrows``).

``TreeModel.save``/``TreeModel.load`` give a flat, versioned ``.npz`` form (SURVEY.md section 8f.4) so a
server never has to unpickle third-party classes; ``tests/golden/models`` holds the shipped
models in that form.
"""
from __future__ import annotations

import io
import json
import pickle
from dataclasses import dataclass, field
from typing import Any, Dict, List, Optional, Sequence, Tuple

import numpy as np

FORMAT_VERSION = 1


class _Bag:
    """Attribute bag standing in for a reference class while unpickling."""

    def __setstate__(self, state):
        if isinstance(state, tuple) and len(state) == 2 and isinstance(state[1], dict):
            # (dict_state, slots_state)
            if state[0]:
                self.__dict__.update(state[0])
            self.__dict__.update(state[1])
        else:
            self.__dict__.update(state)


class _BNBag(_Bag):
    pass


class _GraphBag(_Bag):
    pass


class _CPDBag(_Bag):
    pass


class _ViewBag(_Bag):
    """networkx NodeView: only kept so the pickle stream parses; never used."""

    def __init__(self, *a, **k):
        pass


_CLASS_MAP = {
    ("Models.Bayescard_BN", "Bayescard_BN"): _BNBag,
    ("Pgmpy.models.BayesianModel", "BayesianModel"): _GraphBag,
    ("Pgmpy.factors.discrete.CPD", "TabularCPD"): _CPDBag,
    ("networkx.classes.reportviews", "NodeView"): _ViewBag,
    ("networkx.classes.reportviews", "OutEdgeView"): _ViewBag,
    ("networkx.classes.reportviews", "InEdgeView"): _ViewBag,
    ("networkx.classes.reportviews", "DiDegreeView"): _ViewBag,
    ("networkx.classes.reportviews", "OutDegreeView"): _ViewBag,
    ("networkx.classes.reportviews", "InDegreeView"): _ViewBag,
}

# Explicit (module, name) allow-list: data containers and the numpy array/scalar reconstructors only.  A prefix test
# on the module would let builtins.eval / exec / getattr / __import__ through, i.e. arbitrary code execution.
_ALLOWED_GLOBALS = frozenset(
    [("builtins", n) for n in ("set", "frozenset", "dict", "list", "tuple", "slice", "complex", "bytearray",
                               "int", "float", "bool", "str", "bytes", "range")]
    + [(m, n) for m in ("numpy.core.multiarray", "numpy._core.multiarray") for n in ("_reconstruct", "scalar")]
    + [("numpy", "ndarray"), ("numpy", "dtype"),
       ("numpy.core.numeric", "_frombuffer"), ("numpy._core.numeric", "_frombuffer"),
       ("collections", "OrderedDict"), ("collections", "defaultdict"),
       ("copyreg", "_reconstructor"), ("_codecs", "encode")]
)


class _Interval:
    """pandas Interval stand-in when pandas is absent (only .left/.right/.closed are read)."""

    def __init__(self, left, right, closed="right"):
        self.left, self.right, self.closed = left, right, closed


class RestrictedUnpickler(pickle.Unpickler):
    def find_class(self, module, name):
        key = (module, name)
        if key in _CLASS_MAP:
            return _CLASS_MAP[key]
        if key == ("pandas._libs.interval", "Interval"):
            try:
                from pandas import Interval  # noqa: WPS433

                return Interval
            except Exception:  # pragma: no cover - pandas is in the image
                return _Interval
        if key in _ALLOWED_GLOBALS:
            return super().find_class(module, name)
        raise pickle.UnpicklingError(f"class {module}.{name} is not allowed in a BayesCard model pickle")


def _py(v):
    """numpy scalar -> python scalar (hash/equality preserving: 2019.0 == 2019)."""
    if isinstance(v, np.generic):
        return v.item()
    return v


@dataclass
class TreeModel:
    """Everything the exact-jit path reads from a ``Bayescard_BN`` pickle."""

    table_name: Any
    nrows: Any                                 # int or float, as pickled (affects result types)
    node_names: List[str]                      # original column order (== structure order)
    structure: Tuple[Tuple[int, ...], ...]     # parent index tuples, node_names order
    attr_type: Dict[str, str]
    algorithm: str
    # --- inference topology (topological numbering; index 0..n_infer-1 are the root component) ---
    topo_names: List[str]                      # all nodes, order of align_cpds_in_topological
    infer_names: List[str]                     # nodes of the root component, topological order
    parent: np.ndarray                         # int32[n_infer], -1 for the root, index into infer_names
    card: np.ndarray                           # int32[n_infer]
    cpts: List[np.ndarray]                     # fp64 [card_v, card_pa] ([card_root] for the root)
    dropped_names: List[str]                   # nodes outside the root component (forest trap)
    # --- decode metadata ---
    encoding: Dict[str, Optional[dict]] = field(default_factory=dict)
    n_in_bin: Dict[str, dict] = field(default_factory=dict)
    mapping: Dict[str, Optional[List[Tuple[float, float]]]] = field(default_factory=dict)
    domain: Dict[str, Any] = field(default_factory=dict)
    null_values: Any = field(default_factory=dict)
    n_distinct_mapping: Dict[str, dict] = field(default_factory=dict)
    fanouts: Dict[str, np.ndarray] = field(default_factory=dict)
    fanout_attr: List[str] = field(default_factory=list)
    fanout_attr_inverse: List[str] = field(default_factory=list)
    fanout_attr_positive: List[str] = field(default_factory=list)
    max_parents: Any = None
    n_mcv: Any = None
    n_bins: Any = None
    root: Any = None
    # --- counts behind the CPTs (fit.count_layout order, uint64) and the rows they were counted from; known when the
    #     CPTs were fitted here (fit.refit, structure.learn_tree_model), recovered by fit.counts_from_cpts otherwise.
    #     Neither is stored in the .npz / .bcm files: the CPTs determine them.
    counts: Optional[np.ndarray] = None
    fit_rows: Optional[int] = None

    # ------------------------------------------------------------------ derived
    @property
    def n_nodes(self) -> int:
        return len(self.infer_names)

    def index_of(self, name: str) -> int:
        return self._index[name]

    def __post_init__(self):
        self._index = {n: i for i, n in enumerate(self.infer_names)}
        self.children: List[List[int]] = [[] for _ in self.infer_names]
        for v, p in enumerate(self.parent):
            if p >= 0:
                self.children[int(p)].append(v)

    @property
    def n_cpt_entries(self) -> int:
        return int(sum(c.size for c in self.cpts))

    @property
    def flops_dense(self) -> int:
        """ALGORITHMIC flop per query: one FMA per non-root CPT entry (SURVEY.md section 8d)."""
        return int(2 * sum(c.size for v, c in enumerate(self.cpts) if self.parent[v] >= 0))

    def fan_vector(self, v: int) -> Optional[np.ndarray]:
        f = self.fanouts.get(self.infer_names[v])
        if f is None:
            return None
        f = np.asarray(f, dtype=np.float64)
        return f if f.size == int(self.card[v]) else None

    # ------------------------------------------------------------------ arena packing
    def pack_arena(self, row_align: int = 4):
        """fp32 CPT arena, nodes in topological order, every row 16 B aligned.

        Layout of node v: ``card_v`` rows of ``stride_v = round_up(card_pa, row_align)`` floats,
        ``T_v[c, p]`` at ``off_v + c*stride_v + p``; the root is one row of ``card_root`` floats.
        Padding entries are 0.  Returns ``(arena fp32[...], off int64[n], stride int32[n])``.
        """
        offs, strides, total = [], [], 0
        for v, t in enumerate(self.cpts):
            cols = t.shape[1] if t.ndim == 2 else t.shape[0]
            rows = t.shape[0] if t.ndim == 2 else 1
            stride = -(-cols // row_align) * row_align
            offs.append(total)
            strides.append(stride)
            total += rows * stride
        arena = np.zeros(max(total, row_align), dtype=np.float32)
        for v, t in enumerate(self.cpts):
            rows = t.shape[0] if t.ndim == 2 else 1
            cols = t.shape[1] if t.ndim == 2 else t.shape[0]
            view = arena[offs[v]: offs[v] + rows * strides[v]].reshape(rows, strides[v])
            view[:, :cols] = np.asarray(t, dtype=np.float64).reshape(rows, cols)
        return arena, np.asarray(offs, dtype=np.int64), np.asarray(strides, dtype=np.int32)

    def pack_fanouts(self, row_align: int = 4):
        """fp32 fan-out arena: ``fan_off[v] = -1`` if node v has no fan-out vector."""
        offs, total, chunks = [], 0, []
        for v in range(self.n_nodes):
            f = self.fan_vector(v)
            if f is None:
                offs.append(-1)
                continue
            n = -(-f.size // row_align) * row_align
            buf = np.zeros(n, dtype=np.float32)
            buf[: f.size] = f
            offs.append(total)
            chunks.append(buf)
            total += n
        arena = np.concatenate(chunks) if chunks else np.zeros(row_align, dtype=np.float32)
        return arena, np.asarray(offs, dtype=np.int64)

    # ------------------------------------------------------------------ flat file format
    def _meta(self) -> dict:
        meta = {
            "format_version": FORMAT_VERSION,
            "table_name": _jsonable(self.table_name),
            "nrows": _jsonable(self.nrows),
            "node_names": self.node_names,
            "structure": [list(map(int, s)) for s in self.structure],
            "attr_type": self.attr_type,
            "algorithm": self.algorithm,
            "topo_names": self.topo_names,
            "infer_names": self.infer_names,
            "dropped_names": self.dropped_names,
            "encoding": {k: (None if v is None else [[_jsonable(a), int(b)] for a, b in v.items()])
                         for k, v in self.encoding.items()},
            "n_in_bin": {k: None if v is None else [[int(b), (int(d) if isinstance(d, int) else [[_jsonable(a), float(w)] for a, w in d.items()])]
                             for b, d in v.items()] for k, v in self.n_in_bin.items()},
            "mapping": {k: (None if v is None else [[float(a), float(b)] for a, b in v])
                        for k, v in self.mapping.items()},
            "domain": {k: _jsonable(v) for k, v in self.domain.items()},
            "null_values": _jsonable(self.null_values),
            "n_distinct_mapping": {k: [[_jsonable(a), _jsonable(b)] for a, b in v.items()]
                                   for k, v in self.n_distinct_mapping.items()},
            "fanout_attr": self.fanout_attr,
            "fanout_attr_inverse": self.fanout_attr_inverse,
            "fanout_attr_positive": self.fanout_attr_positive,
            "max_parents": _jsonable(self.max_parents),
            "n_mcv": _jsonable(self.n_mcv),
            "n_bins": _jsonable(self.n_bins),
            "root": _jsonable(self.root),
        }
        return meta

    def save(self, path: str) -> None:
        meta = self._meta()
        arrays = {"parent": self.parent.astype(np.int32), "card": self.card.astype(np.int32)}
        for v, t in enumerate(self.cpts):
            arrays[f"cpt_{v}"] = np.asarray(t, dtype=np.float64)
        for k, f in self.fanouts.items():
            arrays["fan_" + k] = np.asarray(f, dtype=np.float64)
        arrays["meta_json"] = np.frombuffer(json.dumps(meta).encode("utf-8"), dtype=np.uint8)
        np.savez_compressed(path, **arrays)

    @staticmethod
    def load(path: str) -> "TreeModel":
        with np.load(path, allow_pickle=False) as z:
            meta = json.loads(bytes(z["meta_json"]).decode("utf-8"))
            if meta["format_version"] != FORMAT_VERSION:
                raise ValueError(f"unsupported model format version {meta['format_version']}")
            parent = z["parent"].astype(np.int32)
            card = z["card"].astype(np.int32)
            cpts = [z[f"cpt_{v}"] for v in range(len(parent))]
            fanouts = {k[4:]: z[k] for k in z.files if k.startswith("fan_")}
        return TreeModel._from_meta(meta, parent, card, cpts, fanouts)

    @staticmethod
    def _from_meta(meta, parent, card, cpts, fanouts) -> "TreeModel":
        enc = {k: (None if v is None else {_unjson(a): int(b) for a, b in v}) for k, v in meta["encoding"].items()}
        nib = {k: None if v is None else {int(b): (d if isinstance(d, int) else {_unjson(a): float(w) for a, w in d}) for b, d in v}
               for k, v in meta["n_in_bin"].items()}
        mapping = {k: (None if v is None else [(float(a), float(b)) for a, b in v]) for k, v in meta["mapping"].items()}
        return TreeModel(
            table_name=_unjson(meta["table_name"]), nrows=meta["nrows"], node_names=meta["node_names"],
            structure=tuple(tuple(s) for s in meta["structure"]), attr_type=meta["attr_type"],
            algorithm=meta["algorithm"], topo_names=meta["topo_names"], infer_names=meta["infer_names"],
            parent=parent, card=card, cpts=cpts, dropped_names=meta["dropped_names"],
            encoding=enc, n_in_bin=nib, mapping=mapping,
            domain={k: _unjson(v) for k, v in meta["domain"].items()},
            null_values=_unjson(meta["null_values"]),
            n_distinct_mapping={k: {_unjson(a): _unjson(b) for a, b in v} for k, v in meta["n_distinct_mapping"].items()},
            fanouts=fanouts, fanout_attr=meta["fanout_attr"], fanout_attr_inverse=meta["fanout_attr_inverse"],
            fanout_attr_positive=meta["fanout_attr_positive"], max_parents=_unjson(meta["max_parents"]),
            n_mcv=_unjson(meta["n_mcv"]), n_bins=_unjson(meta["n_bins"]), root=_unjson(meta["root"]),
        )


    # ------------------------------------------------------------------ flat, mmap-able model file (".bcm")
    def save_flat(self, path: str) -> None:
        """One flat, versioned, mmap-able file: what ``bc_model_create_from_file`` (csrc/bc_modelfile.cc, which documents
        the layout) uploads without touching Python or pickle, plus the decode tables as a JSON section
        (SURVEY.md section 8f item 4)."""
        import struct

        arena, off, stride = self.pack_arena()
        fan, foff = self.pack_fanouts()
        has_fan = bool((foff >= 0).any())
        cpt64 = np.concatenate([np.asarray(t, dtype=np.float64).reshape(-1) for t in self.cpts])
        meta = self._meta()
        meta["fan_names"] = [k for k in self.fanouts]
        meta["fan_sizes"] = [int(np.asarray(self.fanouts[k]).size) for k in self.fanouts]
        meta["fan64"] = [np.asarray(self.fanouts[k], dtype=np.float64).reshape(-1).tolist() for k in self.fanouts]
        mbytes = json.dumps(meta).encode("utf-8")
        sections = [
            (np.ascontiguousarray(self.parent, dtype="<i4").tobytes(), 64),
            (np.ascontiguousarray(self.card, dtype="<i4").tobytes(), 64),
            (np.ascontiguousarray(off, dtype="<i8").tobytes(), 64),
            (np.ascontiguousarray(stride, dtype="<i4").tobytes(), 64),
            (np.ascontiguousarray(foff, dtype="<i8").tobytes(), 64),
            (np.ascontiguousarray(arena, dtype="<f4").tobytes(), 4096),
            (np.ascontiguousarray(fan, dtype="<f4").tobytes() if has_fan else b"", 64),
            (np.ascontiguousarray(cpt64, dtype="<f8").tobytes(), 64),
            (mbytes, 64),
        ]
        offs, pos = [], 128
        for data, align in sections:
            pos = -(-pos // align) * align
            offs.append(pos)
            pos += len(data)
        header = struct.pack("<8sII4Q9QQ", b"BCB200M\0", 1, self.n_nodes, arena.size, fan.size if has_fan else 0, cpt64.size,
                             len(mbytes), *offs, pos)
        assert len(header) == 128
        with open(path, "wb") as f:
            f.write(header)
            at = 128
            for (data, _), o in zip(sections, offs):
                f.write(b"\0" * (o - at))
                f.write(data)
                at = o + len(data)

    @staticmethod
    def load_flat(path: str) -> "TreeModel":
        """Host-side twin of ``bc_model_create_from_file``: the same file through ``mmap``, no pickle."""
        import mmap
        import struct

        with open(path, "rb") as f:
            mm = mmap.mmap(f.fileno(), 0, access=mmap.ACCESS_READ)
        try:
            if len(mm) < 128:
                raise ValueError(f"{path}: not a flat model file (shorter than its header)")
            (magic, version, n, arena_floats, fan_floats, n64, meta_bytes, o_parent, o_card, o_off, o_stride, o_foff, o_arena, o_fan,
             o_cpt64, o_meta, file_bytes) = struct.unpack("<8sII4Q9QQ", mm[:128])
            if magic != b"BCB200M\0":
                raise ValueError(f"{path}: bad magic (not a bayescard_b200 flat model file)")
            if version != 1:
                raise ValueError(f"{path}: unsupported flat model file version {version}")
            if file_bytes != len(mm):
                raise ValueError(f"{path}: truncated or padded file (size differs from the header)")
            for o, ln in ((o_parent, 4 * n), (o_card, 4 * n), (o_cpt64, 8 * n64), (o_meta, meta_bytes)):
                if o + ln > len(mm):
                    raise ValueError(f"{path}: a section lies outside the file")
            parent = np.frombuffer(mm, dtype="<i4", count=n, offset=o_parent).astype(np.int32)
            card = np.frombuffer(mm, dtype="<i4", count=n, offset=o_card).astype(np.int32)
            cpt64 = np.frombuffer(mm, dtype="<f8", count=n64, offset=o_cpt64).copy()
            meta = json.loads(bytes(mm[o_meta:o_meta + meta_bytes]).decode("utf-8"))
        finally:
            mm.close()
        cpts, at = [], 0
        for v in range(n):
            shape = (int(card[v]),) if parent[v] < 0 else (int(card[v]), int(card[parent[v]]))
            size = int(np.prod(shape))
            cpts.append(cpt64[at:at + size].reshape(shape))
            at += size
        fanouts = {k: np.asarray(v, dtype=np.float64) for k, v in zip(meta["fan_names"], meta["fan64"])}
        return TreeModel._from_meta(meta, parent, card, cpts, fanouts)


def _jsonable(v):
    v = _py(v)
    if isinstance(v, (set, frozenset)):
        return {"__set__": sorted(_jsonable(x) for x in v)}
    if isinstance(v, tuple):
        return {"__tuple__": [_jsonable(x) for x in v]}
    if isinstance(v, np.ndarray):
        return [_jsonable(x) for x in v.tolist()]
    if isinstance(v, list):
        return [_jsonable(x) for x in v]
    if isinstance(v, dict):
        return {"__dict__": [[_jsonable(a), _jsonable(b)] for a, b in v.items()]}
    if isinstance(v, float) and v != v:
        return {"__nan__": 1}
    if isinstance(v, float) and v in (float("inf"), float("-inf")):
        return {"__inf__": 1 if v > 0 else -1}
    return v


def _unjson(v):
    if isinstance(v, dict):
        if "__set__" in v:
            return set(_unjson(x) for x in v["__set__"])
        if "__tuple__" in v:
            return tuple(_unjson(x) for x in v["__tuple__"])
        if "__dict__" in v:
            return {_unjson(a): _unjson(b) for a, b in v["__dict__"]}
        if "__nan__" in v:
            return float("nan")
        if "__inf__" in v:
            return float("inf") * v["__inf__"]
    if isinstance(v, list):
        return [_unjson(x) for x in v]
    return v


# ---------------------------------------------------------------------- pickle -> TreeModel

def topological_order(structure: Sequence[Sequence[int]]) -> List[int]:
    """Order produced by ``align_cpds_in_topological`` (reference Models/Bayescard_BN.py:340-349).

    Repeated sweeps over the columns in index order; a column is appended during a sweep as soon
    as all of its parents have been appended (possibly earlier in the same sweep).
    """
    order: List[int] = []
    placed = set()
    n = len(structure)
    while len(order) < n:
        before = len(order)
        for i, deps in enumerate(structure):
            if i in placed:
                continue
            if all(d in placed for d in deps):
                order.append(i)
                placed.add(i)
        if len(order) == before:
            raise ValueError("structure has a cycle")
    return order


def tree_model_from_object(bn: Any) -> TreeModel:
    """Build a TreeModel from an unpickled ``Bayescard_BN``-shaped object (bag or real)."""
    d = bn.__dict__
    node_names = list(d["node_names"])
    structure = tuple(tuple(int(x) for x in s) for s in d["structure"])
    if any(len(s) > 1 for s in structure):
        raise ValueError("exact-jit supports Chow-Liu trees only (max_parents=1); "
                         "reference Models/Bayescard_BN.py:135 asserts the same")
    algorithm = d.get("algorithm", "chow-liu")
    order = topological_order(structure)
    topo_names = [node_names[i] for i in order]

    model = d["model"]
    cpd_by_var = {}
    for cpd in model.__dict__["cpds"] if isinstance(model, _Bag) else model.cpds:
        cd = cpd.__dict__
        cpd_by_var[cd["variable"]] = cd
    # first node of the graph as the reference's get_root() sees it (ExactInference.py:53)
    gdict = model.__dict__
    if "_node" in gdict:
        first = next(iter(gdict["_node"]))
    else:  # a real networkx graph
        first = list(model.nodes)[0]
    par_name = {}
    for i, deps in enumerate(structure):
        par_name[node_names[i]] = node_names[deps[0]] if deps else None
    # cross-check the graph recorded in the CPDs against `structure`
    for name, cd in cpd_by_var.items():
        vars_ = list(cd["variables"])
        rec_parent = vars_[1] if len(vars_) > 1 else None
        if rec_parent != par_name[name]:
            raise ValueError(f"CPD of {name} records parent {rec_parent}, structure says {par_name[name]}")
    root = first
    while par_name[root] is not None:
        root = par_name[root]
    in_comp = set()
    for n in topo_names:  # parents precede children in topo_names
        if n == root or (par_name[n] in in_comp):
            in_comp.add(n)
    infer_names = [n for n in topo_names if n in in_comp]
    dropped = [n for n in topo_names if n not in in_comp]
    idx = {n: i for i, n in enumerate(infer_names)}
    parent = np.full(len(infer_names), -1, dtype=np.int32)
    card = np.zeros(len(infer_names), dtype=np.int32)
    cpts = []
    for v, n in enumerate(infer_names):
        cd = cpd_by_var[n]
        vals = np.ascontiguousarray(np.asarray(cd["values"], dtype=np.float64))
        if par_name[n] is not None:
            parent[v] = idx[par_name[n]]
            if vals.ndim != 2:
                raise ValueError(f"CPD of {n} has rank {vals.ndim}, expected [card, card_parent]")
        else:
            vals = vals.reshape(-1)
        card[v] = vals.shape[0]
        cpts.append(vals)
    for v in range(len(infer_names)):
        if parent[v] >= 0 and cpts[v].shape[1] != card[parent[v]]:
            raise ValueError("CPT shape does not match the parent's cardinality")

    def clean_map(m):
        return {_py(k): _py(v) for k, v in m.items()}

    encoding = {k: (None if v is None else clean_map(v)) for k, v in d.get("encoding", {}).items()}
    n_in_bin = {}
    for k, v in d.get("n_in_bin", {}).items():
        if v is None:
            n_in_bin[k] = None
            continue
        n_in_bin[k] = {int(b): (int(w) if isinstance(_py(w), int) else {_py(a): float(x) for a, x in w.items()})
                       for b, w in v.items()}
    mapping = {}
    for k, v in d.get("mapping", {}).items():
        if v is None or len(v) == 0:
            mapping[k] = None
        else:
            mapping[k] = [(float(v[i].left), float(v[i].right)) for i in range(len(v))]
    fanouts = {}
    for k, f in (d.get("fanouts") or {}).items():
        fanouts[k] = np.asarray(f, dtype=np.float64).reshape(-1)
    nv = d.get("null_values")
    if isinstance(nv, dict):
        nv = {k: _py(v) for k, v in nv.items()}
    return TreeModel(
        table_name=d.get("table_name"), nrows=_py(d["nrows"]), node_names=node_names, structure=structure,
        attr_type=dict(d["attr_type"]), algorithm=algorithm, topo_names=topo_names, infer_names=infer_names,
        parent=parent, card=card, cpts=cpts, dropped_names=dropped, encoding=encoding, n_in_bin=n_in_bin,
        mapping=mapping, domain={k: _domain_clean(v) for k, v in d.get("domain", {}).items()},
        null_values=nv if nv is not None else [],
        n_distinct_mapping={k: clean_map(v) for k, v in (d.get("n_distinct_mapping") or {}).items()},
        fanouts=fanouts, fanout_attr=list(d.get("fanout_attr", [])),
        fanout_attr_inverse=list(d.get("fanout_attr_inverse", [])),
        fanout_attr_positive=list(d.get("fanout_attr_positive", [])),
        max_parents=_py(d.get("max_parents")), n_mcv=_py(d.get("n_mcv")), n_bins=_py(d.get("n_bins")),
        root=_py(d.get("root")),
    )


def _domain_clean(v):
    if isinstance(v, tuple):
        return tuple(_py(x) for x in v)
    if isinstance(v, np.ndarray):
        return [_py(x) for x in v.tolist()]
    if isinstance(v, list):
        return [_py(x) for x in v]
    return _py(v)


def load_pickle(path_or_bytes) -> TreeModel:
    """Read a reference ``Bayescard_BN`` pickle (optionally bz2, as ``BN_Single.save(compress=True)``)."""
    if isinstance(path_or_bytes, (bytes, bytearray)):
        data = bytes(path_or_bytes)
    else:
        with open(path_or_bytes, "rb") as f:
            data = f.read()
    if data[:3] == b"BZh":
        import bz2

        data = bz2.decompress(data)
    bn = RestrictedUnpickler(io.BytesIO(data)).load()
    return tree_model_from_object(bn)


def load_model(path: str) -> TreeModel:
    """Load a reference pickle (``*.pkl``), the ``.npz`` fixture form or the flat mmap-able ``.bcm`` file."""
    with open(path, "rb") as f:
        magic = f.read(8)
    if magic == b"BCB200M\0":
        return TreeModel.load_flat(path)
    if magic[:2] == b"PK":
        return TreeModel.load(path)
    return load_pickle(path)
