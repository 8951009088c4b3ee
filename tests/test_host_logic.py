"""CPU tests of the host side: loader, SQL front end, predicate compiler, descriptor packing, the
C-ABI library's exported symbols and its host-only entry points (no compute calls without a GPU)."""
import copy
import ctypes
import os
import re

import ctypes as C

import numpy as np
import pytest

import golden_util as G
from bayescard_b200 import _lib as L
from bayescard_b200.decode import PredicateCompiler, dense_to_wsparse, unpack_ranges
from bayescard_b200.engine import DeviceModel, ShardedModel, gen_range_queries_host
from bayescard_b200.loader import TreeModel, topological_order
from bayescard_b200.sql_front import parse_query_single_table
from oracle import bayescard_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _as_map(bins, wts):
    w = np.asarray(wts, dtype=np.float64).reshape(-1)
    if w.size == 1 and len(bins) > 1:
        w = np.full(len(bins), w[0])
    return {int(b): float(x) for b, x in zip(bins, w)}


# ------------------------------------------------------------------------------------ loader
def test_models_shapes_match_survey():
    """SURVEY.md section 8a: node counts, CPT entries and algorithmic flop of the shipped models."""
    expect = {"dmv": (10, 10882, 21756), "census": (68, 3335, 6654), "imdb0": (9, 20398, 40782),
              "imdb1": (9, 30284, 60564), "imdb2": (9, 23402, 46800), "imdb3": (9, 30509, 61004),
              "imdb4": (10, 28096, 56178)}
    for name, (n, entries, flops) in expect.items():
        m = G.model(name)
        assert (m.n_nodes, m.n_cpt_entries, m.flops_dense) == (n, entries, flops)
        assert m.parent[0] == -1 and all(0 <= m.parent[v] < v for v in range(1, n))
        for v in range(1, n):
            assert np.allclose(m.cpts[v].sum(axis=0), 1.0, atol=1e-9)
        arena, off, stride = m.pack_arena()
        assert arena.dtype == np.float32 and all(o % 4 == 0 for o in off) and all(s % 4 == 0 for s in stride)
        for v in range(1, n):
            t = arena[off[v]: off[v] + m.card[v] * stride[v]].reshape(m.card[v], stride[v])
            assert np.array_equal(t[:, : m.cpts[v].shape[1]], m.cpts[v].astype(np.float32))


def test_topological_order_rule():
    # Models/Bayescard_BN.py:340-349: sweeps in index order, a column is placed as soon as its parent is
    assert topological_order(((), (0,), (3,), (1,), (5,), (1,))) == [0, 1, 3, 5, 2, 4]
    assert topological_order(((1,), ())) == [1, 0]
    with pytest.raises(ValueError):
        topological_order(((1,), (0,)))


def _reference_shaped_pickle(tm, monkeypatch):
    """A pickle laid out like the shipped ``Bayescard_BN`` pickles, written from a stored model: the three reference
    classes under their module paths, CPDs as ``TabularCPD`` attribute dicts, ``mapping`` as lists of
    ``pandas._libs.interval.Interval`` (the path older pandas releases pickle it under)."""
    import importlib
    import pickle
    import sys
    import types

    def interval_reduce(self):
        return type(self), (self.left, self.right, self.closed)

    classes = {}
    for module, name, body in (("Models.Bayescard_BN", "Bayescard_BN", {}), ("Pgmpy.models.BayesianModel", "BayesianModel", {}),
                               ("Pgmpy.factors.discrete.CPD", "TabularCPD", {}),
                               ("pandas._libs.interval", "Interval", {"__reduce__": interval_reduce})):
        cls = type(name, (), {"__module__": module, **body})
        parts = module.split(".")
        for i in range(1, len(parts) + 1):
            prefix = ".".join(parts[:i])
            if prefix not in sys.modules:
                try:
                    importlib.import_module(prefix)
                except ImportError:
                    monkeypatch.setitem(sys.modules, prefix, types.ModuleType(prefix))
        monkeypatch.setattr(sys.modules[module], name, cls, raising=False)
        classes[name] = cls

    def obj(cls, **state):
        o = cls.__new__(cls)
        o.__dict__.update(state)
        return o

    cpds = []
    for v, n in enumerate(tm.infer_names):
        variables = [n] if tm.parent[v] < 0 else [n, tm.infer_names[tm.parent[v]]]
        cpds.append(obj(classes["TabularCPD"], variable=n, variables=variables, values=tm.cpts[v].copy()))
    graph = obj(classes["BayesianModel"], cpds=cpds, _node={n: {} for n in tm.infer_names + tm.dropped_names})
    mapping = {k: None if v is None else [obj(classes["Interval"], left=lo, right=hi, closed="right") for lo, hi in v]
               for k, v in tm.mapping.items()}
    bn = obj(classes["Bayescard_BN"], table_name=tm.table_name, nrows=tm.nrows, node_names=list(tm.node_names),
             structure=[list(s) for s in tm.structure], attr_type=dict(tm.attr_type), algorithm=tm.algorithm, model=graph,
             encoding=tm.encoding, n_in_bin=tm.n_in_bin, mapping=mapping, domain=tm.domain, null_values=tm.null_values,
             n_distinct_mapping=tm.n_distinct_mapping, fanouts=tm.fanouts, fanout_attr=tm.fanout_attr,
             fanout_attr_inverse=tm.fanout_attr_inverse, fanout_attr_positive=tm.fanout_attr_positive,
             max_parents=tm.max_parents, n_mcv=tm.n_mcv, n_bins=tm.n_bins, root=tm.root)
    return pickle.dumps(bn, protocol=4)


def test_pickle_loader_matches_flat_models(monkeypatch):
    """The restricted unpickler on pickles in the shipped models' class layout, written from the stored flat models
    (which were converted from the shipped pickles): it must give back the same models, with no reference class imported."""
    import bz2

    from bayescard_b200.loader import load_pickle

    for name in ("dmv", "imdb3"):
        b = G.model(name)
        blob = _reference_shaped_pickle(b, monkeypatch)
        for a in (load_pickle(blob), load_pickle(bz2.compress(blob))):
            assert a.infer_names == b.infer_names and a.nrows == b.nrows and type(a.nrows) is type(b.nrows)
            assert all(np.array_equal(x, y) for x, y in zip(a.cpts, b.cpts))
            assert a.encoding == b.encoding and a.mapping == b.mapping and a.n_in_bin == b.n_in_bin
            assert np.array_equal(a.parent, b.parent) and a.dropped_names == b.dropped_names and a.topo_names == b.topo_names


def test_restricted_unpickler_rejects_foreign_classes():
    import pickle

    from bayescard_b200.loader import load_pickle

    blob = pickle.dumps(os.system)  # a global outside the allow list
    with pytest.raises(pickle.UnpicklingError):
        load_pickle(blob)

    class _Evil:  # builtins.eval through __reduce__: a module-prefix allow-list would run it
        def __init__(self, fn, args):
            self.fn, self.args = fn, args

        def __reduce__(self):
            return self.fn, self.args

    import builtins

    marker = os.path.join(os.path.dirname(__file__), "_pwned_marker")
    for fn, args in ((builtins.eval, (f"open({marker!r}, 'w').close()",)),
                     (builtins.exec, ("import os",)),
                     (builtins.getattr, ("abc", "upper")),
                     (builtins.__import__, ("os",)),
                     (os.system, ("true",))):
        with pytest.raises(pickle.UnpicklingError):
            load_pickle(pickle.dumps(_Evil(fn, args)))
    assert not os.path.exists(marker)


# ------------------------------------------------------------------------------------ sql + decode
@pytest.mark.parametrize("name", ["dmv", "census"])
def test_sql_and_decode_match_reference(name):
    m = G.model(name)
    pc = PredicateCompiler(m)
    for r in G.load(f"{name}_workload.json.gz")["queries"]:
        parsed = parse_query_single_table(r["sql"], m)
        ref = G.unjson(r["parsed"])
        assert list(parsed) == list(ref)
        for k in parsed:
            assert (list(parsed[k]) == list(ref[k])) if isinstance(ref[k], list) else (parsed[k] == ref[k])
        before = copy.deepcopy(parsed)
        bins, wts = pc.decode(parsed)
        assert parsed == before, "decode must not mutate its input"
        if r["decoded"] is None:
            assert bins is None
            continue
        for k, rb in r["decoded"]["bins"].items():
            assert _as_map(bins[k], wts[k]) == pytest.approx(_as_map(rb, r["decoded"]["weights"][k]), rel=1e-15)


@pytest.mark.parametrize("i", range(5))
def test_decode_imdb_cases(i):
    m = G.model(f"imdb{i}")
    pc = PredicateCompiler(m)
    for r in G.load("imdb_cases.json.gz")[f"imdb{i}"]:
        if "decoded" not in r:
            continue
        bins, wts = pc.decode(G.unjson(r["query"]))
        if r["decoded"] is None:
            assert bins is None
            continue
        for k, rb in r["decoded"]["bins"].items():
            assert list(bins[k]) == rb, (k, r["query"])  # order too (continuous walk order)
            assert np.allclose(np.asarray(wts[k], dtype=float).reshape(-1), r["decoded"]["weights"][k], rtol=1e-15)


def test_decode_quirks():
    for r in G.load("quirk_cases.json.gz")["cases"]:
        m = G.model(r["model"])
        pc = PredicateCompiler(m)
        q = G.unjson(r["query"])
        if r.get("error") == "KeyError":
            with pytest.raises(KeyError):
                pc.decode(q)
        elif r["kind"] == "decode":
            bins, wts = pc.decode(q)
            for k, rb in r["decoded"]["bins"].items():
                assert list(bins[k]) == rb
                assert np.allclose(wts[k], r["decoded"]["weights"][k], rtol=1e-15)


# ------------------------------------------------------------------------------------ packing
def bits_weights(m, desc, mask=None):
    """BITS rows -> dense fp64 weights per node (CPU; the inverse of PredicateCompiler.pack)."""
    bits = np.unpackbits(np.asarray(desc, dtype=np.uint8), axis=1, bitorder="little")
    W, off = [], 0
    for v in range(m.n_nodes):
        w = bits[:, off: off + int(m.card[v])].astype(np.float64)
        off += int(m.card[v])
        f = m.fan_vector(v)
        if mask is not None and f is not None:
            bit = ((mask[:, v // 32] >> np.uint32(v % 32)) & 1).astype(bool)
            w = np.where(bit[:, None], w * f[None, :], w)
        W.append(w)
    return W


def test_bits_and_sparse_forms_of_range_queries():
    """RANGE_U8 rows, BITS rows and SPARSE (CSR) entries of the same seeded queries agree; the host twin of
    the generator writes the same queries in both forms."""
    m = G.model("census")
    pc = PredicateCompiler(m)
    dm = DeviceModel(m, device=-1, specialize=False)
    desc = gen_range_queries_host(m, 5, 40, 3000, 1, 14)
    lo, hi = unpack_ranges(m, desc)
    bits = pc.pack_bits(lo, hi)
    assert bits.shape[1] == dm.desc_stride(L.DESC_BITS) and bits.shape[1] % 16 == 0
    W1, W2 = O.range_weights(m, lo, hi), bits_weights(m, bits)
    assert all(np.array_equal(a, b) for a, b in zip(W1, W2))
    assert np.array_equal(dm.bits_offset, pc.geometry()[0])
    full = pc.pack_bits(np.zeros((1, m.n_nodes), int), (m.card - 1)[None, :])
    assert np.array_equal(full.view(np.uint32)[0], dm.bits_default())
    row_off, entries = pc.pack_sparse(lo, hi)
    ro2, en2 = dm.gen_sparse_queries_host(5, 40, 3000, 1, 14)
    assert np.array_equal(row_off, ro2) and np.array_equal(entries, en2)
    k = np.diff(row_off.astype(np.int64))
    assert k.min() >= 0 and k.max() <= 14 and entries.size == k.sum()
    dm.close()


@pytest.mark.parametrize("name", ["dmv", "census", "imdb2"])
def test_pack_is_equivalent_to_decoded_weights(name):
    """Descriptors, unpacked on the CPU and pushed through the dense fp64 form, reproduce the reference."""
    m = G.model(name)
    pc = PredicateCompiler(m)
    cases = G.load("infer_cases.json.gz")[name][:120]
    decoded = [({k: list(v) for k, v in r["bins"].items()}, {k: np.asarray(v) for k, v in r["weights"].items()})
               for r in cases]
    fans = [r["fanout"] for r in cases]
    r_idx, r_desc, d_idx, d_desc, mask = pc.pack(decoded, fans)
    assert len(r_idx) + len(d_idx) == len(cases) and len(r_idx) > 0 and len(d_idx) > 0
    got = np.zeros(len(cases))
    got[r_idx] = O.dense_tree(m, bits_weights(m, r_desc, mask[r_idx]))
    off = np.concatenate([[0], np.cumsum([-(-int(c) // 4) * 4 for c in m.card])[:-1]])
    W = []
    for v in range(m.n_nodes):
        w = d_desc[:, off[v]: off[v] + m.card[v]].astype(np.float64)
        f = m.fan_vector(v)
        if f is not None:
            bit = ((mask[d_idx, v // 32] >> np.uint32(v % 32)) & 1).astype(bool)
            w = np.where(bit[:, None], w * f[None, :], w)
        W.append(w)
    got[d_idx] = O.dense_tree(m, W)
    ref = np.asarray([np.asarray(r["p"]["value"]).reshape(-1)[0] for r in cases])
    # dense descriptors carry fp32 weights: 6e-8 relative per weight
    assert np.allclose(got, ref, rtol=5e-7, atol=0)


# ------------------------------------------------------------------------------------ C ABI
def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "bayescard_b200.h")).read()
    declared = set(re.findall(r"^BC_API [^;(]*?\b(bc_[a-z0-9_]+)\(", header, flags=re.M))
    assert declared == set(L.EXPORTED_SYMBOLS), declared ^ set(L.EXPORTED_SYMBOLS)
    h = ctypes.CDLL(L.LIB_PATH)
    for sym in declared:
        assert hasattr(h, sym), sym
    assert b"sm_100a" in L.lib().bc_version()


def test_no_cpu_fallback_without_device():
    """Creating a device model on a machine without CUDA must fail loudly, never fall back."""
    try:
        import torch

        if torch.cuda.is_available():
            pytest.skip("a GPU is present")
    except ImportError:
        pass
    with pytest.raises(L.BayesCardError):
        DeviceModel(G.model("dmv"), device=0)


def test_host_only_model_codegen_and_generator():
    m = G.model("census")
    dm = DeviceModel(m, device=-1, specialize=False)
    src = dm.spec_source()
    assert "bc_spec_bits" in src and "bc_spec_dense" in src and ".target sm_100a" in src
    # one FFMA per non-zero non-root CPT entry plus the root row
    nz = sum(int(np.count_nonzero(c.astype(np.float32))) for c in m.cpts)
    assert dm.spec_ffma() == nz
    assert dm.flops_dense == m.flops_dense and dm.dense_width == sum(-(-int(c) // 4) * 4 for c in m.card)
    with pytest.raises(L.BayesCardError):
        dm.run_host(np.zeros((1, dm.desc_stride(L.DESC_RANGE_U8)), dtype=np.uint8), L.DESC_RANGE_U8)
    # generator: deterministic, per-index reproducible, k columns constrained, bounds inside the domain
    a = gen_range_queries_host(m, 7, 0, 512, 1, 14)
    b = gen_range_queries_host(m, 7, 100, 50, 1, 14)
    assert np.array_equal(a[100:150], b)
    lo, hi = unpack_ranges(m, a)
    assert np.all(lo <= hi) and np.all(hi < m.card[None, :])
    k = ((lo > 0) | (hi < m.card[None, :] - 1)).sum(axis=1)
    assert k.max() <= 14 and k.mean() > 4
    dm.close()


@pytest.mark.parametrize("name", G.MODEL_NAMES)
def test_flat_model_file_round_trip(name, tmp_path):
    """SURVEY 8f item 4: one mmap-able file instead of the pickle.  The Python reader gives back the same TreeModel;
    the C reader (bc_model_create_from_file, host-only model: no GPU needed) builds the same model as the array entry
    point -- equal code-generator hash means equal topology and equal fp32 arena bit for bit."""
    tm = G.model(name)
    path = str(tmp_path / (name + ".bcm"))
    tm.save_flat(path)
    back = TreeModel.load_flat(path)
    assert np.array_equal(back.parent, tm.parent) and np.array_equal(back.card, tm.card)
    assert all(np.array_equal(a, b) for a, b in zip(back.cpts, tm.cpts))
    assert back._meta() == tm._meta()
    assert set(back.fanouts) == set(tm.fanouts) and all(np.array_equal(back.fanouts[k], tm.fanouts[k]) for k in tm.fanouts)
    a, b = DeviceModel(tm, device=-1, specialize=False), DeviceModel.from_flat_file(path, device=-1, specialize=False)
    assert a.spec_hash() == b.spec_hash() and a.flops_dense == b.flops_dense and a.dense_width == b.dense_width
    assert np.array_equal(a.bits_offset, b.bits_offset)
    a.close()
    b.close()


def test_flat_model_file_rejects_damaged_files(tmp_path):
    tm = G.model("dmv")
    good = str(tmp_path / "dmv.bcm")
    tm.save_flat(good)
    raw = open(good, "rb").read()
    cases = {"truncated": raw[:-100], "magic": b"NOTAMODL" + raw[8:], "version": raw[:8] + (7).to_bytes(4, "little") + raw[12:],
             "short": raw[:64], "section": raw[:48] + (1 << 40).to_bytes(8, "little") + raw[56:]}
    # counts whose byte size wraps in 64 bits (4 * (2^62 + k) == 4 * k): must be rejected before they are multiplied
    arena_floats, fan_floats = int.from_bytes(raw[16:24], "little"), int.from_bytes(raw[24:32], "little")
    cases["wrap_arena"] = raw[:16] + ((1 << 62) + arena_floats).to_bytes(8, "little") + raw[24:]
    cases["wrap_fan"] = raw[:24] + ((1 << 62) + fan_floats).to_bytes(8, "little") + raw[32:]
    cases["wrap_cpt64"] = raw[:32] + ((1 << 61) + int.from_bytes(raw[32:40], "little")).to_bytes(8, "little") + raw[40:]
    for what, data in cases.items():
        bad = str(tmp_path / (what + ".bcm"))
        open(bad, "wb").write(data)
        h = ctypes.c_void_p()
        rc = L.lib().bc_model_create_from_file(-1, os.fsencode(bad), ctypes.byref(h))
        assert rc != 0 and not h.value, what
        assert L.lib().bc_last_error()
        if what != "section" and not what.startswith("wrap_"):  # (the Python reader does not touch the device-only sections)
            with pytest.raises(ValueError):
                TreeModel.load_flat(bad)
    h = ctypes.c_void_p()
    assert L.lib().bc_model_create_from_file(-1, os.fsencode(str(tmp_path / "missing.bcm")), ctypes.byref(h)) != 0


@pytest.mark.parametrize("name", ["dmv", "imdb0", "imdb3"])
def test_wsparse_packer_round_trip(name):
    """WSPARSE (include/bayescard_b200.h): the vectorised packer against a plain expansion of its own output, on the
    golden expectation cases (fractional n_distinct weights, IN lists, empty predicates) and on synthetic rows with holes."""
    m = G.model(name)
    pc = PredicateCompiler(m)
    cases = [r for r in G.load("infer_cases.json.gz")[name] if "error" not in r]
    decoded = [({k: list(v) for k, v in r["bins"].items()}, {k: np.asarray(v) for k, v in r["weights"].items()}) for r in cases]
    _, _, _, dense, _ = pc.pack(decoded, [r["fanout"] for r in cases], force_dense=True)
    rng = np.random.default_rng(3)
    holes = np.repeat(dense, 5, axis=0) * (rng.random((dense.shape[0] * 5, dense.shape[1])) < 0.8)
    off, acc = [], 0
    for v in range(m.n_nodes):
        off.append(acc)
        acc += -(-int(m.card[v]) // 4) * 4
    for rows in (dense, holes.astype(np.float32), np.zeros((0, dense.shape[1]), dtype=np.float32)):
        row_off, words = dense_to_wsparse(m, rows)
        assert row_off.dtype == np.uint32 and words.dtype == np.uint32 and row_off.size == rows.shape[0] + 1
        back = np.zeros_like(rows)
        for v in range(m.n_nodes):
            back[:, off[v]:off[v] + int(m.card[v])] = 1.0
        for q in range(rows.shape[0]):
            i = int(row_off[q])
            seen = set()
            while i < int(row_off[q + 1]):
                h = int(words[i])
                col, cont, first, cnt = h & 0x7FFF, (h >> 15) & 1, (h >> 16) & 0xFF, h >> 24
                assert col < m.n_nodes and first + cnt <= int(m.card[col]) and (cont == 1) == (col in seen)
                seen.add(col)
                if not cont:
                    back[q, off[col]:off[col] + int(m.card[col])] = 0.0
                back[q, off[col] + first:off[col] + first + cnt] = words[i + 1:i + 1 + cnt].view(np.float32)
                i += 1 + cnt
            assert i == int(row_off[q + 1])
        for v in range(m.n_nodes):
            assert np.array_equal(back[:, off[v]:off[v] + int(m.card[v])], rows[:, off[v]:off[v] + int(m.card[v])])
        if rows is dense:   # real factor lists touch a few columns: an order of magnitude fewer bytes than DENSE rows
            assert words.nbytes + row_off.nbytes < rows.nbytes / 4
    with pytest.raises(ValueError):
        dense_to_wsparse(m, np.zeros((2, dense.shape[1] + 4), dtype=np.float32))


def _wsparse_expand(m, row_off, words, nq):
    """Plain restatement of wsparse_to_dense_kernel (csrc/bc_convert.cu) for the packer tests."""
    off, acc = [], 0
    for v in range(m.n_nodes):
        off.append(acc)
        acc += -(-int(m.card[v]) // 4) * 4
    back = np.zeros((nq, acc), dtype=np.float32)
    for v in range(m.n_nodes):
        back[:, off[v]:off[v] + int(m.card[v])] = 1.0
    for q in range(nq):
        i = int(row_off[q])
        while i < int(row_off[q + 1]):
            h = int(words[i])
            col, cont, first, cnt = h & 0x7FFF, (h >> 15) & 1, (h >> 16) & 0xFF, h >> 24
            assert col < m.n_nodes and first + cnt <= int(m.card[col])
            if not cont:
                back[q, off[col]:off[col] + int(m.card[col])] = 0.0
            back[q, off[col] + first:off[col] + first + cnt] = words[i + 1:i + 1 + cnt].view(np.float32)
            i += 1 + cnt
        assert i == int(row_off[q + 1])
    return back, off


def test_wsparse_run_of_256_states():
    """A 256-state column with non-zero weights at states 0 and 255 is one run of 256 states: the 8-bit count field
    would wrap to 0, so the packer sends 255 + a one-state continuation run."""
    from bayescard_b200.synth import make_tree_model

    m = make_tree_model(3, [256, 200, 256], seed=5)
    rng = np.random.default_rng(0)
    rows = np.ones((6, 256 + 200 + 256), dtype=np.float32)
    rows[0, :256] = 0.0
    rows[0, 0] = 0.25
    rows[0, 255] = 0.5                          # the advisor's case
    rows[1, :256] = rng.random(256).astype(np.float32) + 0.1   # all 256 states weighted
    rows[2, 456:] = 0.0
    rows[2, 456 + 1] = 1.0
    rows[2, 456 + 255] = 0.125                  # run of 255: no continuation
    rows[3, 456:] = (rng.random(256) < 0.5).astype(np.float32)
    rows[3, 456] = 1.0
    rows[3, 456 + 255] = 1.0
    rows[4, 256:456] = 0.0                      # an all-zero column: run of 0 states
    row_off, words = dense_to_wsparse(m, rows)
    back, off = _wsparse_expand(m, row_off, words, rows.shape[0])
    assert np.array_equal(back, rows)
    # row 0: header(255) + 255 weights + header(cont, first 255, 1) + 1 weight
    assert int(row_off[1] - row_off[0]) == 1 + 255 + 1 + 1
    h0, h1 = int(words[0]), int(words[256])
    assert (h0 >> 24, (h0 >> 16) & 0xFF, (h0 >> 15) & 1) == (255, 0, 0)
    assert (h1 >> 24, (h1 >> 16) & 0xFF, (h1 >> 15) & 1, h1 & 0x7FFF) == (1, 255, 1, 0)


def _fused_plan(dm):
    info = np.zeros(8, dtype=np.int32)
    rc = L.lib().bc_model_fused_plan(dm._h, info.ctypes.data, None, 0)
    if rc != 0:
        return None, None, L.lib().bc_last_error().decode()
    edges = np.zeros((int(info[0]), 8), dtype=np.int32)
    L.check(L.lib().bc_model_fused_plan(dm._h, info.ctypes.data, edges.ctypes.data, edges.shape[0]))
    return info, edges, ""


@pytest.mark.parametrize("name", G.MODEL_NAMES)
def test_fused_kernel_plan_invariants(name):
    """K3's host-side plan (edge schedule + tensor-memory columns), checked without a GPU on a host-only model: every edge once,
    children before parents, exactly one `first` message per internal node, and no two allocations that are alive at the
    same edge (the accumulators; a message from its first child's edge to its own edge, the root's to the end) share a column."""
    from bayescard_b200.synth import make_tree_model

    m = G.model(name)
    dm = DeviceModel(m, device=-1, specialize=False)
    info, edges, why = _fused_plan(dm)
    assert info is not None, why
    n_edges, tmem_cols, ctas, smem, d_col, d_cols, root_col, _ = (int(x) for x in info)
    tail = None
    assert n_edges == m.n_nodes - 1 - (tail is not None) and tmem_cols == 512 and ctas == 1 and smem <= 227 * 1024
    assert d_col in (128, 192)    # the A ring (2-3 stages of 32 hi + 32 lo columns) sits below the accumulators
    child = edges[:, 0]
    assert sorted(child.tolist()) == [v for v in range(1, m.n_nodes) if v != tail]
    own = {int(v): e for e, v in enumerate(child)}
    parent = {int(v): int(m.parent[v]) for v in child}
    first_seen = {}
    for e, (v, K, N, n_pad, col_v, col_pa, first, nkb) in enumerate(edges.tolist()):
        pa = parent[v]
        assert K == int(m.card[v]) and N == int(m.card[pa]) and n_pad == -(-N // 16) * 16 and nkb == -(-K // 32)
        assert pa == 0 or pa == tail or own[pa] > e        # children before parents
        assert bool(first) == (pa not in first_seen)       # the first message overwrites, the others multiply
        first_seen.setdefault(pa, e)
        has_kids = v in first_seen
        assert (col_v >= 0) == has_kids                    # a leaf has no message in tensor memory
        if has_kids:
            assert first_seen[v] < e                       # all of v's children are done
    if tail is None:
        assert root_col == int(edges[own[next(v for v in own if parent[v] == 0)], 5])
    # column ranges alive at each edge
    spans = [("A ring + D", 0, d_col + d_cols, 0, n_edges)]
    col_of = {parent[int(r[0])]: int(r[5]) for r in edges}
    for node, start in first_seen.items():
        end = n_edges if node == 0 or node == tail else own[node]
        width = -(-int(m.card[node]) // 8) * 8
        if node == 0 and col_of[node] < 0:
            # the root's message stays in the epilogue warps' registers: all edges into the root are consecutive
            into_root = [e for e, v in enumerate(child) if parent[int(v)] == 0]
            assert into_root == list(range(into_root[0], into_root[-1] + 1)) and int(m.card[0]) <= 96
            continue
        spans.append((node, col_of[node], col_of[node] + width, start, end))
    for i, (a, a0, a1, as_, ae) in enumerate(spans):
        assert 0 <= a0 < a1 <= tmem_cols, (a, a0, a1)
        for b, b0, b1, bs, be in spans[i + 1:]:
            if as_ <= be and bs <= ae:                     # lifetimes overlap
                assert a1 <= b0 or b1 <= a0, (a, b)
    dm.close()
    # a model that does not fit is declined with a reason; a wide tree with small domains is planned
    big = DeviceModel(make_tree_model(10, 200, seed=10, dtype=np.float32), device=-1, specialize=False)
    info, _, why = _fused_plan(big)
    assert info is None and "tensor memory" in why
    big.close()
    wide = DeviceModel(make_tree_model(100, 10, seed=100, dtype=np.float32), device=-1, specialize=False)
    info, edges, why = _fused_plan(wide)
    assert info is not None and int(info[0]) == 99, why
    wide.close()


K3_PLAN_SHAPES = {
    "star_root_split": ([-1, 0, 0, 0, 0, 0, 0], [40, 50, 33, 64, 7, 50, 21]),
    "chain": ([-1, 0, 1, 2, 3], [8, 40, 60, 50, 33]),
    "root_two_internal": ([-1, 0, 0, 1, 1, 2, 2, 0], [30, 45, 52, 20, 61, 33, 17, 9]),
    "hub_112_columns": ([-1, 0, 1, 1, 1, 1], [5, 110, 40, 50, 60, 70]),
    "root_100_states": ([-1, 0, 0, 0, 3], [100, 20, 30, 40, 50]),
    "deep_hub_tail": ([-1, 0, 1, 2, 3, 3, 3, 3], [3, 12, 70, 84, 80, 9, 77, 50]),
    "two_hubs": ([-1, 0, 1, 1, 1, 0, 5, 5, 5], [6, 60, 30, 40, 50, 72, 20, 64, 33]),
    "hub_two_runs_under_a_chain": ([-1, 0, 1, 2, 2, 3, 3, 4, 4], [4, 30, 110, 20, 25, 9, 9, 8, 8]),
}


@pytest.mark.parametrize("name", list(G.MODEL_NAMES) + sorted(K3_PLAN_SHAPES))
def test_fused_kernel_step_sequence(name):
    """K3's step sequence (bc_model_fused_sequence), checked without a GPU: every edge once; the tail = the maximal suffix of edges
    that are the only message into their parent (at least one body edge stays); tail edges keep their order, never use the
    register accumulator, and the first of them comes BEFORE the first body write into the message it reads -- the end of the
    first run into that node when the node's message lives in registers, its first edge when it is updated in tensor memory
    (the bug the GPU tree-shape tests found); the nodes a tail edge reads or writes own their tensor-memory columns outright."""
    from bayescard_b200.synth import make_tree_model

    if name in K3_PLAN_SHAPES:
        parent, cards = K3_PLAN_SHAPES[name]
        m = make_tree_model(len(cards), cards, seed=1, dtype=np.float32, parent=parent)
    else:
        m = G.model(name)
    dm = DeviceModel(m, device=-1, specialize=False)
    info, edges, why = _fused_plan(dm)
    if info is None:
        dm.close()
        pytest.skip(f"K3 declines this model: {why}")
    n_edges = int(info[0])
    seq, flags = np.zeros(n_edges, dtype=np.uint8), np.zeros(n_edges, dtype=np.uint8)
    n_tail = C.c_int32()
    L.check(L.lib().bc_model_fused_sequence(dm._h, seq.ctypes.data, flags.ctypes.data, n_edges, C.byref(n_tail)))
    n_tail = n_tail.value
    n_body = n_edges - n_tail
    child = edges[:, 0].tolist()
    par = [int(m.parent[v]) for v in child]
    n_msgs = {p: par.count(p) for p in set(par)}
    assert sorted(int(x) & 127 for x in seq) == list(range(n_edges))
    # the tail: maximal suffix of only-message edges, one body edge at least
    want_tail = 0
    while want_tail < n_edges - 1 and n_msgs[par[n_edges - 1 - want_tail]] == 1:
        want_tail += 1
    assert n_tail == want_tail and n_body >= 1
    pos = {int(x) & 127: i for i, x in enumerate(seq)}
    for e in range(n_edges):
        assert bool(int(seq[pos[e]]) & 128) == (e >= n_body)
        run_first = e == 0 or par[e - 1] != par[e]
        run_last = e == n_edges - 1 or par[e + 1] != par[e]
        assert bool(flags[e] & 1) == run_first and bool(flags[e] & 2) == run_last
        if e >= n_body:
            assert not flags[e] & 4                     # a tail edge never touches the register accumulator
        else:
            assert bool(flags[e] & 4) == (int(edges[e, 3]) <= 96)
    body_order = [int(x) for x in seq if not int(x) & 128]
    tail_order = [int(x) & 127 for x in seq if int(x) & 128]
    assert body_order == list(range(n_body)) and tail_order == list(range(n_body, n_edges))
    if n_tail:
        hub = child[n_body]                             # the node whose message the first tail edge reads
        into_hub = [e for e in range(n_body) if par[e] == hub]
        assert into_hub, "the node below the chain has children (else it would be part of the chain)"
        in_regs = bool(flags[into_hub[0]] & 4)
        first_write = next(e for e in into_hub if flags[e] & 2) if in_regs else into_hub[0]
        assert pos[n_body] < pos[first_write], (name, seq.tolist())
        # pinned nodes own their columns: no other message overlaps them
        pinned = {child[e] for e in range(n_body, n_edges)} | {par[e] for e in range(n_body, n_edges)}
        col_of = {}
        for e in range(n_edges):
            if int(edges[e, 4]) >= 0:
                col_of[child[e]] = int(edges[e, 4])
            if int(edges[e, 5]) >= 0:
                col_of[par[e]] = int(edges[e, 5])
        width = lambda v: -(-int(m.card[v]) // 8) * 8
        for v in pinned:
            if v not in col_of:
                continue                                # (the root in registers)
            for u, c in col_of.items():
                if u != v:
                    assert col_of[v] + width(v) <= c or c + width(u) <= col_of[v], (name, v, u)
    dm.close()


def test_shard_split():
    assert ShardedModel.split(10, 4) == [(0, 2), (2, 4), (4, 6), (6, 10)]
    assert ShardedModel.split(3, 8)[-1] == (0, 3)


def test_reference_arm_query_stream_equals_the_c_generator():
    """bench.py --impl reference regenerates the seeded query stream in pure Python (baseline/ref_runner.py) so that the
    reference arm loads none of this repository's native code: it must be the stream the C generator produces."""
    import sys

    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from baseline import ref_runner as RR
    from bayescard_b200.engine import gen_range_queries_host

    for name, first, kmin, kmax in (("census", 0, 1, 14), ("census", 123456789012, 1, 14), ("dmv", 7, 1, 5), ("imdb3", 99, 0, 9)):
        m = G.model(name)
        lo, hi = RR.gen_ranges([int(c) for c in m.card], 0, first, 200, kmin, kmax)
        lo2, hi2 = unpack_ranges(m, gen_range_queries_host(m, 0, first, 200, kmin, kmax))
        assert np.array_equal(lo, lo2) and np.array_equal(hi, hi2), name


def test_staged_reference_reproduces_the_golden_probabilities():
    """baseline/_ref (the byte-for-byte staged reference that bench.py times) against the committed golden vectors."""
    import sys

    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from baseline import ref_runner as RR

    if not RR.available():
        pytest.skip("baseline/_ref not staged on this machine")
    bn = RR.load_bn("dmv")
    rows = [r for r in G.load("dmv_workload.json.gz")["queries"] if r.get("decoded")][:60]
    for r in rows:
        q = {k: list(v) for k, v in r["decoded"]["bins"].items()}
        nd = {k: np.asarray(v) for k, v in r["decoded"]["weights"].items()}
        p = bn.query(q, n_distinct=nd, return_prob=True)[0]
        want = np.asarray(r["card"]["value"]).reshape(-1)[0] / bn.nrows
        assert abs(float(np.asarray(p).reshape(-1)[0]) - want) <= 1e-12 * max(abs(want), 1e-300)


@pytest.mark.parametrize("name", ["census", "dmv", "imdb3"])
def test_packed_wire_format_round_trip(name):
    """PACKED (include/bayescard_b200.h): the host packer against a plain bit-stream decoder -- same columns, bounds and
    IN-list continuation as the SPARSE entries it was made from; geometry; refusals."""
    m = G.model(name)
    dm = DeviceModel(m, device=-1, specialize=False)
    w, cb, sb = dm.packed_geometry()
    assert w == cb + 2 * sb and (1 << cb) >= m.n_nodes and (1 << sb) >= int(m.card.max()) and (1 << (cb - 1)) < max(m.n_nodes, 2)
    n = 1000
    row_off, entries = dm.gen_sparse_queries_host(5, 17, n, 0, min(14, m.n_nodes))
    # IN lists: duplicate some entries as continuation entries (same column, cont bit) right behind their first
    rng = np.random.default_rng(1)
    ro2, en2 = [0], []
    for q in range(n):
        for e in entries[row_off[q]:row_off[q + 1]]:
            en2.append(int(e))
            if rng.random() < 0.2:
                col, lo, hi = int(e) & 0x7FFF, (int(e) >> 16) & 0xFF, int(e) >> 24
                en2.append(col | (1 << 15) | (min(hi, lo + 1) << 16) | (hi << 24))
        ro2.append(len(en2))
    row_off, entries = np.asarray(ro2, dtype=np.uint32), np.asarray(en2, dtype=np.uint32)
    klen, blk, payload = dm.pack_sparse(row_off, entries)
    assert klen.dtype == np.uint8 and klen.size == n and blk.size == (n + 127) // 128 + 1
    assert np.array_equal(klen, np.diff(row_off.astype(np.int64))) and int(blk[-1]) == entries.size
    assert payload.nbytes == ((entries.size * w + 31) // 32 + 2) * 4
    words = np.frombuffer(payload.tobytes(), dtype=np.uint32)
    e = 0
    for q in range(n):
        if q % 128 == 0:
            assert int(blk[q // 128]) == e
        prev = -1
        for x in entries[row_off[q]:row_off[q + 1]]:
            bit = e * w
            v = ((int(words[bit >> 5]) | (int(words[(bit >> 5) + 1]) << 32)) >> (bit & 31)) & ((1 << w) - 1)
            col, lo, hi = v & ((1 << cb) - 1), (v >> cb) & ((1 << sb) - 1), v >> (cb + sb)
            assert (col, lo, hi) == (int(x) & 0x7FFF, (int(x) >> 16) & 0xFF, int(x) >> 24)
            assert ((int(x) >> 15) & 1) == (col == prev)
            prev = col
            e += 1
    # an ungrouped continuation entry is not representable
    bad = np.asarray([3 | (1 << 15) | (1 << 24)], dtype=np.uint32)
    with pytest.raises(L.BayesCardError):
        dm.pack_sparse(np.asarray([0, 1], dtype=np.uint32), bad)
    # empty batch
    k0, b0, p0 = dm.pack_sparse(np.zeros(1, dtype=np.uint32), np.zeros(0, dtype=np.uint32))
    assert k0.size == 0 and b0.tolist() == [0] and p0.nbytes == 8
    dm.close()
