"""GROUP BY one column: bc_marginal_batch (specialised marginal kernel and expansion), Bayescard_BN.groupby*, the SQL
front end, against the fp64 oracle (groupby_oracle.marginal = oracle.dense_tree with the target's weights masked to each
state in turn).  Tolerance 1e-5 relative, as the other GPU parity tests."""
import os
import re

import numpy as np
import pytest

import golden_util as G
import groupby_oracle as GO
from bayescard_b200 import _lib as L
from bayescard_b200.decode import PredicateCompiler, unpack_ranges
from bayescard_b200.engine import DeviceModel, launch_count
from bayescard_b200.model import Bayescard_BN
from bayescard_b200.sql_front import parse_groupby_single_table, parse_query_single_table
from oracle import bayescard_oracle as O

RTOL = 1e-5


def assert_close(got, ref, what=""):
    got, ref = np.asarray(got, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    err = np.abs(got - ref) / np.maximum(np.abs(ref), 1e-300)
    err[(ref == 0) & (got == 0)] = 0
    assert err.max() <= RTOL, (what, float(err.max()), np.unravel_index(int(err.argmax()), err.shape))


def targets_of(name):
    m = G.model(name)
    return list(range(m.n_nodes)) if name == "dmv" else sorted(set(GO.tree_targets(m).values()))


# ------------------------------------------------------------------------------------ oracle (no GPU)
@pytest.mark.parametrize("seed", range(12))
def test_oracle_equals_brute_force_on_tiny_trees(seed):
    from bayescard_b200.synth import make_tree_model

    rng = np.random.default_rng(seed)
    n = int(rng.integers(1, 7))
    tm = make_tree_model(n, rng.integers(1, 5, size=n), seed=seed)
    W = [rng.random(int(c)) * (rng.random(int(c)) < 0.8) for c in tm.card]
    for t in range(n):
        got = GO.marginal(tm, W, t)
        assert np.allclose(got, GO.brute_force(tm, W, t), rtol=1e-12, atol=0)
        assert np.isclose(got.sum(), O.dense_tree(tm, W), rtol=1e-12)


def test_oracle_bins_sum_to_dense_tree_on_batches():
    m = G.model("dmv")
    dm = DeviceModel(m, device=-1, specialize=False)
    lo, hi = unpack_ranges(m, dm.gen_range_queries_host(3, 0, 64, 1, 6))
    W = O.range_weights(m, lo, hi)
    ref = O.dense_tree(m, W)
    for t in range(m.n_nodes):
        assert np.allclose(GO.marginal(m, W, t).sum(axis=1), ref, rtol=1e-12, atol=0)
    dm.close()


# ------------------------------------------------------------------------------------ code generator (no GPU)
def test_marginal_source_on_host_only_models():
    lib = L.lib()
    for name in ("census", "dmv"):
        m = G.model(name)
        dm = DeviceModel(m, device=-1, specialize=False)
        nz = sum(int(np.count_nonzero(np.asarray(c, dtype=np.float32))) for c in m.cpts)
        hashes = set()
        for t in range(m.n_nodes):
            src = dm.marginal_source(t)
            assert src == dm.marginal_source(t), "generator is not deterministic"
            assert "bc_marg_bits" in src and "bc_marg_dense" in src and ".target sm_100a" in src
            assert f"target: {t}  card: {int(m.card[t])}" in src
            # one FMA-pipe instruction per non-zero CPT entry of the whole tree, as in the spec module
            assert re.search(r"BC_SPEC_FFMA=(\d+)", src).group(1) == str(nz)
            hashes.add(dm.marginal_hash(t))
        assert len(hashes) == m.n_nodes and dm.spec_hash() not in hashes
        # out-of-range targets: BC_EINVAL from the library, ValueError from Python
        for bad in (-1, m.n_nodes):
            assert lib.bc_model_marginal_source(dm._h, bad, None, 0) == -1
            assert lib.bc_model_marginal_hash(dm._h, bad) == 0
            assert lib.bc_marginal_batch(dm._h, None, 1, L.DESC_BITS, bad, None, L.KERNEL_AUTO, None) == -1
            with pytest.raises(ValueError):
                dm.marginal_source(bad)
        # a host-only model cannot run, RANGE rows are refused
        assert lib.bc_marginal_batch(dm._h, None, 0, L.DESC_BITS, 0, None, L.KERNEL_AUTO, None) == -1
        with pytest.raises(L.BayesCardError):
            dm.run_marginal_host(np.zeros((1, dm.desc_stride(L.DESC_BITS)), dtype=np.uint8), L.DESC_BITS, 0)
        with pytest.raises(ValueError):
            dm.specialize_marginal(m.n_nodes)
        dm.close()


@pytest.mark.parametrize("name", ["dmv", "synthetic"])
def test_generated_marginal_arithmetic_on_the_host(name):
    """The generated bc_marg_bits / bc_marg_dense bodies, interpreted on the host in fp32 for a few rows, against the fp64
    oracle: every target of DMV and of a synthetic tree with exact zeros in its CPTs."""
    from bayescard_b200.synth import make_tree_model, random_range_queries

    if name == "dmv":
        m = G.model("dmv")
    else:
        m = make_tree_model(9, [3, 7, 5, 2, 6, 4, 8, 3, 5], seed=4, dtype=np.float32)
        m.cpts[3][0, :] = 0.0   # an all-zero row and scattered exact zeros
        m.cpts[6][:, 1] = np.where(np.arange(8) % 2 == 0, 0.0, m.cpts[6][:, 1])
    dm = DeviceModel(m, device=-1, specialize=False)
    pc = PredicateCompiler(m)
    nq = 3
    lo, hi = random_range_queries(m, nq, seed=1, kmax=m.n_nodes)
    bits = pc.pack_bits(lo, hi)
    W = O.range_weights(m, lo, hi)
    rng = np.random.default_rng(2)
    Wd = [(np.asarray(w) * (0.25 + 0.75 * rng.random((nq, 1)))).astype(np.float32) for w in W]
    dense = np.zeros((nq, dm.dense_width), dtype=np.float32)
    for v in range(m.n_nodes):
        o = int(dm.dense_offset[v])
        dense[:, o:o + int(m.card[v])] = Wd[v]
    Wd = [w.astype(np.float64) for w in Wd]
    for t in range(m.n_nodes):
        src = dm.marginal_source(t)
        ref, ref_d = GO.marginal(m, W, t), GO.marginal(m, Wd, t)
        for q in range(nq):
            assert_close(GO.interpret(src, "bc_marg_bits", bits[q].tobytes()), ref[q], (name, t, q, "bits"))
            assert_close(GO.interpret(src, "bc_marg_dense", dense[q].tobytes()), ref_d[q], (name, t, q, "dense"))
    dm.close()


def test_marginal_modules_assemble_for_sm_100a(tmp_path):
    """Every target of DMV and IMDB 0-4, and the root, deepest, widest and a leaf of Census, through ptxas -arch=sm_100a."""
    for name in G.MODEL_NAMES:
        m = G.model(name)
        nodes = targets_of(name) if name == "census" else range(m.n_nodes)
        GO.assemble_marginals(m, nodes, str(tmp_path / name))
        assert len(os.listdir(tmp_path / name)) == len(set(nodes)), name


# ------------------------------------------------------------------------------------ SQL front end + value selection (no GPU)
def _bn(name):
    return Bayescard_BN(G.model(name), device=-1, infer_algo="exact-jit")


def test_parse_groupby_single_table():
    bn = _bn("dmv")
    col = next(c for c in bn.tree.infer_names if bn.attr_type[c] != "continuous")
    rows = G.load("dmv_workload.json.gz")["queries"]
    sql = rows[0]["sql"]
    where = sql.split(" WHERE ")[1].rstrip(";").strip()
    q, c = parse_groupby_single_table(f"SELECT {col}, COUNT(*) FROM dmv WHERE {where} GROUP BY {col}", bn)
    assert c == col and q == parse_query_single_table(sql, bn)
    q, c = parse_groupby_single_table(f"select COUNT(*), {col} from dmv group by {col};", bn)
    assert c == col and q == {}
    with pytest.raises(ValueError):   # two grouping columns
        parse_groupby_single_table(f"SELECT {col}, COUNT(*) FROM dmv GROUP BY {col}, {bn.tree.infer_names[1]}", bn)
    with pytest.raises(ValueError):   # unknown column
        parse_groupby_single_table("SELECT nope, COUNT(*) FROM dmv GROUP BY nope", bn)
    with pytest.raises(ValueError):   # select list is not (column, COUNT(*))
        parse_groupby_single_table(f"SELECT {bn.tree.infer_names[1]}, COUNT(*) FROM dmv GROUP BY {col}", bn)
    with pytest.raises(ValueError):   # no GROUP BY
        parse_groupby_single_table(sql, bn)


@pytest.mark.parametrize("name", ["dmv", "census"])
def test_value_selection_agrees_with_the_decoder(name):
    bn = _bn(name)
    pc = PredicateCompiler(bn.tree)
    checked = 0
    for r in G.load(f"{name}_workload.json.gz")["queries"]:
        for attr, val in parse_query_single_table(r["sql"], bn).items():
            col = pc.cols[attr]
            if col.kind == "continuous" or col.enc is None:
                continue
            sel = pc.select_values(attr, val)
            b, w = pc.decode({attr: val})
            if b is None:
                assert sel is None or not sel.any(), (attr, val)
                continue
            assert sel is not None
            keys = list(col.pair)
            per_bin = {}
            for k, s in zip(keys, sel):
                if s:
                    bb, ww = col.pair[k]
                    per_bin[int(bb)] = per_bin.get(int(bb), 0) + ww
            assert sorted(per_bin) == sorted(int(x) for x in b[attr]), (attr, val)
            for x, wx in zip(b[attr], np.asarray(w[attr]).reshape(-1)):
                assert np.isclose(min(per_bin[int(x)], 1), wx, rtol=1e-12, atol=0), (attr, val, x)
            checked += 1
    assert checked > 50


# ------------------------------------------------------------------------------------ GPU
_dm = {}


@pytest.fixture(scope="module")
def marg_cache():
    """The marginal cubins of every model and target the GPU tests use, assembled in parallel into the library's cache
    directory (ptxas, as the ahead-of-time spec build does; the driver JIT would compile them one at a time)."""
    for name in G.MODEL_NAMES:
        GO.assemble_marginals(G.model(name), targets_of(name), L.SPEC_CACHE_DIR)
    return L.SPEC_CACHE_DIR


def spec_model(name, cache) -> DeviceModel:
    if name not in _dm:
        dm = DeviceModel(G.model(name), device=0, specialize=False)
        for t in targets_of(name):
            assert dm.specialize_marginal(t, cache), dm.marginal_error.get(t)
        _dm[name] = dm
    return _dm[name]


def _cases(name):
    """infer_cases (bins, fractional weights) plus, for DMV and Census, the workload's predicates decoded."""
    m = G.model(name)
    cases = [r for r in G.load("infer_cases.json.gz")[name] if "error" not in r]
    decoded = [({k: list(v) for k, v in r["bins"].items()}, {k: np.asarray(v) for k, v in r["weights"].items()}) for r in cases]
    if name in ("dmv", "census"):
        bn = _bn(name)
        pc = PredicateCompiler(m)
        for r in G.load(f"{name}_workload.json.gz")["queries"]:
            b, w = pc.decode(parse_query_single_table(r["sql"], bn))
            if b is not None:
                decoded.append((b, w))
    decoded.append(({}, {}))   # no predicate at all
    return decoded


def _weights(m, decoded, idx):
    per = [O.dense_weights(m, decoded[i][0], decoded[i][1]) for i in idx]
    return [np.stack([p[v] for p in per]) for v in range(m.n_nodes)]


@pytest.mark.gpu
@pytest.mark.parametrize("name", G.MODEL_NAMES)
def test_marginal_kernels_match_the_oracle(name, marg_cache):
    m = G.model(name)
    dm = spec_model(name, marg_cache)
    plain = DeviceModel(m, device=0, specialize=False)   # no marginal module attached: AUTO expands
    pc = PredicateCompiler(m)
    decoded = _cases(name)
    for force_dense in (False, True):
        b_idx, b_desc, d_idx, d_desc, _ = pc.pack(decoded, force_dense=force_dense)
        for idx, desc, fmt in ((b_idx, b_desc, L.DESC_BITS), (d_idx, d_desc, L.DESC_DENSE_F32)):
            if not len(idx):
                continue
            W = _weights(m, decoded, idx)
            total = plain.run_host(desc, fmt, None, L.KERNEL_GENERIC)
            for t in targets_of(name):
                ref = GO.marginal(m, W, t)
                for kernel, model in ((L.KERNEL_SPEC, dm), (L.KERNEL_GENERIC, plain), (L.KERNEL_AUTO, plain)):
                    got = model.run_marginal_host(desc, fmt, t, kernel)
                    assert got.shape == ref.shape
                    assert_close(got, ref, (name, t, fmt, kernel, force_dense))
                    if kernel == L.KERNEL_SPEC:
                        assert_close(got.astype(np.float64).sum(axis=1), total, (name, t, fmt, "sum over bins"))
    plain.close()


@pytest.mark.gpu
def test_spec_marginal_is_one_launch_and_dispatch(marg_cache):
    import torch

    m = G.model("dmv")
    dm = spec_model("dmv", marg_cache)
    n, t = 5000, 2
    desc = torch.empty((n, dm.desc_stride(L.DESC_RANGE_U8)), dtype=torch.uint8, device="cuda:0")
    bits = torch.empty((n, dm.desc_stride(L.DESC_BITS)), dtype=torch.uint8, device="cuda:0")
    out = torch.empty((n, int(m.card[t])), dtype=torch.float32, device="cuda:0")
    st = torch.cuda.current_stream().cuda_stream
    dm.gen_range_queries_device(5, 0, n, 1, 8, desc.data_ptr(), st)
    dm.convert_device(desc.data_ptr(), L.DESC_RANGE_U8, bits.data_ptr(), L.DESC_BITS, n, st)
    torch.cuda.synchronize()
    for kernel in (L.KERNEL_SPEC, L.KERNEL_AUTO):
        before = launch_count()
        dm.run_marginal_device(bits.data_ptr(), n, L.DESC_BITS, t, out.data_ptr(), kernel, st)
        assert launch_count() - before == 1, kernel
    torch.cuda.synchronize()
    spec = out.cpu().numpy().copy()
    dm.run_marginal_device(bits.data_ptr(), n, L.DESC_BITS, t, out.data_ptr(), L.KERNEL_GENERIC, st)
    torch.cuda.synchronize()
    assert_close(spec, out.cpu().numpy(), "spec vs expansion on device buffers")
    # n == 0: no launch; RANGE rows refused; SPEC without a module: BC_ECOMPILE
    before = launch_count()
    dm.run_marginal_device(0, 0, L.DESC_BITS, t, 0, L.KERNEL_SPEC, st)
    assert launch_count() == before
    with pytest.raises(L.BayesCardError):
        dm.run_marginal_device(desc.data_ptr(), n, L.DESC_RANGE_U8, t, out.data_ptr(), L.KERNEL_AUTO, st)
    plain = DeviceModel(m, device=0, specialize=False)
    rc = L.lib().bc_marginal_batch(plain._h, bits.data_ptr(), n, L.DESC_BITS, t, out.data_ptr(), L.KERNEL_SPEC, None)
    assert rc == -4
    # the driver-JIT route (no cache directory) attaches the same kernel
    assert plain.specialize_marginal(t, ""), plain.marginal_error.get(t)
    plain.run_marginal_device(bits.data_ptr(), n, L.DESC_BITS, t, out.data_ptr(), L.KERNEL_SPEC, st)
    torch.cuda.synchronize()
    assert np.array_equal(out.cpu().numpy(), spec)
    plain.close()


@pytest.mark.gpu
@pytest.mark.parametrize("target", [5, 3])
def test_expansion_on_a_model_without_spec_module(target):
    """A synthetic tree with a 257-state column (beyond K3 and the 8-bit wire formats) and no specialised module: AUTO
    serves GROUP BY through the expansion; BITS and fractional DENSE rows."""
    from bayescard_b200.synth import make_tree_model, random_range_queries

    cards = [7, 130, 33, 257, 64, 5, 90, 200, 17, 128, 40, 3]
    tm = make_tree_model(len(cards), cards, seed=12, dtype=np.float32)
    dm2 = DeviceModel(tm, device=0, specialize=False)
    lo, hi = random_range_queries(tm, 700, seed=2, kmax=6)
    pc = PredicateCompiler(tm)
    W = O.range_weights(tm, lo, hi)
    ref = GO.marginal(tm, W, target)
    assert_close(dm2.run_marginal_host(pc.pack_bits(lo, hi), L.DESC_BITS, target, L.KERNEL_AUTO), ref, "BITS via AUTO")
    rng = np.random.default_rng(1)
    dense = np.full((len(lo), dm2.dense_width), np.nan, dtype=np.float32)
    Wd = []
    for v in range(tm.n_nodes):
        wv = (W[v] * (0.25 + 0.75 * rng.random((len(lo), 1)))).astype(np.float32)
        Wd.append(wv.astype(np.float64))
        o = int(dm2.dense_offset[v])
        dense[:, o:o + int(tm.card[v])] = wv
    assert_close(dm2.run_marginal_host(dense, L.DESC_DENSE_F32, target, L.KERNEL_AUTO), GO.marginal(tm, Wd, target), "DENSE via AUTO")
    dm2.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["dmv", "census"])
def test_groupby_matches_per_value_queries(name):
    m = G.model(name)
    bn = Bayescard_BN.load(os.path.join(G.GOLD, "models", name + ".npz"), device=0, infer_algo="exact-jit")
    bn.init_inference_method()
    pc = bn.infer_machine.compiler
    # the two categorical columns with the most values (<= 100, to keep the per-value oracle loop short)
    cols = [c for c in m.infer_names if pc.cols[c].enc is not None and len(pc.cols[c].pair) <= 100]
    cols = sorted(cols, key=lambda c: -len(pc.cols[c].pair))[:2]
    rows = G.load(f"{name}_workload.json.gz")["queries"][:40]
    queries = [parse_query_single_table(r["sql"], bn) for r in rows] + [{}]
    for col in cols:
        GO.assemble_marginals(m, [m.infer_names.index(col)], L.SPEC_CACHE_DIR)
        keys, est = bn.groupby_batch(queries, col)
        assert bn.infer_machine._single.specialize_marginal(m.infer_names.index(col))   # served by the specialised kernel
        assert est.shape == (len(queries), len(keys)) and keys == list(pc.cols[col].pair)
        for i, q in enumerate(queries):
            sel = pc.select_values(col, q[col]) if col in q else np.ones(len(keys), dtype=bool)
            rest = {k: v for k, v in q.items() if k != col}
            ref = np.zeros(len(keys))
            if sel is not None:
                for j, k in enumerate(keys):
                    if sel[j]:
                        ref[j] = float(np.asarray(O.bn_query(m, {**rest, col: k})).reshape(-1)[0])
            assert_close(est[i], ref, (name, col, i))
        d = bn.groupby(queries[-1], col)   # no predicate: the column's marginal, summing to nrows
        assert np.isclose(sum(d.values()), m.nrows, rtol=1e-5)
        assert bn.groupby_batch([], col)[1].shape == (0, len(keys))
        other = next(c for c in cols if c != col)
        _, ez = bn.groupby_batch([{col: "no such value"}, {other: "no such value"}], col)   # undecodable: zero rows
        assert not ez.any()
    with pytest.raises(ValueError):
        bn.groupby_batch(queries[:1], "no_such_column")
    sql = [f"SELECT {cols[0]}, COUNT(*) FROM {name} GROUP BY {cols[0]}", f"SELECT {cols[1]}, COUNT(*) FROM {name} GROUP BY {cols[1]}"]
    res = bn.groupby_sql_batch(sql)
    for r, c in zip(res, cols[:2]):
        assert list(r.values()) == list(bn.groupby_batch([{}], c)[1][0])
    bn.close()


@pytest.mark.gpu
def test_groupby_continuous_column_bins_sum_to_query():
    import copy

    m = G.model("imdb3")
    bn = Bayescard_BN(m, device=0, infer_algo="exact-jit", specialize=False)
    bn.init_inference_method()
    col = next(c for c in m.infer_names if m.attr_type[c] == "continuous")
    qs = [G.unjson(r["query"]) for r in G.load("imdb_cases.json.gz")["imdb3"] if "error" not in r]
    qs = [q for q in qs if any(k in m._index for k in q)][:60]
    # a range from the middle of bin 2 to the middle of bin 5: the predicate stays in the descriptor with its coverage
    # weights (0.5, 1, 1, 0.5), so the other bins are 0 and bins 2..5 are those weights times the column's marginal
    edges = m.mapping[col]
    qs.append({col: ((edges[2][0] + edges[2][1]) / 2, (edges[5][0] + edges[5][1]) / 2)})
    keys, est = bn.groupby_batch(qs, col, return_prob=True)
    assert keys == [tuple(e) for e in edges]
    ref = bn.query_batch([copy.deepcopy(q) for q in qs], return_prob=True)
    assert_close(est.sum(axis=1), ref, "continuous bins sum to query")
    full = bn.groupby({}, col, return_prob=True)
    marginal = np.asarray([full[k] for k in keys])
    cover = np.zeros(len(keys))
    cover[2:6] = [0.5, 1.0, 1.0, 0.5]
    assert_close(est[-1], cover * marginal, "range predicate on the grouping column")
    bn.close()
