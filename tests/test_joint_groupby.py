"""GROUP BY two columns: ``bc_joint_marginal_batch``, its generated joint module and its expansion, and the Python surface
(``Bayescard_BN.groupby_batch`` with a pair of columns, ``parse_groupby_single_table``), against the fp64 oracle."""
from __future__ import annotations

import copy
import itertools
import os
import re
import subprocess

import numpy as np
import pytest

import golden_util as G
import groupby_oracle as GO
import join_groupby_oracle as JO
import joint_groupby_oracle as JG
from bayescard_b200 import _lib as L
from bayescard_b200.decode import PredicateCompiler
from bayescard_b200.engine import DeviceModel, launch_count
from bayescard_b200.model import Bayescard_BN
from bayescard_b200.sql_front import parse_groupby_single_table
from oracle import bayescard_oracle as O

RTOL = 1e-5
CAP = 32768   # BC_JOINT_MAX_FFMA
EINVAL, ECOMPILE, ELIMIT = -1, -4, -5


def assert_close(got, ref, what="", rtol=RTOL):
    got, ref = np.atleast_1d(np.asarray(got, dtype=np.float64)), np.atleast_1d(np.asarray(ref, dtype=np.float64))
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    err = np.abs(got - ref) / np.maximum(np.abs(ref), 1e-300)
    err[(ref == 0) & (got == 0)] = 0
    assert err.max() <= rtol, (what, float(err.max()), np.unravel_index(int(err.argmax()), err.shape))


def _depth(m):
    d = [0] * m.n_nodes
    for v in range(1, m.n_nodes):
        d[v] = d[int(m.parent[v])] + 1
    return d


def census_pairs(m):
    """Siblings, ancestor/descendant both ways, LCA = root with the two deepest leaves of different root subtrees, the root
    with a leaf, and the widest pair."""
    d = _depth(m)
    kids = {}
    for v in range(1, m.n_nodes):
        kids.setdefault(int(m.parent[v]), []).append(v)
    sib = next(tuple(k[:2]) for k in kids.values() if len(k) >= 2)
    child = max(range(1, m.n_nodes), key=lambda v: d[v])
    anc = int(m.parent[int(m.parent[child])]) if d[child] >= 2 else int(m.parent[child])
    top = {}
    for v in range(1, m.n_nodes):
        t = v
        while int(m.parent[t]) != 0:
            t = int(m.parent[t])
        if t not in top or d[v] > d[top[t]]:
            top[t] = v
    deep = sorted(top.values(), key=lambda v: -d[v])[:2]
    inner = set(int(p) for p in m.parent[1:])
    leaf = max((v for v in range(m.n_nodes) if v not in inner), key=lambda v: d[v])
    wide = sorted(range(m.n_nodes), key=lambda v: -int(m.card[v]))[:2]
    return [sib, (anc, child), (child, anc), tuple(deep), (0, leaf), (wide[0], wide[1])]


def _pairs_under_cap(dm, m, ordered=False):
    out = []
    for a, b in (itertools.permutations(range(m.n_nodes), 2) if ordered else itertools.combinations(range(m.n_nodes), 2)):
        if L.lib().bc_model_joint_source(dm._h, a, b, None, 0) > 0:
            out.append((a, b))
    return out


def _synthetic_fan_model():
    from bayescard_b200.synth import make_tree_model

    m = make_tree_model(8, [3, 5, 1, 4, 2, 6, 3, 4], seed=9, dtype=np.float32)
    m.cpts[3][0, :] = 0.0   # an all-zero row and scattered exact zeros
    m.cpts[5][:, 0] = np.where(np.arange(6) % 2 == 0, 0.0, m.cpts[5][:, 0])
    rng = np.random.default_rng(3)
    for v in (0, 3, 5, 7):
        f = rng.uniform(0.5, 20.0, int(m.card[v]))
        if v == 5:
            f[1] = 0.0
        m.fanouts[m.infer_names[v]] = f
    return m


def _rows(m, dm, nq, seed, kmax=None):
    """BITS rows of random range queries, DENSE rows with fractional weights, and their fp64 weights."""
    from bayescard_b200.synth import random_range_queries

    pc = PredicateCompiler(m)
    lo, hi = random_range_queries(m, nq, seed=seed, kmax=kmax or m.n_nodes)
    bits = pc.pack_bits(lo, hi)
    rng = np.random.default_rng(seed)
    W = O.range_weights(m, lo, hi)
    Wd = [(np.asarray(w) * (0.25 + 0.75 * rng.random((nq, 1)))).astype(np.float32) for w in W]
    dense = np.zeros((nq, dm.dense_width), dtype=np.float32)
    for v in range(m.n_nodes):
        o = int(dm.dense_offset[v])
        dense[:, o:o + int(m.card[v])] = Wd[v]
    return lo, hi, bits, dense, W, [w.astype(np.float64) for w in Wd]


def _interp(src, entry, row, m, a, b, mask=None):
    return JO.interpret_masked(src, entry, row, mask).reshape(int(m.card[a]), int(m.card[b]))


# ------------------------------------------------------------------------------------ oracle (no GPU)
@pytest.mark.parametrize("seed", range(4))
def test_oracle_against_brute_force(seed):
    from bayescard_b200.synth import make_tree_model

    cards = [[2, 3, 1, 2, 3], [3, 1, 2, 2, 2], [1, 2, 3, 2, 1], [2, 2, 2, 3, 2]][seed]
    m = make_tree_model(5, cards, seed=seed, dtype=np.float64)
    m.cpts[1] = np.asarray(m.cpts[1]).copy()
    m.cpts[1].reshape(int(m.card[1]), -1)[0, :] = 0.0   # exact zeros
    rng = np.random.default_rng(seed)
    W = [rng.random(int(c)) * (rng.random(int(c)) < 0.8) for c in m.card]
    total = O.dense_tree(m, W)
    for a, b in itertools.permutations(range(5), 2):
        J = JG.joint(m, W, a, b)
        assert_close(J, JG.brute_force(m, W, a, b), (a, b))
        assert_close(J.sum(axis=1), GO.marginal(m, W, a), (a, b, "sum over j"))
        assert_close(J.sum(axis=0), GO.marginal(m, W, b), (a, b, "sum over i"))
        assert_close(J.sum(), total, (a, b, "total"))


# ------------------------------------------------------------------------------------ code generator (no GPU)
def test_sources_headers_and_hashes():
    for name in ("dmv", "census"):
        m = G.model(name)
        dm = DeviceModel(m, device=-1, specialize=False)
        spec_src = dm.spec_source()
        others = {dm.spec_hash()} | {dm.marginal_hash(v) for v in range(m.n_nodes)}
        pairs = _pairs_under_cap(dm, m) if name == "dmv" else census_pairs(m)
        hashes = set()
        for a, b in pairs:
            src = dm.joint_source(a, b)
            assert src == dm.joint_source(a, b), "generator is not deterministic"
            assert ".target sm_100a" in src and ".visible .entry bc_joint_bits(" in src and ".visible .entry bc_joint_dense(" in src
            assert f"bc_joint_meta[4] = {{{re.search(r'BC_SPEC_THREADS=(\d+)', src).group(1)}, {a}, {b}, 1}}" in src
            X = int(re.search(r"  X: (\d+)", src).group(1))
            assert X in (a, b)
            assert int(re.search(r"BC_SPEC_FFMA=(\d+)", src).group(1)) == JG.joint_ffma(m, a, b, X), (name, a, b)
            assert int(re.search(r"FMA-pipe=(\d+)", src).group(1)) <= CAP
            for h in (dm.joint_hash(a, b), dm.joint_hash(b, a)):
                assert h not in others
                hashes.add(h)
        ordered = {p for a, b in pairs for p in ((a, b), (b, a))}
        assert len(hashes) == len(ordered), "(a, b) and (b, a) must name different cache entries"
        assert dm.spec_source() == spec_src
        dm.close()


def test_loop_node_choice_prefers_a_on_a_tie():
    """Two leaves of one parent with equal CPT shapes: both choices cost the same, the generator loops over a."""
    from bayescard_b200.synth import make_tree_model

    m = make_tree_model(3, [3, 4, 4], seed=1, dtype=np.float32, parent=[-1, 0, 0])
    m.cpts[2] = np.asarray(m.cpts[1]).copy()
    dm = DeviceModel(m, device=-1, specialize=False)
    for a, b in ((1, 2), (2, 1)):
        assert re.search(r"  X: (\d+)", dm.joint_source(a, b)).group(1) == str(a)
    dm.close()


def test_hash_follows_a_cpt_update_on_the_path():
    m = G.model("census")
    dm = DeviceModel(m, device=-1, specialize=False)
    a, b = census_pairs(m)[3]
    h0 = dm.joint_hash(a, b)
    m2 = copy.deepcopy(m)
    T = np.asarray(m2.cpts[b], dtype=np.float64).copy()
    T.reshape(int(m2.card[b]), -1)[:, 0] = 1.0 / int(m2.card[b])
    m2.cpts[b] = T
    dm2 = DeviceModel(m2, device=-1, specialize=False)
    assert dm2.joint_hash(a, b) != h0
    assert dm2.joint_source(a, b) != dm.joint_source(a, b)
    dm.close()
    dm2.close()


def test_argument_errors():
    lib = L.lib()
    m = G.model("dmv")
    dm = DeviceModel(m, device=-1, specialize=False)
    n = m.n_nodes
    for a, b in ((1, 1), (-1, 2), (2, n), (n, 0)):
        assert lib.bc_model_joint_source(dm._h, a, b, None, 0) == EINVAL, (a, b)
        assert lib.bc_model_joint_hash(dm._h, a, b) == 0
        assert lib.bc_model_specialize_joint(dm._h, a, b, None) == EINVAL
    assert lib.bc_joint_marginal_batch(None, None, 1, L.DESC_BITS, None, 0, 1, None, L.KERNEL_AUTO, None) == EINVAL
    # a host-only model cannot run (n_queries == 0 too)
    assert lib.bc_joint_marginal_batch(dm._h, None, 0, L.DESC_BITS, None, 0, 1, None, L.KERNEL_AUTO, None) == EINVAL
    assert lib.bc_model_specialize_joint(dm._h, 0, 1, None) == EINVAL
    # above the cap: BC_ELIMIT naming the count and the cap
    wide = sorted(range(n), key=lambda v: -int(m.card[v]))[:2]
    assert lib.bc_model_joint_source(dm._h, wide[0], wide[1], None, 0) == ELIMIT
    msg = lib.bc_last_error().decode()
    assert str(CAP) in msg and re.search(r"\d+ FMA-pipe instructions", msg), msg
    with pytest.raises(L.BayesCardError):
        dm.joint_source(wide[0], wide[1])
    with pytest.raises(ValueError):
        dm.joint_source(3, 3)
    dm.close()
    if not _has_gpu():
        return
    dmg = DeviceModel(m, device=0, specialize=False)
    out = np.zeros(1, dtype=np.float32)
    row = np.zeros(64, dtype=np.uint8)
    for a, b, fmt in ((1, 1, L.DESC_BITS), (-1, 1, L.DESC_BITS), (0, n, L.DESC_BITS), (0, 1, L.DESC_RANGE_U8)):
        assert lib.bc_joint_marginal_batch(dmg._h, row.ctypes.data, 1, fmt, None, a, b, out.ctypes.data, L.KERNEL_AUTO, None) == EINVAL
    assert lib.bc_joint_marginal_batch(dmg._h, None, 1, L.DESC_BITS, None, 0, 1, None, L.KERNEL_AUTO, None) == EINVAL
    assert not dmg.specialize_joint(wide[0], wide[1], "") and str(CAP) in dmg.joint_error[(wide[0], wide[1])]
    dmg.close()


def _has_gpu():
    try:
        import torch

        return torch.cuda.is_available()
    except Exception:  # noqa: BLE001
        return False


def _check_interpreted(m, dm, pairs, nq=1, seed=3, masks=False):
    lo, hi, bits, dense, W, Wd = _rows(m, dm, nq, seed)
    rng = np.random.default_rng(seed)
    for a, b in pairs:
        src = dm.joint_source(a, b)
        if masks:
            fan = JO.fan_nodes(m)
            mask = np.zeros((nq, dm.mask_words), dtype=np.uint32)
            for q in range(nq):
                for v in fan:
                    if rng.random() < 0.6:
                        mask[q, v >> 5] |= np.uint32(1 << (v & 31))
            Wm = O.range_weights(m, lo, hi, mask)
            Wdm = []
            for v in range(m.n_nodes):
                f = m.fan_vector(v)
                w = Wd[v]
                if f is not None:
                    bit = ((mask[:, v // 32] >> np.uint32(v % 32)) & 1).astype(bool)
                    w = np.where(bit[:, None], w * np.asarray(f, dtype=np.float64)[None, :], w)
                Wdm.append(w)
            cases = [(mask, Wm, Wdm), (None, W, Wd)]
        else:
            cases = [(None, W, Wd)]
        for mask, Wb, Wdb in cases:
            ref, ref_d = JG.joint(m, Wb, a, b), JG.joint(m, Wdb, a, b)
            for q in range(nq):
                mq = None if mask is None else mask[q]
                assert_close(_interp(src, "bc_joint_bits", bits[q].tobytes(), m, a, b, mq), ref[q], (a, b, q, "bits", mask is None))
                assert_close(_interp(src, "bc_joint_dense", dense[q].tobytes(), m, a, b, mq), ref_d[q], (a, b, q, "dense", mask is None))


def test_generated_joint_arithmetic_dmv():
    """The generated bodies of every DMV pair under the cap interpreted in fp32, against the fp64 oracle."""
    m = G.model("dmv")
    dm = DeviceModel(m, device=-1, specialize=False)
    pairs = _pairs_under_cap(dm, m)
    assert len(pairs) >= 30
    _check_interpreted(m, dm, pairs + [(b, a) for a, b in pairs[::7]])
    dm.close()


def test_generated_joint_arithmetic_census():
    m = G.model("census")
    dm = DeviceModel(m, device=-1, specialize=False)
    _check_interpreted(m, dm, census_pairs(m), nq=2)
    dm.close()


def test_generated_joint_arithmetic_fanout_tree():
    """Every ordered pair of a synthetic tree with fan-out vectors, exact zeros and a one-state column, with random masks
    and a NULL mask."""
    m = _synthetic_fan_model()
    dm = DeviceModel(m, device=-1, specialize=False)
    _check_interpreted(m, dm, list(itertools.permutations(range(m.n_nodes), 2)), nq=2, masks=True)
    dm.close()


def _ptxas(src, tmp_path, tag):
    ptx = tmp_path / f"{tag}.ptx"
    ptx.write_text(src)
    res = subprocess.run([os.environ.get("PTXAS", "/usr/local/cuda/bin/ptxas"), "-arch=sm_100a", "-O3", "-v", "-o",
                          str(tmp_path / f"{tag}.cubin"), str(ptx)], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-2000:]
    return res.stderr


def test_joint_modules_assemble_for_sm_100a(tmp_path):
    jobs = []
    dmv = G.model("dmv")
    dm = DeviceModel(dmv, device=-1, specialize=False)
    pairs = _pairs_under_cap(dm, dmv)
    jobs += [("dmv", dm.joint_source(a, b)) for a, b in (pairs[0], pairs[len(pairs) // 2], pairs[-1])]
    dm.close()
    cen = G.model("census")
    dm = DeviceModel(cen, device=-1, specialize=False)
    jobs += [("census", dm.joint_source(a, b)) for a, b in census_pairs(cen)[1:4]]
    dm.close()
    im = G.model("imdb1")
    dm = DeviceModel(im, device=-1, specialize=False)
    jobs += [("imdb1", dm.joint_source(0, im.n_nodes - 1))]
    dm.close()
    for k, (name, src) in enumerate(jobs):
        log = _ptxas(src, tmp_path, f"{name}{k}")
        assert log.count("Used") >= 2, log


# ------------------------------------------------------------------------------------ SQL (no GPU)
def test_parse_two_column_groupby():
    bn = Bayescard_BN(G.model("dmv"), device=-1)
    c1, c2, c3 = bn.tree.infer_names[1], bn.tree.infer_names[2], bn.tree.infer_names[3]
    q, c = parse_groupby_single_table(f"SELECT {c1}, {c2}, COUNT(*) FROM dmv GROUP BY {c1}, {c2}", bn)
    assert q == {} and c == (c1, c2)
    q, c = parse_groupby_single_table(f"select count(*), {c2}, {c1} from dmv group by {c2},{c1};", bn)
    assert c == (c2, c1)
    q1, c = parse_groupby_single_table(f"SELECT {c1}, COUNT(*) FROM dmv GROUP BY {c1}", bn)
    assert c == c1   # one column is still a string
    for bad in (f"SELECT {c1}, COUNT(*) FROM dmv GROUP BY {c1}, {c2}",                    # select list != group
                f"SELECT {c1}, {c1}, COUNT(*) FROM dmv GROUP BY {c1}, {c1}",              # a repeated column
                f"SELECT {c1}, {c2}, {c3}, COUNT(*) FROM dmv GROUP BY {c1}, {c2}, {c3}",  # three columns
                f"SELECT {c1}, nope, COUNT(*) FROM dmv GROUP BY {c1}, nope",              # unknown column
                f"SELECT {c1}, {c2} FROM dmv GROUP BY {c1}, {c2}"):                       # no COUNT(*)
        with pytest.raises(ValueError):
            parse_groupby_single_table(bad, bn)


def test_pair_argument_errors_in_python():
    bn = Bayescard_BN(G.model("imdb0"), device=-1)
    fan_col = bn.tree.infer_names[JO.fan_nodes(bn.tree)[0]]
    with pytest.raises(ValueError):
        bn.groupby_batch([{}], ("title.kind_id", fan_col))
    with pytest.raises(ValueError):
        bn.groupby_batch([{}], ("title.kind_id", "title.kind_id"))
    with pytest.raises(ValueError):
        bn.expectation_groupby_batch([{}], [[]], (fan_col, "title.kind_id"))


# ------------------------------------------------------------------------------------ GPU
def _assemble_joints(tm, pairs, cache_dir):
    """``ptxas`` the joint modules of ``pairs`` into ``cache_dir/joint_<hash>.cubin`` in parallel (the driver JIT compiles
    one module at a time)."""
    from concurrent.futures import ThreadPoolExecutor

    dm = DeviceModel(tm, device=-1, specialize=False)
    jobs = [(os.path.join(cache_dir, "joint_%016x.cubin" % dm.joint_hash(a, b)), dm.joint_source(a, b)) for a, b in pairs]
    dm.close()
    os.makedirs(cache_dir, exist_ok=True)

    def one(job):
        out, src = job
        if os.path.exists(out):
            return
        d = os.path.dirname(out)
        ptx = out + ".ptx"
        with open(ptx, "w") as f:
            f.write(src)
        res = subprocess.run([os.environ.get("PTXAS", "/usr/local/cuda/bin/ptxas"), "-arch=sm_100a", "-O3", "-o", out + ".tmp", ptx],
                             capture_output=True, text=True, cwd=d)
        os.remove(ptx)
        assert res.returncode == 0, res.stderr[-2000:]
        os.replace(out + ".tmp", out)

    with ThreadPoolExecutor(max_workers=os.cpu_count() or 4) as ex:
        list(ex.map(one, jobs))


def _device_rows(m, dm, nq, seed):
    """BITS and DENSE rows of ``nq`` random queries with their fp64 weights: at most four constrained columns, so that on
    Census every group stays inside the normal fp32 range (results below 1e-38 are not carried)."""
    _, _, bits, dense, W, Wd = _rows(m, dm, nq, seed, kmax=4)
    return bits, dense, W, Wd


@pytest.fixture(scope="module")
def joint_cache(tmp_path_factory):
    d = str(tmp_path_factory.mktemp("joint_cache"))
    for name in ("dmv", "census"):
        m = G.model(name)
        dm = DeviceModel(m, device=-1, specialize=False)
        pairs = _pairs_under_cap(dm, m) if name == "dmv" else census_pairs(m)
        dm.close()
        _assemble_joints(m, pairs, d)
        GO.assemble_marginals(m, sorted({v for p in pairs for v in p}), d)
    return d


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["dmv", "census"])
def test_joint_module_matches_the_oracle(name, joint_cache):
    """The joint module of every DMV pair under the cap and of the Census set, BITS and DENSE, ragged batch sizes; sums over
    j / i against bc_expectation_marginal_batch, the total against bc_query_batch; the module against the expansion."""
    m = G.model(name)
    dm = DeviceModel(m, device=0, specialize=False)
    plain = DeviceModel(m, device=0, specialize=False)   # nothing attached: AUTO expands through the query kernels
    host = DeviceModel(m, device=-1, specialize=False)
    pairs = _pairs_under_cap(host, m) if name == "dmv" else census_pairs(m)
    host.close()
    bits, dense, W, Wd = _device_rows(m, dm, 257, seed=5)
    for k, (a, b) in enumerate(pairs):
        assert dm.specialize_joint(a, b, joint_cache), dm.joint_error.get((a, b))
        nq = (1, 31, 257, 200)[k % 4]
        for desc, fmt, Wx in ((bits, L.DESC_BITS, W), (dense, L.DESC_DENSE_F32, Wd)):
            ref = JG.joint(m, [w[:nq] for w in Wx], a, b)
            got = dm.run_joint_host(desc[:nq], fmt, a, b, L.KERNEL_SPEC)
            assert_close(got, ref, (name, a, b, fmt, nq))
            assert_close(dm.run_joint_host(desc[:nq], fmt, a, b, L.KERNEL_AUTO), ref, (name, a, b, fmt, "auto"))
            if k % 5 == 0:
                exp = plain.run_joint_host(desc[:nq], fmt, a, b, L.KERNEL_AUTO)
                assert_close(exp, ref, (name, a, b, fmt, "expansion"))
                assert_close(got, exp, (name, a, b, fmt, "module vs expansion"), rtol=2e-5)
                g64 = got.astype(np.float64)
                assert_close(g64.sum(axis=2), plain.run_marginal_host(desc[:nq], fmt, a, L.KERNEL_GENERIC), (name, a, b, "sum j"))
                assert_close(g64.sum(axis=1), plain.run_marginal_host(desc[:nq], fmt, b, L.KERNEL_GENERIC), (name, a, b, "sum i"))
                assert_close(g64.sum(axis=(1, 2)), plain.run_host(desc[:nq], fmt, None, L.KERNEL_GENERIC), (name, a, b, "total"))
    dm.close()
    plain.close()


@pytest.mark.gpu
def test_expansions_match_the_oracle(joint_cache):
    """AUTO without the joint module (with and without b's marginal module), K1 and K3 through the expansion."""
    m = G.model("census")
    pairs = census_pairs(m)
    with_marg = DeviceModel(m, device=0, specialize=False)
    plain = DeviceModel(m, device=0, specialize=False)
    bits, dense, W, Wd = _device_rows(m, plain, 100, seed=8)
    for a, b in pairs:
        assert with_marg.specialize_marginal(b, joint_cache)
        for desc, fmt, Wx in ((bits, L.DESC_BITS, W), (dense, L.DESC_DENSE_F32, Wd)):
            ref = JG.joint(m, Wx, a, b)
            for model, kernel in ((with_marg, L.KERNEL_AUTO), (plain, L.KERNEL_AUTO), (plain, L.KERNEL_GENERIC), (plain, L.KERNEL_FUSED)):
                try:
                    got = model.run_joint_host(desc, fmt, a, b, kernel)
                except L.BayesCardError as e:   # K3 serves a model or it does not (BC_ELIMIT)
                    assert kernel == L.KERNEL_FUSED and "error -5" in str(e), e
                    continue
                assert_close(got, ref, (a, b, fmt, kernel, model is with_marg))
    with_marg.close()
    plain.close()


@pytest.mark.gpu
def test_imdb_joint_module_with_fanout_masks(tmp_path):
    from join_groupby_oracle import fan_nodes

    m = G.model("imdb1")
    pc = PredicateCompiler(m)
    cases = [r for r in G.load("infer_cases.json.gz")["imdb1"] if "error" not in r]
    decoded = [({k: list(v) for k, v in r["bins"].items()}, {k: np.asarray(v) for k, v in r["weights"].items()}) for r in cases]
    decoded.append(({}, {}))
    fan = [m.infer_names[v] for v in fan_nodes(m)]
    rng = np.random.default_rng(2)
    fans = [[f for f in fan if rng.random() < 0.6 or f in bb] for bb, _ in decoded]
    host = DeviceModel(m, device=-1, specialize=False)
    pairs = [(a, b) for a, b in ((0, m.n_nodes - 1), (1, 2), (m.n_nodes - 1, 0))
             if L.lib().bc_model_joint_source(host._h, a, b, None, 0) > 0]
    host.close()
    assert pairs
    _assemble_joints(m, pairs, str(tmp_path))
    dm = DeviceModel(m, device=0, specialize=False)
    plain = DeviceModel(m, device=0, specialize=False)
    for a, b in pairs:
        assert dm.specialize_joint(a, b, str(tmp_path)), dm.joint_error.get((a, b))
        b_idx, b_desc, d_idx, d_desc, mask = pc.pack(decoded, fans, force_dense=False)
        for idx, desc, fmt in ((b_idx, b_desc, L.DESC_BITS), (d_idx, d_desc, L.DESC_DENSE_F32)):
            if not len(idx):
                continue
            mk = np.ascontiguousarray(mask[idx])
            per = [O.dense_weights(m, decoded[i][0], decoded[i][1], fans[i]) for i in idx]
            Wm = [np.stack([p[v] for p in per]) for v in range(m.n_nodes)]
            ref = JG.joint(m, Wm, a, b)
            assert_close(dm.run_joint_host(desc, fmt, a, b, L.KERNEL_SPEC, mk), ref, (a, b, fmt, "spec"))
            assert_close(plain.run_joint_host(desc, fmt, a, b, L.KERNEL_AUTO, mk), ref, (a, b, fmt, "expansion"))
    dm.close()
    plain.close()


@pytest.mark.gpu
def test_launches_and_missing_module(joint_cache):
    import torch

    m = G.model("dmv")
    dm = DeviceModel(m, device=0, specialize=False)
    a, b = 1, 2
    bits, _, _, _ = _device_rows(m, dm, 64, seed=1)
    d_desc = torch.from_numpy(bits.reshape(-1).view(np.uint8)).to("cuda:0")
    d_out = torch.empty((64, int(m.card[a]), int(m.card[b])), dtype=torch.float32, device="cuda:0")
    st = torch.cuda.current_stream().cuda_stream
    lib = L.lib()
    assert lib.bc_joint_marginal_batch(dm._h, d_desc.data_ptr(), 64, L.DESC_BITS, None, a, b, d_out.data_ptr(), L.KERNEL_SPEC,
                                       st) == ECOMPILE
    before = launch_count()
    dm.run_joint_device(d_desc.data_ptr(), 0, L.DESC_BITS, a, b, d_out.data_ptr(), L.KERNEL_AUTO, st)
    assert launch_count() == before
    assert dm.specialize_joint(a, b, joint_cache)
    for kernel in (L.KERNEL_SPEC, L.KERNEL_AUTO):
        before = launch_count()
        dm.run_joint_device(d_desc.data_ptr(), 64, L.DESC_BITS, a, b, d_out.data_ptr(), kernel, st)
        assert launch_count() - before == 1, kernel
    torch.cuda.synchronize()
    dm.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["dmv", "census"])
def test_groupby_two_columns_matches_per_pair_queries(name, joint_cache):
    m = G.model(name)
    bn = Bayescard_BN(m, device=0, infer_algo="exact-jit")
    bn.init_inference_method()
    pc = bn.infer_machine.compiler
    cat = [c for c in m.infer_names if pc.cols[c].kind != "continuous" and pc.cols[c].enc is not None]
    cat = sorted(cat, key=lambda c: int(m.card[m._index[c]]))
    ca, cb = cat[len(cat) // 2], cat[len(cat) // 2 + 1]
    rng = np.random.default_rng(6)
    qs = []
    for _ in range(12):
        q = {}
        for c in rng.choice(cat, size=3, replace=False):
            vals = list(pc.cols[c].pair)
            q[str(c)] = [vals[i] for i in sorted(rng.choice(len(vals), size=max(1, len(vals) // 2), replace=False))]
        qs.append(q)
    qs += [{}, {ca: ["no such value"]}]
    keys, est = bn.groupby_batch([copy.deepcopy(q) for q in qs], (ca, cb))
    ka, kb = list(pc.cols[ca].pair), list(pc.cols[cb].pair)
    assert keys == list(itertools.product(ka, kb)) and est.shape == (len(qs), len(ka) * len(kb))
    for i, q in enumerate(qs):
        rest = {k: v for k, v in q.items() if k not in (ca, cb)}
        sa = pc.select_values(ca, q[ca]) if ca in q else np.ones(len(ka), dtype=bool)
        sb = pc.select_values(cb, q[cb]) if cb in q else np.ones(len(kb), dtype=bool)
        per = [{**copy.deepcopy(rest), ca: [va], cb: [vb]} for va, vb in keys]
        ref = bn.query_batch(per)
        if sa is None or sb is None:
            ref[:] = 0
        else:
            ref *= np.outer(sa, sb).reshape(-1)
        assert_close(est[i], ref, (name, i), rtol=2e-5)
        # the fp64 oracle, per pair
        for j in range(0, len(keys), max(1, len(keys) // 7)):
            bb, w = O.query_decoding(m, copy.deepcopy(per[j]))
            exp = 0.0 if (bb is None or ref[j] == 0) else float(np.asarray(O.dense_tree(m, O.dense_weights(m, bb, w))).reshape(-1)[0]) * bn.nrows
            assert_close(est[i, j], exp, (name, i, j, "oracle"), rtol=2e-5)
    assert np.all(est[-1] == 0)
    bn.infer_machine.close()


@pytest.mark.gpu
def test_groupby_continuous_and_categorical_on_imdb_and_sql():
    """A continuous column (its bins as keys, its predicate kept) with a categorical one: group (bin, v) is the continuous
    column's group under the query with the categorical predicate replaced by ``= v``.  Texts grouping by one and by two
    columns go in one groupby_sql_batch."""
    m = G.model("imdb3")
    bn = Bayescard_BN(m, device=0, infer_algo="exact-jit")
    bn.init_inference_method()
    pc = bn.infer_machine.compiler
    cont, cat = "movie_keyword.keyword_id", "title.kind_id"
    assert pc.cols[cont].kind == "continuous"
    qs = [{}, {cat: [1, 2]}, {cont: (1000.0, 50000.0)}, {cont: (1000.0, 50000.0), cat: [7]}]
    keys, est = bn.groupby_batch([copy.deepcopy(q) for q in qs], (cont, cat))
    kc, _ = bn.groupby_batch([{}], cont)
    kk = list(pc.cols[cat].pair)
    assert keys == list(itertools.product(kc, kk)) and est.shape == (len(qs), len(kc) * len(kk))
    E = est.reshape(len(qs), len(kc), len(kk))
    for j, v in enumerate(kk):
        per = [{**{k: x for k, x in q.items() if k != cat}, cat: [v]} for q in qs]
        _, ref = bn.groupby_batch(per, cont)
        sel = np.asarray([pc.select_values(cat, q[cat])[j] if cat in q else True for q in qs], dtype=float)
        assert_close(E[:, :, j], ref * sel[:, None], ("key", v), rtol=2e-5)
    texts = [f"SELECT {cat}, {cont}, COUNT(*) FROM title WHERE {cat} IN [1, 2] GROUP BY {cat}, {cont}",
             f"SELECT {cat}, COUNT(*) FROM title GROUP BY {cat}",
             f"SELECT {cont}, {cat}, COUNT(*) FROM title GROUP BY {cont}, {cat}"]
    res = bn.groupby_sql_batch(texts)
    _, e2 = bn.groupby_batch([{cat: [1, 2]}], (cat, cont))
    _, e1 = bn.groupby_batch([{}], cat)
    assert list(res[0]) == list(itertools.product(kk, kc)) and list(res[2]) == keys
    assert np.array_equal(list(res[0].values()), e2[0]) and np.array_equal(list(res[1].values()), e1[0])
    assert_close(list(res[2].values()), est[0], "text batch vs query batch")   # (rows packed with other queries)
    bn.infer_machine.close()


@pytest.mark.gpu
def test_joint_follows_an_update(joint_cache):
    """After an update the joint module is forgotten, its hash moves (no stale cubin can attach) and the module built again
    computes what the expansion computes on the new CPTs."""
    from bayescard_b200 import fit as F

    m = copy.deepcopy(G.model("census"))
    a, b = census_pairs(m)[1]
    dm = DeviceModel(m, device=0, specialize=False)
    dm.attach_counts(F.counts_from_cpts(m.parent, m.card, m.cpts, F.infer_fit_rows(m)))
    assert dm.specialize_joint(a, b, joint_cache)
    h0 = dm.joint_hash(a, b)
    bits, _, _, _ = _device_rows(m, dm, 50, seed=4)
    before = dm.run_joint_host(bits, L.DESC_BITS, a, b, L.KERNEL_SPEC)
    rng = np.random.default_rng(1)
    rows = np.stack([rng.integers(0, int(c), size=200000) for c in m.card], axis=1).astype(np.uint8)
    touched = dm.update(inserted=rows)
    assert a in touched and b in touched
    assert (a, b) not in dm._joint_built and dm.joint_hash(a, b) != h0
    with pytest.raises(L.BayesCardError):   # the old module is gone
        dm.run_joint_host(bits, L.DESC_BITS, a, b, L.KERNEL_SPEC)
    ref = dm.run_joint_host(bits, L.DESC_BITS, a, b, L.KERNEL_GENERIC)
    assert dm.specialize_joint(a, b, joint_cache)   # generated again for the new CPTs (the cache holds only the old hash)
    got = dm.run_joint_host(bits, L.DESC_BITS, a, b, L.KERNEL_SPEC)
    assert_close(got, ref, "module after update vs expansion after update", rtol=2e-5)
    assert not np.allclose(got, before, rtol=1e-3)
    assert_close(got.astype(np.float64).sum(axis=(1, 2)), dm.run_host(bits, L.DESC_BITS, None, L.KERNEL_GENERIC), "total")
    dm.close()
