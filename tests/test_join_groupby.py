"""GROUP BY over fan-out expectations: bc_expectation_marginal_batch (the specialised marginal kernel with a fan-out mask and
the expansion that carries the mask), Bayescard_BN.expectation_groupby_batch, BN_ensemble.groupby_batch and the job-light
GROUP BY planner, against the fp64 oracle (join_groupby_oracle: groupby_oracle.marginal with the fan-out vectors multiplied
into W).  Tolerances: 1e-5 relative for marginals, 2e-5 for join estimates, as the other GPU parity tests."""
import copy
import hashlib
import json
import os
import re

import numpy as np
import pytest

import golden_util as G
import groupby_oracle as GO
import join_groupby_oracle as JO
from bayescard_b200 import _lib as L
from bayescard_b200.decode import PredicateCompiler
from bayescard_b200.engine import DeviceModel, launch_count
from bayescard_b200.joblight import (BN_INDEX, GROUP_VALUE, groupby_value_plan, parse_job_light_groupby, plan_star_groupby,
                                     plan_star_query)
from bayescard_b200.model import Bayescard_BN
from oracle import bayescard_oracle as O

RTOL = 1e-5
IMDB = [f"imdb{i}" for i in range(5)]
# a categorical column of every joined table but movie_keyword (keyword_id is continuous)
JOINED_COLUMN = {"movie_info_idx": "info_type_id", "movie_info": "info_type_id", "cast_info": "role_id",
                 "movie_companies": "company_type_id"}
ALIAS = {"title": "t", "movie_info_idx": "mi_idx", "movie_info": "mi", "cast_info": "ci", "movie_companies": "mc"}


def assert_close(got, ref, what="", rtol=RTOL):
    got, ref = np.asarray(got, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    err = np.abs(got - ref) / np.maximum(np.abs(ref), 1e-300)
    err[(ref == 0) & (got == 0)] = 0
    assert err.max() <= rtol, (what, float(err.max()), np.unravel_index(int(err.argmax()), err.shape))


def _norm(src):
    src = re.sub(r"marginal generator \(version \d+,", "marginal generator (version V,", src)
    return re.sub(r"bc_marg_meta\[4\] = \{(\d+), (\d+), \d+, (\d+)\}", r"bc_marg_meta[4] = {\1, \2, V, \3}", src)


def _rand_masks(m, nq, target, rng, predicated=()):
    """Mask rows over the model's fan-out nodes: the target's bit and the bits of nodes on its root path always set when
    they carry a fan-out vector, the other fan-out bits at random, plus ``predicated`` nodes."""
    path = []
    v = target
    while v >= 0:
        path.append(v)
        v = int(m.parent[v]) if v > 0 else -1
    fan = JO.fan_nodes(m)
    mask = np.zeros((nq, (m.n_nodes + 31) // 32), dtype=np.uint32)
    for q in range(nq):
        for v in fan:
            if v in path or v in predicated or rng.random() < 0.5:
                mask[q, v >> 5] |= np.uint32(1 << (v & 31))
    return mask


def _joblight_sqls():
    return [r["sql"] for r in G.load("job_light.json.gz")["queries"]]


def _groupby_texts():
    """Every shipped job-light query grouped by title.kind_id, title.production_year and one joined table's categorical
    column (the first table of its FROM list that has one)."""
    out = []
    for sql in _joblight_sqls():
        body = re.match(r"(?is)^\s*select\s+count\(\*\)\s+(from\s+.*?);?\s*$", sql).group(1)
        cols = ["t.kind_id", "t.production_year"]
        order = [p.split()[0] for p in re.split(r"(?i)\s+where\s+", body[5:])[0].split(",")]
        joined = next((t for t in order if t in JOINED_COLUMN), None)
        if joined is not None:
            cols.append(f"{ALIAS[joined]}.{JOINED_COLUMN[joined]}")
        for c in cols:
            out.append(f"SELECT {c}, COUNT(*) {body} GROUP BY {c}")
    return out


def _join_sizes():
    return {i: float(G.model(f"imdb{i}").nrows) for i in range(5)}


def _per_value_cardinalities(ens, plans):
    """``BN_ensemble.cardinality_batch`` of per-value plans; NaN where a plan has an undecodable expectation factor (the
    reference raises ``AttributeError`` there, and the whole batch with it)."""
    parsed = ens.parse_query_all([copy.deepcopy(p) for p in plans])
    bad = np.asarray([any(f["query"] is None and len(f["expectation"]) for f in tq[1:]) for tq in parsed], dtype=bool)
    out = np.full(len(parsed), np.nan)
    ok = np.nonzero(~bad)[0]
    if len(ok):
        out[ok] = ens.cardinality_batch([parsed[i] for i in ok])
    return out


def _host_bns():
    bns = {}
    for i in range(5):
        bns[i] = Bayescard_BN(G.model(f"imdb{i}"), device=-1)
        bns[i].init_inference_method()
    return bns


# ------------------------------------------------------------------------------------ code generator (no GPU)
def test_marginal_sources_without_fanout_are_unchanged():
    """DMV and Census have no fan-out vectors: the marginal module of every target is the one generated before the kernels
    took a fan-out mask, byte for byte apart from the generator version (sha256 fixture from that generator)."""
    with open(os.path.join(G.GOLD, "marginal_sources_v1.json")) as f:
        ref = json.load(f)["sha256"]
    for name in ("dmv", "census"):
        m = G.model(name)
        dm = DeviceModel(m, device=-1, specialize=False)
        assert len(ref[name]) == m.n_nodes
        for t in range(m.n_nodes):
            src = dm.marginal_source(t)
            assert "marginal generator (version 2," in src and "%pfm ld.global.nc.u32" not in src
            assert hashlib.sha256(_norm(src).encode()).hexdigest() == ref[name][t], (name, t)
        dm.close()


def test_imdb_marginal_sources_carry_the_mask():
    for name in IMDB:
        m = G.model(name)
        dm = DeviceModel(m, device=-1, specialize=False)
        nz = sum(int(np.count_nonzero(np.asarray(c, dtype=np.float32))) for c in m.cpts)
        hashes = set()
        for t in range(m.n_nodes):
            src = dm.marginal_source(t)
            assert src == dm.marginal_source(t), "generator is not deterministic"
            assert "@%pfm ld.global.nc.u32" in src   # the mask words are loaded only for a non-NULL mask
            # fan-out multiplies are not counted: one FMA-pipe instruction per non-zero CPT entry
            assert re.search(r"BC_SPEC_FFMA=(\d+)", src).group(1) == str(nz)
            hashes.add(dm.marginal_hash(t))
        assert len(hashes) == m.n_nodes and dm.spec_hash() not in hashes
        dm.close()


def test_imdb_marginal_modules_assemble_for_sm_100a(tmp_path):
    for name in IMDB:
        m = G.model(name)
        GO.assemble_marginals(m, range(m.n_nodes), str(tmp_path / name))
        assert len(os.listdir(tmp_path / name)) == m.n_nodes, name


def _synthetic_fan_model():
    from bayescard_b200.synth import make_tree_model

    m = make_tree_model(9, [3, 7, 5, 2, 6, 4, 8, 3, 5], seed=4, dtype=np.float32)
    m.cpts[3][0, :] = 0.0   # an all-zero row and scattered exact zeros
    m.cpts[6][:, 1] = np.where(np.arange(8) % 2 == 0, 0.0, m.cpts[6][:, 1])
    rng = np.random.default_rng(7)
    for v in (0, 2, 3, 6, 8):   # the root, inner nodes and a leaf carry fan-out vectors (one with an exact zero)
        f = rng.uniform(0.5, 20.0, int(m.card[v]))
        if v == 6:
            f[2] = 0.0
        m.fanouts[m.infer_names[v]] = f
    return m


@pytest.mark.parametrize("name", IMDB + ["synthetic"])
def test_generated_masked_marginal_arithmetic_on_the_host(name):
    """The generated bodies interpreted in fp32 with mask rows, against the fp64 oracle: every target; the masks hold the
    target's bit, the bits of its path and a fan-out column that also has a predicate (the bit multiplies the predicate's
    weights); the NULL mask is the unmasked marginal."""
    from bayescard_b200.synth import random_range_queries

    m = G.model(name) if name != "synthetic" else _synthetic_fan_model()
    dm = DeviceModel(m, device=-1, specialize=False)
    pc = PredicateCompiler(m)
    nq = 2
    lo, hi = random_range_queries(m, nq, seed=3, kmax=m.n_nodes)
    fan = JO.fan_nodes(m)
    pred_fan = fan[len(fan) // 2]
    lo[:, pred_fan] = 0
    hi[:, pred_fan] = max(0, int(m.card[pred_fan]) - 2)   # a predicate on a fan-out column
    bits = pc.pack_bits(lo, hi)
    rng = np.random.default_rng(5)
    for t in range(m.n_nodes):
        src = dm.marginal_source(t)
        mask = _rand_masks(m, nq, t, rng, predicated=(pred_fan,))
        W = O.range_weights(m, lo, hi, mask)
        Wd = [(np.asarray(w) * (0.25 + 0.75 * rng.random((nq, 1)))).astype(np.float32) for w in O.range_weights(m, lo, hi)]
        dense = np.zeros((nq, dm.dense_width), dtype=np.float32)
        for v in range(m.n_nodes):
            o = int(dm.dense_offset[v])
            dense[:, o:o + int(m.card[v])] = Wd[v]
        Wdm = []
        for v in range(m.n_nodes):
            w = Wd[v].astype(np.float64)
            f = m.fan_vector(v)
            if f is not None:
                bit = ((mask[:, v // 32] >> np.uint32(v % 32)) & 1).astype(bool)
                w = np.where(bit[:, None], w * np.asarray(f, dtype=np.float64)[None, :], w)
            Wdm.append(w)
        ref, ref_d = GO.marginal(m, W, t), GO.marginal(m, Wdm, t)
        ref0 = GO.marginal(m, O.range_weights(m, lo, hi), t)
        for q in range(nq):
            assert_close(JO.interpret_masked(src, "bc_marg_bits", bits[q].tobytes(), mask[q]), ref[q], (name, t, q, "bits"))
            assert_close(JO.interpret_masked(src, "bc_marg_dense", dense[q].tobytes(), mask[q]), ref_d[q], (name, t, q, "dense"))
            assert_close(JO.interpret_masked(src, "bc_marg_bits", bits[q].tobytes(), None), ref0[q], (name, t, q, "NULL mask"))
    dm.close()


def test_masked_marginal_argument_errors():
    lib = L.lib()
    m = G.model("imdb0")
    dm = DeviceModel(m, device=-1, specialize=False)
    mask = np.zeros(4, dtype=np.uint32)
    for bad in (-1, m.n_nodes):
        assert lib.bc_expectation_marginal_batch(dm._h, None, 1, L.DESC_BITS, mask.ctypes.data, bad, None, L.KERNEL_AUTO, None) == -1
    assert lib.bc_expectation_marginal_batch(None, None, 1, L.DESC_BITS, None, 0, None, L.KERNEL_AUTO, None) == -1
    # a host-only model cannot run (n_queries == 0 too), RANGE rows are refused
    assert lib.bc_expectation_marginal_batch(dm._h, None, 0, L.DESC_BITS, None, 0, None, L.KERNEL_AUTO, None) == -1
    assert lib.bc_expectation_marginal_batch(dm._h, None, 1, L.DESC_RANGE_U8, mask.ctypes.data, 0, None, L.KERNEL_AUTO, None) == -1
    row = np.zeros((2, dm.desc_stride(L.DESC_BITS)), dtype=np.uint8)
    with pytest.raises(ValueError):   # one mask row per query
        dm.run_marginal_host(row, L.DESC_BITS, 0, L.KERNEL_AUTO, np.zeros((3, dm.mask_words), dtype=np.uint32))
    with pytest.raises(L.BayesCardError):
        dm.run_marginal_host(row, L.DESC_BITS, 0, L.KERNEL_AUTO, np.zeros((2, dm.mask_words), dtype=np.uint32))
    dm.close()
    bn = Bayescard_BN(m, device=-1)
    fan_col = m.infer_names[JO.fan_nodes(m)[0]]
    with pytest.raises(ValueError):   # GROUP BY a fan-out column
        bn.expectation_groupby_batch([{}], [[]], fan_col)
    with pytest.raises(ValueError):   # one fan-out list per query
        bn.expectation_groupby_batch([{}, {}], [[]], "title.kind_id")


# ------------------------------------------------------------------------------------ job-light GROUP BY planner (no GPU)
def test_groupby_plan_equals_the_per_value_plans():
    """For every shipped job-light query grouped by kind_id, production_year and a joined table's column: the GROUP BY plan
    with the placeholder replaced by v is plan_star_query of the per-value text, for every key of every BN."""
    js = _join_sizes()
    bns = _host_bns()
    checked = 0
    for sql in _groupby_texts():
        planned = plan_star_groupby(sql, js)
        column = planned["column"]
        keys = list(dict.fromkeys(k for i in range(5) if column in bns[i].tree._index
                                  for k in bns[i].infer_machine.compiler.cols[column].pair))
        assert keys
        holders = [f for f in planned["plan"][1:] if column in f["query"]]
        assert holders and all(f["query"][column] is GROUP_VALUE for f in holders)
        for v in keys:
            text = JO.per_value_sql(sql, v)
            if text is None:
                continue
            got = groupby_value_plan(planned, v)
            ref = plan_star_query(text, js)
            assert got[0] == ref[0] and len(got) == len(ref), (sql, v)
            for a, b in zip(got[1:], ref[1:]):
                assert (a["bn_index"], a["inverse"], a["expectation"]) == (b["bn_index"], b["inverse"], b["expectation"]), (sql, v)
                assert a["query"] == b["query"], (sql, v)
            checked += 1
    assert checked > 10000


def test_parse_job_light_groupby():
    sql = ("SELECT t.production_year, COUNT(*) FROM title t,movie_info mi WHERE t.id=mi.movie_id AND mi.info_type_id=3 "
           "AND t.production_year>2000 GROUP BY t.production_year;")
    order, conds, table, col = parse_job_light_groupby(sql)
    assert order == ["movie_info"] and (table, col) == ("title", "production_year")
    p = plan_star_groupby(sql, _join_sizes())
    assert p["column"] == "title.production_year" and p["where"] == (2000 + 0.1, np.inf)
    assert parse_job_light_groupby(sql.replace("SELECT t.production_year, COUNT(*)", "select count(*), t.production_year"))[2:] == (
        "title", "production_year")
    for bad in (sql.replace("GROUP BY t.production_year", ""),                                   # no GROUP BY
                sql.replace("SELECT t.production_year,", "SELECT t.kind_id,"),                   # select list != group
                sql.replace("t.production_year, COUNT", "ci.role_id, COUNT").replace("BY t.production_year", "BY ci.role_id")):
        # (the last one: an alias outside FROM)
        with pytest.raises(ValueError):
            parse_job_light_groupby(bad)


def test_continuous_grouping_columns_are_refused():
    from bayescard_b200.ensemble import BN_ensemble

    ens = BN_ensemble(bns=_host_bns())
    js = _join_sizes()
    for sql in ("SELECT mk.keyword_id, COUNT(*) FROM title t,movie_keyword mk WHERE t.id=mk.movie_id AND t.kind_id=1 "
                "GROUP BY mk.keyword_id",
                "SELECT mc.company_id, COUNT(*) FROM title t,movie_companies mc WHERE t.id=mc.movie_id GROUP BY mc.company_id"):
        p = plan_star_groupby(sql, js)
        with pytest.raises(ValueError):
            ens.groupby_batch([p], p["column"])


# ------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def marg_cache():
    for name in IMDB:
        m = G.model(name)
        GO.assemble_marginals(m, range(m.n_nodes), L.SPEC_CACHE_DIR)
    return L.SPEC_CACHE_DIR


def _imdb_cases(name, rng):
    """infer_cases of the model (bins, fractional weights) plus a query without predicates, each with a random subset of
    the model's fan-out columns (a predicated one included where a query has one)."""
    m = G.model(name)
    cases = [r for r in G.load("infer_cases.json.gz")[name] if "error" not in r]
    decoded = [({k: list(v) for k, v in r["bins"].items()}, {k: np.asarray(v) for k, v in r["weights"].items()}) for r in cases]
    decoded.append(({}, {}))
    fan = [m.infer_names[v] for v in JO.fan_nodes(m)]
    fans = [[f for f in fan if rng.random() < 0.6 or f in b] for b, _ in decoded]
    return decoded, fans


@pytest.mark.gpu
@pytest.mark.parametrize("name", IMDB)
def test_masked_marginals_match_the_oracle(name, marg_cache):
    m = G.model(name)
    rng = np.random.default_rng(11)
    spec = DeviceModel(m, device=0, specialize=False)
    for t in range(m.n_nodes):
        assert spec.specialize_marginal(t, marg_cache), spec.marginal_error.get(t)
    plain = DeviceModel(m, device=0, specialize=False)   # no marginal module attached: AUTO expands
    pc = PredicateCompiler(m)
    decoded, fans = _imdb_cases(name, rng)
    for force_dense in (False, True):
        b_idx, b_desc, d_idx, d_desc, mask = pc.pack(decoded, fans, force_dense=force_dense)
        for idx, desc, fmt in ((b_idx, b_desc, L.DESC_BITS), (d_idx, d_desc, L.DESC_DENSE_F32)):
            if not len(idx):
                continue
            mk = np.ascontiguousarray(mask[idx])
            assert mk.any()
            total = plain.run_host(desc, fmt, mk, L.KERNEL_GENERIC)
            for t in range(m.n_nodes):
                ref = JO.masked_marginal(m, [decoded[i] for i in idx], [fans[i] for i in idx], t)
                for kernel, model in ((L.KERNEL_SPEC, spec), (L.KERNEL_GENERIC, plain), (L.KERNEL_FUSED, plain), (L.KERNEL_AUTO, plain)):
                    got = model.run_marginal_host(desc, fmt, t, kernel, mk)
                    assert got.shape == ref.shape
                    assert_close(got, ref, (name, t, fmt, kernel, force_dense))
                    if kernel == L.KERNEL_SPEC:   # row sums are bc_query_batch with the same mask
                        assert_close(got.astype(np.float64).sum(axis=1), total, (name, t, fmt, "sum over bins"))
    spec.close()
    plain.close()


@pytest.mark.gpu
def test_mask_has_no_effect_without_fanout_vectors_and_spec_is_one_launch(marg_cache):
    import torch

    m = G.model("dmv")
    GO.assemble_marginals(m, [2], L.SPEC_CACHE_DIR)
    dm = DeviceModel(m, device=0, specialize=False)
    assert dm.specialize_marginal(2, L.SPEC_CACHE_DIR), dm.marginal_error.get(2)
    n, t = 5000, 2
    desc = torch.empty((n, dm.desc_stride(L.DESC_RANGE_U8)), dtype=torch.uint8, device="cuda:0")
    bits = torch.empty((n, dm.desc_stride(L.DESC_BITS)), dtype=torch.uint8, device="cuda:0")
    out = torch.empty((n, int(m.card[t])), dtype=torch.float32, device="cuda:0")
    mask = torch.from_numpy(np.random.default_rng(3).integers(0, 2**32, size=(n, dm.mask_words), dtype=np.uint32)).to("cuda:0")
    st = torch.cuda.current_stream().cuda_stream
    dm.gen_range_queries_device(5, 0, n, 1, 8, desc.data_ptr(), st)
    dm.convert_device(desc.data_ptr(), L.DESC_RANGE_U8, bits.data_ptr(), L.DESC_BITS, n, st)
    for kernel in (L.KERNEL_SPEC, L.KERNEL_GENERIC):
        dm.run_marginal_device(bits.data_ptr(), n, L.DESC_BITS, t, out.data_ptr(), kernel, st)
        torch.cuda.synchronize()
        ref = out.cpu().numpy().copy()
        dm.run_marginal_device(bits.data_ptr(), n, L.DESC_BITS, t, out.data_ptr(), kernel, st, mask.data_ptr())
        torch.cuda.synchronize()
        assert np.array_equal(out.cpu().numpy(), ref), kernel
    dm.close()
    # IMDB: a spec call with a mask is one launch
    im = G.model("imdb1")
    dmi = DeviceModel(im, device=0, specialize=False)
    ti = JO.fan_nodes(im)[0]
    assert dmi.specialize_marginal(ti, marg_cache)
    pc = PredicateCompiler(im)
    decoded, fans = _imdb_cases("imdb1", np.random.default_rng(1))
    b_idx, b_desc, _, _, mk = pc.pack(decoded, fans, force_dense=False)
    d_desc = torch.from_numpy(b_desc.reshape(-1)).to("cuda:0")
    d_mask = torch.from_numpy(np.ascontiguousarray(mk[b_idx]).reshape(-1)).to("cuda:0")
    d_out = torch.empty((len(b_idx), int(im.card[ti])), dtype=torch.float32, device="cuda:0")
    torch.cuda.synchronize()
    for kernel in (L.KERNEL_SPEC, L.KERNEL_AUTO):
        before = launch_count()
        dmi.run_marginal_device(d_desc.data_ptr(), len(b_idx), L.DESC_BITS, ti, d_out.data_ptr(), kernel, st, d_mask.data_ptr())
        assert launch_count() - before == 1, kernel
    torch.cuda.synchronize()
    dmi.close()


@pytest.mark.gpu
def test_expectation_groupby_matches_per_value_expectations(marg_cache):
    name = "imdb2"
    m = G.model(name)
    bn = Bayescard_BN(m, device=0, infer_algo="exact-jit")
    bn.init_inference_method()
    fan = [m.infer_names[v] for v in JO.fan_nodes(m)]
    qs = [G.unjson(r["query"]) for r in G.load("imdb_cases.json.gz")[name] if "error" not in r]
    qs = [q for q in qs if any(k in m._index for k in q)][:30] + [{}]
    rng = np.random.default_rng(4)
    fans = [[f for f in fan if rng.random() < 0.5] for _ in qs]
    for col in ("title.kind_id", "cast_info.role_id"):
        keys, est = bn.expectation_groupby_batch([copy.deepcopy(q) for q in qs], fans, col)
        pc = bn.infer_machine.compiler
        assert keys == list(pc.cols[col].pair)
        for i, (q, f) in enumerate(zip(qs, fans)):
            sel = pc.select_values(col, q[col]) if col in q else np.ones(len(keys), dtype=bool)
            rest = {k: v for k, v in q.items() if k != col}
            ref = np.zeros(len(keys))
            if sel is not None and O.query_decoding(m, copy.deepcopy(rest))[0] is not None:
                for j, k in enumerate(keys):
                    if sel[j]:
                        ref[j] = float(np.asarray(O.bn_expectation(m, {**copy.deepcopy(rest), col: k}, f)).reshape(-1)[0])
            assert_close(est[i], ref, (col, i))
        # no fan-out column: groupby_batch
        _, e0 = bn.expectation_groupby_batch([copy.deepcopy(q) for q in qs], [[] for _ in qs], col)
        _, g0 = bn.groupby_batch([copy.deepcopy(q) for q in qs], col)
        assert np.array_equal(e0, g0)
    bn.close()


@pytest.fixture(scope="module")
def ensemble(marg_cache):
    from bayescard_b200.ensemble import BN_ensemble

    bns = {}
    for i in range(5):
        bns[i] = Bayescard_BN(G.model(f"imdb{i}"), device=0, infer_algo="exact-jit")
        bns[i].init_inference_method()
    ens = BN_ensemble(bns=bns)
    yield ens
    for bn in bns.values():
        bn.close()


@pytest.mark.gpu
def test_job_light_groupby_equals_the_per_value_estimates(ensemble):
    from bayescard_b200.joblight import groupby_sql_batch

    js = _join_sizes()
    texts = _groupby_texts()
    res = groupby_sql_batch(ensemble, texts, js)
    assert len(res) == len(texts)
    per_value, where = [], []
    for sql, r in zip(texts, res):
        planned = plan_star_groupby(sql, js)
        for k in r:
            per_value.append((sql, k, r[k], groupby_value_plan(planned, k)))
    ref = _per_value_cardinalities(ensemble, [p for _, _, _, p in per_value])
    bns = ensemble.bns
    nonzero = zeros = 0
    for (sql, k, got, plan), r in zip(per_value, ref):
        if np.isnan(r):   # the per-value estimate would raise: the group is 0
            assert got == 0, (sql, k, got)
            zeros += 1
            continue
        if got != 0:
            assert abs(got - r) <= 2e-5 * abs(r), (sql, k, got, r)
            nonzero += 1
            continue
        # a zero group: not selected by the WHERE clause, missing from a factor's BN, or a factor is 0 (per value: 1)
        planned = plan_star_groupby(sql, js)
        column = planned["column"]
        missing = any(k not in bns[f["bn_index"]].infer_machine.compiler.cols[column].pair
                      for f in planned["plan"][1:] if column in f["query"])
        sel = True
        if planned["where"] is not None:
            holder = next(f for f in planned["plan"][1:] if column in f["query"])
            pc = bns[holder["bn_index"]].infer_machine.compiler
            s = pc.select_values(column, planned["where"])
            keys = list(pc.cols[column].pair)
            sel = s is not None and k in pc.cols[column].pair and bool(s[keys.index(k)])
        assert missing or not sel or r == 1, (sql, k, r)
        zeros += 1
    assert nonzero > 1000 and zeros > 100
    # unselected values and values absent from a factor's BN are exactly 0
    sql = ("SELECT t.production_year, COUNT(*) FROM title t,cast_info ci,movie_info mi WHERE t.id=ci.movie_id AND t.id=mi.movie_id "
           "AND mi.info_type_id=3 AND ci.role_id=1 AND t.production_year>2005 GROUP BY t.production_year")
    # (both joined tables are conditioned, so BN 1 and BN 2 both have factors that hold the grouping column: the keys are the
    # union of their values; a table without a condition contributes only its fan-out, and its BN no factor)
    planned = plan_star_groupby(sql, js)
    assert {f["bn_index"] for f in planned["plan"][1:] if "title.production_year" in f["query"]} == {1, 2}
    r, r_all = groupby_sql_batch(ensemble, [sql, sql.replace(" AND t.production_year>2005", "")], js)
    assert all(v == 0 for k, v in r.items() if not (isinstance(k, float) and 2005 < k and k == int(k)))
    assert any(v > 1 for v in r.values())
    # without the range: the values BN 2 lacks (selected, present in BN 1) are 0, the others are not
    absent = [k for k in r_all if k not in bns[2].infer_machine.compiler.cols["title.production_year"].pair]
    assert absent and all(r_all[k] == 0 for k in absent)
    assert sum(v > 0 for v in r_all.values()) > len(r_all) // 2
    # a seeded sample of (query, group) pairs against the fp64 CPU oracle
    rng = np.random.default_rng(2026)
    cand = [i for i, (_, _, got, _) in enumerate(per_value) if got != 0]
    sample = rng.choice(cand, size=min(300, len(cand)), replace=False)
    obns = {i: G.model(f"imdb{i}") for i in range(5)}
    for i in sample:
        sql, k, got, plan = per_value[i]
        tq = O.ensemble_parse_query_all(obns, [copy.deepcopy(plan)])[0]
        r = float(np.asarray(O.ensemble_cardinality(obns, tq)).reshape(-1)[0])
        assert abs(got - r) <= 2e-5 * abs(r), (sql, k, got, r)
