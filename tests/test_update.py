"""Incremental update of a served model (bc_model_set_counts / bc_model_update, DeviceModel.update, Bayescard_BN.update_rows).

The bar is exactness: after inserting rows I and deleting rows D, the counts are C + count(I) - count(D), the fp64 CPTs are
fit.counts_to_cpts of them bit for bit, and the arena (device and host copy) is pack_arena() of that tree model bit for bit.
Query results are then checked against the fp64 oracle on the updated tree model, through every kernel.
"""
import copy
import ctypes as C
import hashlib
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import golden_util as G  # noqa: E402
import groupby_oracle as GO  # noqa: E402
import structure_oracle as SO  # noqa: E402
from bayescard_b200 import _lib as L  # noqa: E402
from bayescard_b200 import fit as F  # noqa: E402
from bayescard_b200.decode import unpack_ranges  # noqa: E402
from bayescard_b200.loader import TreeModel  # noqa: E402
from bayescard_b200.model import rows_to_topological  # noqa: E402
from bayescard_b200.structure import model_from_counts  # noqa: E402
from oracle import bayescard_oracle as O  # noqa: E402

# rows the shipped models' CPTs were fitted on: nrows, except DMV (16 rows fewer) and the IMDB models fitted on a sample
FIT_ROWS = {"census": 2458285, "dmv": 11575467, "imdb0": 3448422, "imdb1": 10_000_000, "imdb2": 10_000_000,
            "imdb3": 6575448, "imdb4": 4050205}
NVCC = "/usr/local/cuda/bin/nvcc"


def golden_fit():
    d = np.load(os.path.join(G.GOLD, "fit_dmv_shaped.npz"))
    n = len(d["card"])
    return d["parent"].astype(np.int32), d["card"].astype(np.int32), d["table"], [d[f"cpd_{v}"] for v in range(n)]


def flat(counts):
    return np.concatenate([np.asarray(c, dtype=np.uint64).reshape(-1) for c in counts])


def fit_tree_model(parent, card, cpts=None):
    """A TreeModel around a tree in topological order (names c0.. = columns)."""
    names = [f"c{v}" for v in range(len(card))]
    if cpts is None:
        cpts = F.counts_to_cpts(parent, card, np.zeros(F.count_layout(parent, card)[1], dtype=np.uint64))
    return TreeModel(table_name="t", nrows=0, node_names=names,
                     structure=tuple(() if parent[v] < 0 else (int(parent[v]),) for v in range(len(card))),
                     attr_type={k: "categorical" for k in names}, algorithm="chow-liu", topo_names=names, infer_names=names,
                     parent=np.asarray(parent, dtype=np.int32), card=np.asarray(card, dtype=np.int32), cpts=list(cpts),
                     dropped_names=[])


def with_counts(tm, counts):
    out = copy.copy(tm)
    out.cpts = F.counts_to_cpts(tm.parent, tm.card, counts)
    out.counts = np.asarray(counts, dtype=np.uint64)
    return out


def host_only_model(tm):
    arena, off, stride = tm.pack_arena()
    fan, foff = tm.pack_fanouts()
    parent = np.ascontiguousarray(tm.parent, dtype=np.int32)
    card = np.ascontiguousarray(tm.card, dtype=np.int32)
    h = C.c_void_p()
    L.check(L.lib().bc_model_create(-1, tm.n_nodes, parent.ctypes.data, card.ctypes.data, off.ctypes.data, stride.ctypes.data,
                                    arena.ctypes.data, arena.size, foff.ctypes.data, fan.ctypes.data, fan.size, C.byref(h)))
    return h


# ------------------------------------------------------------------------------------ host: counts from CPTs
@pytest.mark.parametrize("name", G.MODEL_NAMES)
def test_counts_from_cpts_round_trips_shipped_models(name):
    tm = G.model(name)
    assert F.infer_fit_rows(tm) == FIT_ROWS[name]
    counts = F.counts_from_cpts(tm.parent, tm.card, tm.cpts, FIT_ROWS[name])
    off, total = F.count_layout(tm.parent, tm.card)
    assert counts.dtype == np.uint64 and counts.size == total
    assert int(counts[: int(tm.card[0])].sum()) == FIT_ROWS[name]
    for v, t in enumerate(F.counts_to_cpts(tm.parent, tm.card, counts)):
        assert np.array_equal(t, np.asarray(tm.cpts[v], dtype=np.float64).reshape(t.shape)), (name, v)
    if FIT_ROWS[name] != int(tm.nrows):
        with pytest.raises(ValueError, match="node"):
            F.counts_from_cpts(tm.parent, tm.card, tm.cpts, int(tm.nrows))


def test_counts_from_reference_cpds_equal_oracle_counts():
    parent, card, table, ref = golden_fit()
    counts = F.counts_from_cpts(parent, card, ref, table.shape[0])
    assert np.array_equal(counts, flat(O.fit_counts(parent, card, table)[0]))
    with pytest.raises(ValueError, match="node"):
        F.counts_from_cpts(parent, card, ref, table.shape[0] + 1)


def test_rows_to_topological_matches_the_oracle_refit():
    """A build_from_table-shaped model (tree learned on a table whose column order is not topological): rows in the table's
    column order, permuted by rows_to_topological, count to the model's own counts and refit to its CPTs."""
    rng = np.random.default_rng(7)
    card = np.asarray([5, 3, 7, 4, 6, 2], dtype=np.int32)
    n = 3000
    table = np.stack([rng.integers(0, c, n) for c in card], axis=1).astype(np.uint8)
    table[:, 0] = (table[:, 3] + rng.integers(0, 2, n)) % 5   # dependencies, so that the tree is not a chain in column order
    table[:, 4] = (table[:, 0] * 2 + rng.integers(0, 2, n)) % 6
    counts, _ = SO.pair_counts(card, table)
    mi = SO.mutual_information(card, counts, n)
    parent = SO.chow_liu(mi, root=2)
    tm = model_from_counts(parent, card, counts, [f"col{i}" for i in range(len(card))], root=2, nrows=n)
    assert tm.infer_names != tm.node_names   # the permutation is not the identity
    topo = rows_to_topological(tm, table)
    assert topo.dtype == np.uint8 and topo.shape == (n, len(card))
    assert np.array_equal(flat(O.fit_counts(tm.parent, tm.card, topo)[0]), tm.counts)
    for a, b in zip(O.fit_cpts(tm.parent, tm.card, topo), tm.cpts):
        assert np.array_equal(a.reshape(b.shape), b)
    assert tm.fit_rows == n
    # other integer types are narrowed after a range check
    assert np.array_equal(rows_to_topological(tm, table.astype(np.int64)), topo)
    with pytest.raises(ValueError):
        rows_to_topological(tm, -table.astype(np.int64) - 1)
    with pytest.raises(ValueError):
        rows_to_topological(tm, table[:, :3])


def test_update_arguments_fail_before_any_device_work():
    parent, card, _, ref = golden_fit()
    tm = fit_tree_model(parent, card, ref)
    lib = L.lib()
    h = host_only_model(tm)
    try:
        _, total = F.count_layout(parent, card)
        counts = np.zeros(total + 1, dtype=np.uint64)
        assert lib.bc_model_set_counts(h, counts.ctypes.data, total + 1) == -1
        assert b"counters" in lib.bc_last_error()
        assert lib.bc_model_set_counts(h, counts.ctypes.data, total) == -1   # right total, but a host-only model
        assert b"host-only" in lib.bc_last_error()
        touched = np.zeros(tm.n_nodes, dtype=np.uint8)
        for elem, stride, msg in ((3, 10, b"element size"), (1, 9, b"row stride"), (1, 10, b"no counts")):
            assert lib.bc_model_update(h, None, 0, None, 0, elem, stride, touched.ctypes.data, None, None) == -1
            assert msg in lib.bc_last_error(), (elem, stride, lib.bc_last_error())
        assert lib.bc_model_update(h, None, 5, None, 0, 1, 10, None, None, None) == -1
        assert b"NULL" in lib.bc_last_error()
        assert lib.bc_model_get_counts(h, 0, 1, counts.ctypes.data) == -1 and b"no counts" in lib.bc_last_error()
        assert lib.bc_model_get_counts(h, 5, 6, counts.ctypes.data) == -1 and b"outside" in lib.bc_last_error()
        # the host copy of the arena is pack_arena()'s, zero-padded
        arena = np.zeros(int(lib.bc_model_arena(h, 0, None, 0)), dtype=np.float32)
        assert lib.bc_model_arena(h, 0, arena.ctypes.data, arena.size) == arena.size
        ref_arena = tm.pack_arena()[0]
        assert np.array_equal(arena[: ref_arena.size], ref_arena) and not arena[ref_arena.size:].any()
    finally:
        lib.bc_model_destroy(h)
    # a card that does not fit uint8 bin ids
    wide = fit_tree_model(np.asarray([-1, 0], dtype=np.int32), np.asarray([3, 300], dtype=np.int32))
    h = host_only_model(wide)
    try:
        assert lib.bc_model_update(h, None, 0, None, 0, 1, 2, None, None, None) == -1
        assert b"300 states" in lib.bc_last_error()
        assert lib.bc_model_update(h, None, 0, None, 0, 2, 2, None, None, None) == -1   # uint16 fits: no counts is next
        assert b"no counts" in lib.bc_last_error()
    finally:
        lib.bc_model_destroy(h)


def _sass_functions(cubin):
    sass = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", cubin], capture_output=True, text=True, check=True).stdout
    out, cur = {}, None
    for line in sass.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1)
            out[cur] = []
        elif cur and line.strip():
            out[cur].append(" ".join(line.split()))
    return out


@pytest.mark.skipif(not os.path.exists(NVCC), reason="needs nvcc")
def test_fit_kernels_unchanged_and_update_kernels_do_not_spill(tmp_path):
    """bc_fit_counts' four kernels compile to the SASS they had before the sign parameter existed; the update kernels
    compile for sm_100a without spills."""
    src = os.path.join(ROOT, "bayescard_b200", "csrc", "bc_fit.cu")
    cubin = str(tmp_path / "fit.cubin")
    res = subprocess.run([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-cubin", "-Xptxas", "-v",
                          "-x", "cu", src, "-o", cubin], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    report = {}
    for m in re.finditer(r"Function properties for (\S+)\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores", res.stderr):
        report[m.group(1)] = int(m.group(3))
    upd = {k: v for k, v in report.items() if "upd_" in k}
    assert len(upd) == 3 and not any(upd.values()), upd
    pin = json.load(open(os.path.join(G.GOLD, "fit_count_sass_v1.json")))
    ver = subprocess.run([NVCC, "--version"], capture_output=True, text=True).stdout
    if f"release {pin['nvcc_release']}," not in ver:
        pytest.skip(f"SASS pinned with nvcc {pin['nvcc_release']}")
    got = {}
    for name, body in _sass_functions(cubin).items():
        m = re.search(r"fit_count_kernelI([ht])Lb([01])ELb0E", name)
        if m:
            key = ("uint8" if m.group(1) == "h" else "uint16") + ("_shared" if m.group(2) == "1" else "_direct")
            got[key] = hashlib.sha256("\n".join(body).encode()).hexdigest()
    assert got == pin["sha256"]


# ------------------------------------------------------------------------------------ GPU
def _rel(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-30))) if a.size else 0.0


def _assert_state(dm, tm_new, counts):
    """Counts, fp64 CPTs and both arenas of an updated model against a fresh model of tm_new."""
    assert np.array_equal(dm.get_counts(), counts)
    want = tm_new.pack_arena()[0]
    for from_device in (True, False):
        a = dm.arena(from_device)
        assert np.array_equal(a[: want.size], want) and not a[want.size:].any(), from_device


@pytest.mark.gpu
def test_golden_split_insert_then_delete_is_exact():
    from bayescard_b200.engine import DeviceModel

    parent, card, table, ref = golden_fit()
    k = 20_011
    tm0 = fit_tree_model(parent, card)
    tmA = F.refit(tm0, table[:k])
    assert tmA.fit_rows == k
    dm = DeviceModel(tmA, device=0, specialize=False)
    dm.attach_counts(tmA.counts)
    touched = dm.update(table[k:])
    assert list(touched) == list(range(len(card)))
    full = flat(O.fit_counts(parent, card, table)[0])
    got = dm.get_counts()
    assert np.array_equal(got, full)
    for v, t in enumerate(F.counts_to_cpts(parent, card, got)):
        assert np.array_equal(t.reshape(ref[v].shape), ref[v]), v
    _assert_state(dm, with_counts(tm0, full), full)
    # deleting the same rows gives back the first part's fit exactly
    dm.update(None, table[k:])
    _assert_state(dm, tmA, tmA.counts)
    dm.close()


@pytest.mark.gpu
def test_mixed_batches_uint16_strides_and_no_op():
    import torch

    from bayescard_b200.engine import DeviceModel

    parent, card, table, _ = golden_fit()
    tm0 = fit_tree_model(parent, card)
    base = F.refit(tm0, table[:30_000])
    dm = DeviceModel(base, device=0, specialize=True)
    assert dm.has_spec, dm.spec_error
    dm.attach_counts(base.counts)
    h0 = dm.spec_hash()
    # an empty update and one whose deltas cancel are no-ops: the spec module stays attached
    assert dm.update(None, None).size == 0
    same = table[40_000:40_100]
    assert dm.update(same, same).size == 0
    assert dm.has_spec and dm.spec_hash() == h0
    _assert_state(dm, base, base.counts)
    # insert with duplicates and delete in one call
    ins = np.concatenate([table[30_000:35_000], table[30_000:30_500]])
    dele = table[:2000]
    dm.update(ins, dele)
    want = base.counts + flat(O.fit_counts(parent, card, ins)[0]) - flat(O.fit_counts(parent, card, dele)[0])
    _assert_state(dm, with_counts(tm0, want), want)
    assert dm.has_spec and dm.spec_hash() != h0    # re-specialised for the new CPTs
    # uint16 rows with a row stride wider than the row, through the device-pointer form
    wide = np.zeros((3000, 13), dtype=np.uint16)
    wide[:, :10] = table[35_000:38_000]
    wide[:, 10:] = 999   # padding columns are never read
    d = torch.from_numpy(wide.reshape(-1).view(np.uint8)).cuda()
    s = torch.cuda.current_stream().cuda_stream
    dm.update(d.data_ptr(), None, n_inserted=3000, elem_bytes=2, row_stride=13, stream=s)
    want = want + flat(O.fit_counts(parent, card, table[35_000:38_000])[0])
    _assert_state(dm, with_counts(tm0, want), want)
    dm.close()


@pytest.mark.gpu
def test_rejected_batches_change_nothing():
    from bayescard_b200.engine import DeviceModel, gen_range_queries_host

    parent, card, table, _ = golden_fit()
    tm0 = fit_tree_model(parent, card)
    base = F.refit(tm0, table[:10_000])
    dm = DeviceModel(base, device=0, specialize=True)
    dm.attach_counts(base.counts)
    desc = gen_range_queries_host(base, 3, 0, 512, 1, 4)
    before = dm.run_host(desc, L.DESC_RANGE_U8)
    h0, spec0 = dm.spec_hash(), dm.has_spec
    bad = table[10_000:10_010].copy()
    bad[3, 4] = card[4]                 # one bin id outside node 4's domain
    with pytest.raises(L.BayesCardError, match="outside the model's domains"):
        dm.update(bad)
    rows = table[10_000:10_001]
    dele = np.concatenate([rows] * int(O.fit_counts(parent, card, table[:10_000])[0][0][rows[0, 0]] + 1))
    with pytest.raises(L.BayesCardError, match=r"node \d+, own bin \d+, parent bin -?\d+"):
        dm.update(None, np.concatenate([dele, table[:5]]))   # node 0's count of that bin cannot go below zero
    _assert_state(dm, base, base.counts)
    assert dm.has_spec == spec0 and dm.spec_hash() == h0
    assert np.array_equal(dm.run_host(desc, L.DESC_RANGE_U8), before)
    dm.close()


def _range_case(tm, n, seed):
    from bayescard_b200.engine import gen_range_queries_host

    desc = gen_range_queries_host(tm, seed, 0, n, 1, 5)
    lo, hi = unpack_ranges(tm, desc)
    return desc, lo, hi


def _updated(tm, counts, dm):
    """tm with the counts the device now holds (checked against the host update)."""
    got = dm.get_counts()
    assert np.array_equal(got, counts)
    out = with_counts(tm, counts)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["dmv", "census"])
def test_every_kernel_after_an_update_single_table(name):
    import torch

    from bayescard_b200.engine import DeviceModel
    from bayescard_b200.synth import sample_table_device

    tm = G.model(name)
    counts = F.counts_from_cpts(tm.parent, tm.card, tm.cpts, F.infer_fit_rows(tm))
    dm = DeviceModel(tm, device=0, specialize=(name == "dmv"))
    dm.attach_counts(counts)
    # 1 % of the rows, drawn from a different model of the same shape (so that the CPTs really move), plus a delete
    other = copy.copy(tm)
    other.cpts = [np.asarray(c)[::-1].copy() if v == 0 else np.asarray(c)[::-1, :].copy() for v, c in enumerate(tm.cpts)]
    ins = sample_table_device(other, 100_000, seed=5)
    s = torch.cuda.current_stream().cuda_stream
    touched = dm.update(ins.data_ptr(), None, n_inserted=ins.shape[0], elem_bytes=ins.element_size(), stream=s)
    assert touched.size == tm.n_nodes
    host_ins = ins.cpu().numpy()
    counts = counts + flat(O.fit_counts(tm.parent, tm.card, host_ins)[0])
    dm.update(None, host_ins[:20_000])
    counts = counts - flat(O.fit_counts(tm.parent, tm.card, host_ins[:20_000])[0])
    tm2 = _updated(tm, counts, dm)
    _assert_state(dm, tm2, counts)
    desc, lo, hi = _range_case(tm2, 4096, 11)
    ref = O.dense_tree(tm2, O.range_weights(tm2, lo, hi))
    old = O.dense_tree(tm, O.range_weights(tm, lo, hi))
    assert _rel(old, ref) > 1e-3          # the update moved the answers
    kernels = [L.KERNEL_GENERIC, L.KERNEL_AUTO] + ([L.KERNEL_SPEC] if name == "dmv" else [L.KERNEL_FUSED])
    if name == "dmv":
        assert dm.has_spec, dm.spec_error   # re-specialised for the new CPTs
    for kernel in kernels:
        assert _rel(dm.run_host(desc, L.DESC_RANGE_U8, None, kernel), ref) < 1e-5, kernel
    dm.close()


@pytest.mark.gpu
def test_imdb_pickle_with_inferred_fit_rows_through_k3_with_fanouts():
    from bayescard_b200.engine import DeviceModel
    from bayescard_b200.synth import sample_table_device

    tm = G.model("imdb1")
    rows = F.infer_fit_rows(tm)
    assert rows == 10_000_000
    counts = F.counts_from_cpts(tm.parent, tm.card, tm.cpts, rows)
    dm = DeviceModel(tm, device=0, specialize=False)
    dm.attach_counts(counts)
    other = copy.copy(tm)
    other.cpts = [np.asarray(c)[::-1].copy() if v == 0 else np.asarray(c)[::-1, :].copy() for v, c in enumerate(tm.cpts)]
    ins = sample_table_device(other, 300_000, seed=9).cpu().numpy()
    dm.update(ins)
    counts = counts + flat(O.fit_counts(tm.parent, tm.card, ins)[0])
    tm2 = _updated(tm, counts, dm)
    _assert_state(dm, tm2, counts)
    desc, lo, hi = _range_case(tm2, 4096, 12)
    mask = np.zeros((desc.shape[0], dm.mask_words), dtype=np.uint32)
    for v in range(tm.n_nodes):
        if tm.fan_vector(v) is not None:
            mask[::2, v // 32] |= np.uint32(1 << (v % 32))
    ref = O.dense_tree(tm2, O.range_weights(tm2, lo, hi, mask))
    for kernel in (L.KERNEL_FUSED, L.KERNEL_AUTO, L.KERNEL_GENERIC):
        assert _rel(dm.run_host(desc, L.DESC_RANGE_U8, mask, kernel), ref) < 1e-5, kernel
    dm.close()


@pytest.mark.gpu
def test_large_domain_tree_through_k2():
    from bayescard_b200.engine import DeviceModel
    from bayescard_b200.synth import make_tree_model, pack_ranges_u16, random_range_queries, sample_table_device

    gen = make_tree_model(5, [300, 600, 400, 500, 300], seed=4, parent=[-1, 0, 1, 1, 0])
    table = sample_table_device(gen, 400_000, seed=1).cpu().numpy().astype(np.uint16)
    base = F.refit(gen, table[:200_000])
    dm = DeviceModel(base, device=0, specialize=False)
    dm.attach_counts(base.counts)
    lo, hi = random_range_queries(base, 2048, seed=3, kmax=3)
    desc = pack_ranges_u16(lo, hi)
    for kernel in (L.KERNEL_GEMM, L.KERNEL_GEMM_SIMT):   # plans built under the old CPTs
        assert _rel(dm.run_host(desc, L.DESC_RANGE_U16, None, kernel), O.dense_tree(base, O.range_weights(base, lo, hi))) < 1e-5
    dm.update(table[200_000:], table[:50_000])
    counts = base.counts + flat(O.fit_counts(base.parent, base.card, table[200_000:])[0]) \
        - flat(O.fit_counts(base.parent, base.card, table[:50_000])[0])
    tm2 = _updated(base, counts, dm)
    _assert_state(dm, tm2, counts)
    ref = O.dense_tree(tm2, O.range_weights(tm2, lo, hi))
    for kernel in (L.KERNEL_GEMM, L.KERNEL_GEMM_SIMT, L.KERNEL_AUTO):
        assert _rel(dm.run_host(desc, L.DESC_RANGE_U16, None, kernel), ref) < 1e-5, kernel
    dm.close()


@pytest.mark.gpu
def test_groupby_after_an_update_and_no_stale_module(tmp_path):
    from bayescard_b200.engine import DeviceModel
    from bayescard_b200.synth import sample_table_device

    tm = G.model("dmv")
    counts = F.counts_from_cpts(tm.parent, tm.card, tm.cpts, FIT_ROWS["dmv"])
    dm = DeviceModel(tm, device=0, specialize=False)
    cache = str(tmp_path)
    dm.specialize(cache)
    target = tm.n_nodes - 1
    assert dm.has_spec and dm.specialize_marginal(target, cache)
    old_hash, old_marg = dm.spec_hash(), dm.marginal_hash(target)
    dm.attach_counts(counts)
    other = copy.copy(tm)
    other.cpts = [np.asarray(c)[::-1].copy() if v == 0 else np.asarray(c)[::-1, :].copy() for v, c in enumerate(tm.cpts)]
    ins = sample_table_device(other, 200_000, seed=2).cpu().numpy()
    dm.update(ins)   # specialize=False at construction: nothing is rebuilt
    assert not dm.has_spec and dm.spec_hash() != old_hash and dm.marginal_hash(target) != old_marg
    counts = counts + flat(O.fit_counts(tm.parent, tm.card, ins)[0])
    tm2 = _updated(tm, counts, dm)
    with pytest.raises(L.BayesCardError):
        dm.run_marginal_host(np.tile(dm.bits_default(), (4, 1)), L.DESC_BITS, target, L.KERNEL_SPEC)
    # the cache holds only the old hashes' images: building attaches a module of the NEW CPTs
    dm.specialize(cache)
    assert dm.specialize_marginal(target, cache)
    desc, lo, hi = _range_case(tm2, 2048, 13)
    ref = O.dense_tree(tm2, O.range_weights(tm2, lo, hi))
    assert _rel(dm.run_host(desc, L.DESC_RANGE_U8, None, L.KERNEL_SPEC), ref) < 1e-5
    bits = np.zeros((desc.shape[0], dm.desc_stride(L.DESC_BITS)), dtype=np.uint8)
    import torch

    d_desc = torch.from_numpy(desc).cuda()
    d_bits = torch.from_numpy(bits).cuda()
    dm.convert_device(d_desc.data_ptr(), L.DESC_RANGE_U8, d_bits.data_ptr(), L.DESC_BITS, desc.shape[0],
                      torch.cuda.current_stream().cuda_stream)
    bits = d_bits.cpu().numpy()
    W = O.range_weights(tm2, lo, hi)
    mref = GO.marginal(tm2, W, target)
    for kernel in (L.KERNEL_SPEC, L.KERNEL_GENERIC):   # the marginal module and the expansion
        got = dm.run_marginal_host(bits, L.DESC_BITS, target, kernel)
        assert _rel(got, mref) < 1e-5 or np.allclose(got, mref, rtol=1e-5, atol=1e-12), kernel
    dm.close()


@pytest.mark.gpu
def test_stream_order_k3_update_k3_without_host_sync():
    import torch

    from bayescard_b200.engine import DeviceModel
    from bayescard_b200.synth import sample_table_device

    tm = G.model("imdb3")
    counts = F.counts_from_cpts(tm.parent, tm.card, tm.cpts, FIT_ROWS["imdb3"])
    dm = DeviceModel(tm, device=0, specialize=False)
    dm.attach_counts(counts)
    other = copy.copy(tm)
    other.cpts = [np.asarray(c)[::-1].copy() if v == 0 else np.asarray(c)[::-1, :].copy() for v, c in enumerate(tm.cpts)]
    ins = sample_table_device(other, 500_000, seed=4)
    n = 8192
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        desc = torch.empty((n, dm.desc_stride(L.DESC_RANGE_U8)), dtype=torch.uint8, device="cuda")
        bits = torch.empty((n, dm.desc_stride(L.DESC_BITS)), dtype=torch.uint8, device="cuda")
        out1 = torch.empty(n, dtype=torch.float32, device="cuda")
        out2 = torch.empty(n, dtype=torch.float32, device="cuda")
    s.wait_stream(torch.cuda.current_stream())
    sp = s.cuda_stream
    dm.gen_range_queries_device(21, 0, n, 1, 5, desc.data_ptr(), sp)
    dm.convert_device(desc.data_ptr(), L.DESC_RANGE_U8, bits.data_ptr(), L.DESC_BITS, n, sp)
    dm.run_device(bits.data_ptr(), n, L.DESC_BITS, out1.data_ptr(), kernel=L.KERNEL_FUSED, stream=sp)
    dm.update(ins.data_ptr(), None, n_inserted=ins.shape[0], elem_bytes=1, stream=sp)
    dm.run_device(bits.data_ptr(), n, L.DESC_BITS, out2.data_ptr(), kernel=L.KERNEL_FUSED, stream=sp)
    s.synchronize()
    lo, hi = unpack_ranges(tm, desc.cpu().numpy())
    counts = counts + flat(O.fit_counts(tm.parent, tm.card, ins.cpu().numpy())[0])
    tm2 = _updated(tm, counts, dm)
    assert _rel(out1.cpu().numpy(), O.dense_tree(tm, O.range_weights(tm, lo, hi))) < 1e-5
    assert _rel(out2.cpu().numpy(), O.dense_tree(tm2, O.range_weights(tm2, lo, hi))) < 1e-5
    dm.close()


@pytest.mark.gpu
def test_bayescard_update_rows_on_a_table_model():
    from bayescard_b200.model import Bayescard_BN

    parent, card, table, ref = golden_fit()
    rng = np.random.default_rng(0)
    perm = rng.permutation(len(card))            # the table's columns in an order that is not topological
    tab = np.ascontiguousarray(table[:, perm])
    k = 25_000
    bn = Bayescard_BN.build_from_table(tab[:k], card[perm], specialize=False)
    bn.init_inference_method()
    names = bn.update_rows(tab[k:])
    assert bn.nrows == table.shape[0] and bn.tree.fit_rows == table.shape[0]
    assert set(names) <= set(bn.node_names)
    want = F.refit(bn.tree, rows_to_topological(bn.tree, tab))
    for a, b in zip(bn.tree.cpts, want.cpts):
        assert np.array_equal(a, b)
    assert np.array_equal(bn.tree.counts, want.counts)
    assert np.array_equal(bn.infer_machine.dev.arena()[: want.pack_arena()[0].size], want.pack_arena()[0])
    q = {bn.node_names[0]: [0], bn.node_names[3]: [1]}
    nd = {k: np.ones(1) for k in q}
    ref_q = float(np.asarray(O.ve_query(want, q, nd)).reshape(-1)[0])
    got_q = float(np.asarray(bn.infer_machine.query(q, nd)).reshape(-1)[0])
    assert ref_q > 0 and abs(got_q - ref_q) <= 1e-5 * ref_q
    bn.close()


@pytest.mark.gpu
def test_sharded_model_replicas_stay_identical():
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from bayescard_b200.engine import ShardedModel

    parent, card, table, _ = golden_fit()
    base = F.refit(fit_tree_model(parent, card), table[:20_000])
    sm = ShardedModel(base, [0, 1], specialize=False)
    sm.attach_counts(base.counts)
    sm.update(table[20_000:], table[:1000])
    a, b = sm.replicas[0].arena(), sm.replicas[1].arena()
    assert np.array_equal(a, b)
    assert np.array_equal(sm.replicas[0].get_counts(), sm.replicas[1].get_counts())
    desc, lo, hi = _range_case(base, 4096, 5)
    r = sm.run_host(desc, L.DESC_RANGE_U8)
    assert np.array_equal(r[:2048], sm.replicas[0].run_host(desc[:2048], L.DESC_RANGE_U8))
    assert np.array_equal(r[2048:], sm.replicas[0].run_host(desc[2048:], L.DESC_RANGE_U8))
    sm.close()
