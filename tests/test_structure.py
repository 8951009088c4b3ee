"""Structure learning (bc_pair_counts / bc_chow_liu + bayescard_b200/structure.py) against the numpy reference in
tests/structure_oracle.py (pair counts, mutual information, Prim) and the existing oracle (CPTs, query probabilities).

Counting is integer work: the bar is bit-exact counts.  Mutual information is fp64 on both sides (1e-12).  The learned
tree is compared with the oracle's Prim where every decision has a margin, and by total MI where ties are exact.
pomegranate cannot run here, so the structure is pinned to the oracle's reading of its loop, not to pomegranate itself.
"""
import itertools
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import golden_util as G  # noqa: E402
from bayescard_b200 import _lib as L  # noqa: E402
from bayescard_b200 import structure as S  # noqa: E402
from bayescard_b200.loader import TreeModel, topological_order  # noqa: E402
from oracle import bayescard_oracle as O  # noqa: E402
import structure_oracle as SO  # noqa: E402


def tree_weight(parent, mi):
    return sum(mi[v, p] for v, p in enumerate(parent) if p >= 0)


def is_spanning_tree(parent, root):
    n = len(parent)
    if parent[root] != -1 or sum(p < 0 for p in parent) != 1:
        return False
    for v in range(n):  # every node reaches the root without a cycle
        seen, u = set(), v
        while u != root:
            if u in seen:
                return False
            seen.add(u)
            u = parent[u]
    return True


# ---------------------------------------------------------------------------------------------------- CPU


def test_pair_count_layout():
    marg, pair, total = S.pair_count_layout([2, 3, 4])
    assert list(marg) == [0, 2, 5]
    assert pair[0, 1] == 9 and pair[0, 2] == 15 and pair[1, 2] == 23 and total == 35
    assert (pair[np.tril_indices(3)] == -1).all()
    rng = np.random.default_rng(0)
    card = [3, 1, 5, 2]
    table = np.stack([rng.integers(0, c, 50) for c in card], axis=1).astype(np.uint8)
    counts, bad = SO.pair_counts(card, table)
    assert bad == 0 and counts.size == S.pair_count_layout(card)[2]
    marg, pair, _ = S.pair_count_layout(card)
    blk = counts[pair[0, 2]: pair[0, 2] + 15].reshape(3, 5)
    want = np.zeros((3, 5), dtype=np.uint64)
    np.add.at(want, (table[:, 0], table[:, 2]), 1)
    assert np.array_equal(blk, want) and np.array_equal(counts[marg[2]: marg[2] + 5], want.sum(axis=0))


def test_oracle_prim_is_a_maximum_spanning_tree():
    rng = np.random.default_rng(1)
    for n in (2, 3, 4, 5, 6):
        edges = list(itertools.combinations(range(n), 2))
        for trial in range(6):
            mi = rng.random((n, n))
            mi = np.triu(mi, 1) + np.triu(mi, 1).T
            best = -1.0
            for sub in itertools.combinations(edges, n - 1):  # all spanning trees (brute force)
                comp = list(range(n))

                def find(x):
                    while comp[x] != x:
                        x = comp[x]
                    return x
                ok = True
                for a, b in sub:
                    ra, rb = find(a), find(b)
                    if ra == rb:
                        ok = False
                        break
                    comp[ra] = rb
                if ok:
                    best = max(best, sum(mi[a, b] for a, b in sub))
            root = trial % n
            parent = SO.chow_liu(mi, root)
            assert is_spanning_tree(parent, root)
            assert abs(tree_weight(parent, mi) - best) < 1e-12


def test_oracle_prim_tie_rule():
    # all equal: x = the root first, y ascending -> a star
    assert list(SO.chow_liu(np.ones((4, 4)), 0)) == [-1, 0, 0, 0]
    assert list(SO.chow_liu(np.ones((4, 4)), 2)) == [2, 2, -1, 2]
    # (0,1) and (0,2) tie: y = 1 first; then (0,3) and (1,3) tie: x = 0, which joined first
    mi = np.zeros((4, 4))
    for a, b, w in ((0, 1, 1.0), (0, 2, 1.0), (0, 3, 0.5), (1, 3, 0.5), (1, 2, 0.2)):
        mi[a, b] = mi[b, a] = w
    assert list(SO.chow_liu(mi, 0)) == [-1, 0, 0, 0]
    # a later-joined x only wins with a strictly larger MI
    mi[2, 3] = mi[3, 2] = 0.6
    assert list(SO.chow_liu(mi, 0)) == [-1, 0, 0, 2]


def toy_table(n=5000, seed=2):
    rng = np.random.default_rng(seed)
    a = rng.integers(0, 4, n)
    b = (a + rng.integers(0, 2, n)) % 5
    c = rng.integers(0, 3, n)
    d = (b * 2 + (rng.random(n) < 0.1)) % 7
    return np.stack([a, b, c, d], axis=1).astype(np.uint8), np.asarray([4, 5, 3, 7])


def test_model_from_counts_numbering_and_round_trip(tmp_path):
    table, card = toy_table()
    counts, bad = SO.pair_counts(card, table)
    mi = SO.mutual_information(card, counts, len(table) - bad)
    for root in (0, 3):
        parent = SO.chow_liu(mi, root)
        tm = S.model_from_counts(parent, card, counts, ["a", "b", "c", "d"], root, "toy", len(table))
        order = topological_order(tm.structure)
        assert tm.infer_names == [tm.node_names[i] for i in order] and tm.topo_names == tm.infer_names
        assert tm.infer_names[0] == tm.node_names[root] and tm.parent[0] == -1
        # the CPTs are pgmpy's MLE of the learned tree (oracle fit on the table permuted to topological order)
        want = O.fit_cpts(tm.parent, tm.card, table[:, order])
        assert all(np.array_equal(x, y) for x, y in zip(tm.cpts, want))
        tm.save(str(tmp_path / "m.npz"))
        tm.save_flat(str(tmp_path / "m.bcm"))
        for back in (TreeModel.load(str(tmp_path / "m.npz")), TreeModel.load_flat(str(tmp_path / "m.bcm"))):
            assert back.structure == tm.structure and back.infer_names == tm.infer_names
            assert np.array_equal(back.parent, tm.parent) and np.array_equal(back.card, tm.card)
            assert all(np.array_equal(x, y) for x, y in zip(back.cpts, tm.cpts))
            assert back.algorithm == "chow-liu" and back.encoding == tm.encoding


def test_bad_arguments_fail_before_any_device_work():
    lib = L.lib()
    card = np.full(200, 100, dtype=np.int32)  # S = 20 000 > 16 384
    rc = lib.bc_pair_counts(0, 200, card.ctypes.data, None, 1, 0, 200, 1, 0, None, None)
    assert rc == L.ELIMIT and b"16384" in lib.bc_last_error()
    card = np.asarray([3, 300], dtype=np.int32)  # 300 does not fit uint8
    rc = lib.bc_pair_counts(0, 2, card.ctypes.data, None, 1, 0, 2, 1, 0, None, None)
    assert rc == -1 and b"card" in lib.bc_last_error()
    card = np.asarray([3, 4], dtype=np.int32)
    rc = lib.bc_pair_counts(0, 2, card.ctypes.data, None, 1, 10, 2, 1, 3 + 4 + 12, None, None)
    assert rc == -1 and b"NULL" in lib.bc_last_error()
    rc = lib.bc_pair_counts(0, 1, card.ctypes.data, None, 1, 0, 1, 1, 3, None, None)
    assert rc == -1 and b"n_cols" in lib.bc_last_error()
    parent = np.zeros(2, dtype=np.int32)
    for root in (-1, 2):
        rc = lib.bc_chow_liu(0, 2, card.ctypes.data, None, 1, 0, 2, root, None, 0, parent.ctypes.data, None, None, None)
        assert rc == -1 and b"root" in lib.bc_last_error()


# ---------------------------------------------------------------------------------------------------- GPU


def gpu_table(tm, n, seed):
    from bayescard_b200.synth import sample_table_device

    t = sample_table_device(tm, n, seed)
    return t.cpu().numpy().view(np.uint16) if t.element_size() == 2 else t.cpu().numpy()


def check_counts(table, card):
    got, bad = S.pair_counts(table, card)
    want, want_bad = SO.pair_counts(card, table)
    assert bad == want_bad and np.array_equal(got, want), (table.shape, list(card))
    return got, bad


@pytest.mark.gpu
def test_gpu_counts_bit_exact():
    d = np.load(os.path.join(G.GOLD, "fit_dmv_shaped.npz"))
    table, card = d["table"], d["card"]
    check_counts(table, card)
    for n in (0, 1, 31, 127, 128, 129, 4097):
        check_counts(table[:n], card)
    rng = np.random.default_rng(4)
    for S_total in (256, 257, 384, 385, 512):  # S a multiple of 128 (and of 256), and one above
        cards = [16] * (S_total // 16) + ([S_total % 16] if S_total % 16 else [])
        t = np.stack([rng.integers(0, c, 3000) for c in cards], axis=1).astype(np.uint8)
        t[:, 3] = t[:, 2]  # co-occurring states inside one window pair
        check_counts(t, cards)
    # uint16, cards above 256, S in the thousands (many window pairs)
    cards = [300, 700, 2, 1200, 260]
    t = np.stack([rng.integers(0, c, 20_000) for c in cards], axis=1).astype(np.uint16)
    t[:, 4] = t[:, 0] % 260
    check_counts(t, cards)
    # 68-column Census-shaped sample
    census = G.model("census")
    check_counts(gpu_table(census, 50_000, 3), census.card)
    # row stride > n_cols: a column slice of a wider table
    import torch

    wide = np.concatenate([table, np.full((len(table), 5), 255, np.uint8)], axis=1)
    d_wide = torch.from_numpy(wide).cuda()
    _, _, total = S.pair_count_layout(card)
    out = torch.empty(total + 1, dtype=torch.int64, device="cuda")
    bad = S.pair_counts_device(card, d_wide.data_ptr(), len(wide), 1, wide.shape[1], out.data_ptr(), 0,
                               torch.cuda.current_stream().cuda_stream, True)
    assert bad == 0 and np.array_equal(out[:total].cpu().numpy().astype(np.uint64), SO.pair_counts(card, table)[0])
    # out-of-domain ids: the rows are skipped, as bc_fit_counts skips them
    from bayescard_b200 import fit as F

    dirty = table[:5000].copy()
    dirty[::7, 4] = 255
    dirty[3::11, 9] = 200
    _, bad = check_counts(dirty, card)
    _, _, fit_bad = F.fit_cpts(d["parent"], card, dirty)
    assert bad == fit_bad > 0


@pytest.mark.gpu
def test_gpu_mutual_information_and_tree():
    d = np.load(os.path.join(G.GOLD, "fit_dmv_shaped.npz"))
    table, card = d["table"], d["card"]
    for t, c in ((table, card), (gpu_table(G.model("census"), 50_000, 3), G.model("census").card)):
        parent, mi, bad = S.chow_liu(t, c)
        counts, want_bad = SO.pair_counts(c, t)
        want = SO.mutual_information(c, counts, len(t) - want_bad)
        assert bad == want_bad
        assert np.all(np.abs(mi - want) <= 1e-12 * np.maximum(np.abs(want), 1e-3))
        assert np.array_equal(S.mutual_information(t, c)[0], mi)
        want_parent = SO.chow_liu(want, 0)
        if np.array_equal(parent, want_parent):
            continue
        # only exact ties may differ: then the device's Prim on the oracle's matrix must agree with the oracle
        assert is_spanning_tree(parent, 0)
        assert abs(tree_weight(parent, want) - tree_weight(want_parent, want)) <= 1e-12 * tree_weight(want_parent, want)
    # DMV-shaped table: every Prim decision has a margin -> the same tree; also for another root
    parent, mi, _ = S.chow_liu(table, card, root=4)
    assert np.array_equal(parent, SO.chow_liu(mi, 4))


@pytest.mark.gpu
def test_gpu_tie_heavy_tables():
    rng = np.random.default_rng(5)
    n = 20_000
    a = rng.integers(0, 6, n)
    cols = [a, a.copy(), np.zeros(n, np.int64), rng.integers(0, 3, n), (a + (rng.random(n) < 0.3)) % 6, a.copy(),
            rng.integers(0, 2, n)]
    card = [6, 6, 1, 3, 6, 6, 2]
    table = np.stack(cols, axis=1).astype(np.uint8)
    for root in (0, 2, 6):
        parent, mi, _ = S.chow_liu(table, card, root)
        want = SO.mutual_information(card, *(lambda c: (c[0], n - c[1]))(SO.pair_counts(card, table)))
        assert is_spanning_tree(parent, root)
        best = tree_weight(SO.chow_liu(want, root), want)
        assert abs(tree_weight(parent, want) - best) <= 1e-12 * max(best, 1.0)
        # duplicated columns tie exactly: the tie rule picks the first-joined x and the smallest y
        assert np.array_equal(parent, SO.chow_liu(mi, root))


@pytest.mark.gpu
def test_gpu_dmv_full_size_tree_counts_equal_fit_counts():
    import torch

    from bayescard_b200 import fit as F

    tm = G.model("dmv")
    n = 11_591_877
    from bayescard_b200.synth import sample_table_device

    t = sample_table_device(tm, n, 7)
    card = np.asarray(tm.card)
    parent, mi, bad = S.chow_liu(t.cpu().numpy(), card)
    assert bad == 0 and np.array_equal(parent, tm.parent), (parent, tm.parent)   # recovery of the shipped tree
    # the learned tree's counts gathered from G equal bc_fit_counts on that tree, bit for bit
    learned = S.learn_tree_model(t.cpu().numpy(), card)
    order = [learned.node_names.index(x) for x in learned.infer_names]
    tt = t[:, order].contiguous()
    off, total = F.count_layout(learned.parent, learned.card)
    counts = torch.empty(total + 1, dtype=torch.int64, device="cuda")
    F.fit_counts_device(learned.parent, learned.card, tt.data_ptr(), n, 1, tm.n_nodes, counts.data_ptr(), 0,
                        torch.cuda.current_stream().cuda_stream)
    want = F.counts_to_cpts(learned.parent, learned.card, counts[:total].cpu().numpy().astype(np.uint64))
    assert all(np.array_equal(a, b) for a, b in zip(learned.cpts, want))
    assert learned.nrows == n


@pytest.mark.gpu
@pytest.mark.parametrize("name,rows", [("imdb1", 1_000_000), ("imdb2", 1_000_000), ("imdb3", 1_000_000),
                                       ("imdb4", 1_000_000), ("imdb0", 1_000_000), ("census", 2_458_285)])
def test_gpu_recovers_shipped_trees(name, rows):
    tm = G.model(name)
    t = gpu_table(tm, rows, 11)
    parent, mi, bad = S.chow_liu(t, tm.card)
    assert bad == 0 and is_spanning_tree(parent, 0)
    if name in ("census", "imdb0"):  # exact population ties (deterministic child columns): equal total MI only
        want = tree_weight(tm.parent, mi)
        assert abs(tree_weight(parent, mi) - want) <= 1e-12 * want
    else:
        assert np.array_equal(parent, tm.parent)


@pytest.mark.gpu
def test_gpu_build_from_table_end_to_end():
    from bayescard_b200.model import Bayescard_BN
    from bayescard_b200.synth import random_range_queries

    tm = G.model("dmv")
    n = 11_591_877
    t = gpu_table(tm, n, 9)
    bn = Bayescard_BN.build_from_table(t, tm.card, names=tm.infer_names, table_name="dmv")
    bn.init_inference_method()
    learned = bn.tree
    assert learned.infer_names == tm.infer_names and np.array_equal(learned.parent, tm.parent)
    lo, hi = random_range_queries(learned, 10_000, seed=3, kmax=5)
    queries = []
    for q in range(len(lo)):
        queries.append({learned.infer_names[v]: list(range(int(lo[q, v]), int(hi[q, v]) + 1))
                        for v in range(learned.n_nodes) if lo[q, v] > 0 or hi[q, v] < learned.card[v] - 1})
    keep = [i for i, q in enumerate(queries) if q]
    got = bn.query_batch([queries[i] for i in keep], return_prob=True)
    lo, hi = lo[keep], hi[keep]
    want = O.dense_tree(learned, O.range_weights(learned, lo, hi))
    assert np.max(np.abs(got - want) / np.maximum(np.abs(want), 1e-30)) < 1e-5
    # against the shipped model the learned one differs by sampling noise only.  A query probability p is a product of
    # at most n_nodes estimated factors, each a ratio of counts of at least ~n p rows, so its relative standard deviation
    # is at most ~sqrt(n_nodes / (n p)), i.e. sqrt(n_nodes p / n) absolute; we allow 6 of those
    shipped = O.dense_tree(tm, O.range_weights(tm, lo, hi))
    bound = 6 * np.sqrt(tm.n_nodes * np.maximum(shipped, got) / n)
    assert np.all(np.abs(got - shipped) <= bound)
    bn.close()
