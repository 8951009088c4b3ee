"""The fan-out mask contract on every query kernel, and output bounds.

``mask_words = ceil(n_nodes / 32)`` uint32 per query; bit v multiplies w_v by ``fanouts[v]`` (include/bayescard_b200.h).  The
shipped models only ever set bits 1-9 of word 0, so the synthetic models here put fan-out vectors on both sides of every word
boundary, on the root, on one-state columns' neighbours and next to all-zero CPT rows:

  wide70          70 columns (3 mask words), cards 1-8 with one-state columns (one a leaf, one with children), fan-out vectors
                  on nodes 0, 31, 32, 33, 63, 64, 69 (one with an exact 0), an all-zero CPT row on node 33 and rows with equal
                  numbers of zeros (the seed row of the generated code is not row 0)
  chain_fan_root  a chain of 6 with fan-out vectors on the root and the leaf: in the marginal of every target below the root,
                  the root has no lambda (the selp between two immediates)
  wide_bits       40 columns, four 200-256-state leaves whose BITS columns cross 32-bit words, fan-out vectors on nodes >= 32
                  (the fused kernel declines it: columns of more than 128 states)
  one_node        a single column with a fan-out vector

Host tests interpret the generated PTX (``join_groupby_oracle.interpret_masked``) and assemble it with ptxas; GPU tests run
every kernel against the fp64 oracle (``oracle.range_weights`` / ``dense_tree``, ``groupby_oracle.marginal``) at 1e-5
relative, compare the host pipelines with the device-buffer launch bit for bit, and check that no entry point writes outside
its n results.  The specialised modules of these models are assembled into a per-session temporary cache, never into the
library's shared one."""
import os

import numpy as np
import pytest

import groupby_oracle as GO
import join_groupby_oracle as JO
from bayescard_b200 import _lib as L
from bayescard_b200 import aot
from bayescard_b200.decode import PredicateCompiler, dense_to_wsparse
from bayescard_b200.engine import DeviceModel
from bayescard_b200.synth import make_tree_model, pack_ranges_u16, random_range_queries
from oracle import bayescard_oracle as O

RTOL = 1e-5
MODELS = ["wide70", "chain_fan_root", "wide_bits", "one_node"]
# targets of the specialised marginal modules under test (wide70: both sides of the word boundaries, node 33 holds the
# all-zero CPT row, 5 and 66 are one-state columns -- 5 with children, 66 a leaf)
MARGINAL_TARGETS = {"wide70": [0, 5, 31, 32, 33, 66, 69], "chain_fan_root": list(range(6)), "wide_bits": [0, 33, 39],
                    "one_node": [0]}
SENTINEL = 0x7FC0DEAD   # a NaN bit pattern no kernel computes
GUARD = 4096            # bytes of guard on each side of an output buffer


# ------------------------------------------------------------------------------------ synthetic models
def with_fanouts(m, nodes, seed, zero=None):
    """Fan-out vectors of 1 - 1000 (fp32-exact, like the IMDB vectors' range) on ``nodes``; ``zero = (node, state)`` makes
    one entry an exact 0."""
    rng = np.random.default_rng(seed)
    for v in nodes:
        f = rng.uniform(1.0, 1000.0, int(m.card[v])).astype(np.float32).astype(np.float64)
        if zero is not None and zero[0] == v:
            f[zero[1]] = 0.0
        m.fanouts[m.infer_names[v]] = f
    return m


def _renormalise(t):
    t /= t.sum(axis=0, keepdims=True)


def _wide70():
    n = 70
    rng = np.random.default_rng(70)
    parent = np.array([-1] + [int(rng.integers(0, i)) for i in range(1, n)], dtype=np.int32)
    card = rng.integers(2, 9, size=n).astype(np.int32)
    inner = set(int(p) for p in parent[1:])
    assert 5 in inner and 66 not in inner and 20 in inner
    card[[5, 20, 66]] = 1          # one-state columns: two with children, one leaf
    card[33] = max(card[33], 4)    # room for an all-zero row
    card[0] = max(card[0], 3)
    m = make_tree_model(n, card, seed=7, dtype=np.float32, parent=parent)
    t = m.cpts[33]
    t[1, :] = 0.0                  # an all-zero CPT row (the state holds no mass whatever its parent)
    _renormalise(t)
    for v in (32, 45):             # one exact zero in row 0: the rows below tie on their number of zeros
        t = m.cpts[v]
        t[0, 0] = 0.0
        _renormalise(t)
    return with_fanouts(m, [0, 31, 32, 33, 63, 64, 69], seed=1, zero=(64, 0))


def _chain_fan_root():
    m = make_tree_model(6, [4, 3, 5, 2, 6, 3], seed=6, dtype=np.float32, parent=[-1, 0, 1, 2, 3, 4])
    return with_fanouts(m, [0, 5], seed=2)


def _wide_bits():
    n = 40
    big = {10: 200, 21: 256, 33: 229, 36: 250}   # leaves: their BITS columns span 7-8 words and cross word boundaries
    rng = np.random.default_rng(40)
    small = [0]
    parent = [-1]
    for i in range(1, n):
        parent.append(int(rng.choice(small)))
        if i not in big:
            small.append(i)
    card = rng.integers(2, 7, size=n).astype(np.int32)
    for v, c in big.items():
        card[v] = c
    m = make_tree_model(n, card, seed=9, dtype=np.float32, parent=parent)
    return with_fanouts(m, [32, 33, 36, 39], seed=3, zero=(33, 200))


def _one_node():
    m = make_tree_model(1, [5], seed=1, dtype=np.float32, parent=[-1])
    return with_fanouts(m, [0], seed=4)


_BUILDERS = {"wide70": _wide70, "chain_fan_root": _chain_fan_root, "wide_bits": _wide_bits, "one_node": _one_node}
_MODELS = {}


def model(name):
    if name not in _MODELS:
        _MODELS[name] = _BUILDERS[name]()
    return _MODELS[name]


def test_synthetic_models_have_the_shapes_under_test():
    m = model("wide70")
    words = (m.n_nodes + 31) // 32
    assert words == 3 and JO.fan_nodes(m) == [0, 31, 32, 33, 63, 64, 69]
    assert (m.card == 1).sum() >= 3 and m.card[66] == 1 and 66 not in set(m.parent[1:].tolist())
    assert m.card.min() == 1 and m.card.max() == 8
    assert not np.asarray(m.cpts[33])[1].any() and (m.fan_vector(64) == 0).sum() == 1
    for v in range(1, m.n_nodes):   # stochastic columns: K1 skips unconstrained subtrees because their sums are 1
        assert np.allclose(np.asarray(m.cpts[v], dtype=np.float64).sum(axis=0), 1.0, atol=1e-6)
    wb = model("wide_bits")
    dm = DeviceModel(wb, device=-1, specialize=False)
    offs = dm.bits_offset
    crossing = [v for v in range(wb.n_nodes) if offs[v] // 32 != (offs[v] + int(wb.card[v]) - 1) // 32]
    assert {10, 21, 33, 36} <= set(crossing) and all(v >= 32 for v in JO.fan_nodes(wb))
    dm.close()


# ------------------------------------------------------------------------------------ queries and the oracle
def all_ones(m):
    row = np.zeros((m.n_nodes + 31) // 32, dtype=np.uint32)
    for v in range(m.n_nodes):
        row[v >> 5] |= np.uint32(1 << (v & 31))
    return row


def rand_masks(m, nq, rng, p=0.5):
    """Random mask rows over the model's nodes (bits at or beyond n_nodes stay clear); row 0 is all ones, row 1 all zeros."""
    bits = rng.random((nq, m.n_nodes)) < p
    mask = np.zeros((nq, (m.n_nodes + 31) // 32), dtype=np.uint32)
    for v in range(m.n_nodes):
        mask[:, v >> 5] |= bits[:, v].astype(np.uint32) << np.uint32(v & 31)
    if nq > 1:
        mask[0], mask[1] = all_ones(m), 0
    return mask


def only_fan_bits(m, mask):
    keep = np.zeros(mask.shape[1], dtype=np.uint32)
    for v in JO.fan_nodes(m):
        keep[v >> 5] |= np.uint32(1 << (v & 31))
    return mask & keep[None, :]


def apply_mask(m, W, mask):
    """fp64 weights with bit v of each row's mask multiplying w_v by fanouts[v] (``mask`` None: unchanged)."""
    out = []
    for v in range(m.n_nodes):
        w = np.asarray(W[v], dtype=np.float64)
        f = m.fan_vector(v)
        if f is not None and mask is not None:
            bit = ((mask[:, v >> 5] >> np.uint32(v & 31)) & 1).astype(bool)
            w = np.where(bit[:, None], w * f[None, :], w)
        out.append(w)
    return out


class Batch:
    """``nq`` random range queries on ``m`` as BITS, DENSE_F32 (fractional weights, NaN in the pad floats) and RANGE rows,
    with their fp64 weights (DENSE rows and weights for the first ``n_dense``)."""

    def __init__(self, m, dm, nq, seed, n_dense=None):
        rng = np.random.default_rng(seed)
        self.nq = nq
        nd = nq if n_dense is None else n_dense
        self.lo, self.hi = random_range_queries(m, nq, seed=seed, kmax=min(m.n_nodes, 12))
        if nq > 2:
            self.lo[2], self.hi[2] = 0, m.card - 1   # unconstrained
        self.W = O.range_weights(m, self.lo[:nd], self.hi[:nd])
        self.bits = PredicateCompiler(m).pack_bits(self.lo, self.hi)
        self.range16 = pack_ranges_u16(self.lo, self.hi)
        self.Wd = []
        self.dense = np.full((nd, dm.dense_width), np.nan, dtype=np.float32)
        for v in range(m.n_nodes):
            w = (self.W[v] * (0.25 + 0.75 * rng.random((nd, 1)))).astype(np.float32)
            self.Wd.append(w.astype(np.float64))
            o = int(dm.dense_offset[v])
            self.dense[:, o:o + int(m.card[v])] = w

    def rows(self, fmt):
        return {L.DESC_BITS: self.bits, L.DESC_DENSE_F32: self.dense, L.DESC_RANGE_U16: self.range16}[fmt]

    def weights(self, fmt):
        return self.Wd if fmt == L.DESC_DENSE_F32 else self.W


def oracle(m, lo, hi, mask, step=16384):
    """fp64 results of range rows ``lo``, ``hi`` with ``mask`` (or None), in slices of ``step`` queries."""
    return np.concatenate([O.dense_tree(m, apply_mask(m, O.range_weights(m, lo[s:s + step], hi[s:s + step]),
                                                      None if mask is None else mask[s:s + step])) for s in range(0, len(lo), step)])


def assert_close(got, ref, what=""):
    got, ref = np.asarray(got, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    err = np.abs(got - ref) / np.maximum(np.abs(ref), 1e-300)
    err[(ref == 0) & (got == 0)] = 0
    assert err.max() <= RTOL, (what, float(err.max()), np.unravel_index(int(err.argmax()), err.shape))


# ------------------------------------------------------------------------------------ host: the generated code
@pytest.mark.parametrize("name", MODELS)
def test_generated_code_applies_multiword_masks_on_the_host(name):
    """bc_spec_bits / bc_spec_dense and bc_marg_bits / bc_marg_dense interpreted in fp32 with random 3-word mask rows, the
    all-ones and the all-zero row and a NULL mask, against the fp64 oracle."""
    m = model(name)
    dm = DeviceModel(m, device=-1, specialize=False)
    rng = np.random.default_rng(17)
    b = Batch(m, dm, 3, seed=5)
    masks = np.concatenate([rand_masks(m, 3, rng), rand_masks(m, 1, rng)])   # all ones, all zeros, two random rows
    cases = [(mask[None, :], mask) for mask in masks] + [(None, None)]
    src = dm.spec_source()
    for q in range(b.nq):
        for ref_mask, mask in cases:
            for fmt, entry in ((L.DESC_BITS, "bc_spec_bits"), (L.DESC_DENSE_F32, "bc_spec_dense")):
                W = apply_mask(m, [w[q:q + 1] for w in b.weights(fmt)], ref_mask)
                got = JO.interpret_masked(src, entry, b.rows(fmt)[q].tobytes(), mask)
                assert_close(got, O.dense_tree(m, W), (name, entry, q, mask))
    for t in MARGINAL_TARGETS[name]:
        msrc = dm.marginal_source(t)
        for q in range(b.nq):
            for ref_mask, mask in cases[1:4] + cases[-1:]:
                for fmt, entry in ((L.DESC_BITS, "bc_marg_bits"), (L.DESC_DENSE_F32, "bc_marg_dense")):
                    W = apply_mask(m, [w[q:q + 1] for w in b.weights(fmt)], ref_mask)
                    got = JO.interpret_masked(msrc, entry, b.rows(fmt)[q].tobytes(), mask)
                    assert_close(got, GO.marginal(m, W, t)[0], (name, entry, t, q, mask))
    dm.close()


def test_generated_code_takes_the_shape_dependent_branches():
    """The branches of the generator that only these models reach are present in the code the tests run."""
    dm = DeviceModel(model("wide70"), device=-1, specialize=False)
    src = dm.spec_source()
    assert "[%rtmp+8]" in src                                     # mask word 2 is loaded
    assert "mad.lo.u64 %rtmp, %rqc, 12, %rfmask;" in src         # 4 * mask_words bytes per query
    assert "mov.f32" in dm.marginal_source(33).split("path node 33")[1]   # the zero register of the all-zero row
    dm.close()
    dc = DeviceModel(model("chain_fan_root"), device=-1, specialize=False)
    for t in range(1, 6):   # the root's only child is on the path: a selp between T_0[c] * fanouts[c] and T_0[c]
        root = dc.marginal_source(t).split("path node 0: card 4 (root)")[1].split("path node 1")[0]
        assert root.count("selp.f32") >= 4, t
    dc.close()


def test_fused_kernel_declines_columns_beyond_128_states():
    """K3 chains every k-step of an edge into one fp32 accumulator; past 128 states below the root that loses the 1e-5
    accuracy, so the planner declines the model with a reason (and AUTO serves it with the other kernels)."""
    import ctypes as C

    info = (C.c_int32 * 8)()
    for name, served in (("wide70", True), ("chain_fan_root", True), ("wide_bits", False)):
        dm = DeviceModel(model(name), device=-1, specialize=False)
        rc = L.lib().bc_model_fused_plan(dm._h, info, None, 0)
        assert (rc == 0) == served, (name, rc)
        if not served:
            assert rc == L.ELIMIT and b"more than 128 states" in L.lib().bc_last_error()
        dm.close()


@pytest.fixture(scope="session")
def cubin_cache(tmp_path_factory):
    """A per-session cache of the synthetic models' cubins: ``assemble(name, targets)`` runs ptxas -arch=sm_100a on the spec
    module and the marginal modules of ``targets`` in parallel (the files bc_model_specialize / _marginal look for)."""
    d = str(tmp_path_factory.mktemp("fanout_cubins"))

    def assemble(name, targets):
        m = model(name)
        if name not in assemble.spec:
            assemble.spec[name] = aot.build_cubin(m, cache_dir=d)
        GO.assemble_marginals(m, targets, d)
        return d

    assemble.spec = {}
    return assemble


def test_generated_modules_assemble_for_sm_100a(cubin_cache):
    """ptxas accepts the spec module and every marginal module of every synthetic model."""
    for name in MODELS:
        m = model(name)
        d = cubin_cache(name, range(m.n_nodes))
        dm = DeviceModel(m, device=-1, specialize=False)
        for f in ["spec_%016x.cubin" % dm.spec_hash()] + ["marg_%016x.cubin" % dm.marginal_hash(t) for t in range(m.n_nodes)]:
            assert os.path.getsize(os.path.join(d, f)) > 0, (name, f)
        dm.close()


# ------------------------------------------------------------------------------------ GPU
def _torch():
    import torch

    return torch


def dev(a):
    """A host array on cuda:0 (raw bytes)."""
    return _torch().from_numpy(np.ascontiguousarray(a).reshape(-1).view(np.uint8)).to("cuda:0")


class Guarded:
    """An output buffer of ``n`` 32-bit words with GUARD bytes of SENTINEL on each side."""

    def __init__(self, n):
        torch = _torch()
        self.n, self.g = n, GUARD // 4
        self.buf = torch.full((2 * self.g + n,), SENTINEL, dtype=torch.int32, device="cuda:0")
        self.ptr = self.buf.data_ptr() + 4 * self.g

    def values(self, dtype=np.float32):
        return self.buf[self.g:self.g + self.n].cpu().numpy().view(dtype)

    def intact(self):
        return bool((self.buf[:self.g] == SENTINEL).all()) and bool((self.buf[self.g + self.n:] == SENTINEL).all())


def spec_model(name, cubin_cache, targets=()):
    m = model(name)
    d = cubin_cache(name, targets)
    dm = DeviceModel(m, device=0, specialize=True, cache_dir=d)
    assert dm.has_spec, dm.spec_error
    for t in targets:
        assert dm.specialize_marginal(t, d), dm.marginal_error.get(t)
    return dm


def run_or_refused(fn, kernel, what):
    """``fn()``, or None when the fused kernel declines the model with BC_ELIMIT and a message."""
    try:
        return fn()
    except L.BayesCardError as e:
        if kernel != L.KERNEL_FUSED or "error -5:" not in str(e) or len(str(e).split("error -5:")[1].strip()) < 5:
            raise
        return None


@pytest.mark.gpu
@pytest.mark.parametrize("name", MODELS)
def test_query_batch_with_multiword_masks(name, cubin_cache):
    """bc_query_batch through K1, SPEC, FUSED and AUTO on BITS, DENSE_F32 and RANGE rows with random mask rows: the fp64
    oracle; a bit on a node without a fan-out vector changes nothing; K2 refuses a mask and serves the NULL mask."""
    m = model(name)
    dm = spec_model(name, cubin_cache)
    b = Batch(m, dm, 2000, seed=11)
    mask = rand_masks(m, b.nq, np.random.default_rng(3))
    fan_only = only_fan_bits(m, mask)
    assert np.array_equal(fan_only, mask) == (name == "one_node")
    served = set()
    for fmt in (L.DESC_BITS, L.DESC_DENSE_F32, L.DESC_RANGE_U16):
        rows = b.rows(fmt)
        ref = O.dense_tree(m, apply_mask(m, b.weights(fmt), mask))
        for kernel in (L.KERNEL_GENERIC, L.KERNEL_SPEC, L.KERNEL_FUSED, L.KERNEL_AUTO):
            got = run_or_refused(lambda: dm.run_host(rows, fmt, mask, kernel), kernel, name)
            if got is None:
                continue
            served.add(kernel)
            assert_close(got, ref, (name, fmt, kernel))
            assert np.array_equal(dm.run_host(rows, fmt, fan_only, kernel), got), (name, fmt, kernel, "bit without a vector")
        assert_close(dm.run_host(rows, fmt, None, L.KERNEL_AUTO), O.dense_tree(m, b.weights(fmt)), (name, fmt, "NULL mask"))
    assert {L.KERNEL_GENERIC, L.KERNEL_SPEC, L.KERNEL_AUTO} <= served
    # K3 serves the small-domain trees; it declines the single node and wide_bits' columns of more than 128 states
    assert (L.KERNEL_FUSED in served) == (name in ("wide70", "chain_fan_root"))
    for kernel in (L.KERNEL_GEMM, L.KERNEL_GEMM_SIMT):
        with pytest.raises(L.BayesCardError, match="error -1:.*fan-out"):
            dm.run_host(b.range16, L.DESC_RANGE_U16, mask, kernel)
        assert_close(dm.run_host(b.range16, L.DESC_RANGE_U16, None, kernel), O.dense_tree(m, b.W), (name, kernel, "K2"))
    dm.close()


@pytest.mark.gpu
def test_fused_dense_rows_ignore_the_next_columns_pad_floats():
    """K3 reads a column's DENSE weights in blocks of 32 floats and issues its last 8-state k-step whole: states K ..
    round_up(K, 8) - 1 hold the column's own pad floats and the NEXT column's weights and pad floats.  With NaN in every pad
    float (the caller's, whatever they hold must not matter) and columns that end in the first half of a k-step followed by
    one-state columns (cards 4 | 1 and 2 | 1), every result must still be the oracle's -- NaN * 0 is NaN, so the whole
    issued tail of the k-step has to be zeroed, not only the column's own pad group."""
    m = make_tree_model(6, [3, 4, 1, 2, 1, 7], seed=12, dtype=np.float32, parent=[-1, 0, 1, 2, 3, 4])
    dm = DeviceModel(m, device=0, specialize=False)
    b = Batch(m, dm, 3000, seed=13)
    assert np.isnan(b.dense).any()
    ref = O.dense_tree(m, b.Wd)
    assert_close(dm.run_host(b.dense, L.DESC_DENSE_F32, None, L.KERNEL_FUSED), ref, "fused, DENSE rows with NaN pads")
    finite = np.nan_to_num(b.dense, nan=0.0)
    assert np.array_equal(dm.run_host(b.dense, L.DESC_DENSE_F32, None, L.KERNEL_FUSED),
                          dm.run_host(finite, L.DESC_DENSE_F32, None, L.KERNEL_FUSED))
    dm.close()


def _rare_equality(m, nq, n_pred, rng):
    """Equality predicates on ``n_pred`` columns, each on a state from the rarer half of its CPT's row mass: joint
    probabilities far below the fp32 range."""
    lo = np.zeros((nq, m.n_nodes), dtype=np.int32)
    hi = np.tile(m.card.astype(np.int32) - 1, (nq, 1))
    rare = []
    for v in range(m.n_nodes):
        t = np.asarray(m.cpts[v], dtype=np.float64)
        mass = t if t.ndim == 1 else t.sum(axis=1)
        live = np.flatnonzero(mass > 0)   # (not the all-zero row: that result is an exact 0)
        rare.append(live[np.argsort(mass[live])][: max(1, len(live) // 2)])
    for q in range(nq):
        for v in rng.choice(m.n_nodes, size=n_pred, replace=False):
            lo[q, v] = hi[q, v] = int(rng.choice(rare[v]))
    return lo, hi


@pytest.mark.gpu
def test_scaled_results_with_multiword_masks(cubin_cache):
    """bc_query_batch_scaled (host and device buffers) through K1, FUSED and AUTO on rare-state equality queries of wide70
    with random mask rows: mantissa * 2^exponent against the fp64 oracle, far below the fp32 range."""
    torch = _torch()
    m = model("wide70")
    dm = DeviceModel(m, device=0, specialize=False)
    rng = np.random.default_rng(8)
    nq = 1500
    lo, hi = _rare_equality(m, nq, 60, rng)
    lo[0], hi[0] = 0, m.card - 1
    mask = rand_masks(m, nq, rng)
    ref = O.dense_tree(m, apply_mask(m, O.range_weights(m, lo, hi), mask))
    assert ((ref > 0) & (ref < 1e-45)).sum() > nq // 2
    bits = PredicateCompiler(m).pack_bits(lo, hi)
    d_bits, d_mask = dev(bits), dev(mask)
    for kernel in (L.KERNEL_GENERIC, L.KERNEL_FUSED, L.KERNEL_AUTO):
        for fmt, rows in ((L.DESC_BITS, bits), (L.DESC_RANGE_U16, pack_ranges_u16(lo, hi))):
            got = dm.run_host_scaled(rows, fmt, mask, kernel)
            err = np.abs(got - ref) / np.maximum(ref, 1e-300)
            err[(ref == 0) & (got == 0)] = 0
            assert err.max() <= RTOL, (kernel, fmt, float(err.max()))
        # device buffers: both output arrays guarded
        om, oe = Guarded(nq), Guarded(nq)
        L.check(L.lib().bc_query_batch_scaled(dm._h, d_bits.data_ptr(), nq, L.DESC_BITS, d_mask.data_ptr(), om.ptr, oe.ptr, kernel,
                                              None))
        torch.cuda.synchronize()
        assert om.intact() and oe.intact(), kernel
        assert np.array_equal(np.ldexp(om.values().astype(np.float64), oe.values(np.int32)),
                              dm.run_host_scaled(bits, L.DESC_BITS, mask, kernel)), kernel
    dm.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", MODELS)
def test_expectation_marginals_with_multiword_masks(name, cubin_cache):
    """bc_expectation_marginal_batch through the spec marginal modules and the expansion via K1 and FUSED, BITS and DENSE
    rows, random mask rows and a NULL mask: the fp64 oracle, and the bins sum to bc_query_batch of the same row and mask."""
    m = model(name)
    targets = MARGINAL_TARGETS[name]
    dm = spec_model(name, cubin_cache, targets)
    b = Batch(m, dm, 400, seed=12)
    mask = rand_masks(m, b.nq, np.random.default_rng(4))
    for fmt in (L.DESC_BITS, L.DESC_DENSE_F32):
        rows = b.rows(fmt)
        for mk in (mask, None):
            W = apply_mask(m, b.weights(fmt), mk)
            total = dm.run_host(rows, fmt, mk, L.KERNEL_GENERIC)
            for t in targets:
                ref = GO.marginal(m, W, t)
                for kernel in (L.KERNEL_SPEC, L.KERNEL_AUTO, L.KERNEL_GENERIC, L.KERNEL_FUSED):
                    got = run_or_refused(lambda: dm.run_marginal_host(rows, fmt, t, kernel, mk), kernel, name)
                    if got is None:
                        continue
                    assert got.shape == ref.shape
                    assert_close(got, ref, (name, fmt, t, kernel, mk is None))
                    if kernel == L.KERNEL_SPEC:
                        assert_close(got.astype(np.float64).sum(axis=1), total, (name, fmt, t, "sum over bins"))
    dm.close()


@pytest.mark.gpu
def test_host_pipelines_offset_mask_rows_per_chunk(cubin_cache):
    """run_host, run_sparse_host, run_packed_host, run_wsparse_host and run_host_scaled on wide70 with mask rows, over
    several chunks each: bit for bit the device-buffer launch on the same rows and masks."""
    torch = _torch()
    m = model("wide70")
    dm = spec_model("wide70", cubin_cache)
    st = torch.cuda.current_stream().cuda_stream

    def on_device(rows, fmt, mask, kernel):
        n = rows.shape[0]
        out = torch.empty(n, dtype=torch.float32, device="cuda:0")
        d_rows, d_mask = dev(rows), dev(mask)
        dm.run_device(d_rows.data_ptr(), n, fmt, out.data_ptr(), d_mask.data_ptr(), kernel, st)
        torch.cuda.synchronize()
        return out.cpu().numpy()

    # DENSE rows: bc_query_batch_host cuts 16 MiB of rows per chunk
    stride = dm.desc_stride(L.DESC_DENSE_F32)
    chunk = max(4096, (16 << 20) // stride)
    b = Batch(m, dm, 2 * chunk + 77, seed=21)
    mask = rand_masks(m, b.nq, np.random.default_rng(5))
    for kernel in (L.KERNEL_GENERIC, L.KERNEL_SPEC):
        assert np.array_equal(dm.run_host(b.dense, L.DESC_DENSE_F32, mask, kernel), on_device(b.dense, L.DESC_DENSE_F32, mask, kernel))
    n = 5000
    sub = slice(0, n)
    pc = PredicateCompiler(m)
    row_off, entries = pc.pack_sparse(b.lo[sub], b.hi[sub])
    klen, blk, payload = dm.pack_sparse(row_off, entries)
    ws_off, ws_words = dense_to_wsparse(m, b.dense[sub])
    env = {k: os.environ.get(k) for k in ("BC_SPARSE_CHUNK", "BC_PACKED_CHUNK", "BC_WSPARSE_CHUNK")}
    os.environ.update(BC_SPARSE_CHUNK="1024", BC_PACKED_CHUNK="1024", BC_WSPARSE_CHUNK="1024")   # five chunks each
    try:
        for kernel in (L.KERNEL_GENERIC, L.KERNEL_SPEC):
            want_bits = on_device(b.bits[sub], L.DESC_BITS, mask[sub], kernel)
            assert np.array_equal(dm.run_sparse_host(row_off, entries, mask[sub], kernel), want_bits), kernel
            assert np.array_equal(dm.run_packed_host(klen, blk, payload, mask[sub], kernel), want_bits), kernel
            want_dense = on_device(b.dense[sub], L.DESC_DENSE_F32, mask[sub], kernel)
            assert np.array_equal(dm.run_wsparse_host(ws_off, ws_words, mask[sub], kernel), want_dense), kernel
    finally:
        for k, v in env.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    # bc_query_batch_scaled_host cuts 64 MiB of rows per chunk (at least 4096)
    ns = 2 * max(4096, (64 << 20) // stride) + 77
    rows = np.tile(b.dense, (-(-ns // b.nq), 1))[:ns]
    mk = rand_masks(m, ns, np.random.default_rng(6))
    om, oe = torch.empty(rows.shape[0], dtype=torch.float32, device="cuda:0"), torch.empty(rows.shape[0], dtype=torch.int32, device="cuda:0")
    d_rows, d_mask = dev(rows), dev(mk)
    L.check(L.lib().bc_query_batch_scaled(dm._h, d_rows.data_ptr(), rows.shape[0], L.DESC_DENSE_F32, d_mask.data_ptr(), om.data_ptr(),
                                          oe.data_ptr(), L.KERNEL_GENERIC, None))
    torch.cuda.synchronize()
    want = np.ldexp(om.cpu().numpy().astype(np.float64), oe.cpu().numpy())
    assert np.array_equal(dm.run_host_scaled(rows, L.DESC_DENSE_F32, mk, L.KERNEL_GENERIC), want)
    dm.close()


def _resident_ctas(cubin, entry, threads):
    """CTAs of ``entry`` one SM holds: the driver's occupancy calculator, which sizes the library's persistent grid."""
    import ctypes as C

    cu = C.CDLL("libcuda.so.1")
    with open(cubin, "rb") as f:
        image = f.read()
    mod, fn, nb = C.c_void_p(), C.c_void_p(), C.c_int()
    assert cu.cuModuleLoadData(C.byref(mod), image) == 0
    try:
        assert cu.cuModuleGetFunction(C.byref(fn), mod, entry.encode()) == 0
        assert cu.cuOccupancyMaxActiveBlocksPerMultiprocessor(C.byref(nb), fn, threads, C.c_size_t(0)) == 0
    finally:
        cu.cuModuleUnload(mod)
    return nb.value


def _batch_sizes(dm, cubin):
    """1, 31, 33, 127, 129, the spec CTA's threads +- 1 and one round of the persistent grid of bc_spec_bits + 1."""
    torch = _torch()
    threads = int(dm.spec_source().split("BC_SPEC_THREADS=")[1].split()[0])
    grid = torch.cuda.get_device_properties(0).multi_processor_count * _resident_ctas(cubin, "bc_spec_bits", threads)
    return sorted({1, 31, 33, 127, 129, threads - 1, threads + 1, grid * threads + 1})


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["wide70", "wide_bits"])
def test_outputs_stay_inside_their_buffers(name, cubin_cache):
    """Every device entry point writes its n results and nothing next to them: K1, SPEC, FUSED and GEMM, the scaled
    mantissa and exponent arrays, the spec marginal module and the expansion -- at batch sizes around the warp, the K3
    tile, the spec CTA and one round of the persistent grid."""
    torch = _torch()
    m = model(name)
    t = MARGINAL_TARGETS[name][-1]
    dm = spec_model(name, cubin_cache, [t])
    sizes = _batch_sizes(dm, cubin_cache.spec[name])
    small = 4096   # DENSE rows, scaled results and marginals up to this size; BITS, RANGE and K2 at every size
    big = Batch(m, dm, sizes[-1], seed=31, n_dense=small)
    mask = rand_masks(m, big.nq, np.random.default_rng(7))
    d_bits, d_dense, d_r16, d_mask = dev(big.bits), dev(big.dense), dev(big.range16), dev(mask)
    # the oracle on the first `small` queries, the last 8192 (the last rounds) and a seeded sample of the rest (NaN elsewhere)
    idx = np.unique(np.concatenate([np.arange(small), np.arange(max(0, big.nq - 8192), big.nq),
                                    np.random.default_rng(8).choice(big.nq, min(big.nq, 8192), replace=False)]))
    ref_b, ref_r = np.full(big.nq, np.nan), np.full(big.nq, np.nan)
    ref_b[idx] = oracle(m, big.lo[idx], big.hi[idx], mask[idx])
    ref_r[idx] = oracle(m, big.lo[idx], big.hi[idx], None)
    ref_d = O.dense_tree(m, apply_mask(m, big.Wd, mask[:small]))
    card = int(m.card[t])
    ref_marg = GO.marginal(m, apply_mask(m, big.W, mask[:small]), t)
    st = torch.cuda.current_stream().cuda_stream

    def check(got, ref, what):
        assert np.isfinite(got).all(), what
        known = ~np.isnan(ref)
        assert_close(got[known], ref[known], what)

    for n in sizes:
        for fmt, d_rows, ref in ((L.DESC_BITS, d_bits, ref_b), (L.DESC_DENSE_F32, d_dense, ref_d)):
            if n > ref.shape[0]:
                continue
            for kernel in (L.KERNEL_GENERIC, L.KERNEL_SPEC, L.KERNEL_FUSED):
                out = Guarded(n)
                try:
                    dm.run_device(d_rows.data_ptr(), n, fmt, out.ptr, d_mask.data_ptr(), kernel, st)
                except L.BayesCardError as e:
                    assert kernel == L.KERNEL_FUSED and "error -5:" in str(e), (n, fmt, kernel, str(e))
                    continue
                torch.cuda.synchronize()
                assert out.intact(), (name, n, fmt, kernel)
                check(out.values(), ref[:n], (name, n, fmt, kernel))
        out = Guarded(n)
        dm.run_device(d_r16.data_ptr(), n, L.DESC_RANGE_U16, out.ptr, 0, L.KERNEL_GEMM, st)
        torch.cuda.synchronize()
        assert out.intact(), (name, n, "GEMM")
        check(out.values(), ref_r[:n], (name, n, "GEMM"))
        if n > small:
            continue
        for kernel in (L.KERNEL_GENERIC, L.KERNEL_FUSED):
            om, oe = Guarded(n), Guarded(n)
            rc = L.lib().bc_query_batch_scaled(dm._h, d_bits.data_ptr(), n, L.DESC_BITS, d_mask.data_ptr(), om.ptr, oe.ptr, kernel, st)
            if rc == -5 and kernel == L.KERNEL_FUSED:
                continue
            L.check(rc)
            torch.cuda.synchronize()
            assert om.intact() and oe.intact(), (name, n, "scaled", kernel)
            assert_close(np.ldexp(om.values().astype(np.float64), oe.values(np.int32)), ref_b[:n], (name, n, "scaled", kernel))
        for kernel in (L.KERNEL_SPEC, L.KERNEL_GENERIC):
            out = Guarded(n * card)
            dm.run_marginal_device(d_bits.data_ptr(), n, L.DESC_BITS, t, out.ptr, kernel, st, d_mask.data_ptr())
            torch.cuda.synchronize()
            assert out.intact(), (name, n, "marginal", kernel)
            assert_close(out.values().reshape(n, card), ref_marg[:n], (name, n, "marginal", kernel))
    dm.close()


@pytest.mark.gpu
def test_spec_work_counter_ring_across_launches_and_streams(cubin_cache):
    """300 consecutive spec launches of varying sizes on one stream (more than the 256 work-counter slots, so every slot is
    reused by a launch of another grid size), then launches alternating between two streams, marginal launches among them
    (they draw from the same ring): each against the fp64 oracle on its own rows."""
    torch = _torch()
    m = model("wide70")
    t = 33
    dm = spec_model("wide70", cubin_cache, [t])
    b = Batch(m, dm, 6000, seed=41)
    mask = rand_masks(m, b.nq, np.random.default_rng(9))
    ref = O.dense_tree(m, apply_mask(m, b.W, mask))
    ref_marg = GO.marginal(m, apply_mask(m, [w[:600] for w in b.W], mask[:600]), t)
    d_bits, d_mask = dev(b.bits), dev(mask)
    stride, mstride = dm.desc_stride(L.DESC_BITS), 4 * dm.mask_words
    rng = np.random.default_rng(10)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    launches = []

    def launch(stream, marginal=False):
        n = int(rng.integers(1, 600 if marginal else 5000))
        a = int(rng.integers(0, (600 if marginal else b.nq) - n + 1))
        out = torch.empty(n * (int(m.card[t]) if marginal else 1), dtype=torch.float32, device="cuda:0")
        args = (d_bits.data_ptr() + a * stride, n, L.DESC_BITS)
        if marginal:
            dm.run_marginal_device(*args, t, out.data_ptr(), L.KERNEL_SPEC, stream.cuda_stream, d_mask.data_ptr() + a * mstride)
        else:
            dm.run_device(*args, out.data_ptr(), d_mask.data_ptr() + a * mstride, L.KERNEL_SPEC, stream.cuda_stream)
        launches.append((a, n, marginal, out))

    for _ in range(300):
        launch(s1)
    for i in range(240):
        launch(s1 if i % 2 == 0 else s2, marginal=i % 5 == 0)
    torch.cuda.synchronize()
    for a, n, marginal, out in launches:
        if marginal:
            assert_close(out.cpu().numpy().reshape(n, -1), ref_marg[a:a + n], ("marginal", a, n))
        else:
            assert_close(out.cpu().numpy(), ref[a:a + n], ("spec", a, n))
    dm.close()
