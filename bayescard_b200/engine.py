"""Device-side model handle: a :class:`~bayescard_b200.loader.TreeModel` uploaded through the C ABI.

``DeviceModel`` owns one ``bc_model*`` (one GPU).  ``ShardedModel`` replicates the CPT arena on several
GPUs and splits a query batch into contiguous ranges, one host thread + stream set per device, no
collective on the data path (SURVEY.md section 8e).  PyTorch is not needed here; callers that hold
torch tensors pass ``tensor.data_ptr()`` and ``torch.cuda.current_stream().cuda_stream``.
"""
from __future__ import annotations

import ctypes as C
import os
import threading
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

from . import _lib as L
from .loader import TreeModel


class DeviceModel:
    def __init__(self, tm: TreeModel, device: int = 0, specialize: bool = True, cache_dir: Optional[str] = None,
                 flat_file: Optional[str] = None):
        self.tm = tm
        self.device = device
        lib = L.lib()
        h = C.c_void_p()
        card = np.ascontiguousarray(tm.card, dtype=np.int32)
        if flat_file is not None:
            # the library maps the file itself: no array of this model crosses the boundary from Python
            L.check(lib.bc_model_create_from_file(device, os.fsencode(flat_file), C.byref(h)))
        else:
            arena, off, stride = tm.pack_arena()
            fan, foff = tm.pack_fanouts()
            parent = np.ascontiguousarray(tm.parent, dtype=np.int32)
            L.check(lib.bc_model_create(device, tm.n_nodes, parent.ctypes.data, card.ctypes.data, off.ctypes.data,
                                        stride.ctypes.data, arena.ctypes.data, arena.size, foff.ctypes.data,
                                        fan.ctypes.data, fan.size, C.byref(h)))
        self._h = h
        self.n_nodes = tm.n_nodes
        self.mask_words = (tm.n_nodes + 31) // 32
        self.dense_width = int(lib.bc_model_dense_width(h))
        self.dense_offset = np.array([lib.bc_model_dense_offset(h, v) for v in range(tm.n_nodes)], dtype=np.int64)
        self.bits_offset = np.array([lib.bc_model_bits_offset(h, v) for v in range(tm.n_nodes)], dtype=np.int64)
        self.flops_dense = int(lib.bc_model_flops_dense(h))
        self.max_card = int(card.max())
        self.spec_error: Optional[str] = None
        self.marginal_error: Dict[int, str] = {}   # target node -> why its specialised marginal kernel is missing
        self._marginal_built: Dict[int, bool] = {}
        self.joint_error: Dict[Tuple[int, int], str] = {}   # ordered pair -> why its joint module is missing
        self._joint_built: Dict[Tuple[int, int], bool] = {}
        self._specialize = specialize and device >= 0   # update() re-specialises under the same policy
        self._cache_dir = cache_dir
        if specialize and device >= 0:
            try:
                self.specialize(cache_dir)
            except L.BayesCardError as e:  # generic CUDA kernel keeps serving; remembered for diagnostics
                self.spec_error = str(e)

    @classmethod
    def from_flat_file(cls, path: str, device: int = 0, specialize: bool = True) -> "DeviceModel":
        """Serve from a flat model file (``TreeModel.save_flat``): decode tables through ``mmap``, CPTs through
        ``bc_model_create_from_file`` -- nothing is unpickled."""
        return cls(TreeModel.load_flat(path), device=device, specialize=specialize, flat_file=path)

    # ------------------------------------------------------------------ lifecycle
    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            L.lib().bc_model_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ specialised kernel
    def specialize(self, cache_dir: Optional[str] = None) -> None:
        cache_dir = L.SPEC_CACHE_DIR if cache_dir is None else cache_dir
        if cache_dir:
            os.makedirs(cache_dir, exist_ok=True)
        L.check(L.lib().bc_model_specialize(self._h, cache_dir.encode() if cache_dir else None))

    @property
    def has_spec(self) -> bool:
        return bool(L.lib().bc_model_has_spec(self._h))

    def spec_source(self) -> str:
        lib = L.lib()
        n = lib.bc_model_spec_source(self._h, None, 0)
        if n < 0:
            L.check(int(n))
        buf = C.create_string_buffer(int(n))
        lib.bc_model_spec_source(self._h, buf, int(n))
        return buf.value.decode()

    def spec_hash(self) -> int:
        return int(L.lib().bc_model_spec_hash(self._h))

    def spec_ffma(self) -> int:
        """FFMA instructions the generated kernel executes per query (exact zeros are skipped)."""
        for line in self.spec_source().splitlines()[:4]:
            if "BC_SPEC_FFMA=" in line:
                return int(line.split("BC_SPEC_FFMA=")[1].split()[0])
        raise L.BayesCardError("generated source has no BC_SPEC_FFMA header")

    def load_image(self, image: bytes) -> None:
        """Attach a compiled specialised image (cubin, or PTX text for the driver JIT)."""
        if not image.endswith(b"\0") and image[:4] != b"\x7fELF":
            image = image + b"\0"  # PTX must be NUL terminated
        buf = C.create_string_buffer(image, len(image))
        L.check(L.lib().bc_model_load_cubin(self._h, buf, len(image)))

    # ------------------------------------------------------------------ GROUP BY one column (per-state marginals)
    def _check_node(self, node: int) -> int:
        node = int(node)
        if not 0 <= node < self.n_nodes:
            raise ValueError(f"node {node} outside the model's {self.n_nodes} nodes")
        return node

    def specialize_marginal(self, node: int, cache_dir: Optional[str] = None) -> bool:
        """Attach the specialised marginal kernel of ``node`` (built on the first call, then kept).  A failure is
        recorded in ``marginal_error[node]`` and not retried; ``marginal_batch`` then serves the node by expansion."""
        node = self._check_node(node)
        if node not in self._marginal_built:
            cache_dir = L.SPEC_CACHE_DIR if cache_dir is None else cache_dir
            try:
                L.check(L.lib().bc_model_specialize_marginal(self._h, node, cache_dir.encode() if cache_dir else None))
                self._marginal_built[node] = True
            except L.BayesCardError as e:
                self.marginal_error[node] = str(e)
                self._marginal_built[node] = False
        return self._marginal_built[node]

    def marginal_source(self, node: int) -> str:
        lib = L.lib()
        node = self._check_node(node)
        n = lib.bc_model_marginal_source(self._h, node, None, 0)
        if n < 0:
            L.check(int(n))
        buf = C.create_string_buffer(int(n))
        lib.bc_model_marginal_source(self._h, node, buf, int(n))
        return buf.value.decode()

    def marginal_hash(self, node: int) -> int:
        return int(L.lib().bc_model_marginal_hash(self._h, self._check_node(node)))

    def run_marginal_device(self, desc_ptr: int, n: int, fmt: int, node: int, out_ptr: int, kernel: int = L.KERNEL_AUTO,
                            stream: int = 0, mask_ptr: int = 0) -> None:
        """``bc_expectation_marginal_batch`` on DEVICE buffers: ``out`` receives ``[n][card(node)]`` fp32; ``mask_ptr``: 0 or
        ``n * mask_words`` uint32 fan-out mask rows (0 is ``bc_marginal_batch``)."""
        L.check(L.lib().bc_expectation_marginal_batch(self._h, desc_ptr or None, n, fmt, mask_ptr or None, int(node), out_ptr or None,
                                                      kernel, stream or None))

    def run_marginal_host(self, desc: np.ndarray, fmt: int, node: int, kernel: int = L.KERNEL_AUTO,
                          mask: Optional[np.ndarray] = None) -> np.ndarray:
        """BITS / DENSE_F32 rows from the host -> ``ndarray [n, card(node)]`` fp32: the per-state mass of ``node`` under
        each row, with the fan-out columns of ``mask`` (``[n, mask_words]`` uint32, or ``None``) multiplied in.  torch moves
        the buffers; the work is ``bc_expectation_marginal_batch``."""
        node = self._check_node(node)
        stride = self.desc_stride(fmt)
        desc = np.ascontiguousarray(desc)
        n = desc.nbytes // stride
        if desc.nbytes != n * stride:
            raise ValueError(f"descriptor buffer of {desc.nbytes} B is not a multiple of the row stride {stride}")
        if mask is not None:
            mask = np.ascontiguousarray(mask, dtype=np.uint32)
            if mask.size != n * self.mask_words:
                raise ValueError("fan-out mask has the wrong size")
        card = int(self.tm.card[node])
        if n == 0 or self.device < 0:   # (the library still validates the arguments)
            L.check(L.lib().bc_expectation_marginal_batch(self._h, None, n, fmt, None, node, None, kernel, None))
            return np.zeros((n, card), dtype=np.float32)
        import torch

        dev = torch.device("cuda", self.device)
        with torch.cuda.device(dev):
            d_desc = torch.from_numpy(desc.reshape(-1).view(np.uint8)).to(dev)
            d_mask = torch.from_numpy(mask.reshape(-1)).to(dev) if mask is not None else None
            d_out = torch.empty(n * card, dtype=torch.float32, device=dev)
            self.run_marginal_device(d_desc.data_ptr(), n, fmt, node, d_out.data_ptr(), kernel,
                                     torch.cuda.current_stream().cuda_stream, d_mask.data_ptr() if d_mask is not None else 0)
            return d_out.cpu().numpy().reshape(n, card)

    # ------------------------------------------------------------------ GROUP BY two columns (joint marginals)
    def _check_pair(self, a: int, b: int):
        a, b = self._check_node(a), self._check_node(b)
        if a == b:
            raise ValueError(f"a joint marginal needs two distinct nodes, got {a} twice")
        return a, b

    def specialize_joint(self, a: int, b: int, cache_dir: Optional[str] = None) -> bool:
        """Attach the joint module of the ordered pair ``(a, b)`` (built on the first call, then kept).  A failure -- such
        as a pair above the generator's size cap -- is recorded in ``joint_error[(a, b)]`` and not retried;
        ``run_joint_*`` then serve the pair by expansion."""
        a, b = self._check_pair(a, b)
        if (a, b) not in self._joint_built:
            cache_dir = L.SPEC_CACHE_DIR if cache_dir is None else cache_dir
            try:
                L.check(L.lib().bc_model_specialize_joint(self._h, a, b, cache_dir.encode() if cache_dir else None))
                self._joint_built[(a, b)] = True
            except L.BayesCardError as e:
                self.joint_error[(a, b)] = str(e)
                self._joint_built[(a, b)] = False
        return self._joint_built[(a, b)]

    def joint_source(self, a: int, b: int) -> str:
        lib = L.lib()
        a, b = self._check_pair(a, b)
        n = lib.bc_model_joint_source(self._h, a, b, None, 0)
        if n < 0:
            L.check(int(n))
        buf = C.create_string_buffer(int(n))
        lib.bc_model_joint_source(self._h, a, b, buf, int(n))
        return buf.value.decode()

    def joint_hash(self, a: int, b: int) -> int:
        a, b = self._check_pair(a, b)
        return int(L.lib().bc_model_joint_hash(self._h, a, b))

    def run_joint_device(self, desc_ptr: int, n: int, fmt: int, a: int, b: int, out_ptr: int, kernel: int = L.KERNEL_AUTO,
                         stream: int = 0, mask_ptr: int = 0) -> None:
        """``bc_joint_marginal_batch`` on DEVICE buffers: ``out`` receives ``[n][card(a)][card(b)]`` fp32; ``mask_ptr``: 0 or
        ``n * mask_words`` uint32 fan-out mask rows."""
        L.check(L.lib().bc_joint_marginal_batch(self._h, desc_ptr or None, n, fmt, mask_ptr or None, int(a), int(b), out_ptr or None,
                                                kernel, stream or None))

    # one call's device output stays below this many bytes (run_joint_host chunks the rows)
    JOINT_OUT_BYTES = 256 << 20

    def run_joint_host(self, desc: np.ndarray, fmt: int, a: int, b: int, kernel: int = L.KERNEL_AUTO,
                       mask: Optional[np.ndarray] = None) -> np.ndarray:
        """BITS / DENSE_F32 rows from the host -> ``ndarray [n, card(a), card(b)]`` fp32: the mass of every pair of states of
        ``a`` and ``b`` under each row, with the fan-out columns of ``mask`` (``[n, mask_words]`` uint32, or ``None``)
        multiplied in.  The rows go in chunks whose output is at most ``JOINT_OUT_BYTES`` on the device."""
        a, b = self._check_pair(a, b)
        stride = self.desc_stride(fmt)
        desc = np.ascontiguousarray(desc)
        n = desc.nbytes // stride
        if desc.nbytes != n * stride:
            raise ValueError(f"descriptor buffer of {desc.nbytes} B is not a multiple of the row stride {stride}")
        if mask is not None:
            mask = np.ascontiguousarray(mask, dtype=np.uint32).reshape(-1)
            if mask.size != n * self.mask_words:
                raise ValueError("fan-out mask has the wrong size")
        ca, cb = int(self.tm.card[a]), int(self.tm.card[b])
        out = np.zeros((n, ca, cb), dtype=np.float32)
        if n == 0 or self.device < 0:   # (the library still validates the arguments)
            L.check(L.lib().bc_joint_marginal_batch(self._h, None, n, fmt, None, a, b, None, kernel, None))
            return out
        import torch

        rows = desc.reshape(-1).view(np.uint8).reshape(n, stride)
        chunk = max(1, self.JOINT_OUT_BYTES // (4 * ca * cb))
        dev = torch.device("cuda", self.device)
        with torch.cuda.device(dev):
            for q0 in range(0, n, chunk):
                q1 = min(n, q0 + chunk)
                d_desc = torch.from_numpy(rows[q0:q1].reshape(-1)).to(dev)
                d_mask = None if mask is None else torch.from_numpy(mask[q0 * self.mask_words:q1 * self.mask_words]).to(dev)
                d_out = torch.empty((q1 - q0) * ca * cb, dtype=torch.float32, device=dev)
                self.run_joint_device(d_desc.data_ptr(), q1 - q0, fmt, a, b, d_out.data_ptr(), kernel,
                                      torch.cuda.current_stream().cuda_stream, d_mask.data_ptr() if d_mask is not None else 0)
                out[q0:q1] = d_out.cpu().numpy().reshape(q1 - q0, ca, cb)
        return out

    # ------------------------------------------------------------------ incremental update (DESIGN.md section 9e)
    def attach_counts(self, counts: np.ndarray) -> None:
        """Keep ``counts`` (uint64, ``fit.count_layout`` order) on the device as the counts behind the CPTs
        (``bc_model_set_counts``).  They must be the counts the CPTs were normalised from (``fit.counts_from_cpts``)."""
        counts = np.ascontiguousarray(counts, dtype=np.uint64)
        L.check(L.lib().bc_model_set_counts(self._h, counts.ctypes.data, counts.size))
        self._marginal_built.clear()
        self.marginal_error.clear()
        self._joint_built.clear()
        self.joint_error.clear()

    def get_counts(self, node_first: int = 0, node_count: Optional[int] = None) -> np.ndarray:
        """The attached counters of nodes ``[node_first, node_first + node_count)`` (default: to the last node)."""
        from .fit import count_layout

        node_count = self.n_nodes - node_first if node_count is None else node_count
        off, total = count_layout(self.tm.parent, self.tm.card)
        off = np.append(off, total)
        if not (0 <= node_first and 0 <= node_count and node_first + node_count <= self.n_nodes):
            raise ValueError(f"nodes [{node_first}, {node_first + node_count}) outside the model's {self.n_nodes} nodes")
        out = np.zeros(int(off[node_first + node_count] - off[node_first]), dtype=np.uint64)
        L.check(L.lib().bc_model_get_counts(self._h, node_first, node_count, out.ctypes.data if out.size else None))
        return out

    def arena(self, from_device: bool = True) -> np.ndarray:
        """The fp32 CPT arena the kernels read (``from_device``) or the library's host copy of it, zero-padded: its first
        ``tm.pack_arena()[0].size`` floats are ``pack_arena()``'s."""
        lib = L.lib()
        n = int(lib.bc_model_arena(self._h, int(from_device), None, 0))
        if n < 0:
            L.check(n)
        out = np.zeros(n, dtype=np.float32)
        rc = int(lib.bc_model_arena(self._h, int(from_device), out.ctypes.data, n))
        if rc < 0:
            L.check(rc)
        return out

    def update(self, inserted=None, deleted=None, n_inserted: int = 0, n_deleted: int = 0, elem_bytes: int = 1,
               row_stride: Optional[int] = None, stream: int = 0) -> np.ndarray:
        """Insert and delete rows of the table the attached counts came from (``bc_model_update``) and return the
        topological indices of the nodes whose counts changed.

        Rows are bin ids with columns in topological order.  Either host arrays (``[n, n_nodes]`` or wider, uint8 /
        uint16; the two tables are given the same width and dtype) or DEVICE addresses with ``n_inserted`` /
        ``n_deleted`` rows, ``elem_bytes`` and ``row_stride`` (elements, default ``n_nodes``) on ``stream``.  Only the CPTs
        move: the tree, the decode metadata and the fan-out vectors stay.  A rejected batch (a bin id outside its domain, a
        delete below zero) raises and leaves the model as it was.  When a count changed, the marginal kernels are
        forgotten and, for a model built with ``specialize=True``, the specialised kernel is built again for the new
        CPTs."""
        host = not (isinstance(inserted, int) or isinstance(deleted, int))
        touched = np.zeros(self.n_nodes, dtype=np.uint8)
        bad = C.c_uint32(0)
        if host:
            tabs = [None if t is None else np.asarray(t) for t in (inserted, deleted)]
            present = [t for t in tabs if t is not None]
            for t in present:
                if t.ndim != 2 or t.shape[1] < self.n_nodes or t.dtype not in (np.uint8, np.uint16):
                    raise ValueError("rows must be [n, >= n_nodes] uint8 or uint16 bin ids")
            dt = np.uint16 if any(t.dtype == np.uint16 for t in present) else np.uint8
            width = max([t.shape[1] for t in present], default=self.n_nodes)
            tabs = [None if t is None else
                    np.ascontiguousarray((t if t.shape[1] == width else np.pad(t, ((0, 0), (0, width - t.shape[1])))).astype(dt, copy=False))
                    for t in tabs]
            n_ins, n_del = [0 if t is None else t.shape[0] for t in tabs]
            if n_ins + n_del and self.device >= 0:
                import torch

                dev = torch.device("cuda", self.device)
                with torch.cuda.device(dev):
                    d = [None if not (t is not None and t.shape[0]) else torch.from_numpy(t.reshape(-1).view(np.uint8)).to(dev)
                         for t in tabs]
                    L.check(L.lib().bc_model_update(self._h, d[0].data_ptr() if d[0] is not None else None, n_ins,
                                                    d[1].data_ptr() if d[1] is not None else None, n_del, np.dtype(dt).itemsize,
                                                    width, touched.ctypes.data, C.byref(bad), torch.cuda.current_stream().cuda_stream or None))
            else:   # (no rows, or a host-only model: the library still validates the arguments)
                L.check(L.lib().bc_model_update(self._h, None, 0, None, 0, np.dtype(dt).itemsize, width, touched.ctypes.data,
                                                C.byref(bad), None))
        else:
            L.check(L.lib().bc_model_update(self._h, inserted or None, n_inserted, deleted or None, n_deleted, elem_bytes,
                                            self.n_nodes if row_stride is None else row_stride, touched.ctypes.data, C.byref(bad),
                                            stream or None))
        nodes = np.flatnonzero(touched)
        if nodes.size:
            self._marginal_built.clear()
            self.marginal_error.clear()
            self._joint_built.clear()
            self.joint_error.clear()
            if self._specialize:
                try:
                    self.specialize(self._cache_dir)
                    self.spec_error = None
                except L.BayesCardError as e:
                    self.spec_error = str(e)
        return nodes

    # ------------------------------------------------------------------ geometry
    def desc_stride(self, fmt: int) -> int:
        s = int(L.lib().bc_model_desc_stride(self._h, fmt))
        if s <= 0:
            raise L.BayesCardError(f"unknown descriptor format {fmt}")
        return s

    # ------------------------------------------------------------------ launches
    def run_device(self, desc_ptr: int, n: int, fmt: int, out_ptr: int, mask_ptr: int = 0,
                   kernel: int = L.KERNEL_AUTO, stream: int = 0) -> None:
        """One stream-ordered launch on DEVICE buffers (raw addresses)."""
        L.check(L.lib().bc_query_batch(self._h, desc_ptr, n, fmt, mask_ptr or None, out_ptr, kernel, stream or None))

    def run_host(self, desc: np.ndarray, fmt: int, mask: Optional[np.ndarray] = None,
                 kernel: int = L.KERNEL_AUTO, out: Optional[np.ndarray] = None) -> np.ndarray:
        """Host buffers in, host fp32 probabilities out (H2D / kernel / D2H pipelined in the library)."""
        stride = self.desc_stride(fmt)
        desc = np.ascontiguousarray(desc)
        n = desc.nbytes // stride
        if desc.nbytes != n * stride:
            raise ValueError(f"descriptor buffer of {desc.nbytes} B is not a multiple of the row stride {stride}")
        if mask is not None:
            mask = np.ascontiguousarray(mask, dtype=np.uint32)
            if mask.size != n * self.mask_words:
                raise ValueError("fan-out mask has the wrong size")
        if out is None:
            out = np.empty(n, dtype=np.float32)
        L.check(L.lib().bc_query_batch_host(self._h, desc.ctypes.data, n, fmt,
                                            mask.ctypes.data if mask is not None else None, out.ctypes.data, kernel))
        return out

    def run_host_scaled(self, desc: np.ndarray, fmt: int, mask: Optional[np.ndarray] = None,
                        kernel: int = L.KERNEL_AUTO) -> np.ndarray:
        """Host buffers in, **fp64** probabilities out, for results beyond the fp32 range (below ~1e-38): the kernels carry
        one power-of-two exponent per query (``bc_query_batch_scaled_host``); the reference computes in fp64
        (``Pgmpy/inference/ExactInference.py:157-177``)."""
        stride = self.desc_stride(fmt)
        desc = np.ascontiguousarray(desc)
        n = desc.nbytes // stride
        if desc.nbytes != n * stride:
            raise ValueError(f"descriptor buffer of {desc.nbytes} B is not a multiple of the row stride {stride}")
        if mask is not None:
            mask = np.ascontiguousarray(mask, dtype=np.uint32)
            if mask.size != n * self.mask_words:
                raise ValueError("fan-out mask has the wrong size")
        out = np.empty(n, dtype=np.float64)
        L.check(L.lib().bc_query_batch_scaled_host(self._h, desc.ctypes.data, n, fmt,
                                                   mask.ctypes.data if mask is not None else None, out.ctypes.data, kernel))
        return out

    def bits_default(self) -> np.ndarray:
        row = np.zeros(self.desc_stride(L.DESC_BITS) // 4, dtype=np.uint32)
        L.check(L.lib().bc_model_bits_default(self._h, row.ctypes.data, row.nbytes))
        return row

    def convert_device(self, src_ptr: int, src_fmt: int, dst_ptr: int, dst_fmt: int, n: int, stream: int = 0) -> None:
        """Stream-ordered descriptor conversion on DEVICE buffers (RANGE_U8 / RANGE_U16 -> BITS)."""
        L.check(L.lib().bc_convert_desc(self._h, src_ptr, src_fmt, dst_ptr, dst_fmt, n, stream or None))

    def expand_sparse_device(self, row_off_ptr: int, entries_ptr: int, n: int, dst_ptr: int, stream: int = 0) -> None:
        L.check(L.lib().bc_expand_sparse(self._h, row_off_ptr, entries_ptr, n, dst_ptr, stream or None))

    def run_wsparse_host(self, row_off: np.ndarray, words: np.ndarray, mask: Optional[np.ndarray] = None,
                         kernel: int = L.KERNEL_AUTO, out: Optional[np.ndarray] = None) -> np.ndarray:
        """WSPARSE rows (weighted runs, ``decode.dense_to_wsparse`` / ``PredicateCompiler.pack_wsparse``) from host
        buffers: H2D, expand to DENSE_F32 on the device, infer, D2H -- pipelined in the library."""
        row_off = np.ascontiguousarray(row_off, dtype=np.uint32)
        words = np.ascontiguousarray(words, dtype=np.uint32)
        n = row_off.size - 1
        if n < 0 or (n > 0 and int(row_off[-1]) > words.size):
            raise ValueError("row_off does not match the words array")
        if mask is not None:
            mask = np.ascontiguousarray(mask, dtype=np.uint32)
            if mask.size != n * self.mask_words:
                raise ValueError("fan-out mask has the wrong size")
        if out is None:
            out = np.empty(n, dtype=np.float32)
        L.check(L.lib().bc_query_batch_wsparse_host(self._h, row_off.ctypes.data, words.ctypes.data if words.size else None, n,
                                                    mask.ctypes.data if mask is not None else None, out.ctypes.data, kernel))
        return out

    def run_sparse_host(self, row_off: np.ndarray, entries: np.ndarray, mask: Optional[np.ndarray] = None,
                        kernel: int = L.KERNEL_AUTO, out: Optional[np.ndarray] = None) -> np.ndarray:
        """SPARSE (CSR) queries from host buffers: H2D, expand to BITS, infer, D2H -- pipelined in the library."""
        row_off = np.ascontiguousarray(row_off, dtype=np.uint32)
        entries = np.ascontiguousarray(entries, dtype=np.uint32)
        n = row_off.size - 1
        if n < 0 or (n > 0 and int(row_off[-1]) > entries.size):
            raise ValueError("row_off does not match the entries array")
        if mask is not None:
            mask = np.ascontiguousarray(mask, dtype=np.uint32)
            if mask.size != n * self.mask_words:
                raise ValueError("fan-out mask has the wrong size")
        if out is None:
            out = np.empty(n, dtype=np.float32)
        L.check(L.lib().bc_query_batch_sparse_host(self._h, row_off.ctypes.data, entries.ctypes.data if entries.size else None,
                                                   n, mask.ctypes.data if mask is not None else None, out.ctypes.data,
                                                   kernel))
        return out

    # ------------------------------------------------------------------ PACKED wire format (17 B per Census query over PCIe)
    def packed_geometry(self):
        """``(entry_bits, col_bits, state_bits)`` of the PACKED wire format for this model."""
        w, cb, sb = C.c_int(), C.c_int(), C.c_int()
        L.check(L.lib().bc_model_packed_geometry(self._h, C.byref(w), C.byref(cb), C.byref(sb)))
        return w.value, cb.value, sb.value

    def pack_sparse(self, row_off: np.ndarray, entries: np.ndarray):
        """SPARSE (CSR) -> PACKED on the host: ``(klen uint8[n], blk_off uint32[ceil(n/128)+1], payload uint8[...])``."""
        row_off = np.ascontiguousarray(row_off, dtype=np.uint32)
        entries = np.ascontiguousarray(entries, dtype=np.uint32)
        n = row_off.size - 1
        klen = np.zeros(max(n, 1), dtype=np.uint8)[:n]
        blk = np.zeros((n + 127) // 128 + 1, dtype=np.uint32)
        w, _, _ = self.packed_geometry()
        ne = int(row_off[-1]) - int(row_off[0]) if n else 0
        payload = np.zeros(((ne * w + 31) // 32 + 2) * 4, dtype=np.uint8)
        used = C.c_size_t()
        L.check(L.lib().bc_pack_sparse(self._h, row_off.ctypes.data, entries.ctypes.data if entries.size else None, n,
                                       klen.ctypes.data if n else None, blk.ctypes.data, payload.ctypes.data, payload.nbytes, C.byref(used)))
        return klen, blk, payload[: used.value]

    def run_packed_host(self, klen: np.ndarray, blk_off: np.ndarray, payload: np.ndarray, mask: Optional[np.ndarray] = None,
                        kernel: int = L.KERNEL_AUTO, out: Optional[np.ndarray] = None) -> np.ndarray:
        """PACKED queries from host buffers: H2D, expand to BITS, infer, D2H -- sub-chunked and pipelined in the library."""
        klen = np.ascontiguousarray(klen, dtype=np.uint8)
        blk_off = np.ascontiguousarray(blk_off, dtype=np.uint32)
        payload = np.ascontiguousarray(payload, dtype=np.uint8)
        n = klen.size
        if blk_off.size != (n + 127) // 128 + 1:
            raise ValueError("blk_off does not match klen")
        if mask is not None:
            mask = np.ascontiguousarray(mask, dtype=np.uint32)
            if mask.size != n * self.mask_words:
                raise ValueError("fan-out mask has the wrong size")
        if out is None:
            out = np.empty(n, dtype=np.float32)
        L.check(L.lib().bc_query_batch_packed_host(self._h, klen.ctypes.data if n else None, blk_off.ctypes.data, payload.ctypes.data,
                                                   payload.nbytes, n, mask.ctypes.data if mask is not None else None, out.ctypes.data, kernel))
        return out

    def submit_packed_host(self, klen: np.ndarray, blk_off: np.ndarray, payload: np.ndarray, out: np.ndarray,
                           mask: Optional[np.ndarray] = None, kernel: int = L.KERNEL_AUTO) -> int:
        """Asynchronous ``run_packed_host``: returns a ticket as soon as the batch is enqueued; ``out`` (pinned, float32[n]) is
        complete after ``wait(ticket)``.  The arrays must be the caller's own contiguous buffers (nothing is copied) and stay
        untouched until then.  Consecutive submissions overlap -- batch i + 1 is copied in while batch i is computed and read
        back -- so a serving loop keeps two batches in flight::

            t_prev = None
            for bufs in batches:                      # double-buffered host memory
                t = dm.submit_packed_host(*bufs.inputs, out=bufs.out)
                if t_prev is not None: dm.wait(t_prev); consume(prev.out)
                t_prev, prev = t, bufs
        """
        n = klen.size
        for a, dt in ((klen, np.uint8), (blk_off, np.uint32), (payload, np.uint8), (out, np.float32)):
            if a.dtype != dt or not a.flags["C_CONTIGUOUS"]:
                raise ValueError("submit_packed_host takes contiguous arrays of the wire dtypes (no copies are made)")
        if blk_off.size != (n + 127) // 128 + 1 or out.size != n:
            raise ValueError("blk_off / out do not match klen")
        if mask is not None and (mask.dtype != np.uint32 or not mask.flags["C_CONTIGUOUS"] or mask.size != n * self.mask_words):
            raise ValueError("fan-out mask has the wrong dtype or size")
        ticket = C.c_uint64()
        L.check(L.lib().bc_query_batch_packed_host_submit(self._h, klen.ctypes.data if n else None, blk_off.ctypes.data, payload.ctypes.data,
                                                          payload.nbytes, n, mask.ctypes.data if mask is not None else None, out.ctypes.data,
                                                          kernel, C.byref(ticket)))
        return int(ticket.value)

    def wait(self, ticket: int) -> None:
        """Blocks until the submission ``ticket`` (and every earlier one) has written its results."""
        L.check(L.lib().bc_pipe_wait(self._h, int(ticket)))

    def gen_sparse_queries_host(self, seed: int, first: int, n: int, kmin: int, kmax: int):
        card = np.ascontiguousarray(self.tm.card, dtype=np.int32)
        row_off = np.zeros(n + 1, dtype=np.uint32)
        entries = np.zeros(max(1, n * min(kmax, self.n_nodes)), dtype=np.uint32)
        ne = C.c_size_t()
        L.check(L.lib().bc_gen_sparse_queries_host(self.n_nodes, card.ctypes.data, seed, first, n, kmin, kmax,
                                                   row_off.ctypes.data, entries.ctypes.data, C.byref(ne)))
        return row_off, entries[: ne.value]

    def gen_range_queries_device(self, seed: int, first: int, n: int, kmin: int, kmax: int, desc_ptr: int,
                                 stream: int = 0) -> None:
        L.check(L.lib().bc_gen_range_queries(self._h, seed, first, n, kmin, kmax, desc_ptr, stream or None))

    def gen_range_queries_host(self, seed: int, first: int, n: int, kmin: int, kmax: int) -> np.ndarray:
        card = np.ascontiguousarray(self.tm.card, dtype=np.int32)
        stride = self.desc_stride(L.DESC_RANGE_U8)
        out = np.zeros((n, stride), dtype=np.uint8)
        L.check(L.lib().bc_gen_range_queries_host(self.n_nodes, card.ctypes.data, seed, first, n, kmin, kmax,
                                                  out.ctypes.data))
        return out


def gen_range_queries_host(tm: TreeModel, seed: int, first: int, n: int, kmin: int, kmax: int) -> np.ndarray:
    """Host twin of the on-device generator (no GPU needed)."""
    card = np.ascontiguousarray(tm.card, dtype=np.int32)
    stride = -(-2 * tm.n_nodes // 4) * 4
    out = np.zeros((n, stride), dtype=np.uint8)
    L.check(L.lib().bc_gen_range_queries_host(tm.n_nodes, card.ctypes.data, seed, first, n, kmin, kmax,
                                              out.ctypes.data))
    return out


def measure_fp32_peak(device: int = 0):
    t, c = C.c_double(), C.c_double()
    L.check(L.lib().bc_measure_fp32_peak(device, C.byref(t), C.byref(c)))
    return t.value, c.value


def launch_count() -> int:
    return int(L.lib().bc_launch_count())


class ShardedModel:
    """The model replicated on several GPUs of ONE process; a batch is split into contiguous ranges, one host thread +
    stream set per device, the results land in one host array (SURVEY.md section 8e; BASELINE.json north_star item 4).
    No collective: the path has no exchange step.  Every ``run_*_host`` of :class:`DeviceModel` has a sharded twin here;
    the C calls release the GIL (ctypes), so the devices really run concurrently."""

    def __init__(self, tm: TreeModel, devices: Sequence[int], specialize: bool = True):
        self.tm = tm
        self.replicas: List[DeviceModel] = [DeviceModel(tm, d, specialize=specialize) for d in devices]
        self.mask_words = self.replicas[0].mask_words
        # one long-lived host thread per device (creating threads per call costs ~0.1 ms, a fifth of a 1 M-query call)
        from concurrent.futures import ThreadPoolExecutor

        self._pool = ThreadPoolExecutor(max_workers=len(self.replicas), thread_name_prefix="bc-shard")

    @staticmethod
    def split(n: int, parts: int, align: int = 1):
        """Equal contiguous ranges, remainder to the last (SURVEY.md section 8e); boundaries on multiples of ``align``."""
        base = n // parts // align * align
        bounds = [i * base for i in range(parts)] + [n]
        return [(bounds[i], bounds[i + 1]) for i in range(parts)]

    def _fan_out(self, n: int, work, align: int = 1, out: Optional[np.ndarray] = None) -> np.ndarray:
        """Run ``work(replica, a, b, out[a:b])`` for every replica's slice on its own thread."""
        if out is None:
            out = np.empty(n, dtype=np.float32)
        futs = [self._pool.submit(work, rep, a, b, out[a:b])
                for rep, (a, b) in zip(self.replicas, self.split(n, len(self.replicas), align)) if b > a]
        errs = [f.exception() for f in futs]   # waits for every slice (no replica may still write into `out` on return)
        for e in errs:
            if e is not None:
                raise e
        return out

    def _mask(self, mask, n):
        if mask is None:
            return None
        mask = np.ascontiguousarray(mask, dtype=np.uint32).reshape(n, self.mask_words)
        return mask

    def run_host(self, desc: np.ndarray, fmt: int, mask: Optional[np.ndarray] = None,
                 kernel: int = L.KERNEL_AUTO) -> np.ndarray:
        stride = self.replicas[0].desc_stride(fmt)
        desc = np.ascontiguousarray(desc).reshape(-1)
        n = desc.nbytes // stride
        rows = desc.view(np.uint8).reshape(n, stride)
        mask = self._mask(mask, n)
        return self._fan_out(n, lambda rep, a, b, o: rep.run_host(rows[a:b], fmt, None if mask is None else mask[a:b], kernel, out=o))

    def run_sparse_host(self, row_off: np.ndarray, entries: np.ndarray, mask: Optional[np.ndarray] = None,
                        kernel: int = L.KERNEL_AUTO) -> np.ndarray:
        """SPARSE (CSR) batch: each replica gets a contiguous CSR slice (the library takes absolute entry indices: the
        slice is ``row_off[a:b+1]`` as it stands plus the whole ``entries`` array, nothing is copied on the host)."""
        row_off = np.ascontiguousarray(row_off, dtype=np.uint32)
        entries = np.ascontiguousarray(entries, dtype=np.uint32)
        n = row_off.size - 1
        mask = self._mask(mask, n)
        return self._fan_out(n, lambda rep, a, b, o: rep.run_sparse_host(row_off[a:b + 1], entries, None if mask is None else mask[a:b],
                                                                      kernel, out=o))

    def run_wsparse_host(self, row_off: np.ndarray, words: np.ndarray, mask: Optional[np.ndarray] = None,
                         kernel: int = L.KERNEL_AUTO) -> np.ndarray:
        row_off = np.ascontiguousarray(row_off, dtype=np.uint32)
        words = np.ascontiguousarray(words, dtype=np.uint32)
        n = row_off.size - 1
        mask = self._mask(mask, n)
        return self._fan_out(n, lambda rep, a, b, o: rep.run_wsparse_host(row_off[a:b + 1], words, None if mask is None else mask[a:b],
                                                                       kernel, out=o))

    def run_packed_host(self, klen: np.ndarray, blk_off: np.ndarray, payload: np.ndarray, mask: Optional[np.ndarray] = None,
                        kernel: int = L.KERNEL_AUTO, out: Optional[np.ndarray] = None) -> np.ndarray:
        """PACKED batch: slices on multiples of the 128-query block, ``blk_off`` keeps absolute entry indices."""
        klen = np.ascontiguousarray(klen, dtype=np.uint8)
        blk_off = np.ascontiguousarray(blk_off, dtype=np.uint32)
        payload = np.ascontiguousarray(payload, dtype=np.uint8)
        n = klen.size
        mask = self._mask(mask, n)

        def work(rep, a, b, o):
            rep.run_packed_host(klen[a:b], blk_off[a // 128:(b + 127) // 128 + 1], payload, None if mask is None else mask[a:b], kernel, out=o)

        return self._fan_out(n, work, align=128, out=out)

    def submit_packed_host(self, klen: np.ndarray, blk_off: np.ndarray, payload: np.ndarray, out: np.ndarray,
                           mask: Optional[np.ndarray] = None, kernel: int = L.KERNEL_AUTO):
        """Asynchronous ``run_packed_host``: every replica's slice is enqueued on its device (``DeviceModel.submit_packed_host``,
        from the replica's own host thread) and the tickets come back; ``out`` (pinned) is complete after ``wait(tickets)``.
        Two batches in flight per device overlap each device's next copy with its kernels and read-back."""
        n = klen.size
        if mask is not None:
            mask = mask.reshape(n, self.mask_words)
        parts = [(rep, a, b) for rep, (a, b) in zip(self.replicas, self.split(n, len(self.replicas), 128)) if b > a]
        futs = [self._pool.submit(rep.submit_packed_host, klen[a:b], blk_off[a // 128:(b + 127) // 128 + 1], payload, out[a:b],
                                  None if mask is None else mask[a:b].reshape(-1), kernel) for rep, a, b in parts]
        tickets, err = [], None
        for (rep, _, _), f in zip(parts, futs):
            e = f.exception()
            if e is None:
                tickets.append((rep, f.result()))
            elif err is None:
                err = e
        if err is not None:
            self.wait(tickets)   # nothing may still write into `out` when the error surfaces
            raise err
        return tickets

    def wait(self, tickets) -> None:
        for rep, t in tickets:
            rep.wait(t)

    def attach_counts(self, counts: np.ndarray) -> None:
        for r in self.replicas:
            r.attach_counts(counts)

    def get_counts(self, node_first: int = 0, node_count: Optional[int] = None) -> np.ndarray:
        return self.replicas[0].get_counts(node_first, node_count)

    def update(self, inserted=None, deleted=None) -> np.ndarray:
        """The same batch (host arrays, see ``DeviceModel.update``) on every replica, each from its own host thread.
        Counts are integers and the normalisation is exact, so the replicas stay bit-identical.  Returns the touched
        nodes."""
        futs = [self._pool.submit(r.update, inserted, deleted) for r in self.replicas]
        errs = [f.exception() for f in futs]
        for e in errs:
            if e is not None:
                raise e
        return futs[0].result()

    def close(self):
        self._pool.shutdown(wait=True)
        for r in self.replicas:
            r.close()
