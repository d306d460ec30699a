"""EdgeIndex: the cached CSR/CSC of a Graph (mirror of reference pgl/utils/edge_index.py).

numpy mode builds on the host through ``pglb_build_index_host`` (twin of the reference's
Cython ``graph_kernel.build_index``); tensor mode builds on the device through
``pglb_csr_build``.  Both are stable, so ``sorted_edges()`` is identical between modes
(the reference's tensor mode depends on paddle.argsort's unspecified tie order,
SURVEY.md appendix B).
"""
import ctypes
import os

import numpy as np
import torch

from .. import _lib, ops
from .helper import check_is_tensor, to_tensor


def _np_ptr(a):
    return ctypes.c_void_p(a.ctypes.data)


def build_index_host(u, v, num_nodes):
    """(degree, sorted_v, sorted_u, sorted_eid, indptr) like graph_kernel.build_index
    (reference pgl/graph_kernel.pyx:59-88); u, v may be strided int64 views."""
    u = np.asarray(u)
    v = np.asarray(v)
    if u.dtype != np.int64:
        u = u.astype(np.int64)
    if v.dtype != np.int64:
        v = v.astype(np.int64)
    E = int(u.shape[0])
    N = int(num_nodes)
    if E and (u.strides[0] % 8 or v.strides[0] % 8 or u.strides[0] <= 0 or v.strides[0] <= 0):
        u = np.ascontiguousarray(u)
        v = np.ascontiguousarray(v)
    degree = np.empty(N, np.int64)
    indptr = np.empty(N + 1, np.int64)
    su = np.empty(E, np.int64)
    sv = np.empty(E, np.int64)
    se = np.empty(E, np.int64)
    us = u.strides[0] // 8 if E else 1
    vs = v.strides[0] // 8 if E else 1
    _lib.check(_lib.lib.pglb_build_index_host(_np_ptr(u), us, _np_ptr(v), vs, E, N, _np_ptr(degree),
                                              _np_ptr(indptr), _np_ptr(su), _np_ptr(sv),
                                              _np_ptr(se)))
    return degree, sv, su, se, indptr


def sorted_successor_csr(u, v, num_nodes):
    """(indptr, cols) keyed by ``u`` with every row's ``v`` in ascending order: the stable index build keyed by
    ``v``, then again keyed by ``u``.  indptr is the one of ``EdgeIndex.from_edges(u, v)``.  Host or device, as the
    inputs are."""
    if check_is_tensor(u, v):
        n = int(num_nodes.item()) if isinstance(num_nodes, torch.Tensor) else int(num_nodes)
        _, by_v_u, by_v_v, _, _ = ops.csr_build(v, u, n)
        _, cols, _, _, indptr = ops.csr_build(by_v_u, by_v_v, n)
    else:
        _, by_v_u, by_v_v, _, _ = build_index_host(v, u, num_nodes)
        _, cols, _, _, indptr = build_index_host(by_v_u, by_v_v, num_nodes)
    return indptr, cols


class EdgeIndex(object):
    """Sorted edges in compressed form, keyed by ``u`` (reference edge_index.py:27-36)."""

    def __init__(self):
        self._max_degree = None

    @classmethod
    def from_edges(cls, u, v, num_nodes, v_bound=None):
        """reference pgl/utils/edge_index.py:38-58.  ``v_bound``: number of nodes on the v side (the kernels
        index feature rows with v): ids outside [0, v_bound) raise instead of corrupting memory later; the u side
        is range-checked by the index build itself (PGLB_ESHAPE)."""
        self = cls()
        self._is_tensor = check_is_tensor(u, v, num_nodes)
        if v_bound is not None and len(v) > 0:
            vb = int(v_bound.item()) if isinstance(v_bound, torch.Tensor) else int(v_bound)
            lo, hi = (int(v.min()), int(v.max()))
            if lo < 0 or hi >= vb:
                raise ValueError("edge endpoint %d outside [0, %d)" % (lo if lo < 0 else hi, vb))
        if self._is_tensor:
            n = int(num_nodes.item()) if isinstance(num_nodes, torch.Tensor) else int(num_nodes)
            u = to_tensor(u)
            v = to_tensor(v)
            self._degree, self._sorted_v, self._sorted_u, self._sorted_eid, self._indptr = \
                ops.csr_build(u, v, n)
        else:
            self._degree, self._sorted_v, self._sorted_u, self._sorted_eid, self._indptr = \
                build_index_host(u, v, num_nodes)
        return self

    @classmethod
    def from_index(cls, sorted_v, sorted_u, sorted_eid, degree, indptr):
        """reference pgl/utils/edge_index.py:60-70."""
        self = cls()
        self._degree = degree
        self._sorted_v = sorted_v
        self._sorted_u = sorted_u
        self._sorted_eid = sorted_eid
        self._indptr = indptr
        self._is_tensor = check_is_tensor(sorted_v, sorted_u, sorted_eid, degree, indptr)
        return self

    @classmethod
    def load(cls, path, mmap_mode="r"):
        """reference pgl/utils/edge_index.py:72-95 (same .npy layout)."""
        self = cls()
        self._degree = np.load(os.path.join(path, "degree.npy"), mmap_mode=mmap_mode)
        self._sorted_u = np.load(os.path.join(path, "sorted_u.npy"), mmap_mode=mmap_mode)
        self._sorted_v = np.load(os.path.join(path, "sorted_v.npy"), mmap_mode=mmap_mode)
        self._sorted_eid = np.load(os.path.join(path, "sorted_eid.npy"), mmap_mode=mmap_mode)
        self._indptr = np.load(os.path.join(path, "indptr.npy"), mmap_mode=mmap_mode)
        self._is_tensor = False
        return self

    @property
    def degree(self):
        return self._degree

    @property
    def max_degree(self):
        """Longest row (cached; one device->host read in tensor mode)."""
        if self._max_degree is None:
            if len(self._degree) == 0:
                self._max_degree = 0
            elif self._is_tensor:
                self._max_degree = int(self._degree.max().item())
            else:
                self._max_degree = int(np.max(self._degree))
        return self._max_degree

    def packed_cols(self, n_src, row_bytes):
        """Cached packed column ids (see ops.pack_cols) for gathers of `row_bytes` rows."""
        cache = self.__dict__.setdefault("_packed_cache", {})
        key = (int(n_src), int(row_bytes) if ops.HOT_L2_BYTES > 0 else 0)
        if key not in cache:
            cache[key] = ops.pack_cols(self._sorted_v, n_src, row_bytes)
        return cache[key]

    def narrow_plan(self, n_src, row_bytes=64):
        """Cached plan of the narrow-row kernel (see ops.narrow_plan).  The row flags depend on the index only; the
        L2 residency hints on how many rows of this width fit the budget, hence the key."""
        cache = self.__dict__.setdefault("_plan_cache", {})
        key = int(row_bytes) if ops.NARROW_HOT_BYTES > 0 else 0
        if key not in cache:
            cache[key] = ops.narrow_plan(self._indptr, self._sorted_v, n_src, row_bytes)
        return cache[key]

    def slot_scale(self, scale_src):
        """scale_src[cols[j]] for every CSR slot j -- the edge values of the normalised adjacency -- cached per scale
        tensor (identity + in-place version counter), so the narrow-row kernel streams 4 bytes per slot instead of
        gathering a 32-byte sector per edge."""
        cache = self.__dict__.setdefault("_slot_scale_cache", {})
        key = (scale_src.data_ptr(), int(scale_src._version), int(scale_src.numel()))
        hit = cache.get("key") == key
        if not hit:
            cache["key"] = key
            cache["val"] = scale_src.reshape(-1)[self._sorted_v].contiguous()
            cache["ref"] = scale_src          # keeps the storage alive, so the data_ptr cannot be recycled
        return cache["val"]

    def csr(self):
        """dict consumed by pgl_b200.ops: rows keyed by u, columns = v, eid per slot."""
        return {"indptr": self._indptr, "cols": self._sorted_v, "eid": self._sorted_eid, "rows": self._sorted_u,
                "degree": self._degree, "max_degree": self.max_degree, "packed": self.packed_cols,
                "plan": self.narrow_plan, "slot_scale": self.slot_scale}

    def view_v(self, u=None):
        """reference pgl/utils/edge_index.py:103-114 (numpy mode only)."""
        if self._is_tensor:
            raise NotImplementedError("not implemented!")
        if u is None:
            return np.split(self._sorted_v, self._indptr[1:-1])
        u = np.array(u, dtype="int64")
        return np.array([self._sorted_v[self._indptr[j]:self._indptr[j + 1]] for j in u],
                        dtype=object)

    def view_eid(self, u=None):
        """reference pgl/utils/edge_index.py:116-127 (numpy mode only)."""
        if self._is_tensor:
            raise NotImplementedError("not implemented!")
        if u is None:
            return np.split(self._sorted_eid, self._indptr[1:-1])
        u = np.array(u, dtype="int64")
        return np.array([self._sorted_eid[self._indptr[j]:self._indptr[j + 1]] for j in u],
                        dtype=object)

    def triples(self):
        """reference pgl/utils/edge_index.py:129-132."""
        return self._sorted_u, self._sorted_v, self._sorted_eid

    def is_tensor(self):
        return self._is_tensor

    def tensor(self, inplace=True, uva=False):
        """reference pgl/utils/edge_index.py:139-178 (UVA out of scope)."""
        if self._is_tensor:
            return self
        if uva:
            raise ValueError("uva mode is not supported by pgl_b200")
        vals = [to_tensor(np.asarray(a)) for a in
                (self._sorted_v, self._sorted_u, self._sorted_eid, self._degree, self._indptr)]
        if inplace:
            self._sorted_v, self._sorted_u, self._sorted_eid, self._degree, self._indptr = vals
            self._is_tensor = True
            return self
        return EdgeIndex.from_index(sorted_v=vals[0], sorted_u=vals[1], sorted_eid=vals[2],
                                    degree=vals[3], indptr=vals[4])

    def numpy(self, inplace=True):
        """reference pgl/utils/edge_index.py:180-206 (without its inplace degree/indptr bug,
        SURVEY.md appendix B)."""
        if not self._is_tensor:
            return self
        vals = [a.cpu().numpy() for a in
                (self._sorted_v, self._sorted_u, self._sorted_eid, self._degree, self._indptr)]
        if inplace:
            self._sorted_v, self._sorted_u, self._sorted_eid, self._degree, self._indptr = vals
            self._is_tensor = False
            return self
        return EdgeIndex.from_index(sorted_v=vals[0], sorted_u=vals[1], sorted_eid=vals[2],
                                    degree=vals[3], indptr=vals[4])

    def dump(self, path):
        """reference pgl/utils/edge_index.py:208-219."""
        if self._is_tensor:
            self.numpy(inplace=False).dump(path)
            return
        if not os.path.exists(path):
            os.makedirs(path)
        np.save(os.path.join(path, "degree.npy"), self._degree)
        np.save(os.path.join(path, "sorted_v.npy"), self._sorted_v)
        np.save(os.path.join(path, "sorted_u.npy"), self._sorted_u)
        np.save(os.path.join(path, "sorted_eid.npy"), self._sorted_eid)
        np.save(os.path.join(path, "indptr.npy"), self._indptr)
