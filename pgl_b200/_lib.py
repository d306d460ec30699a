"""ctypes binding of libpglb.so (include/pglb.h).  The product path has no fallback: if the
shared library is missing this module raises at import time."""
import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_int, c_int64, c_size_t, c_uint64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PGLB_LIB") or os.path.join(_HERE, "libpglb.so")
METIS_PATH = os.path.join(_HERE, "third_party", "libmetis_i64.so")

PGLB_OK = 0
PGLB_CUDA_ERR_BASE = 1000
REDUCE = {"sum": 0, "mean": 1, "max": 2, "min": 3}
MSG = {"copy": 0, "add": 1, "sub": 2, "mul": 3, "div": 4}
BCAST_FULL, BCAST_HEAD, BCAST_SCALAR = 0, 1, 2
WALK_UNIFORM, WALK_NODE2VEC, WALK_NODE2VEC_PLUS = 0, 1, 2


class PglbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libpglb error %d: %s" % (code, msg))
        self.code = code


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "pgl_b200: %s not found. Build it first with `python pgl_b200/build.py` "
            "(or __graft_entry__.build()); there is no CPU / eager fallback." % LIB_PATH)
    return ctypes.CDLL(LIB_PATH)


lib = _load()

_p = c_void_p
_i64 = c_int64

_SIGS = {
    "pglb_version": (c_int, []),
    "pglb_last_error": (c_char_p, []),
    "pglb_launch_count": (c_int64, []),
    "pglb_csr_build_ws": (c_int, [_i64, _i64, POINTER(c_size_t)]),
    "pglb_csr_build": (c_int, [_p, _i64, _p, _i64, _i64, _i64, _p, _p, _p, _p, _p, _p, c_size_t, _p]),
    "pglb_build_index_host": (c_int, [_p, _i64, _p, _i64, _i64, _i64, _p, _p, _p, _p, _p]),
    "pglb_segment_ids_ws": (c_int, [_i64, POINTER(c_size_t)]),
    "pglb_segment_ids": (c_int, [_p, _i64, _i64, _p, _p, _p, _p, c_size_t, _p]),
    "pglb_segment_indptr": (c_int, [_p, _i64, _i64, _p, _p]),
    "pglb_spmm_csr_ws": (c_int, [_i64, _i64, _i64, POINTER(c_size_t)]),
    "pglb_spmm_csr_f32": (c_int, [_p, _p, _p, _p, _i64, _p, _i64, c_int, _p, _i64, _i64, _i64, _i64,
                                  _i64, _i64, c_int, c_int, _p, _p, _p, _i64, c_int, _p, c_size_t, _p]),
    "pglb_narrow_plan_ws": (c_int, [_i64, POINTER(c_size_t)]),
    "pglb_narrow_plan": (c_int, [_p, _p, _p, _i64, _i64, _i64, _p, _p, _p, _p, c_size_t, _p]),
    "pglb_spmm_narrow_ws": (c_int, [_i64, _i64, POINTER(c_size_t)]),
    "pglb_spmm_narrow_f32": (c_int, [_p, _p, _p, _p, _p, _i64, _p, _i64, _i64, _i64, _i64, _i64, c_int, _p, _p, _p,
                                     c_int, _p, c_size_t, _p]),
    "pglb_memcpy2d_async": (c_int, [_p, c_size_t, _p, c_size_t, c_size_t, c_size_t, c_int, _p]),
    "pglb_ipc_alloc": (c_int, [c_size_t, POINTER(c_void_p), _p]),
    "pglb_ipc_free": (c_int, [_p]),
    "pglb_ipc_open": (c_int, [_p, POINTER(c_void_p)]),
    "pglb_ipc_close": (c_int, [_p]),
    "pglb_pack_cols": (c_int, [_p, _i64, _i64, _p, _i64, _p, _p]),
    "pglb_send_uv_f32": (c_int, [_p, _p, _p, _i64, _p, _i64, _i64, _i64, c_int, _p, _p]),
    "pglb_gather_rows_f32": (c_int, [_p, _i64, _p, _i64, _i64, _i64, _p, _i64, _p]),
    "pglb_scatter_rows_f32": (c_int, [_p, _i64, _p, _i64, _i64, _p, _i64, _p]),
    "pglb_edge_softmax_csr_ws": (c_int, [_i64, POINTER(c_size_t)]),
    "pglb_edge_softmax_csr_f32": (c_int, [_p, _p, _p, _p, _i64, _i64, _i64, _p, c_size_t, _p]),
    "pglb_degree_norm_f32": (c_int, [_p, _i64, _p, _p]),
    "pglb_sample_count": (c_int, [_p, _p, _i64, _i64, _p, _p, _p]),
    "pglb_sample_fill": (c_int, [_p, _p, _p, _p, _i64, _i64, ctypes.c_uint64, _p, _p, _p, _p]),
    "pglb_reindex_table_init": (c_int, [_p, _i64, _p]),
    "pglb_reindex_graph_ws": (c_int, [_i64, POINTER(c_size_t)]),
    "pglb_reindex_graph": (c_int, [_p, _i64, _p, _p, _i64, _p, _p, _p, _p, _p, _p, c_size_t, _p]),
    "pglb_copy2d_kernel_async": (c_int, [_p, c_size_t, _p, c_size_t, c_size_t, _i64, c_int, _p]),
    "pglb_linear_tf32x3_f32": (c_int, [_p, _i64, _p, _p, _p, _i64, _i64, _i64, _i64, c_int, _p]),
    "pglb_gat_fused_csr_f32": (c_int, [_p, _p, _p, _i64, _p, _p, ctypes.c_float, _p, _i64, _i64, _i64, _i64,
                                       _i64, _i64, _p, c_size_t, _p]),
    "pglb_head_dots_f32": (c_int, [_p, _i64, _i64, _i64, _i64, _p, _p, _p, _p, _p]),
    "pglb_gat_fused_train_csr_f32": (c_int, [_p, _p, _p, _i64, _p, _p, ctypes.c_float, _p, _i64, _p, _i64, _i64,
                                             _i64, _i64, _i64, _p, c_size_t, _p]),
    "pglb_gat_bwd_edge_f32": (c_int, [_p, _p, _p, _p, _i64, _p, _i64, _p, _i64, _p, _p, _p, ctypes.c_float,
                                      _i64, _i64, _i64, _p, _p, _p]),
    "pglb_gat_attention_csr_f32": (c_int, [_p, _p, _p, _p, ctypes.c_float, _p, _i64, _i64, _i64, _p,
                                           c_size_t, _p]),
    "pglb_sddmm_dot_f32": (c_int, [_p, _p, _p, _i64, _p, _i64, _i64, _i64, _i64, _p, _p]),
    "pglb_edge_softmax_bwd_csr_f32": (c_int, [_p, _p, _p, _p, _p, _i64, _i64, _i64, _p]),
    "pglb_maxmin_bwd_f32": (c_int, [_p, _p, _p, _p, _p, _p, _i64, _i64, _p]),
    "pglb_debug_task_trace": (c_int, [_p, _i64]),
    "pglb_map_nodes": (c_int, [_p, _i64, _p, _i64, _p, _p, _p]),
    "pglb_map_edges": (c_int, [_p, _i64, _p, _i64, _p, _i64, _p, _p, _p]),
    "pglb_invert_perm": (c_int, [_p, _i64, _p, _p]),
    "pglb_halo_plan_ws": (c_int, [_i64, _i64, POINTER(c_size_t)]),
    "pglb_halo_plan_count": (c_int, [_p, _i64, _i64, _i64, _i64, _p, _p, _p, c_size_t, _p]),
    "pglb_halo_plan_fill": (c_int, [_p, _i64, _i64, _i64, _i64, _p, _i64, _p, _p, _p, _p, _p, _p, c_size_t, _p]),
    "pglb_metis_partition": (c_int, [c_char_p, _i64, _p, _p, _i64, _p, _p, c_int, _p]),
    "pglb_random_walk": (c_int, [_p, _p, _i64, _p, _i64, _i64, c_int, c_double, c_double, c_uint64, _p, _i64, _p]),
    "pglb_random_walk_host": (c_int, [_p, _p, _i64, _p, _i64, _i64, c_int, c_double, c_double, c_uint64, _p, _i64]),
    "pglb_skip_gram_ws": (c_int, [_i64, _i64, POINTER(c_size_t)]),
    "pglb_skip_gram_count": (c_int, [_p, _i64, _i64, _i64, _i64, c_uint64, _p, _p, c_size_t, _p]),
    "pglb_skip_gram_fill": (c_int, [_p, _i64, _i64, _i64, _i64, c_uint64, _p, _p, _p, _p, c_size_t, _p]),
}

for _name, (_res, _args) in _SIGS.items():
    _f = getattr(lib, _name)
    _f.restype = _res
    _f.argtypes = _args


def check(rc):
    if rc != PGLB_OK:
        msg = lib.pglb_last_error()
        raise PglbError(rc, msg.decode("utf-8", "replace") if msg else "")


def launch_count():
    return int(lib.pglb_launch_count())
