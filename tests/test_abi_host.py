"""CPU-side tests: the C-ABI library loads and exports every symbol include/pglb.h declares,
argument validation happens before any device work, and the host entry points
(build_index_host, METIS) match the reference-generated golden fixtures bit for bit."""
import ctypes
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


def test_header_symbols_exported():
    from pgl_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "pglb.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    names = sorted(set(re.findall(r"\b(pglb_[a-z0-9_]+)\s*\(", hdr)))
    assert len(names) >= 18
    for n in names:
        assert hasattr(_lib.lib, n), "libpglb.so does not export %s" % n
        assert n in _lib._SIGS, "ctypes signature missing for %s" % n
    assert _lib.lib.pglb_version() == 100


def test_error_convention():
    from pgl_b200 import _lib
    lib = _lib.lib
    need = ctypes.c_size_t(0)
    assert lib.pglb_csr_build_ws(-1, 5, ctypes.byref(need)) == -1
    assert b"negative" in lib.pglb_last_error()
    assert lib.pglb_spmm_csr_ws(10, 100, 16, None) == -1
    # invalid enums / shapes are rejected without touching the device
    rc = lib.pglb_spmm_csr_f32(None, None, None, None, 4, None, 0, 0, None, 4, 10, 10, 5, 4, 1,
                               0, 9, None, None, None, -1, 0, None, 0, None)
    assert rc == -1 and b"reduce_op" in lib.pglb_last_error()
    rc = lib.pglb_send_uv_f32(None, None, None, 1, None, 1, 5, 4, 0, None, None)
    assert rc == -1
    with pytest.raises(_lib.PglbError):
        _lib.check(rc)
    # zero-sized problems are OK no-ops
    assert lib.pglb_spmm_csr_f32(None, None, None, None, 4, None, 0, 0, None, 4, 0, 0, 0, 4, 1, 0,
                                 0, None, None, None, -1, 0, None, 0, None) == 0


def test_build_index_host_vs_reference_golden():
    from pgl_b200.utils.edge_index import build_index_host
    g = np.load(os.path.join(GOLDEN, "ref_build_index.npz"))
    for name in ("tiny", "uniform", "powerlaw", "gaps"):
        n = int(g[name + "_n"])
        deg, sv, su, se, ip = build_index_host(g[name + "_u"], g[name + "_v"], n)
        assert (deg == g[name + "_degree"]).all()
        assert (sv == g[name + "_sorted_v"]).all()
        assert (su == g[name + "_sorted_u"]).all()
        assert (se == g[name + "_sorted_eid"]).all()
        assert (ip == g[name + "_indptr"]).all()
    # strided views of an [E,2] array are read in place
    e = np.stack([g["uniform_v"], g["uniform_u"]], 1)
    deg, sv, su, se, ip = build_index_host(e[:, 1], e[:, 0], int(g["uniform_n"]))
    assert (se == g["uniform_sorted_eid"]).all() and (sv == g["uniform_sorted_v"]).all()
    from pgl_b200 import _lib
    with pytest.raises(_lib.PglbError):
        build_index_host(np.array([7]), np.array([0]), 3)


def test_metis_vs_reference_golden():
    from pgl_b200 import _lib, partition
    if not os.path.exists(os.environ.get("PGLB_LIBMETIS") or _lib.METIS_PATH):   # the library metis_csr loads
        pytest.skip("libmetis_i64.so not built")
    m = np.load(os.path.join(GOLDEN, "ref_metis.npz"))
    n = int(m["n"])
    for k in (2, 8):
        part = partition.metis_csr(n, m["indptr"], m["sorted_v"], k)
        assert (part == m["part_%d" % k]).all()
        assert set(np.unique(part)) == set(range(k))
    part = partition.metis_csr(n, m["indptr"], m["sorted_v"], 8,
                               node_weights=m["node_weights_scaled"])
    assert (part == m["part_8_nw"]).all()
    assert (partition._metis_weight_scale(m["node_weights_raw"]) == m["node_weights_scaled"]).all()
    # the Graph-level API (numpy mode) goes through the same CSR
    import pgl_b200 as pgl
    g = pgl.Graph(edges=m["edges"], num_nodes=n)
    assert (pgl.partition.metis_partition(g, 8) == m["part_8"]).all()
    assert (pgl.partition.metis_partition(g, 1) == 0).all()
    rp = pgl.partition.random_partition(g, 4)
    assert rp.shape == (n,) and np.bincount(rp).max() - np.bincount(rp).min() <= 1
    with pytest.raises(_lib.PglbError):
        partition.metis_csr(n, m["indptr"], m["sorted_v"], 2, libmetis_path="/nonexistent/libmetis.so")


def test_numpy_mode_graph(kat, tmp_path):
    import pgl_b200 as pgl
    k = kat["degree"]
    g = pgl.Graph(edges=[tuple(e) for e in k["edges"]], num_nodes=k["num_nodes"])
    assert not g.is_tensor()
    assert (g.indegree() == np.array(k["indegree"])).all()
    assert (g.outdegree() == np.array(k["outdegree"])).all()
    assert (g.indegree(nodes=k["subset"]) == np.array(k["indegree"])[k["subset"]]).all()
    assert (g.outdegree(nodes=k["subset"]) == np.array(k["outdegree"])[k["subset"]]).all()
    s, d, e = g.sorted_edges("dst")
    assert (np.diff(d) >= 0).all()
    with pytest.raises(ValueError):
        g.sorted_edges("foo")
    # send / recv need tensor mode
    with pytest.raises(ValueError):
        g.send(lambda s, d, e: {}, src_feat={})
    with pytest.raises(ValueError):
        g.recv(lambda m: m, {})
    with pytest.raises(ValueError):
        g.send_recv(np.zeros((5, 2), np.float32))
    succ = g.successor()
    assert [set(x) for x in succ] == [{1}, {2}, set(), {4}, set()]
    # dump / load keep the reference's .npy layout, including the cached CSR
    p = str(tmp_path / "g")
    g.dump(p)
    for f in ("num_nodes.npy", "edges.npy", "num_graph.npy", "adj_dst/indptr.npy",
              "adj_src/sorted_eid.npy"):
        assert os.path.exists(os.path.join(p, f)), f
    g2 = pgl.Graph.load(p)
    assert (np.asarray(g2.indegree()) == np.array(k["indegree"])).all()
    assert g2.num_nodes == k["num_nodes"] and (np.asarray(g2.edges) == g.edges).all()
    # batching
    j = pgl.Graph.batch([g, g])
    assert j.num_graph == 2 and j.num_nodes == 10
    assert j.graph_node_id.tolist() == [0] * 5 + [1] * 5
    assert j.graph_edge_id.tolist() == [0] * 3 + [1] * 3


def test_tensor_mode_requires_cuda():
    import torch
    import pgl_b200 as pgl
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    g = pgl.Graph(edges=[(0, 1)], num_nodes=2)
    with pytest.raises(RuntimeError, match="CUDA"):
        g.tensor()
    with pytest.raises(RuntimeError, match="CUDA"):
        pgl.ops.aggregate_copy(torch.zeros(2, 4), {}, 2)


def test_argument_validation_of_the_newer_entries():
    """Dense transform, sampling and reindex entries: shapes and pointers are checked before any
    device work, zero-sized problems are no-ops (no GPU needed for either)."""
    from pgl_b200 import _lib
    lib = _lib.lib
    one = ctypes.c_void_p(16)   # a non-NULL, 16-byte aligned dummy: must never be dereferenced here
    # pglb_linear_tf32x3_f32(x, ldx, w, bias, out, ldo, M, K, N, act, stream)
    assert lib.pglb_linear_tf32x3_f32(None, 128, None, None, None, 128, 0, 128, 128, 0, None) == 0
    assert lib.pglb_linear_tf32x3_f32(one, 130, one, None, one, 128, 10, 130, 128, 0, None) < 0
    assert b"K must be" in lib.pglb_last_error()
    assert lib.pglb_linear_tf32x3_f32(one, 128, one, None, one, 96, 10, 128, 96, 0, None) < 0
    assert b"N must be" in lib.pglb_last_error()
    assert lib.pglb_linear_tf32x3_f32(one, 128, one, None, one, 128, 10, 128, 128, 7, None) < 0
    assert lib.pglb_linear_tf32x3_f32(None, 128, one, None, one, 128, 10, 128, 128, 0, None) < 0
    assert lib.pglb_linear_tf32x3_f32(one, 126, one, None, one, 128, 10, 124, 128, 0, None) < 0  # ldx % 4
    # sampling
    assert lib.pglb_sample_fill(None, None, None, None, 0, 5, 1, None, None, None, None) == 0
    assert lib.pglb_sample_fill(one, one, None, one, 3, 5000, 1, one, one, None, None) < 0
    assert b"4096" in lib.pglb_last_error()
    assert lib.pglb_sample_fill(None, one, None, one, 3, 5, 1, one, one, None, None) < 0
    assert lib.pglb_sample_count(None, None, -1, 5, None, one, None) < 0
    # reindex
    need = ctypes.c_size_t(0)
    assert lib.pglb_reindex_graph_ws(1000, ctypes.byref(need)) == 0 and need.value >= 2 * 8 * 1000
    assert lib.pglb_reindex_graph_ws(-1, ctypes.byref(need)) < 0
    assert lib.pglb_reindex_table_init(None, 0, None) == 0
    assert lib.pglb_reindex_table_init(None, 10, None) < 0
    assert lib.pglb_reindex_graph(one, 3, one, one, 5, one, one, one, one, one, one, 8, None) < 0
    assert b"workspace" in lib.pglb_last_error()


def test_plain_c_consumer(tmp_path):
    """include/pglb.h + libpglb.so from plain C (gcc, no Python in the loop): the binding a maintainer of
    the reference would write links the same way (INTEGRATION.md section B)."""
    import shutil
    import subprocess
    if shutil.which("gcc") is None:
        pytest.skip("gcc not available")
    from pgl_b200 import _lib
    libdir = os.path.dirname(_lib.LIB_PATH) if hasattr(_lib, "LIB_PATH") else os.path.join(ROOT, "pgl_b200")
    exe = str(tmp_path / "c_abi_smoke")
    cmd = ["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
           os.path.join(ROOT, "tests", "c_abi_smoke.c"), "-o", exe, "-L", libdir, "-lpglb",
           "-Wl,-rpath," + libdir]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout
    r = subprocess.run([exe], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0 and "C_ABI_OK indegree=[1 2 1 0 1]" in r.stdout, (r.returncode, r.stdout)
