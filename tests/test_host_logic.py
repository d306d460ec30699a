"""CPU tests of host-side helpers that need no device: broadcast classification, partition
helpers, the builder, workspace sizing through the C-ABI."""
import ctypes
import os

import numpy as np
import pytest

REF_GK = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_graph_kernel.npz")


def test_classify_bcast():
    from pgl_b200 import ops
    from pgl_b200._lib import BCAST_FULL, BCAST_HEAD, BCAST_SCALAR
    assert ops.classify_bcast((10, 8, 16), (50, 8, 1)) == (BCAST_HEAD, 16)
    assert ops.classify_bcast((10, 8, 16), (50, 1, 1)) == (BCAST_SCALAR, 1)
    assert ops.classify_bcast((10, 8, 16), (50, 8, 16)) == (BCAST_FULL, 1)
    assert ops.classify_bcast((10, 128), (50, 1)) == (BCAST_SCALAR, 1)
    assert ops.classify_bcast((10, 2, 3, 4), (50, 2, 1, 1)) == (BCAST_HEAD, 12)
    assert ops.classify_bcast((10, 8, 16), (50, 1, 16)) is None  # needs expand()


def test_workspace_queries_and_version():
    from pgl_b200 import _lib
    lib = _lib.lib
    need = ctypes.c_size_t(0)
    _lib.check(lib.pglb_spmm_csr_ws(10_000_000, 100_000_000, 128, ctypes.byref(need)))
    assert 0 < need.value < (1 << 30)  # partial buffers of the cfg5 aggregation stay well below 1 GB
    small = ctypes.c_size_t(0)
    _lib.check(lib.pglb_spmm_csr_ws(100, 1000, 128, ctypes.byref(small)))
    assert small.value <= need.value
    _lib.check(lib.pglb_edge_softmax_csr_ws(1000, ctypes.byref(small)))
    assert small.value >= 256
    assert isinstance(_lib.launch_count(), int)
    # host-only entry points validate before touching CUDA
    assert lib.pglb_memcpy2d_async(None, 0, None, 0, 0, 0, 1, None) == 0
    assert lib.pglb_memcpy2d_async(None, 16, None, 16, 16, 1, 1, None) == -1
    assert lib.pglb_ipc_open(None, None) == -1
    assert lib.pglb_gat_fused_csr_f32(None, None, None, 128, None, None, 0.2, None, 128, 10, 10, 5, 8,
                                      20, None, 0, None) == -4  # H*head_dim > 128: unsupported shape


def test_block_partition_and_relabel():
    import pgl_b200 as pgl
    from pgl_b200.distributed.halo import block_offsets, relabel_by_partition
    p = pgl.partition.block_partition(10, 4)
    assert p.tolist() == [0, 0, 0, 1, 1, 1, 2, 2, 2, 3]
    new_id, off = relabel_by_partition(p, 4)
    assert off == block_offsets(10, 4) and new_id.tolist() == list(range(10))


def test_builder_is_loadable_without_the_library():
    import __graft_entry__ as ge
    b = ge.load_builder()
    assert os.path.basename(b.LIB) == "libpglb.so" and callable(b.build_all)
    # up to date => no-op
    assert b.build_lib() == b.LIB


def test_gen_edges_and_bytes_model():
    import torch
    import bench
    e = bench.gen_edges(torch, 1000, 5000, 0.8, 7, "cpu")
    assert e.shape == (5000, 2) and int(e.min()) >= 0 and int(e.max()) < 1000
    # SURVEY section 8d: 572 B/edge at D=128, N/E = 0.1 (+ the two norm vectors)
    b = bench.algorithmic_bytes(10_000_000, 100_000_000, 128)
    assert abs(b / 100_000_000 - 572.8) < 0.1
    # the CPU arm's row sample: rows dst < n_s with ALL their in-edges; the GCN restatement on it equals numpy
    en = e.numpy()
    src, dst = np.ascontiguousarray(en[:, 0]), np.ascontiguousarray(en[:, 1])
    lib = bench._load_oracle_c()
    prob = bench.CpuGcn(lib, src, dst, 1000, 8, 0.1, threads=2)
    assert prob.n_s == 100 and (prob.dst < 100).all() and prob.e_s == int((dst < 100).sum())
    x = np.random.default_rng(1).standard_normal((1000, 8)).astype(np.float32)
    norm = bench.cpu_norm(np.bincount(dst, minlength=1000))
    for threads in (1, 2):
        t, det = prob.run(x, norm, threads)
        want = np.zeros((100, 8), np.float32)
        xs = x * norm[:, None]
        for s_, d_ in zip(prob.src, prob.dst):
            want[d_] += xs[s_]
        want *= norm[:100, None]
        assert np.array_equal(prob.out, want) and t > 0 and det["sample_edges"] == prob.e_s
    st = bench.parity_stats(prob.out, want)
    assert st["pass"] and st["bit_exact_rows"] == 100 and st["max_rel_err"] == 0.0
    bad = want.copy()
    bad[3, 2] += 1.0
    assert not bench.parity_stats(bad, want)["pass"]


def test_relabel_matches_reference_graph_kernel():
    from pgl_b200.utils import relabel
    ref = np.load(REF_GK)   # inputs and the reference's own compiled map_nodes / map_edges on them
    old, nodes, edges, eid = (ref["relabel_" + k] for k in ("old", "nodes", "edges", "eid"))
    reindex = {int(o): i for i, o in enumerate(old)}
    mn = relabel.map_nodes(nodes, reindex)
    me = relabel.map_edges(eid, edges, reindex)
    assert mn.tolist() == [reindex[int(v)] for v in nodes]
    assert me.tolist() == [[reindex[int(a)], reindex[int(b)]] for a, b in edges[eid]]
    assert np.array_equal(ref["relabel_map_nodes"], mn)
    assert np.array_equal(ref["relabel_map_edges"], me)


def test_bench_reference_arm_contract():
    """bench.py --impl reference runs anywhere (no GPU, oracle port only) and prints one JSON line
    with the keys the driver reads."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--nodes",
                        "20000", "--edges", "200000", "--steps", "2", "--warmup", "1"],
                       capture_output=True, text=True, timeout=300, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step",
              "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in line, k
    assert line["impl"] == "reference" and line["value"] > 0 and line["cpu_baseline"]["kind"] == "port"
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["cpu_baseline"]["cores"] >= 1
    # non-zero ranks of a torchrun launch exit 0 without work
    r2 = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference"],
                        capture_output=True, text=True, timeout=120, env=dict(os.environ, RANK="1", CUDA_VISIBLE_DEVICES=""))
    assert r2.returncode == 0 and r2.stdout.strip() == ""


def test_bigraph_host_mode():
    """BiGraph in numpy mode: indexes come from the host build (twin of the reference's Cython
    build_index), degrees / sorted_edges follow reference bigraph.py:594-681, message passing
    refuses to run until .tensor() (bigraph.py:1157,1181)."""
    import pgl_b200 as pgl
    edges = np.array([[0, 1], [2, 0], [2, 1], [1, 1], [3, 0]], np.int64)
    g = pgl.BiGraph(edges)
    assert not g.is_tensor() and int(g.src_num_nodes) == 4 and int(g.dst_num_nodes) == 2
    assert g.indegree().tolist() == [2, 3] and g.outdegree().tolist() == [1, 1, 2, 1]
    assert g.indegree([1]).tolist() == [3]
    src, dst, eid = g.sorted_edges("dst")
    assert dst.tolist() == [0, 0, 1, 1, 1] and eid.tolist() == [1, 4, 0, 2, 3]
    assert src.tolist() == [2, 3, 0, 2, 1]
    src, dst, eid = g.sorted_edges("src")
    assert src.tolist() == [0, 1, 2, 2, 3] and eid.tolist() == [0, 3, 1, 2, 4]
    assert g.src_nodes.tolist() == [0, 1, 2, 3] and g.dst_nodes.tolist() == [0, 1]
    with pytest.raises(ValueError):
        g.sorted_edges("both")
    with pytest.raises(ValueError):
        g.send(lambda s, d, e: {}, src_feat={})
    with pytest.raises(ValueError):
        g.recv(lambda m: m, {})
    g2 = pgl.BiGraph(edges, src_num_nodes=6, dst_num_nodes=5)
    assert len(g2.indegree()) == 5 and len(g2.outdegree()) == 6


def test_pgl_import_alias():
    """`import pgl` (SURVEY 7.2) resolves to pgl_b200: same module objects, sub-packages included."""
    import pgl
    import pgl_b200
    import pgl.nn as nn
    import pgl.nn.functional as GF
    import pgl.math as pm
    from pgl.utils import op as uop
    assert pgl.Graph is pgl_b200.Graph and pgl.BiGraph is pgl_b200.BiGraph
    assert nn.GCNConv is pgl_b200.nn.GCNConv and GF is pgl_b200.nn.functional
    assert pm.segment_sum is pgl_b200.math.segment_sum and uop is pgl_b200.utils.op


def test_bench_balanced_row_bounds():
    """bench.py's destination-row blocks: contiguous, cover every row, nearly equal in-edge counts (hubs included)."""
    import torch
    import bench
    rng = np.random.default_rng(9)
    indeg = rng.integers(0, 5, 10000)
    indeg[[17, 4000, 9000]] = [30000, 20000, 10000]       # hubs
    t = torch.from_numpy(indeg.astype(np.int64))
    for parts in (1, 2, 4, 8):
        b = bench.balanced_row_bounds(torch, t, parts)
        assert b[0] == 0 and b[-1] == 10000 and len(b) == parts + 1 and all(b[i] <= b[i + 1] for i in range(parts))
        per = [int(indeg[b[i]:b[i + 1]].sum()) for i in range(parts)]
        assert sum(per) == int(indeg.sum())
        assert max(per) <= indeg.sum() / parts + indeg.max()   # within one (hub) row of the ideal share
    assert bench.block_bounds(10, 4, 0) == (0, 3) and bench.block_bounds(10, 4, 3) == (8, 10)
    assert bench.parse_grid(type("A", (), {"grid": ""})(), 8) == (8, 1)
    assert bench.parse_grid(type("A", (), {"grid": "2x4"})(), 8) == (2, 4)


def test_sampling_subgraph_matches_reference_relabelling():
    """pgl.sampling.subgraph (reference pgl/sampling/custom.py:23-83): edges renumbered exactly as the reference's
    compiled map_edges does with the {node: position} dict, features sliced by nodes / eid."""
    import pgl_b200 as pgl
    ref = np.load(REF_GK)   # inputs and the reference's own compiled map_edges on them
    edges, nodes = ref["subgraph_edges"], ref["subgraph_nodes"]
    rng = np.random.default_rng(0)
    n = 30
    g = pgl.Graph(edges=edges, num_nodes=n, node_feat={"x": rng.standard_normal((n, 3)).astype(np.float32)},
                  edge_feat={"w": rng.standard_normal((60, 2)).astype(np.float32)})
    eid = np.flatnonzero(np.isin(edges[:, 0], nodes) & np.isin(edges[:, 1], nodes))
    sg = pgl.sampling.subgraph(g, nodes, eid=eid)
    reindex = {int(v): i for i, v in enumerate(nodes)}
    want = np.array([[reindex[int(a)], reindex[int(b)]] for a, b in edges[eid]])
    assert (np.asarray(sg.edges) == want).all() and sg.num_nodes == 20
    assert (sg.node_feat["x"] == g.node_feat["x"][nodes]).all() and (sg.edge_feat["w"] == g.edge_feat["w"][eid]).all()
    assert np.array_equal(ref["subgraph_map_edges"], np.asarray(sg.edges))
    sg2 = pgl.sampling.subgraph(g, nodes, edges=edges[eid], with_edge_feat=False)
    assert (np.asarray(sg2.edges) == want).all() and not sg2.edge_feat
    with pytest.raises(ValueError):
        pgl.sampling.subgraph(g, nodes)
    with pytest.raises(ValueError):
        pgl.sampling.subgraph(g, nodes, edges=edges[eid])      # edge features need eid
