"""Generate the committed golden fixtures under tests/golden/.

Run in the build container (where /root/reference exists):  python tests/golden/make_golden.py

Two kinds of fixture:
1. ``kat.json`` -- the reference's own known-answer tests for the send/recv path,
   transcribed by hand from /root/reference/tests (file:line cited per entry).  These
   are inputs + expected outputs; no reference code is executed for them.
2. ``ref_build_index.npz`` / ``ref_metis.npz`` -- outputs of the REFERENCE's compiled
   ``pgl.graph_kernel`` (built by oracle/build.py into oracle/_ref/) on seeded inputs:
   ``build_index`` (pgl/graph_kernel.pyx:59-88) and ``metis_partition``
   (pgl/graph_kernel.pyx:434-472, K-way, as pgl/partition.py:83-90 calls it).
3. ``ref_graph_kernel.npz`` -- outputs of the same compiled module for the seeded inputs the
   relabelling and index tests draw (``map_nodes`` / ``map_edges`` / ``build_index``), plus a fixed
   set of small edge lists (empty, one node, duplicates, self loops, ids beyond the largest one)
   with their ``build_index`` results, so those tests compare with the reference everywhere.
   ``python tests/golden/make_golden.py graph_kernel`` rewrites only this file.
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import build as obuild  # noqa: E402


def kats():
    k = {}
    nfeat5 = [[1, 2, 3, 4], [2, 3, 4, 5], [3, 4, 5, 6], [4, 5, 6, 7], [5, 6, 7, 8]]
    edges5 = [[0, 1], [1, 2], [3, 4], [4, 1], [1, 0]]
    k["send_recv_sum"] = {
        "cite": "tests/test_graph.py:337-357",
        "num_nodes": 5, "edges": edges5, "nfeat": nfeat5,
        "ground": [[2, 3, 4, 5], [6, 8, 10, 12], [2, 3, 4, 5], [0, 0, 0, 0], [4, 5, 6, 7]],
    }
    k["send_and_recv"] = {
        "cite": "tests/test_graph.py:359-410",
        "num_nodes": 5, "edges": edges5, "nfeat": nfeat5,
        "msg_ground": [[1, 2, 3, 4], [2, 3, 4, 5], [4, 5, 6, 7], [5, 6, 7, 8], [2, 3, 4, 5]],
        "recv_ground": [[2, 3, 4, 5], [6, 8, 10, 12], [2, 3, 4, 5], [0, 0, 0, 0], [4, 5, 6, 7]],
    }
    k["send_func"] = {
        "cite": "tests/test_graph.py:292-335",
        "num_nodes": 4, "edges": [[0, 1], [1, 2], [2, 3]],
        "nfeat": [[0], [1], [2], [3]], "efeat": [[0], [1], [2]],
        "target_src": [[0], [1], [2]], "target_dst": [[1], [2], [3]], "target_edge": [[0], [1], [2]],
    }
    k["degree"] = {
        "cite": "tests/test_graph.py:101-140",
        "num_nodes": 5, "edges": [[0, 1], [1, 2], [3, 4]],
        "indegree": [0, 1, 1, 0, 1], "outdegree": [1, 1, 0, 1, 0], "subset": [1, 2, 3],
    }
    k["segment_softmax"] = {
        "cite": "tests/test_math.py:32-49",
        "data": [[1, 2, 3], [3, 2, 1], [4, 5, 6]], "seg_ids": [0, 0, 1],
        "ground": [[0.11920292, 0.5, 0.880797], [0.880797, 0.5, 0.11920292], [1, 1, 1]],
    }
    k["segment_softmax_overflow"] = {
        "cite": "tests/test_math.py:51-66",
        "data": [[1, 2, 0.003], [3, 2, 10000000000], [4, 5, 6]], "seg_ids": [0, 0, 1],
        "ground": [[0.11920292, 0.5, 0], [0.880797, 0.5, 1], [1, 1, 1]],
    }
    k["edge_softmax"] = {
        "cite": "tests/test_graph_op.py:56-68 (exact float equality asserted)",
        "num_nodes": 3, "edges": [[0, 0], [0, 1], [0, 2], [1, 1], [1, 2], [2, 2]],
        "logits": [1, 1, 1, 1, 1, 1],
        "dst": ["1", "1/2", "1/3", "1/2", "1/3", "1/3"],
        "src": ["1/3", "1/3", "1/3", "1/2", "1/2", "1"],
    }
    k["send_ue_recv_add_sum"] = {
        "cite": "tests/test_dist_graph.py:115-137",
        "num_nodes": 5, "edges": edges5, "nfeat": nfeat5, "efeat": [1, 1, 1, 1, 1],
        "ground": [[3, 4, 5, 6], [8, 10, 12, 14], [3, 4, 5, 6], [0, 0, 0, 0], [5, 6, 7, 8]],
    }
    k["segment_docstrings"] = {
        "cite": "pgl/math.py:72-75,105-110,137-142,170-175",
        "data": [[1, 2, 3], [3, 2, 1], [4, 5, 6]], "seg_ids": [0, 0, 1],
        "sum": [[4, 4, 4], [4, 5, 6]], "mean": [[2, 2, 2], [4, 5, 6]],
        "min": [[1, 2, 1], [4, 5, 6]], "max": [[3, 2, 3], [4, 5, 6]],
    }
    k["bigraph_send_recv_sum"] = {
        "cite": "tests/test_bigraph.py:390-412 (rectangular: 5 src x 4 dst)",
        "src_num_nodes": 5, "dst_num_nodes": 4,
        "edges": [[0, 1], [1, 2], [3, 3], [4, 1], [1, 0]], "src_nfeat": nfeat5,
        "ground": [[2, 3, 4, 5], [6, 8, 10, 12], [2, 3, 4, 5], [4, 5, 6, 7]],
    }
    k["bigraph_recv_src"] = {
        "cite": "tests/test_bigraph.py:414-507 (the only recv_mode='src' KAT in the tree)",
        "src_num_nodes": 5, "dst_num_nodes": 4,
        "edges": [[0, 1], [1, 2], [3, 3], [4, 1], [1, 0]],
        "dst_nfeat": [[2, 3, 4, 5], [3, 4, 5, 6], [4, 5, 6, 7], [5, 6, 7, 8]],
        "dst_msg_ground": [[3, 4, 5, 6], [4, 5, 6, 7], [5, 6, 7, 8], [3, 4, 5, 6], [2, 3, 4, 5]],
        "dst_recv": [[3, 4, 5, 6], [6, 8, 10, 12], [0, 0, 0, 0], [5, 6, 7, 8], [3, 4, 5, 6]],
    }
    k["readme_toy"] = {
        "cite": "README.md:64-92 (BASELINE config 1; feature = randn(5,100) seed 0)",
        "num_nodes": 5, "edges": [[0, 1], [1, 2], [3, 4]], "dim": 100, "seed": 0,
        "copy_rows": {"1": 0, "2": 1, "4": 3}, "zero_rows": [0, 3],
    }
    k["ref_probe_build_index"] = {
        "cite": "SURVEY.md section 8c: reference build_index run on the test_graph.py 5-edge graph",
        "num_nodes": 5, "edges": edges5,
        "indegree": [1, 2, 1, 0, 1], "indptr": [0, 1, 3, 4, 4, 5], "eid": [4, 0, 3, 1, 2],
    }
    return k


def power_law_edges(n, e, seed):
    rng = np.random.default_rng(seed)
    w = np.power(np.arange(1, n + 1, dtype=np.float64), -0.8)
    cdf = np.cumsum(w) / np.sum(w)
    s = np.minimum(np.searchsorted(cdf, rng.random(e)), n - 1)
    d = np.minimum(np.searchsorted(cdf, rng.random(e)), n - 1)
    p = rng.permutation(n)
    return p[s].astype(np.int64), p[d].astype(np.int64)


BUILD_INDEX_FIELDS = ("degree", "sorted_v", "sorted_u", "sorted_eid", "indptr")
INDEX_CASES = 80


def index_cases(seed=17):
    """Small (u, v, num_nodes) edge lists shaped like tests/test_property_index.py draws them."""
    rng = np.random.default_rng(seed)
    cases = [(np.zeros(0, np.int64), np.zeros(0, np.int64), 1), (np.zeros(0, np.int64), np.zeros(0, np.int64), 6),
             (np.zeros(3, np.int64), np.zeros(3, np.int64), 1)]
    while len(cases) < INDEX_CASES:
        n = int(rng.integers(1, 41))
        e = int(rng.integers(0, 121))
        u = rng.integers(0, n, e).astype(np.int64)
        v = rng.integers(0, n, e).astype(np.int64)
        cases.append((u, v, n + int(rng.integers(0, 6))))
    return cases


def graph_kernel_fixtures(gk):
    """Every input is stored next to the reference's output on it: the tests read both."""
    out = {}
    # map_nodes / map_edges with the {old id: position} dict: tests/test_host_logic.py ("relabel") and
    # tests/test_gpu_localgraph.py ("localgraph")
    for name, seed, ids, n_old, n_nodes, n_edges, n_eid in (("relabel", 3, 50, 20, 30, 40, 15),
                                                            ("localgraph", 401, 5000, 2000, 3000, 4000, 1500)):
        rng = np.random.default_rng(seed)
        old = rng.permutation(ids)[:n_old].astype(np.int64)
        nodes = rng.choice(old, n_nodes)
        edges = rng.choice(old, (n_edges, 2)).astype(np.int64)
        eid = rng.integers(0, n_edges, n_eid).astype(np.int64)
        reindex = {int(o): i for i, o in enumerate(old)}
        out.update({name + "_old": old, name + "_nodes": nodes, name + "_edges": edges, name + "_eid": eid,
                    name + "_map_nodes": np.asarray(gk.map_nodes(nodes, reindex)),
                    name + "_map_edges": np.asarray(gk.map_edges(eid, edges, reindex))})
    # pgl.sampling.subgraph's renumbering of the edges inside `nodes` (tests/test_host_logic.py)
    rng = np.random.default_rng(0)
    edges = rng.integers(0, 30, (60, 2)).astype(np.int64)
    nodes = rng.permutation(30)[:20].astype(np.int64)
    eid = np.flatnonzero(np.isin(edges[:, 0], nodes) & np.isin(edges[:, 1], nodes))
    reindex = {int(v): i for i, v in enumerate(nodes)}
    out["subgraph_edges"], out["subgraph_nodes"] = edges, nodes
    out["subgraph_map_edges"] = np.asarray(gk.map_edges(np.arange(len(eid), dtype=np.int64), edges[eid], reindex))

    def index_case(name, u, v, n):
        out[name + "_u"], out[name + "_v"], out[name + "_n"] = u, v, np.int64(n)
        for f, a in zip(BUILD_INDEX_FIELDS, gk.build_index(u, v, n)):
            out[name + "_" + f] = np.asarray(a)

    # build_index: three seeded edge lists (tests/test_oracle_golden.py) and the small cases
    # (tests/test_property_index.py)
    rng = np.random.default_rng(5)
    for i, (n, e) in enumerate(((1, 0), (3, 10), (500, 5000))):
        index_case("seeded%d" % i, rng.integers(0, n, e).astype(np.int64), rng.integers(0, n, e).astype(np.int64), n)
    for i, (u, v, n) in enumerate(index_cases()):
        index_case("case%02d" % i, u, v, n)
    np.savez_compressed(os.path.join(HERE, "ref_graph_kernel.npz"), **out)


def main():
    gk = obuild.load_ref_graph_kernel()
    if gk is None:
        obuild.build_ref()
        gk = obuild.load_ref_graph_kernel()
    graph_kernel_fixtures(gk)
    if sys.argv[1:] == ["graph_kernel"]:
        return
    with open(os.path.join(HERE, "kat.json"), "w") as f:
        json.dump(kats(), f, indent=1)

    out = {}
    cases = [("tiny", 7, 0, 1), ("uniform", 50, 400, 2), ("powerlaw", 1000, 20000, 3),
             ("gaps", 64, 100, 4)]
    for name, n, e, seed in cases:
        if name == "uniform" or name == "gaps":
            rng = np.random.default_rng(seed)
            u = rng.integers(0, n if name == "uniform" else n // 4, e).astype(np.int64)
            v = rng.integers(0, n, e).astype(np.int64)
        elif name == "tiny":
            u = np.zeros(0, np.int64)
            v = np.zeros(0, np.int64)
        else:
            v, u = power_law_edges(n, e, seed)
        deg, sv, su, se, ip = gk.build_index(u, v, n)
        out[name + "_n"] = np.int64(n)
        out[name + "_u"] = u
        out[name + "_v"] = v
        out[name + "_degree"] = deg
        out[name + "_sorted_v"] = sv
        out[name + "_sorted_u"] = su
        out[name + "_sorted_eid"] = se
        out[name + "_indptr"] = ip
    np.savez_compressed(os.path.join(HERE, "ref_build_index.npz"), **out)

    # METIS: symmetric random graph, 200 nodes, as pgl/partition.py:66-90 feeds it
    rng = np.random.default_rng(11)
    n = 200
    a = rng.integers(0, n, 900)
    b = rng.integers(0, n, 900)
    keep = a != b
    a, b = a[keep], b[keep]
    und = np.unique(np.stack([np.minimum(a, b), np.maximum(a, b)], 1), axis=0)
    edges = np.concatenate([und, und[:, ::-1]], 0).astype(np.int64)
    deg, sv, su, se, ip = gk.build_index(edges[:, 1].copy(), edges[:, 0].copy(), n)
    m = {"n": np.int64(n), "edges": edges, "indptr": ip, "sorted_v": sv}
    for nparts in (2, 8):
        m["part_%d" % nparts] = gk.metis_partition(n, ip, sv, nparts=nparts, recursive=False)
    nw = (rng.random(n) * 5).astype(np.float32)
    nws = ((nw - nw.min()) / (nw.max() - nw.min() + 1e-5) * 1000).astype("int64") + 1
    m["node_weights_raw"] = nw
    m["node_weights_scaled"] = nws
    m["part_8_nw"] = gk.metis_partition(n, ip, sv, nparts=8, node_weights=nws, recursive=False)
    np.savez_compressed(os.path.join(HERE, "ref_metis.npz"), **m)
    print("golden fixtures written to", HERE)


if __name__ == "__main__":
    main()
