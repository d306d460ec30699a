"""Partition -> local-graph pipeline on the device (csrc/localgraph.cu, SURVEY.md section 8f rank 3): integer work,
so every comparison is bit-exact -- against the reference's own compiled Cython helpers (graph_kernel.map_nodes /
map_edges, their outputs stored in tests/golden), against numpy restatements, and against the torch-op plan the
CPU (gloo) tests of the host logic use."""
import os

import numpy as np
import pytest
import torch

from oracle import oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pgl():
    import pgl_b200
    return pgl_b200


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def test_map_nodes_and_edges_vs_reference_cython(pgl):
    from pgl_b200.utils import relabel
    # inputs and the reference's own compiled helpers on them (tests/golden/make_golden.py)
    ref = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_graph_kernel.npz"))
    old, nodes, edges, eid = (ref["localgraph_" + k] for k in ("old", "nodes", "edges", "eid"))
    reindex = {int(o): i for i, o in enumerate(old)}
    table = relabel.dense_table(reindex, size=5000, device="cuda")
    mn = relabel.map_nodes(dev(nodes), table).cpu().numpy()
    me = relabel.map_edges(dev(eid), dev(edges), table).cpu().numpy()
    assert mn.tolist() == [reindex[int(v)] for v in nodes]
    assert me.tolist() == [[reindex[int(a)], reindex[int(b)]] for a, b in edges[eid]]
    all_e = pgl.ops.map_edges(None, dev(edges), table).cpu().numpy()
    assert (all_e == relabel.map_edges(np.arange(4000), edges, reindex)).all()
    assert np.array_equal(ref["localgraph_map_nodes"], mn)
    assert np.array_equal(ref["localgraph_map_edges"], me)
    # ids outside the table: -1 (non-strict) / IndexError (strict), never a wild read
    bad_nodes = dev(np.array([1, 5000, -3, 7], dtype=np.int64))
    got = pgl.ops.map_nodes(bad_nodes, table, strict=False).cpu().numpy()
    assert got[1] == -1 and got[2] == -1
    with pytest.raises(IndexError):
        pgl.ops.map_nodes(bad_nodes, table)
    with pytest.raises(IndexError):
        pgl.ops.map_edges(dev(np.array([4000], dtype=np.int64)), dev(edges), table)
    # empty inputs
    assert pgl.ops.map_nodes(dev(np.zeros(0, np.int64)), table).numel() == 0
    assert pgl.ops.map_edges(dev(np.zeros(0, np.int64)), dev(edges), table).shape == (0, 2)


@pytest.mark.parametrize("n,k", [(10, 1), (1000, 4), (200000, 8), (50000, 64)])
def test_partition_relabel_is_the_stable_argsort(pgl, n, k):
    from pgl_b200.distributed.halo import relabel_by_partition
    rng = np.random.default_rng(402 + n)
    part = rng.integers(0, k, n).astype(np.int64)
    if k > 2:
        part[part == 1] = 0   # an empty part
    new_id, offsets = pgl.ops.partition_relabel(dev(part), k)
    want_id, want_off = relabel_by_partition(part, k)
    assert (new_id.cpu().numpy() == want_id).all()
    assert offsets.cpu().numpy().tolist() == want_off
    # convention of apps/GNNAutoScale/graph_partition.py:94-101: permutation = argsort(part), ids ascend inside a part
    perm = np.argsort(part, kind="stable")
    assert (new_id.cpu().numpy()[perm] == np.arange(n)).all()


def numpy_plan(edges, lo, hi, offsets):
    src, dst = edges[:, 0], edges[:, 1]
    eid = np.nonzero((dst >= lo) & (dst < hi))[0]
    s = src[eid]
    remote = (s < lo) | (s >= hi)
    halo = np.unique(s[remote])
    col = np.where(remote, np.searchsorted(halo, s) + (hi - lo), s - lo)
    recv = [int(((halo >= offsets[p]) & (halo < offsets[p + 1])).sum()) for p in range(len(offsets) - 1)]
    return eid, dst[eid] - lo, col, halo, recv


@pytest.mark.parametrize("n,e,k", [(3000, 40000, 4), (100000, 1500000, 8), (64, 10, 3)])
def test_halo_plan_kernels_vs_numpy_and_torch_ops(pgl, n, e, k):
    from pgl_b200.distributed.halo import HaloPlan, block_offsets
    edges = O.chung_lu_edges(n, e, exponent=0.8, seed=411 + n)
    ed = dev(edges)
    offsets = block_offsets(n, k)
    for r in range(k):
        lo, hi = offsets[r], offsets[r + 1]
        eid, dl, cl, halo, recv = pgl.ops.halo_plan(ed, n, lo, hi, offsets)
        w_eid, w_dl, w_cl, w_halo, w_recv = numpy_plan(edges, lo, hi, offsets)
        assert (eid.cpu().numpy() == w_eid).all()
        assert (dl.cpu().numpy() == w_dl).all()
        assert (cl.cpu().numpy() == w_cl).all()
        assert (halo.cpu().numpy() == w_halo).all()
        assert recv.cpu().numpy().tolist() == w_recv and w_recv[r] == 0
    # the class, world 1 (no collective): kernels == the torch-op construction of the CPU tests
    a = HaloPlan.build(ed, n, [0, n], 0, 1)
    b = HaloPlan.build(ed, n, [0, n], 0, 1, force_torch=True)
    for name in ("eid", "dst_local", "col_local", "halo_ids"):
        assert torch.equal(getattr(a, name), getattr(b, name)), name
    assert a.n_halo == 0 and a.recv_counts == b.recv_counts


def test_halo_plan_edge_cases(pgl):
    n = 100
    offsets = [0, 50, 50, 100]   # an empty part in the middle
    edges = np.array([[0, 60], [99, 1], [70, 2], [70, 3], [10, 4], [3, 3]], dtype=np.int64)
    ed = dev(edges)
    eid, dl, cl, halo, recv = pgl.ops.halo_plan(ed, n, 0, 50, offsets)
    assert eid.tolist() == [1, 2, 3, 4, 5] and dl.tolist() == [1, 2, 3, 4, 3]
    assert halo.tolist() == [70, 99] and cl.tolist() == [51, 50, 50, 10, 3] and recv.tolist() == [0, 0, 2]
    eid, dl, cl, halo, recv = pgl.ops.halo_plan(ed, n, 50, 50, offsets)   # owns nothing
    assert eid.numel() == 0 and halo.numel() == 0 and recv.tolist() == [0, 0, 0]
    eid, dl, cl, halo, recv = pgl.ops.halo_plan(dev(np.zeros((0, 2), np.int64)), n, 0, 50, offsets)   # no edges
    assert eid.numel() == 0 and halo.numel() == 0
    with pytest.raises(IndexError):
        pgl.ops.halo_plan(dev(np.array([[0, 100]], dtype=np.int64)), n, 0, 50, offsets)


def test_partition_to_local_aggregation_matches_the_global_result(pgl):
    """part -> relabel -> per-rank local graph -> aggregation over [own rows | halo rows] == the owned rows of the
    global aggregation (oracle), for every rank of a 4-way partition, on one GPU."""
    n, e, d, k = 6000, 90000, 32, 4
    edges = O.chung_lu_edges(n, e, exponent=0.8, seed=421)
    rng = np.random.default_rng(422)
    x = rng.standard_normal((n, d)).astype(np.float32)
    part = rng.integers(0, k, n).astype(np.int64)
    want = O.send_u_recv(x, edges[:, 0], edges[:, 1], "sum")
    new_id, off_t = pgl.ops.partition_relabel(dev(part), k)
    offsets = off_t.tolist()
    e2 = pgl.ops.map_edges(None, dev(edges), new_id)
    x2 = torch.empty(n, d, device="cuda")
    x2[new_id] = dev(x)            # row new_id[i] of the relabelled matrix = row i of the original
    inv = torch.empty_like(new_id)
    inv[new_id] = torch.arange(n, device="cuda")
    for r in range(k):
        lo, hi = offsets[r], offsets[r + 1]
        eid, dl, cl, halo, recv = pgl.ops.halo_plan(e2, n, lo, hi, offsets)
        x_ext = torch.cat([x2[lo:hi], x2[halo]], 0).contiguous()
        from pgl_b200.utils.edge_index import EdgeIndex
        deg, sv, su, se, ip = pgl.ops.csr_build(dl, cl, hi - lo)
        csr = EdgeIndex.from_index(sorted_v=sv, sorted_u=su, sorted_eid=se, degree=deg, indptr=ip).csr()
        out = pgl.ops.aggregate_copy(x_ext, csr, hi - lo, "sum")
        orig_rows = inv[lo:hi].cpu().numpy()
        got = out.cpu().numpy()
        err = np.abs(got - want[orig_rows]).max() / max(np.abs(want).max(), 1e-12)
        assert err <= 1e-5, (r, err)
