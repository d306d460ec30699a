"""GPU tests of the random walks and skip-gram pairs (csrc/walk.cu, pgl_b200/sampling/walk.py): the device walks
equal the host twin's bit for bit (which tests/test_walk_host.py pins to the reference's rules and probabilities),
the tensor return type, and skip_gram_pairs against the oracle's restatement of skip_gram_gen_pair."""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import walk_oracle as W  # noqa: E402  (tests/walk_oracle.py)

pytestmark = pytest.mark.gpu

M64 = (1 << 64) - 1


def mix64(z):
    z = (z + 0x9e3779b97f4a7c15) & M64
    z = ((z ^ (z >> 30)) * 0xbf58476d1ce4e5b9) & M64
    z = ((z ^ (z >> 27)) * 0x94d049bb133111eb) & M64
    return z ^ (z >> 31)


@pytest.fixture(scope="module")
def graphs():
    import pgl_b200 as pgl
    n, e = 3000, 40000
    edges = O.chung_lu_edges(n, e, exponent=0.9, seed=901)                # hub rows and dead ends
    extra = np.array([[5, 5], [5, 5], [6, 9], [6, 9], [6, 9]], np.int64)   # self-loops, multi-edges
    edges = np.concatenate([edges, extra])
    n += 3                                                                  # isolated nodes
    g_np = pgl.Graph(edges=edges, num_nodes=n)
    g_t = pgl.Graph(edges=edges, num_nodes=n).tensor()
    return g_np, g_t, edges, n


def padded(walks, width):
    out = np.full((len(walks), width), -1, np.int64)
    for i, w in enumerate(walks):
        out[i, :len(w)] = w
    return out


def test_device_walks_equal_host_twin(graphs):
    from pgl_b200.sampling import node2vec_walk, node2vec_walk_plus, random_walk
    g_np, g_t, edges, n = graphs
    rng = np.random.default_rng(902)
    nodes = np.concatenate([np.arange(n), rng.integers(0, n, 500)]).astype(np.int64)
    nodes_d = torch.from_numpy(nodes).cuda()
    for depth in (0, 1, 2, 40):
        for fn, kind in ((random_walk, "random"), (node2vec_walk, "node2vec"), (node2vec_walk_plus, "plus")):
            for p, q in ((0.25, 0.25), (4.0, 0.5), (1e-3, 1.0), (1.0, 1.0)):
                if kind == "random" and (p, q) != (1.0, 1.0):
                    continue
                kw = {} if kind == "random" else {"p": p, "q": q}
                width = W.walk_length(kind, depth, p, q)
                dev = fn(g_t, nodes_d, depth, seed=77, **kw)
                assert dev.shape == (len(nodes), width) and dev.dtype == torch.int64
                host = padded(fn(g_np, nodes, depth, seed=77, **kw), width)
                assert np.array_equal(dev.cpu().numpy(), host), (kind, depth, p, q)


def test_device_walks_grid_stride(graphs):
    """More walks than one launch holds threads (the kernels loop over warps of walks)."""
    from pgl_b200.sampling import node2vec_walk, random_walk
    g_np, g_t, edges, n = graphs
    nodes = np.random.default_rng(903).integers(0, n, 400000).astype(np.int64)
    for fn, kw in ((random_walk, {}), (node2vec_walk, {"p": 0.25, "q": 4.0})):
        dev = fn(g_t, torch.from_numpy(nodes).cuda(), 12, seed=5, **kw)
        host = fn(g_np, nodes, 12, seed=5, **kw)
        assert np.array_equal(dev.cpu().numpy(), padded(host, dev.shape[1]))


def test_tensor_return_type_and_padding(graphs):
    from pgl_b200.sampling import node2vec_walk, random_walk
    g_np, g_t, edges, n = graphs
    succ_deg = np.bincount(edges[:, 0], minlength=n)
    dead = int(np.flatnonzero(succ_deg == 0)[0])
    nodes = [0, dead, 5, 5]
    outs = [random_walk(g_t, x, 6, seed=1) for x in (nodes, np.array(nodes), torch.tensor(nodes, device="cuda"))]
    for o in outs:
        assert o.is_cuda and o.dtype == torch.int64 and o.shape == (4, 6)
        assert torch.equal(o, outs[0])
    o = outs[0].cpu().numpy()
    assert (o[:, 0] == nodes).all() and (o[1, 1:] == -1).all()
    for row in o:                                                   # -1 only as a suffix
        k = int((row >= 0).sum())
        assert (row[:k] >= 0).all() and (row[k:] == -1).all()
    assert not np.array_equal(o[2], o[3]) or succ_deg[5] <= 1      # repeated start: its own walk
    e = node2vec_walk(g_t, [], 5, p=2.0, q=0.5)
    assert e.shape == (0, 6) and e.is_cuda


def sg_windows(seed, w, length, win):
    base = mix64(seed ^ mix64(w))
    return [1 + ((mix64((base + i) & M64) * win) >> 64) for i in range(length)]


def test_skip_gram_pairs_vs_oracle(graphs):
    from pgl_b200.sampling import node2vec_walk, skip_gram_pairs
    g_np, g_t, edges, n = graphs
    walks = node2vec_walk(g_t, torch.arange(0, n, 7, device="cuda"), 9, p=0.5, q=2.0, seed=3).cpu().numpy()
    crafted = np.array([[1, 2, 1, 2, 3, -1, -1, -1, -1, -1],
                        [5, 5, 5, -1, -1, -1, -1, -1, -1, -1],
                        [4, -1, -1, -1, -1, -1, -1, -1, -1, -1],
                        [-1] * 10,
                        [8, 9, 8, 9, 8, 9, 8, 9, 8, 9]], np.int64)
    for arr in (walks, crafted):
        for win, seed in ((1, 2), (5, 11), (10, 0xABCDEF)):
            t = torch.from_numpy(arr).cuda()
            src, dst = skip_gram_pairs(t, win_size=win, seed=seed)
            ws, wd = [], []
            for w, row in enumerate(arr):
                walk = row[row >= 0] if (row >= 0).all() else row[:int(np.argmax(row < 0))]
                s, d = W.skip_gram_gen_pair(walk, sg_windows(seed, w, len(walk), win))
                ws.append(s)
                wd.append(d)
            assert np.array_equal(src.cpu().numpy(), np.concatenate(ws)), (win, seed)
            assert np.array_equal(dst.cpu().numpy(), np.concatenate(wd)), (win, seed)
    # a strided view is read in place
    t = torch.from_numpy(crafted).cuda()
    a = skip_gram_pairs(t[:, :5], win_size=3, seed=4)
    b = skip_gram_pairs(t[:, :5].contiguous(), win_size=3, seed=4)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


def test_import_pgl_alias_on_tensor_graph(graphs):
    import pgl
    g_np, g_t, edges, n = graphs
    w = pgl.sampling.node2vec_walk(g_t, [0, 1, 2], 5, p=0.25, q=0.25, seed=9)
    assert w.shape == (3, 6) and w.is_cuda
    with pytest.raises(ValueError):
        g_t.successor([0])                                          # still numpy-mode only


def test_out_of_range_start_raises_before_launch(graphs):
    import pgl_b200 as pgl
    from pgl_b200.sampling import node2vec_walk, random_walk
    g_np, g_t, edges, n = graphs
    g_t.successor_csr()
    torch.cuda.synchronize()
    before = pgl.ops.launch_count()
    with pytest.raises(IndexError):
        random_walk(g_t, torch.tensor([0, n], device="cuda"), 5)
    with pytest.raises(IndexError):
        node2vec_walk(g_t, [-1], 5, p=2.0, q=2.0)
    assert pgl.ops.launch_count() == before
