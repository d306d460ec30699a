"""Random walks and skip-gram pairs (mirror of reference pgl/sampling/walk.py:23-183 and
graph_kernel.skip_gram_gen_pair, pgl/graph_kernel.pyx:343-364) on the sm_100a kernels of csrc/walk.cu.

A numpy-mode graph walks on the host twin ``pglb_random_walk_host`` and returns the reference's list of lists; a
tensor-mode graph walks on the device and returns one int64 CUDA tensor ``[len(nodes), W]`` padded with -1.  Both
produce the same walks for the same seed: walk ``i`` is a pure function of ``(seed, i, graph, nodes[i], depth, p, q)``
(the RNG and the sampling rule are written out in include/pglb.h)."""
import ctypes
import math

import numpy as np
import torch

from .. import ops
from .._lib import WALK_NODE2VEC, WALK_NODE2VEC_PLUS, WALK_UNIFORM, check, lib

__all__ = ["random_walk", "node2vec_walk", "node2vec_walk_plus", "skip_gram_pairs"]

_U64 = 0xFFFFFFFFFFFFFFFF


def _seed(seed):
    """``None`` draws a 63-bit seed from numpy's global RNG, so ``np.random.seed`` makes walks reproducible."""
    if seed is None:
        return int(np.random.randint(0, np.iinfo(np.int64).max, dtype=np.int64))
    return int(seed) & _U64


def _check_pq(p, q):
    for name, v in (("p", p), ("q", q)):
        v = float(v)
        if not math.isfinite(v) or v <= 0:
            raise ValueError("node2vec %s must be finite and > 0, got %r" % (name, v))


def _walk(graph, nodes, steps, mode, p, q, seed):
    steps = max(int(steps), 0)
    W = steps + 1
    seed = _seed(seed)
    n_nodes = int(graph._n)
    indptr, cols = graph.successor_csr()
    p_ = lambda t: ctypes.c_void_p(t.data_ptr() if isinstance(t, torch.Tensor) else t.ctypes.data)  # noqa: E731
    if not graph.is_tensor():
        nodes = np.asarray(nodes.cpu().numpy() if isinstance(nodes, torch.Tensor) else nodes, np.int64).reshape(-1)
        n = int(nodes.shape[0])
        if n == 0:
            return []
        if nodes.min() < 0 or nodes.max() >= n_nodes:
            raise IndexError("walk start node outside [0, %d)" % n_nodes)
        out = np.empty((n, W), np.int64)
        check(lib.pglb_random_walk_host(p_(indptr), p_(cols), n_nodes, p_(nodes), n, steps, mode, float(p),
                                        float(q), seed, p_(out), W))
        lens = (out >= 0).sum(axis=1).tolist()
        return [row[:k] for row, k in zip(out.tolist(), lens)]
    dev = indptr.device
    if isinstance(nodes, torch.Tensor):
        ops.require_cuda(nodes)
        nodes = nodes.to(device=dev, dtype=torch.int64).reshape(-1).contiguous()
    else:
        nodes = torch.from_numpy(np.asarray(nodes, np.int64).reshape(-1).copy()).to(dev)
    n = int(nodes.shape[0])
    out = torch.empty((n, W), dtype=torch.int64, device=dev)
    if n == 0:
        return out
    lo, hi = torch.stack(torch.aminmax(nodes)).tolist()
    if lo < 0 or hi >= n_nodes:
        raise IndexError("walk start node outside [0, %d)" % n_nodes)
    with torch.cuda.device(dev):
        check(lib.pglb_random_walk(p_(indptr), p_(cols), n_nodes, p_(nodes), n, steps, mode, float(p), float(q), seed,
                                   p_(out), W, ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
    return out


def random_walk(graph, nodes, max_depth, seed=None):
    """Uniform random walks from every node of ``nodes`` (reference pgl/sampling/walk.py:23-64).

    A walk takes ``max_depth - 1`` steps, so it has at most ``max_depth`` nodes (``max_depth <= 0``: the start node
    alone), and ends early at the first node without successors.  Every step picks one of the current node's
    out-edges uniformly, so a neighbour reached by two parallel edges is twice as likely.

    Returns a list of lists of ints for a numpy-mode graph; for a tensor-mode graph an int64 CUDA tensor
    ``[len(nodes), max(max_depth, 1)]`` whose row ``i`` starts with ``nodes[i]`` and is padded with -1.
    ``seed``: walks are a pure function of it; ``None`` draws one from numpy's global RNG.
    A start node outside ``[0, num_nodes)`` raises IndexError."""
    return _walk(graph, nodes, int(max_depth) - 1, WALK_UNIFORM, 1.0, 1.0, seed)


def _node2vec(graph, nodes, max_depth, p, q, seed, mode):
    _check_pq(p, q)
    if p == 1.0 and q == 1.0:  # the reference's shortcut, one node shorter: kept because window sizes see it
        return random_walk(graph, nodes, max_depth, seed=seed)
    return _walk(graph, nodes, int(max_depth), mode, p, q, seed)


def node2vec_walk(graph, nodes, max_depth, p=1.0, q=1.0, seed=None):
    """node2vec walks (reference pgl/sampling/walk.py:67-122; Grover & Leskovec 2016).

    A walk takes ``max_depth`` steps, so it has at most ``max_depth + 1`` nodes; when ``p == q == 1`` this is
    ``random_walk(graph, nodes, max_depth)``, one node shorter, as in the reference.  The first step is uniform.
    After it every out-edge of the current node is weighted ``1/p`` if it leads back to the previous node, ``1`` if
    it leads to a successor of the previous node, ``1/q`` otherwise, and one edge is drawn with probability
    proportional to its weight (exactly; the reference's float32 loop can return None).  Return types, padding,
    ``seed`` and IndexError as ``random_walk``; ``p`` or ``q`` not finite or ``<= 0`` raises ValueError."""
    return _node2vec(graph, nodes, max_depth, p, q, seed, WALK_NODE2VEC)


def node2vec_walk_plus(graph, nodes, max_depth, p=1.0, q=1.0, seed=None):
    """node2vec walks whose weight-1 set is the union of the successors of every earlier node of the walk, not
    only of the previous one (reference pgl/sampling/walk.py:125-183).  Everything else as ``node2vec_walk``."""
    return _node2vec(graph, nodes, max_depth, p, q, seed, WALK_NODE2VEC_PLUS)


def skip_gram_pairs(walks, win_size=5, seed=None):
    """Skip-gram (center, context) pairs of a batch of walks: graph_kernel.skip_gram_gen_pair
    (reference pgl/graph_kernel.pyx:343-364) applied to every row of ``walks`` in one call.

    ``walks``: int64 CUDA tensor ``[n, W]`` as the tensor-mode walks return it (a row is a walk followed by -1).
    Position ``i`` of a walk draws a window ``r_i`` in ``[1, win_size]`` and pairs with every ``j`` in
    ``[i - r_i, i + r_i]`` inside the walk whose node differs from ``walk[i]``.  Returns ``(src, dst)`` int64 CUDA
    tensors ordered by walk, then ``i``, then ``j``; the windows are a pure function of ``(seed, walk row, i)``
    (include/pglb.h)."""
    ops.require_cuda(walks)
    if walks.dim() != 2:
        raise ValueError("walks must be [n, W], got shape %s" % (tuple(walks.shape),))
    win_size = int(win_size)
    if win_size < 1:
        raise ValueError("win_size must be >= 1, got %d" % win_size)
    walks = walks.to(torch.int64)
    if walks.stride(1) != 1:
        walks = walks.contiguous()
    n, W = int(walks.shape[0]), int(walks.shape[1])
    ldw = int(walks.stride(0)) if n > 1 else W
    dev = walks.device
    seed = _seed(seed)
    m = n * W
    offsets = torch.empty(m + 1, dtype=torch.int64, device=dev)
    need = ctypes.c_size_t(0)
    check(lib.pglb_skip_gram_ws(n, W, ctypes.byref(need)))
    ws = ops.workspace(dev, need.value)
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    p_ = lambda t: ctypes.c_void_p(t.data_ptr())  # noqa: E731
    with torch.cuda.device(dev):
        check(lib.pglb_skip_gram_count(p_(walks), n, W, ldw, win_size, seed, p_(offsets), p_(ws), ws.numel(),
                                       stream))
    total = int(offsets[m].item())
    src = torch.empty(total, dtype=torch.int64, device=dev)
    dst = torch.empty(total, dtype=torch.int64, device=dev)
    if total > 0:
        with torch.cuda.device(dev):
            check(lib.pglb_skip_gram_fill(p_(walks), n, W, ldw, win_size, seed, p_(offsets), p_(src), p_(dst),
                                          p_(ws), ws.numel(), stream))
    return src, dst
