"""Random walks on the host (no GPU): the oracle's node2vec probabilities against the reference's compiled sampler
(tests/golden/ref_node2vec.npz), the host twin pglb_random_walk_host (what a numpy-mode graph walks on, and the
device kernels' reference) against the reference's length rules and the oracle's transition probabilities, a Python
restatement of the RNG and sampling scheme documented in include/pglb.h, and argument checks of the C-ABI."""
import ctypes
import math
import os
import sys
from collections import Counter

import numpy as np
import pytest

from oracle import oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import walk_oracle as W  # noqa: E402  (tests/walk_oracle.py)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
M64 = (1 << 64) - 1
MAX_REJECT, WORDS_PER_STEP = 32, 128


@pytest.fixture(scope="module")
def pgl():
    import pgl_b200
    return pgl_b200


def chi2(counts, probs):
    counts, probs = np.asarray(counts, np.float64), np.asarray(probs, np.float64)
    exp = probs * counts.sum()
    assert (counts[exp == 0] == 0).all(), (counts, probs)
    k = exp > 0
    return float(((counts[k] - exp[k]) ** 2 / exp[k]).sum()), int(k.sum()) - 1


def chi2_ok(counts, probs):
    # fixed inputs and seeds: deterministic.  The bound is the 1e-6 upper tail for dof <= 10 (about 40).
    stat, dof = chi2(counts, probs)
    return stat < 40, (stat, dof)


# ---- 1. the oracle against the reference's compiled node2vec_sample / node2vec_plus_sample ----------------------

def test_oracle_probs_match_reference_golden():
    z = np.load(os.path.join(GOLDEN, "ref_node2vec.npz"))
    assert int(z["draws"]) >= 100000
    for c in range(int(z["num_cases"])):
        succ, seen, prev = z["c%d_succ" % c], z["c%d_prev_succ" % c], int(z["c%d_prev" % c])
        p, q = float(z["c%d_p" % c]), float(z["c%d_q" % c])
        vals, probs = W.node2vec_value_probs(succ, seen, prev, p, q)
        assert (vals == z["c%d_values" % c]).all()
        for name in ("plain", "plus"):
            counts = z["c%d_%s_counts" % (c, name)]
            assert counts[-1] == 0  # the reference never fell through to None on these cases
            ok, info = chi2_ok(counts[:-1], probs)
            assert ok, (c, name, info)
        want_seen = np.unique(np.concatenate([seen, succ]))
        assert (z["c%d_plus_next_seen" % c] == want_seen).all()


def test_oracle_walk_length_rules():
    assert W.walk_length("random", 5) == 5 and W.walk_length("random", 0) == 1 and W.walk_length("random", -3) == 1
    assert W.walk_length("node2vec", 5, 0.5, 2) == 6 and W.walk_length("node2vec", 5, 1.0, 1.0) == 5
    assert W.walk_length("plus", 0, 2, 2) == 1
    src, dst = W.skip_gram_gen_pair([7, 8, 7, 9], [1, 2, 1, 3])
    assert list(zip(src.tolist(), dst.tolist())) == [(7, 8), (8, 7), (8, 7), (8, 9), (7, 8), (7, 9), (9, 7), (9, 8), (9, 7)]


# ---- 2. host twin: the reference's walk contract -----------------------------------------------------------------

def small_graph(seed=5, n=60, e=400):
    edges = O.chung_lu_edges(n, e, exponent=0.9, seed=seed)
    edges = np.concatenate([edges, [[3, 3], [3, 3], [4, 7], [4, 7]]])        # self-loops and parallel edges
    return edges, n + 4                                                         # 4 isolated nodes at the end


def successors(edges, n):
    s = [[] for _ in range(n)]
    for u, v in edges.tolist():
        s[u].append(v)
    return s


def check_walks(walks, nodes, edges, n, width):
    have = set(map(tuple, edges.tolist()))
    succ = successors(edges, n)
    assert len(walks) == len(nodes)
    for w, v in zip(walks, nodes):
        assert w[0] == v and 1 <= len(w) <= width
        assert all((a, b) in have for a, b in zip(w[:-1], w[1:]))
        if len(w) < width:
            assert len(succ[w[-1]]) == 0                                      # ended early only at a dead end


def test_host_walks_follow_edges_and_length_rules(pgl):
    from pgl_b200.sampling import node2vec_walk, node2vec_walk_plus, random_walk
    edges, n = small_graph()
    g = pgl.Graph(edges=edges, num_nodes=n)
    nodes = list(range(n)) + [3, 3, n - 1]                                    # repeated and isolated starts
    for d in (0, 1, 2, 7):
        check_walks(random_walk(g, nodes, d, seed=1), nodes, edges, n, W.walk_length("random", d))
        for fn, kind in ((node2vec_walk, "node2vec"), (node2vec_walk_plus, "plus")):
            for p, q in ((0.25, 4.0), (4.0, 0.25), (1e-3, 1.0)):
                w = fn(g, nodes, d, p=p, q=q, seed=2)
                check_walks(w, nodes, edges, n, W.walk_length(kind, d, p, q))
            # p == q == 1 is random_walk(max_depth), one node shorter
            assert fn(g, nodes, d, p=1.0, q=1.0, seed=3) == random_walk(g, nodes, d, seed=3)
    assert random_walk(g, [n - 1, n - 2], 5, seed=0) == [[n - 1], [n - 2]]
    assert random_walk(g, [], 5, seed=0) == [] and node2vec_walk(g, np.zeros(0, np.int64), 5, 2, 2) == []
    w = random_walk(g, [0] * 50, 10, seed=4)                                  # a repeated start gives other walks
    assert len(set(map(tuple, w))) > 40


def test_host_walks_seeding(pgl):
    from pgl_b200.sampling import node2vec_walk, random_walk
    edges, n = small_graph()
    g = pgl.Graph(edges=edges, num_nodes=n)
    nodes = np.arange(n)
    a = node2vec_walk(g, nodes, 10, p=0.5, q=2.0, seed=11)
    assert a == node2vec_walk(g, nodes, 10, p=0.5, q=2.0, seed=11)
    assert a != node2vec_walk(g, nodes, 10, p=0.5, q=2.0, seed=12)
    # walk i depends on (seed, i, nodes[i]) only: a prefix of the batch walks the same
    assert node2vec_walk(g, nodes[:5], 10, p=0.5, q=2.0, seed=11) == a[:5]
    np.random.seed(123)
    b = random_walk(g, nodes, 8)
    np.random.seed(123)
    assert random_walk(g, nodes, 8) == b
    assert random_walk(g, nodes, 8) != b


def test_host_walks_argument_errors(pgl):
    from pgl_b200.sampling import node2vec_walk, node2vec_walk_plus, random_walk
    edges, n = small_graph()
    g = pgl.Graph(edges=edges, num_nodes=n)
    with pytest.raises(IndexError):
        random_walk(g, [0, n], 3)
    with pytest.raises(IndexError):
        node2vec_walk(g, [-1], 3, p=2.0)
    for p, q in ((0.0, 1.0), (1.0, -2.0), (float("inf"), 1.0), (1.0, float("nan"))):
        for fn in (node2vec_walk, node2vec_walk_plus):
            with pytest.raises(ValueError):
                fn(g, [0], 3, p=p, q=q)


def test_successor_csr_rows_sorted(pgl):
    edges, n = small_graph()
    g = pgl.Graph(edges=edges, num_nodes=n)
    indptr, cols = g.successor_csr()
    assert g.successor_csr()[1] is cols                                       # cached
    assert (indptr == g.adj_src_index._indptr).all()
    succ = successors(edges, n)
    for v in range(n):
        assert cols[indptr[v]:indptr[v + 1]].tolist() == sorted(succ[v])


# ---- 3. host twin transition frequencies against the oracle's exact probabilities -------------------------------

def context_graph(prev_in_row=True):
    """Walks from node 0 reach (0, 1, 2) with probability 1/2; from there the next draw has prev = 1, cur = 2,
    node2vec's seen set succ(1) = {2} and node2vec+'s succ(0) | succ(1) = {1, 2, 5}.  Node 2's row has duplicates,
    a self-loop, the previous node (unless prev_in_row is False), and node 3, which nothing before it reaches."""
    succ = {0: [1, 5], 1: [2], 2: [0, 1, 2, 3, 5, 5, 6], 3: [2], 5: [0], 6: [2]}
    if not prev_in_row:
        succ[2].remove(1)
    edges = np.array([(u, v) for u, vs in succ.items() for v in vs], np.int64)
    return edges, 7, succ


# (1e-3, 1, False): the envelope is 1/p = 1000 and no candidate reaches it, so about 97% of these steps reject 32
# draws and take the inverse-CDF fallback
@pytest.mark.parametrize("p,q,prev_in_row", [(0.25, 4.0, True), (4.0, 0.25, True), (1e-3, 1.0, True),
                                             (1.0, 1e-3, True), (1e-3, 1.0, False)])
def test_host_transition_frequencies(pgl, p, q, prev_in_row):
    from pgl_b200.sampling import node2vec_walk, node2vec_walk_plus, random_walk
    edges, n, succ = context_graph(prev_in_row)
    g = pgl.Graph(edges=edges, num_nodes=n)
    walks_n = 60000
    vals = np.array(sorted(set(succ[2])))
    # uniform: the step from node 2, every slot equally likely
    w = random_walk(g, [2] * walks_n, 2, seed=7)
    cnt = Counter(x[1] for x in w)
    ok, info = chi2_ok([cnt[v] for v in vals], W.node2vec_value_probs(succ[2], [], -1, 1.0, 1.0)[1])
    assert ok, info
    for fn, seen in ((node2vec_walk, succ[1]), (node2vec_walk_plus, sorted(set(succ[0]) | set(succ[1])))):
        w = fn(g, [0] * walks_n, 3, p=p, q=q, seed=8)
        cnt = Counter(x[3] for x in w if x[:3] == [0, 1, 2])
        assert sum(cnt.values()) > walks_n // 3
        _, probs = W.node2vec_value_probs(succ[2], seen, 1, p, q)
        ok, info = chi2_ok([cnt[v] for v in vals], probs)
        assert ok, (fn.__name__, p, q, info)


# ---- 4. a restatement of the documented RNG and sampling scheme reproduces the host twin exactly -----------------

def mix64(z):
    z = (z + 0x9e3779b97f4a7c15) & M64
    z = ((z ^ (z >> 30)) * 0xbf58476d1ce4e5b9) & M64
    z = ((z ^ (z >> 27)) * 0x94d049bb133111eb) & M64
    return z ^ (z >> 31)


def thresholds(p, q):
    w = (1.0 / p, 1.0, 1.0 / q)
    m = max(w)
    return [max(1, int(math.floor(x / m * 4294967296.0))) for x in w]


def model_walk(succ_sorted, start, i, steps, mode, p, q, seed):
    """include/pglb.h, statement by statement, with set membership instead of the binary search."""
    T = thresholds(p, q) if mode else None
    wb = mix64(seed ^ mix64(i))
    word = lambda t, k: mix64((wb + WORDS_PER_STEP * t + k) & M64)  # noqa: E731
    walk = [start]
    for t in range(steps):
        row = succ_sorted[walk[-1]]
        d = len(row)
        if d == 0:
            break
        if mode == 0 or t == 0:
            walk.append(row[(word(t, 0) * d) >> 64])
            continue
        prev = walk[-2]
        seen = set(succ_sorted[prev]) if mode == 1 else set().union(*(succ_sorted[v] for v in walk[:-1]))
        thr = lambda x: T[0] if x == prev else (T[1] if x in seen else T[2])  # noqa: E731
        nxt = None
        for k in range(MAX_REJECT):
            x = row[(word(t, 2 * k) * d) >> 64]
            if (word(t, 2 * k + 1) >> 32) < thr(x):
                nxt = x
                break
        if nxt is None:
            ws = [thr(x) for x in row]
            target = (word(t, 2 * MAX_REJECT) * sum(ws)) >> 64
            nxt = row[int(np.searchsorted(np.cumsum(ws), target, "right"))]
        walk.append(nxt)
    return walk


def test_rng_model_reproduces_host_twin(pgl):
    from pgl_b200.sampling import node2vec_walk, node2vec_walk_plus, random_walk
    edges, n = small_graph(seed=9, n=40, e=300)
    g = pgl.Graph(edges=edges, num_nodes=n)
    succ_sorted = [sorted(s) for s in successors(edges, n)]
    nodes = list(range(n)) + [0, 0, 3]
    seed = 0xFEEDFACECAFEBEEF
    got = random_walk(g, nodes, 9, seed=seed)
    assert got == [model_walk(succ_sorted, v, i, 8, 0, 1, 1, seed) for i, v in enumerate(nodes)]
    for p, q in ((0.25, 4.0), (1e-3, 1.0), (3.0, 0.5)):
        for fn, mode in ((node2vec_walk, 1), (node2vec_walk_plus, 2)):
            got = fn(g, nodes, 8, p=p, q=q, seed=seed)
            want = [model_walk(succ_sorted, v, i, 8, mode, p, q, seed) for i, v in enumerate(nodes)]
            assert got == want, (fn.__name__, p, q)


# ---- 5. C-ABI argument checks (no device work) -------------------------------------------------------------------

def test_walk_abi_rejects_bad_arguments():
    from pgl_b200 import _lib
    lib = _lib.lib
    one = ctypes.c_void_p(16)   # non-NULL dummy: must never be dereferenced here
    EINVAL, ESHAPE, EWORKSPACE = -1, -2, -3
    # pglb_random_walk(indptr, cols, N, nodes, n, steps, mode, p, q, seed, out, ldo, stream)
    assert lib.pglb_random_walk(None, None, 5, None, 0, 3, 0, 1.0, 1.0, 1, None, 4, None) == 0
    assert lib.pglb_random_walk(one, one, 5, one, 3, 3, 7, 1.0, 1.0, 1, one, 4, None) == EINVAL
    assert b"mode" in lib.pglb_last_error()
    for p, q in ((0.0, 1.0), (1.0, -1.0), (float("inf"), 1.0), (float("nan"), 1.0)):
        assert lib.pglb_random_walk(one, one, 5, one, 3, 3, 1, p, q, 1, one, 4, None) == EINVAL
    assert lib.pglb_random_walk(one, one, 5, one, 3, 3, 2, 0.5, 2.0, 1, one, 3, None) == ESHAPE
    assert lib.pglb_random_walk(None, one, 5, one, 3, 3, 0, 1.0, 1.0, 1, one, 4, None) == EINVAL
    assert lib.pglb_random_walk(one, one, 5, one, -1, 3, 0, 1.0, 1.0, 1, one, 4, None) == EINVAL
    assert lib.pglb_random_walk(one, one, 5, one, 3, -1, 0, 1.0, 1.0, 1, one, 4, None) == EINVAL
    # host twin: an id outside [0, N) is refused before any step
    indptr = np.array([0, 1, 1], np.int64)
    cols = np.array([1], np.int64)
    nodes = np.array([0, 2], np.int64)
    out = np.zeros((2, 3), np.int64)
    ptr = lambda a: ctypes.c_void_p(a.ctypes.data)  # noqa: E731
    assert lib.pglb_random_walk_host(ptr(indptr), ptr(cols), 2, ptr(nodes), 2, 2, 0, 1.0, 1.0, 1, ptr(out), 3) == ESHAPE
    assert b"out of range" in lib.pglb_last_error()
    nodes[1] = 1
    assert lib.pglb_random_walk_host(ptr(indptr), ptr(cols), 2, ptr(nodes), 2, 2, 0, 1.0, 1.0, 1, ptr(out), 3) == 0
    assert out.tolist() == [[0, 1, -1], [1, -1, -1]]
    assert lib.pglb_random_walk_host(ptr(indptr), None, 2, ptr(nodes), 2, 2, 0, 1.0, 1.0, 1, ptr(out), 3) == EINVAL
    # skip-gram
    need = ctypes.c_size_t(0)
    assert lib.pglb_skip_gram_ws(10, 5, ctypes.byref(need)) == 0 and need.value >= 10 * 8
    assert lib.pglb_skip_gram_ws(-1, 5, ctypes.byref(need)) == EINVAL
    big = need.value
    assert lib.pglb_skip_gram_count(one, 10, 5, 5, 0, 1, one, one, big, None) == EINVAL
    assert b"win_size" in lib.pglb_last_error()
    assert lib.pglb_skip_gram_count(one, 10, 5, 4, 3, 1, one, one, big, None) == ESHAPE
    assert lib.pglb_skip_gram_count(one, 10, 5, 5, 3, 1, one, one, 8, None) == EWORKSPACE
    assert lib.pglb_skip_gram_count(one, 10, 5, 5, 3, 1, None, one, big, None) == EINVAL
    assert lib.pglb_skip_gram_fill(one, 10, 5, 5, 3, 1, None, one, one, one, big, None) == EINVAL
    assert lib.pglb_skip_gram_fill(None, 0, 5, 5, 3, 1, None, None, None, one, big, None) == 0
