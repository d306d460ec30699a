"""CPU restatement of the reference's random walks and skip-gram pairs (pgl/sampling/walk.py:23-183,
pgl/graph_kernel.pyx:142-224 node2vec_sample / node2vec_plus_sample, pgl/graph_kernel.pyx:343-364
skip_gram_gen_pair).  TEST INFRASTRUCTURE ONLY: tests/test_walk_host.py, tests/test_gpu_walk.py and the
reference-loop leg of scripts/bench_walk.py use it as the checker; pgl_b200 never imports it.

The exact node2vec probabilities are pinned to the reference's compiled sampler by
tests/golden/ref_node2vec.npz (written by tests/golden/make_walk_golden.py)."""
import numpy as np


def walk_length(kind, max_depth, p=1.0, q=1.0):
    """Most nodes a walk of the reference can have.  random_walk loops ``max_depth - 1`` times
    (walk.py:42); node2vec_walk / node2vec_walk_plus loop ``max_depth`` times (walk.py:94, 152), except that
    ``p == q == 1`` returns random_walk(max_depth) (walk.py:82-83, 140-141).  A walk also ends at the first
    node without successors (walk.py:44-53)."""
    if kind != "random" and not (p == 1.0 and q == 1.0):
        return max(int(max_depth), 0) + 1
    return max(int(max_depth) - 1, 0) + 1


def node2vec_probs(succ, seen, prev, p, q):
    """Exact probability of every candidate slot of node2vec_sample / node2vec_plus_sample
    (graph_kernel.pyx:142-224): slot j weighs 1/p when succ[j] == prev, 1 when succ[j] is in ``seen`` (the
    previous node's successors; for node2vec+ every earlier node's), 1/q otherwise; one slot per edge, so a
    duplicated successor collects the weight of each of its slots.  The reference draws with rand() and a
    float32 subtract-and-compare loop; this is the distribution that loop approximates."""
    seen = set(int(x) for x in seen)
    w = np.array([1.0 / p if int(x) == prev else (1.0 if int(x) in seen else 1.0 / q) for x in succ], np.float64)
    return w / w.sum()


def node2vec_value_probs(succ, seen, prev, p, q):
    """node2vec_probs summed per distinct successor: (values ascending, probabilities)."""
    succ = np.asarray(succ, np.int64)
    pr = node2vec_probs(succ, seen, prev, p, q)
    vals, inv = np.unique(succ, return_inverse=True)
    return vals, np.bincount(inv, weights=pr, minlength=len(vals))


def reference_walks(succ_of, nodes, max_depth, kind="random", p=1.0, q=1.0, rng=None):
    """The reference's walk loops (walk.py:23-183) restated over ``succ_of(v)`` (successor array of v): one
    Python-level draw per walk per step, with a set of the previous node's successors (node2vec) or of every
    earlier node's (node2vec+) built for each draw as graph_kernel.node2vec_sample does, and numpy's RNG
    for rand().  Returns a list of lists."""
    rng = np.random.default_rng(0) if rng is None else rng
    if kind != "random" and p == 1.0 and q == 1.0:
        kind = "random"
    steps = walk_length(kind, max_depth, p, q) - 1
    walks = []
    for v in nodes:
        walk = [int(v)]
        prev, seen = -1, []
        for _ in range(steps):
            succ = succ_of(walk[-1])
            if len(succ) == 0:
                break
            if kind == "random":
                nxt = int(succ[int(rng.random() * len(succ))])
            else:
                pr = node2vec_probs(succ, seen, prev, p, q)
                nxt = int(succ[min(int(np.searchsorted(np.cumsum(pr), rng.random() * pr.sum(), "right")),
                                   len(succ) - 1)])
                seen = list(set(seen) | set(succ.tolist())) if kind == "plus" else succ
                prev = walk[-1]
            walk.append(nxt)
        walks.append(walk)
    return walks


def skip_gram_gen_pair(walk, windows):
    """graph_kernel.skip_gram_gen_pair (graph_kernel.pyx:343-364) with the window of every position given
    (the reference draws them with np.random.randint(1, win_size + 1)): position i pairs with every j in
    [i - windows[i], i + windows[i]] clipped to the walk, skipping j with walk[j] == walk[i].  (src, dst)."""
    walk = list(walk)
    n = len(walk)
    src, dst = [], []
    for i in range(n):
        left, right = max(i - int(windows[i]), 0), min(i + int(windows[i]), n - 1)
        for j in range(left, right + 1):
            if walk[i] == walk[j]:
                continue
            src.append(walk[i])
            dst.append(walk[j])
    return np.asarray(src, np.int64), np.asarray(dst, np.int64)
