"""Generate tests/golden/ref_node2vec.npz from the REFERENCE's compiled ``pgl.graph_kernel`` (built by
oracle/build.py into oracle/_ref/, where the reference sources exist):  python tests/golden/make_walk_golden.py

For fixed (succ, prev_succ, prev, p, q) cases it stores how often ``node2vec_sample`` and ``node2vec_plus_sample``
(pgl/graph_kernel.pyx:142-224) return each candidate in NODE2VEC_DRAWS calls, and the seen set
``node2vec_plus_sample`` hands to the next step.  The tests read only the .npz.  The reference draws with C
``rand()`` without a seed call, so a rerun in a fresh process writes the same counts.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import build as obuild  # noqa: E402

NODE2VEC_DRAWS = 100000
# (succ, prev_succ, prev, p, q): duplicates in succ, the previous node among the candidates or not, the first step
# (prev -1, nothing seen), p and q from {0.25, 1, 4}
NODE2VEC_CASES = (
    ([1, 2, 3, 4, 5], [2, 3], 1, 0.25, 4.0),
    ([1, 2, 3, 4, 5], [2, 3], 1, 4.0, 0.25),
    ([1, 1, 2, 3, 3, 3, 7], [3, 9], 1, 1.0, 4.0),
    ([5, 6, 7, 8], [], -1, 0.25, 0.25),
    ([10, 11, 12, 13], [11, 12, 99], 9, 0.25, 1.0),
    ([0, 2, 2, 4, 6, 8], [0, 2, 4], 0, 4.0, 4.0),
    ([3, 3, 3, 5], [5], 3, 0.25, 0.25),
    ([1, 2, 3, 4, 5, 6, 7, 8, 9, 10], [2, 4, 6, 8, 10], 5, 1.0, 0.25),
)


def node2vec_fixtures(gk):
    out = {"num_cases": np.int64(len(NODE2VEC_CASES)), "draws": np.int64(NODE2VEC_DRAWS)}
    for c, (succ, prev_succ, prev, p, q) in enumerate(NODE2VEC_CASES):
        succ_a, prev_a = np.array(succ, np.int64), np.array(prev_succ, np.int64)
        vals = np.unique(succ_a)
        out.update({"c%d_succ" % c: succ_a, "c%d_prev_succ" % c: prev_a, "c%d_prev" % c: np.int64(prev),
                    "c%d_p" % c: np.float64(p), "c%d_q" % c: np.float64(q), "c%d_values" % c: vals})
        for name, fn in (("plain", gk.node2vec_sample), ("plus", gk.node2vec_plus_sample)):
            counts = np.zeros(len(vals) + 1, np.int64)   # last entry: the reference returned None
            seen = None
            for _ in range(NODE2VEC_DRAWS):
                r = fn(succ_a, prev_a, prev, p, q)
                if name == "plus" and r is not None:
                    r, seen = r
                counts[len(vals) if r is None else int(np.searchsorted(vals, r))] += 1
            out["c%d_%s_counts" % (c, name)] = counts
            if name == "plus":
                out["c%d_plus_next_seen" % c] = np.sort(np.asarray(seen, np.int64))
    np.savez_compressed(os.path.join(HERE, "ref_node2vec.npz"), **out)


def main():
    gk = obuild.load_ref_graph_kernel()
    if gk is None:
        obuild.build_ref()
        gk = obuild.load_ref_graph_kernel()
    node2vec_fixtures(gk)
    print("written", os.path.join(HERE, "ref_node2vec.npz"))


if __name__ == "__main__":
    main()
