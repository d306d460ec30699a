"""Property-based checks (hypothesis) of the integer half on the CPU side of the C-ABI: for arbitrary small
edge lists -- empty, single node, duplicates, self loops, gaps in the id range, num_nodes larger than the
largest id -- pglb_build_index_host == the numpy oracle == the loop restatement, plus the structural
invariants a CSR must satisfy; on a fixed set of such edge lists also == the reference's own compiled
graph_kernel.build_index (outputs stored by tests/golden/make_golden.py).  Also the reindex oracle against
a dictionary restatement."""
import os

import numpy as np
from hypothesis import given, settings, strategies as st

from oracle import oracle as O

REF_GK = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_graph_kernel.npz")
FIELDS = ("degree", "sorted_v", "sorted_u", "sorted_eid", "indptr")


@st.composite
def edge_lists(draw):
    n = draw(st.integers(1, 40))
    e = draw(st.integers(0, 120))
    u = draw(st.lists(st.integers(0, n - 1), min_size=e, max_size=e))
    v = draw(st.lists(st.integers(0, n - 1), min_size=e, max_size=e))
    extra = draw(st.integers(0, 5))
    return n + extra, np.array(u, np.int64), np.array(v, np.int64)


@settings(max_examples=150, deadline=None)
@given(edge_lists())
def test_build_index_host_matches_oracle(case):
    from pgl_b200.utils.edge_index import build_index_host
    n, u, v = case
    got = build_index_host(u, v, n)
    want = O.build_index(u, v, n)
    loops = O.build_index_loops(u, v, n)
    for a, b, c in zip(got, want, loops):
        assert (np.asarray(a) == np.asarray(b)).all() and (np.asarray(b) == np.asarray(c)).all()
    degree, sorted_v, sorted_u, sorted_eid, indptr = got
    assert indptr[0] == 0 and indptr[-1] == len(u) and (np.diff(indptr) == degree).all()
    assert (np.diff(sorted_u) >= 0).all()                                   # keyed by u
    assert (u[sorted_eid] == sorted_u).all() and (v[sorted_eid] == sorted_v).all()
    for r in range(n):                                                      # stable: ascending edge id per row
        assert (np.diff(sorted_eid[indptr[r]:indptr[r + 1]]) > 0).all()
    assert sorted(sorted_eid.tolist()) == list(range(len(u)))


def test_build_index_host_matches_reference_cases():
    from pgl_b200.utils.edge_index import build_index_host
    g = np.load(REF_GK)
    cases = sorted({k.split("_")[0] for k in g.files if k.startswith("case")})
    assert len(cases) >= 50
    for c in cases:
        u, v, n = g[c + "_u"], g[c + "_v"], int(g[c + "_n"])
        for impl in (build_index_host, O.build_index, O.build_index_loops):
            for f, a in zip(FIELDS, impl(u, v, n)):
                assert np.array_equal(np.asarray(a), g[c + "_" + f]), (c, impl.__name__, f)


@settings(max_examples=100, deadline=None)
@given(st.integers(1, 12).flatmap(lambda n: st.tuples(
    st.permutations(list(range(30))).map(lambda p: p[:n]),
    st.lists(st.integers(0, 5), min_size=n, max_size=n))), st.randoms(use_true_random=False))
def test_reindex_oracle_first_appearance(xc, rnd):
    x, count = xc
    nb = [rnd.randrange(30) for _ in range(sum(count))]
    src, dst, out = O.reindex_graph(x, nb, count)
    assert out[:len(x)].tolist() == list(x) and len(set(out.tolist())) == len(out)
    assert (out[src] == np.asarray(nb, np.int64)).all()                     # the mapping inverts
    assert dst.tolist() == [i for i, c in enumerate(count) for _ in range(c)]
    seen, order = set(x), []
    for v in nb:
        if v not in seen:
            seen.add(v)
            order.append(v)
    assert out[len(x):].tolist() == order
