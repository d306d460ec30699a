"""GPU neighbour sampling (mirror of reference pgl/sampling/sage.py:130-155): csrc/sampling.cu, validated on
hardware in round 2 (tests/test_gpu_sampling.py, DESIGN.md section 4.11).  Random walks and skip-gram pairs (mirror
of reference pgl/sampling/walk.py): csrc/walk.cu (DESIGN.md section 4.13)."""
from .custom import subgraph  # noqa: F401
from .sage import NeighborSampler, reindex_graph, sample_neighbors  # noqa: F401
from .walk import node2vec_walk, node2vec_walk_plus, random_walk, skip_gram_pairs  # noqa: F401
