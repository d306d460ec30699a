"""Random-walk input pipeline timing (DeepWalk / node2vec, DESIGN.md section 4.13) on the cfg5 graph
(bench.gen_edges: 10M nodes / 100M edges, Chung-Lu exponent 0.8).  Prints one JSON line:

* full-graph legs: random_walk from every node at walk_len 40 (examples/deepwalk's default), node2vec_walk and
  node2vec_walk_plus at p = q = 0.25 (examples/node2vec/config.yaml), skip_gram_pairs at win_size 10 over the
  first --sg-walks random walks (the pairs of every walk, about 4e9, would need about 70 GB);
* the same modes on a DeepWalk-sized batch (1 024 start nodes), where launch overhead dominates;
* for comparison on a fixed subsample: the host twin (pglb_random_walk_host) and the reference's per-walk,
  per-step loop restated in Python (tests/walk_oracle.py reference_walks).

kernel_ms: CUDA events around the C-ABI launch alone, averaged over --iters after warm-up.  call_ms: the public
call, which also range-checks the start nodes (one read-back).  steps_per_s counts the steps walks actually took.
The byte model per step is the least DRAM/L2 traffic of a uniform step; node2vec adds per draw one column sector
and the binary search of the previous row (node2vec+: of every earlier row).  Usage:
python scripts/bench_walk.py [--nodes N --edges E --iters K]."""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402  (gen_edges)

UNIFORM_STEP_BYTES = 16 + 32 + 8   # indptr pair, one 32-byte column sector, the 8-byte output entry


def gpu_identity():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": r.stdout.strip()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nodes", type=int, default=10_000_000)
    ap.add_argument("--edges", type=int, default=100_000_000)
    ap.add_argument("--exponent", type=float, default=0.8)
    ap.add_argument("--seed", type=int, default=20240922)
    ap.add_argument("--walk-len", type=int, default=40)
    ap.add_argument("--pq", type=float, default=0.25)
    ap.add_argument("--sg-walks", type=int, default=1_000_000)
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--host-walks", type=int, default=20000)
    ap.add_argument("--ref-walks", type=int, default=50)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_walk.py needs a CUDA device")
    import pgl_b200 as pgl
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import walk_oracle as W
    from pgl_b200._lib import WALK_NODE2VEC, WALK_NODE2VEC_PLUS, WALK_UNIFORM, check, lib
    from pgl_b200.sampling import node2vec_walk, node2vec_walk_plus, random_walk, skip_gram_pairs

    dev = torch.device("cuda", 0)
    n = args.nodes
    edges = bench.gen_edges(torch, n, args.edges, args.exponent, args.seed, dev)
    g = pgl.Graph(edges=edges, num_nodes=n)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    indptr, cols = g.successor_csr()
    torch.cuda.synchronize()
    res = {"gpu": gpu_identity(),
           "workload": "cfg5 Chung-Lu exp %.1f, %d nodes / %d edges; walk_len %d, p = q = %g"
                       % (args.exponent, n, args.edges, args.walk_len, args.pq),
           "successor_csr_build_ms": (time.perf_counter() - t0) * 1e3,
           "uniform_step_bytes": UNIFORM_STEP_BYTES, "legs": {}}
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    stream = lambda: ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)  # noqa: E731
    P = lambda t: ctypes.c_void_p(t.data_ptr())  # noqa: E731

    modes = (("random_walk", WALK_UNIFORM, args.walk_len - 1, random_walk, {}),
             ("node2vec_walk", WALK_NODE2VEC, args.walk_len, node2vec_walk, {"p": args.pq, "q": args.pq}),
             ("node2vec_walk_plus", WALK_NODE2VEC_PLUS, args.walk_len, node2vec_walk_plus,
              {"p": args.pq, "q": args.pq}))

    def leg(name, nodes, mode, steps, fn, kw):
        m = int(nodes.shape[0])
        out = torch.empty((m, steps + 1), dtype=torch.int64, device=dev)

        def launch():
            check(lib.pglb_random_walk(P(indptr), P(cols), n, P(nodes), m, steps, mode, args.pq, args.pq, 1234,
                                       P(out), steps + 1, stream()))
        launch()
        torch.cuda.synchronize()
        a, b = ev(), ev()
        a.record()
        for _ in range(args.iters):
            launch()
        b.record()
        torch.cuda.synchronize()
        kms = a.elapsed_time(b) / args.iters
        taken = int((out >= 0).sum().item()) - m
        fn(g, nodes, steps + (1 if mode == WALK_UNIFORM else 0), seed=1234, **kw)   # warm the public call
        torch.cuda.synchronize()
        t = time.perf_counter()
        for _ in range(args.iters):
            fn(g, nodes, steps + (1 if mode == WALK_UNIFORM else 0), seed=1234, **kw)
        torch.cuda.synchronize()
        cms = (time.perf_counter() - t) * 1e3 / args.iters
        r = {"walks": m, "steps_taken": taken, "kernel_ms": kms, "call_ms": cms,
             "steps_per_s": taken / (kms * 1e-3)}
        if mode == WALK_UNIFORM:
            r["model_GBs"] = taken * UNIFORM_STEP_BYTES / (kms * 1e-3) / 1e9
        return r, out

    all_nodes = torch.arange(n, device=dev)
    batch = torch.from_numpy(np.random.default_rng(7).integers(0, n, 1024)).to(dev)
    walks = None
    for name, mode, steps, fn, kw in modes:
        r, out = leg(name, all_nodes, mode, steps, fn, kw)
        res["legs"][name + "_full"] = r
        if mode == WALK_UNIFORM:
            walks = out
        else:
            del out
        res["legs"][name + "_batch1024"] = leg(name, batch, mode, steps, fn, kw)[0]
    res["node2vec_plus_over_node2vec"] = (res["legs"]["node2vec_walk_plus_full"]["kernel_ms"]
                                          / res["legs"]["node2vec_walk_full"]["kernel_ms"])

    # skip-gram pairs at win_size 10
    for name, w in (("skip_gram_pairs_%d_walks" % args.sg_walks, walks[:args.sg_walks]),
                    ("skip_gram_pairs_batch1024", walks[:1024])):
        src, dst = skip_gram_pairs(w, win_size=10, seed=5)
        del src, dst
        torch.cuda.synchronize()
        t = time.perf_counter()
        for _ in range(args.iters):
            src, dst = skip_gram_pairs(w, win_size=10, seed=5)
            del src, dst
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t) * 1e3 / args.iters
        pairs = int(skip_gram_pairs(w, win_size=10, seed=5)[0].shape[0])
        res["legs"][name] = {"walks": int(w.shape[0]), "pairs": pairs, "call_ms": ms,
                             "pairs_per_s": pairs / (ms * 1e-3), "out_GBs": pairs * 16 / (ms * 1e-3) / 1e9}
    del walks

    # host twin and the reference loop, on a fixed subsample of start nodes
    ip_h, cols_h = indptr.cpu().numpy(), cols.cpu().numpy()
    sub = np.random.default_rng(8).integers(0, n, args.host_walks).astype(np.int64)
    for name, mode, steps, fn, kw in modes:
        out = np.empty((len(sub), steps + 1), np.int64)
        t = time.perf_counter()
        check(lib.pglb_random_walk_host(ctypes.c_void_p(ip_h.ctypes.data), ctypes.c_void_p(cols_h.ctypes.data), n,
                                        ctypes.c_void_p(sub.ctypes.data), len(sub), steps, mode, args.pq, args.pq,
                                        1234, ctypes.c_void_p(out.ctypes.data), steps + 1))
        s = time.perf_counter() - t
        taken = int((out >= 0).sum()) - len(sub)
        res["legs"][name + "_host_twin"] = {"walks": len(sub), "steps_taken": taken, "ms": s * 1e3,
                                            "steps_per_s": taken / s}
        kind = {WALK_UNIFORM: "random", WALK_NODE2VEC: "node2vec", WALK_NODE2VEC_PLUS: "plus"}[mode]
        depth = steps + (1 if mode == WALK_UNIFORM else 0)
        rsub = sub[:args.ref_walks]
        t = time.perf_counter()
        ref = W.reference_walks(lambda v: cols_h[ip_h[v]:ip_h[v + 1]], rsub, depth, kind, args.pq, args.pq)
        s = time.perf_counter() - t
        taken = sum(len(w) - 1 for w in ref)
        res["legs"][name + "_reference_loop"] = {"walks": len(rsub), "steps_taken": taken, "ms": s * 1e3,
                                                 "steps_per_s": taken / s}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
