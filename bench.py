#!/usr/bin/env python
"""bench.py -- edges/sec per GCN layer (128-d feat) on synthetic power-law graphs.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config cfg5|cfg3|cfg4]
                    [--dump-outputs DIR]

One "step" = one GCN-layer aggregation over the whole graph: ``send_recv(sum)`` with both
degree-norm scalings (reference pgl/nn/conv.py:242-250 around graph.py:860), i.e. the SpMM the
BASELINE.md roofline table is written for.  Workload (BASELINE.json configs[4], "cfg5"):
10M nodes / 100M edges Chung-Lu power-law graph (exponent 0.8, ids randomly permuted,
duplicates and self loops kept), 128-d float32 features.

N > 1 (torchrun, one rank per GPU): the default layout shards the FEATURE COLUMNS (every rank holds the
whole CSR and 128/N columns of every row: a copy-message aggregation is independent per column, so the
step needs no exchange at all -- the reference's own large-feature example shards columns the same way,
examples/.../dist_feat.py:31-49); ``--shard rows`` keeps the 1-D row partition (METIS or block) + halo
exchange of round 1.

Prints ONE JSON line (rank 0).  Keys follow the driver contract; additionally
  roofline      dominant kernel vs the measured HBM copy bandwidth (MEASURED_PEAKS.json)
  cpu_baseline  the oracle's C restatement of the reference CPU loop on a bounded sample
  parity        the GPU result checked against that oracle output on the same inputs, in this run
  e2e           same metric through the public API with pinned HOST buffers (H2D + D2H inside)
  full_layer    GCNConv(128,128).forward (aggregation + dense transform + bias + ReLU) edges/s

``--config cfg3`` (GATConv on RMAT 1M/10M) and ``--config cfg4`` (3-layer GraphSAGE on a products-shape
graph) time BASELINE.json configs[2] and configs[3] with their own roofline models.

``--dump-outputs DIR`` writes what the timed path returned in its last timed step to DIR/<name>.npy
(float32, one row per output row, the row numbers in DIR/<name>_rows.npy; see dump_outputs), so that two
builds run with the same arguments -- hence the same seeded inputs -- can be compared output for output.
"""
import argparse
import ctypes
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the package is imported from the tree, which bench.py leaves as it found it

FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback
PARITY_TOL = 1e-4           # north_star: "correctness matching reference PGL within 1e-4 relative"
DUMP_BYTES = 48 << 20       # --dump-outputs: bytes of all files of one run together (every rank included)
DUMP_SEED = 0


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg5", choices=["cfg5", "cfg3", "cfg4"])
    ap.add_argument("--nodes", type=int, default=10_000_000)
    ap.add_argument("--edges", type=int, default=100_000_000)
    ap.add_argument("--dim", type=int, default=128)
    ap.add_argument("--exponent", type=float, default=0.8)
    ap.add_argument("--seed", type=int, default=20240922)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-full-layer", action="store_true")
    ap.add_argument("--shard", default=os.environ.get("PGLB_SHARD", "cols"), choices=["cols", "rows"])
    ap.add_argument("--grid", default=os.environ.get("PGLB_GRID", ""),
                    help="N > 1, --shard cols: RrxRc = row groups x column groups (default: 2 column groups)")
    ap.add_argument("--partition", default="block", choices=["block", "metis"])
    ap.add_argument("--halo", default=os.environ.get("PGLB_HALO_MODE", "p2p"), choices=["nccl", "p2p"])
    ap.add_argument("--overlap", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned to DIR/<name>.npy (float32; a fixed seeded sample "
                         "of the rows when the output is larger than %d MiB)" % (DUMP_BYTES >> 20))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def host_threads():
    """CPU threads this process may really use: the affinity mask, capped by a cgroup CPU quota if
    one is set (os.cpu_count() reports the machine, not the container)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    quota = None
    try:
        q = open("/sys/fs/cgroup/cpu.max").read().split()           # cgroup v2: "<quota|max> <period>"
        if q[0] != "max":
            quota = int(q[0]) / int(q[1])
    except Exception:
        try:                                                           # cgroup v1
            cq = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            cp = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if cq > 0 and cp > 0:
                quota = cq / cp
        except Exception:
            pass
    if quota is not None:
        n = min(n, max(1, int(quota + 0.999)))
    return max(1, n)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def algorithmic_bytes(n_dst, n_edges, dim):
    """SURVEY.md section 8d: E*(4D+8) + N*4D + (N+1)*8, plus the two norm vectors."""
    return n_edges * (4 * dim + 8) + n_dst * 4 * dim + (n_dst + 1) * 8 + 2 * n_dst * 4


def gen_edges(torch, n, e, exponent, seed, device):
    """Chung-Lu power-law graph: w_i ~ (i+1)^-exponent, src,dst ~ Cat(w) iid via the float64
    inverse CDF, ids relabelled by a fixed random permutation; duplicates/self loops kept."""
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    w = torch.arange(1, n + 1, device=device, dtype=torch.float64).pow_(-exponent)
    cdf = torch.cumsum(w, 0)
    cdf /= cdf[-1].clone()
    del w
    perm = torch.randperm(n, generator=g, device=device)
    out = torch.empty((e, 2), dtype=torch.int64, device=device)
    chunk = 1 << 24
    for col in (0, 1):
        for s in range(0, e, chunk):
            m = min(chunk, e - s)
            r = torch.rand(m, generator=g, device=device, dtype=torch.float64)
            idx = torch.searchsorted(cdf, r).clamp_(max=n - 1)
            out[s:s + m, col] = perm[idx]
    return out


def gen_features(torch, n, d, seed, device):
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    return torch.randn(n, d, device=device, generator=g)


def rmat_edges(torch, scale, e, a=0.57, b=0.19, c=0.19, seed=1, device="cuda"):
    """RMAT (a, b, c, d) = (0.57, 0.19, 0.19, 0.05), noise off, duplicates / self loops kept (SURVEY 8d cfg3)."""
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    src = torch.zeros(e, dtype=torch.int64, device=device)
    dst = torch.zeros(e, dtype=torch.int64, device=device)
    for _ in range(scale):
        r = torch.rand(e, generator=g, device=device)
        sb = (r >= a + b).to(torch.int64)
        db = (((r >= a) & (r < a + b)) | (r >= a + b + c)).to(torch.int64)
        src = src * 2 + sb
        dst = dst * 2 + db
    return torch.stack([src, dst], 1)


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons while the timed region runs (NVML)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop_evt = threading.Event()

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {
                "hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4),
                "hw_power_brake_slowdown": getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80),
            }
            get = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                nv.nvmlDeviceGetCurrentClocksThrottleReasons
            while not self._stop_evt.is_set():
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = get(h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
                time.sleep(0.05)
        except Exception as ex:  # NVML missing: report that instead of inventing numbers
            self.reasons.add("nvml_unavailable:%s" % type(ex).__name__)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------
# CPU legs (oracle = checker / reported baseline; never on the product path)
# ------------------------------------------------------------------------------------------

def _ptr(a):
    return ctypes.c_void_p(a.ctypes.data)


def _i64(v):
    return ctypes.c_int64(int(v))


def _load_oracle_c():
    """The oracle's C library as build() left it.  bench.py writes nothing into the tree (it may be read-only):
    a missing or out-of-date library is compiled into a temporary directory instead."""
    import tempfile
    from oracle import build as obuild
    with tempfile.TemporaryDirectory(prefix="pglb_oracle_") as tmp:
        return ctypes.CDLL(obuild.build_oracle_c(out=os.path.join(tmp, "liboracle_c.so")))


class CpuGcn(object):
    """The oracle's restatement of the reference CPU path for ONE GCN-layer aggregation
    (pgl/nn/conv.py:242-250): ``feature * norm`` -> send_u_recv(sum) -> ``output * norm``, on the rows
    dst < n_s of the workload with ALL their in-edges (ids are randomly permuted, so this is a uniform
    row sample; frac = 1 is the whole graph) and the full feature matrix.

    ``run(threads)``: threads == 1 -> the sequential COO loop (Paddle's CPU send_u_recv contract);
    threads > 1 -> the row-threaded CSR twin (bit-identical results, oracle/oracle_c.c)."""

    def __init__(self, lib, src_np, dst_np, n, dim, frac, threads, n_rows=None):
        """n: rows of the feature matrix (sources); n_rows: destination rows of this edge list (default n)."""
        self.lib, self.n, self.dim, self.frac = lib, int(n), int(dim), float(frac)
        self.n_rows = int(n if n_rows is None else n_rows)
        self.e_total = int(len(src_np))
        if frac >= 1.0:
            self.n_s, self.src, self.dst = self.n_rows, src_np, dst_np
        else:
            self.n_s = max(1, int(self.n_rows * frac))
            m = dst_np < self.n_s
            self.src = np.ascontiguousarray(src_np[m])
            self.dst = np.ascontiguousarray(dst_np[m])
        self.e_s = int(len(self.src))
        self.ip = self.sv = None
        if threads > 1:
            # dst-keyed CSR of the sample (graph preparation, like the GPU's cached index: not timed)
            deg = np.empty(self.n_s, np.int64)
            self.ip = np.empty(self.n_s + 1, np.int64)
            self.sv = np.empty(self.e_s, np.int64)
            su = np.empty(self.e_s, np.int64)
            se = np.empty(self.e_s, np.int64)
            rc = lib.orc_build_index(_ptr(self.dst), _ptr(self.src), _i64(self.e_s), _i64(self.n_s),
                                     _ptr(deg), _ptr(self.sv), _ptr(su), _ptr(se), _ptr(self.ip))
            assert rc == 0
            del su, se, deg
        self.sample = ("rows dst < %d (%.2f%% of the graph's rows with all their in-edges: %d of %d edges), "
                       "full %d-row feature matrix" % (self.n_s, 100.0 * self.n_s / self.n_rows, self.e_s,
                                                       self.e_total, self.n))
        self.xs = None
        self.out = None

    def run(self, x_np, norm_np, threads, scaled=True, norm_dst_np=None):
        """One pass.  Returns (seconds charged, detail).  The source scaling touches all N rows whatever
        the sample is; its time is charged in proportion to the sample (frac), everything else in full."""
        lib, d = self.lib, self.dim
        if self.out is None:
            self.out = np.empty((self.n_s, d), np.float32)
        t_scale_in = 0.0
        xin = x_np
        if scaled:
            if self.xs is None:
                self.xs = np.empty_like(x_np)
            t0 = time.perf_counter()
            lib.orc_scale_rows_f32(_ptr(x_np), _ptr(norm_np), _i64(self.n), _i64(d), _ptr(self.xs), int(threads))
            t_scale_in = time.perf_counter() - t0
            xin = self.xs
        t0 = time.perf_counter()
        if threads > 1:
            lib.orc_send_u_recv_csr_f32(_ptr(xin), _ptr(self.ip), _ptr(self.sv), _i64(self.n_s), _i64(d), 0,
                                        _ptr(self.out), int(threads))
        else:
            lib.orc_send_u_recv_f32(_ptr(xin), _ptr(self.src), _ptr(self.dst), _i64(self.e_s), _i64(self.n_s),
                                    _i64(d), 0, _ptr(self.out))
        t_agg = time.perf_counter() - t0
        t_scale_out = 0.0
        if scaled:
            t0 = time.perf_counter()
            nd = norm_np if norm_dst_np is None else norm_dst_np   # norm of the destination rows (local numbering)
            lib.orc_scale_rows_f32(_ptr(self.out), _ptr(nd), _i64(self.n_s), _i64(d), _ptr(self.out),
                                   int(threads))
            t_scale_out = time.perf_counter() - t0
        charged = t_scale_in * min(1.0, self.n_s / self.n_rows) + t_agg + t_scale_out
        return charged, {"scale_src_s_full_matrix": t_scale_in, "aggregate_s": t_agg, "scale_dst_s": t_scale_out,
                         "charged_s": charged, "threads": int(threads), "sample_edges": self.e_s,
                         "sample_rows": self.n_s, "edges_per_s": self.e_s / charged if charged > 0 else None}


def parity_stats(got, want, tol=PARITY_TOL):
    """got / want: float32 [rows, d] numpy.  max_rel_err = max |got - want| / max |want| (the tests' metric);
    row_rel_err normalises every row by its own largest entry."""
    got = np.asarray(got)
    want = np.asarray(want)
    diff = np.abs(got.astype(np.float64) - want.astype(np.float64))
    scale = float(np.abs(want).max()) if want.size else 1.0
    row_scale = np.maximum(np.abs(want).max(axis=1), 1e-30)
    row_err = diff.max(axis=1) / row_scale
    exact = int((got.view(np.uint32) == want.view(np.uint32)).all(axis=1).sum())
    res = {"rows": int(want.shape[0]), "cols": int(want.shape[1]),
           "max_rel_err": float(diff.max() / max(scale, 1e-30)) if want.size else 0.0,
           "max_row_rel_err": float(row_err.max()) if want.size else 0.0,
           "bit_exact_rows": exact, "tol": tol}
    res["pass"] = bool(res["max_rel_err"] <= tol and np.isfinite(res["max_rel_err"]))
    return res


def cpu_norm(indeg_np):
    from oracle import oracle as O
    return np.ascontiguousarray(O.degree_norm(indeg_np).reshape(-1))


def main_reference(args):
    """The reference's own CPU implementation of the path on the box's host cores, same config as the GPU arm:
    the whole cfg5 graph when one pass fits the budget (it does on a multi-core host: about a second on 16
    threads), both norm scalings included."""
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = host_threads()
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    n, d = args.nodes, args.dim
    edges = gen_edges(torch, n, args.edges, args.exponent, args.seed, dev)
    src_np = np.ascontiguousarray(edges[:, 0].cpu().numpy())
    dst_np = np.ascontiguousarray(edges[:, 1].cpu().numpy())
    del edges
    x_np = gen_features(torch, n, d, args.seed + 1, dev).cpu().numpy()
    if dev == "cuda":
        torch.cuda.empty_cache()
    norm_np = cpu_norm(np.bincount(dst_np, minlength=n)[:n])
    lib = _load_oracle_c()
    # budget: the whole --steps/--warmup run within a few minutes
    total_steps = max(1, args.steps + args.warmup)
    per = max(0.5, min(12.0, 200.0 / total_steps))
    probe = CpuGcn(lib, src_np, dst_np, n, d, 0.02, threads)
    t_probe, _ = probe.run(x_np, norm_np, threads)
    t_probe2, _ = probe.run(x_np, norm_np, threads)
    full_est = min(t_probe, t_probe2) / 0.02
    frac = 1.0 if full_est <= per else max(0.02, per / full_est)
    del probe
    prob = CpuGcn(lib, src_np, dst_np, n, d, frac, threads)
    vals, info = [], None
    for i in range(args.warmup + args.steps):
        t, info = prob.run(x_np, norm_np, threads)
        if i >= args.warmup:
            vals.append(prob.e_s / t)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"gcn_aggregate": prob.out})
    v = float(np.median(vals))
    line = {
        "impl": "reference", "metric": "edges/sec per GCN layer (128-d feat)", "value": v,
        "unit": "edges/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * args.edges / v, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args), "same_workload_as_gpu_arm": frac >= 1.0,
                   "note": "reference CPU path restated (Paddle unavailable in this image): oracle/oracle_c.c -- "
                           "feature*norm, send_u_recv(sum) as the row-threaded CSR twin of Paddle's sequential "
                           "COO loop (bit-identical results), output*norm; all host threads"},
        "cpu_baseline": {"value": v, "unit": "edges/s", "cores": threads, "kind": "port",
                         "sample": prob.sample, "detail": info},
        "e2e": {"value": v, "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def workload_name(args):
    return ("cfg5 synthetic power-law (Chung-Lu exp %.1f) %d nodes / %d edges, %d-d f32, GCN-layer "
            "SpMM aggregation: send_recv(sum) + both degree-norm scalings" %
            (args.exponent, args.nodes, args.edges, args.dim))


# ------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------

def _ev(torch):
    return torch.cuda.Event(enable_timing=True)


def timed_steps(torch, step, steps, dist=None):
    """EXACTLY `steps` calls bracketed by synchronize (+ barrier) on both sides; per-step CUDA events on the
    launching stream.  Returns (total_ms, sorted per-step ms, what the last call returned).  Only the last
    call's result is kept, so earlier results are freed as soon as their call returns."""
    evs = [(_ev(torch), _ev(torch)) for _ in range(steps)]
    last = None
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    b0, b1 = _ev(torch), _ev(torch)
    b0.record()
    for i, (a, b) in enumerate(evs):
        a.record()
        if i + 1 < steps:
            step()
        else:
            last = step()
        b.record()
    b1.record()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    return b0.elapsed_time(b1), sorted(a.elapsed_time(b) for a, b in evs), last


def dump_outputs(path, outputs, rank=0, world=1):
    """--dump-outputs: every array in `outputs` ({name: torch tensor or numpy array}) -> path/<name>.npy as float32
    rows [k, a[0].size], and path/<name>_rows.npy (float64 [k]): which rows of `a` they are (names suffixed with
    the rank when several ranks write).  An array larger than its share of DUMP_BYTES is stored as a fixed sample
    of its rows (DUMP_SEED, ascending row order): the same rows in every run with the same arguments.  Row i of
    the single-GPU cfg5 output is graph row i, in both arms; the reference arm's output holds only the rows it
    timed (dst < n_s, all of them when config.same_workload_as_gpu_arm)."""
    os.makedirs(path, exist_ok=True)
    share = DUMP_BYTES // (world * len(outputs))
    for name, a in outputs.items():
        rows = a.reshape(a.shape[0], -1)
        k = min(rows.shape[0], max(1, share // (4 * max(1, rows.shape[1]) + 8)))
        idx = np.arange(rows.shape[0])
        if k < rows.shape[0]:
            idx = np.sort(np.random.default_rng(DUMP_SEED).choice(rows.shape[0], k, replace=False))
            if isinstance(rows, np.ndarray):
                rows = rows[idx]
            else:
                import torch
                rows = rows[torch.from_numpy(idx).to(rows.device)]
        if not isinstance(rows, np.ndarray):
            rows = rows.float().cpu().numpy()
        fname = name if world == 1 else "%s_rank%d" % (name, rank)
        np.save(os.path.join(path, fname + ".npy"), np.ascontiguousarray(rows, dtype=np.float32))
        np.save(os.path.join(path, fname + "_rows.npy"), idx.astype(np.float64))


def read_traffic(key):
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        try:
            return json.load(open(tp)).get(key)
        except Exception:
            return None
    return None


def kernel_name(num_edges=None, num_rows=None):
    v5 = os.environ.get("PGLB_STREAM_V5")
    try:
        from pgl_b200 import ops
        return ops.stream_kernel_name(num_edges, num_rows)
    except Exception:
        return "spmm_stream (PGLB_STREAM_V5=%s)" % v5


def main_ours(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    import pgl_b200 as pgl
    from pgl_b200 import ops
    import pgl_b200.nn.functional as GF

    if args.config == "cfg3":
        result = bench_gat(args, torch, pgl, ops, GF, dev) if rank == 0 else None
    elif args.config == "cfg4":
        result = bench_sage(args, torch, dist, pgl, ops, GF, dev, world, rank)
    elif world > 1 and args.shard == "rows":
        result = bench_row_sharded(args, torch, dist, pgl, dev, world, rank)
    else:
        result = bench_gcn(args, torch, dist if world > 1 else None, pgl, ops, GF, dev, world, rank)
    if rank == 0 and result is not None:
        print(json.dumps(result))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if result is not None and result.get("parity") and result["parity"].get("pass") is False:
        raise SystemExit("bench.py: parity check against the oracle FAILED: %r" % (result["parity"],))


def parse_grid(args, world):
    """(row groups Rr, column groups Rc).  Default for N > 1: Rr = N, Rc = 1 -- every GPU aggregates the in-edges of its
    block of destination rows from a local replica of the source features (the reference's DistGPUGraph layout,
    pgl/graph.py:1490: edges by destination, features replicated -- minus its all-reduce of the [N, D] output, which a
    row-sharded output does not need).  `--grid 1xN` is the pure column shard, anything between a mix; DESIGN.md
    section 5 has the measured table and what each layout costs a full layer."""
    if world == 1:
        return 1, 1
    if args.grid:
        rr, rc = (int(v) for v in args.grid.lower().split("x"))
    else:
        rr, rc = world, 1
    assert rr * rc == world, "--grid RrxRc must multiply to the number of ranks"
    return rr, rc


def block_bounds(n, parts, i):
    """[lo, hi) of the i-th of `parts` nearly equal contiguous blocks of range(n)."""
    base, rem = divmod(n, parts)
    lo = i * base + min(i, rem)
    return lo, lo + base + (1 if i < rem else 0)


def balanced_row_bounds(torch, indeg, parts):
    """Row-block boundaries with (nearly) equal numbers of in-edges per block: a block of rows costs what its edges
    cost, and a power-law graph's hubs make equal ROW counts unequal work."""
    n = int(indeg.shape[0])
    if parts == 1:
        return [0, n]
    csum = torch.cumsum(indeg, 0)
    total = int(csum[-1].item())
    targets = torch.tensor([total * k // parts for k in range(1, parts)], device=indeg.device, dtype=csum.dtype)
    cuts = torch.searchsorted(csum, targets).tolist()
    b = [0] + [min(max(int(c) + 1, 1), n) for c in cuts] + [n]
    for i in range(1, len(b)):           # strictly increasing even on degenerate inputs
        b[i] = max(b[i], b[i - 1])
    return b


def bench_gcn(args, torch, dist, pgl, ops, GF, dev, world, rank):
    """cfg5 at 1 GPU; at N GPUs on an Rr x Rc grid: rank (r, c) owns destination rows block r and feature columns
    block c of every source row (column blocks are replicated across the Rr row groups, as the reference's
    DistGPUGraph replicates whole features).  No exchange inside the aggregation for any grid."""
    n, e, d = args.nodes, args.edges, args.dim
    rr, rc = parse_grid(args, world)
    r, c = rank // rc, rank % rc
    emu = os.environ.get("PGLB_BENCH_EMULATE", "")   # development aid: "RrxRc:rank" times ONE rank's shard on one GPU
    if emu and world == 1:
        gspec, rk = emu.split(":")
        rr, rc = (int(v) for v in gspec.lower().split("x"))
        r, c = int(rk) // rc, int(rk) % rc
    assert d % rc == 0 and (d // rc) % 4 == 0, "feature width must split into 16-byte column slices"
    dl = d // rc
    c0 = c * dl
    hbm_gbs, peak_src = peaks()

    t0 = time.perf_counter()
    edges = gen_edges(torch, n, e, args.exponent, args.seed, dev)   # same seed: every rank sees the whole graph
    torch.cuda.synchronize()
    t_gen = time.perf_counter() - t0
    indeg = torch.bincount(edges[:, 1], minlength=n)
    bounds = balanced_row_bounds(torch, indeg, rr)                   # identical on every rank
    lo, hi = bounds[r], bounds[r + 1]
    n_loc = hi - lo
    norm = ops.degree_norm(indeg).reshape(-1)                        # global clip(in-degree, 1)^-0.5
    if rr > 1:
        m = (edges[:, 1] >= lo) & (edges[:, 1] < hi)
        edges_loc = torch.stack([edges[m, 0], edges[m, 1] - lo], 1)  # my rows' in-edges, destinations renumbered
        del m
    else:
        edges_loc = edges
    e_loc = int(edges_loc.shape[0])
    g = pgl.Graph(edges=edges_loc, num_nodes=n)
    s0, s1 = _ev(torch), _ev(torch)
    g._fwd_csr()                     # first call pays one-off costs (module load, workspace growth): not the build time
    g2 = pgl.Graph(edges=edges_loc, num_nodes=n)
    torch.cuda.synchronize()
    s0.record()
    g2._fwd_csr()                    # device CSR build, steady state
    s1.record()
    torch.cuda.synchronize()
    t_csr_ms = s0.elapsed_time(s1)
    del g2
    fwd = g._csr_for_rows(n_loc)     # dst-CSR truncated to my rows (the rows behind them have no in-edges)
    norm_dst = norm[lo:hi].contiguous()
    x_full = gen_features(torch, n, d, args.seed + 1, dev)
    x = x_full if rc == 1 else x_full[:, c0:c0 + dl].contiguous()
    del x_full
    torch.cuda.empty_cache()
    out = torch.empty(n_loc, dl, device=dev)
    packed = ops._packed_of(fwd, x)  # cached per graph: packed column ids (wide rows) or the narrow-row plan

    def step():
        return ops._spmm_raw(fwd["indptr"], fwd["cols"], x, n_loc, "sum", scale_src=norm,
                             scale_dst=norm_dst, max_degree=fwd["max_degree"], out=out, packed=packed)

    warm = max(args.warmup, 3)
    for _ in range(warm):
        step()
    torch.cuda.synchronize()
    sampler = ClockSampler(dev.index)
    sampler.start()
    l0 = ops.launch_count()
    total_ms, per, last = timed_steps(torch, step, args.steps, dist)
    launches = ops.launch_count() - l0
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"gcn_aggregate": last}, rank, world)
    kern_ms = float(np.mean(per))
    b_alg = algorithmic_bytes(n_loc, e_loc, dl)    # this rank's kernel: its edges, its rows, its columns
    achieved = b_alg / (kern_ms * 1e-3) / 1e9
    per_rank = None
    if dist is not None:
        t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t[0].item())
        lt = torch.tensor([launches], device=dev, dtype=torch.int64)
        dist.all_reduce(lt)
        launches = int(lt.item())
        mine = {"rank": rank, "grid_pos": [r, c], "rows": n_loc, "edges": e_loc, "cols": dl, "kernel_ms": kern_ms,
                "algorithmic_bytes": b_alg, "achieved_GBs": achieved}
        per_rank = [None] * world
        dist.all_gather_object(per_rank, mine)
        slow = min(per_rank, key=lambda q: q["achieved_GBs"])   # the roofline line quotes the least efficient rank
        kern_ms, b_alg, achieved = slow["kernel_ms"], slow["algorithmic_bytes"], slow["achieved_GBs"]
    ms_step = total_ms / args.steps
    value = e / (ms_step * 1e-3)

    # ---- parity against the oracle, in this run ---------------------------------------------
    cpu = None
    parity = None
    if not args.no_cpu:
        try:
            cpu, parity = cpu_and_parity(args, torch, dist, ops, fwd, edges_loc, indeg, x, norm, norm_dst, out, step,
                                         dev, world, rank, n, n_loc, lo, c0, dl)
        except Exception as ex:
            cpu = {"value": None, "unit": "edges/s", "cores": 1, "kind": "port", "sample": "failed: %r" % (ex,)}
            parity = {"pass": None, "error": repr(ex)[:300]}

    # ---- full GCN layer ------------------------------------------------------------------------
    full = None
    if not args.no_full_layer:
        try:
            full = full_layer(args, torch, dist, pgl, ops, g, step, x, norm, dev, world, rank, rr, rc, r, c, n, n_loc,
                              e, d, dl)
        except Exception as ex:
            full = {"value": None, "error": repr(ex)[:300]}

    # ---- e2e: public API, pinned host buffers, H2D of the step's input + D2H of its result inside
    e2e = None
    if not args.no_e2e:
        try:
            e2e = e2e_host(args, torch, dist, ops, g, fwd, x, norm, norm_dst, dev, world, rank, rr, rc, r, c, bounds, n,
                           n_loc, e, dl)
        except Exception as ex:
            e2e = {"value": None, "unit": "edges/s", "error": repr(ex)[:300]}

    if world == 1:
        par = "single GPU"
    else:
        par = ("%d x %d grid: %d destination-row groups x %d feature-column groups; a rank holds the in-edges of its "
               "%d rows and %d of the %d feature columns of ALL source rows (column blocks replicated across the row "
               "groups); the aggregation needs no exchange (full_layer adds the re-shard to whole rows)" %
               (rr, rc, rr, rc, n_loc, dl, d))
    return {
        "metric": "edges/sec per GCN layer (128-d feat)", "value": value, "unit": "edges/s",
        "n_gpus": world, "steps": args.steps, "warmup": warm, "ms_per_step": ms_step,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": workload_name(args),
                   "l2": "inputs (%.2f GB of feature rows per GPU) larger than L2" % (n * dl * 4 / 1e9),
                   "parallelism": par, "grid": [rr, rc], "row_blocks": "balanced by in-edge count", "csr_build_ms": t_csr_ms, "graph_gen_s": t_gen,
                   "max_in_degree": int(fwd["max_degree"]), "index_dtype": "int64",
                   "packed_cols": packed is not None, "narrow_plan": isinstance(packed, ops.NarrowPlan),
                   "l2_hints": bool(packed.hints if isinstance(packed, ops.NarrowPlan) else (packed is not None and packed[1])),
                   "stream_v5": os.environ.get("PGLB_STREAM_V5", "default"), "per_rank": per_rank},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm_gbs, "unit": "GB/s",
                     "frac": achieved / hbm_gbs,
                     "traffic": read_traffic("spmm_csr_kernel_bytes_per_launch" if world == 1 else
                                             "grid%dx%d_bytes_per_launch" % (rr, rc)),
                     "peak_source": peak_src, "frac_of_nominal_8000GBs": achieved / 8000.0,
                     "algorithmic_bytes": b_alg,
                     "note": "the least efficient rank's kernel: E_r*(4*Dl+8) + N_r*4*Dl + (N_r+1)*8 + 2*N_r*4 bytes "
                             "(its edges, its rows, Dl = %d columns) over its mean kernel time (CUDA events around each "
                             "step on the launching stream)" % dl,
                     "kernel": kernel_name(e_loc, n_loc) if dl > 64 else "spmm_narrow2_kernel (+ empty_rows, fix-up kernels)",
                     "kernel_ms_mean": kern_ms,
                     "kernel_ms_p10": per[len(per) // 10], "kernel_ms_p90": per[(len(per) * 9) // 10]},
        "cpu_baseline": cpu, "parity": parity, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
        "full_layer": full,
    }


def cpu_and_parity(args, torch, dist, ops, fwd, edges_loc, gdeg, x, norm, norm_dst, out, step, dev, world, rank, n,
                   n_loc, lo, c0, dl):
    """Rank 0: the oracle's 1-thread COO pass on a bounded row sample (cpu_baseline).  Every rank: its block of the
    GPU output (its rows, its columns) on a row sample against the oracle's output for the same inputs --
    (a) the GCN-normalised aggregation (tolerance 1e-4: the kernel fuses x*norm into an FMA),
    (b) the plain sum: BIT-EXACT on every row of <= 1024 in-edges for the wide-row kernels (same summation order),
        rounding-level for the narrow-row kernel, and long rows judged against an fp64 sum."""
    lib = _load_oracle_c()
    src_np = np.ascontiguousarray(edges_loc[:, 0].cpu().numpy())
    dst_np = np.ascontiguousarray(edges_loc[:, 1].cpu().numpy())
    x_np = x.cpu().numpy()
    norm_np = norm.cpu().numpy()
    indeg = fwd["degree"][:n_loc].cpu().numpy()
    # the oracle's norm needs the GLOBAL in-degree of every source (the ranks' norm vector came from the same counts)
    gdeg_np = gdeg.cpu().numpy()
    norm_ref = cpu_norm(gdeg_np)
    norm_dst_ref = np.ascontiguousarray(norm_ref[lo:lo + n_loc])
    threads = host_threads()
    cpu = None
    if rank == 0:
        # calibrate: about 12 s of single-thread work
        probe = CpuGcn(lib, src_np, dst_np, n, dl, 0.005, 1, n_rows=n_loc)
        t1, _ = probe.run(x_np, norm_ref, 1, norm_dst_np=norm_dst_ref)
        frac = min(1.0, max(0.005, 0.005 * float(os.environ.get("PGLB_BENCH_CPU_SECONDS", "12")) / max(t1, 1e-3)))
        del probe
    else:
        frac = 0.0
    if dist is not None:
        ft = torch.tensor([frac], device=dev, dtype=torch.float64)
        dist.broadcast(ft, 0)
        frac = float(ft.item())
    if rank != 0:
        frac = min(frac, 0.02)  # the other ranks only check: a 2 % sample of their rows
    prob = CpuGcn(lib, src_np, dst_np, n, dl, frac, threads, n_rows=n_loc)
    n_s = prob.n_s
    if rank == 0:
        t1, det1 = prob.run(x_np, norm_ref, 1, norm_dst_np=norm_dst_ref)
        cpu = {"value": prob.e_s / t1, "unit": "edges/s", "cores": 1, "kind": "port", "sample": prob.sample,
               "detail": {"coo_1thread": det1}}
        want = prob.out.copy()
        if threads > 1:
            tt, dett = prob.run(x_np, norm_ref, threads, norm_dst_np=norm_dst_ref)
            cpu["detail"]["csr_threads"] = dict(dett, identical_to_coo=bool(np.array_equal(want, prob.out)))
    else:
        prob.run(x_np, norm_ref, threads, norm_dst_np=norm_dst_ref)
        want = prob.out.copy()
    step()
    torch.cuda.synchronize()
    got = out[:n_s].cpu().numpy()
    parity = parity_stats(got, want)
    parity["norm_bit_exact"] = bool(np.array_equal(norm_np, norm_ref))
    # (b) plain sum
    prob.run(x_np, norm_ref, threads, scaled=False)
    plain = ops._spmm_raw(fwd["indptr"], fwd["cols"], x, n_loc, "sum", max_degree=fwd["max_degree"],
                          packed=ops._packed_of(fwd, x))
    torch.cuda.synchronize()
    gp = plain[:n_s].cpu().numpy()
    del plain
    short = indeg[:n_s] <= 1024
    ex_rows = (gp.view(np.uint32) == prob.out.view(np.uint32)).all(axis=1)
    ps = parity_stats(gp, prob.out)
    # rows of more than 1024 in-edges are cut into tasks whose partial sums are added in task order: a different
    # (deterministic) fp32 grouping than the oracle's one-by-one loop.  Both are judged against an fp64 sum of the
    # same row (torch on the device, a checker like the oracle) -- the sequential fp32 loop itself drifts by
    # ~1e-4 of the result on an 800 000-term row.
    long_rows = np.flatnonzero(~short)
    pick = long_rows[np.argsort(indeg[long_rows])[::-1][:64]] if len(long_rows) else long_rows
    err_gpu = err_orc = 0.0
    ip_t, cols_t = fwd["indptr"], fwd["cols"]
    for rrow in pick.tolist():
        a0, a1 = int(ip_t[rrow].item()), int(ip_t[rrow + 1].item())
        ref64 = x[cols_t[a0:a1]].double().sum(0).cpu().numpy()
        sc = max(float(np.abs(ref64).max()), 1e-30)
        err_gpu = max(err_gpu, float(np.abs(gp[rrow].astype(np.float64) - ref64).max() / sc))
        err_orc = max(err_orc, float(np.abs(prob.out[rrow].astype(np.float64) - ref64).max() / sc))
    parity["plain_sum"] = {"max_rel_err_vs_oracle": ps["max_rel_err"], "bit_exact_rows": int(ex_rows.sum()),
                           "rows_le_1024_edges": int(short.sum()),
                           "all_rows_le_1024_bit_exact": bool(ex_rows[short].all()),
                           "rows_gt_1024_edges": int((~short).sum()), "long_rows_checked_vs_fp64": int(len(pick)),
                           "long_rows_rel_err_vs_fp64": {"gpu": err_gpu, "oracle_fp32_loop": err_orc}}
    # the wide-row kernels sum rows of <= 1024 slots in slot order (bit-exact is part of the bar); the narrow-row
    # kernel (column blocks of <= 64 floats) regroups a row's sum by 32-slot ranges: deterministic, equal to rounding
    need_exact = dl > 64
    parity["plain_sum"]["bit_exact_required"] = need_exact
    short_ok = parity["plain_sum"]["all_rows_le_1024_bit_exact"] if need_exact else \
        bool(parity_stats(gp[short], prob.out[short])["max_rel_err"] <= 1e-5)
    parity["pass"] = bool(parity["pass"] and short_ok and err_gpu <= 3e-5)
    parity["what"] = ("rank %d: GPU output rows [%d, %d) of the graph, columns [%d, %d) vs oracle/oracle_c.c on the same "
                      "edges and features" % (rank, lo, lo + n_s, c0, c0 + dl))
    if dist is not None:
        allp = [None] * world
        dist.all_gather_object(allp, parity)
        parity = {"pass": all(bool(q["pass"]) for q in allp), "tol": PARITY_TOL,
                  "max_rel_err": max(q["max_rel_err"] for q in allp),
                  "rows": sum(q["rows"] for q in allp),
                  "bit_exact_rows": sum(q["plain_sum"]["bit_exact_rows"] for q in allp), "per_rank": allp}
    else:
        parity["bit_exact_rows_gcn"] = parity["bit_exact_rows"]
        parity["bit_exact_rows"] = parity["plain_sum"]["bit_exact_rows"]
    return cpu, parity


def full_layer(args, torch, dist, pgl, ops, g, step, x, norm, dev, world, rank, rr, rc, r, c, n, n_loc, e, d, dl):
    """GCNConv(128,128,relu).forward.  N = 1: the public layer.  N > 1: aggregate my block (no exchange) ->
    all-to-all inside my row group ([rows, D/Rc] -> [rows/Rc, D]) -> dense transform + bias + ReLU of those rows."""
    kf = max(3, args.steps // 4)
    if world == 1:
        conv = pgl.nn.GCNConv(d, d, activation="relu").to(dev)
        with torch.no_grad():
            for _ in range(3):
                y = conv(g, x)
            torch.cuda.synchronize()
            f0, f1 = _ev(torch), _ev(torch)
            f0.record()
            for _ in range(kf):
                y = conv(g, x)
            f1.record()
            torch.cuda.synchronize()
            full_ms = f0.elapsed_time(f1) / kf
        del y
        return {"value": e / (full_ms * 1e-3), "unit": "edges/s", "ms": full_ms,
                "what": "GCNConv(128,128,relu).forward: aggregation + dense transform with bias + ReLU in its "
                        "epilogue (3xTF32 on tcgen05 tensor cores, csrc/linear_tcgen05.cu)"}
    from pgl_b200.distributed import ColumnShardedGraph
    groups = [dist.new_group(list(range(q * rc, (q + 1) * rc))) for q in range(rr)]   # every rank creates every group
    cs = ColumnShardedGraph(None, d, rc, c, group=groups[r])
    torch.manual_seed(7)
    w = (torch.randn(d, d, device=dev) / d ** 0.5).contiguous()
    b = torch.zeros(d, device=dev)

    def layer():
        agg = step()
        rows = cs.to_rows(agg) if rc > 1 else agg
        return ops.linear_tc(rows, w, b, "relu")

    with torch.no_grad():
        for _ in range(3):
            layer()
        torch.cuda.synchronize()
        dist.barrier()
        f0, f1 = _ev(torch), _ev(torch)
        f0.record()
        for _ in range(kf):
            layer()
        f1.record()
        torch.cuda.synchronize()
        dist.barrier()
        t = torch.tensor([f0.elapsed_time(f1) / kf], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        full_ms = float(t.item())
    return {"value": e / (full_ms * 1e-3), "unit": "edges/s", "ms": full_ms,
            "what": "GCN layer on the %d x %d grid: aggregate my block (no exchange) -> NCCL all-to-all inside my row group "
                    "to whole rows -> dense transform + bias + ReLU; output row-sharded [N/%d, %d].  Re-replicating the "
                    "output columns for a NEXT layer (all-gather across the %d row groups) is not included" %
                    (rr, rc, world, d, rr)}


def e2e_host(args, torch, dist, ops, g, fwd, x, norm, norm_dst, dev, world, rank, rr, rc, r, c, bounds, n, n_loc, e, dl):
    """Features start in pinned host memory and the result ends in pinned host memory, every step.
    N = 1: the public host-buffer API (HostAggregator.submit / wait pipelines successive steps; `single_call_ms` is
    one blocking Graph.send_recv_host).  N > 1: every rank uploads only ITS row block of its column block (the
    feature matrix crosses PCIe once in total, not once per row group), the row groups complete each other's
    replicas by an NCCL all-gather over NVLink (distributed.GridHostAggregator), then kernel and download."""
    if world == 1:
        x_host = torch.empty((n, dl), dtype=torch.float32, pin_memory=True)
        x_host.copy_(x)
        out_host = torch.empty((n_loc, dl), dtype=torch.float32, pin_memory=True)
        chunks = int(os.environ.get("PGLB_E2E_CHUNKS", "2"))
        blocking = g.host_aggregator(n, dl, chunks, 1)
        for _ in range(2):
            blocking(x_host, out_host, "sum", scale_src=norm, scale_dst=norm_dst)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        blocking(x_host, out_host, "sum", scale_src=norm, scale_dst=norm_dst)
        single_ms = (time.perf_counter() - t0) * 1e3
        ref = ops._spmm_raw(fwd["indptr"], fwd["cols"], x, n_loc, "sum", scale_src=norm, scale_dst=norm_dst,
                            max_degree=fwd["max_degree"], packed=ops._packed_of(fwd, x))
        diff_single = float((out_host.to(dev) - ref).abs().max().item())
        del blocking
        agg = ops.HostAggregator(fwd, n, n_loc, dl, dev, int(os.environ.get("PGLB_E2E_PIPE_CHUNKS", "1")), depth=2)
        submit = lambda: agg.submit(x_host, out_host, "sum", scale_src=norm, scale_dst=norm_dst)   # noqa: E731
        h2d, d2h = n * dl * 4, n_loc * dl * 4
        api = ("Graph.host_aggregator(...).submit / wait (sum + degree norms) on a resident graph: features from pinned "
               "host memory, result back in pinned host memory, every step; successive steps are double-buffered so the "
               "upload of step i+1 overlaps kernel + download of step i.  single_call_ms = one blocking "
               "Graph.send_recv_host call (%d column chunks)" % chunks)
    else:
        from pgl_b200.distributed import GridHostAggregator
        ub = [block_bounds(n, rr, q)[0] for q in range(rr)] + [n]    # upload split of the source rows: even blocks
        lo, hi = ub[r], ub[r + 1]
        x_host = torch.empty((hi - lo, dl), dtype=torch.float32, pin_memory=True)
        x_host.copy_(x[lo:hi])
        out_host = torch.empty((n_loc, dl), dtype=torch.float32, pin_memory=True)
        agg = GridHostAggregator(fwd, n, n_loc, dl, dev, rr, rc, r, c, ub)
        t0 = None
        for _ in range(2):
            agg.wait(agg.submit(x_host, out_host, "sum", scale_src=norm, scale_dst=norm_dst))
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        agg.wait(agg.submit(x_host, out_host, "sum", scale_src=norm, scale_dst=norm_dst))
        single_ms = (time.perf_counter() - t0) * 1e3
        ref = ops._spmm_raw(fwd["indptr"], fwd["cols"], x, n_loc, "sum", scale_src=norm, scale_dst=norm_dst,
                            max_degree=fwd["max_degree"], packed=ops._packed_of(fwd, x))
        diff_single = float((out_host.to(dev) - ref).abs().max().item())
        submit = lambda: agg.submit(x_host, out_host, "sum", scale_src=norm, scale_dst=norm_dst)   # noqa: E731
        h2d, d2h = (hi - lo) * dl * 4, n_loc * dl * 4
        api = ("distributed.GridHostAggregator.submit / wait: every rank uploads its row block of its column block from "
               "pinned host memory (the matrix crosses PCIe once in total), NCCL all-gather over NVLink completes the "
               "source replica of each row group, aggregation, output block back to pinned host memory; two buffer sets, "
               "upload of step i+1 overlaps step i.  single_call_ms = one step alone")
    out_host.zero_()
    for _ in range(2):
        agg.wait(submit())
    ke = max(3, min(args.steps, 8))
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    q0, q1 = _ev(torch), _ev(torch)
    q0.record()
    tickets = [submit() for _ in range(ke)]
    for t in tickets:
        torch.cuda.current_stream().wait_event(t)
    q1.record()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    e2e_ms = q0.elapsed_time(q1) / ke
    diff_pipe = float((out_host.to(dev) - ref).abs().max().item())
    del ref
    if dist is not None:
        t = torch.tensor([e2e_ms, single_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms, single_ms = float(t[0].item()), float(t[1].item())
        bt = torch.tensor([h2d, d2h], device=dev, dtype=torch.float64)
        dist.all_reduce(bt)
        h2d, d2h = int(bt[0].item()), int(bt[1].item())
    return {"value": e / (e2e_ms * 1e-3), "unit": "edges/s",
            "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
            "ms_per_step": e2e_ms, "steps": ke, "single_call_ms": single_ms,
            "max_abs_diff_vs_resident": max(diff_single, diff_pipe), "api": api}


# ------------------------------------------------------------------------------------------
# N > 1, 1-D row partition + halo exchange (round 1's layout; the north_star's METIS variant)
# ------------------------------------------------------------------------------------------

def bench_row_sharded(args, torch, dist, pgl, dev, world, rank):
    from pgl_b200.distributed import ShardedGraph
    from pgl_b200 import ops
    n, e, d = args.nodes, args.edges, args.dim
    hbm_gbs, peak_src = peaks()
    edges = gen_edges(torch, n, e, args.exponent, args.seed, dev)
    sg = ShardedGraph.from_global_edges(edges, n, world, rank, method=args.partition,
                                        mode=args.halo, overlap=args.overlap)
    torch.cuda.empty_cache()
    x_ext, x_local = sg.features(d)  # features live inside the exchange buffer: no staging copy
    x_full = gen_features(torch, n, d, args.seed + 1, dev)
    owned = sg.owned_global_ids() if hasattr(sg, "owned_global_ids") else None
    if owned is not None:
        x_local.copy_(x_full[owned])
    else:
        g0 = torch.Generator(device=dev)
        g0.manual_seed(args.seed + 1 + rank)
        x_local.copy_(torch.randn(sg.n_local, d, device=dev, generator=g0))
    norm_l = sg.local_norm()

    def step():
        return sg.gcn_aggregate(x_local, norm_l)

    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    sampler = ClockSampler(dev.index)
    sampler.start()
    l0 = ops.launch_count()
    total_ms, per, last = timed_steps(torch, step, args.steps, dist)
    launches = ops.launch_count() - l0
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"gcn_aggregate": last}, rank, world)
    del last
    ms = torch.tensor([total_ms], device=dev, dtype=torch.float64)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_step = float(ms.item()) / args.steps
    stats = sg.stats()
    allstats = [None] * world
    dist.all_gather_object(allstats, stats)
    comp = sg.time_split(x_local, norm_l, iters=3)
    allcomp = [None] * world
    dist.all_gather_object(allcomp, comp)
    value = e / (ms_step * 1e-3)
    # the timed kernel's own bytes (VERDICT r1 weak 7: no exchange term in the aggregation's roofline)
    b_alg = max(algorithmic_bytes(s["n_local"], s["e_local"], d) for s in allstats)
    agg_ms = max(c["aggregate_ms"] for c in allcomp)
    achieved = b_alg / (agg_ms * 1e-3) / 1e9

    parity = None
    if not args.no_cpu and owned is not None:
        try:
            # oracle on a sample of MY rows: global edges whose dst is one of my first rows
            lib = _load_oracle_c()
            k = min(int(owned.numel()), 20000)
            mine = owned[:k]
            sel = torch.zeros(n, dtype=torch.bool, device=dev)
            sel[mine] = True
            m = sel[edges[:, 1]]
            relabel = torch.full((n,), -1, dtype=torch.int64, device=dev)
            relabel[mine] = torch.arange(k, device=dev)
            src_np = np.ascontiguousarray(edges[m, 0].cpu().numpy())
            dst_np = np.ascontiguousarray(relabel[edges[m, 1]].cpu().numpy())
            indeg = torch.bincount(edges[:, 1], minlength=n)
            norm_ref = cpu_norm(indeg.cpu().numpy())
            xs = np.ascontiguousarray(x_full.cpu().numpy() * norm_ref[:, None])
            want = np.empty((k, d), np.float32)
            lib.orc_send_u_recv_f32(_ptr(xs), _ptr(src_np), _ptr(dst_np), _i64(len(src_np)), _i64(k), _i64(d), 0,
                                    _ptr(want))
            want *= norm_ref[mine.cpu().numpy()][:, None]
            got = step()[:k].cpu().numpy()
            parity = parity_stats(got, want)
            allp = [None] * world
            dist.all_gather_object(allp, parity)
            parity = {"pass": all(p["pass"] for p in allp), "tol": PARITY_TOL,
                      "max_rel_err": max(p["max_rel_err"] for p in allp), "rows": sum(p["rows"] for p in allp),
                      "bit_exact_rows": sum(p["bit_exact_rows"] for p in allp), "per_rank": allp}
        except Exception as ex:
            parity = {"pass": None, "error": repr(ex)[:300]}
    del x_full
    return {
        "metric": "edges/sec per GCN layer (128-d feat)", "value": value, "unit": "edges/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": workload_name(args), "l2": "inputs larger than L2",
                   "parallelism": "%d-way 1-D row partition (%s) + halo exchange (%s%s)" %
                                  (world, args.partition, sg.mode, ", overlapped" if sg.overlap else ""),
                   "per_rank": allstats, "time_split_ms": allcomp},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm_gbs, "unit": "GB/s",
                     "frac": achieved / hbm_gbs, "traffic": None, "peak_source": peak_src,
                     "note": "slowest rank's local aggregation kernel over its own algorithmic bytes; the "
                             "exchange is in time_split_ms"},
        "cpu_baseline": None, "parity": parity, "e2e": None,
        "gpu_launches": int(launches), "clocks": clocks,
    }


# ------------------------------------------------------------------------------------------
# cfg3: GATConv(128 -> 8 x 16) on RMAT scale 20 / 10M edges (BASELINE.json configs[2])
# ------------------------------------------------------------------------------------------

def bench_gat(args, torch, pgl, ops, GF, dev):
    n, e, H, Dh = 1 << 20, 10_000_000, 8, 16
    hbm_gbs, peak_src = peaks()
    edges = rmat_edges(torch, 20, e, seed=1, device=dev)
    g = pgl.Graph(edges=edges, num_nodes=n)
    x = gen_features(torch, n, 128, 2, dev)
    torch.manual_seed(3)
    conv = pgl.nn.GATConv(128, Dh, feat_drop=0, attn_drop=0, num_heads=H).to(dev)
    conv.eval()
    csr = g._fwd_csr()
    with torch.no_grad():
        f = (x @ conv.linear.weight + conv.linear.bias).reshape(-1, H, Dh).contiguous()
        a_s = (f * conv.weight_src).sum(-1).contiguous()
        a_d = (f * conv.weight_dst).sum(-1).contiguous()

        def step():
            return ops.gat_fused(csr, f, a_s, a_d, 0.2)

        for _ in range(max(args.warmup, 3)):
            step()
        sampler = ClockSampler(dev.index)
        sampler.start()
        l0 = ops.launch_count()
        total_ms, per, last = timed_steps(torch, step, args.steps)
        launches = ops.launch_count() - l0
        clocks = sampler.stop()
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"gat_aggregate": last})
        del last
        for _ in range(3):
            conv(g, x)
        torch.cuda.synchronize()
        f0, f1 = _ev(torch), _ev(torch)
        f0.record()
        for _ in range(5):
            conv(g, x)
        f1.record()
        torch.cuda.synchronize()
        layer_ms = f0.elapsed_time(f1) / 5
        # parity at full size: sampled rows against the oracle's op-by-op GAT aggregation
        parity = None
        if not args.no_cpu:
            try:
                parity = gat_parity(torch, edges, n, f, a_s, a_d, step(), H, Dh)
            except Exception as ex:
                parity = {"pass": None, "error": repr(ex)[:300]}
    training = gat_training_leg(torch, pgl, ops, GF, g, f, a_s, a_d, H, Dh)
    ms_step = total_ms / args.steps
    kern_ms = float(np.mean(per))
    # SURVEY 8d cfg3: per edge 8 + 32 + 512 + 32 (alpha write, training only) ; per node 32 + 512 + 8.
    # The single-pass inference kernel writes no alpha: 552 B/edge.
    b_alg = e * (8 + 32 + 512) + n * (32 + 512 + 8)
    achieved = b_alg / (kern_ms * 1e-3) / 1e9
    return {
        "metric": "edges/sec per GAT layer aggregation (8 heads x 16, edge softmax fused)", "value": e / (ms_step * 1e-3),
        "unit": "edges/s", "n_gpus": 1, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "cfg3 RMAT scale 20 (0.57,0.19,0.19,0.05), %d nodes / %d edges, GATConv(128 -> 8x16) eval: "
                               "single-pass attention + softmax + aggregation" % (n, e),
                   "max_in_degree": int(csr["max_degree"]), "l2": "features (0.5 GB) larger than L2"},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm_gbs, "unit": "GB/s", "frac": achieved / hbm_gbs,
                     "traffic": read_traffic("gat_fused_bytes_per_launch"), "peak_source": peak_src,
                     "algorithmic_bytes": b_alg, "kernel": "spmm_gat5_kernel (fused GAT, TMA gather4)",
                     "kernel_ms_mean": kern_ms,
                     "note": "SURVEY 8d cfg3 model without the alpha write (inference): E*552 + N*552 bytes; with the "
                             "training-time alpha write the model is 6.42 GB"},
        "parity": parity, "cpu_baseline": None, "e2e": None, "gpu_launches": int(launches), "clocks": clocks,
        "full_layer": {"ms": layer_ms, "value": e / (layer_ms * 1e-3), "unit": "edges/s",
                       "what": "GATConv.forward (linear + attention logits + fused aggregation)"},
        "training": training,
    }


def gat_training_leg(torch, pgl, ops, GF, g, f, a_s, a_d, H, Dh, iters=5):
    """Forward + backward of the attention + aggregation part of GATConv under autograd: the fused path
    (ops._GatFused: single-pass forward keeping lse, backward edge kernel + reverse-CSR aggregations) next to the
    op-by-op path (send_uv, LeakyReLU, edge_softmax, send_ue_recv, each with its own backward), and the largest
    relative difference between their gradients at full size."""
    try:
        go = gen_features(torch, f.shape[0], H * Dh, 7, f.device).reshape(-1, H, Dh)
        res = {}
        grads = {}
        for name in ("fused", "op_by_op"):
            fa, sa, da = [t.detach().clone().requires_grad_(True) for t in (f, a_s, a_d)]

            def one():
                for t in (fa, sa, da):
                    t.grad = None
                if name == "fused":
                    out = ops.gat_fused_train(g._fwd_csr(), g._bwd_csr, fa, sa, da, 0.2)
                else:
                    al = g.send_uv(sa, da, "add")
                    al = torch.nn.functional.leaky_relu(al, 0.2)
                    al = GF.edge_softmax(g, al)
                    out = g.send_ue_recv(fa, al.reshape(-1, H, 1), "mul", "sum")
                out.backward(go)

            with torch.enable_grad():
                one()
                one()
                torch.cuda.synchronize()
                e0, e1 = _ev(torch), _ev(torch)
                e0.record()
                for _ in range(iters):
                    one()
                e1.record()
                torch.cuda.synchronize()
            res[name + "_fwd_bwd_ms"] = e0.elapsed_time(e1) / iters
            grads[name] = [t.grad.detach().clone() for t in (fa, sa, da)]

        def rel(a, b):
            return float((a - b).abs().max() / b.abs().max().clamp(min=1e-30))
        res["grad_max_rel_diff"] = {k: rel(a, b) for k, a, b in zip(("f", "attn_src", "attn_dst"), grads["fused"],
                                                                     grads["op_by_op"])}
        res["pass"] = all(v <= 5e-4 for v in res["grad_max_rel_diff"].values())
        return res
    except Exception as ex:   # never lose the timing line to the extra leg
        return {"pass": None, "error": repr(ex)[:300]}


def gat_parity(torch, edges, n, f, a_s, a_d, got, H, Dh, rows=4096):
    """Oracle (numpy, op by op as pgl/nn/conv.py:308-346) on a row sample at full size."""
    dev = f.device
    g0 = torch.Generator(device=dev)
    g0.manual_seed(11)
    pick = torch.randperm(n, generator=g0, device=dev)[:rows]
    sel = torch.zeros(n, dtype=torch.bool, device=dev)
    sel[pick] = True
    m = sel[edges[:, 1]]
    src = edges[m, 0].cpu().numpy()
    dst = edges[m, 1].cpu().numpy()
    fn, asn, adn = f.cpu().numpy(), a_s.cpu().numpy(), a_d.cpu().numpy()
    order = np.argsort(dst, kind="stable")
    src, dst = src[order], dst[order]
    lg = asn[src] + adn[dst]
    lg = np.where(lg >= 0, lg, np.float32(0.2) * lg).astype(np.float32)
    want = np.zeros((n, H, Dh), np.float32)
    bounds = np.flatnonzero(np.r_[True, dst[1:] != dst[:-1], True])
    for i in range(len(bounds) - 1):
        lo, hi = bounds[i], bounds[i + 1]
        l = lg[lo:hi]
        ex = np.exp(l - l.max(axis=0, keepdims=True))
        al = (ex / ex.sum(axis=0, keepdims=True)).astype(np.float32)
        want[dst[lo]] = (fn[src[lo:hi]] * al[:, :, None]).sum(axis=0)
    pk = pick.cpu().numpy()
    return parity_stats(got.reshape(n, H * Dh)[pick].cpu().numpy(), want[pk].reshape(len(pk), H * Dh))


# ------------------------------------------------------------------------------------------
# cfg4: 3 x GraphSageConv(mean) 100 -> 128 -> 128 -> 47, products-shape stand-in (BASELINE.json configs[3])
# ------------------------------------------------------------------------------------------

def bench_sage(args, torch, dist, pgl, ops, GF, dev, world, rank):
    n, und = 2_449_029, 61_859_140
    hbm_gbs, peak_src = peaks()
    half = gen_edges(torch, n, und, 0.6, 5, dev)
    edges = torch.cat([half, half.flip(1)], 0)
    del half
    e = int(edges.shape[0])
    x = gen_features(torch, n, 100, 4, dev)
    dims = [100, 128, 128, 47]
    torch.manual_seed(6)
    layers = [pgl.nn.GraphSageConv(dims[i], dims[i + 1], aggr_func="mean").to(dev) for i in range(3)]
    if world > 1:
        return bench_sage_sharded(args, torch, dist, pgl, ops, dev, world, rank, edges, x, layers, dims, n, e)
    g = pgl.Graph(edges=edges, num_nodes=n)
    fwd = g._fwd_csr()

    def forward():
        h = x
        for i, conv in enumerate(layers):
            h = conv(g, h, act="relu" if i < 2 else None)
        return h

    per_layer = []
    with torch.no_grad():
        for _ in range(max(args.warmup, 3)):
            forward()
        sampler = ClockSampler(dev.index)
        sampler.start()
        l0 = ops.launch_count()
        total_ms, per, last = timed_steps(torch, forward, args.steps)
        launches = ops.launch_count() - l0
        clocks = sampler.stop()
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"sage_forward": last})
        del last
        h = x
        for i, conv in enumerate(layers):
            d = dims[i]
            agg = lambda: g.send_recv(h, "mean")   # noqa: E731
            for _ in range(3):
                agg()
            t_ms, p_, _ = timed_steps(torch, agg, 5)
            b_alg = e * (4 * d + 8) + n * 4 * d + (n + 1) * 8
            per_layer.append({"in": d, "out": dims[i + 1], "aggregation_ms": t_ms / 5,
                              "agg_alg_GBs": b_alg / (t_ms / 5) / 1e6,
                              "agg_roofline_frac": b_alg / (t_ms / 5) / 1e6 / hbm_gbs})
            h = conv(g, h, act="relu" if i < 2 else None)
        parity = None
        if not args.no_cpu:
            try:
                k = 20000
                lib = _load_oracle_c()
                m = edges[:, 1] < k
                src_np = np.ascontiguousarray(edges[m, 0].cpu().numpy())
                dst_np = np.ascontiguousarray(edges[m, 1].cpu().numpy())
                x_np = x.cpu().numpy()
                want = np.empty((k, 100), np.float32)
                lib.orc_send_u_recv_f32(_ptr(x_np), _ptr(src_np), _ptr(dst_np), _i64(len(src_np)), _i64(k), _i64(100), 1,
                                        _ptr(want))
                parity = parity_stats(g.send_recv(x, "mean")[:k].cpu().numpy(), want)
                parity["what"] = "layer-1 mean aggregation (400-byte rows), rows dst < %d vs oracle_c" % k
            except Exception as ex:
                parity = {"pass": None, "error": repr(ex)[:300]}
    ms_step = total_ms / args.steps
    agg0 = per_layer[0]
    return {
        "metric": "edges/sec per GraphSAGE forward (3 layers, mean aggregation)", "value": 3 * e / (ms_step * 1e-3),
        "unit": "edges/s", "n_gpus": 1, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "cfg4 ogbn-products-shape stand-in (Chung-Lu exp 0.6, symmetrised): %d nodes / %d directed "
                               "edges, X [N,100] f32; 3 x GraphSageConv(mean) 100->128->128->47, full-batch forward" % (n, e),
                   "max_in_degree": int(fwd["max_degree"]), "layers": per_layer,
                   "sector_note": "400-byte rows start on 16-byte, not 128-byte, boundaries: a row touches 13 or 14 "
                                  "32-byte sectors for 12.5 useful (sector efficiency 0.89-0.96)"},
        "roofline": {"bound": "hbm", "achieved": agg0["agg_alg_GBs"], "peak": hbm_gbs, "unit": "GB/s",
                     "frac": agg0["agg_roofline_frac"], "traffic": read_traffic("sage_l1_bytes_per_launch"),
                     "peak_source": peak_src, "kernel": kernel_name(e, n),
                     "note": "layer-1 mean aggregation (D = 100): E*(4D+8) + N*4D + (N+1)*8 = 416 B/edge model"},
        "parity": parity, "cpu_baseline": None, "e2e": None, "gpu_launches": int(launches), "clocks": clocks,
    }


def bench_sage_sharded(args, torch, dist, pgl, ops, dev, world, rank, edges, x, layers, dims, n, e):
    """cfg4 as north_star states it: METIS world-way row partition + halo exchange per layer (ShardedGraph),
    every rank owning its nodes' rows."""
    from pgl_b200.distributed import ShardedGraph
    hbm_gbs, peak_src = peaks()
    method = args.partition
    sg = ShardedGraph.from_global_edges(edges, n, world, rank, method=method, mode=args.halo, overlap=args.overlap)
    owned = sg.owned_global_ids()
    for conv in layers:   # same weights on every rank
        for p in conv.parameters():
            dist.broadcast(p.data, 0)
    bufs = {}

    import torch.nn.functional as F
    x_own = x[owned].contiguous()

    def forward():
        h = x_own
        for i, conv in enumerate(layers):
            d = dims[i]
            if d not in bufs:
                bufs[d] = sg.features(d)
            x_ext, x_local = bufs[d]
            x_local.copy_(h)
            neigh = sg.send_recv(x_local, "mean")            # halo exchange + local mean aggregation
            h = conv.self_linear(h) + conv.neigh_linear(neigh)   # reference pgl/nn/conv.py:106-115
            if i < 2:
                h = F.relu(h)
            h = F.normalize(h, dim=1)
        return h

    with torch.no_grad():
        for _ in range(max(args.warmup, 3)):
            forward()
        sampler = ClockSampler(dev.index)
        sampler.start()
        l0 = ops.launch_count()
        total_ms, per, last = timed_steps(torch, forward, args.steps, dist)
        launches = ops.launch_count() - l0
        clocks = sampler.stop()
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"sage_forward": last}, rank, world)
        del last
    t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / args.steps
    stats = sg.stats()
    allstats = [None] * world
    dist.all_gather_object(allstats, stats)
    parity = None
    if not args.no_cpu:
        try:   # layer-1 mean aggregation (halo exchange + local kernel) of my first rows vs the oracle on the global graph
            lib = _load_oracle_c()
            k = min(int(owned.numel()), 20000)
            mine = owned[:k]
            sel = torch.zeros(n, dtype=torch.bool, device=dev)
            sel[mine] = True
            m = sel[edges[:, 1]]
            relabel = torch.full((n,), -1, dtype=torch.int64, device=dev)
            relabel[mine] = torch.arange(k, device=dev)
            src_np = np.ascontiguousarray(edges[m, 0].cpu().numpy())
            dst_np = np.ascontiguousarray(relabel[edges[m, 1]].cpu().numpy())
            x_np = x.cpu().numpy()
            want = np.empty((k, dims[0]), np.float32)
            lib.orc_send_u_recv_f32(_ptr(x_np), _ptr(src_np), _ptr(dst_np), _i64(len(src_np)), _i64(k), _i64(dims[0]), 1,
                                    _ptr(want))
            x_ext, x_local = bufs[dims[0]]
            x_local.copy_(x_own)
            got = sg.send_recv(x_local, "mean")[:k].cpu().numpy()
            p1 = parity_stats(got, want)
            allp = [None] * world
            dist.all_gather_object(allp, p1)
            parity = {"pass": all(q["pass"] for q in allp), "tol": PARITY_TOL,
                      "max_rel_err": max(q["max_rel_err"] for q in allp), "rows": sum(q["rows"] for q in allp),
                      "bit_exact_rows": sum(q["bit_exact_rows"] for q in allp),
                      "what": "layer-1 mean aggregation incl. the halo exchange, first %d owned rows of every rank vs oracle_c" % k}
        except Exception as ex:
            parity = {"pass": None, "error": repr(ex)[:300]}
    return {
        "metric": "edges/sec per GraphSAGE forward (3 layers, mean aggregation)", "value": 3 * e / (ms_step * 1e-3),
        "unit": "edges/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "cfg4 products-shape stand-in, %d nodes / %d directed edges, 3 x GraphSageConv(mean)" % (n, e),
                   "parallelism": "%d-way %s row partition + halo exchange (%s) per layer" % (world, method, sg.mode),
                   "per_rank": allstats},
        "roofline": {"bound": "hbm", "achieved": None, "peak": hbm_gbs, "unit": "GB/s", "frac": None, "traffic": None,
                     "peak_source": peak_src, "note": "multi-layer sharded forward: see per_rank for halo sizes"},
        "parity": parity, "cpu_baseline": None, "e2e": None, "gpu_launches": int(launches), "clocks": clocks,
    }


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        main_reference(a)
    else:
        main_ours(a)
