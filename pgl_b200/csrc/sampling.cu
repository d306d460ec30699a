// sampling.cu -- neighbour sampling + reindex for mini-batch GraphSAGE (SURVEY 8f rank 4).
// Replaces `paddle.geometric.sample_neighbors` and `paddle.geometric.reindex_graph` as called by the
// reference's GPU sampler (pgl/sampling/sage.py:130-155, NeighborSampler.sample_neighbors), on the
// cached dst-CSR (`row` = adj_dst_index._sorted_v, `colptr` = adj_dst_index._indptr).
//
// sample_neighbors: one warp per input node.  deg <= k (or k < 0): the whole neighbour list, in CSR
// order.  deg > k: a uniform k-subset WITHOUT replacement by Floyd's algorithm (k draws, each checked
// against the at most k positions already chosen, warp-parallel) -- O(k) work however long the row is,
// so a 10^6-edge hub costs the same as a 30-edge row.  Draws come from a counter-based hash of
// (seed, input position, draw), so the result is a pure function of the arguments.
//
// reindex_graph: ids are compacted in first-appearance order (input nodes first, then new neighbours in
// the order they occur) like Paddle's op, with a dense lookup table instead of a hash map: the caller
// owns a `table` of num_nodes int64 filled with INT64_MAX; the call leaves it filled with INT64_MAX
// again (only touched entries are reset), so it is allocated once per graph.
//
// Runs on hardware and is tested there (tests/test_gpu_sampling.py, DESIGN.md section 4.11); the CPU restatement of
// both kernels is tests/test_sampling_model.py.
#include <limits.h>

#include "common.cuh"

namespace pglb {

__device__ __forceinline__ unsigned long long mix64(unsigned long long z) {
    z += 0x9e3779b97f4a7c15ull;
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
    return z ^ (z >> 31);
}

__global__ void __launch_bounds__(256) sample_count_kernel(const int64_t *__restrict__ indptr,
                                                           const int64_t *__restrict__ nodes, int64_t n,
                                                           int64_t k, int64_t *__restrict__ count) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t v = nodes[i];
    const int64_t deg = indptr[v + 1] - indptr[v];
    count[i] = (k < 0 || deg <= k) ? deg : k;
}

// offsets = exclusive scan of count.  Dynamic shared memory: warps * k ints (chosen positions).
__global__ void __launch_bounds__(256) sample_fill_kernel(const int64_t *__restrict__ indptr,
                                                          const int64_t *__restrict__ row,
                                                          const int64_t *__restrict__ eid,
                                                          const int64_t *__restrict__ nodes, int64_t n,
                                                          int64_t k, unsigned long long seed,
                                                          const int64_t *__restrict__ offsets,
                                                          int64_t *__restrict__ out_neighbors,
                                                          int64_t *__restrict__ out_eids) {
    extern __shared__ int chosen_all[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    const int64_t i = (int64_t)blockIdx.x * wpb + warp;
    if (i >= n) return;
    const int64_t v = nodes[i];
    const int64_t start = indptr[v];
    const int64_t deg = indptr[v + 1] - start;
    const int64_t o = offsets[i];
    if (k < 0 || deg <= k) {
        for (int64_t j = lane; j < deg; j += 32) {
            out_neighbors[o + j] = row[start + j];
            if (out_eids) out_eids[o + j] = eid ? eid[start + j] : start + j;
        }
        return;
    }
    int *chosen = chosen_all + (size_t)warp * k;
    // Floyd: for j = deg-k .. deg-1: t = U[0, j]; insert t unless already chosen, else insert j
    const unsigned long long base = mix64(seed ^ mix64((unsigned long long)i));
    for (int64_t c = 0; c < k; ++c) {
        const int64_t j = deg - k + c;
        const unsigned long long r = mix64(base + (unsigned long long)c);
        int t = (int)__umul64hi(r, (unsigned long long)(j + 1));
        bool hit = false;
        for (int64_t q = lane; q < c; q += 32) hit |= (chosen[q] == t);
        if (__any_sync(0xffffffffu, hit)) t = (int)j;
        if (lane == 0) chosen[c] = t;
        __syncwarp();
    }
    for (int64_t c = lane; c < k; c += 32) {
        const int64_t p = start + chosen[c];
        out_neighbors[o + c] = row[p];
        if (out_eids) out_eids[o + c] = eid ? eid[p] : p;
    }
}

// ---- reindex ---------------------------------------------------------------------------------------
constexpr long long RX_EMPTY = LLONG_MAX;

__global__ void __launch_bounds__(256) rx_mark_seeds_kernel(const int64_t *__restrict__ x, int64_t n,
                                                            long long *__restrict__ table) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) table[x[i]] = i;
}

__global__ void __launch_bounds__(256) rx_first_pos_kernel(const int64_t *__restrict__ nb, int64_t m,
                                                           int64_t n, long long *__restrict__ table) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p < m) atomicMin(table + nb[p], (long long)(n + p));  // seeds hold a value < n: untouched
}

__global__ void __launch_bounds__(256) rx_flag_kernel(const int64_t *__restrict__ nb, int64_t m, int64_t n,
                                                      const long long *__restrict__ table,
                                                      int64_t *__restrict__ flag) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p < m) flag[p] = (table[nb[p]] == (long long)(n + p)) ? 1 : 0;
}

// rank = exclusive scan of flag.  dst[p] = input position owning slot p (binary search in offsets).
__global__ void __launch_bounds__(256) rx_emit_kernel(const int64_t *__restrict__ x, const int64_t *__restrict__ nb,
                                                      const int64_t *__restrict__ offsets, int64_t n, int64_t m,
                                                      const long long *__restrict__ table,
                                                      const int64_t *__restrict__ flag,
                                                      const int64_t *__restrict__ rank,
                                                      int64_t *__restrict__ src, int64_t *__restrict__ dst,
                                                      int64_t *__restrict__ out_nodes,
                                                      int64_t *__restrict__ num_out) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p < n) out_nodes[p] = x[p];
    if (p == 0) *num_out = n + (m > 0 ? rank[m - 1] + flag[m - 1] : 0);
    if (p >= m) return;
    const int64_t v = nb[p];
    const long long t = table[v];
    if (t < n) {
        src[p] = t;
    } else {
        const int64_t id = n + rank[t - n];
        src[p] = id;
        if (flag[p]) out_nodes[id] = v;
    }
    int64_t lo = 0, hi = n;  // last i with offsets[i] <= p  (offsets has n + 1 entries, offsets[n] = m)
    while (hi - lo > 1) {
        const int64_t mid = (lo + hi) >> 1;
        if (offsets[mid] <= p) lo = mid; else hi = mid;
    }
    dst[p] = lo;
}

__global__ void __launch_bounds__(256) rx_reset_kernel(const int64_t *__restrict__ x, int64_t n,
                                                       const int64_t *__restrict__ nb, int64_t m,
                                                       long long *__restrict__ table) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p < n) table[x[p]] = RX_EMPTY;
    if (p < m) table[nb[p]] = RX_EMPTY;
}

__global__ void __launch_bounds__(256) fill_i64_kernel(long long *p, int64_t n, long long v) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        p[i] = v;
}

// single-block exclusive scan is enough for mini-batch sizes; large inputs go through 2048-wide tiles
__global__ void __launch_bounds__(1024) small_exclusive_scan_kernel(const int64_t *__restrict__ in, int64_t n,
                                                                    int64_t *__restrict__ out,
                                                                    int64_t *__restrict__ total) {
    __shared__ int64_t wsum[32];
    __shared__ int64_t carry_s;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    for (int64_t b0 = 0; b0 < n; b0 += 1024) {
        const int64_t i = b0 + threadIdx.x;
        const int64_t v = i < n ? in[i] : 0;
        int64_t incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int64_t t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) wsum[w] = incl;
        __syncthreads();
        int64_t base = 0, tot = 0;
        for (int j = 0; j < 32; ++j) {
            if (j < w) base += wsum[j];
            tot += wsum[j];
        }
        const int64_t c = carry_s;
        if (i < n) out[i] = c + base + incl - v;
        __syncthreads();
        if (threadIdx.x == 0) carry_s = c + tot;
        __syncthreads();
    }
    if (threadIdx.x == 0 && total) *total = carry_s;
}

static inline unsigned blocks_for(int64_t n, int t = 256) { return (unsigned)std::max<int64_t>((n + t - 1) / t, 1); }

}  // namespace pglb

using namespace pglb;

extern "C" int pglb_sample_count(const int64_t *indptr, const int64_t *nodes, int64_t n, int64_t sample_size,
                                 int64_t *count, int64_t *offsets, void *stream) {
    PGLB_CHECK_ARG(n >= 0, PGLB_EINVAL, "pglb_sample_count: negative node count");
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    PGLB_CHECK_ARG(offsets, PGLB_EINVAL, "pglb_sample_count: NULL offsets");
    if (n > 0) {
        PGLB_CHECK_ARG(indptr && nodes && count, PGLB_EINVAL, "pglb_sample_count: NULL pointer");
        sample_count_kernel<<<blocks_for(n), 256, 0, s>>>(indptr, nodes, n, sample_size, count);
        PGLB_LAUNCH_CHECK("sample_count_kernel");
    }
    // offsets[0..n) = exclusive scan, offsets[n] = total
    small_exclusive_scan_kernel<<<1, 1024, 0, s>>>(count, n, offsets, offsets + n);
    PGLB_LAUNCH_CHECK("small_exclusive_scan_kernel");
    return PGLB_OK;
}

extern "C" int pglb_sample_fill(const int64_t *indptr, const int64_t *row, const int64_t *eid,
                                const int64_t *nodes, int64_t n, int64_t sample_size, uint64_t seed,
                                const int64_t *offsets, int64_t *out_neighbors, int64_t *out_eids,
                                void *stream) {
    PGLB_CHECK_ARG(n >= 0, PGLB_EINVAL, "pglb_sample_fill: negative node count");
    PGLB_CHECK_ARG(sample_size <= 4096, PGLB_ESHAPE,
                   "pglb_sample_fill: sample_size %lld > 4096 is not supported", (long long)sample_size);
    if (n == 0) return PGLB_OK;
    PGLB_CHECK_ARG(indptr && row && nodes && offsets && out_neighbors, PGLB_EINVAL,
                   "pglb_sample_fill: NULL pointer");
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    const int64_t k = sample_size;
    int wpb = 8;
    if (k > 0) wpb = (int)std::max<int64_t>(1, std::min<int64_t>(8, (48 * 1024) / (k * 4)));
    const size_t smem = k > 0 ? (size_t)wpb * (size_t)k * sizeof(int) : 0;
    const unsigned grid = (unsigned)((n + wpb - 1) / wpb);
    sample_fill_kernel<<<grid, wpb * 32, smem, s>>>(indptr, row, eid, nodes, n, k, (unsigned long long)seed,
                                                    offsets, out_neighbors, out_eids);
    PGLB_LAUNCH_CHECK("sample_fill_kernel");
    return PGLB_OK;
}

extern "C" int pglb_reindex_table_init(int64_t *table, int64_t num_nodes, void *stream) {
    PGLB_CHECK_ARG(num_nodes >= 0 && (table || num_nodes == 0), PGLB_EINVAL, "pglb_reindex_table_init: bad argument");
    if (num_nodes == 0) return PGLB_OK;
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    const unsigned grid = (unsigned)std::min<int64_t>((num_nodes + 255) / 256, (int64_t)sm_count() * 16);
    fill_i64_kernel<<<grid, 256, 0, s>>>(reinterpret_cast<long long *>(table), num_nodes, RX_EMPTY);
    PGLB_LAUNCH_CHECK("fill_i64_kernel");
    return PGLB_OK;
}

extern "C" int pglb_reindex_graph_ws(int64_t num_neighbors, size_t *ws_bytes) {
    PGLB_CHECK_ARG(num_neighbors >= 0 && ws_bytes, PGLB_EINVAL, "pglb_reindex_graph_ws: bad argument");
    *ws_bytes = 2 * align_up(sizeof(int64_t) * (size_t)std::max<int64_t>(num_neighbors, 1), 256);
    return PGLB_OK;
}

extern "C" int pglb_reindex_graph(const int64_t *x, int64_t n, const int64_t *neighbors,
                                  const int64_t *offsets, int64_t m, int64_t *table, int64_t *reindex_src,
                                  int64_t *reindex_dst, int64_t *out_nodes, int64_t *num_out, void *ws,
                                  size_t ws_bytes, void *stream) {
    PGLB_CHECK_ARG(n >= 0 && m >= 0, PGLB_EINVAL, "pglb_reindex_graph: negative size");
    PGLB_CHECK_ARG(num_out && (n == 0 || (x && out_nodes && table)), PGLB_EINVAL, "pglb_reindex_graph: NULL pointer");
    PGLB_CHECK_ARG(m == 0 || (neighbors && offsets && reindex_src && reindex_dst && table && n > 0),
                   PGLB_EINVAL, "pglb_reindex_graph: NULL pointer");
    size_t need = 0;
    pglb_reindex_graph_ws(m, &need);
    PGLB_CHECK_ARG(ws_bytes >= need && (ws || m == 0), PGLB_EWORKSPACE,
                   "pglb_reindex_graph: workspace of %zu bytes needed (got %zu)", need, ws_bytes);
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    long long *tab = reinterpret_cast<long long *>(table);
    int64_t *flag = reinterpret_cast<int64_t *>(ws);
    int64_t *rank = reinterpret_cast<int64_t *>(reinterpret_cast<char *>(ws) + need / 2);
    if (n > 0) {
        rx_mark_seeds_kernel<<<blocks_for(n), 256, 0, s>>>(x, n, tab);
        PGLB_LAUNCH_CHECK("rx_mark_seeds_kernel");
    }
    if (m > 0) {
        rx_first_pos_kernel<<<blocks_for(m), 256, 0, s>>>(neighbors, m, n, tab);
        PGLB_LAUNCH_CHECK("rx_first_pos_kernel");
        rx_flag_kernel<<<blocks_for(m), 256, 0, s>>>(neighbors, m, n, tab, flag);
        PGLB_LAUNCH_CHECK("rx_flag_kernel");
        small_exclusive_scan_kernel<<<1, 1024, 0, s>>>(flag, m, rank, nullptr);
        PGLB_LAUNCH_CHECK("small_exclusive_scan_kernel");
    }
    const int64_t span = std::max(n, m);
    rx_emit_kernel<<<blocks_for(span), 256, 0, s>>>(x, neighbors, offsets, n, m, tab, flag, rank, reindex_src,
                                                    reindex_dst, out_nodes, num_out);
    PGLB_LAUNCH_CHECK("rx_emit_kernel");
    if (span > 0) {
        rx_reset_kernel<<<blocks_for(span), 256, 0, s>>>(x, n, neighbors, m, tab);
        PGLB_LAUNCH_CHECK("rx_reset_kernel");
    }
    return PGLB_OK;
}
