// walk.cu -- random walks (uniform, node2vec, node2vec+) and skip-gram pairs: the input pipeline of DeepWalk /
// node2vec (reference pgl/sampling/walk.py:23-183, pgl/graph_kernel.pyx:142-224 node2vec_sample /
// node2vec_plus_sample, pgl/graph_kernel.pyx:343-364 skip_gram_gen_pair).
//
// Walks read the row-sorted successor CSR (the src-CSR's indptr, each row's columns ascending), so "is x a
// successor of v" is a binary search.  Every draw comes from the counter-based hash documented in include/pglb.h,
// and all sampling arithmetic is integer: the host twin (pglb_random_walk_host, same file) and the kernels share
// the step functions below and produce the same walks bit for bit.
//
// Kernel: one walk per thread, the walk's state in registers, a grid-stride loop over warps of 32 walks.  The
// node2vec kernels keep a warp's lanes on the same step so that a step whose 32 rejection draws all failed can run
// the exact inverse-CDF fallback over the row with the whole warp (two passes of a 32-wide integer prefix sum).
#include <math.h>

#include "common.cuh"

namespace pglb {
namespace {

constexpr int WALK_T = 256;
// blocks per SM each kernel is built for: the uniform kernel fits 32 registers (2048 threads an SM); the node2vec
// kernels need about 53 without spills (1024 threads an SM)
template <int MODE>
constexpr int walk_blocks_per_sm() { return MODE == PGLB_WALK_UNIFORM ? 8 : 4; }
constexpr unsigned FULL = 0xffffffffu;

__host__ __device__ __forceinline__ uint64_t wmix64(uint64_t z) {
    z += 0x9e3779b97f4a7c15ull;
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
    return z ^ (z >> 31);
}

__host__ __device__ __forceinline__ uint64_t mulhi64(uint64_t a, uint64_t b) {
#ifdef __CUDA_ARCH__
    return __umul64hi(a, b);
#else
    return (uint64_t)(((unsigned __int128)a * b) >> 64);
#endif
}

// word k of step t of the walk whose base is wb = wmix64(seed ^ wmix64(i))
__host__ __device__ __forceinline__ uint64_t walk_word(uint64_t wb, int64_t t, int k) {
    return wmix64(wb + (uint64_t)t * PGLB_WALK_WORDS_PER_STEP + (uint64_t)k);
}

// cols[lo, hi) is ascending: binary search for x
__host__ __device__ __forceinline__ bool row_has(const int64_t *cols, int64_t lo, int64_t hi, int64_t x) {
    while (lo < hi) {
        const int64_t mid = lo + ((hi - lo) >> 1);
        const int64_t c = cols[mid];
        if (c == x) return true;
        if (c < x) lo = mid + 1; else hi = mid;
    }
    return false;
}

// Threshold of candidate x at step t >= 1 of a walk whose nodes so far are hist[0..t] (hist[t] = current node):
// class 0 (x is the previous node) -> T0, class 1 (x in the seen set) -> T1, otherwise T2.
template <int MODE>
__host__ __device__ __forceinline__ uint64_t walk_threshold(int64_t x, const int64_t *hist, int64_t t,
                                                            const int64_t *indptr, const int64_t *cols, uint64_t T0,
                                                            uint64_t T1, uint64_t T2) {
    const int64_t prev = hist[t - 1];
    if (x == prev) return T0;
    if constexpr (MODE == PGLB_WALK_NODE2VEC) {
        return row_has(cols, indptr[prev], indptr[prev + 1], x) ? T1 : T2;
    } else {
        for (int64_t k = 0; k < t; ++k) {  // node2vec+: the successors of every earlier node
            const int64_t v = hist[k];
            if (row_has(cols, indptr[v], indptr[v + 1], x)) return T1;
        }
        return T2;
    }
}

// ---- device ------------------------------------------------------------------------------------------------

__device__ __forceinline__ uint64_t warp_incl_scan(uint64_t v, int lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint64_t u = __shfl_up_sync(FULL, v, o);
        if (lane >= o) v += u;
    }
    return v;
}

template <int MODE>
__global__ void __launch_bounds__(WALK_T, walk_blocks_per_sm<MODE>()) walk_kernel(const int64_t *__restrict__ indptr,
                                                      const int64_t *__restrict__ cols, int64_t N,
                                                      const int64_t *__restrict__ nodes, int64_t n, int64_t steps,
                                                      uint64_t seed, uint64_t T0, uint64_t T1, uint64_t T2,
                                                      int64_t *out, int64_t ldo) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t base = warp * 32; base < n; base += nwarps * 32) {  // warp-uniform loop
        const int64_t i = base + lane;
        const bool valid = i < n;
        int64_t *row = out + (valid ? i : 0) * ldo;
        int64_t cur = valid ? nodes[i] : -1;
        if (cur >= N) cur = -1;  // callers reject such ids; a row of -1 rather than a wild read
        if (valid) row[0] = cur;
        const uint64_t wb = wmix64(seed ^ wmix64((uint64_t)i));
        bool alive = cur >= 0;
        int64_t len = alive ? 1 : 0;
        for (int64_t t = 0; t < steps; ++t) {
            if (MODE == PGLB_WALK_UNIFORM) {
                if (!alive) break;
            } else if (!__any_sync(FULL, alive)) {
                break;
            }
            int64_t nxt = -1, s = 0, d = 0;
            bool fb = false;
            if (alive) {
                s = __ldg(indptr + cur);
                d = __ldg(indptr + cur + 1) - s;
                if (d == 0) {
                    alive = false;
                } else if (MODE == PGLB_WALK_UNIFORM || t == 0) {
                    nxt = __ldg(cols + s + (int64_t)mulhi64(walk_word(wb, t, 0), (uint64_t)d));
                } else {
                    fb = true;
                    for (int k = 0; k < PGLB_WALK_MAX_REJECT; ++k) {
                        const int64_t x = __ldg(cols + s + (int64_t)mulhi64(walk_word(wb, t, 2 * k), (uint64_t)d));
                        const uint64_t T = walk_threshold<MODE>(x, row, t, indptr, cols, T0, T1, T2);
                        if ((walk_word(wb, t, 2 * k + 1) >> 32) < T) {
                            nxt = x;
                            fb = false;
                            break;
                        }
                    }
                }
            }
            if (MODE != PGLB_WALK_UNIFORM) {
                __syncwarp();  // the fallback reads other lanes' rows
                unsigned m = __ballot_sync(FULL, fb);
                while (m) {
                    const int src = __ffs(m) - 1;
                    m &= m - 1;
                    const int64_t s_ = __shfl_sync(FULL, s, src), d_ = __shfl_sync(FULL, d, src);
                    const int64_t *h = out + __shfl_sync(FULL, i, src) * ldo;
                    const uint64_t wb_ = __shfl_sync(FULL, wb, src);
                    uint64_t tot = 0;
                    for (int64_t j = lane; j < d_; j += 32)
                        tot += walk_threshold<MODE>(__ldg(cols + s_ + j), h, t, indptr, cols, T0, T1, T2);
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(FULL, tot, o);
                    const uint64_t target = mulhi64(walk_word(wb_, t, 2 * PGLB_WALK_MAX_REJECT), tot);
                    uint64_t carry = 0;
                    int64_t pick = 0;
                    for (int64_t j0 = 0; j0 < d_; j0 += 32) {
                        const int64_t j = j0 + lane;
                        const uint64_t w =
                            j < d_ ? walk_threshold<MODE>(__ldg(cols + s_ + j), h, t, indptr, cols, T0, T1, T2) : 0;
                        const uint64_t incl = warp_incl_scan(w, lane);
                        const unsigned hit = __ballot_sync(FULL, j < d_ && carry + incl > target);
                        if (hit) {
                            pick = j0 + __ffs(hit) - 1;
                            break;
                        }
                        carry += __shfl_sync(FULL, incl, 31);
                    }
                    if (lane == src) nxt = __ldg(cols + s_ + pick);
                }
            }
            if (alive) {
                row[t + 1] = nxt;
                cur = nxt;
                len = t + 2;
            }
        }
        if (valid)
            for (int64_t k = len; k <= steps; ++k) row[k] = -1;
    }
}

// ---- skip-gram ---------------------------------------------------------------------------------------------

// len[w] = entries of row w before its first -1
__global__ void __launch_bounds__(256) sg_len_kernel(const int64_t *__restrict__ walks, int64_t n, int64_t W,
                                                     int64_t ldw, int64_t *__restrict__ len) {
    for (int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; w < n; w += (int64_t)gridDim.x * blockDim.x) {
        const int64_t *row = walks + w * ldw;
        int64_t l = 0;
        while (l < W && row[l] != -1) ++l;
        len[w] = l;
    }
}

__device__ __forceinline__ void sg_window(const int64_t *__restrict__ len, int64_t W, int64_t win, uint64_t seed,
                                          int64_t p, int64_t &w, int64_t &i, int64_t &lo, int64_t &hi) {
    w = p / W;
    i = p - w * W;
    const int64_t l = len[w];
    if (i >= l) {
        lo = 1;
        hi = 0;
        return;
    }
    const int64_t r = 1 + (int64_t)mulhi64(wmix64(wmix64(seed ^ wmix64((uint64_t)w)) + (uint64_t)i), (uint64_t)win);
    lo = i - r < 0 ? 0 : i - r;
    hi = i + r > l - 1 ? l - 1 : i + r;
}

// offsets[p + 1] = number of pairs position p emits; offsets[0] = 0
__global__ void __launch_bounds__(256) sg_count_kernel(const int64_t *__restrict__ walks, int64_t n, int64_t W,
                                                       int64_t ldw, int64_t win, uint64_t seed,
                                                       const int64_t *__restrict__ len, int64_t *__restrict__ offsets) {
    const int64_t m = n * W;
    for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < m; p += (int64_t)gridDim.x * blockDim.x) {
        int64_t w, i, lo, hi;
        sg_window(len, W, win, seed, p, w, i, lo, hi);
        const int64_t *row = walks + w * ldw;
        int64_t c = 0;
        if (lo <= hi) {
            const int64_t a = row[i];
            for (int64_t j = lo; j <= hi; ++j) c += row[j] != a;
        }
        offsets[p + 1] = c;
        if (p == 0) offsets[0] = 0;
    }
}

__global__ void __launch_bounds__(256) sg_fill_kernel(const int64_t *__restrict__ walks, int64_t n, int64_t W,
                                                      int64_t ldw, int64_t win, uint64_t seed,
                                                      const int64_t *__restrict__ len,
                                                      const int64_t *__restrict__ offsets, int64_t *__restrict__ src,
                                                      int64_t *__restrict__ dst) {
    const int64_t m = n * W;
    for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < m; p += (int64_t)gridDim.x * blockDim.x) {
        int64_t w, i, lo, hi;
        sg_window(len, W, win, seed, p, w, i, lo, hi);
        const int64_t *row = walks + w * ldw;
        int64_t o = offsets[p];
        if (lo > hi) continue;
        const int64_t a = row[i];
        for (int64_t j = lo; j <= hi; ++j) {
            const int64_t b = row[j];
            if (b == a) continue;
            src[o] = a;
            dst[o] = b;
            ++o;
        }
    }
}

inline unsigned grid_for(int64_t items, int per_sm_blocks) {
    const int64_t want = (items + 255) / 256;
    return (unsigned)std::max<int64_t>(1, std::min<int64_t>(want, (int64_t)sm_count() * per_sm_blocks));
}

// 2^32 * w / max(w) for w = (1/p, 1, 1/q), at least 1 so that every candidate keeps a non-zero weight
void walk_thresholds(double p, double q, uint64_t *T) {
    const double w[3] = {1.0 / p, 1.0, 1.0 / q};
    const double M = fmax(w[0], fmax(w[1], w[2]));
    for (int c = 0; c < 3; ++c) {
        const double v = floor(w[c] / M * 4294967296.0);
        T[c] = v < 1.0 ? 1 : (uint64_t)v;
    }
}

int walk_check(const char *who, int64_t N, int64_t n, int64_t steps, int mode, double p, double q, int64_t ldo,
               const void *indptr, const void *nodes, const void *out) {
    PGLB_CHECK_ARG(N >= 0 && n >= 0 && steps >= 0, PGLB_EINVAL, "%s: negative size", who);
    PGLB_CHECK_ARG(mode == PGLB_WALK_UNIFORM || mode == PGLB_WALK_NODE2VEC || mode == PGLB_WALK_NODE2VEC_PLUS,
                   PGLB_EINVAL, "%s: unknown mode %d", who, mode);
    PGLB_CHECK_ARG(mode == PGLB_WALK_UNIFORM || (isfinite(p) && isfinite(q) && p > 0 && q > 0), PGLB_EINVAL,
                   "%s: p and q must be finite and > 0", who);
    PGLB_CHECK_ARG(ldo >= steps + 1, PGLB_ESHAPE, "%s: ldo %lld < steps + 1", who, (long long)ldo);
    PGLB_CHECK_ARG(n == 0 || (indptr && nodes && out), PGLB_EINVAL, "%s: NULL pointer", who);
    return PGLB_OK;
}

}  // namespace
}  // namespace pglb

using namespace pglb;

extern "C" int pglb_random_walk(const int64_t *indptr, const int64_t *cols, int64_t N, const int64_t *nodes, int64_t n,
                                int64_t steps, int mode, double p, double q, uint64_t seed, int64_t *out, int64_t ldo,
                                void *stream) {
    const int rc = walk_check("pglb_random_walk", N, n, steps, mode, p, q, ldo, indptr, nodes, out);
    if (rc != PGLB_OK || n == 0) return rc;
    uint64_t T[3] = {1, 1, 1};
    if (mode != PGLB_WALK_UNIFORM) walk_thresholds(p, q, T);
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    const unsigned grid = grid_for(n, mode == PGLB_WALK_UNIFORM ? walk_blocks_per_sm<PGLB_WALK_UNIFORM>()
                                                                : walk_blocks_per_sm<PGLB_WALK_NODE2VEC>());
    if (mode == PGLB_WALK_UNIFORM)
        walk_kernel<PGLB_WALK_UNIFORM><<<grid, WALK_T, 0, s>>>(indptr, cols, N, nodes, n, steps, seed, T[0], T[1],
                                                               T[2], out, ldo);
    else if (mode == PGLB_WALK_NODE2VEC)
        walk_kernel<PGLB_WALK_NODE2VEC><<<grid, WALK_T, 0, s>>>(indptr, cols, N, nodes, n, steps, seed, T[0], T[1],
                                                                T[2], out, ldo);
    else
        walk_kernel<PGLB_WALK_NODE2VEC_PLUS><<<grid, WALK_T, 0, s>>>(indptr, cols, N, nodes, n, steps, seed, T[0],
                                                                     T[1], T[2], out, ldo);
    PGLB_LAUNCH_CHECK("walk_kernel");
    return PGLB_OK;
}

template <int MODE>
static void walk_host(const int64_t *indptr, const int64_t *cols, const int64_t *nodes, int64_t n, int64_t steps,
                      uint64_t seed, const uint64_t *T, int64_t *out, int64_t ldo) {
    for (int64_t i = 0; i < n; ++i) {
        int64_t *row = out + i * ldo;
        int64_t cur = nodes[i];
        row[0] = cur;
        const uint64_t wb = wmix64(seed ^ wmix64((uint64_t)i));
        int64_t len = 1;
        for (int64_t t = 0; t < steps; ++t) {
            const int64_t s = indptr[cur], d = indptr[cur + 1] - s;
            if (d == 0) break;
            int64_t nxt = -1;
            if (MODE == PGLB_WALK_UNIFORM || t == 0) {
                nxt = cols[s + (int64_t)mulhi64(walk_word(wb, t, 0), (uint64_t)d)];
            } else {
                for (int k = 0; k < PGLB_WALK_MAX_REJECT && nxt < 0; ++k) {
                    const int64_t x = cols[s + (int64_t)mulhi64(walk_word(wb, t, 2 * k), (uint64_t)d)];
                    if ((walk_word(wb, t, 2 * k + 1) >> 32) < walk_threshold<MODE>(x, row, t, indptr, cols, T[0], T[1], T[2]))
                        nxt = x;
                }
                if (nxt < 0) {  // exact inverse CDF over the row's integer weights
                    uint64_t tot = 0;
                    for (int64_t j = 0; j < d; ++j)
                        tot += walk_threshold<MODE>(cols[s + j], row, t, indptr, cols, T[0], T[1], T[2]);
                    const uint64_t target = mulhi64(walk_word(wb, t, 2 * PGLB_WALK_MAX_REJECT), tot);
                    uint64_t acc = 0;
                    for (int64_t j = 0; j < d; ++j) {
                        acc += walk_threshold<MODE>(cols[s + j], row, t, indptr, cols, T[0], T[1], T[2]);
                        if (acc > target) {
                            nxt = cols[s + j];
                            break;
                        }
                    }
                }
            }
            row[t + 1] = nxt;
            cur = nxt;
            len = t + 2;
        }
        for (int64_t k = len; k <= steps; ++k) row[k] = -1;
    }
}

extern "C" int pglb_random_walk_host(const int64_t *indptr, const int64_t *cols, int64_t N, const int64_t *nodes,
                                     int64_t n, int64_t steps, int mode, double p, double q, uint64_t seed,
                                     int64_t *out, int64_t ldo) {
    const int rc = walk_check("pglb_random_walk_host", N, n, steps, mode, p, q, ldo, indptr, nodes, out);
    if (rc != PGLB_OK || n == 0) return rc;
    PGLB_CHECK_ARG(cols || indptr[N] == 0, PGLB_EINVAL, "pglb_random_walk_host: NULL cols");
    for (int64_t i = 0; i < n; ++i)
        PGLB_CHECK_ARG(nodes[i] >= 0 && nodes[i] < N, PGLB_ESHAPE,
                       "pglb_random_walk_host: node id %lld out of range [0,%lld)", (long long)nodes[i],
                       (long long)N);
    uint64_t T[3] = {1, 1, 1};
    if (mode != PGLB_WALK_UNIFORM) walk_thresholds(p, q, T);
    if (mode == PGLB_WALK_UNIFORM)
        walk_host<PGLB_WALK_UNIFORM>(indptr, cols, nodes, n, steps, seed, T, out, ldo);
    else if (mode == PGLB_WALK_NODE2VEC)
        walk_host<PGLB_WALK_NODE2VEC>(indptr, cols, nodes, n, steps, seed, T, out, ldo);
    else
        walk_host<PGLB_WALK_NODE2VEC_PLUS>(indptr, cols, nodes, n, steps, seed, T, out, ldo);
    return PGLB_OK;
}

static int sg_check(const char *who, int64_t n, int64_t W, int64_t ldw, int64_t win, const void *walks, void *ws,
                    size_t ws_bytes) {
    PGLB_CHECK_ARG(n >= 0 && W >= 0, PGLB_EINVAL, "%s: negative size", who);
    PGLB_CHECK_ARG(win >= 1, PGLB_EINVAL, "%s: win_size must be >= 1", who);
    PGLB_CHECK_ARG(ldw >= W, PGLB_ESHAPE, "%s: ldw %lld < W %lld", who, (long long)ldw, (long long)W);
    PGLB_CHECK_ARG(n == 0 || W == 0 || walks, PGLB_EINVAL, "%s: NULL walks", who);
    size_t need = 0;
    pglb_skip_gram_ws(n, W, &need);
    PGLB_CHECK_ARG(ws_bytes >= need && (ws || n * W == 0), PGLB_EWORKSPACE,
                   "%s: workspace of %zu bytes needed (got %zu)", who, need, ws_bytes);
    return PGLB_OK;
}

extern "C" int pglb_skip_gram_ws(int64_t n, int64_t W, size_t *ws_bytes) {
    PGLB_CHECK_ARG(n >= 0 && W >= 0 && ws_bytes, PGLB_EINVAL, "pglb_skip_gram_ws: bad argument");
    *ws_bytes = align_up(sizeof(int64_t) * (size_t)std::max<int64_t>(n, 1), 256) + scan_i64_ws_bytes(n * W);
    return PGLB_OK;
}

extern "C" int pglb_skip_gram_count(const int64_t *walks, int64_t n, int64_t W, int64_t ldw, int64_t win_size,
                                    uint64_t seed, int64_t *offsets, void *ws, size_t ws_bytes, void *stream) {
    int rc = sg_check("pglb_skip_gram_count", n, W, ldw, win_size, walks, ws, ws_bytes);
    if (rc != PGLB_OK) return rc;
    PGLB_CHECK_ARG(offsets, PGLB_EINVAL, "pglb_skip_gram_count: NULL offsets");
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    const int64_t m = n * W;
    if (m == 0) {
        PGLB_CUDA(cudaMemsetAsync(offsets, 0, sizeof(int64_t), s));
        return PGLB_OK;
    }
    int64_t *len = reinterpret_cast<int64_t *>(ws);
    void *scan_tmp = reinterpret_cast<char *>(ws) + align_up(sizeof(int64_t) * (size_t)n, 256);
    sg_len_kernel<<<grid_for(n, 8), 256, 0, s>>>(walks, n, W, ldw, len);
    PGLB_LAUNCH_CHECK("sg_len_kernel");
    sg_count_kernel<<<grid_for(m, 8), 256, 0, s>>>(walks, n, W, ldw, win_size, seed, len, offsets);
    PGLB_LAUNCH_CHECK("sg_count_kernel");
    return scan_i64(offsets + 1, offsets + 1, m, /*inclusive=*/1, scan_tmp, s);
}

extern "C" int pglb_skip_gram_fill(const int64_t *walks, int64_t n, int64_t W, int64_t ldw, int64_t win_size,
                                   uint64_t seed, const int64_t *offsets, int64_t *src, int64_t *dst, void *ws,
                                   size_t ws_bytes, void *stream) {
    int rc = sg_check("pglb_skip_gram_fill", n, W, ldw, win_size, walks, ws, ws_bytes);
    if (rc != PGLB_OK) return rc;
    const int64_t m = n * W;
    if (m == 0) return PGLB_OK;
    PGLB_CHECK_ARG(offsets && src && dst, PGLB_EINVAL, "pglb_skip_gram_fill: NULL pointer");
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    sg_fill_kernel<<<grid_for(m, 8), 256, 0, s>>>(walks, n, W, ldw, win_size, seed,
                                                  reinterpret_cast<const int64_t *>(ws), offsets, src, dst);
    PGLB_LAUNCH_CHECK("sg_fill_kernel");
    return PGLB_OK;
}
