// Diffusion re-ranking (mdir_b200.Diffusion; Iscen et al., CVPR 2017): a mutual kNN graph of the database, built once,
// and per query a truncated conjugate-gradient solve of (I - alpha S_LL) f = y on the query's shortlist L.
// The semantics are restated in tests/diffusion_reference.py (diffusion_graph / diffusion_search).
//
// Graph.  knn_ids / knn_s are the certified fp32 top-(k+1) of every used slot against the database (Index.search,
// ordered by score desc, id asc; -1 padding): row r is slot r's list.  N(i) is that list without i itself, or without
// its last entry when i is not in it.  (i, j) is an edge iff j in N(i) and i in N(j); its weight is max(s, 0)^gamma with
// s taken from the list of the lower slot, so w is symmetric bit for bit; d_i sums w over N(i) in list order;
// S_ij = w_ij / (sqrtf(d_i) sqrtf(d_j)) (a product of square roots: the square of a tiny degree would underflow).
//
// Solve.  One CTA per query (a persistent grid over the queries); CG in fp64 on the fp32 graph weights.  Every step's arithmetic depends only on the query's
// own shortlist and the graph, and every reduction runs in a fixed order (per-thread strided sums, an xor-shuffle tree
// per warp, the warp partials summed in warp order), so a query's result is the same bits alone or in any batch.
//
// Combine (offline diffusion).  A table of every slot's own diffusion truncated to `width` entries, and per query the
// weighted sum of the table rows of its top-k_q (diffusion_combine_kernel).
#include <cuda_bf16.h>

#include <cfloat>

#include "common.cuh"

namespace mdir {

constexpr int kDiffMaxTrunc = 2048;       // shortlist rows per query (4 fp64 CG vectors + 64-bit sort keys in smem)
constexpr int kDiffMaxK = 255;            // neighbours per row
constexpr int kDiffThreads = 512;
constexpr int kDiffWarps = kDiffThreads / 32;
constexpr int kDiffCtas = 2 * kNumSMs;    // persistent solve grid: two 512-thread CTAs per SM

// first slot s in [0, n_used) with slot_id[s] == id, or -1
__device__ __forceinline__ int64_t diff_slot_of(const uint32_t* __restrict__ slot_id, int64_t n_used, int32_t id) {
    if (id == -1) return -1;
    int64_t lo = 0, hi = n_used;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (slot_id[mid] < (uint32_t)id) lo = mid + 1;
        else hi = mid;
    }
    return lo < n_used && slot_id[lo] == (uint32_t)id ? lo : -1;
}

// One warp per row i.  Lane l handles raw list positions l, l + 32, ... in chunks of 32, so the ballot prefix keeps the
// mutual neighbours in N(i) order.  Membership i in N(j) is a linear scan of j's raw list for the ids of i and of j.
__global__ void __launch_bounds__(256) diffusion_graph_kernel(const int32_t* __restrict__ knn_ids, const float* __restrict__ knn_s,
                                                              int64_t n_used, int k, const uint32_t* __restrict__ slot_id, float gamma,
                                                              int32_t* __restrict__ nbr, float* __restrict__ w, float* __restrict__ deg) {
    __shared__ float wbuf[8][kDiffMaxK + 1];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int64_t i = (int64_t)blockIdx.x * 8 + wid;
    if (i >= n_used) return;
    const int kr = k + 1;
    const int32_t* ri = knn_ids + i * kr;
    const int32_t id_i = (int32_t)slot_id[i];
    int self_pos = -1;
    for (int p = lane; p < kr; p += 32)
        if (ri[p] == id_i) self_pos = p;
    self_pos = __reduce_max_sync(0xffffffffu, self_pos);
    int n_out = 0;
    for (int p0 = 0; p0 < kr; p0 += 32) {
        const int p = p0 + lane;
        bool mutual = false;
        int64_t j = -1;
        float wij = 0.f;
        if (p < kr && p != self_pos && (self_pos >= 0 || p < k)) {
            const int32_t id_j = ri[p];
            j = diff_slot_of(slot_id, n_used, id_j);
            if (j >= 0) {
                const int32_t* rj = knn_ids + j * kr;
                int pi = -1, pj = -1;
                for (int t = 0; t < kr; ++t) {
                    const int32_t v = rj[t];
                    if (v == id_i) pi = t;
                    if (v == id_j) pj = t;
                }
                mutual = pi >= 0 && (pj >= 0 || pi < k);
                if (mutual) {
                    const float s = i < j ? knn_s[i * kr + p] : knn_s[j * kr + pi];
                    wij = powf(fmaxf(s, 0.f), gamma);
                }
            }
        }
        const unsigned bal = __ballot_sync(0xffffffffu, mutual);
        if (mutual) {
            const int o = n_out + __popc(bal & ((1u << lane) - 1u));
            nbr[i * k + o] = (int32_t)j;
            w[i * k + o] = wij;
            wbuf[wid][o] = wij;
        }
        n_out += __popc(bal);
    }
    for (int o = n_out + lane; o < k; o += 32) {
        nbr[i * k + o] = -1;
        w[i * k + o] = 0.f;
    }
    __syncwarp();
    if (lane == 0) {
        float d = 0.f;
        for (int o = 0; o < n_out; ++o) d += wbuf[wid][o];
        deg[i] = d;
    }
}

__global__ void __launch_bounds__(256) diffusion_normalize_kernel(const int32_t* __restrict__ nbr, const float* w,
                                                                  const float* __restrict__ deg, int64_t n_used, int k, float* S) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_used * k) return;
    const int32_t j = nbr[e];
    const float wij = w[e];
    S[e] = j >= 0 && wij > 0.f ? wij / (sqrtf(deg[e / k]) * sqrtf(deg[j])) : 0.f;
}

// Block sum in a fixed order (an xor-shuffle tree per warp, then the warps in order); every thread returns the same bits.
__device__ __forceinline__ double diff_block_sum(double v, double* red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();                                   // red's previous readers are done
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = 0.0;
#pragma unroll
    for (int t = 0; t < kDiffWarps; ++t) s += red[t];
    return s;
}

__host__ __device__ inline size_t diff_ws_cta_bytes(int trunc, int k) {
    const size_t a = ((size_t)trunc * k * 2 + 255) & ~(size_t)255;
    const size_t b = ((size_t)trunc * k * 4 + 255) & ~(size_t)255;
    return a + b;
}

__global__ void __launch_bounds__(kDiffThreads) diffusion_solve_kernel(
        const int32_t* __restrict__ L_ids, const float* __restrict__ L_s, int n_q, int trunc, const uint32_t* __restrict__ slot_id,
        int64_t n_used, const int32_t* __restrict__ nbr, const float* __restrict__ S, int k, int k_q, float gamma, double alpha,
        int iters, double rtol, int k_out, uint8_t* __restrict__ ws, float* __restrict__ f_out, int32_t* __restrict__ ids_out,
        const int64_t* __restrict__ n_used_dev, const int32_t* __restrict__ status) {
    extern __shared__ __align__(16) uint8_t smem[];
    uint64_t* keys = reinterpret_cast<uint64_t*>(smem);                       // kDiffMaxTrunc
    double* x = reinterpret_cast<double*>(keys + kDiffMaxTrunc);
    double* r = x + kDiffMaxTrunc;
    double* p = r + kDiffMaxTrunc;
    double* ap = p + kDiffMaxTrunc;
    uint16_t* cnt = reinterpret_cast<uint16_t*>(ap + kDiffMaxTrunc);
    __shared__ double red[kDiffWarps];
    __shared__ int s_n;
    __shared__ int64_t s_used;
    // this CTA's local ELL of S_LL, column-major: entry c of row u at c * trunc + u (u16 local index, fp32 S)
    uint16_t* ell_idx = reinterpret_cast<uint16_t*>(ws + (size_t)blockIdx.x * diff_ws_cta_bytes(trunc, k));
    float* ell_val = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(ell_idx) + (((size_t)trunc * k * 2 + 255) & ~(size_t)255));
    const int tid = threadIdx.x;
    if (tid == 0) s_used = n_used_dev ? *n_used_dev : n_used;
    __syncthreads();
    n_used = s_used;

    for (int q = blockIdx.x; q < n_q; q += gridDim.x) {
        if (status && status[q] != 0) {                                      // a flagged shortlist: no rows
            for (int j = tid; j < k_out; j += kDiffThreads) {
                f_out[(int64_t)q * k_out + j] = -INFINITY;
                ids_out[(int64_t)q * k_out + j] = -1;
            }
            continue;
        }
        const int32_t* ids = L_ids + (int64_t)q * trunc;
        const float* sc = L_s + (int64_t)q * trunc;
        // (0) |L|: search pads its rows with id -1 after the live rows it found
        if (tid == 0) s_n = trunc;
        __syncthreads();
        for (int u = tid; u < trunc; u += kDiffThreads)
            if (ids[u] == -1) atomicMin(&s_n, u);
        __syncthreads();
        const int n = s_n;
        int npow = 32;
        while (npow < n) npow <<= 1;
        // (1) + (2) the shortlist's slots, sorted with their positions
        for (int u = tid; u < npow; u += kDiffThreads) {
            uint64_t key = ~0ull;
            if (u < n) {
                const int64_t s = diff_slot_of(slot_id, n_used, ids[u]);
                key = ((uint64_t)(s >= 0 ? (uint32_t)s : 0xffffffffu) << 32) | (uint32_t)u;
            }
            keys[u] = key;
        }
        __syncthreads();
        bitonic_sort_smem(keys, npow);
        // (3) local ELL of S_LL: row u keeps the neighbours of its slot that are in L, in the graph's order
        for (int t = tid; t < n; t += kDiffThreads) {
            const uint64_t kt = keys[t];
            const uint32_t slot = (uint32_t)(kt >> 32);
            const int u = (int)(uint32_t)kt;
            int c = 0;
            if (slot != 0xffffffffu) {
                for (int e = 0; e < k; ++e) {
                    const int32_t j = nbr[(int64_t)slot * k + e];
                    if (j < 0) break;                                        // mutual neighbours first, then padding
                    int lo = 0, hi = n;
                    while (lo < hi) {
                        const int mid = (lo + hi) >> 1;
                        if ((uint32_t)(keys[mid] >> 32) < (uint32_t)j) lo = mid + 1;
                        else hi = mid;
                    }
                    if (lo < n && (uint32_t)(keys[lo] >> 32) == (uint32_t)j) {
                        ell_idx[(size_t)c * trunc + u] = (uint16_t)(uint32_t)keys[lo];
                        ell_val[(size_t)c * trunc + u] = S[(int64_t)slot * k + e];
                        ++c;
                    }
                }
            }
            cnt[u] = (uint16_t)c;
        }
        // (4) CG from x = 0: scipy.sparse.linalg.cg's recurrences in fp64 on the fp32 S.  fp32 vectors lose about
        // eps_32 / (1 - alpha) of max |f|: 4e-5 on a clique of duplicate rows at alpha = 0.99
        double yy = 0.0;
        for (int u = tid; u < n; u += kDiffThreads) {
            const double y = u < k_q ? pow((double)fmaxf(sc[u], 0.f), (double)gamma) : 0.0;
            x[u] = 0.0;
            r[u] = y;
            yy += y * y;
        }
        yy = diff_block_sum(yy, red);                                        // its syncs also publish cnt and the ELL
        const double atol = rtol * sqrt(yy);
        double rho_prev = 1.0;
        for (int it = 0; yy > 0.0 && it < iters; ++it) {
            double rr = 0.0;
            for (int u = tid; u < n; u += kDiffThreads) rr += r[u] * r[u];
            const double rho = diff_block_sum(rr, red);
            if (sqrt(rho) < atol || rho == 0.0) break;                        // rho == 0: r is 0, x is exact (rtol = 0)
            const double beta = it > 0 ? rho / rho_prev : 0.0;
            for (int u = tid; u < n; u += kDiffThreads) p[u] = it > 0 ? p[u] * beta + r[u] : r[u];
            __syncthreads();
            double pq = 0.0;
            for (int u = tid; u < n; u += kDiffThreads) {
                double acc = 0.0;
                const int c = cnt[u];
                for (int e = 0; e < c; ++e) acc = fma((double)ell_val[(size_t)e * trunc + u], p[ell_idx[(size_t)e * trunc + u]], acc);
                const double v = p[u] - alpha * acc;
                ap[u] = v;
                pq += p[u] * v;
            }
            const double a = rho / diff_block_sum(pq, red);
            for (int u = tid; u < n; u += kDiffThreads) {
                x[u] += a * p[u];
                r[u] -= a * ap[u];
            }
            rho_prev = rho;
        }
        __syncthreads();
        // (5) rank L by (f desc, position asc) and emit the top k_out with their ids
        for (int u = tid; u < npow; u += kDiffThreads) keys[u] = u < n ? make_key((float)x[u], (uint32_t)u) : ~0ull;
        __syncthreads();
        bitonic_sort_smem(keys, npow);
        for (int j = tid; j < k_out; j += kDiffThreads) {
            const bool ok = j < n;
            const int u = ok ? (int)(uint32_t)keys[j] : 0;
            f_out[(int64_t)q * k_out + j] = ok ? (float)x[u] : -INFINITY;
            ids_out[(int64_t)q * k_out + j] = ok ? ids[u] : -1;
        }
        __syncthreads();                                                     // keys / x are rewritten by the next query
    }
}

constexpr size_t kDiffSmem = (size_t)kDiffMaxTrunc * (8 + 4 * 8 + 2);   // keys, x / r / p / Ap, counts: 84 KB

// ---- incremental graph update (Diffusion.add / restore / remove) ---------------------------------------------------
// Raw lists hold (k + 1) entries per slot; an entry's key is make_key(score, id) (smaller = better), ~0 for padding.
constexpr int kMergeCols = 32;            // target rows per CTA of diffusion_merge_kernel
constexpr int kMergeWarps = 8;
constexpr int kMergeStage = 128;          // new keys a warp stages before merging them into its row's list

__device__ __forceinline__ uint64_t diff_entry_key(const int32_t* ids, const float* s, int64_t e) {
    const int32_t id = ids[e];
    return id == -1 ? ~0ull : make_key(s[e], (uint32_t)id);
}
__device__ __forceinline__ bool diff_live(const uint32_t* __restrict__ live, int64_t slot) {
    return (live[slot >> 5] >> (slot & 31)) & 1u;
}

// eps[j] = bf16_eps of row j of q32 (n_q, D) taken as a query: range_tau_kernel's norms and bound.
__global__ void __launch_bounds__(256) diffusion_batch_eps_kernel(const float* __restrict__ q32, int D, const float* __restrict__ db_stats,
                                                                  float* __restrict__ eps) {
    __shared__ float red[32];
    const int q = blockIdx.x;
    float q2 = 0.f, qt2 = 0.f, qf2 = 0.f;
    for (int i = threadIdx.x; i < D; i += blockDim.x) {
        const float v = q32[(int64_t)q * D + i];
        const float vt = __bfloat162float(__float2bfloat16_rn(v));
        q2 = fmaf(v, v, q2);
        qt2 = fmaf(vt, vt, qt2);
        qf2 = fmaf(v - vt, v - vt, qf2);
    }
    q2 = block_sum(q2, red);
    qt2 = block_sum(qt2, red);
    qf2 = block_sum(qf2, red);
    if (threadIdx.x == 0) eps[q] = bf16_eps(db_stats, q2, qt2, qf2, D);
}

// The reverse merge of a batch B into the raw lists of the target rows i (rows of the plane's chunk whose bit in `live`
// is set), one CTA per tile of kMergeCols rows, in two kernels on the same grid.  plane (nb, ld) fp32 = the bf16 scores
// of B (queries) against the chunk's rows.
// (1) diffusion_screen_kernel: pair (i, j) passes when its bf16 score >= fsub_rd(score(T_i), eps[j]), T_i the key of
//     entry k of i's list (every pair passes when that entry is padding).  Passing pairs go to the CTA's segment through a
//     warp-aggregated shared-memory counter; cnt[tile] is exact even past `cap`, so that the host re-runs an overflowed
//     tile with room.
// (2) diffusion_merge_kernel, for a tile with cnt <= cap: one warp per passing pair re-scores it with rescore_row, row i
//     as the query (the build's roles and summation order), and accepts key(s_ij, id_j) < T_i; then one warp per target
//     row stages its accepted keys and rank-merges them into the sorted list (keys are unique: B's ids are in no target
//     list), keeping the first k + 1.  rep[tile] = list entries replaced (0 when the tile overflowed: no list touched).
// T_i and the screen limit of the tile's kMergeCols target rows (s_ts NaN: row i is not a target, nothing passes)
__device__ __forceinline__ void diff_tile_thresholds(int64_t row0, int64_t n_rows, const uint32_t* __restrict__ live, const int32_t* knn_ids,
                                                     const float* knn_s, int k, uint64_t* s_T, float* s_ts) {
    if (threadIdx.x < kMergeCols) {
        const int64_t i = row0 + threadIdx.x;
        const bool ok = threadIdx.x < n_rows && diff_live(live, i);
        const uint64_t T = ok ? diff_entry_key(knn_ids, knn_s, i * (k + 1) + k) : 0ull;     // 0: no key is smaller
        s_T[threadIdx.x] = T;
        s_ts[threadIdx.x] = !ok ? NAN : T == ~0ull ? -INFINITY : key_score(T);
    }
    __syncthreads();
}

__global__ void __launch_bounds__(kMergeWarps * 32) diffusion_screen_kernel(
        const float* __restrict__ plane, int64_t ld, int nb, int64_t col0, int64_t n_cols, const int32_t* __restrict__ tiles,
        const uint32_t* __restrict__ live, const float* __restrict__ eps, const int32_t* __restrict__ knn_ids, const float* __restrict__ knn_s,
        int k, uint64_t* __restrict__ seg, int cap, int32_t* __restrict__ cnt) {
    __shared__ uint64_t s_T[kMergeCols];
    __shared__ float s_ts[kMergeCols];
    __shared__ int s_cnt;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t tile = tiles ? (int64_t)tiles[blockIdx.x] : col0 / kMergeCols + blockIdx.x;
    const int64_t c_lo = tile * kMergeCols - col0;             // the tile's first column of the plane
    uint64_t* ent = seg + (int64_t)blockIdx.x * 2 * cap;        // (column << 32 | batch row)
    if (threadIdx.x == 0) s_cnt = 0;
    diff_tile_thresholds(col0 + c_lo, n_cols - c_lo, live, knn_ids, knn_s, k, s_T, s_ts);
    // (1) screen: warp w reads batch rows w, w + 8, ...; lane = column (coalesced 128-byte rows of the plane)
    const float ts = s_ts[lane];
    if (__any_sync(0xffffffffu, ts == ts)) {
        const float* col = plane + c_lo + lane;
        for (int j0 = warp; j0 < nb; j0 += 4 * kMergeWarps) {
            float v[4];                                         // four rows' loads in flight per lane
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int j = j0 + u * kMergeWarps;
                v[u] = ts == ts && j < nb ? __ldg(col + (int64_t)j * ld) : 0.f;
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int j = j0 + u * kMergeWarps;
                const bool pass = ts == ts && j < nb && v[u] >= __fsub_rd(ts, __ldg(eps + min(j, nb - 1)));
                const unsigned bal = __ballot_sync(0xffffffffu, pass);
                if (bal) {
                    int base = 0;
                    if (lane == 0) base = atomicAdd(&s_cnt, __popc(bal));
                    base = __shfl_sync(0xffffffffu, base, 0);
                    const int o = base + __popc(bal & ((1u << lane) - 1u));
                    if (pass && o < cap) ent[o] = ((uint64_t)lane << 32) | (uint32_t)j;
                }
            }
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) cnt[tile] = s_cnt;
}

// Runs after diffusion_screen_kernel on the same grid: a tile whose count exceeds cap is left as it is.
__global__ void __launch_bounds__(kMergeWarps * 32, 1) diffusion_merge_kernel(
        int64_t col0, int64_t n_cols, const int32_t* __restrict__ tiles, const uint32_t* __restrict__ live, const int64_t* __restrict__ bslot,
        const float* __restrict__ db32, int D, const uint32_t* __restrict__ slot_id, int32_t* __restrict__ knn_ids, float* __restrict__ knn_s,
        int k, uint64_t* __restrict__ seg, int cap, const int32_t* __restrict__ cnt, int32_t* __restrict__ rep) {
    __shared__ uint64_t s_T[kMergeCols];
    __shared__ float s_ts[kMergeCols];
    __shared__ uint64_t s_lst[kMergeWarps][kDiffMaxK + 1], s_out[kMergeWarps][kDiffMaxK + 1], s_stage[kMergeWarps][kMergeStage];
    __shared__ int s_rep;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int kr = k + 1;
    const int64_t tile = tiles ? (int64_t)tiles[blockIdx.x] : col0 / kMergeCols + blockIdx.x;
    const int64_t c_lo = tile * kMergeCols - col0;
    const int n = cnt[tile];
    if (n > cap) {
        if (threadIdx.x == 0) rep[tile] = 0;
        return;
    }
    uint64_t* ent = seg + (int64_t)blockIdx.x * 2 * cap;        // (column << 32 | batch row), then the accepted keys
    uint64_t* acc = ent + cap;
    if (threadIdx.x == 0) s_rep = 0;
    diff_tile_thresholds(col0 + c_lo, n_cols - c_lo, live, knn_ids, knn_s, k, s_T, s_ts);
    // (2) re-score every passing pair in fp32
    for (int e = warp; e < n; e += kMergeWarps) {
        const uint64_t en = ent[e];
        const int c = (int)(en >> 32);
        const int64_t i = col0 + c_lo + c, j = bslot[(uint32_t)en];
        const float s = rescore_row(db32 + j * D, db32 + i * D, D, lane);
        const uint64_t key = make_key(s, slot_id[j]);
        if (lane == 0) acc[e] = key < s_T[c] ? key : ~0ull;
    }
    __syncthreads();
    // (3) merge, one warp per target row
    uint64_t* lst = s_lst[warp];
    uint64_t* out = s_out[warp];
    uint64_t* stage = s_stage[warp];
    int replaced = 0;
    for (int c = warp; c < kMergeCols; c += kMergeWarps) {
        if (s_ts[c] != s_ts[c]) continue;
        const int64_t i = col0 + c_lo + c;
        for (int p = lane; p < kr; p += 32) lst[p] = diff_entry_key(knn_ids, knn_s, i * kr + p);
        int ns = 0, n_new = 0;
        for (int e0 = 0; e0 < n; e0 += 32) {
            const int e = e0 + lane;
            const uint64_t key = e < n && (int)(ent[e] >> 32) == c ? acc[e] : ~0ull;
            const unsigned bal = __ballot_sync(0xffffffffu, key != ~0ull);
            if (key != ~0ull) stage[ns + __popc(bal & ((1u << lane) - 1u))] = key;
            ns += __popc(bal);
            n_new += __popc(bal);
            if (ns > kMergeStage - 32 || (e0 + 32 >= n && ns > 0)) {
                __syncwarp();
                // ranks in the union: old entry p -> p + #(staged keys below it); staged key -> #(staged below) + #(old below)
                for (int p = lane; p < kr; p += 32) {
                    const uint64_t a = lst[p];
                    int r = p;
                    for (int t = 0; t < ns; ++t) r += stage[t] < a;
                    if (r < kr) out[r] = a;
                }
                for (int t = lane; t < ns; t += 32) {
                    const uint64_t b = stage[t];
                    int r = 0;
                    for (int u = 0; u < ns; ++u) r += stage[u] < b;
                    int lo = 0, hi = kr;
                    while (lo < hi) {
                        const int mid = (lo + hi) >> 1;
                        if (lst[mid] < b) lo = mid + 1;
                        else hi = mid;
                    }
                    r += lo;
                    if (r < kr) out[r] = b;
                }
                __syncwarp();
                for (int p = lane; p < kr; p += 32) lst[p] = out[p];
                __syncwarp();
                ns = 0;
            }
        }
        if (n_new == 0) continue;
        // entries of the merged list that were not in the old one, then the list written back
        for (int p = lane; p < kr; p += 32) {
            const uint64_t key = lst[p];
            if (key == ~0ull) continue;
            int lo = 0, hi = kr;
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (diff_entry_key(knn_ids, knn_s, i * kr + mid) < key) lo = mid + 1;
                else hi = mid;
            }
            replaced += !(lo < kr && diff_entry_key(knn_ids, knn_s, i * kr + lo) == key);
        }
        __syncwarp();
        for (int p = lane; p < kr; p += 32) {
            const uint64_t key = lst[p];
            knn_ids[i * kr + p] = key == ~0ull ? -1 : (int32_t)(uint32_t)key;
            knn_s[i * kr + p] = key == ~0ull ? -INFINITY : key_score(key);
        }
        __syncwarp();
    }
    replaced = warp_sum_int(replaced);
    if (lane == 0 && replaced) atomicAdd(&s_rep, replaced);
    __syncthreads();
    if (threadIdx.x == 0) rep[tile] = s_rep;
}

// One warp per used slot: a removed slot's list becomes padding; a live slot whose list holds an id that is no longer
// live (or no longer held by any used slot) gets flag 1, else 0.
__global__ void __launch_bounds__(256) diffusion_stale_kernel(int32_t* __restrict__ knn_ids, float* __restrict__ knn_s, int64_t n_used, int k,
                                                              const uint32_t* __restrict__ slot_id, const uint32_t* __restrict__ live,
                                                              uint8_t* __restrict__ flag) {
    const int lane = threadIdx.x & 31;
    const int64_t i = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (i >= n_used) return;
    const int kr = k + 1;
    if (!diff_live(live, i)) {
        for (int p = lane; p < kr; p += 32) {
            knn_ids[i * kr + p] = -1;
            knn_s[i * kr + p] = -INFINITY;
        }
        if (lane == 0) flag[i] = 0;
        return;
    }
    bool stale = false;
    for (int p = lane; p < kr; p += 32) {
        const int32_t id = knn_ids[i * kr + p];
        if (id == -1) continue;
        const int64_t s = diff_slot_of(slot_id, n_used, id);
        stale |= s < 0 || !diff_live(live, s);
    }
    stale = __any_sync(0xffffffffu, stale);
    if (lane == 0) flag[i] = stale ? 1 : 0;
}

// ---- offline diffusion (DiffusionTable.search) ------------------------------------------------------------------------
// Table row of slot s: the top `width` (id, f) of that row's own diffusion (k_q = 1).  A query's f_j is the sum over the
// k_q rows L_u of its top-k_q of w_u F[slot(L_u)][j], w_u = max(s_u, 0)^gamma, over the union of those table rows.
constexpr int kCombMaxKq = 128;           // u takes 7 bits of a staged key
constexpr int kCombMaxWidth = 1024;       // e takes 10 bits
constexpr int kCombMaxEntries = 8192;     // k_q * width: 64-bit keys, fp32 sums and head flags, 104 KB of smem
constexpr int kCombThreads = 512;
constexpr int kCombCtas = 2 * kNumSMs;

__host__ __device__ inline int comb_npow(int n) {
    int p = 32;
    while (p < n) p <<= 1;
    return p;
}
__host__ __device__ inline size_t comb_smem_bytes(int n) { return ((size_t)comb_npow(n) * (8 + 4 + 1) + 15) & ~(size_t)15; }

// One CTA per query (a persistent grid).  (1) L's ids -> slots, w_u in fp64; (2) key (id, u, e) per live table entry,
// bitonic-sorted; (3) the first entry of each id's run sums its run in key order (ascending u) in fp64, as
// f = f + w_u * F with separate roundings; (4) the run heads re-keyed make_key((float)f, id), sorted, top k_out emitted.
// No atomics and fixed orders: a query's result is the same bits alone or in any batch.
__global__ void __launch_bounds__(kCombThreads, 2) diffusion_combine_kernel(
        const int32_t* __restrict__ L_ids, const float* __restrict__ L_s, int n_q, int k_q, const uint32_t* __restrict__ slot_id,
        int64_t n_used, const int32_t* __restrict__ tab_ids, const float* __restrict__ tab_f, int width, float gamma, int k_out,
        float* __restrict__ f_out, int32_t* __restrict__ ids_out, const int64_t* __restrict__ n_used_dev, const int32_t* __restrict__ status) {
    extern __shared__ __align__(16) uint8_t smem[];
    __shared__ int64_t s_slot[kCombMaxKq];
    __shared__ double s_w[kCombMaxKq];
    __shared__ int64_t s_used;
    const int n = k_q * width, npow = comb_npow(n);
    uint64_t* keys = reinterpret_cast<uint64_t*>(smem);
    float* fsum = reinterpret_cast<float*>(keys + npow);
    uint8_t* head = reinterpret_cast<uint8_t*>(fsum + npow);
    const int tid = threadIdx.x;
    constexpr int kIdShift = 17;
    if (tid == 0) s_used = n_used_dev ? *n_used_dev : n_used;
    __syncthreads();
    n_used = s_used;

    for (int q = blockIdx.x; q < n_q; q += gridDim.x) {
        if (status && status[q] != 0) {                                      // a flagged top-k_q: no rows
            for (int j = tid; j < k_out; j += kCombThreads) {
                f_out[(int64_t)q * k_out + j] = -INFINITY;
                ids_out[(int64_t)q * k_out + j] = -1;
            }
            continue;
        }
        for (int u = tid; u < k_q; u += kCombThreads) {
            s_slot[u] = diff_slot_of(slot_id, n_used, L_ids[(int64_t)q * k_q + u]);
            s_w[u] = pow((double)fmaxf(L_s[(int64_t)q * k_q + u], 0.f), (double)gamma);
        }
        __syncthreads();
        for (int t = tid; t < npow; t += kCombThreads) {
            uint64_t key = ~0ull;
            if (t < n) {
                const int u = t / width, e = t - u * width;
                const int64_t s = s_slot[u];
                const int32_t id = s >= 0 ? tab_ids[s * width + e] : -1;
                if (id != -1) key = ((uint64_t)(uint32_t)id << kIdShift) | ((uint64_t)u << 10) | (uint64_t)e;
            }
            keys[t] = key;
        }
        __syncthreads();
        bitonic_sort_smem(keys, npow);
        for (int t = tid; t < npow; t += kCombThreads) {
            const uint64_t kt = keys[t];
            const uint64_t id = kt >> kIdShift;                    // padding: 2^47 - 1, no id
            const bool h = kt != ~0ull && (t == 0 || (keys[t - 1] >> kIdShift) != id);
            if (h) {
                double f = 0.0;
                for (int r = t; r < npow && (keys[r] >> kIdShift) == id; ++r) {
                    const int u = (int)((keys[r] >> 10) & (kCombMaxKq - 1)), e = (int)(keys[r] & (kCombMaxWidth - 1));
                    f = __dadd_rn(f, __dmul_rn(s_w[u], (double)tab_f[s_slot[u] * width + e]));
                }
                fsum[t] = (float)f;
            }
            head[t] = h;
        }
        __syncthreads();
        for (int t = tid; t < npow; t += kCombThreads)
            keys[t] = head[t] ? make_key(fsum[t], (uint32_t)(keys[t] >> kIdShift)) : ~0ull;
        __syncthreads();
        bitonic_sort_smem(keys, npow);
        for (int j = tid; j < k_out; j += kCombThreads) {
            const uint64_t kt = j < npow ? keys[j] : ~0ull;
            const bool ok = kt != ~0ull;
            f_out[(int64_t)q * k_out + j] = ok ? key_score(kt) : -INFINITY;
            ids_out[(int64_t)q * k_out + j] = ok ? (int32_t)(uint32_t)kt : -1;
        }
        __syncthreads();                                                     // keys / s_slot are rewritten by the next query
    }
}

}  // namespace mdir

using namespace mdir;

extern "C" int mdir_diffusion_graph(const int32_t* knn_ids, const float* knn_s, int64_t n_used, int k, const uint32_t* slot_id,
                                    float gamma, int32_t* nbr, float* w, float* deg, void* stream) {
    MDIR_CHECK_ARG(knn_ids && knn_s && slot_id && nbr && w && deg && n_used >= 0 && k >= 1 && k <= kDiffMaxK);
    MDIR_CHECK_ARG(gamma > 0.f && gamma <= FLT_MAX);
    if (n_used == 0) return 0;
    diffusion_graph_kernel<<<(unsigned)((n_used + 7) / 8), 256, 0, (cudaStream_t)stream>>>(knn_ids, knn_s, n_used, k, slot_id, gamma,
                                                                                          nbr, w, deg);
    MDIR_LAUNCH_CHECK();
    return 0;
}

extern "C" int mdir_diffusion_normalize(const int32_t* nbr, const float* w, const float* deg, int64_t n_used, int k, float* S,
                                        void* stream) {
    MDIR_CHECK_ARG(nbr && w && deg && S && n_used >= 0 && k >= 1 && k <= kDiffMaxK);
    const int64_t n = n_used * k;
    if (n == 0) return 0;
    diffusion_normalize_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(nbr, w, deg, n_used, k, S);
    MDIR_LAUNCH_CHECK();
    return 0;
}

extern "C" int mdir_diffusion_batch_eps(const float* q32, int n_q, int D, const float* db_stats, float* eps, void* stream) {
    MDIR_CHECK_ARG(q32 && db_stats && eps && n_q >= 0 && D >= 1);
    if (n_q == 0) return 0;
    diffusion_batch_eps_kernel<<<n_q, 256, 0, (cudaStream_t)stream>>>(q32, D, db_stats, eps);
    MDIR_LAUNCH_CHECK();
    return 0;
}

extern "C" int mdir_diffusion_merge(const float* plane, int64_t ld, int nb, int64_t col0, int64_t n_cols, const int32_t* tiles, int n_tiles,
                                    const uint32_t* live, const float* eps, const int64_t* bslot, const float* db32, int D,
                                    const uint32_t* slot_id, int32_t* knn_ids, float* knn_s, int k, uint64_t* seg, int cap, int32_t* cnt,
                                    int32_t* rep, void* stream) {
    MDIR_CHECK_ARG(plane && live && eps && bslot && db32 && slot_id && knn_ids && knn_s && seg && cnt && rep);
    MDIR_CHECK_ARG(nb >= 1 && n_cols >= 0 && ld >= n_cols && col0 >= 0 && col0 % kMergeCols == 0 && D >= 1 && k >= 1 && k <= kDiffMaxK);
    MDIR_CHECK_ARG(cap >= 1 && (tiles == nullptr || n_tiles >= 0));
    const int64_t grid = tiles ? n_tiles : (n_cols + kMergeCols - 1) / kMergeCols;
    if (grid == 0) return 0;
    MDIR_CHECK_ARG(grid < ((int64_t)1 << 31));
    diffusion_screen_kernel<<<(unsigned)grid, kMergeWarps * 32, 0, (cudaStream_t)stream>>>(plane, ld, nb, col0, n_cols, tiles, live, eps, knn_ids,
                                                                                           knn_s, k, seg, cap, cnt);
    MDIR_LAUNCH_CHECK();
    diffusion_merge_kernel<<<(unsigned)grid, kMergeWarps * 32, 0, (cudaStream_t)stream>>>(col0, n_cols, tiles, live, bslot, db32, D, slot_id, knn_ids,
                                                                                          knn_s, k, seg, cap, cnt, rep);
    MDIR_LAUNCH_CHECK();
    return 0;
}

extern "C" int mdir_diffusion_stale_rows(int32_t* knn_ids, float* knn_s, int64_t n_used, int k, const uint32_t* slot_id, const uint32_t* live,
                                         uint8_t* flag, void* stream) {
    MDIR_CHECK_ARG(knn_ids && knn_s && slot_id && live && flag && n_used >= 0 && k >= 1 && k <= kDiffMaxK);
    if (n_used == 0) return 0;
    diffusion_stale_kernel<<<(unsigned)((n_used + 7) / 8), 256, 0, (cudaStream_t)stream>>>(knn_ids, knn_s, n_used, k, slot_id, live, flag);
    MDIR_LAUNCH_CHECK();
    return 0;
}

extern "C" size_t mdir_diffusion_solve_workspace_bytes(int n_q, int trunc, int k) {
    if (n_q <= 0 || trunc < 1 || trunc > kDiffMaxTrunc || k < 1 || k > kDiffMaxK) return 0;
    return (size_t)(n_q < kDiffCtas ? n_q : kDiffCtas) * diff_ws_cta_bytes(trunc, k);
}

extern "C" int mdir_diffusion_solve_dev(const int32_t* L_ids, const float* L_s, int n_q, int trunc, const uint32_t* slot_id, int64_t n_used,
                                        const int32_t* nbr, const float* S, int k, int k_q, float gamma, double alpha, int iters, double rtol,
                                        int k_out, void* ws, size_t ws_bytes, float* f_out, int32_t* ids_out, const int64_t* n_used_dev,
                                        const int32_t* status, void* stream) {
    MDIR_CHECK_ARG(L_ids && L_s && slot_id && nbr && S && f_out && ids_out && n_q >= 0 && n_used >= 0);
    MDIR_CHECK_ARG(trunc >= 1 && trunc <= kDiffMaxTrunc && k >= 1 && k <= kDiffMaxK);
    MDIR_CHECK_ARG(k_q >= 1 && k_q <= trunc && k_out >= 1 && k_out <= trunc);
    MDIR_CHECK_ARG(alpha > 0.0 && alpha < 1.0 && gamma > 0.f && gamma <= FLT_MAX && iters >= 1 && iters <= 1000 && rtol >= 0.0);
    if (n_q == 0) return 0;
    MDIR_CHECK_ARG(ws && ws_bytes >= mdir_diffusion_solve_workspace_bytes(n_q, trunc, k));
    static PerDeviceOnce once;
    if (once.first() != 0) MDIR_CUDA(cudaFuncSetAttribute(diffusion_solve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kDiffSmem));
    const int grid = n_q < kDiffCtas ? n_q : kDiffCtas;
    diffusion_solve_kernel<<<grid, kDiffThreads, kDiffSmem, (cudaStream_t)stream>>>(L_ids, L_s, n_q, trunc, slot_id, n_used, nbr, S, k, k_q,
                                                                                   gamma, alpha, iters, rtol, k_out, (uint8_t*)ws, f_out,
                                                                                   ids_out, n_used_dev, status);
    MDIR_LAUNCH_CHECK();
    return 0;
}

extern "C" int mdir_diffusion_solve(const int32_t* L_ids, const float* L_s, int n_q, int trunc, const uint32_t* slot_id, int64_t n_used,
                                    const int32_t* nbr, const float* S, int k, int k_q, float gamma, double alpha, int iters, double rtol,
                                    int k_out, void* ws, size_t ws_bytes, float* f_out, int32_t* ids_out, void* stream) {
    return mdir_diffusion_solve_dev(L_ids, L_s, n_q, trunc, slot_id, n_used, nbr, S, k, k_q, gamma, alpha, iters, rtol, k_out, ws, ws_bytes,
                                    f_out, ids_out, nullptr, nullptr, stream);
}

extern "C" int mdir_diffusion_combine_dev(const int32_t* L_ids, const float* L_s, int n_q, int k_q, const uint32_t* slot_id, int64_t n_used,
                                          const int32_t* tab_ids, const float* tab_f, int width, float gamma, int k_out, float* f_out,
                                          int32_t* ids_out, const int64_t* n_used_dev, const int32_t* status, void* stream) {
    MDIR_CHECK_ARG(L_ids && L_s && slot_id && tab_ids && tab_f && f_out && ids_out && n_q >= 0 && n_used >= 0);
    MDIR_CHECK_ARG(k_q >= 1 && k_q <= kCombMaxKq && width >= 1 && width <= kCombMaxWidth && k_q * width <= kCombMaxEntries);
    MDIR_CHECK_ARG(k_out >= 1 && k_out <= kCombMaxEntries && gamma > 0.f && gamma <= FLT_MAX);
    if (n_q == 0) return 0;
    static PerDeviceOnce once;
    if (once.first() != 0)
        MDIR_CUDA(cudaFuncSetAttribute(diffusion_combine_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)comb_smem_bytes(kCombMaxEntries)));
    const int grid = n_q < kCombCtas ? n_q : kCombCtas;
    diffusion_combine_kernel<<<grid, kCombThreads, comb_smem_bytes(k_q * width), (cudaStream_t)stream>>>(
            L_ids, L_s, n_q, k_q, slot_id, n_used, tab_ids, tab_f, width, gamma, k_out, f_out, ids_out, n_used_dev, status);
    MDIR_LAUNCH_CHECK();
    return 0;
}

extern "C" int mdir_diffusion_combine(const int32_t* L_ids, const float* L_s, int n_q, int k_q, const uint32_t* slot_id, int64_t n_used,
                                      const int32_t* tab_ids, const float* tab_f, int width, float gamma, int k_out, float* f_out,
                                      int32_t* ids_out, void* stream) {
    return mdir_diffusion_combine_dev(L_ids, L_s, n_q, k_q, slot_id, n_used, tab_ids, tab_f, width, gamma, k_out, f_out, ids_out, nullptr,
                                      nullptr, stream);
}
