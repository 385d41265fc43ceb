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
        int iters, double rtol, int k_out, uint8_t* __restrict__ ws, float* __restrict__ f_out, int32_t* __restrict__ ids_out) {
    extern __shared__ __align__(16) uint8_t smem[];
    uint64_t* keys = reinterpret_cast<uint64_t*>(smem);                       // kDiffMaxTrunc
    double* x = reinterpret_cast<double*>(keys + kDiffMaxTrunc);
    double* r = x + kDiffMaxTrunc;
    double* p = r + kDiffMaxTrunc;
    double* ap = p + kDiffMaxTrunc;
    uint16_t* cnt = reinterpret_cast<uint16_t*>(ap + kDiffMaxTrunc);
    __shared__ double red[kDiffWarps];
    __shared__ int s_n;
    // this CTA's local ELL of S_LL, column-major: entry c of row u at c * trunc + u (u16 local index, fp32 S)
    uint16_t* ell_idx = reinterpret_cast<uint16_t*>(ws + (size_t)blockIdx.x * diff_ws_cta_bytes(trunc, k));
    float* ell_val = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(ell_idx) + (((size_t)trunc * k * 2 + 255) & ~(size_t)255));
    const int tid = threadIdx.x;

    for (int q = blockIdx.x; q < n_q; q += gridDim.x) {
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

extern "C" size_t mdir_diffusion_solve_workspace_bytes(int n_q, int trunc, int k) {
    if (n_q <= 0 || trunc < 1 || trunc > kDiffMaxTrunc || k < 1 || k > kDiffMaxK) return 0;
    return (size_t)(n_q < kDiffCtas ? n_q : kDiffCtas) * diff_ws_cta_bytes(trunc, k);
}

extern "C" int mdir_diffusion_solve(const int32_t* L_ids, const float* L_s, int n_q, int trunc, const uint32_t* slot_id, int64_t n_used,
                                    const int32_t* nbr, const float* S, int k, int k_q, float gamma, double alpha, int iters, double rtol,
                                    int k_out, void* ws, size_t ws_bytes, float* f_out, int32_t* ids_out, void* stream) {
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
                                                                                   ids_out);
    MDIR_LAUNCH_CHECK();
    return 0;
}
