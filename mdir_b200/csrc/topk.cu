// Selection machinery around the similarity scan: radix-select of the k-th key, candidate
// finalisation (bitonic sort in shared memory), fp32 shortlist re-scoring, fp32 -> bf16 packing.
// All orderings are on the 64-bit key (score descending, index ascending) of common.cuh, so
// results equal np.argsort(-scores, kind='stable')[:k] bit for bit.
#include <cuda_bf16.h>

#include "common.cuh"

namespace mdir {

__device__ __forceinline__ uint32_t sample_pos_to_idx(int64_t i, int sample_stride, uint32_t idx_base) {
    if (sample_stride <= 1) return idx_base + (uint32_t)i;
    const int64_t j = i / MDIR_SCAN_TILE_ROWS, r = i - j * MDIR_SCAN_TILE_ROWS;
    return idx_base + (uint32_t)(j * sample_stride * MDIR_SCAN_TILE_ROWS + r);
}

// kth smallest (1-based) of ONE 32-bit value per thread of a 1024-thread block (4 radix passes of
// one element each).  Used to bound the selection: the kth smallest of the per-thread minima is an
// upper bound B of the kth smallest key overall, so only the few keys <= B take part in the real
// selection passes (the warp-aggregated histogram update is the expensive part of a pass).
__device__ __forceinline__ uint32_t block_kth_of_thread_values(uint32_t val, uint32_t kth, uint32_t* hist, uint32_t* s_prefix,
                                                               uint32_t* s_k) {
    const int lane = threadIdx.x & 31;
    __syncthreads();
    if (threadIdx.x == 0) { *s_prefix = 0u; *s_k = kth; }
    for (int pass = 0; pass < 4; ++pass) {
        const int shift = 24 - 8 * pass;
        if (threadIdx.x < 256) hist[threadIdx.x] = 0u;
        __syncthreads();
        const uint32_t prefix = *s_prefix;
        const uint32_t himask = pass == 0 ? 0u : (0xffffffffu << (shift + 8));
        const bool hit = (val & himask) == prefix;
        if (__any_sync(0xffffffffu, hit)) {
            const int d = (int)((val >> shift) & 0xffu);
            const unsigned peers = match_digit8(d, hit);
            if (hit && lane == (__ffs(peers) - 1)) atomicAdd(&hist[d], (uint32_t)__popc(peers));
        }
        __syncthreads();
        if (threadIdx.x < 32) {
            uint32_t before;
            const int b = find_bin_warp0(hist, *s_k, &before);
            if (lane == 0) {
                *s_k -= before;
                *s_prefix = prefix | ((uint32_t)b << shift);
            }
        }
        __syncthreads();
    }
    const uint32_t r = *s_prefix;
    __syncthreads();
    return r;
}

// One CTA (1024 threads) per query.  MSB-first 8-bit radix select on the 32-bit score key
// (4 passes over the L2-resident score row, warp-aggregated shared-memory histogram updates).
// tau = (kth-best score key << 32) | index limit: normally 0xffffffff (the rows tying the kth
// score are all wanted); when more rows tie than are wanted, 4 more passes select the lowest
// indices among them, so exactly kth rows have key <= tau.  Those rows are appended to cand.
__global__ void __launch_bounds__(1024) select_kth_kernel(const float* __restrict__ scores, int64_t ld, int64_t n, int kth,
                                                          int sample_stride, uint32_t idx_base, uint64_t* __restrict__ tau,
                                                          uint64_t* __restrict__ cand, int64_t cand_row, uint32_t* __restrict__ seg_counts,
                                                          int n_seg, int cap) {
    __shared__ uint32_t hist[256];
    __shared__ uint32_t s_prefix;
    __shared__ uint32_t s_k;
    __shared__ uint32_t s_n;
    __shared__ uint32_t s_ties;
    const int q = blockIdx.x;
    const int lane = threadIdx.x & 31;
    const float* sc = scores + (int64_t)q * ld;
    uint32_t result;
    uint32_t idx_limit = 0xffffffffu;      // index part of tau (all ties pass unless narrowed below)
    const int64_t n_round = (n + 8191) & ~(int64_t)8191;
    if ((int64_t)kth > n) {
        result = 0xffffffffu;
    } else {
        uint32_t bound = 0xffffffffu;
        if (kth <= 1024) {                 // see block_kth_of_thread_values: one extra streaming pass for the bound
            uint32_t mymin = 0xffffffffu;
            for (int64_t base = 0; base < n_round; base += 8 * 1024) {
                float v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const int64_t i = base + u * 1024 + threadIdx.x;
                    v[u] = i < n ? __ldg(sc + i) : 0.f;
                }
#pragma unroll
                for (int u = 0; u < 8; ++u)
                    if (base + u * 1024 + threadIdx.x < n) mymin = min(mymin, desc_key(v[u]));
            }
            bound = block_kth_of_thread_values(mymin, (uint32_t)kth, hist, &s_prefix, &s_k);
        }
        if (threadIdx.x == 0) { s_prefix = 0u; s_k = (uint32_t)kth; }
        for (int pass = 0; pass < 4; ++pass) {
            const int shift = 24 - 8 * pass;
            if (threadIdx.x < 256) hist[threadIdx.x] = 0u;
            __syncthreads();
            const uint32_t prefix = s_prefix;
            const uint32_t himask = pass == 0 ? 0u : (0xffffffffu << (shift + 8));
            // 8 independent loads in flight per thread (the row is L2-resident; latency-bound otherwise)
            for (int64_t base = 0; base < n_round; base += 8 * 1024) {
                float v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const int64_t i = base + u * 1024 + threadIdx.x;
                    v[u] = i < n ? __ldg(sc + i) : 0.f;
                }
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const int64_t i = base + u * 1024 + threadIdx.x;
                    const bool valid = i < n;
                    const uint32_t key = desc_key(v[u]);
                    const bool hit = valid && key <= bound && ((key & himask) == prefix);
                    if (__any_sync(0xffffffffu, hit)) {
                        const int d = (int)((key >> shift) & 0xffu);
                        const unsigned peers = match_digit8(d, hit);
                        if (hit && lane == (__ffs(peers) - 1)) atomicAdd(&hist[d], (uint32_t)__popc(peers));
                    }
                }
            }
            __syncthreads();
            if (threadIdx.x < 32) {
                uint32_t before;
                const int b = find_bin_warp0(hist, s_k, &before);
                if (lane == 0) {
                    s_k -= before;
                    s_prefix = prefix | ((uint32_t)b << shift);
                    s_ties = hist[b];
                }
            }
            __syncthreads();
        }
        result = s_prefix;
        // s_k of the s_ties rows that tie the kth score are wanted.  When not all of them are, the
        // lowest indices win (stable-argsort order): radix-select the s_k-th smallest index among them.
        if (s_k < s_ties) {
            __syncthreads();
            if (threadIdx.x == 0) s_prefix = 0u;
            for (int pass = 0; pass < 4; ++pass) {
                const int shift = 24 - 8 * pass;
                if (threadIdx.x < 256) hist[threadIdx.x] = 0u;
                __syncthreads();
                const uint32_t prefix = s_prefix;
                const uint32_t himask = pass == 0 ? 0u : (0xffffffffu << (shift + 8));
                for (int64_t base = 0; base < n_round; base += 1024) {
                    const int64_t i = base + threadIdx.x;
                    const bool valid = i < n;
                    const float v = valid ? __ldg(sc + i) : 0.f;
                    const uint32_t idx = sample_pos_to_idx(valid ? i : 0, sample_stride, idx_base);
                    const bool hit = valid && (desc_key(v) == result) && ((idx & himask) == prefix);
                    if (__any_sync(0xffffffffu, hit)) {
                        const int d = (int)((idx >> shift) & 0xffu);
                        const unsigned peers = match_digit8(d, hit);
                        if (hit && lane == (__ffs(peers) - 1)) atomicAdd(&hist[d], (uint32_t)__popc(peers));
                    }
                }
                __syncthreads();
                if (threadIdx.x < 32) {
                    uint32_t before;
                    const int b = find_bin_warp0(hist, s_k, &before);
                    if (lane == 0) {
                        s_k -= before;
                        s_prefix = prefix | ((uint32_t)b << shift);
                    }
                }
                __syncthreads();
            }
            idx_limit = s_prefix;
        }
    }
    const uint64_t tau_key = ((uint64_t)result << 32) | (uint64_t)idx_limit;
    __syncthreads();          // s_prefix / s_k / s_ties share a vector word with s_n: every read of them is done
    if (threadIdx.x == 0) { tau[q] = tau_key; s_n = 0u; }
    if (cand) {
        __syncthreads();
        for (int64_t base = 0; base < n_round; base += 8 * 1024) {
            float v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int64_t i = base + u * 1024 + threadIdx.x;
                v[u] = i < n ? __ldg(sc + i) : -INFINITY;
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int64_t i = base + u * 1024 + threadIdx.x;
                if (i < n && desc_key(v[u]) <= result) {
                    const uint64_t key = make_key(v[u], sample_pos_to_idx(i, sample_stride, idx_base));
                    if (key <= tau_key) {
                        const uint32_t pos = atomicAdd(&s_n, 1u);
                        if (pos < (uint32_t)cap) cand[(int64_t)q * cand_row + pos] = key;
                    }
                }
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) seg_counts[(int64_t)q * n_seg] = s_n;      // segment 0 of this query
        for (int sg = 1 + threadIdx.x; sg < n_seg; sg += blockDim.x) seg_counts[(int64_t)q * n_seg + sg] = 0u;   // producers of the next pass start from 0
    }
}

// Register-resident variant for n <= 32 * 1024 rows (the usual sample size): every thread keeps its
// 32 score keys in registers, so the 4 (+4) radix passes and the append pass never re-read the row.
__global__ void __launch_bounds__(1024, 1) select_kth_reg_kernel(const float* __restrict__ scores, int64_t ld, int n, int kth,
                                                                 int sample_stride, uint32_t idx_base, uint64_t* __restrict__ tau,
                                                                 uint64_t* __restrict__ cand, int64_t cand_row,
                                                                 uint32_t* __restrict__ seg_counts, int n_seg, int cap, int approx) {
    __shared__ uint32_t hist[256];
    __shared__ uint32_t s_prefix, s_k, s_n, s_ties;
    const int q = blockIdx.x;
    const int lane = threadIdx.x & 31;
    const float* sc = scores + (int64_t)q * ld;
    uint32_t key[32];
#pragma unroll
    for (int u = 0; u < 32; ++u) {
        const int i = u * 1024 + threadIdx.x;
        key[u] = i < n ? desc_key(__ldg(sc + i)) : 0xffffffffu;     // padding sorts last (and is never valid)
    }
    uint32_t result = 0xffffffffu, idx_limit = 0xffffffffu;
    if (kth <= n) {
        uint32_t bound = 0xffffffffu;
        if (kth <= 1024) {
            uint32_t mymin = 0xffffffffu;
#pragma unroll
            for (int u = 0; u < 32; ++u)
                if (u * 1024 + (int)threadIdx.x < n) mymin = min(mymin, key[u]);
            bound = block_kth_of_thread_values(mymin, (uint32_t)kth, hist, &s_prefix, &s_k);
        }
        // approx: the bound itself is a valid threshold (>= kth keys are <= it, typically ~7 % more than kth)
        const bool use_bound = approx && kth <= 1024;
        if (threadIdx.x == 0) { s_prefix = use_bound ? bound : 0u; s_k = use_bound ? 0u : (uint32_t)kth; s_ties = 0u; }
        if (use_bound) __syncthreads();
        for (int pass = 0; pass < (use_bound ? 0 : 4); ++pass) {
            const int shift = 24 - 8 * pass;
            if (threadIdx.x < 256) hist[threadIdx.x] = 0u;
            __syncthreads();
            const uint32_t prefix = s_prefix;
            const uint32_t himask = pass == 0 ? 0u : (0xffffffffu << (shift + 8));
#pragma unroll
            for (int u = 0; u < 32; ++u) {
                const bool valid = u * 1024 + (int)threadIdx.x < n;
                const bool hit = valid && key[u] <= bound && ((key[u] & himask) == prefix);
                if (__any_sync(0xffffffffu, hit)) {
                    const int d = (int)((key[u] >> shift) & 0xffu);
                    const unsigned peers = match_digit8(d, hit);
                    if (hit && lane == (__ffs(peers) - 1)) atomicAdd(&hist[d], (uint32_t)__popc(peers));
                }
            }
            __syncthreads();
            if (threadIdx.x < 32) {
                uint32_t before;
                const int b = find_bin_warp0(hist, s_k, &before);
                if (lane == 0) {
                    s_k -= before;
                    s_prefix = prefix | ((uint32_t)b << shift);
                    s_ties = hist[b];
                }
            }
            __syncthreads();
        }
        result = s_prefix;
        if (s_k < s_ties) {            // more rows tie the kth score than are wanted: lowest indices win
            __syncthreads();
            if (threadIdx.x == 0) s_prefix = 0u;
            for (int pass = 0; pass < 4; ++pass) {
                const int shift = 24 - 8 * pass;
                if (threadIdx.x < 256) hist[threadIdx.x] = 0u;
                __syncthreads();
                const uint32_t prefix = s_prefix;
                const uint32_t himask = pass == 0 ? 0u : (0xffffffffu << (shift + 8));
#pragma unroll
                for (int u = 0; u < 32; ++u) {
                    const int i = u * 1024 + threadIdx.x;
                    const uint32_t idx = sample_pos_to_idx(i, sample_stride, idx_base);
                    const bool hit = i < n && key[u] == result && ((idx & himask) == prefix);
                    if (__any_sync(0xffffffffu, hit)) {
                        const int d = (int)((idx >> shift) & 0xffu);
                        const unsigned peers = match_digit8(d, hit);
                        if (hit && lane == (__ffs(peers) - 1)) atomicAdd(&hist[d], (uint32_t)__popc(peers));
                    }
                }
                __syncthreads();
                if (threadIdx.x < 32) {
                    uint32_t before;
                    const int b = find_bin_warp0(hist, s_k, &before);
                    if (lane == 0) {
                        s_k -= before;
                        s_prefix = prefix | ((uint32_t)b << shift);
                    }
                }
                __syncthreads();
            }
            idx_limit = s_prefix;
        }
    }
    const uint64_t tau_key = ((uint64_t)result << 32) | (uint64_t)idx_limit;
    __syncthreads();          // s_prefix / s_k / s_ties share a vector word with s_n: every read of them is done
    if (threadIdx.x == 0) { tau[q] = tau_key; s_n = 0u; }
    if (cand) {
        __syncthreads();
#pragma unroll
        for (int u = 0; u < 32; ++u) {
            const int i = u * 1024 + threadIdx.x;
            if (i < n && key[u] <= result) {
                // key = (desc_key(score) << 32) | idx: the upper half is exactly the register key
                const uint64_t k64 = ((uint64_t)key[u] << 32) | (uint64_t)sample_pos_to_idx(i, sample_stride, idx_base);
                if (k64 <= tau_key) {
                    const uint32_t pos = atomicAdd(&s_n, 1u);
                    if (pos < (uint32_t)cap) cand[(int64_t)q * cand_row + pos] = k64;
                }
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) seg_counts[(int64_t)q * n_seg] = s_n;
        for (int sg = 1 + threadIdx.x; sg < n_seg; sg += blockDim.x) seg_counts[(int64_t)q * n_seg + sg] = 0u;
    }
}

// ---- thread-block-cluster helpers (distributed shared memory) for the split re-scoring in topk_finalize_kernel
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// address of `p` (a shared-memory object of this kernel) inside CTA `rank` of the cluster
__device__ __forceinline__ uint32_t cluster_map(const void* p, uint32_t rank) {
    const uint32_t a = (uint32_t)__cvta_generic_to_shared(p);
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(rank));
    return r;
}
__device__ __forceinline__ uint64_t cluster_ld_u64(uint32_t a) {
    uint64_t v;
    asm volatile("ld.shared::cluster.u64 %0, [%1];" : "=l"(v) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ void cluster_st_u64(uint32_t a, uint64_t v) {
    asm volatile("st.shared::cluster.u64 [%0], %1;" ::"r"(a), "l"(v) : "memory");
}
__device__ __forceinline__ int cluster_ld_s32(uint32_t a) {
    int v;
    asm volatile("ld.shared::cluster.s32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
    return v;
}

// fp32 dot product of one database row with the query staged in shared memory, one warp per row
__device__ __forceinline__ float rescore_row(const float* __restrict__ a, const float* qs, int D, int lane) {
    float acc = 0.f;
    if ((D & 3) == 0) {
        const float4* a4 = reinterpret_cast<const float4*>(a);
        const float4* b4 = reinterpret_cast<const float4*>(qs);
        const int n4 = D >> 2;
        float acc1 = 0.f, acc2 = 0.f, acc3 = 0.f;
        int i = lane;
        for (; i + 96 < n4; i += 128) {            // 4 independent 128-bit loads in flight per lane
            const float4 x0 = __ldg(a4 + i), x1 = __ldg(a4 + i + 32), x2 = __ldg(a4 + i + 64), x3 = __ldg(a4 + i + 96);
            const float4 y0 = b4[i], y1 = b4[i + 32], y2 = b4[i + 64], y3 = b4[i + 96];
            acc = fmaf(x0.x, y0.x, acc); acc = fmaf(x0.y, y0.y, acc); acc = fmaf(x0.z, y0.z, acc); acc = fmaf(x0.w, y0.w, acc);
            acc1 = fmaf(x1.x, y1.x, acc1); acc1 = fmaf(x1.y, y1.y, acc1); acc1 = fmaf(x1.z, y1.z, acc1); acc1 = fmaf(x1.w, y1.w, acc1);
            acc2 = fmaf(x2.x, y2.x, acc2); acc2 = fmaf(x2.y, y2.y, acc2); acc2 = fmaf(x2.z, y2.z, acc2); acc2 = fmaf(x2.w, y2.w, acc2);
            acc3 = fmaf(x3.x, y3.x, acc3); acc3 = fmaf(x3.y, y3.y, acc3); acc3 = fmaf(x3.z, y3.z, acc3); acc3 = fmaf(x3.w, y3.w, acc3);
        }
        for (; i < n4; i += 32) {
            const float4 x = __ldg(a4 + i), y = b4[i];
            acc = fmaf(x.x, y.x, acc); acc = fmaf(x.y, y.y, acc); acc = fmaf(x.z, y.z, acc); acc = fmaf(x.w, y.w, acc);
        }
        acc = (acc + acc1) + (acc2 + acc3);
    } else {
        for (int i = lane; i < D; i += 32) acc = fmaf(a[i], qs[i], acc);
    }
    return warp_sum(acc);
}

// The k smallest of the cnt unique keys in skeys[0, cnt) (1024-thread block), sorted ascending into out[0, min(k, cnt))
// (padded with ~0 up to kpow2), without the 8 MSB radix passes: candidates of one query share sign and exponent, so
// ONE histogram over 1024 bins linear between the smallest and the largest key separates them; the bins up to the
// one where the running count reaches k hold k + a few keys, which are compacted behind the list (skeys[cnt, cnt + 1024))
// and rank-counted.  Returns false (nothing written) when those bins hold more than 1024 keys (massive ties): the
// caller then takes the radix path.  scratch: 64 words.
__device__ __forceinline__ bool topk_hist_select(uint64_t* skeys, int cnt, int k, int kpow2, uint64_t* out, uint32_t* hist, uint32_t* s_n,
                                                 uint32_t* scratch) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    uint32_t mn = 0xffffffffu, mx = 0u;
    for (int i = threadIdx.x; i < cnt; i += blockDim.x) {
        const uint32_t h = (uint32_t)(skeys[i] >> 32);
        mn = min(mn, h);
        mx = max(mx, h);
    }
    mn = __reduce_min_sync(0xffffffffu, mn);
    mx = __reduce_max_sync(0xffffffffu, mx);
    if (lane == 0) { scratch[w] = mn; scratch[32 + w] = mx; }
    hist[threadIdx.x] = 0u;
    if (threadIdx.x == 0) *s_n = 0u;
    __syncthreads();
    mn = scratch[lane];
    mx = scratch[32 + lane];
    mn = __reduce_min_sync(0xffffffffu, mn);
    mx = __reduce_max_sync(0xffffffffu, mx);
    const float scale = 1024.0f / ((float)(mx - mn) + 1.0f);
    auto bin_of = [&](uint64_t key) { return min(1023, (int)((float)((uint32_t)(key >> 32) - mn) * scale)); };     // monotone in the key
    for (int i = threadIdx.x; i < cnt; i += blockDim.x) atomicAdd(&hist[bin_of(skeys[i])], 1u);
    __syncthreads();
    // inclusive scan over the 1024 bins, one per thread
    const uint32_t c = hist[threadIdx.x];
    uint32_t incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    __syncthreads();                                   // scratch (min / max) fully read
    if (lane == 31) scratch[w] = incl;
    __syncthreads();
    uint32_t pre = 0;
    for (int j = 0; j < w; ++j) pre += scratch[j];
    incl += pre;
    // the first bin where the running count reaches k: everything up to it is wanted
    if (incl >= (uint32_t)k && incl - c < (uint32_t)k) { scratch[32] = threadIdx.x; scratch[33] = incl; }
    if (threadIdx.x == 1023 && incl < (uint32_t)k) { scratch[32] = 1023u; scratch[33] = incl; }      // fewer than k keys in all
    __syncthreads();
    const int b_star = (int)scratch[32];
    const int take = (int)scratch[33];
    if (take > 1024) return false;
    uint64_t* sel = skeys + cnt;
    for (int i = threadIdx.x; i < cnt; i += blockDim.x) {
        const uint64_t key = skeys[i];
        if (bin_of(key) <= b_star) sel[atomicAdd(s_n, 1u)] = key;
    }
    for (int i = threadIdx.x; i < kpow2; i += blockDim.x) out[i] = ~0ull;
    __syncthreads();
    if ((int)threadIdx.x < take) {
        const uint64_t mine = sel[threadIdx.x];
        int r = 0;
        for (int j = 0; j < take; ++j) r += sel[j] < mine ? 1 : 0;
        if (r < kpow2) out[r] = mine;
    }
    __syncthreads();
    return true;
}

// Rescore entries [j0, j0 + n) of the key list at shared-memory address `list` of cluster rank 0 (DSMEM when this
// CTA is a helper): one warp per row, rows interleaved over the CS CTAs of the cluster.
// fp32 dot products of TWO database rows with the staged query, both rows' loads in flight together
__device__ __forceinline__ void rescore_row2(const float* __restrict__ a0, const float* __restrict__ a1, const float* qs, int D, int lane,
                                             float& r0, float& r1) {
    if ((D & 3) != 0) {
        r0 = rescore_row(a0, qs, D, lane);
        r1 = rescore_row(a1, qs, D, lane);
        return;
    }
    const float4* p0 = reinterpret_cast<const float4*>(a0);
    const float4* p1 = reinterpret_cast<const float4*>(a1);
    const float4* b4 = reinterpret_cast<const float4*>(qs);
    const int n4 = D >> 2;
    float s0a = 0.f, s0b = 0.f, s1a = 0.f, s1b = 0.f;
    int i = lane;
    for (; i + 96 < n4; i += 128) {           // 2 x 4 independent 128-bit loads in flight per lane (4 KB per warp)
        const float4 x0 = __ldg(p0 + i), x1 = __ldg(p0 + i + 32), x2 = __ldg(p0 + i + 64), x3 = __ldg(p0 + i + 96);
        const float4 z0 = __ldg(p1 + i), z1 = __ldg(p1 + i + 32), z2 = __ldg(p1 + i + 64), z3 = __ldg(p1 + i + 96);
        float4 y = b4[i];
        s0a = fmaf(x0.x, y.x, s0a); s0a = fmaf(x0.y, y.y, s0a); s0a = fmaf(x0.z, y.z, s0a); s0a = fmaf(x0.w, y.w, s0a);
        s1a = fmaf(z0.x, y.x, s1a); s1a = fmaf(z0.y, y.y, s1a); s1a = fmaf(z0.z, y.z, s1a); s1a = fmaf(z0.w, y.w, s1a);
        y = b4[i + 32];
        s0b = fmaf(x1.x, y.x, s0b); s0b = fmaf(x1.y, y.y, s0b); s0b = fmaf(x1.z, y.z, s0b); s0b = fmaf(x1.w, y.w, s0b);
        s1b = fmaf(z1.x, y.x, s1b); s1b = fmaf(z1.y, y.y, s1b); s1b = fmaf(z1.z, y.z, s1b); s1b = fmaf(z1.w, y.w, s1b);
        y = b4[i + 64];
        s0a = fmaf(x2.x, y.x, s0a); s0a = fmaf(x2.y, y.y, s0a); s0a = fmaf(x2.z, y.z, s0a); s0a = fmaf(x2.w, y.w, s0a);
        s1a = fmaf(z2.x, y.x, s1a); s1a = fmaf(z2.y, y.y, s1a); s1a = fmaf(z2.z, y.z, s1a); s1a = fmaf(z2.w, y.w, s1a);
        y = b4[i + 96];
        s0b = fmaf(x3.x, y.x, s0b); s0b = fmaf(x3.y, y.y, s0b); s0b = fmaf(x3.z, y.z, s0b); s0b = fmaf(x3.w, y.w, s0b);
        s1b = fmaf(z3.x, y.x, s1b); s1b = fmaf(z3.y, y.y, s1b); s1b = fmaf(z3.z, y.z, s1b); s1b = fmaf(z3.w, y.w, s1b);
    }
    for (; i < n4; i += 32) {
        const float4 x = __ldg(p0 + i), z = __ldg(p1 + i), y = b4[i];
        s0a = fmaf(x.x, y.x, s0a); s0a = fmaf(x.y, y.y, s0a); s0a = fmaf(x.z, y.z, s0a); s0a = fmaf(x.w, y.w, s0a);
        s1a = fmaf(z.x, y.x, s1a); s1a = fmaf(z.y, y.y, s1a); s1a = fmaf(z.z, y.z, s1a); s1a = fmaf(z.w, y.w, s1a);
    }
    r0 = warp_sum(s0a + s0b);
    r1 = warp_sum(s1a + s1b);
}

// Rescore entries [j0, j0 + n) of the key list at shared-memory address `list` of cluster rank 0 (DSMEM when this
// CTA is a helper): one warp per row, rows interleaved over the CS CTAs of the cluster, two rows of a warp in flight
// together (a row is 4 * D bytes gathered from HBM: latency, not bandwidth, is what a warp waits for).
template <int CS>
__device__ __forceinline__ void rescore_share(uint64_t* local_list, uint32_t remote_list, bool remote, int j0, int n, int crank,
                                              const float* __restrict__ db32, int64_t n_db, uint32_t idx_base, const float* qs, int D) {
    const int lane = threadIdx.x & 31;
    for (int j = (threadIdx.x >> 5) * CS + crank; j < n; j += 64 * CS) {
        const int jb = j + 32 * CS;                       // this warp's second row of the round
        const uint64_t key0 = remote ? cluster_ld_u64(remote_list + 8u * (uint32_t)(j0 + j)) : local_list[j0 + j];
        uint64_t key1 = ~0ull;
        if (jb < n) key1 = remote ? cluster_ld_u64(remote_list + 8u * (uint32_t)(j0 + jb)) : local_list[j0 + jb];
        const uint32_t g0 = (uint32_t)key0, g1 = (uint32_t)key1;
        const int64_t row0 = (int64_t)g0 - (int64_t)idx_base, row1 = (int64_t)g1 - (int64_t)idx_base;
        const bool ok0 = key0 != ~0ull && row0 >= 0 && row0 < n_db, ok1 = key1 != ~0ull && row1 >= 0 && row1 < n_db;
        float s0 = 0.f, s1 = 0.f;
        if (ok0 && ok1) rescore_row2(db32 + row0 * D, db32 + row1 * D, qs, D, lane, s0, s1);
        else if (ok0) s0 = rescore_row(db32 + row0 * D, qs, D, lane);
        else if (ok1) s1 = rescore_row(db32 + row1 * D, qs, D, lane);
        const uint64_t n0 = ok0 ? make_key(s0, g0) : ~0ull, n1 = ok1 ? make_key(s1, g1) : ~0ull;
        __syncwarp();
        if (lane == 0) {
            if (remote) {
                cluster_st_u64(remote_list + 8u * (uint32_t)(j0 + j), n0);
                if (jb < n) cluster_st_u64(remote_list + 8u * (uint32_t)(j0 + jb), n1);
            } else {
                local_list[j0 + j] = n0;
                if (jb < n) local_list[j0 + jb] = n1;
            }
        }
    }
}

// One CTA (1024 threads) per query.  The candidates of a query live in n_seg segments of its
// cand row (segment 0: cap0 slots, the others cap_l slots each; seg_counts holds how many each
// producer appended).  They are compacted into shared memory; when there are many more than k,
// the k best are first isolated by an in-smem MSB radix select (keys are unique) and only those
// are sorted.  dynamic smem = (smem_cap + sl_cap) * 8 (+ D * 4 when re-scoring) bytes.
//
// Re-scoring (db32 != NULL) with the shortlist CERTIFICATE (db_stats != NULL).  The k best keys by bf16 score are
// re-scored exactly in fp32 (one warp per row).  Let t be the k_out-th best fp32 score among them and eps a bound
// on |bf16-path score - fp32 score| for any database row against this query:
//     eps = max_r ||bf16(x_r) - x_r|| * ||bf16(q)||  +  max_r ||x_r|| * ||bf16(q) - q||        (Cauchy-Schwarz on the
//           + 1.25 * D * 2^-24 * max_r ||x_r|| * ||q||                                          two rounding residuals,
// (db_stats = {max_r ||bf16(x_r) - x_r||^2, max_r ||x_r||^2}, from mdir_pack_stats).           + fp32 accumulation)
// A row whose bf16 score is below t - eps cannot reach the fp32 top k_out.  Every candidate at or above t - eps that
// is not yet in the shortlist is appended ("extension") and re-scored too; t can only rise, so one round suffices.
// The answer is then PROVEN equal to the exact fp32 top k_out of the whole shard provided the candidate list
// contains every row with bf16 score >= t - eps, i.e. the filter threshold tau[q] is not tighter than that bound
// and nothing overflowed.  Otherwise status bit 1 (uncertified) is raised and the host widens the selection.
// q_eps != NULL: the filter scores came from another encoding (the int8 scan) and q_eps[q] is that encoding's bound
// for query q (mdir_pack_q_i8), used instead of the bf16 formula above.
// status[q]: bit 0 = a candidate segment / the staging area overflowed, bit 1 = not certified.
template <int CS>      // CS = CTAs per query (thread-block cluster size): rank 0 selects and sorts, all ranks share the fp32 re-scoring
__global__ void __launch_bounds__(1024) topk_finalize_kernel(const uint64_t* __restrict__ cand, int64_t cand_row,
                                                             const uint32_t* __restrict__ seg_counts, int n_seg, int cap0, int cap_l,
                                                             int k, int smem_cap, int sl_cap, float* __restrict__ out_scores,
                                                             int32_t* __restrict__ out_idx, uint64_t* __restrict__ out_keys,
                                                             uint64_t* __restrict__ tau, int32_t* __restrict__ overflow,
                                                             const float* __restrict__ db32, int64_t n_db, uint32_t idx_base,
                                                             const float* __restrict__ q32, int D, int k_out,
                                                             const float* __restrict__ db_stats, const float* __restrict__ q_eps) {
    extern __shared__ uint64_t skeys[];
    __shared__ uint32_t hist[256];
    __shared__ uint64_t s_prefix;
    __shared__ uint32_t s_k, s_done, s_out;
    __shared__ int s_off[MDIR_CAND_SEGS + 1];
    __shared__ int s_ovf;
    __shared__ int s_hdr[3];                      // rank 0 -> helpers: {shortlist length, offset of the list in skeys, extension length}
    __shared__ uint64_t s_tkey;
    __shared__ float s_red[96];
    __shared__ uint32_t hist_sel[1024];
    uint64_t* sorted = skeys + smem_cap;          // sl_cap entries: the sorted selection; with re-scoring the shortlist + its extension
    const int q = blockIdx.x / CS;
    const int crank = CS > 1 ? (int)cluster_ctarank() : 0;
    const int lane = threadIdx.x & 31;
    int kpow2 = 32;
    while (kpow2 < k) kpow2 <<= 1;
    if (CS > 1 && crank != 0) {
        // helper CTA of the cluster: stage the query, then re-score its share of the shortlist and of the extension
        float* qs = reinterpret_cast<float*>(sorted + sl_cap);
        for (int i = threadIdx.x; i < D; i += blockDim.x) qs[i] = q32[(int64_t)q * D + i];
        __syncthreads();
        cluster_sync_all();                                            // (1) shortlist ready in rank 0's shared memory
        const int nk = cluster_ld_s32(cluster_map(&s_hdr[0], 0));
        const int off = cluster_ld_s32(cluster_map(&s_hdr[1], 0));
        const uint32_t rk0 = cluster_map(skeys + off, 0);
        rescore_share<CS>(nullptr, rk0, true, 0, nk, crank, db32, n_db, idx_base, qs, D);
        cluster_sync_all();                                            // (2) every share is back in rank 0
        cluster_sync_all();                                            // (3) extension ready
        const int n_ext = cluster_ld_s32(cluster_map(&s_hdr[2], 0));
        rescore_share<CS>(nullptr, rk0, true, nk, n_ext, crank, db32, n_db, idx_base, qs, D);
        cluster_sync_all();                                            // (4) extension shares are back
        return;
    }
    const uint64_t tau_in = tau ? tau[q] : ~0ull;
    // segment offsets (exclusive scan of the clamped counts) by warp 0; the (at most 5) count loads of a lane are all
    // issued before the first is used
    if (threadIdx.x < 32) {
        constexpr int kRounds = (MDIR_CAND_SEGS + 31) / 32;
        uint32_t raw[kRounds];
#pragma unroll
        for (int i = 0; i < kRounds; ++i) {
            const int sg = i * 32 + lane;
            raw[i] = sg < n_seg ? seg_counts[(int64_t)q * n_seg + sg] : 0u;
        }
        int run = 0, ovf = 0;
#pragma unroll
        for (int i = 0; i < kRounds; ++i) {
            const int sg = i * 32 + lane;
            int c = 0;
            if (sg < n_seg) {
                const uint32_t cp = (uint32_t)(sg == 0 ? cap0 : cap_l);
                if (raw[i] > cp) ovf = 1;
                c = (int)min(raw[i], cp);
            }
            int incl = c;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += t;
            }
            if (sg < n_seg) s_off[sg] = run + incl - c;
            run += __shfl_sync(0xffffffffu, incl, 31);
        }
        ovf = __any_sync(0xffffffffu, ovf);
        if (lane == 0) { s_off[n_seg] = run; s_ovf = ovf; }
    }
    __syncthreads();
    const int total = s_off[n_seg];
    const int cnt = min(total, smem_cap);
    const bool ovf_any = s_ovf || total > smem_cap;
    {   // compaction by OUTPUT slot: slot p belongs to the segment found by a binary search over the offsets, so every
        // thread's loads are independent of each other (a warp-per-segment loop paid one global latency per segment)
        const uint64_t* row = cand + (int64_t)q * cand_row;
        for (int p = threadIdx.x; p < cnt; p += blockDim.x) {
            int lo = 0, hi = n_seg;                               // last segment with s_off[sg] <= p
            while (hi - lo > 1) {
                const int mid = (lo + hi) >> 1;
                if (s_off[mid] <= p) lo = mid; else hi = mid;
            }
            const int64_t base = lo == 0 ? 0 : (int64_t)cap0 + (int64_t)(lo - 1) * cap_l;
            skeys[p] = row[base + (p - s_off[lo])];
        }
    }
    __syncthreads();
    const uint64_t* res;       // ascending keys, at least min(k, cnt) valid
    int nres;
    if (cnt > k + 96 && cnt + 1024 <= smem_cap &&
        topk_hist_select(skeys, cnt, k, kpow2, sorted, hist_sel, &s_out, reinterpret_cast<uint32_t*>(s_red))) {
        // the k best keys isolated by ONE histogram over bins linear between the extreme keys, then rank-counted
        res = sorted;
        nres = min(cnt, k);
    } else if (cnt <= 1024 && cnt + kpow2 <= smem_cap) {
        // few candidates: rank-counting sort (cnt^2 / 1024 comparisons per thread, no barriers inside)
        uint64_t mine = ~0ull;
        int r = 0;
        if ((int)threadIdx.x < cnt) {
            mine = skeys[threadIdx.x];
            for (int j = 0; j < cnt; ++j) r += skeys[j] < mine ? 1 : 0;          // keys are unique
        }
        __syncthreads();
        if ((int)threadIdx.x < cnt) skeys[r] = mine;
        for (int i = cnt + threadIdx.x; i < cnt + kpow2 && i < smem_cap; i += blockDim.x) skeys[i] = ~0ull;
        __syncthreads();
        res = skeys;
        nres = cnt;
    } else if (cnt <= 2 * kpow2 || cnt <= 1024) {
        int n = 32;
        while (n < cnt) n <<= 1;
        for (int i = cnt + threadIdx.x; i < n; i += blockDim.x) skeys[i] = ~0ull;
        __syncthreads();
        bitonic_sort_smem(skeys, n);
        res = skeys;
        nres = cnt;
    } else {
        if (threadIdx.x == 0) { s_prefix = 0ull; s_k = (uint32_t)k; s_done = 0u; s_out = 0u; }
        __syncthreads();
        const int cnt_round = (cnt + 1023) & ~1023;
        uint64_t thresh = ~0ull;
        for (int pass = 0; pass < 8; ++pass) {
            const int shift = 56 - 8 * pass;
            if (threadIdx.x < 256) hist[threadIdx.x] = 0u;
            __syncthreads();
            const uint64_t prefix = s_prefix;
            const uint64_t himask = pass == 0 ? 0ull : (~0ull << (shift + 8));
            for (int i = threadIdx.x; i < cnt_round; i += 1024) {
                const bool valid = i < cnt;
                const uint64_t key = valid ? skeys[i] : 0ull;
                const bool hit = valid && ((key & himask) == prefix);
                if (__any_sync(0xffffffffu, hit)) {
                    const int d = (int)((key >> shift) & 0xffu);
                    const unsigned peers = match_digit8(d, hit);
                    if (hit && lane == (__ffs(peers) - 1)) atomicAdd(&hist[d], (uint32_t)__popc(peers));
                }
            }
            __syncthreads();
            if (threadIdx.x < 32) {
                uint32_t before;
                const int b = find_bin_warp0(hist, s_k, &before);
                if (lane == 0) {
                    const uint32_t need = s_k - before;
                    s_k = need;
                    s_prefix = prefix | ((uint64_t)b << shift);
                    // the whole bin is wanted: everything with this prefix is in the top k
                    if (need == hist[b] || shift == 0) s_done = 1u;
                }
            }
            __syncthreads();
            if (s_done) {
                thresh = s_prefix | (shift ? ((1ull << shift) - 1ull) : 0ull);
                break;
            }
        }
        for (int i = threadIdx.x; i < kpow2; i += blockDim.x) sorted[i] = ~0ull;
        __syncthreads();
        for (int i = threadIdx.x; i < cnt; i += blockDim.x) {
            const uint64_t key = skeys[i];
            if (key <= thresh) {
                const uint32_t pos = atomicAdd(&s_out, 1u);
                if (pos < (uint32_t)kpow2) sorted[pos] = key;
            }
        }
        __syncthreads();
        bitonic_sort_smem(sorted, kpow2);
        res = sorted;
        nres = min(cnt, k);
    }
    int status = ovf_any ? 1 : 0;
    if (threadIdx.x == 0 && ovf_any && tau && nres > 0) tau[q] = res[min(k, nres) - 1];
    int k_emit = k;
    if (db32) {
        // ---- exact fp32 re-scoring of the bf16 shortlist (+ certified extension) ----
        uint64_t* sl = sorted;
        float* qs = reinterpret_cast<float*>(sorted + sl_cap);
        const int nk = min(k, nres);
        if (res != sl) {                           // small candidate sets were sorted in place: move the shortlist out
            for (int j = threadIdx.x; j < nk; j += blockDim.x) sl[j] = res[j];
        }
        float q2 = 0.f, qt2 = 0.f, qf2 = 0.f;
        for (int i = threadIdx.x; i < D; i += blockDim.x) {
            const float v = q32[(int64_t)q * D + i];
            qs[i] = v;
            const float vt = __bfloat162float(__float2bfloat16_rn(v));
            q2 = fmaf(v, v, q2);
            qt2 = fmaf(vt, vt, qt2);
            qf2 = fmaf(v - vt, v - vt, qf2);
        }
        if (threadIdx.x == 0) { s_hdr[0] = nk; s_hdr[1] = (int)(sl - skeys); s_hdr[2] = 0; s_out = 0u; s_tkey = ~0ull; }
        __syncthreads();
        const uint64_t last16 = nk > 0 ? sl[nk - 1] : 0ull;          // worst bf16 key inside the shortlist
        float eps = 0.f;
        if (db_stats && q_eps) {
            eps = q_eps[q];
        } else if (db_stats) {
            // one block reduction for the three sums
            q2 = warp_sum(q2); qt2 = warp_sum(qt2); qf2 = warp_sum(qf2);
            const int wi = threadIdx.x >> 5;
            if (lane == 0) { s_red[wi] = q2; s_red[32 + wi] = qt2; s_red[64 + wi] = qf2; }
            __syncthreads();
            q2 = warp_sum(s_red[lane]); qt2 = warp_sum(s_red[32 + lane]); qf2 = warp_sum(s_red[64 + lane]);
            const float e_max = sqrtf(db_stats[0]), x_max = sqrtf(db_stats[1]);
            eps = e_max * sqrtf(qt2) + x_max * sqrtf(qf2) + 1.25f * (float)D * 5.9604645e-8f * x_max * sqrtf(q2);
            eps = eps * 1.001f + 1e-7f;                              // slack for evaluating the bound itself in fp32
        }
        __syncthreads();
        if (CS > 1) cluster_sync_all();                                // (1) helpers may read the shortlist
        rescore_share<CS>(sl, 0u, false, 0, nk, 0, db32, n_db, idx_base, qs, D);
        if (CS > 1) cluster_sync_all();                                // (2) helpers' shares have landed
        __syncthreads();
        int n_ext = 0;
        if (db_stats) {
            // t = k_out-th best re-scored key (rank counting; the in-place bitonic sort when the shortlist is long)
            if (nk >= k_out) {
                if (nk <= 1024) {
                    if ((int)threadIdx.x < nk) {
                        const uint64_t mine = sl[threadIdx.x];
                        int r = 0;
                        for (int j = 0; j < nk; ++j) {
                            const uint64_t o = sl[j];
                            r += (o < mine || (o == mine && j < (int)threadIdx.x)) ? 1 : 0;
                        }
                        if (r == k_out - 1) s_tkey = mine;
                    }
                } else {
                    for (int j = nk + threadIdx.x; j < kpow2; j += blockDim.x) sl[j] = ~0ull;
                    __syncthreads();
                    bitonic_sort_smem(sl, kpow2);
                    if (threadIdx.x == 0) s_tkey = sl[k_out - 1];
                }
            }
            __syncthreads();
            const uint64_t tkey = s_tkey;
            // every row whose bf16 score is >= t - eps must be re-scored: bound key B (all index bits set)
            const uint64_t bound = tkey == ~0ull ? ~0ull : ((uint64_t)desc_key(key_score(tkey) - eps) << 32) | 0xffffffffull;
            const int ext_cap = sl_cap - nk;
            for (int i = threadIdx.x; i < cnt; i += blockDim.x) {
                const uint64_t key = skeys[i];
                if (key > last16 && key <= bound && key != ~0ull) {
                    const uint32_t pos = atomicAdd(&s_out, 1u);
                    if (pos < (uint32_t)ext_cap) sl[nk + pos] = key;
                }
            }
            __syncthreads();
            n_ext = min((int)s_out, ext_cap);
            // complete iff the candidate list holds every row with key <= bound: tau not tighter, nothing dropped
            if ((int)s_out > ext_cap || bound > tau_in || ovf_any) status |= 2;
            if (threadIdx.x == 0) s_hdr[2] = n_ext;
            __syncthreads();
        }
        if (CS > 1) cluster_sync_all();                                // (3) helpers may read the extension
        rescore_share<CS>(sl, 0u, false, nk, n_ext, 0, db32, n_db, idx_base, qs, D);
        if (CS > 1) cluster_sync_all();                                // (4) extension shares have landed
        __syncthreads();
        const int n_all = nk + n_ext;
        if (n_all <= 1024) {
            // rank-counting sort into the (no longer needed) candidate staging area
            if ((int)threadIdx.x < n_all) {
                const uint64_t mine = sl[threadIdx.x];
                int r = 0;
                for (int j = 0; j < n_all; ++j) {
                    const uint64_t o = sl[j];
                    r += (o < mine || (o == mine && j < (int)threadIdx.x)) ? 1 : 0;
                }
                skeys[r] = mine;
            }
            __syncthreads();
            res = skeys;
        } else {
            int n = 32;
            while (n < n_all) n <<= 1;
            for (int j = n_all + threadIdx.x; j < n; j += blockDim.x) sl[j] = ~0ull;
            __syncthreads();
            bitonic_sort_smem(sl, n);
            res = sl;
        }
        nres = n_all;
        k_emit = k_out;
    }
    if (threadIdx.x == 0 && overflow) overflow[q] = status;
    for (int j = threadIdx.x; j < k_emit; j += blockDim.x) {
        const uint64_t key = j < nres ? res[j] : ~0ull;
        const bool ok = j < nres && key != ~0ull;
        if (out_scores) out_scores[(int64_t)q * k_emit + j] = ok ? key_score(key) : -INFINITY;
        if (out_idx) out_idx[(int64_t)q * k_emit + j] = ok ? (int32_t)(uint32_t)key : -1;
        if (out_keys) out_keys[(int64_t)q * k_emit + j] = ok ? key : ~0ull;
    }
}

// One warp per (query, shortlist entry): exact fp32 dot product against the fp32 master copy.
__global__ void __launch_bounds__(256) rescore_f32_kernel(const float* __restrict__ db32, int64_t n_db, uint32_t idx_base,
                                                          const float* __restrict__ q32, int n_q, int D,
                                                          const int32_t* __restrict__ idx, int kk, uint64_t* __restrict__ out_keys) {
    const int lane = threadIdx.x & 31;
    const int64_t item = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (item >= (int64_t)n_q * kk) return;
    const int q = (int)(item / kk);
    const int32_t gi = idx[item];
    const int64_t row = (int64_t)(uint32_t)gi - (int64_t)idx_base;
    if (gi < 0 || row < 0 || row >= n_db) {
        if (lane == 0) out_keys[item] = ~0ull;
        return;
    }
    const float* a = db32 + row * D;
    const float* b = q32 + (int64_t)q * D;
    float acc = 0.f;
    if ((D & 3) == 0) {
        const float4* a4 = reinterpret_cast<const float4*>(a);
        const float4* b4 = reinterpret_cast<const float4*>(b);
        for (int i = lane; i < (D >> 2); i += 32) {
            const float4 x = a4[i], y = b4[i];
            acc = fmaf(x.x, y.x, acc); acc = fmaf(x.y, y.y, acc); acc = fmaf(x.z, y.z, acc); acc = fmaf(x.w, y.w, acc);
        }
    } else {
        for (int i = lane; i < D; i += 32) acc = fmaf(a[i], b[i], acc);
    }
    acc = warp_sum(acc);
    if (lane == 0) out_keys[item] = make_key(acc, (uint32_t)gi);
}

// fp32 -> bf16 (round-to-nearest-even) packing into the row-major (n, D) layout the scan wants.
// src_is_Dxn: src is the reference's (D, n) column-per-image matrix -> tiled transpose.
__global__ void __launch_bounds__(256) pack_bf16_rows_kernel(const float* __restrict__ src, int64_t total, __nv_bfloat16* __restrict__ dst) {
    const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i + 3 < total) {
        const float4 v = *reinterpret_cast<const float4*>(src + i);
        __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
        uint2 o;
        o.x = *reinterpret_cast<uint32_t*>(&lo);
        o.y = *reinterpret_cast<uint32_t*>(&hi);
        *reinterpret_cast<uint2*>(dst + i) = o;
    } else {
        for (int64_t j = i; j < total; ++j) dst[j] = __float2bfloat16_rn(src[j]);
    }
}

__global__ void __launch_bounds__(256) pack_bf16_transpose_kernel(const float* __restrict__ src, int64_t n, int D,
                                                                  __nv_bfloat16* __restrict__ dst) {
    __shared__ float tile[32][33];
    const int64_t n0 = (int64_t)blockIdx.x * 32;
    const int d0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 32 x 8
    for (int r = ty; r < 32; r += 8) {
        const int d = d0 + r;
        const int64_t i = n0 + tx;
        tile[r][tx] = (d < D && i < n) ? src[(int64_t)d * n + i] : 0.f;
    }
    __syncthreads();
    for (int r = ty; r < 32; r += 8) {
        const int64_t i = n0 + r;
        const int d = d0 + tx;
        if (i < n && d < D) dst[i * D + d] = __float2bfloat16_rn(tile[tx][r]);
    }
}

// alpha-QE / DBA accumulation (NOT in the reference; SURVEY.md App. E).  One CTA per query:
// acc[q, :] = sum_j max(s_j, 0)^alpha * db32[idx_j - idx_base, :] over the entries this shard owns.
__global__ void __launch_bounds__(256) qe_accumulate_kernel(const float* __restrict__ db32, int64_t n_db, uint32_t idx_base, int D,
                                                            const int32_t* __restrict__ idx, const float* __restrict__ scores,
                                                            int n_qe, float alpha, float* __restrict__ acc) {
    __shared__ float w_s[256];
    __shared__ int64_t row_s[256];
    const int q = blockIdx.x;
    for (int j = threadIdx.x; j < n_qe; j += blockDim.x) {
        const int32_t gi = idx[(int64_t)q * n_qe + j];
        const int64_t row = (int64_t)(uint32_t)gi - (int64_t)idx_base;
        const bool own = gi >= 0 && row >= 0 && row < n_db;
        row_s[j] = own ? row : -1;
        w_s[j] = own ? powf(fmaxf(scores[(int64_t)q * n_qe + j], 0.f), alpha) : 0.f;
    }
    __syncthreads();
    for (int d = threadIdx.x; d < D; d += blockDim.x) {
        float a = 0.f;
        for (int j = 0; j < n_qe; ++j)
            if (row_s[j] >= 0) a = fmaf(w_s[j], db32[row_s[j] * D + d], a);
        acc[(int64_t)q * D + d] = a;
    }
}

// out[n, :] = (a[n, :] + b[n, :]) / ||a[n, :] + b[n, :]||   (b may be NULL)
__global__ void __launch_bounds__(256) add_l2n_kernel(const float* a, const float* b, int D, float* out) {
    __shared__ float red[32];
    const int n = blockIdx.x;
    float s = 0.f;
    for (int d = threadIdx.x; d < D; d += blockDim.x) {
        const float v = a[(int64_t)n * D + d] + (b ? b[(int64_t)n * D + d] : 0.f);
        s += v * v;
    }
    s = block_sum(s, red);
    const float inv = 1.0f / sqrtf(s);
    for (int d = threadIdx.x; d < D; d += blockDim.x)
        out[(int64_t)n * D + d] = (a[(int64_t)n * D + d] + (b ? b[(int64_t)n * D + d] : 0.f)) * inv;
}

}  // namespace mdir

using namespace mdir;

extern "C" uint64_t mdir_make_key(float score, uint32_t index) { return make_key(score, index); }
extern "C" float mdir_key_score(uint64_t key) { return key_score(key); }

extern "C" int mdir_select_kth(const float* scores, int64_t ld, int64_t n, int n_q, int kth, int sample_stride,
                               uint32_t idx_base, uint64_t* tau, uint64_t* cand, int64_t cand_row, uint32_t* seg_counts, int n_seg,
                               int cap, int approx, void* stream) {
    MDIR_CHECK_ARG(scores && tau && n >= 0 && n_q >= 0 && kth >= 1 && ld >= n);
    MDIR_CHECK_ARG(cand == nullptr || (seg_counts != nullptr && cap >= 1 && n_seg >= 1 && cand_row >= cap));
    if (n_q == 0) return 0;
    if (n <= 32 * 1024) {
        select_kth_reg_kernel<<<n_q, 1024, 0, (cudaStream_t)stream>>>(scores, ld, (int)n, kth, sample_stride, idx_base, tau, cand,
                                                                      cand_row, seg_counts, n_seg, cap, approx);
        MDIR_LAUNCH_CHECK();
        return 0;
    }
    select_kth_kernel<<<n_q, 1024, 0, (cudaStream_t)stream>>>(scores, ld, n, kth, sample_stride, idx_base, tau, cand, cand_row,
                                                              seg_counts, n_seg, cap);
    MDIR_LAUNCH_CHECK();
    return 0;
}

static int launch_finalize(const uint64_t* cand, int64_t cand_row, const uint32_t* seg_counts, int n_seg, int cap0, int cap_l, int n_q,
                           int k, float* out_scores, int32_t* out_idx, uint64_t* out_keys, uint64_t* tau, int32_t* overflow,
                           const float* db32, int64_t n_db, uint32_t idx_base, const float* q32, int D, int k_out, const float* db_stats,
                           void* stream, const float* q_eps = nullptr) {
    MDIR_CHECK_ARG(cand && seg_counts && n_seg >= 1 && n_seg <= MDIR_CAND_SEGS && cap0 >= 0 && n_q >= 0 && k >= 1 && k <= 4096);
    MDIR_CHECK_ARG(n_seg == 1 || cap_l >= 1);
    MDIR_CHECK_ARG(cand_row >= (int64_t)cap0 + (int64_t)(n_seg - 1) * cap_l);
    if (n_q == 0) return 0;
    int kpow2 = 32;
    while (kpow2 < k) kpow2 <<= 1;
    // shared-memory staging capacity: everything the segments can hold, at most 16384 keys
    int64_t want = (int64_t)cap0 + (int64_t)(n_seg - 1) * cap_l;
    int smem_cap = 1024;
    while (smem_cap < want && smem_cap < 16384) smem_cap <<= 1;
    // mdir_tune: a smaller staging area (two CTAs fit on an SM); a query with more candidates raises the overflow bit
    if (g_finalize_stage_cap > 0 && smem_cap > g_finalize_stage_cap) smem_cap = g_finalize_stage_cap;
    if (smem_cap < 2 * kpow2) smem_cap = 2 * kpow2;
    // with re-scoring the selection area also takes the certified extension of the shortlist (as many keys again).  The
    // int8 route's bound reaches ~5x as many rows: ~0.09 % of a unit-norm randn shard at D = 2048 against ~0.02 % for
    // bf16, so its area grows with the shard -- room for 0.2 % of it, a power of two (the bitonic sorts), <= 2,048 keys
    int sl_cap = db32 ? 2 * kpow2 : kpow2;
    if (db32 && q_eps) {
        const int64_t want = (int64_t)kpow2 + n_db / 512;
        while (sl_cap < want && sl_cap < 2048) sl_cap <<= 1;
    }
    size_t smem = (size_t)(smem_cap + sl_cap) * 8;
    if (db32) {
        MDIR_CHECK_ARG(q32 && D > 0 && D <= 8192 && k_out >= 1 && k_out <= k && n_db >= 0);
        MDIR_CHECK_ARG((((uintptr_t)db32 | (uintptr_t)q32) & 15) == 0);
        MDIR_CHECK_ARG(db_stats == nullptr || tau != nullptr);          // the certificate compares against the filter threshold
        smem += (size_t)D * 4;
    }
    // 227 KB per CTA minus the kernel's static arrays: the deepest selection (4096-row shortlist) leaves room for D <= 7168
    constexpr int kFinalizeMaxSmem = 232448 - 7424;
    MDIR_CHECK_ARG(smem <= (size_t)kFinalizeMaxSmem);
    static PerDeviceOnce once;
    if (once.first() != 0) {
        const int max_smem = kFinalizeMaxSmem;
        MDIR_CUDA(cudaFuncSetAttribute(topk_finalize_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
        MDIR_CUDA(cudaFuncSetAttribute(topk_finalize_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
    }
    const int sm_count = device_sm_count();
    // fp32 re-scoring gathers shortlist x D x 4 bytes per query from one CTA; while the batch leaves SMs idle, a
    // 2-CTA cluster per query splits those rows (rank 1 reads / writes the shortlist through distributed shared memory)
    if (db32 && g_finalize_cluster && 2 * n_q <= sm_count) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(2 * n_q);
        cfg.blockDim = dim3(1024);
        cfg.dynamicSmemBytes = smem;
        cfg.stream = (cudaStream_t)stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = 2;
        attr[0].val.clusterDim.y = 1;
        attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        MDIR_CUDA(cudaLaunchKernelEx(&cfg, topk_finalize_kernel<2>, cand, cand_row, seg_counts, n_seg, cap0, cap_l, k, smem_cap, sl_cap, out_scores,
                                     out_idx, out_keys, tau, overflow, db32, n_db, idx_base, q32, D, k_out, db_stats, q_eps));
        MDIR_LAUNCH_CHECK();
        return 0;
    }
    topk_finalize_kernel<1><<<n_q, 1024, smem, (cudaStream_t)stream>>>(cand, cand_row, seg_counts, n_seg, cap0, cap_l, k, smem_cap, sl_cap,
                                                                        out_scores, out_idx, out_keys, tau, overflow, db32, n_db, idx_base,
                                                                        q32, D, k_out, db_stats, q_eps);
    MDIR_LAUNCH_CHECK();
    return 0;
}

extern "C" int mdir_topk_finalize(const uint64_t* cand, int64_t cand_row, const uint32_t* seg_counts, int n_seg, int cap0, int cap_l,
                                  int n_q, int k, float* out_scores, int32_t* out_idx, uint64_t* out_keys, uint64_t* tau,
                                  int32_t* overflow, void* stream) {
    return launch_finalize(cand, cand_row, seg_counts, n_seg, cap0, cap_l, n_q, k, out_scores, out_idx, out_keys, tau, overflow, nullptr, 0,
                           0, nullptr, 0, 0, nullptr, stream);
}

extern "C" int mdir_topk_finalize_rescore(const uint64_t* cand, int64_t cand_row, const uint32_t* seg_counts, int n_seg, int cap0,
                                          int cap_l, int n_q, int shortlist, int k_out, const float* db32, int64_t n_db,
                                          uint32_t idx_base, const float* q32, int D, const float* db_stats, float* out_scores,
                                          int32_t* out_idx, uint64_t* out_keys, uint64_t* tau, int32_t* overflow, void* stream) {
    MDIR_CHECK_ARG(db32 != nullptr);
    return launch_finalize(cand, cand_row, seg_counts, n_seg, cap0, cap_l, n_q, shortlist, out_scores, out_idx, out_keys, tau, overflow,
                           db32, n_db, idx_base, q32, D, k_out, db_stats, stream);
}

extern "C" int mdir_topk_finalize_rescore_eps(const uint64_t* cand, int64_t cand_row, const uint32_t* seg_counts, int n_seg, int cap0,
                                              int cap_l, int n_q, int shortlist, int k_out, const float* db32, int64_t n_db,
                                              uint32_t idx_base, const float* q32, int D, const float* db_stats, const float* q_eps,
                                              float* out_scores, int32_t* out_idx, uint64_t* out_keys, uint64_t* tau, int32_t* overflow,
                                              void* stream) {
    MDIR_CHECK_ARG(db32 != nullptr && db_stats != nullptr && q_eps != nullptr);
    return launch_finalize(cand, cand_row, seg_counts, n_seg, cap0, cap_l, n_q, shortlist, out_scores, out_idx, out_keys, tau, overflow,
                           db32, n_db, idx_base, q32, D, k_out, db_stats, stream, q_eps);
}

// db_stats for the shortlist certificate: {max_r ||bf16(x_r) - x_r||^2, max_r ||x_r||^2} over the rows of a shard.
// Non-negative floats order like their bit patterns, so the maxima are atomicMax on the uint view.
namespace mdir {
__global__ void __launch_bounds__(256) pack_stats_kernel(const float* __restrict__ db32, const __nv_bfloat16* __restrict__ db16, int64_t n, int D,
                                                         uint32_t* __restrict__ stats) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
    float e_max = 0.f, x_max = 0.f;
    for (int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < n; r += warps) {
        const float* a = db32 + r * D;
        const __nv_bfloat16* b = db16 + r * D;
        float e2 = 0.f, x2 = 0.f;
        for (int i = lane; i < D; i += 32) {
            const float x = a[i];
            const float d = __bfloat162float(b[i]) - x;
            e2 = fmaf(d, d, e2);
            x2 = fmaf(x, x, x2);
        }
        e_max = fmaxf(e_max, warp_sum(e2));
        x_max = fmaxf(x_max, warp_sum(x2));
    }
    if (lane == 0) {
        // 1 ulp-scale head room for the order of the fp32 summation above
        atomicMax(&stats[0], __float_as_uint(e_max * 1.0001f));
        atomicMax(&stats[1], __float_as_uint(x_max * 1.0001f));
    }
}
}  // namespace mdir

extern "C" int mdir_pack_stats(const float* db32, const uint16_t* db16, int64_t n, int D, float* stats, void* stream) {
    MDIR_CHECK_ARG(db32 && db16 && stats && n >= 0 && D > 0);
    MDIR_CUDA(cudaMemsetAsync(stats, 0, 2 * sizeof(float), (cudaStream_t)stream));
    if (n == 0) return 0;
    const int64_t blocks = (n + 7) / 8;
    pack_stats_kernel<<<(unsigned)(blocks < 148 * 8 ? blocks : 148 * 8), 256, 0, (cudaStream_t)stream>>>(
        db32, reinterpret_cast<const __nv_bfloat16*>(db16), n, D, reinterpret_cast<uint32_t*>(stats));
    MDIR_LAUNCH_CHECK();
    return 0;
}

// ---- int8 first pass of the certified serving scan (mdir_sim_scan_fused_i8) --------------------------------------
// Symmetric quantisation of one value: v / s rounded to nearest even, clamped to the int8 range [-127, 127].
namespace mdir {
__device__ __forceinline__ float quant_i8(float v, float s) {
    return s > 0.f ? fminf(fmaxf(rintf(__fdiv_rn(v, s)), -127.f), 127.f) : 0.f;
}

// One warp per database row: the int8 row x8_r with s_r = max_i |x_ri| / 127, and in the same pass the certificate's
// database terms stats = {max_r ||bf16(x_r) - x_r||^2, max_r ||x_r||^2, max_r ||x_r - s_r x8_r||^2,
// max_r ||x_r - s_r x8_r||^2 / ||x_r||^2} (the last one selects the route, see Index).
__global__ void __launch_bounds__(256) pack_stats_i8_kernel(const float* __restrict__ db32, const __nv_bfloat16* __restrict__ db16, int64_t n,
                                                            int D, uint32_t* __restrict__ stats, int8_t* __restrict__ db8,
                                                            float* __restrict__ row_scale) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
    float e_max = 0.f, x_max = 0.f, e8_max = 0.f, rel_max = 0.f;
    for (int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < n; r += warps) {
        const float* a = db32 + r * D;
        const __nv_bfloat16* b = db16 + r * D;
        float e2 = 0.f, x2 = 0.f, m = 0.f;
        for (int i = lane; i < D; i += 32) {
            const float x = a[i];
            const float d = __bfloat162float(b[i]) - x;
            e2 = fmaf(d, d, e2);
            x2 = fmaf(x, x, x2);
            m = fmaxf(m, fabsf(x));
        }
        e2 = warp_sum(e2);
        x2 = warp_sum(x2);
        const float s = __fdiv_rn(warp_max(m), 127.f);
        float q2 = 0.f;
        for (int i = lane * 4; i < D; i += 128) {          // D % 128 == 0: four int8 per lane and step
            const float4 x = *reinterpret_cast<const float4*>(a + i);
            const float c0 = quant_i8(x.x, s), c1 = quant_i8(x.y, s), c2 = quant_i8(x.z, s), c3 = quant_i8(x.w, s);
            char4 o;
            o.x = (signed char)c0; o.y = (signed char)c1; o.z = (signed char)c2; o.w = (signed char)c3;
            *reinterpret_cast<char4*>(db8 + r * D + i) = o;
            const float d0 = fmaf(-s, c0, x.x), d1 = fmaf(-s, c1, x.y), d2 = fmaf(-s, c2, x.z), d3 = fmaf(-s, c3, x.w);
            q2 = fmaf(d0, d0, fmaf(d1, d1, fmaf(d2, d2, fmaf(d3, d3, q2))));
        }
        q2 = warp_sum(q2);
        if (lane == 0) row_scale[r] = s;
        e_max = fmaxf(e_max, e2);
        x_max = fmaxf(x_max, x2);
        e8_max = fmaxf(e8_max, q2);
        if (x2 > 0.f) rel_max = fmaxf(rel_max, q2 / x2);
    }
    if (lane == 0) {
        // head room for the order of the fp32 summations above (the int8 residual also for its fmaf rounding)
        atomicMax(&stats[0], __float_as_uint(e_max * 1.0001f));
        atomicMax(&stats[1], __float_as_uint(x_max * 1.0001f));
        atomicMax(&stats[2], __float_as_uint(e8_max * 1.001f));
        atomicMax(&stats[3], __float_as_uint(rel_max * 1.001f));
    }
}

// One warp per query row of the int8 scan's B operand: q ~ s_hi * hi + s_lo * lo with hi = quant(q, s_hi),
// lo = quant(q - s_hi * hi, s_lo) (two int8 planes: the query's own rounding nearly vanishes from the bound), and the
// query's certificate bound for |int8-path score - fp32 score| over every row of the shard:
//     eps = e8 ||q^|| + x ||q - q^||                          (Cauchy-Schwarz on the two rounding residuals)
//         + 1.25 D 2^-24 x ||q||                               (fp32 accumulation of the exact re-score)
//         + 8 2^-24 (x + e8) (||s_hi hi|| + ||s_lo lo||)     (s32 -> fp32 conversion and the scale products of the scan)
// with e8 = max_r ||x_r - s_r x8_r||, x = max_r ||x_r|| (stats).  Rows n_q .. n_pad - 1 of the planes are zero.
__global__ void __launch_bounds__(32) pack_q_i8_kernel(const float* __restrict__ q32, int n_q, int n_pad, int D, const float* __restrict__ stats,
                                                       int8_t* __restrict__ q8, float* __restrict__ q_scale, float* __restrict__ q_eps) {
    const int q = blockIdx.x, lane = threadIdx.x;
    int8_t* hi_row = q8 + (int64_t)q * D;
    int8_t* lo_row = q8 + (int64_t)(n_pad + q) * D;
    if (q >= n_q) {
        for (int i = lane * 4; i < D; i += 128) {
            *reinterpret_cast<char4*>(hi_row + i) = make_char4(0, 0, 0, 0);
            *reinterpret_cast<char4*>(lo_row + i) = make_char4(0, 0, 0, 0);
        }
        return;
    }
    const float* v = q32 + (int64_t)q * D;
    float m = 0.f, q2 = 0.f;
    for (int i = lane; i < D; i += 32) {
        const float x = v[i];
        m = fmaxf(m, fabsf(x));
        q2 = fmaf(x, x, q2);
    }
    const float s_hi = __fdiv_rn(warp_max(m), 127.f);
    float m2 = 0.f;
    for (int i = lane; i < D; i += 32) m2 = fmaxf(m2, fabsf(fmaf(-s_hi, quant_i8(v[i], s_hi), v[i])));
    const float s_lo = __fdiv_rn(warp_max(m2), 127.f);
    float h2 = 0.f, l2 = 0.f, qh2 = 0.f, d2 = 0.f;
    for (int i = lane * 4; i < D; i += 128) {
        const float4 x = *reinterpret_cast<const float4*>(v + i);
        const float xs[4] = {x.x, x.y, x.z, x.w};
        signed char ho[4], lo[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float h = quant_i8(xs[j], s_hi);
            const float r = fmaf(-s_hi, h, xs[j]);
            const float l = quant_i8(r, s_lo);
            const float d = fmaf(-s_lo, l, r);                 // q - q^ (the residual's own rounding: within the 1.001 below)
            const float qh = fmaf(s_lo, l, s_hi * h);
            ho[j] = (signed char)h;
            lo[j] = (signed char)l;
            h2 = fmaf(h, h, h2);
            l2 = fmaf(l, l, l2);
            qh2 = fmaf(qh, qh, qh2);
            d2 = fmaf(d, d, d2);
        }
        *reinterpret_cast<char4*>(hi_row + i) = make_char4(ho[0], ho[1], ho[2], ho[3]);
        *reinterpret_cast<char4*>(lo_row + i) = make_char4(lo[0], lo[1], lo[2], lo[3]);
    }
    q2 = warp_sum(q2); h2 = warp_sum(h2); l2 = warp_sum(l2); qh2 = warp_sum(qh2); d2 = warp_sum(d2);
    if (lane == 0) {
        const float x_max = sqrtf(stats[1]), e8 = sqrtf(stats[2]);
        const float u = 5.9604645e-8f;
        float eps = e8 * sqrtf(qh2) + x_max * sqrtf(d2) + 1.25f * (float)D * u * x_max * sqrtf(q2) +
                    8.f * u * (x_max + e8) * (s_hi * sqrtf(h2) + s_lo * sqrtf(l2));
        q_scale[2 * q] = s_hi;
        q_scale[2 * q + 1] = s_lo;
        q_eps[q] = eps * 1.001f + 1e-7f;                       // slack for evaluating the bound itself in fp32
    }
}
}  // namespace mdir

extern "C" int mdir_pack_stats_i8(const float* db32, const uint16_t* db16, int64_t n, int D, float* stats, int8_t* db8, float* row_scale,
                                  void* stream) {
    MDIR_CHECK_ARG(db32 && db16 && stats && db8 && row_scale && n >= 0 && D > 0 && D % 128 == 0);
    MDIR_CHECK_ARG((((uintptr_t)db32 | (uintptr_t)db8) & 15) == 0);
    MDIR_CUDA(cudaMemsetAsync(stats, 0, 4 * sizeof(float), (cudaStream_t)stream));
    if (n == 0) return 0;
    const int64_t blocks = (n + 7) / 8;
    pack_stats_i8_kernel<<<(unsigned)(blocks < 148 * 8 ? blocks : 148 * 8), 256, 0, (cudaStream_t)stream>>>(
        db32, reinterpret_cast<const __nv_bfloat16*>(db16), n, D, reinterpret_cast<uint32_t*>(stats), db8, row_scale);
    MDIR_LAUNCH_CHECK();
    return 0;
}

extern "C" int mdir_pack_q_i8(const float* q32, int n_q, int D, const float* stats, int8_t* q8, float* q_scale, float* q_eps, void* stream) {
    MDIR_CHECK_ARG(q32 && stats && q8 && q_scale && q_eps && n_q >= 1 && n_q <= 128 && D > 0 && D % 128 == 0);
    MDIR_CHECK_ARG((((uintptr_t)q32 | (uintptr_t)q8) & 15) == 0);
    const int n_pad = (n_q + 15) & ~15;
    pack_q_i8_kernel<<<n_pad, 32, 0, (cudaStream_t)stream>>>(q32, n_q, n_pad, D, stats, q8, q_scale, q_eps);
    MDIR_LAUNCH_CHECK();
    return 0;
}

extern "C" int mdir_rescore_f32(const float* db32, int64_t n_db, uint32_t idx_base, const float* q32, int n_q, int D,
                                const int32_t* idx, int kk, uint64_t* out_keys, void* stream) {
    MDIR_CHECK_ARG(db32 && q32 && idx && out_keys && n_db >= 0 && n_q >= 0 && D > 0 && kk >= 1);
    MDIR_CHECK_ARG((((uintptr_t)db32 | (uintptr_t)q32) & 15) == 0);
    const int64_t items = (int64_t)n_q * kk;
    if (items == 0) return 0;
    rescore_f32_kernel<<<(unsigned)((items + 7) / 8), 256, 0, (cudaStream_t)stream>>>(db32, n_db, idx_base, q32, n_q, D, idx, kk,
                                                                                      out_keys);
    MDIR_LAUNCH_CHECK();
    return 0;
}

extern "C" int mdir_pack_bf16(const float* src, int64_t n, int D, int src_is_Dxn, uint16_t* dst, void* stream) {
    MDIR_CHECK_ARG(src && dst && n >= 0 && D > 0);
    if (n == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    if (!src_is_Dxn) {
        MDIR_CHECK_ARG((((uintptr_t)src & 15) | ((uintptr_t)dst & 7)) == 0);
        const int64_t total = n * D;
        const int64_t threads = (total + 3) / 4;
        pack_bf16_rows_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(src, total, (__nv_bfloat16*)dst);
    } else {
        dim3 grid((unsigned)((n + 31) / 32), (unsigned)((D + 31) / 32));
        MDIR_CHECK_ARG(grid.y <= 65535);
        pack_bf16_transpose_kernel<<<grid, 256, 0, st>>>(src, n, D, (__nv_bfloat16*)dst);
    }
    MDIR_LAUNCH_CHECK();
    return 0;
}

extern "C" int mdir_qe_accumulate(const float* db32, int64_t n_db, uint32_t idx_base, int D, const int32_t* idx, const float* scores,
                                  int n_q, int n_qe, float alpha, float* acc, void* stream) {
    MDIR_CHECK_ARG(db32 && idx && scores && acc && n_db >= 0 && D > 0 && n_q >= 0 && n_qe >= 1 && n_qe <= 256);
    if (n_q == 0) return 0;
    qe_accumulate_kernel<<<n_q, 256, 0, (cudaStream_t)stream>>>(db32, n_db, idx_base, D, idx, scores, n_qe, alpha, acc);
    MDIR_LAUNCH_CHECK();
    return 0;
}

extern "C" int mdir_add_l2n(const float* a, const float* b, int n, int D, float* out, void* stream) {
    MDIR_CHECK_ARG(a && out && n >= 0 && D > 0);
    if (n == 0) return 0;
    add_l2n_kernel<<<n, 256, 0, (cudaStream_t)stream>>>(a, b, D, out);
    MDIR_LAUNCH_CHECK();
    return 0;
}
