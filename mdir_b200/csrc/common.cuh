// Shared helpers for libmdir_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>

#include "../../include/mdir_b200.h"

namespace mdir {

void set_error(const std::string& s);
int fail_arg(const char* what);

#define MDIR_CHECK_ARG(cond)                                              \
    do {                                                                  \
        if (!(cond)) return ::mdir::fail_arg(#cond);                      \
    } while (0)

#define MDIR_CUDA(expr)                                                   \
    do {                                                                  \
        cudaError_t _e = (expr);                                          \
        if (_e != cudaSuccess) {                                          \
            ::mdir::set_error(std::string(#expr) + ": " + cudaGetErrorString(_e)); \
            return (int)_e;                                               \
        }                                                                 \
    } while (0)

extern unsigned long long g_launches;   // kernels launched by this library (bench.py's gpu_launches)
// SM-partitioning knobs (mdir_tune): a serving pipeline that runs finalize + exchange of step t beside the scan of step
// t + 1 caps the scan's persistent grid and keeps finalize off thread-block clusters, so that both fit at once
extern int g_scan_max_ctas;            // 0 = no cap
extern int g_finalize_cluster;         // 1 = 2-CTA clusters when SMs are idle (default)
extern int g_finalize_stage_cap;       // 0 = stage everything the segments can hold (<= 16384 keys); else at most this many

#define MDIR_LAUNCH_CHECK()                                               \
    do {                                                                  \
        ++::mdir::g_launches;                                             \
        cudaError_t _e = cudaGetLastError();                              \
        if (_e != cudaSuccess) {                                          \
            ::mdir::set_error(std::string("kernel launch: ") + cudaGetErrorString(_e)); \
            return (int)_e;                                               \
        }                                                                 \
    } while (0)

constexpr int kNumSMs = 148;

// Per-device "already done" flag: cudaFuncSetAttribute and the SM count are per DEVICE, so a
// process that drives cuda:0 and then cuda:1 must repeat them (a process-wide static would skip the second device).
constexpr int kMaxDevices = 64;
struct PerDeviceOnce {
    bool done[kMaxDevices] = {};
    // true exactly once per device ordinal (the current device); -1 on a CUDA error
    int first() {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) return -1;
        if (done[dev]) return 0;
        done[dev] = true;
        return 1;
    }
};
// Persistent-grid size for n_work equal work items on at most max_ctas SMs: the smallest grid that needs the same
// number of rounds as max_ctas would (489 tiles on 148 SMs are 4 rounds either way; 123 CTAs x 4 rounds keep every
// CTA busy to the end, where 148 CTAs leave 103 SMs idle during a last round that then runs at a third of the HBM rate).
inline int balanced_grid(int64_t n_work, int max_ctas) {
    if (n_work <= 0 || max_ctas <= 0) return 1;
    if (n_work <= max_ctas) return (int)n_work;
    const int64_t rounds = (n_work + max_ctas - 1) / max_ctas;
    return (int)((n_work + rounds - 1) / rounds);
}

// SM count of the current device (cached per ordinal); 0 on error
inline int device_sm_count() {
    static int cache[kMaxDevices] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) return 0;
    if (!cache[dev]) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return 0;
        cache[dev] = n;
    }
    return cache[dev];
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ int warp_sum_int(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Block-wide sum for blockDim.x <= 1024 (multiple of 32); red must hold 32 floats.
__device__ __forceinline__ float block_sum(float v, float* red) {
    v = warp_sum(v);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    __syncthreads();
    if (lane == 0) red[w] = v;
    __syncthreads();
    float r = (lane < nw) ? red[lane] : 0.f;
    r = warp_sum(r);
    return r;   // every warp holds the total
}

// Lanes of the warp whose 8-bit digit equals this lane's, among the lanes with valid == true
// (9 ballots + logic).  MATCH.ANY computes the same thing but is an order of magnitude slower on this
// part when the warp holds many distinct values, which is the common case for radix digits.
__device__ __forceinline__ unsigned match_digit8(int d, bool valid) {
    unsigned peers = __ballot_sync(0xffffffffu, valid);
#pragma unroll
    for (int b = 0; b < 8; ++b) {
        const bool bit = (d >> b) & 1;
        const unsigned bal = __ballot_sync(0xffffffffu, bit);
        peers &= bit ? bal : ~bal;
    }
    return peers;
}

// One-warp helper: given hist[256] and the remaining rank k (1-based), find the bin where the
// running count reaches k.  Returns the bin; *before = items in earlier bins.
__device__ __forceinline__ int find_bin_warp0(const uint32_t* hist, uint32_t k, uint32_t* before) {
    const int lane = threadIdx.x & 31;
    uint32_t loc[8], sum = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) { loc[j] = hist[lane * 8 + j]; sum += loc[j]; }
    uint32_t incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    const uint32_t excl = incl - sum;
    const unsigned hit = __ballot_sync(0xffffffffu, incl >= k);
    const int src = hit ? (__ffs(hit) - 1) : 31;
    int bin = 0;
    uint32_t acc = excl;
    if (lane == src) {
        int j = 0;
        for (; j < 7; ++j) {
            if (acc + loc[j] >= k) break;
            acc += loc[j];
        }
        bin = lane * 8 + j;
    }
    bin = __shfl_sync(0xffffffffu, bin, src);
    acc = __shfl_sync(0xffffffffu, acc, src);
    *before = acc;
    return bin;
}

// fp32 dot product of one database row with a query (in shared or global memory), one warp per row.  The summation
// order is that of each row of rescore_row2 (topk.cu), so a row's fp32 score does not depend on whether it was
// re-scored alone or as one of a pair: every finalize path, range_gather_kernel and the diffusion graph update give the
// same bits for the same row.
__device__ __forceinline__ float rescore_row(const float* __restrict__ a, const float* qs, int D, int lane) {
    float acc = 0.f;
    if ((D & 3) == 0) {
        const float4* a4 = reinterpret_cast<const float4*>(a);
        const float4* b4 = reinterpret_cast<const float4*>(qs);
        const int n4 = D >> 2;
        float sa = 0.f, sb = 0.f;
        int i = lane;
        for (; i + 96 < n4; i += 128) {            // 4 independent 128-bit loads in flight per lane
            const float4 x0 = __ldg(a4 + i), x1 = __ldg(a4 + i + 32), x2 = __ldg(a4 + i + 64), x3 = __ldg(a4 + i + 96);
            const float4 y0 = b4[i], y1 = b4[i + 32], y2 = b4[i + 64], y3 = b4[i + 96];
            sa = fmaf(x0.x, y0.x, sa); sa = fmaf(x0.y, y0.y, sa); sa = fmaf(x0.z, y0.z, sa); sa = fmaf(x0.w, y0.w, sa);
            sb = fmaf(x1.x, y1.x, sb); sb = fmaf(x1.y, y1.y, sb); sb = fmaf(x1.z, y1.z, sb); sb = fmaf(x1.w, y1.w, sb);
            sa = fmaf(x2.x, y2.x, sa); sa = fmaf(x2.y, y2.y, sa); sa = fmaf(x2.z, y2.z, sa); sa = fmaf(x2.w, y2.w, sa);
            sb = fmaf(x3.x, y3.x, sb); sb = fmaf(x3.y, y3.y, sb); sb = fmaf(x3.z, y3.z, sb); sb = fmaf(x3.w, y3.w, sb);
        }
        for (; i < n4; i += 32) {
            const float4 x = __ldg(a4 + i), y = b4[i];
            sa = fmaf(x.x, y.x, sa); sa = fmaf(x.y, y.y, sa); sa = fmaf(x.z, y.z, sa); sa = fmaf(x.w, y.w, sa);
        }
        acc = sa + sb;
    } else {
        for (int i = lane; i < D; i += 32) acc = fmaf(a[i], qs[i], acc);
    }
    return warp_sum(acc);
}

// The certified bound on |bf16-path score - fp32 score| of any database row against a query q (topk_finalize_kernel
// derives it): q2 = ||q||^2, qt2 = ||bf16(q)||^2, qf2 = ||q - bf16(q)||^2, db_stats = {max_r ||bf16(x_r) - x_r||^2,
// max_r ||x_r||^2} (mdir_pack_stats).  The bound is symmetric in the two rows when db_stats covers q's row as well.
__device__ __forceinline__ float bf16_eps(const float* __restrict__ db_stats, float q2, float qt2, float qf2, int D) {
    const float e_max = sqrtf(db_stats[0]), x_max = sqrtf(db_stats[1]);
    float eps = e_max * sqrtf(qt2) + x_max * sqrtf(qf2) + 1.25f * (float)D * 5.9604645e-8f * x_max * sqrtf(q2);
    eps = eps * 1.001f + 1e-7f;                              // slack for evaluating the bound itself in fp32
    return eps;
}

__device__ __forceinline__ void bitonic_sort_smem(uint64_t* a, int n) {
    for (int kk = 2; kk <= n; kk <<= 1) {
        for (int j = kk >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < n; i += blockDim.x) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const uint64_t x = a[i], y = a[ixj];
                    const bool asc = (i & kk) == 0;
                    if ((x > y) == asc) { a[i] = y; a[ixj] = x; }
                }
            }
            __syncthreads();
        }
    }
}

// ---- 64-bit candidate keys: smaller key == better (score desc, index asc) --------
__host__ __device__ __forceinline__ uint32_t f32_bits(float f) {
#ifdef __CUDA_ARCH__
    return __float_as_uint(f);
#else
    union { float f; uint32_t u; } c; c.f = f; return c.u;
#endif
}
__host__ __device__ __forceinline__ float bits_f32(uint32_t u) {
#ifdef __CUDA_ARCH__
    return __uint_as_float(u);
#else
    union { float f; uint32_t u; } c; c.u = u; return c.f;
#endif
}
// ascending-orderable transform of an fp32, with -0 canonicalised to +0 so that
// +-0 tie exactly as they do under numpy's comparison sort.
__host__ __device__ __forceinline__ uint32_t orderable(float f) {
    uint32_t u = f32_bits(f);
    if ((u << 1) == 0u) u = 0u;
    return u ^ ((u >> 31) ? 0xffffffffu : 0x80000000u);
}
// descending-score key: smaller == better.  NaN scores (the reference produces NaN rows for missing
// images) rank last, in index order, exactly as np.argsort(-scores) places them.
__host__ __device__ __forceinline__ uint32_t desc_key(float score) {
    return (score != score) ? 0xffffffffu : ~orderable(score);
}
__host__ __device__ __forceinline__ uint64_t make_key(float score, uint32_t idx) {
    return ((uint64_t)desc_key(score) << 32) | (uint64_t)idx;
}
__host__ __device__ __forceinline__ float key_score(uint64_t key) {
    uint32_t o = ~(uint32_t)(key >> 32);
    uint32_t u = o ^ ((o >> 31) ? 0x80000000u : 0xffffffffu);
    return bits_f32(u);
}

}  // namespace mdir
