// In-place compaction of a mutable index (Index.compact): the live rows of the used slots move, in order, to slots
// [0, n_live) of every plane (bf16 rows, fp32 master, int8 rows, row scales, slot -> id map), the freed slots are
// zero-filled and the live bitmap and the device-side scan extent describe the result.
//
// The destination of live slot s is the number of live slots before it: an exclusive prefix popcount over the bitmap
// words (mdir_compact_prefix) plus the popcount of the lower bits of its own word.  dest(s) <= s, so a parallel gather
// over all slots at once would read rows another CTA has already overwritten.  The host sweeps chunks [lo, hi) of slots
// in ascending order (search.compaction_schedule); the live rows of a chunk go to [dst0, dst0 + n_dst), which ends at
// or below hi, so a chunk only overwrites rows already read.  A chunk whose destinations end at or below lo
// (dst0 + n_dst <= lo) moves directly in one launch, its reads and writes disjoint; any other chunk is staged: one
// launch gathers its live rows into scratch, the next writes them to their destinations.  Scratch is one chunk.
#include <cuda_bf16.h>

#include "common.cuh"

namespace mdir {

struct CompactPlanes {
    uint8_t* p[5];           // db16, db32, db8, row_scale, slot_id (NULL: the plane does not exist)
    int64_t row_bytes[5];
};

__device__ __forceinline__ void copy_row_bytes(uint8_t* __restrict__ dst, const uint8_t* __restrict__ src, int64_t bytes) {
    if ((bytes & 15) == 0) {
        const uint4* s = reinterpret_cast<const uint4*>(src);
        uint4* d = reinterpret_cast<uint4*>(dst);
        for (int64_t i = threadIdx.x; i < (bytes >> 4); i += blockDim.x) d[i] = s[i];
    } else {
        for (int64_t i = threadIdx.x; i < bytes; i += blockDim.x) dst[i] = src[i];
    }
}

// prefix[w] = live slots in words [0, w), prefix[n_words] = all of them.  One CTA: each thread sums a contiguous run of
// words, an exclusive scan over the threads, then each thread writes the prefixes of its run.
__global__ void __launch_bounds__(1024) compact_prefix_kernel(const uint32_t* __restrict__ live, int64_t n_words, int64_t* __restrict__ prefix) {
    __shared__ int64_t part[1024];
    const int t = threadIdx.x;
    const int64_t per = (n_words + 1023) / 1024;
    const int64_t w0 = (int64_t)t * per, w1 = min(n_words, w0 + per);
    int64_t sum = 0;
    for (int64_t w = w0; w < w1; ++w) sum += __popc(live[w]);
    part[t] = sum;
    __syncthreads();
    for (int off = 1; off < 1024; off <<= 1) {        // inclusive Hillis-Steele scan
        const int64_t v = t >= off ? part[t - off] : 0;
        __syncthreads();
        part[t] += v;
        __syncthreads();
    }
    int64_t run = part[t] - sum;
    for (int64_t w = w0; w < w1; ++w) {
        prefix[w] = run;
        run += __popc(live[w]);
    }
    if (t == 1023) prefix[n_words] = part[1023];
}

// MODE 0 (direct): live slot s of [lo, hi) -> slot dest(s).  MODE 1 (gather): -> scratch row dest(s) - dst0.
// MODE 2 (scatter): scratch row i -> slot dst0 + i.  One CTA per slot (modes 0, 1) or per scratch row (mode 2).
template <int MODE>
__global__ void __launch_bounds__(128) compact_move_kernel(CompactPlanes pl, CompactPlanes scr, const uint32_t* __restrict__ live,
                                                           const int64_t* __restrict__ prefix, int64_t lo, int64_t dst0) {
    int64_t src, dst;
    if (MODE == 2) {
        src = blockIdx.x;
        dst = dst0 + blockIdx.x;
    } else {
        const int64_t s = lo + blockIdx.x;
        const uint32_t w = live[s >> 5];
        const uint32_t bit = (uint32_t)(s & 31);
        if (!((w >> bit) & 1u)) return;
        const int64_t dest = prefix[s >> 5] + __popc(w & ((1u << bit) - 1u));
        src = s;
        dst = MODE == 0 ? dest : dest - dst0;
    }
#pragma unroll
    for (int k = 0; k < 5; ++k) {
        if (!pl.p[k]) continue;
        const int64_t rb = pl.row_bytes[k];
        const uint8_t* from = (MODE == 2 ? scr.p[k] : pl.p[k]) + src * rb;
        uint8_t* to = (MODE == 1 ? scr.p[k] : pl.p[k]) + dst * rb;
        copy_row_bytes(to, from, rb);
    }
}

// The bitmap after compaction: ones on [0, n_live), zeros after; and the scan extent.
__global__ void __launch_bounds__(256) compact_finish_kernel(uint32_t* __restrict__ live, int64_t n_words, int64_t n_live,
                                                             int64_t* __restrict__ n_scan) {
    const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (w == 0 && n_scan) *n_scan = n_live;
    if (w >= n_words) return;
    const int64_t r0 = w * 32;
    live[w] = r0 + 32 <= n_live ? 0xffffffffu : (r0 >= n_live ? 0u : (1u << (uint32_t)(n_live - r0)) - 1u);
}

static CompactPlanes make_planes(uint16_t* db16, float* db32, int8_t* db8, float* row_scale, uint32_t* slot_id, int D) {
    CompactPlanes pl;
    pl.p[0] = reinterpret_cast<uint8_t*>(db16);
    pl.p[1] = reinterpret_cast<uint8_t*>(db32);
    pl.p[2] = reinterpret_cast<uint8_t*>(db8);
    pl.p[3] = reinterpret_cast<uint8_t*>(row_scale);
    pl.p[4] = reinterpret_cast<uint8_t*>(slot_id);
    pl.row_bytes[0] = (int64_t)D * 2;
    pl.row_bytes[1] = (int64_t)D * 4;
    pl.row_bytes[2] = (int64_t)D;
    pl.row_bytes[3] = 4;
    pl.row_bytes[4] = 4;
    return pl;
}

// Scratch for `rows` rows of the planes that exist, one 256-byte aligned section per plane.  scr == NULL: size only.
static size_t scratch_layout(const CompactPlanes& pl, int64_t rows, uint8_t* base, CompactPlanes* scr) {
    size_t off = 0;
    for (int k = 0; k < 5; ++k) {
        if (scr) {
            scr->p[k] = pl.p[k] ? base + off : nullptr;
            scr->row_bytes[k] = pl.row_bytes[k];
        }
        if (pl.p[k]) off += ((size_t)(rows * pl.row_bytes[k]) + 255) & ~(size_t)255;
    }
    return off;
}

}  // namespace mdir

using namespace mdir;

extern "C" size_t mdir_compact_scratch_bytes(int64_t rows, int D, int has_fp32, int has_i8) {
    if (rows < 0 || D <= 0) return 0;
    uint16_t one16;
    float one32;
    int8_t one8;
    uint32_t id;
    const CompactPlanes pl = make_planes(&one16, has_fp32 ? &one32 : nullptr, has_i8 ? &one8 : nullptr, has_i8 ? &one32 : nullptr, &id, D);
    return scratch_layout(pl, rows, nullptr, nullptr);
}

extern "C" int mdir_compact_prefix(const uint32_t* live, int64_t n_words, int64_t* word_prefix, void* stream) {
    MDIR_CHECK_ARG(live && word_prefix && n_words >= 0);
    compact_prefix_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(live, n_words, word_prefix);
    MDIR_LAUNCH_CHECK();
    return 0;
}

extern "C" int mdir_compact_move(uint16_t* db16, float* db32, int8_t* db8, float* row_scale, uint32_t* slot_id, int64_t capacity, int D,
                                 const uint32_t* live, const int64_t* word_prefix, int64_t lo, int64_t hi, int64_t dst0, int64_t n_dst,
                                 void* scratch, size_t scratch_bytes, void* stream) {
    MDIR_CHECK_ARG(db16 && slot_id && live && word_prefix && D > 0 && D % 8 == 0 && (!db8 || (row_scale && D % 16 == 0)));
    MDIR_CHECK_ARG(0 <= lo && lo <= hi && hi <= capacity && hi - lo <= 0x7fffffff);
    MDIR_CHECK_ARG(dst0 >= 0 && n_dst >= 0 && n_dst <= hi - lo && dst0 + n_dst <= hi);     // destinations never pass the chunk
    if (n_dst == 0) return 0;
    const CompactPlanes pl = make_planes(db16, db32, db8, row_scale, slot_id, D);
    CompactPlanes scr = pl;
    cudaStream_t st = (cudaStream_t)stream;
    if (!scratch) {
        MDIR_CHECK_ARG(dst0 + n_dst <= lo);            // direct: the destinations lie below every row this chunk reads
        compact_move_kernel<0><<<(unsigned)(hi - lo), 128, 0, st>>>(pl, scr, live, word_prefix, lo, dst0);
        MDIR_LAUNCH_CHECK();
        return 0;
    }
    MDIR_CHECK_ARG(scratch_layout(pl, n_dst, static_cast<uint8_t*>(scratch), &scr) <= scratch_bytes);
    compact_move_kernel<1><<<(unsigned)(hi - lo), 128, 0, st>>>(pl, scr, live, word_prefix, lo, dst0);
    MDIR_LAUNCH_CHECK();
    compact_move_kernel<2><<<(unsigned)n_dst, 128, 0, st>>>(pl, scr, live, word_prefix, lo, dst0);
    MDIR_LAUNCH_CHECK();
    return 0;
}

extern "C" int mdir_compact_finish(uint16_t* db16, float* db32, int8_t* db8, float* row_scale, uint32_t* slot_id, int D, uint32_t* live,
                                   int64_t n_words, int64_t n_live, int64_t n_used, int64_t* n_scan, void* stream) {
    MDIR_CHECK_ARG(db16 && slot_id && live && D > 0 && 0 <= n_live && n_live <= n_used && n_used <= n_words * 32);
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t n_free = n_used - n_live;
    if (n_free > 0) {
        MDIR_CUDA(cudaMemsetAsync(db16 + n_live * D, 0, (size_t)(n_free * D) * 2, st));
        if (db32) MDIR_CUDA(cudaMemsetAsync(db32 + n_live * D, 0, (size_t)(n_free * D) * 4, st));
        if (db8) MDIR_CUDA(cudaMemsetAsync(db8 + n_live * D, 0, (size_t)(n_free * D), st));
        if (row_scale) MDIR_CUDA(cudaMemsetAsync(row_scale + n_live, 0, (size_t)n_free * 4, st));
        MDIR_CUDA(cudaMemsetAsync(slot_id + n_live, 0xff, (size_t)n_free * 4, st));      // no id
    }
    compact_finish_kernel<<<(unsigned)((n_words + 255) / 256 + (n_words == 0)), 256, 0, st>>>(live, n_words, n_live, n_scan);
    MDIR_LAUNCH_CHECK();
    return 0;
}
