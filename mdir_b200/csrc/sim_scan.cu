// Query x database similarity as a dense contraction on tcgen05 / TMEM tiles fed by TMA.
// Replaces np.dot(vecs.T, qvecs) (mdir/components/optim/score/cirscore.py:69) and fuses the
// selection half of np.argsort (cirscore.py:70) into the epilogue so that the n_db-wide
// score rows never land in HBM in FILTER mode.
//
// One persistent CTA per SM, 192 threads, warp-specialised:
//   warp 0      TMA producer: per k-block one 256x64 bf16 box of the database (A operand,
//               32 KB, SWIZZLE_128B) + one N x 64 box of the queries (B operand, L2-resident)
//   warp 1      TMEM allocator + single-thread tcgen05.mma issuer: two M=128 accumulators
//               (db rows 0-127 / 128-255 of the tile) x N query columns, fp32, double-buffered
//               in TMEM (4 x 128 columns = all 512)
//   warps 2-5   epilogue: tcgen05.ld 32x32b (lane = db row, column = query); DENSE/SAMPLE
//               modes store scores query-major (coalesced: 32 lanes = 32 consecutive rows),
//               FILTER mode compares against the per-query threshold key and appends the rare
//               survivors (expected k*n_tiles/n_sample per query) to the candidate lists.
// Orientation: database rows sit on the UMMA M axis so that no MMA rows are wasted on the
// 70 -> 80 padded queries (SURVEY.md section 7, hard part 1).
#include <cuda.h>

#include "common.cuh"

namespace mdir {

constexpr int kBlockM = MDIR_SCAN_TILE_ROWS;   // 256 db rows per tile = two UMMA M=128 halves
constexpr int kBlockKBytes = 128;               // one 128-byte swizzle row per operand row and k-block:
                                                //   64 bf16 (UMMA_K = 16) or 32 fp32/tf32 (UMMA_K = 8): 4 MMAs of 32 bytes either way
constexpr int kKSteps = 4;
constexpr int kABytes = kBlockM * kBlockKBytes;  // 32768
constexpr int kMaxN = 256;               // queries resident per pass (UMMA N); the in-kernel threshold exchange handles <= 128
constexpr int kMaxStages = 8;
constexpr int kThreads = 192;
constexpr uint32_t kTmemCols = 512;
constexpr int kChainKBlocks = 4;        // k-blocks (16 MMAs) per chained accumulation chunk of the tf32 DENSE scan
constexpr int kMaxWideQ = 1024;          // queries of one wide FILTER / SAMPLE launch (their filter state lives in shared memory)
constexpr int kChainMaxN = 96;          // queries per launch of the chained scan (96 KB of running sums + 2 operand stages)
constexpr int kMaxAccBufs = 3;          // accumulator tiles resident in TMEM (2 halves x acc_stride columns each)

constexpr uint64_t kEvictNormal = 0x1000000000000000ull;
constexpr uint64_t kEvictFirst = 0x12F0000000000000ull;
constexpr uint64_t kEvictLast = 0x14F0000000000000ull;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra LAB_DONE;\n"
        "bra LAB_WAIT;\n"
        "LAB_DONE:\n"
        "}\n" ::"r"(bar), "r"(parity)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int x, int y, uint64_t hint) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(dst), "l"(map), "r"(bar), "r"(x), "r"(y), "l"(hint)
        : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// operand kinds of sim_scan_kernel: bf16 x bf16 and tf32 x tf32 (fp32 accumulators), s8 x s8 (s32 accumulators)
constexpr int kKindBf16 = 0, kKindTf32 = 1, kKindI8 = 2;

template <int KIND>
__device__ __forceinline__ void umma_ss(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    if (KIND == kKindI8) {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "setp.ne.b32 p, %4, 0;\n"
            "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n"
            "}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
            : "memory");
    } else if (KIND == kKindTf32) {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "setp.ne.b32 p, %4, 0;\n"
            "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
            "}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
            : "memory");
    } else {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "setp.ne.b32 p, %4, 0;\n"
            "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
            "}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
            : "memory");
    }
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor layout):
// start>>4 [0,14) | LBO>>4 = 1 [16,30) | SBO>>4 = 64 (8 rows x 128 B) [32,46) | version 1 [46,48) | layout 2 [61,64)
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t saddr) {
    return (uint64_t)((saddr >> 4) & 0x3fffu) | ((uint64_t)1 << 16) | ((uint64_t)64 << 32) | ((uint64_t)1 << 46) |
           ((uint64_t)2 << 61);
}

struct ScanParams {
    int64_t n_db;
    int n_q, n_pad, num_k_blocks, n_tiles;
    int mode, sample_stride, n_sample, n_work, num_stages;
    float* dense_out;
    int64_t dense_ld;
    const uint64_t* tau;
    uint32_t idx_base;
    uint64_t* cand;          // (n_q, cap_s + 148 * cap_l): segment 0 = select kernel, segment 1 + cta = this CTA
    uint32_t* seg_counts;    // (n_q, MDIR_CAND_SEGS)
    int cap_s, cap_l;
    uint64_t db_hint;
    // DENSE mode only: the k-blocks are split over k_split CTAs per tile; split ks writes its partial sums to
    // dense_out + ks * split_stride (the caller adds the k_split partial planes in a fixed order)
    int k_split, kb_per_split;
    int64_t split_stride;
    // DENSE mode only: CHAINED accumulation.  The tensor core's fp32 accumulator truncates once per MMA, so a long K
    // loop drifts by up to (number of MMAs) x ulp(|score|) (~4.6e-5 relative at 3 x 2048 tf32 elements).  With
    // chain > 1 the K loop of a tile is cut into `chain` chunks of kb_per_chain k-blocks that the SAME CTA runs back
    // to back; the epilogue of a chunk adds its TMEM partial to a running sum the CTA keeps in SHARED memory behind the
    // operand ring (256 rows x n_pad fp32, one rounded fp32 add per chunk; each thread owns its own entries, so no
    // barrier), and the last chunk's epilogue writes sum + partial to dense_out.  Drift: (MMAs per chunk) x ulp.
    int chain, kb_per_chain;
    // DENSE mode only: more than one block of n_pad queries in ONE launch (work item = (tile, query block), the blocks
    // of a tile adjacent in the round-robin so that its database rows are read from HBM once): n_q_total queries in all
    int n_qblocks, n_q_total;
    // FUSED mode only (threshold + filter in one launch): every CTA's first tile is a sample tile; the best two keys
    // of each 32-row group go to grp_top (n_q, grid, 8, 2); CTA q selects the kth smallest of query q's grid*16
    // values as the threshold, published through tau_rw; sync = {arrivals 1, arrivals 2, unused, exits}
    int acc_bufs, acc_stride;     // TMEM: acc_bufs accumulator tiles of 2 x acc_stride columns (3 x 2 x 80 when N <= 80, else 2 x 2 x 128);
                                  // int8: acc_bufs accumulators of ONE 128-row half each (see sim_scan_kernel)
    int kth;
    uint32_t* grp_top;
    uint32_t* sync;
    uint64_t* tau_rw;
    // int8 only: score(row r, query q) = s_r * (s_hi[q] * acc_hi + s_lo[q] * acc_lo), the query as two int8 planes
    // (rows [0, n_pad) = hi, [n_pad, 2 n_pad) = lo of the B operand)
    const float* row_scale;      // s_r, n_db entries
    const float* q_scale;        // {s_hi, s_lo} per query
    // live-row bitmap (NULL: every row < n_db is live): bit r & 31 of word r >> 5 set = row r is live.  A dead row
    // is scored like a row past the end: never a candidate, -inf in the SAMPLE / DENSE outputs, no pass-A key.
    const uint32_t* live;
};

constexpr int MDIR_SCAN_FUSED = 3;      // internal mode behind mdir_sim_scan_fused_bf16

struct WorkItem {
    int tile, ks, kb0, nkb, j, chunk, last, qb;
};

__device__ __forceinline__ int tile_of_work(const ScanParams& p, int j);

__device__ __forceinline__ WorkItem decode_work(const ScanParams& p, int j) {
    WorkItem w;
    w.qb = 0;
    if (p.mode == MDIR_SCAN_DENSE && p.k_split > 1) {
        w.tile = j / p.k_split;
        w.ks = j - w.tile * p.k_split;
        w.kb0 = w.ks * p.kb_per_split;
        w.nkb = min(p.kb_per_split, p.num_k_blocks - w.kb0);
    } else if (p.n_qblocks > 1) {
        // wide launch: work item = (tile-level item, query block), the blocks of a tile adjacent in the round-robin
        const int jt = j / p.n_qblocks;
        w.qb = j - jt * p.n_qblocks;
        w.tile = tile_of_work(p, jt);
        w.ks = 0;
        w.kb0 = 0;
        w.nkb = p.num_k_blocks;
        w.j = jt;
        w.chunk = 0;
        w.last = 1;
        return w;
    } else {
        w.tile = tile_of_work(p, j);
        w.ks = 0;
        w.kb0 = 0;
        w.nkb = p.num_k_blocks;
    }
    w.j = j;
    w.chunk = 0;
    w.last = 1;
    return w;
}

// The it-th work item of this CTA (persistent round-robin); false when the CTA is done.  In FUSED mode item 0 is
// the CTA's own sample tile and the rest walk the non-sample tiles exactly like FILTER mode.
__device__ __forceinline__ bool next_item(const ScanParams& p, int it, WorkItem& w) {
    if (p.chain > 1) {                    // DENSE, chained chunks: chunk c of the CTA's (it / chain)-th tile
        const int t = it / p.chain, c = it - t * p.chain;
        const int tile = (int)blockIdx.x + t * (int)gridDim.x;
        if (tile >= p.n_tiles) return false;
        w.tile = tile;
        w.ks = 0;
        w.qb = 0;
        w.kb0 = c * p.kb_per_chain;
        w.nkb = min(p.kb_per_chain, p.num_k_blocks - w.kb0);
        w.j = tile;
        w.chunk = c;
        w.last = c == p.chain - 1 ? 1 : 0;
        return true;
    }
    int j = (int)blockIdx.x + it * (int)gridDim.x;
    if (p.mode == MDIR_SCAN_FUSED) {
        if (it == 0) {
            w.tile = (int)blockIdx.x * p.sample_stride;
            w.ks = 0;
            w.qb = 0;
            w.kb0 = 0;
            w.nkb = p.num_k_blocks;
            w.j = (int)blockIdx.x;
            w.chunk = 0;
            w.last = 1;
            return true;
        }
        j -= (int)gridDim.x;
    }
    if (j >= p.n_work) return false;
    w = decode_work(p, j);
    return true;
}

// Bounded spin on a device-scope arrival counter (one thread).  ~4 s worst case, then gives up: the caller turns
// that into a candidate overflow, which the host recovers through the dense route instead of hanging.
__device__ __forceinline__ bool spin_until(const uint32_t* ctr, uint32_t target) {
    const volatile uint32_t* c = ctr;
    for (int i = 0; i < (1 << 25); ++i) {
        if (*c >= target) return true;
        __nanosleep(100);
    }
    return false;
}

__device__ __forceinline__ int tile_of_work(const ScanParams& p, int j) {
    if (p.mode == MDIR_SCAN_DENSE) return j;
    if (p.mode == MDIR_SCAN_SAMPLE) return j * p.sample_stride;
    // FILTER: every tile that is not a sample tile
    if (p.n_sample == 0) return j;
    const int per = p.sample_stride - 1;
    const int in_groups = p.n_sample * per;
    if (j < in_groups) {
        const int g = j / per;
        return g * p.sample_stride + 1 + (j - g * per);
    }
    return p.n_sample * p.sample_stride + (j - in_groups);
}

// 16 scores (columns c0 .. c0 + 15 of this warp's TMEM lanes) of one accumulator.  int8: the hi plane's s32 sums sit in
// columns [0, n_pad), the lo plane's in [n_pad, 2 n_pad); s_r is this lane's row scale and qsc the per-query scales.
template <int KIND>
__device__ __forceinline__ void acc_scores16(uint32_t taddr, int c0, int n_pad, float s_r, const float* qsc, float (&s)[16]) {
    uint32_t v[16];
    tmem_ld16(taddr + (uint32_t)c0, v);
    if (KIND == kKindI8) {
        uint32_t lo[16];
        tmem_ld16(taddr + (uint32_t)(n_pad + c0), lo);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const float2 sc = *reinterpret_cast<const float2*>(qsc + 2 * (c0 + i));
            s[i] = __fmul_rn(__fmaf_rn((float)(int)v[i], sc.x, __fmul_rn((float)(int)lo[i], sc.y)), s_r);
        }
    } else {
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 16; ++i) s[i] = __uint_as_float(v[i]);
    }
}

// KIND = kKindI8 (FUSED mode only): the accumulators rotate per 128-row HALF rather than per tile.  Two planes of up
// to 80 queries make N = 160 columns per half, so two whole tiles (640 columns) no longer fit TMEM's 512; three
// half-accumulators (480) do.  Half index i = 2 * item + h lives in buffer i % acc_bufs: the MMAs of the next tile wait
// only for the epilogue of this tile's first half, and the second half's epilogue overlaps them.
template <int KIND>
__global__ void __launch_bounds__(kThreads, 1) sim_scan_kernel(const __grid_constant__ CUtensorMap tmap_db,
                                                                const __grid_constant__ CUtensorMap tmap_q, const ScanParams p) {
    constexpr bool TF32 = KIND == kKindTf32;
    constexpr bool I8 = KIND == kKindI8;
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t full_bar[kMaxStages];
    __shared__ __align__(8) uint64_t empty_bar[kMaxStages];
    __shared__ __align__(8) uint64_t tmem_full_bar[kMaxAccBufs];
    __shared__ __align__(8) uint64_t tmem_empty_bar[kMaxAccBufs];
    __shared__ uint32_t tmem_base_s;
    __shared__ uint64_t tau_s0[kMaxN];
    __shared__ float tau_f0[kMaxN];
    __shared__ uint32_t cand_n0[kMaxN];    // candidates this CTA has appended per query (CTA-private list: no global atomics)
    __shared__ __align__(8) float qsc[I8 ? 2 * 128 : 2];    // int8: {s_hi, s_lo} per query

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t b_bytes = (uint32_t)p.n_pad * 128u * (I8 ? 2u : 1u);
    const uint32_t stage_bytes = (uint32_t)kABytes + b_bytes;
    // per-query filter state: the static arrays for one block of queries; behind the operand ring for a wide launch
    // (n_qblocks blocks of n_pad queries: thresholds and counters of all n_q_total queries stay resident)
    uint64_t* tau_s = tau_s0;
    float* tau_f = tau_f0;
    uint32_t* cand_n = cand_n0;
    const int n_state = p.n_qblocks > 1 ? p.n_qblocks * p.n_pad : kMaxN;
    if (p.n_qblocks > 1 && p.mode == MDIR_SCAN_FILTER) {
        uint8_t* wide = smem_raw + (smem_base - smem_u32(smem_raw)) + (uint32_t)p.num_stages * stage_bytes;
        tau_s = reinterpret_cast<uint64_t*>(wide);
        tau_f = reinterpret_cast<float*>(tau_s + n_state);
        cand_n = reinterpret_cast<uint32_t*>(tau_f + n_state);
    }

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_db) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_q) : "memory");
        for (int s = 0; s < p.num_stages; ++s) {
            mbar_init(smem_u32(&full_bar[s]), 1);
            mbar_init(smem_u32(&empty_bar[s]), 1);
        }
        for (int b = 0; b < p.acc_bufs; ++b) {
            mbar_init(smem_u32(&tmem_full_bar[b]), 1);
            mbar_init(smem_u32(&tmem_empty_bar[b]), 4);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(kTmemCols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (p.mode == MDIR_SCAN_FUSED) {
        for (int c = threadIdx.x; c < kMaxN; c += kThreads) cand_n[c] = 0u;
        if (I8)
            for (int c = threadIdx.x; c < 2 * p.n_pad; c += kThreads) qsc[c] = c < 2 * p.n_q ? p.q_scale[c] : 0.f;
    } else if (p.mode == MDIR_SCAN_FILTER) {
        for (int c = threadIdx.x; c < n_state; c += kThreads) {
            uint64_t t = c < p.n_q_total ? p.tau[c] : 0ull;
            tau_s[c] = t;
            tau_f[c] = ((uint32_t)(t >> 32) == 0xffffffffu) ? -INFINITY : key_score(t);
            cand_n[c] = 0u;
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;

    if (warp == 0) {
        // ------------------------------------------------------------ TMA producer
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            WorkItem w;
            for (int it = 0; next_item(p, it, w); ++it) {
                const int row0 = w.tile * kBlockM;
                for (int kb = w.kb0; kb < w.kb0 + w.nkb; ++kb) {
                    mbar_wait(smem_u32(&empty_bar[stage]), phase ^ 1u);
                    const uint32_t fb = smem_u32(&full_bar[stage]);
                    const uint32_t a_dst = smem_base + (uint32_t)stage * stage_bytes;
                    mbar_expect_tx(fb, stage_bytes);
                    constexpr int kElemsPerBlock = TF32 ? 32 : (I8 ? 128 : 64);
                    tma_load_2d(a_dst, &tmap_db, fb, kb * kElemsPerBlock, row0, p.db_hint);
                    tma_load_2d(a_dst + kABytes, &tmap_q, fb, kb * kElemsPerBlock, w.qb * p.n_pad, kEvictLast);
                    if (++stage == p.num_stages) { stage = 0; phase ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------ MMA issuer
        if (lane == 0) {
            // instruction descriptor: D format [4,6) = 1 (f32) or 2 (s32), A/B format [7,10)/[10,13) = 1 (bf16 / signed
            // int8) or 2 (tf32), K-major A/B, N>>3 [17,23), M>>4 [24,29); int8: N = both query planes
            constexpr uint32_t fmt = TF32 ? 2u : 1u;
            constexpr uint32_t dfmt = I8 ? 2u : 1u;
            const uint32_t n_mma = (uint32_t)p.n_pad * (I8 ? 2u : 1u);
            const uint32_t idesc = (dfmt << 4) | (fmt << 7) | (fmt << 10) | ((n_mma >> 3) << 17) | ((128u >> 4) << 24);
            int stage = 0;
            uint32_t phase = 0;
            WorkItem w;
            for (int it = 0; next_item(p, it, w); ++it) {
                const int b = it % p.acc_bufs;
                const uint32_t acc_phase = (uint32_t)(it / p.acc_bufs) & 1u;
                uint32_t d_half[2];
                if (I8) {
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const int i = 2 * it + h, hb = i % p.acc_bufs;
                        mbar_wait(smem_u32(&tmem_empty_bar[hb]), ((uint32_t)(i / p.acc_bufs) & 1u) ^ 1u);
                        d_half[h] = tmem_base + (uint32_t)hb * (uint32_t)p.acc_stride;
                    }
                } else {
                    mbar_wait(smem_u32(&tmem_empty_bar[b]), acc_phase ^ 1u);
#pragma unroll
                    for (int h = 0; h < 2; ++h) d_half[h] = tmem_base + (uint32_t)(b * 2 + h) * (uint32_t)p.acc_stride;
                }
                tc_fence_after();
                const int nkb = w.nkb;
                for (int kb = 0; kb < nkb; ++kb) {
                    mbar_wait(smem_u32(&full_bar[stage]), phase);
                    tc_fence_after();
                    const uint32_t a_base = smem_base + (uint32_t)stage * stage_bytes;
                    const uint32_t b_base = a_base + kABytes;
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
#pragma unroll
                        for (int k = 0; k < kKSteps; ++k) {
                            const uint64_t ad = umma_desc_sw128(a_base + (uint32_t)h * (128u * 128u) + (uint32_t)k * 32u);
                            const uint64_t bd = umma_desc_sw128(b_base + (uint32_t)k * 32u);
                            umma_ss<KIND>(d_half[h], ad, bd, idesc, (kb | k) != 0 ? 1u : 0u);
                        }
                    }
                    umma_commit(smem_u32(&empty_bar[stage]));     // frees the smem slot when these MMAs retire
                    if (++stage == p.num_stages) { stage = 0; phase ^= 1u; }
                }
                if (I8) {                                          // accumulators of this tile are complete
                    umma_commit(smem_u32(&tmem_full_bar[(2 * it) % p.acc_bufs]));
                    umma_commit(smem_u32(&tmem_full_bar[(2 * it + 1) % p.acc_bufs]));
                } else {
                    umma_commit(smem_u32(&tmem_full_bar[b]));
                }
            }
        }
    } else {
        // ------------------------------------------------------------ epilogue (warps 2..5)
        const int quarter = warp & 3;                  // TMEM lane quarter this warp may read
        const int64_t cand_row = (int64_t)p.cap_s + (int64_t)kNumSMs * p.cap_l;
        const int64_t cand_seg_off = (int64_t)p.cap_s + (int64_t)blockIdx.x * p.cap_l;
        const int emode = p.mode == MDIR_SCAN_FUSED ? MDIR_SCAN_FILTER : p.mode;
        float* chain_sum = reinterpret_cast<float*>(smem_raw + (smem_base - smem_u32(smem_raw)) + (uint32_t)p.num_stages * stage_bytes);
        WorkItem w;
        for (int it = 0; next_item(p, it, w); ++it) {
            const int b = it % p.acc_bufs;
            const uint32_t acc_phase = (uint32_t)(it / p.acc_bufs) & 1u;
            const int tile = w.tile;
            float* dense_out = p.dense_out + (int64_t)w.ks * p.split_stride + (int64_t)w.qb * p.n_pad * p.dense_ld;
            const int nq_here = p.n_qblocks > 1 ? min(p.n_pad, p.n_q_total - w.qb * p.n_pad) : p.n_q;     // queries of this item's block
            // int8: this lane's row scales of both halves, loaded before the accumulator waits so that their latency hides
            // under the MMAs instead of stalling the epilogue (and with it the release of the TMEM buffer)
            float s_rh[2] = {0.f, 0.f};
            if (I8) {
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int64_t row = (int64_t)tile * kBlockM + h * 128 + quarter * 32 + lane;
                    if (row < p.n_db) s_rh[h] = __ldg(p.row_scale + row);
                }
            }
            // live bits of this lane's rows in both halves: the 32 rows of a warp and half are one aligned bitmap word, so
            // this is one broadcast load per warp and half, also issued before the accumulator waits
            uint32_t live_w[2] = {0xffffffffu, 0xffffffffu};
            if (p.live) {
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int64_t row0 = (int64_t)tile * kBlockM + h * 128 + quarter * 32;
                    live_w[h] = row0 < p.n_db ? __ldg(p.live + (row0 >> 5)) : 0u;
                }
            }
            // TMEM column of half h of this item's accumulators, and (int8) the barrier slot / phase of that half
            auto acc_col = [&](int h) -> uint32_t {
                return I8 ? (uint32_t)((2 * it + h) % p.acc_bufs) * (uint32_t)p.acc_stride : (uint32_t)(b * 2 + h) * (uint32_t)p.acc_stride;
            };
            if (!I8 || (p.mode == MDIR_SCAN_FUSED && it == 0)) {
                for (int h = 0; h < (I8 ? 2 : 1); ++h) {
                    const int i = I8 ? 2 * it + h : it;
                    mbar_wait(smem_u32(&tmem_full_bar[i % p.acc_bufs]), (uint32_t)(i / p.acc_bufs) & 1u);
                }
                tc_fence_after();
            }
            if (p.mode == MDIR_SCAN_FUSED && it == 0) {
                // ---- pass A over the sample tile: best two keys of each 32-row group (this warp x half), per query
                const int et = (int)threadIdx.x - 64;
#pragma unroll 1
                for (int h = 0; h < 2; ++h) {
                    const int64_t row = (int64_t)tile * kBlockM + h * 128 + quarter * 32 + lane;
                    const bool row_ok = row < p.n_db && (((h ? live_w[1] : live_w[0]) >> lane) & 1u);
                    const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + acc_col(h);
                    const float s_r = h ? s_rh[1] : s_rh[0];
#pragma unroll 1
                    for (int c0 = 0; c0 < p.n_pad; c0 += 16) {
                        float v[16];
                        acc_scores16<KIND>(taddr, c0, p.n_pad, s_r, qsc, v);
                        uint32_t m1 = 0xffffffffu, m2 = 0xffffffffu;
#pragma unroll
                        for (int i = 0; i < 16; ++i) {
                            const uint32_t key = row_ok ? desc_key(v[i]) : 0xffffffffu;
                            const uint32_t a = __reduce_min_sync(0xffffffffu, key);
                            const unsigned who = __ballot_sync(0xffffffffu, key == a);
                            const uint32_t key2 = (lane == __ffs(who) - 1) ? 0xffffffffu : key;
                            const uint32_t bb = __reduce_min_sync(0xffffffffu, key2);
                            if (lane == i) { m1 = a; m2 = bb; }
                        }
                        if (lane < 16 && c0 + lane < p.n_q) {
                            uint32_t* dst = p.grp_top + (((int64_t)(c0 + lane) * gridDim.x + blockIdx.x) * 8 + (quarter * 2 + h)) * 2;
                            *reinterpret_cast<uint2*>(dst) = make_uint2(m1, m2);
                        }
                    }
                }
                // ---- grid-wide arrival 1, then CTA q turns query q's grid*16 values into its threshold
                __shared__ uint32_t sel_hist[256];
                __shared__ uint32_t sel_prefix, sel_k, sel_ok;
                asm volatile("bar.sync 1, 128;" ::: "memory");
                if (et == 0) {
                    __threadfence();
                    atomicAdd(&p.sync[0], 1u);
                    sel_ok = 1u;
                }
                const int n_val = (int)gridDim.x * 16;
                for (int q = blockIdx.x; q < p.n_q; q += gridDim.x) {
                    if (et == 0) {
                        if (!spin_until(&p.sync[0], gridDim.x)) sel_ok = 0u;
                        __threadfence();
                        sel_prefix = 0u;
                        sel_k = (uint32_t)p.kth;
                    }
                    asm volatile("bar.sync 1, 128;" ::: "memory");
                    constexpr int kPer = (kNumSMs * 16 + 127) / 128;
                    uint32_t vals[kPer];
                    const uint32_t* src = p.grp_top + (int64_t)q * n_val;
#pragma unroll
                    for (int k = 0; k < kPer; ++k) {
                        const int i = et + 128 * k;
                        vals[k] = i < n_val ? __ldcg(src + i) : 0xffffffffu;
                    }
                    uint32_t result = 0xffffffffu;
                    if (p.kth <= n_val) {
                        for (int pass = 0; pass < 4; ++pass) {
                            const int shift = 24 - 8 * pass;
                            sel_hist[et] = 0u;
                            sel_hist[et + 128] = 0u;
                            asm volatile("bar.sync 1, 128;" ::: "memory");
                            const uint32_t prefix = sel_prefix;
                            const uint32_t himask = pass == 0 ? 0u : (0xffffffffu << (shift + 8));
#pragma unroll
                            for (int k = 0; k < kPer; ++k)
                                if (et + 128 * k < n_val && (vals[k] & himask) == prefix) atomicAdd(&sel_hist[(vals[k] >> shift) & 255u], 1u);
                            asm volatile("bar.sync 1, 128;" ::: "memory");
                            if (warp == 2) {
                                uint32_t before;
                                const int bin = find_bin_warp0(sel_hist, sel_k, &before);
                                __syncwarp();                       // every lane has read sel_k before lane 0 rewrites it
                                if (lane == 0) {
                                    sel_prefix = prefix | ((uint32_t)bin << shift);
                                    sel_k -= before;
                                }
                            }
                            asm volatile("bar.sync 1, 128;" ::: "memory");
                        }
                        // only the publishing thread reads it (it also rewrites it next round).  volatile: the compiler
                        // otherwise loads sel_prefix on every thread and selects by predicate -- harmless, but the other
                        // threads' speculative read then races with this thread's next-round store (racecheck)
                        if (et == 0) result = *reinterpret_cast<volatile uint32_t*>(&sel_prefix);
                    }
                    if (et == 0) {
                        p.tau_rw[q] = sel_ok ? (((uint64_t)result << 32) | 0xffffffffull) : 0ull;
                        __threadfence();
                        atomicAdd(&p.sync[1], 1u);
                    }
                }
                // ---- grid-wide arrival 2: every threshold is published
                if (et == 0) {
                    if (!spin_until(&p.sync[1], (uint32_t)p.n_q)) sel_ok = 0u;
                    __threadfence();
                }
                asm volatile("bar.sync 1, 128;" ::: "memory");
                {
                    const bool ok = sel_ok != 0u;
                    const uint64_t tq = (ok && et < p.n_q) ? __ldcg(reinterpret_cast<const unsigned long long*>(p.tau_rw) + et) : 0ull;
                    tau_s[et] = tq;
                    tau_f[et] = ((uint32_t)(tq >> 32) == 0xffffffffu) ? -INFINITY : key_score(tq);
                    if (!ok) cand_n[et] = (uint32_t)p.cap_l + 1u;        // barrier timed out: report overflow, never hang
                }
                asm volatile("bar.sync 1, 128;" ::: "memory");
            }
#pragma unroll 1
            for (int h = 0; h < 2; ++h) {
                const int r_in_tile = h * 128 + quarter * 32 + lane;
                const int64_t row = (int64_t)tile * kBlockM + r_in_tile;
                const bool row_in = row < p.n_db;
                const bool row_ok = row_in && (((h ? live_w[1] : live_w[0]) >> lane) & 1u);      // no dynamic index: no stack
                if (I8) {
                    const int i = 2 * it + h;
                    mbar_wait(smem_u32(&tmem_full_bar[i % p.acc_bufs]), (uint32_t)(i / p.acc_bufs) & 1u);
                    tc_fence_after();
                }
                const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + acc_col(h);
                const float s_r = h ? s_rh[1] : s_rh[0];
                const int64_t out_row = (p.mode == MDIR_SCAN_SAMPLE ? (int64_t)w.j * kBlockM : (int64_t)tile * kBlockM) + r_in_tile;
                const uint32_t gidx = p.idx_base + (uint32_t)row;
#pragma unroll 1
                for (int c0 = 0; c0 < p.n_pad; c0 += 16) {
                    float v[16];
                    acc_scores16<KIND>(taddr, c0, p.n_pad, s_r, qsc, v);
                    if (emode != MDIR_SCAN_FILTER) {
                        // rows past the end of the database only exist in the compact SAMPLE buffer: mark them -inf, and
                        // dead rows too
                        if (p.chain > 1) {
                            // chained chunk: running sum of this thread's row in shared memory (column-major, 128 rows
                            // per (half, column): conflict-free); only the last chunk touches dense_out
                            float* sum = chain_sum + ((int64_t)(h * p.n_pad + c0) * 128 + quarter * 32 + lane);
                            if (w.chunk == 0) {
#pragma unroll
                                for (int i = 0; i < 16; ++i) sum[i * 128] = v[i];
                            } else if (!w.last) {
#pragma unroll
                                for (int i = 0; i < 16; ++i) sum[i * 128] = __fadd_rn(sum[i * 128], v[i]);
                            } else if (row_ok) {
#pragma unroll
                                for (int i = 0; i < 16; ++i)
                                    if (c0 + i < p.n_q)
                                        dense_out[(int64_t)(c0 + i) * p.dense_ld + out_row] = __fadd_rn(sum[i * 128], v[i]);
                            }
                        } else if (row_in || p.mode == MDIR_SCAN_SAMPLE) {
#pragma unroll
                            for (int i = 0; i < 16; ++i)
                                if (c0 + i < nq_here)
                                    dense_out[(int64_t)(c0 + i) * p.dense_ld + out_row] = row_ok ? v[i] : -INFINITY;
                        }
                    } else if (row_ok) {
                        const int qo = w.qb * p.n_pad + c0;               // first query of these 16 columns
#pragma unroll
                        for (int i = 0; i < 16; ++i) {
                            const float s = v[i];
                            if (s >= tau_f[qo + i] && c0 + i < nq_here) {
                                const uint64_t key = make_key(s, gidx);
                                if (key <= tau_s[qo + i]) {
                                    const uint32_t pos = atomicAdd(&cand_n[qo + i], 1u);      // shared memory, rare
                                    if (pos < (uint32_t)p.cap_l)
                                        p.cand[(int64_t)(qo + i) * cand_row + cand_seg_off + pos] = key;
                                }
                            }
                        }
                    }
                }
                if (I8) {                                  // this half's accumulator is free for the MMAs of a later tile
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(smem_u32(&tmem_empty_bar[(2 * it + h) % p.acc_bufs]));
                }
            }
            if (!I8) {
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(smem_u32(&tmem_empty_bar[b]));
            }
        }
        if (emode == MDIR_SCAN_FILTER) {
            asm volatile("bar.sync 1, 128;" ::: "memory");       // the four epilogue warps only
            for (int t = (int)threadIdx.x - 64; t < p.n_q_total; t += 128) {
                p.seg_counts[(int64_t)t * MDIR_CAND_SEGS + 1 + blockIdx.x] = cand_n[t];
                if (p.mode == MDIR_SCAN_FUSED && blockIdx.x == 0) {
                    // no select kernel in this route: segment 0 and the segments of absent CTAs are empty
                    p.seg_counts[(int64_t)t * MDIR_CAND_SEGS] = 0u;
                    for (int s = 1 + (int)gridDim.x; s < MDIR_CAND_SEGS; ++s) p.seg_counts[(int64_t)t * MDIR_CAND_SEGS + s] = 0u;
                }
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
    }
    if (p.mode == MDIR_SCAN_FUSED && threadIdx.x == 0) {
        // the last CTA out re-arms the arrival counters for the next launch on this workspace
        if (atomicAdd(&p.sync[3], 1u) == gridDim.x - 1) {
            p.sync[0] = 0u;
            p.sync[1] = 0u;
            p.sync[3] = 0u;
            __threadfence();
        }
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)ptr;
    }
    return fn;
}

static int make_tmap(CUtensorMap* map, int kind, const void* ptr, uint64_t rows, uint64_t cols, uint32_t box_rows) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) {
        set_error("cuTensorMapEncodeTiled entry point unavailable");
        return MDIR_E_DRIVER;
    }
    cuuint64_t gdim[2] = {cols, rows};
    const uint32_t esz = kind == kKindTf32 ? 4u : (kind == kKindI8 ? 1u : 2u);
    cuuint64_t gstride[1] = {cols * esz};
    cuuint32_t box[2] = {(cuuint32_t)(kBlockKBytes / esz), box_rows};      // one 128-byte swizzle row per operand row
    cuuint32_t estr[2] = {1, 1};
    const CUtensorMapDataType dt = kind == kKindTf32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                   : (kind == kKindI8 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16);
    CUresult r = fn(map, dt, 2, const_cast<void*>(ptr), gdim, gstride, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed with CUresult " + std::to_string((int)r));
        return MDIR_E_DRIVER;
    }
    return 0;
}

}  // namespace mdir

using namespace mdir;

// kind: kKindBf16 / kKindTf32 (bool false / true at the older call sites) or kKindI8 (FUSED mode only; q = the two
// int8 planes of mdir_pack_q_i8, row_scale / q_scale = s_r and {s_hi, s_lo})
static int launch_scan(int kind, const void* db, int64_t n_db, const void* q, int n_q, int D, int mode, int sample_stride, int n_sample,
                       float* dense_out, int64_t dense_ld, const uint64_t* tau, uint32_t idx_base, uint64_t* cand,
                       uint32_t* seg_counts, int cap_s, int cap_l, void* stream, int k_split = 1, int64_t split_stride = 0,
                       int kth = 0, uint32_t* fused_ws = nullptr, uint64_t* tau_rw = nullptr, int n_q_total = 0,
                       const float* row_scale = nullptr, const float* q_scale = nullptr, const uint32_t* live = nullptr) {
    const bool tf32 = kind == kKindTf32, i8 = kind == kKindI8;
    const int esz = tf32 ? 4 : (i8 ? 1 : 2);
    MDIR_CHECK_ARG(db && q && n_db >= 1 && n_q >= 1 && n_q <= kMaxN && D >= 16 / esz && (D % (16 / esz)) == 0);
    MDIR_CHECK_ARG((((uintptr_t)db | (uintptr_t)q) & 15) == 0);
    MDIR_CHECK_ARG(mode >= 0 && mode <= MDIR_SCAN_FUSED);
    MDIR_CHECK_ARG(n_db + (int64_t)idx_base <= ((int64_t)1 << 32));
    MDIR_CHECK_ARG(!i8 || (mode == MDIR_SCAN_FUSED && row_scale && q_scale));
    MDIR_CHECK_ARG(!live || !tf32);
    ScanParams p;
    p.row_scale = row_scale;
    p.q_scale = q_scale;
    p.live = live;
    p.n_db = n_db;
    p.n_q = n_q;
    p.n_pad = (n_q + 15) & ~15;
    const int elems_per_block = kBlockKBytes / esz;
    p.num_k_blocks = (D + elems_per_block - 1) / elems_per_block;
    const int64_t n_tiles64 = (n_db + kBlockM - 1) / kBlockM;
    MDIR_CHECK_ARG(n_tiles64 < ((int64_t)1 << 23));
    p.n_tiles = (int)n_tiles64;
    p.mode = mode;
    p.sample_stride = sample_stride;
    p.n_sample = n_sample;
    p.k_split = 1;
    p.kb_per_split = p.num_k_blocks;
    p.split_stride = split_stride;
    p.chain = 1;
    p.kb_per_chain = p.num_k_blocks;
    p.n_qblocks = 1;
    p.n_q_total = n_q;
    if (n_q_total > n_q) {
        // several blocks of n_pad queries in one launch (bf16, no split-K): one ramp instead of one per block, and the
        // database tile of a work item is re-read from L2, not HBM, by the other query blocks
        MDIR_CHECK_ARG(!tf32 && k_split == 1 && n_q == p.n_pad && mode != MDIR_SCAN_FUSED);
        p.n_q_total = n_q_total;
        p.n_qblocks = (n_q_total + p.n_pad - 1) / p.n_pad;
        MDIR_CHECK_ARG(p.n_qblocks * p.n_pad <= kMaxWideQ || mode == MDIR_SCAN_DENSE);
        MDIR_CHECK_ARG((int64_t)p.n_tiles * p.n_qblocks < ((int64_t)1 << 30));
    }
    // TMEM (512 columns): 3 tiles of 2 x 80 columns, 2 of 2 x 128, or -- 129..256 queries, the tensor-bound shapes
    // (DBA, all-pairs): AI = n_q FLOP/B crosses the ~214 FLOP/B ridge -- ONE tile of 2 x 256 (the epilogue of a tile is
    // then not overlapped with the next tile's MMAs: ~10 % of a D = 2048 tile)
    p.acc_bufs = p.n_pad <= 80 ? 3 : (p.n_pad <= 128 ? 2 : 1);
    p.acc_stride = p.n_pad <= 80 ? 80 : (p.n_pad <= 128 ? 128 : 256);
    if (i8) {
        // half-accumulators of both query planes: 3 x 160 columns up to 80 queries, else 2 x (2 n_pad) (= one tile)
        p.acc_stride = 2 * p.n_pad;
        p.acc_bufs = p.n_pad <= 80 ? 3 : 2;
    }
    p.kth = 0;
    p.grp_top = nullptr;
    p.sync = nullptr;
    p.tau_rw = nullptr;
    if (mode == MDIR_SCAN_DENSE) {
        MDIR_CHECK_ARG(dense_out && dense_ld >= n_db);
        if (k_split > 1) {
            p.kb_per_split = (p.num_k_blocks + k_split - 1) / k_split;
            p.k_split = (p.num_k_blocks + p.kb_per_split - 1) / p.kb_per_split;     // every split gets >= 1 k-block
        }
        p.n_work = p.n_tiles * p.k_split;
        if (n_q_total > n_q) p.n_work = p.n_tiles * p.n_qblocks;
        if (tf32 && p.k_split == 1 && p.num_k_blocks > 2 * kChainKBlocks) {
            // fp32-faithful path: at most 16 truncating MMAs per TMEM accumulation (see ScanParams::chain)
            if (p.n_pad > kChainMaxN) {
                // the running sums (256 x n_pad fp32) share the CTA's shared memory with the operand ring: wider query
                // blocks go as two launches
                const int n0 = ((n_q / 2) + 15) & ~15;
                int rc = launch_scan(kind, db, n_db, q, n0, D, mode, sample_stride, n_sample, dense_out, dense_ld, tau, idx_base, cand, seg_counts,
                                     cap_s, cap_l, stream);
                if (rc) return rc;
                return launch_scan(kind, db, n_db, static_cast<const uint8_t*>(q) + (size_t)n0 * D * esz, n_q - n0, D, mode, sample_stride, n_sample,
                                   dense_out + (int64_t)n0 * dense_ld, dense_ld, tau, idx_base, cand, seg_counts, cap_s, cap_l, stream);
            }
            p.kb_per_chain = kChainKBlocks;
            p.chain = (p.num_k_blocks + kChainKBlocks - 1) / kChainKBlocks;
        }
    } else if (mode == MDIR_SCAN_SAMPLE) {
        MDIR_CHECK_ARG(dense_out && n_sample >= 1 && sample_stride >= 1);
        MDIR_CHECK_ARG((int64_t)(n_sample - 1) * sample_stride < p.n_tiles);
        MDIR_CHECK_ARG(dense_ld >= (int64_t)n_sample * kBlockM);
        p.n_work = n_sample * p.n_qblocks;
    } else if (mode == MDIR_SCAN_FUSED) {
        // one sample tile per CTA, all CTAs co-resident (the in-kernel arrival counters rely on it)
        MDIR_CHECK_ARG(tau_rw && fused_ws && cand && seg_counts && cap_l >= 1 && kth >= 1 && n_q <= 128);
        const int sm_count = device_sm_count();
        MDIR_CHECK_ARG(sm_count > 0);
        int g = sm_count < kNumSMs ? sm_count : kNumSMs;
        if (g_scan_max_ctas > 0 && g > g_scan_max_ctas) g = g_scan_max_ctas;      // leave SMs to a concurrent finalize (mdir_tune)
        if (g > p.n_tiles / 2) g = p.n_tiles / 2;
        MDIR_CHECK_ARG(g >= 1);
        g = balanced_grid(p.n_tiles, g);          // every CTA scans the same number of tiles (its sample tile included)
        p.n_sample = g;
        p.sample_stride = p.n_tiles / g;
        p.n_work = p.n_tiles - g;
        p.kth = kth;
        p.grp_top = fused_ws + 4;
        p.sync = fused_ws;
        p.tau_rw = tau_rw;
    } else {
        MDIR_CHECK_ARG(tau && cand && seg_counts && cap_s >= 0 && cap_l >= 1);
        MDIR_CHECK_ARG(n_sample >= 0 && (n_sample == 0 || sample_stride >= 2));
        MDIR_CHECK_ARG(n_sample == 0 || (int64_t)(n_sample - 1) * sample_stride < p.n_tiles);
        p.n_work = (p.n_tiles - n_sample) * p.n_qblocks;
    }
    p.dense_out = dense_out;
    p.dense_ld = dense_ld;
    p.tau = tau;
    p.idx_base = idx_base;
    p.cand = cand;
    p.seg_counts = seg_counts;
    p.cap_s = cap_s;
    p.cap_l = cap_l;
    // a database that fits L2 (126 MB) is worth keeping there across query blocks / passes
    p.db_hint = ((int64_t)n_db * D * esz > (int64_t)96 * 1024 * 1024) ? kEvictFirst : kEvictNormal;
    if (p.n_work <= 0 && mode != MDIR_SCAN_FUSED) return 0;

    const int stage_bytes = kABytes + p.n_pad * 128 * (i8 ? 2 : 1);
    int chain_bytes = p.chain > 1 ? kBlockM * p.n_pad * 4 : 0;            // running sums of the chained tf32 DENSE scan
    if (p.n_qblocks > 1 && mode == MDIR_SCAN_FILTER) chain_bytes = p.n_qblocks * p.n_pad * 16;      // wide FILTER: per-query thresholds + counters
    int stages = (232448 - 1024 - 8192 - chain_bytes) / stage_bytes;      // 8 KB left for the static shared arrays
    if (stages > kMaxStages) stages = kMaxStages;
    MDIR_CHECK_ARG(stages >= 2);
    p.num_stages = stages;
    const size_t smem = (size_t)stages * stage_bytes + 1024 + chain_bytes;

    CUtensorMap tmap_db, tmap_q;
    int rc = make_tmap(&tmap_db, kind, db, (uint64_t)n_db, (uint64_t)D, kBlockM);
    if (rc) return rc;
    const int q_rows = i8 ? 2 * p.n_pad : p.n_q_total;         // int8: hi plane rows [0, n_pad), lo plane rows [n_pad, 2 n_pad)
    rc = make_tmap(&tmap_q, kind, q, (uint64_t)q_rows, (uint64_t)D, (uint32_t)(i8 ? 2 * p.n_pad : p.n_pad));
    if (rc) return rc;

    static PerDeviceOnce once;
    if (once.first() != 0) {
        MDIR_CUDA(cudaFuncSetAttribute(sim_scan_kernel<kKindBf16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448 - 8192));
        MDIR_CUDA(cudaFuncSetAttribute(sim_scan_kernel<kKindTf32>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448 - 8192));
        MDIR_CUDA(cudaFuncSetAttribute(sim_scan_kernel<kKindI8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448 - 8192));
    }
    const int n_ctas_wanted = p.chain > 1 ? p.n_tiles : p.n_work;
    int grid = mode == MDIR_SCAN_FUSED ? p.n_sample : balanced_grid(n_ctas_wanted, kNumSMs);
    if (p.n_qblocks > 1) {
        // CTA c takes items c, c + grid, ...: with grid coprime to the number of query blocks it meets every block equally
        // often (148 CTAs and 8 blocks would give each CTA only two of them -- and each query's candidates only a
        // quarter of the per-CTA segments, four times as full)
        auto gcd = [](int a, int b) { while (b) { const int t = a % b; a = b; b = t; } return a; };
        while (grid > 1 && gcd(grid, p.n_qblocks) != 1) --grid;
    }
    if (mode == MDIR_SCAN_FUSED) {
        // the in-kernel threshold exchange is a grid-wide rendezvous: launch COOPERATIVELY, so the runtime guarantees
        // that all `grid` CTAs are co-resident (or fails the launch) instead of the kernel relying on an empty device
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(grid);
        cfg.blockDim = dim3(kThreads);
        cfg.dynamicSmemBytes = smem;
        cfg.stream = (cudaStream_t)stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeCooperative;
        attr[0].val.cooperative = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        if (i8) MDIR_CUDA(cudaLaunchKernelEx(&cfg, sim_scan_kernel<kKindI8>, tmap_db, tmap_q, p));
        else MDIR_CUDA(cudaLaunchKernelEx(&cfg, sim_scan_kernel<kKindBf16>, tmap_db, tmap_q, p));
        MDIR_LAUNCH_CHECK();
        return 0;
    }
    if (tf32) sim_scan_kernel<kKindTf32><<<grid, kThreads, smem, (cudaStream_t)stream>>>(tmap_db, tmap_q, p);
    else sim_scan_kernel<kKindBf16><<<grid, kThreads, smem, (cudaStream_t)stream>>>(tmap_db, tmap_q, p);
    MDIR_LAUNCH_CHECK();
    return 0;
}

extern "C" int mdir_sim_scan_bf16_live(const uint16_t* db, int64_t n_db, const uint16_t* q, int n_q, int D, int mode, int sample_stride,
                                       int n_sample, float* dense_out, int64_t dense_ld, const uint64_t* tau, uint32_t idx_base,
                                       uint64_t* cand, uint32_t* seg_counts, int cap_s, int cap_l, const uint32_t* live, void* stream) {
    return launch_scan(kKindBf16, db, n_db, q, n_q, D, mode, sample_stride, n_sample, dense_out, dense_ld, tau, idx_base, cand, seg_counts,
                       cap_s, cap_l, stream, 1, 0, 0, nullptr, nullptr, 0, nullptr, nullptr, live);
}

extern "C" int mdir_sim_scan_bf16(const uint16_t* db, int64_t n_db, const uint16_t* q, int n_q, int D, int mode, int sample_stride,
                                  int n_sample, float* dense_out, int64_t dense_ld, const uint64_t* tau, uint32_t idx_base,
                                  uint64_t* cand, uint32_t* seg_counts, int cap_s, int cap_l, void* stream) {
    return mdir_sim_scan_bf16_live(db, n_db, q, n_q, D, mode, sample_stride, n_sample, dense_out, dense_ld, tau, idx_base, cand, seg_counts,
                                   cap_s, cap_l, nullptr, stream);
}

extern "C" int mdir_sim_scan_dense_bf16(const uint16_t* db, int64_t n_db, const uint16_t* q, int n_q, int D, float* dense_out, int64_t dense_ld,
                                        void* stream) {
    // all of a (possibly > 128-query) block of queries in ONE launch: (tile, 128-query block) work items
    // 128 queries per work item: 256 (all of TMEM for one tile, no accumulator double-buffering, three 64 KB stages) was
    // measured 8-10 % slower on both the 512-D and the 2048-D shape
    const int blk = n_q < 128 ? n_q : 128;
    return launch_scan(kKindBf16, db, n_db, q, blk, D, MDIR_SCAN_DENSE, 0, 0, dense_out, dense_ld, nullptr, 0, nullptr, nullptr, 0, 0, stream, 1, 0, 0,
                       nullptr, nullptr, n_q > blk ? n_q : 0);
}

extern "C" int mdir_sim_scan_wide_bf16_live(const uint16_t* db, int64_t n_db, const uint16_t* q, int n_q, int D, int mode, int sample_stride,
                                            int n_sample, float* dense_out, int64_t dense_ld, const uint64_t* tau, uint32_t idx_base,
                                            uint64_t* cand, uint32_t* seg_counts, int cap_s, int cap_l, const uint32_t* live, void* stream) {
    // mdir_sim_scan_bf16 for 129 .. 1024 queries in one launch (DENSE: any number): blocks of 128 queries per work item
    MDIR_CHECK_ARG(n_q >= 1 && (mode == MDIR_SCAN_DENSE || n_q <= kMaxWideQ));
    const int blk = n_q < 128 ? n_q : 128;
    return launch_scan(kKindBf16, db, n_db, q, blk, D, mode, sample_stride, n_sample, dense_out, dense_ld, tau, idx_base, cand, seg_counts, cap_s,
                       cap_l, stream, 1, 0, 0, nullptr, nullptr, n_q > blk ? n_q : 0, nullptr, nullptr, live);
}

extern "C" int mdir_sim_scan_wide_bf16(const uint16_t* db, int64_t n_db, const uint16_t* q, int n_q, int D, int mode, int sample_stride,
                                       int n_sample, float* dense_out, int64_t dense_ld, const uint64_t* tau, uint32_t idx_base,
                                       uint64_t* cand, uint32_t* seg_counts, int cap_s, int cap_l, void* stream) {
    return mdir_sim_scan_wide_bf16_live(db, n_db, q, n_q, D, mode, sample_stride, n_sample, dense_out, dense_ld, tau, idx_base, cand, seg_counts,
                                        cap_s, cap_l, nullptr, stream);
}

extern "C" size_t mdir_sim_scan_fused_workspace_bytes(int n_q) {
    return (4 + (size_t)(n_q > 0 ? n_q : 0) * kNumSMs * 16) * sizeof(uint32_t);
}

extern "C" int mdir_sim_scan_fused_bf16_live(const uint16_t* db, int64_t n_db, const uint16_t* q, int n_q, int D, int kth, uint64_t* tau,
                                             uint32_t idx_base, uint64_t* cand, uint32_t* seg_counts, int cap_s, int cap_l, void* ws,
                                             const uint32_t* live, void* stream) {
    MDIR_CHECK_ARG(ws && (((uintptr_t)ws) & 15) == 0);
    return launch_scan(kKindBf16, db, n_db, q, n_q, D, MDIR_SCAN_FUSED, 0, 0, nullptr, 0, nullptr, idx_base, cand, seg_counts, cap_s, cap_l,
                       stream, 1, 0, kth, static_cast<uint32_t*>(ws), tau, 0, nullptr, nullptr, live);
}

extern "C" int mdir_sim_scan_fused_bf16(const uint16_t* db, int64_t n_db, const uint16_t* q, int n_q, int D, int kth, uint64_t* tau,
                                        uint32_t idx_base, uint64_t* cand, uint32_t* seg_counts, int cap_s, int cap_l, void* ws,
                                        void* stream) {
    return mdir_sim_scan_fused_bf16_live(db, n_db, q, n_q, D, kth, tau, idx_base, cand, seg_counts, cap_s, cap_l, ws, nullptr, stream);
}

extern "C" int mdir_sim_scan_fused_i8_live(const int8_t* db8, const float* row_scale, int64_t n_db, const int8_t* q8, const float* q_scale,
                                           int n_q, int D, int kth, uint64_t* tau, uint32_t idx_base, uint64_t* cand, uint32_t* seg_counts,
                                           int cap_s, int cap_l, void* ws, const uint32_t* live, void* stream) {
    MDIR_CHECK_ARG(ws && (((uintptr_t)ws) & 15) == 0 && D % 128 == 0);
    return launch_scan(kKindI8, db8, n_db, q8, n_q, D, MDIR_SCAN_FUSED, 0, 0, nullptr, 0, nullptr, idx_base, cand, seg_counts, cap_s, cap_l,
                       stream, 1, 0, kth, static_cast<uint32_t*>(ws), tau, 0, row_scale, q_scale, live);
}

extern "C" int mdir_sim_scan_fused_i8(const int8_t* db8, const float* row_scale, int64_t n_db, const int8_t* q8, const float* q_scale,
                                      int n_q, int D, int kth, uint64_t* tau, uint32_t idx_base, uint64_t* cand, uint32_t* seg_counts,
                                      int cap_s, int cap_l, void* ws, void* stream) {
    return mdir_sim_scan_fused_i8_live(db8, row_scale, n_db, q8, q_scale, n_q, D, kth, tau, idx_base, cand, seg_counts, cap_s, cap_l, ws,
                                       nullptr, stream);
}

extern "C" int mdir_sim_scan_tf32(const float* db, int64_t n_db, const float* q, int n_q, int D, int mode, int sample_stride,
                                  int n_sample, float* dense_out, int64_t dense_ld, const uint64_t* tau, uint32_t idx_base,
                                  uint64_t* cand, uint32_t* seg_counts, int cap_s, int cap_l, void* stream) {
    return launch_scan(kKindTf32, db, n_db, q, n_q, D, mode, sample_stride, n_sample, dense_out, dense_ld, tau, idx_base, cand, seg_counts,
                       cap_s, cap_l, stream);
}

// fp32 -> [hi | hi | lo] (role 0, database side) or [hi | lo | hi] (role 1, query side) with hi = x truncated to
// tf32 (10 explicit mantissa bits) and lo = x - hi (exact): scanning the two (n, 3D) matrices against each other
// with kind::tf32 accumulates hi*hi + hi*lo + lo*hi in fp32, i.e. an fp32-faithful dot product (3xTF32).
__global__ void __launch_bounds__(256) split_tf32x3_kernel(const float* __restrict__ src, int64_t n, int D, int role, float* __restrict__ dst) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n * D) return;
    const int64_t r = i / D;
    const int d = (int)(i - r * D);
    const float x = src[i];
    const float hi = __uint_as_float(__float_as_uint(x) & 0xffffe000u);
    const float lo = x - hi;
    float* o = dst + r * 3 * (int64_t)D;
    o[d] = hi;
    o[D + d] = role == 0 ? hi : lo;
    o[2 * D + d] = role == 0 ? lo : hi;
}

extern "C" int mdir_split_tf32x3(const float* src, int64_t n, int D, int role, float* dst, void* stream) {
    MDIR_CHECK_ARG(src && dst && n >= 0 && D > 0 && (role == 0 || role == 1));
    if (n == 0) return 0;
    const int64_t total = n * D;
    split_tf32x3_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(src, n, D, role, dst);
    MDIR_LAUNCH_CHECK();
    return 0;
}

// ---- Lw projection on the tensor cores: out = normalise(P[:dims] (v - m)) with 3xTF32 (fp32-faithful) -------------
namespace mdir {

// (v - m) -> [hi | lo | hi] (query-side role of the 3xTF32 split), rows [r0, r0 + nb)
__global__ void __launch_bounds__(256) center_split_kernel(const float* __restrict__ v, const float* __restrict__ m, int nb, int D,
                                                           float* __restrict__ dst) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)nb * D) return;
    const int64_t r = i / D;
    const int d = (int)(i - r * D);
    const float x = v[i] - (m ? m[d] : 0.f);
    const float hi = __uint_as_float(__float_as_uint(x) & 0xffffe000u);
    float* o = dst + r * 3 * (int64_t)D;
    o[d] = hi;
    o[D + d] = x - hi;
    o[2 * D + d] = hi;
}

// out[i] = sum_ks partial[ks * split_stride + i] in a fixed order (deterministic), 4 elements per thread
__global__ void __launch_bounds__(256) sum_partials_kernel(const float* __restrict__ partial, int k_split, int64_t split_stride,
                                                           int64_t total, float* __restrict__ out) {
    const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i >= total) return;
    if (i + 3 < total && (split_stride & 3) == 0) {
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
        int ks = 0;
        for (; ks + 3 < k_split; ks += 4) {                       // 4 independent 128-bit loads in flight
            const float4 v0 = *reinterpret_cast<const float4*>(partial + (int64_t)ks * split_stride + i);
            const float4 v1 = *reinterpret_cast<const float4*>(partial + (int64_t)(ks + 1) * split_stride + i);
            const float4 v2 = *reinterpret_cast<const float4*>(partial + (int64_t)(ks + 2) * split_stride + i);
            const float4 v3 = *reinterpret_cast<const float4*>(partial + (int64_t)(ks + 3) * split_stride + i);
            a.x = (((a.x + v0.x) + v1.x) + v2.x) + v3.x; a.y = (((a.y + v0.y) + v1.y) + v2.y) + v3.y;
            a.z = (((a.z + v0.z) + v1.z) + v2.z) + v3.z; a.w = (((a.w + v0.w) + v1.w) + v2.w) + v3.w;
        }
        for (; ks < k_split; ++ks) {
            const float4 v = *reinterpret_cast<const float4*>(partial + (int64_t)ks * split_stride + i);
            a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
        }
        *reinterpret_cast<float4*>(out + i) = a;
    } else {
        for (int64_t e = i; e < total && e < i + 4; ++e) {
            float a = 0.f;
            for (int ks = 0; ks < k_split; ++ks) a += partial[(int64_t)ks * split_stride + e];
            out[e] = a;
        }
    }
}

// x / (||x||_2 + eps) per row, in place (rows of `dims` floats)
__global__ void __launch_bounds__(256) row_l2n_kernel(float* x, int dims, float eps) {
    __shared__ float red[32];
    float* row = x + (int64_t)blockIdx.x * dims;
    float s = 0.f;
    for (int j = threadIdx.x; j < dims; j += blockDim.x) { const float v = row[j]; s += v * v; }
    s = block_sum(s, red);
    const float inv = 1.0f / (sqrtf(s) + eps);
    for (int j = threadIdx.x; j < dims; j += blockDim.x) row[j] *= inv;
}

// sum of the k_split partial planes (fixed order) fused with the row renormalisation: one CTA per descriptor.
// dims % 4 == 0 and 16-byte aligned planes (always true here: dims comes from the 256-row tiles of the scan).
__global__ void __launch_bounds__(256) sum_partials_l2n_kernel(const float* __restrict__ partial, int k_split, int64_t split_stride, int dims,
                                                               float eps, float* __restrict__ out) {
    __shared__ float red[32];
    const float* src = partial + (int64_t)blockIdx.x * dims;
    float* row = out + (int64_t)blockIdx.x * dims;
    float s = 0.f;
    for (int j = threadIdx.x * 4; j < dims; j += blockDim.x * 4) {
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
        int ks = 0;
        for (; ks + 7 < k_split; ks += 8) {                       // 8 independent 128-bit loads in flight, summed in plane order
            float4 v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) v[u] = *reinterpret_cast<const float4*>(src + (int64_t)(ks + u) * split_stride + j);
#pragma unroll
            for (int u = 0; u < 8; ++u) { a.x += v[u].x; a.y += v[u].y; a.z += v[u].z; a.w += v[u].w; }
        }
        for (; ks < k_split; ++ks) {
            const float4 v = *reinterpret_cast<const float4*>(src + (int64_t)ks * split_stride + j);
            a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
        }
        *reinterpret_cast<float4*>(row + j) = a;
        s += a.x * a.x + a.y * a.y + a.z * a.z + a.w * a.w;
    }
    s = block_sum(s, red);
    const float inv = 1.0f / (sqrtf(s) + eps);
    for (int j = threadIdx.x * 4; j < dims; j += blockDim.x * 4) {              // each thread re-reads only its own writes
        float4 a = *reinterpret_cast<float4*>(row + j);
        a.x *= inv; a.y *= inv; a.z *= inv; a.w *= inv;
        *reinterpret_cast<float4*>(row + j) = a;
    }
}

// Blocks of <= 128 descriptors; with more than one block two of them run concurrently (caller's stream + an internal
// one), each on half of the SMs, instead of back to back on all of them: the chain of small kernels per block is
// latency-bound, so two half-width chains finish in about the time of one.
static void whiten_blocks(int n, int* n_blocks, int* block_rows) {
    constexpr int kWhitenBlock = 128;           // descriptors per projection block (double-buffered TMEM accumulators)
    const int nblk = (n + kWhitenBlock - 1) / kWhitenBlock;
    int rows = (n + nblk - 1) / nblk;
    rows = (rows + 15) & ~15;
    if (rows > kWhitenBlock) rows = kWhitenBlock;
    *n_blocks = (n + rows - 1) / rows;
    *block_rows = rows;
}

static int whiten_plan(int D, int dims, int n_concurrent, int* k_split) {
    const int tiles = (dims + kBlockM - 1) / kBlockM;
    const int nkb = (3 * D + 31) / 32;
    int ks = (kNumSMs / n_concurrent) / tiles;
    if (ks < 1) ks = 1;
    if (ks > nkb) ks = nkb;
    const int per = (nkb + ks - 1) / ks;
    *k_split = (nkb + per - 1) / per;
    return 0;
}

}  // namespace mdir

static size_t whiten_slot_floats(int rows, int D, int dims, int ks) {
    return (((size_t)rows * 3 * D + (size_t)ks * rows * dims) + 63) & ~(size_t)63;
}

extern "C" size_t mdir_whiten_tc_workspace_bytes(int n, int D, int dims) {
    if (n <= 0 || D <= 0 || dims <= 0) return 0;
    int nblk, rows, ks;
    whiten_blocks(n, &nblk, &rows);
    const int conc = nblk > 1 ? 2 : 1;
    whiten_plan(D, dims, conc, &ks);
    return conc * whiten_slot_floats(rows, D, dims, ks) * 4 + 512;
}

extern "C" int mdir_whiten_project_tc(const float* v, const float* m, int n, int D, const float* Px3, int dims, float renorm_eps,
                                      float* out, void* ws, void* stream) {
    MDIR_CHECK_ARG(v && Px3 && out && ws && n >= 0 && D > 0 && (D % 4) == 0 && dims > 0);
    MDIR_CHECK_ARG((((uintptr_t)Px3 | (uintptr_t)ws) & 15) == 0);
    if (n == 0) return 0;
    int nblk, rows, ks;
    whiten_blocks(n, &nblk, &rows);
    const int conc = nblk > 1 ? 2 : 1;
    whiten_plan(D, dims, conc, &ks);
    const size_t slot = whiten_slot_floats(rows, D, dims, ks);
    float* ws0 = (float*)(((uintptr_t)ws + 255) & ~(uintptr_t)255);

    // fork: odd blocks run on an internal stream (created once per process), joined before returning; both the fork
    // and the join are event edges, so the whole thing is capturable into a CUDA graph
    static cudaStream_t side_dev[kMaxDevices] = {};
    static cudaEvent_t ev_fork_dev[kMaxDevices] = {}, ev_join_dev[kMaxDevices] = {};
    int cur_dev = 0;
    MDIR_CUDA(cudaGetDevice(&cur_dev));
    MDIR_CHECK_ARG(cur_dev >= 0 && cur_dev < kMaxDevices);
    cudaStream_t& side = side_dev[cur_dev];
    cudaEvent_t &ev_fork = ev_fork_dev[cur_dev], &ev_join = ev_join_dev[cur_dev];
    cudaStream_t main_st = (cudaStream_t)stream;
    if (conc > 1) {
        if (!side) {
            MDIR_CUDA(cudaStreamCreateWithFlags(&side, cudaStreamNonBlocking));
            MDIR_CUDA(cudaEventCreateWithFlags(&ev_fork, cudaEventDisableTiming));
            MDIR_CUDA(cudaEventCreateWithFlags(&ev_join, cudaEventDisableTiming));
        }
        MDIR_CUDA(cudaEventRecord(ev_fork, main_st));
        MDIR_CUDA(cudaStreamWaitEvent(side, ev_fork, 0));
    }
    for (int b = 0; b < nblk; ++b) {
        const int r0 = b * rows;
        const int nb = (n - r0) < rows ? (n - r0) : rows;
        cudaStream_t st = (b & 1) ? side : main_st;
        float* vx3 = ws0 + (size_t)(b & 1) * slot;
        float* partial = vx3 + (size_t)rows * 3 * D;
        const int64_t total = (int64_t)nb * D;
        center_split_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(v + (size_t)r0 * D, m, nb, D, vx3);
        MDIR_LAUNCH_CHECK();
        const int64_t split_stride = (int64_t)nb * dims;
        int rc = launch_scan(kKindTf32, Px3, dims, vx3, nb, 3 * D, MDIR_SCAN_DENSE, 0, 0, partial, dims, nullptr, 0, nullptr, nullptr, 0, 0,
                             (void*)st, ks, split_stride);
        if (rc) return rc;
        // launch_scan may have reduced the split count; recompute it the same way
        const int nkb = (3 * D + 31) / 32;
        const int per = (nkb + ks - 1) / ks;
        const int ks_eff = ks > 1 ? (nkb + per - 1) / per : 1;
        float* o = out + (size_t)r0 * dims;
        if (renorm_eps >= 0.f && (dims & 3) == 0 && (((uintptr_t)o | (uintptr_t)partial) & 15) == 0) {
            sum_partials_l2n_kernel<<<nb, 256, 0, st>>>(partial, ks_eff, split_stride, dims, renorm_eps, o);
        } else if (renorm_eps >= 0.f) {
            sum_partials_kernel<<<(unsigned)((split_stride / 4 + 256) / 256), 256, 0, st>>>(partial, ks_eff, split_stride, split_stride, o);
            MDIR_LAUNCH_CHECK();
            row_l2n_kernel<<<nb, 256, 0, st>>>(o, dims, renorm_eps);
        } else {
            sum_partials_kernel<<<(unsigned)((split_stride / 4 + 256) / 256), 256, 0, st>>>(partial, ks_eff, split_stride, split_stride, o);
        }
        MDIR_LAUNCH_CHECK();
    }
    if (conc > 1) {
        MDIR_CUDA(cudaEventRecord(ev_join, side));
        MDIR_CUDA(cudaStreamWaitEvent(main_st, ev_join, 0));
    }
    return 0;
}
