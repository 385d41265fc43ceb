// One-call composites over the component launchers: what a host language binds when it wants "the head" or "the
// top-k" as a single entry point (SURVEY.md section 8b, C-ABI face: mdir_gem_head, mdir_sim_topk_bf16).  Pure host
// code: planning + a chain of the extern "C" launchers of this library on the caller's stream; no allocation, no
// synchronisation, every scratch buffer comes out of the caller's workspace.
#include "common.cuh"

namespace mdir {

constexpr int kTile = MDIR_SCAN_TILE_ROWS;
constexpr int kMaxQ = 128;
constexpr int kCapS = 8192;                          // segment 0 (select kernel) capacity, three-launch / dense routes
constexpr int kCapL = 96;                            // per-CTA segment capacity, three-launch route
constexpr int64_t kCandRow = kCapS + 148 * (int64_t)kCapL;
constexpr int kFusedCapL = (int)(kCandRow / 148);    // one-launch route: the whole row shared by the CTA segments
constexpr int kMaxSampleTiles = 512;
constexpr int kTargetCand = 4500;
constexpr int64_t kDenseRowsMax = (int64_t)kMaxSampleTiles * kTile;      // the score region holds 128 x this many floats

static size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

struct TopkWs {
    uint16_t* q16;
    uint64_t* tau;
    uint32_t* segcnt;
    uint8_t* fused;
    uint64_t* cand;
    float* scores;
    size_t total;
};

static TopkWs topk_layout(void* ws, int D) {
    TopkWs w;
    uint8_t* p = reinterpret_cast<uint8_t*>(align256(reinterpret_cast<size_t>(ws)));
    const uint8_t* p0 = reinterpret_cast<const uint8_t*>(ws);
    w.q16 = reinterpret_cast<uint16_t*>(p);      p += align256((size_t)kMaxQ * D * 2);
    w.tau = reinterpret_cast<uint64_t*>(p);      p += align256((size_t)kMaxQ * 8);
    w.segcnt = reinterpret_cast<uint32_t*>(p);   p += align256((size_t)kMaxQ * MDIR_CAND_SEGS * 4);
    w.fused = p;                                 p += align256(mdir_sim_scan_fused_workspace_bytes(kMaxQ));
    w.cand = reinterpret_cast<uint64_t*>(p);     p += align256((size_t)kMaxQ * kCandRow * 8);
    w.scores = reinterpret_cast<float*>(p);      p += align256((size_t)kMaxQ * kDenseRowsMax * 4);
    w.total = (size_t)(p - p0);
    return w;
}

// 1.25 k rounded up to a multiple of 64 (whole rounds of the 2 x 32 re-scoring warps); the certified extension
// of mdir_topk_finalize_rescore adds whatever else is needed.  Same rule as mdir_b200/search.py:default_shortlist.
static int default_shortlist(int k) {
    const int b = (5 * k + 3) / 4;
    return (b + 63) / 64 * 64;
}

}  // namespace mdir

using namespace mdir;

extern "C" size_t mdir_sim_topk_workspace_bytes(int D) {
    if (D <= 0) return 0;
    return topk_layout(nullptr, D).total + 256;
}

// Host-only: which route a top-k over n_db rows with selection depth kth takes on a device with sm_count SMs.
// route 0 = dense (every score, exact select), 1 = one-launch threshold + filter scan, 2 = sample / select / filter.
// n_sample / stride = the three-launch sampling plan (n_sample tiles at that stride), reported on routes 1 and 2: a
// caller that may not take the one-launch route (more than 128 queries, or the route disabled) falls back to it.  Zero
// only when no three-launch plan exists (route 0).  No CUDA call.
extern "C" int mdir_topk_plan(int64_t n_db, int kth, int sm_count, int* route, int* n_sample, int* stride) {
    MDIR_CHECK_ARG(route && n_sample && stride && n_db >= 0 && kth >= 1 && sm_count >= 1);
    *route = 0;
    *n_sample = 0;
    *stride = 0;
    const int64_t n_tiles = (n_db + kTile - 1) / kTile;
    if (n_tiles < 64) return 0;
    int64_t want = ((int64_t)kth * n_tiles + kTargetCand - 1) / kTargetCand;
    if (want > 148) want = (want + 147) / 148 * 148;
    int64_t ns = want < n_tiles / 4 ? want : n_tiles / 4;
    if (ns > kMaxSampleTiles) ns = kMaxSampleTiles;
    if (ns < 32) ns = 32;
    const int64_t st = n_tiles / ns;
    if (ns * kTile >= 2 * (int64_t)kth && st >= 2) {
        *route = 2;
        *n_sample = (int)ns;
        *stride = (int)st;
    }
    int64_t g = sm_count < 148 ? sm_count : 148;
    if (g > n_tiles / 2) g = n_tiles / 2;
    g = balanced_grid(n_tiles, (int)g);          // the grid mdir_sim_scan_fused_bf16 launches
    if (g * 16 >= 2 * (int64_t)kth && 1.25 * kth * (double)n_tiles / ((double)g * (double)g) <= kFusedCapL / 2.0) *route = 1;
    return 0;
}

extern "C" int mdir_sim_topk_bf16(const uint16_t* db16, const float* db32, const float* db_stats, int64_t n_db, const float* q32, int n_q, int D, int k, int shortlist,
                                  uint32_t idx_base, int route, float* out_scores, int32_t* out_idx, uint64_t* out_keys, int32_t* overflow,
                                  void* ws, void* stream) {
    MDIR_CHECK_ARG(db16 && q32 && ws && out_scores && out_idx && overflow);
    MDIR_CHECK_ARG(n_q >= 0 && n_q <= kMaxQ && D >= 8 && (D % 8) == 0 && k >= 1 && n_db >= k && route >= 0 && route <= 1);
    if (n_q == 0) return 0;
    int kth = k;
    if (db32) {
        int64_t s = shortlist > 0 ? shortlist : default_shortlist(k);
        if (s > n_db) s = n_db;
        if (s > kth) kth = (int)s;
    }
    MDIR_CHECK_ARG(kth <= 4096);
    const TopkWs w = topk_layout(ws, D);
    int rc = mdir_pack_bf16(q32, n_q, D, 0, w.q16, stream);
    if (rc) return rc;
    const int64_t n_tiles = (n_db + kTile - 1) / kTile;

    // route planning: the planner Index.search uses too (search.py:Index._route); only route 2 reads the sampling plan
    const int sm_count = device_sm_count();
    MDIR_CHECK_ARG(sm_count > 0);
    int plan_route = 0, n_sample = 0, stride = 0;
    if (route == 0) mdir_topk_plan(n_db, kth, sm_count, &plan_route, &n_sample, &stride);
    const bool fused = plan_route == 1;
    if (plan_route != 2) n_sample = 0;
    int cap0 = kCapS, cap_l = kCapL;
    if (fused) {
        MDIR_CUDA(cudaMemsetAsync(w.fused, 0, 16, (cudaStream_t)stream));       // the kernel's arrival counters
        rc = mdir_sim_scan_fused_bf16(db16, n_db, w.q16, n_q, D, kth, w.tau, idx_base, w.cand, w.segcnt, 0, kFusedCapL, w.fused, stream);
        if (rc) return rc;
        cap0 = 0;
        cap_l = kFusedCapL;
    } else if (n_sample > 0) {
        const int64_t ld = kDenseRowsMax, rows = (int64_t)n_sample * kTile;
        rc = mdir_sim_scan_bf16(db16, n_db, w.q16, n_q, D, MDIR_SCAN_SAMPLE, stride, n_sample, w.scores, ld, nullptr, 0, nullptr, nullptr, 0, 0,
                                stream);
        if (rc) return rc;
        rc = mdir_select_kth(w.scores, ld, rows, n_q, kth, stride, idx_base, w.tau, w.cand, kCandRow, w.segcnt, MDIR_CAND_SEGS, kCapS, 1, stream);
        if (rc) return rc;
        rc = mdir_sim_scan_bf16(db16, n_db, w.q16, n_q, D, MDIR_SCAN_FILTER, stride, n_sample, nullptr, 0, w.tau, idx_base, w.cand, w.segcnt,
                                kCapS, kCapL, stream);
        if (rc) return rc;
    } else {
        // dense route: every score, exact kth-key select (emits exactly kth keys: cannot overflow).  Small databases
        // and the recovery after an overflow; limited by the score region of the workspace.
        MDIR_CHECK_ARG(n_db <= kDenseRowsMax);
        rc = mdir_sim_scan_bf16(db16, n_db, w.q16, n_q, D, MDIR_SCAN_DENSE, 0, 0, w.scores, n_db, nullptr, 0, nullptr, nullptr, 0, 0, stream);
        if (rc) return rc;
        rc = mdir_select_kth(w.scores, n_db, n_db, n_q, kth, 0, idx_base, w.tau, w.cand, kCandRow, w.segcnt, MDIR_CAND_SEGS, kCapS, 0, stream);
        if (rc) return rc;
    }
    const int64_t cand_row = cap0 + 148 * (int64_t)cap_l;
    if (db32)
        return mdir_topk_finalize_rescore(w.cand, cand_row, w.segcnt, MDIR_CAND_SEGS, cap0, cap_l, n_q, kth, k, db32, n_db, idx_base, q32, D,
                                          db_stats, out_scores, out_idx, out_keys, w.tau, overflow, stream);
    return mdir_topk_finalize(w.cand, cand_row, w.segcnt, MDIR_CAND_SEGS, cap0, cap_l, n_q, k, out_scores, out_idx, out_keys, w.tau, overflow,
                              stream);
}

extern "C" size_t mdir_gem_head_workspace_bytes(int n_img, int S, int C, int dims) {
    if (n_img <= 0 || S <= 0 || C <= 0) return 0;
    size_t b = align256((size_t)n_img * S * C * 4) + align256((size_t)n_img * C * 4) + 512;
    if (dims > 0) b += align256(mdir_whiten_tc_workspace_bytes(n_img, C, dims));
    return b;
}

extern "C" int mdir_gem_head(int kind, const float* x, const int64_t* off, const int32_t* hw, int n_img, int S, int C, int hw_uniform, float p,
                             float eps, float msp, const float* m, const float* P, const float* Px3, int dims, float* out, void* ws,
                             void* stream) {
    MDIR_CHECK_ARG(x && out && ws && n_img >= 0 && S >= 1 && C >= 1);
    MDIR_CHECK_ARG((P == nullptr && Px3 == nullptr) || dims >= 1);
    if (n_img == 0) return 0;
    uint8_t* b = reinterpret_cast<uint8_t*>(align256(reinterpret_cast<size_t>(ws)));
    float* pooled = reinterpret_cast<float*>(b);
    b += align256((size_t)n_img * S * C * 4);
    const bool whiten = P != nullptr || Px3 != nullptr;
    float* agg = whiten ? reinterpret_cast<float*>(b) : out;
    b += align256((size_t)n_img * C * 4);
    int rc = mdir_pool(kind, x, off, hw, n_img * S, C, hw_uniform, p, eps, pooled, stream);
    if (rc) return rc;
    // L2N's eps and the +1e-6 of the Lw renormalisation are constants of the reference (normalization.py:12, wrapper.py:195)
    rc = mdir_ms_aggregate(pooled, n_img, S, C, 1e-6f, msp, nullptr, agg, stream);
    if (rc || !whiten) return rc;
    if (Px3 != nullptr && n_img > 4 && (C % 4) == 0) return mdir_whiten_project_tc(agg, m, n_img, C, Px3, dims, 1e-6f, out, b, stream);
    MDIR_CHECK_ARG(P != nullptr);
    return mdir_whiten_project(agg, m, n_img, C, P, dims, 1e-6f, out, stream);
}
