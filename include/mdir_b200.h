/*
 * mdir_b200.h -- C ABI of libmdir_b200.so: hand-written sm_100a kernels for the
 * post-backbone retrieval hot path of jenicek/mdir (SURVEY.md section 8).
 *
 * The reference is pure Python and has NO FFI; its plug-in mechanism is four dict
 * registries (SURVEY.md 8b).  Every entry point below therefore cites the
 * reference Python call it replaces (file:line relative to the reference root);
 * INTEGRATION.md shows the ctypes stub a maintainer would add on the reference
 * side.  Conventions: plain device pointers + sizes + a cudaStream_t passed as
 * void*; no allocation, no synchronisation, no torch types; every function
 * returns 0 on success, a positive cudaError_t, or a negative MDIR_E_* code, and
 * mdir_last_error() describes the last failure on the calling thread.
 */
#ifndef MDIR_B200_H
#define MDIR_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MDIR_ABI_VERSION 2

#define MDIR_E_ARG      (-1)   /* invalid argument (shape/alignment/range) */
#define MDIR_E_DRIVER   (-2)   /* driver entry point (cuTensorMapEncodeTiled) unavailable */
#define MDIR_E_DEVICE   (-3)   /* not an sm_100 device */

int         mdir_abi_version(void);
const char* mdir_last_error(void);
/* 0 when the current device is compute capability 10.x with >= 148 SMs usable. */
int         mdir_device_check(void);
/* number of kernels this library has launched in this process (for bench accounting) */
uint64_t    mdir_launch_count(void);

/* Process-wide SM-partitioning knobs, read at launch time (so a value set around a CUDA-graph capture is baked into
 * that graph): MDIR_TUNE_SCAN_MAX_CTAS caps the persistent grid of mdir_sim_scan_fused_bf16 (0 = all SMs),
 * MDIR_TUNE_FINALIZE_CLUSTER = 0 keeps mdir_topk_finalize_rescore on single CTAs.  A serving pipeline that runs the
 * finalize + exchange of step t beside the scan of step t + 1 uses both so that the two kernels fit at once.        */
#define MDIR_TUNE_SCAN_MAX_CTAS 1
#define MDIR_TUNE_FINALIZE_CLUSTER 2
#define MDIR_TUNE_FINALIZE_STAGE_CAP 3   /* keys staged per query by finalize (0 = everything the segments can hold); more -> overflow bit */
int         mdir_tune(int key, int value);

/* ---------------------------------------------------------------- pooling ---
 * kind: 0 = GeM, 1 = MAC, 2 = SPoC.
 * Replaces LF.gem / LF.mac / LF.spoc
 *   (mdir/external/cirtorch/layers/functional.py:11-22) called by
 *   GeM/MAC/SPoC.forward (mdir/external/cirtorch/layers/pooling.py:12-47).
 * x holds n_maps feature maps; map i is C contiguous planes of hw[i] floats
 * starting at x + off[i] (floats).  off/hw are DEVICE arrays; both NULL means a
 * uniform (n_maps, C, hw_uniform) NCHW batch.  out: (n_maps, C) fp32.         */
#define MDIR_POOL_GEM  0
#define MDIR_POOL_MAC  1
#define MDIR_POOL_SPOC 2
int mdir_pool(int kind, const float* x, const int64_t* off, const int32_t* hw,
              int n_maps, int C, int hw_uniform, float p, float eps,
              float* out, void* stream);

/* L2N over dim=1 of an (N, C, inner) tensor: x / (||x||_2 + eps)
 * Replaces LF.l2n (cirtorch/layers/functional.py:130-131).                    */
int mdir_l2n(const float* x, int N, int C, int inner, float eps, float* out, void* stream);

/* Per image: L2N each of S pooled vectors (eps added to the norm), then
 * v = (sum_s o_s^msp / S)^(1/msp); v /= ||v|| (no eps); optionally v -= m.
 * Replaces ImageRetrievalNet.forward's norm(pool(o)) (cirtorch/networks/
 * imageretrievalnet.py:107) + CirMultiscaleAggregation.aggregate_tensor
 * (mdir/components/data/wrapper.py:109-119) + the centring of
 * CirtorchWhiten.postprocess (wrapper.py:194).
 * pooled: (n_img, S, C); m: (C) or NULL; out: (n_img, C).
 * l2n_eps < 0 means the S vectors are already L2-normalised (skip that step). */
int mdir_ms_aggregate(const float* pooled, int n_img, int S, int C, float l2n_eps,
                      float msp, const float* m, float* out, void* stream);

/* out[n, j] = sum_d P[j, d] * (v[n, d] - m[d]) for j < dims, then (optionally)
 * out[n, :] /= (||out[n, :]||_2 + renorm_eps)  when renorm_eps >= 0.
 * Replaces CirtorchWhiten.postprocess (wrapper.py:193-195) and, batched,
 * whitenapply (mdir/external/cirtorch/utils/whiten.py:4-12).
 * v: (n, D); m: (D) or NULL; P: (>=dims, D) row-major fp32; out: (n, dims).   */
int mdir_whiten_project(const float* v, const float* m, int n, int D, const float* P, int dims,
                        float renorm_eps, float* out, void* stream);

/* The same projection on the tensor cores (3xTF32 = fp32-faithful) for batches: Px3 is
 * mdir_split_tf32x3(P[:dims_total], role 0) = (dims_total, 3D) fp32, built once per Lw.
 * ws: mdir_whiten_tc_workspace_bytes(n, D, dims) bytes.  D % 4 == 0.                 */
size_t mdir_whiten_tc_workspace_bytes(int n, int D, int dims);
int mdir_whiten_project_tc(const float* v, const float* m, int n, int D, const float* Px3, int dims,
                           float renorm_eps, float* out, void* ws, void* stream);

/* ------------------------------------------------------------------ CLAHE ---
 * Bit-exact cv2.createCLAHE(clipLimit=clip, tileGridSize=(tiles_x,tiles_y)).apply
 * on a batch of ragged 8UC1 images.  Replaces ChannelClahe.apply's cv2 call
 * (mdir/components/data/transform/functional.py:109-117).
 * descs: DEVICE array of n_img descriptors (byte offsets into src/dst).
 * ws: device workspace of mdir_clahe_workspace_bytes() bytes (the per-tile LUTs). */
typedef struct {
    int64_t src_off;    /* byte offset of pixel (0,0) in src */
    int64_t dst_off;    /* byte offset of pixel (0,0) in dst */
    int32_t H, W;
    int32_t src_pitch;  /* bytes between rows */
    int32_t dst_pitch;
} mdir_image_desc;
size_t mdir_clahe_workspace_bytes(int n_img, int tiles_x, int tiles_y);
int mdir_clahe_u8(const uint8_t* src, uint8_t* dst, const mdir_image_desc* descs,
                  int n_img, int max_H, int max_W, double clip, int tiles_x, int tiles_y,
                  void* ws, void* stream);

/* RGB <-> Lab around CLAHE on the device, following OpenCV's float code path as the reference
 * calls it (rgb2normspace / normspace2rgb, mdir/components/data/transform/functional.py:24-48,
 * ImageClahe.apply :120-129).  Images are contiguous HWC float32 in [0,1]; descs is a DEVICE array.
 *   lut       (33,33,33,4) int16: OpenCV's RGB2Lab interpolation lattice {L,a,b,0} (LAB_BASE 2^14)
 *   gamma_tab (1024,4) fp32: cubic-spline coefficients of the sRGB gamma (Lab2RGBfloat)
 * mdir_rgb_to_l_u8:      L plane as uint8 = trunc((L/100)*255)   -> feed to mdir_clahe_u8
 * mdir_lab_clahe_to_rgb: (a, b of the original pixel) + CLAHE'd uint8 L -> RGB float32 HWC       */
typedef struct {
    int64_t rgb_off;   /* float offset of pixel (0,0) in the rgb INPUT buffer */
    int64_t out_off;   /* float offset of pixel (0,0) in the rgb OUTPUT buffer of mdir_lab_clahe_to_rgb */
    int64_t l_off;     /* byte offset of the image's L plane in the uint8 L buffers */
    int32_t H, W;
} mdir_rgb_desc;
int mdir_rgb_to_l_u8(const float* rgb, const mdir_rgb_desc* descs, int n_img, int64_t max_pixels,
                     const int16_t* lut, uint8_t* l_out, void* stream);
int mdir_lab_clahe_to_rgb(const float* rgb, const mdir_rgb_desc* descs, int n_img, int64_t max_pixels,
                          const int16_t* lut, const float* gamma_tab, const uint8_t* l_in, float* out,
                          void* stream);

/* ------------------------------------------------------- similarity search ---
 * Replaces np.dot(vecs.T, qvecs) + np.argsort(-scores, axis=0)
 * (mdir/components/optim/score/cirscore.py:69-70).
 *
 * Descriptor matrices on the device are ROW-major (n, D) bf16 ("K-major"), D % 8
 * == 0.  mdir_pack_bf16 converts from fp32, optionally from the reference's
 * (D, n) column-per-image layout (cirtorch/networks/imageretrievalnet.py:291).  */
int mdir_pack_bf16(const float* src, int64_t n, int D, int src_is_Dxn, uint16_t* dst, void* stream);

/* One streaming pass of the database against <= 256 resident queries on
 * tcgen05/TMEM tiles fed by TMA (256 db rows per tile, fp32 accumulate).  Up to 128 queries the TMEM
 * accumulators are double / triple buffered (the HBM-bound serving shapes); 129..256 queries use all 512 TMEM
 * columns for one tile: arithmetic intensity = n_q FLOP per database byte, above the ~214 FLOP/B ridge of this part,
 * i.e. the tensor-bound shapes (database-side augmentation, all-pairs scores).
 *   mode MDIR_SCAN_DENSE   : write every score, out[q * dense_ld + row]
 *   mode MDIR_SCAN_SAMPLE  : only tiles t = j*sample_stride (j < n_sample), written
 *                            compactly: out[q * dense_ld + j*256 + r]
 *   mode MDIR_SCAN_FILTER  : all tiles EXCEPT the sample tiles (n_sample may be 0);
 *                            a score is appended to the query's candidates iff its 64-bit
 *                            key (mdir key order: score desc, index asc) <= tau[q].
 * Candidate storage (no global atomics: every producer owns a segment):
 *   cand       (n_q, cap_s + 148*cap_l) u64 keys; per query, segment 0 = [0, cap_s) belongs
 *              to mdir_select_kth, segment 1+c = [cap_s + c*cap_l, +cap_l) to scan CTA c
 *   seg_counts (n_q, MDIR_CAND_SEGS) u32: how many keys each producer appended (may exceed
 *              the segment capacity: the surplus was dropped, mdir_topk_finalize reports
 *              overflow and a tightened tau, and the caller re-scans).  Caller zeroes it.
 * Keys carry idx_base + row so shards emit global indices.                      */
#define MDIR_SCAN_DENSE  0
#define MDIR_SCAN_SAMPLE 1
#define MDIR_SCAN_FILTER 2
#define MDIR_SCAN_TILE_ROWS 256
#define MDIR_CAND_SEGS 149
int mdir_sim_scan_bf16(const uint16_t* db, int64_t n_db, const uint16_t* q, int n_q, int D,
                       int mode, int sample_stride, int n_sample,
                       float* dense_out, int64_t dense_ld,
                       const uint64_t* tau, uint32_t idx_base,
                       uint64_t* cand, uint32_t* seg_counts, int cap_s, int cap_l, void* stream);

/* Dense bf16 scores of ANY number of queries in one launch: out (n_q, n_db) fp32 query-major with pitch dense_ld
 * (np.dot(vecs.T, qvecs).T, cirscore.py:69).  Work items are (256-row tile, 128-query block) pairs, the blocks of a
 * tile adjacent in the persistent round-robin, so the database is streamed from HBM once and the kernel ramps up once
 * instead of once per 128 queries (the all-pairs / full-ranks shapes, BASELINE config C3).                          */
int mdir_sim_scan_dense_bf16(const uint16_t* db, int64_t n_db, const uint16_t* q, int n_q, int D,
                             float* dense_out, int64_t dense_ld, void* stream);

/* mdir_sim_scan_bf16 for more than 128 queries in ONE launch (SAMPLE / FILTER: up to 1,024; DENSE: any number): work
 * items are (tile, 128-query block) pairs, so a database tile is read from HBM once for all its query blocks and the
 * scan of a large query batch (DBA, all-pairs ranking) becomes tensor-bound.  tau, cand, seg_counts, dense_out are
 * indexed by the query's position in q exactly as for mdir_sim_scan_bf16; results are bit-identical to per-block launches. */
int mdir_sim_scan_wide_bf16(const uint16_t* db, int64_t n_db, const uint16_t* q, int n_q, int D, int mode,
                            int sample_stride, int n_sample, float* dense_out, int64_t dense_ld,
                            const uint64_t* tau, uint32_t idx_base, uint64_t* cand, uint32_t* seg_counts,
                            int cap_s, int cap_l, void* stream);

/* Threshold + filter in ONE launch (the large-database route of the top-k search; replaces the
 * SAMPLE scan -> mdir_select_kth -> FILTER scan chain and its two extra launches).  Every
 * persistent CTA first scans one sample tile (tiles c * (n_tiles / grid)), publishes the two best
 * keys of each of its eight 32-row groups, and after a grid-wide arrival counter CTA q selects the
 * kth smallest of query q's grid*16 values: a valid threshold, because those values are keys of
 * kth distinct rows.  After a second arrival counter every CTA filters its sample tile (still in
 * TMEM) and then the rest of the database exactly like MDIR_SCAN_FILTER.  Writes tau[q], the
 * candidate segments 1.. and ALL n_q * MDIR_CAND_SEGS segment counters (segment 0 stays empty).
 * ws: mdir_sim_scan_fused_workspace_bytes(n_q) bytes, 16-byte aligned, ZEROED ONCE by the caller
 * before first use (the kernel re-arms its counters itself).  Needs n_db >= 512 rows.  The launch is
 * COOPERATIVE (cudaLaunchAttributeCooperative): the runtime guarantees the grid's co-residency, which
 * the in-kernel rendezvous needs, or fails the launch; should an arrival counter still not be
 * reached within ~4 s the segments report overflow instead of hanging.                        */
size_t mdir_sim_scan_fused_workspace_bytes(int n_q);
int mdir_sim_scan_fused_bf16(const uint16_t* db, int64_t n_db, const uint16_t* q, int n_q, int D,
                             int kth, uint64_t* tau, uint32_t idx_base,
                             uint64_t* cand, uint32_t* seg_counts, int cap_s, int cap_l,
                             void* ws, void* stream);

/* mdir_sim_scan_fused_bf16 with int8 operands (tcgen05 kind::i8, s32 accumulate): the first pass of the
 * certified fp32 search reads n_db * D + 4 n_db bytes instead of 2 n_db * D.  db8 (n_db, D) int8 rows and
 * row_scale[n_db] from mdir_pack_stats_i8; q8 / q_scale from mdir_pack_q_i8 (two int8 planes per query).
 * Filter score = row_scale[r] * (s_hi * <x8_r, hi> + s_lo * <x8_r, lo>) in fp32; keys, segments and
 * counters exactly as mdir_sim_scan_fused_bf16.  D % 128 == 0, n_q <= 128.                  */
int mdir_sim_scan_fused_i8(const int8_t* db8, const float* row_scale, int64_t n_db, const int8_t* q8,
                           const float* q_scale, int n_q, int D, int kth, uint64_t* tau, uint32_t idx_base,
                           uint64_t* cand, uint32_t* seg_counts, int cap_s, int cap_l,
                           void* ws, void* stream);

/* The same scan with fp32 operands consumed as TF32 (tcgen05 kind::tf32, fp32 accumulate):
 * db (n_db, D) and q (n_q, D) row-major fp32, D % 4 == 0.  Used directly it is the TF32
 * similarity variant; fed the (n, 3D) matrices written by mdir_split_tf32x3 (role 0 for the
 * database side, role 1 for the query side) it computes hi*hi + hi*lo + lo*hi = an
 * fp32-faithful ("3xTF32") dot product.                                              */
int mdir_sim_scan_tf32(const float* db, int64_t n_db, const float* q, int n_q, int D,
                       int mode, int sample_stride, int n_sample,
                       float* dense_out, int64_t dense_ld,
                       const uint64_t* tau, uint32_t idx_base,
                       uint64_t* cand, uint32_t* seg_counts, int cap_s, int cap_l, void* stream);
int mdir_split_tf32x3(const float* src, int64_t n, int D, int role, float* dst, void* stream);

/* key helpers exposed for tests: key = (~orderable(score) << 32) | index        */
uint64_t mdir_make_key(float score, uint32_t index);
float    mdir_key_score(uint64_t key);

/* For each query: radix-select the kth best (score desc, index asc) key among
 * scores[q*ld + i], i < n, and set tau[q] to it (exactly kth rows have key <= tau).
 * The index part of a key = pos_to_idx(i): i itself, or for a compact sample
 * ((i/256)*sample_stride)*256 + i%256, plus idx_base.  When cand != NULL the kth items
 * with key <= tau are written to segment 0 of the query's cand row (row pitch cand_row
 * keys, capacity cap), seg_counts[q*n_seg + 0] is set to their number and the other
 * n_seg - 1 counters of the query are zeroed (ready for the FILTER scan that follows).
 * approx != 0 relaxes tau to any valid upper bound of the kth key (>= kth rows pass, typically
 * a few % more): enough for a filter threshold and about half the work.               */
int mdir_select_kth(const float* scores, int64_t ld, int64_t n, int n_q, int kth,
                    int sample_stride, uint32_t idx_base,
                    uint64_t* tau, uint64_t* cand, int64_t cand_row, uint32_t* seg_counts, int n_seg,
                    int cap, int approx, void* stream);

/* For each query: gather the candidate keys of its n_seg segments (segment 0 holds up to
 * cap0 keys, the others cap_l each), emit the best k as (score fp32, index int32) rows of
 * out_*(n_q, k) (padded with -inf / -1), and set overflow[q] = 1 and tau[q] = kth key of
 * what was kept when a segment (or the 16384-key staging area) overflowed.
 * Also the shard merge and the post-rescoring sort: n_seg = 1, cap0 = keys per query.  */
int mdir_topk_finalize(const uint64_t* cand, int64_t cand_row, const uint32_t* seg_counts, int n_seg,
                       int cap0, int cap_l, int n_q, int k,
                       float* out_scores, int32_t* out_idx, uint64_t* out_keys,
                       uint64_t* tau, int32_t* overflow, void* stream);

/* mdir_topk_finalize + exact fp32 re-scoring fused: selects the `shortlist` best keys (bf16
 * scores), recomputes their dot products in fp32 from db32 (rows idx - idx_base of this shard)
 * against q32[q], re-sorts and emits the best k_out (out_* are (n_q, k_out)).
 * Shortlist CERTIFICATE (db_stats != NULL, then tau != NULL): with t = the k_out-th best fp32
 * score and eps = a Cauchy-Schwarz bound on |bf16-path score - fp32 score| over the whole shard
 * (from db_stats = mdir_pack_stats output and the query's own rounding residual), every candidate
 * whose bf16 score is >= t - eps is re-scored as well, and status bit 1 is raised unless the
 * candidate list provably holds all such rows (tau[q] not tighter than t - eps, no overflow):
 * a clear status means the emitted rows ARE the exact fp32 top k_out of the shard.
 * overflow[q] is a status word: bit 0 = a segment / the staging area overflowed (re-scan),
 * bit 1 = not certified (widen the selection: larger shortlist, eventually the dense route). */
int mdir_topk_finalize_rescore(const uint64_t* cand, int64_t cand_row, const uint32_t* seg_counts, int n_seg,
                               int cap0, int cap_l, int n_q, int shortlist, int k_out,
                               const float* db32, int64_t n_db, uint32_t idx_base, const float* q32, int D,
                               const float* db_stats,
                               float* out_scores, int32_t* out_idx, uint64_t* out_keys,
                               uint64_t* tau, int32_t* overflow, void* stream);
/* mdir_topk_finalize_rescore for filter scores of another encoding (mdir_sim_scan_fused_i8): q_eps[q]
 * (mdir_pack_q_i8) is that encoding's bound for query q, used instead of the bf16 one; db_stats must
 * still be given.  The extension area grows with the shard (0.2 % of n_db rows, 256 .. 2,048 keys).  */
int mdir_topk_finalize_rescore_eps(const uint64_t* cand, int64_t cand_row, const uint32_t* seg_counts, int n_seg,
                                   int cap0, int cap_l, int n_q, int shortlist, int k_out,
                                   const float* db32, int64_t n_db, uint32_t idx_base, const float* q32, int D,
                                   const float* db_stats, const float* q_eps,
                                   float* out_scores, int32_t* out_idx, uint64_t* out_keys,
                                   uint64_t* tau, int32_t* overflow, void* stream);
#define MDIR_STATUS_OVERFLOW    1
#define MDIR_STATUS_UNCERTIFIED 2

/* stats[2] (device) = {max_r ||bf16(x_r) - x_r||_2^2, max_r ||x_r||_2^2} over the n rows of a shard:
 * the database half of the certificate's error bound.  db16 = mdir_pack_bf16(db32).            */
int mdir_pack_stats(const float* db32, const uint16_t* db16, int64_t n, int D, float* stats, void* stream);

/* mdir_pack_stats plus, in the same pass, the int8 plane of the shard: db8 (n, D) with a symmetric
 * per-row scale row_scale[r] = max_i |x_ri| / 127 (x8 = rint(x / s_r), round half even), and
 * stats[4] = {the two above, max_r ||x_r - s_r x8_r||^2, max_r ||x_r - s_r x8_r||^2 / ||x_r||^2}.
 * D % 128 == 0; db32 and db8 16-byte aligned.                                               */
int mdir_pack_stats_i8(const float* db32, const uint16_t* db16, int64_t n, int D, float* stats,
                       int8_t* db8, float* row_scale, void* stream);

/* The query operand of mdir_sim_scan_fused_i8 and its certificate bound, one launch: q8 (2 n_pad, D),
 * n_pad = n_q rounded up to 16, rows [0, n_pad) = hi = rint(q / s_hi), rows [n_pad, 2 n_pad) =
 * lo = rint((q - s_hi hi) / s_lo) (padding rows zero), s_hi = max|q| / 127, s_lo = max|q - s_hi hi| / 127,
 * q_scale (n_q, 2) = {s_hi, s_lo}; q_eps[n_q] = the bound on |int8-path score - fp32 score| over every
 * row of the shard described by stats (mdir_pack_stats_i8).  n_q <= 128, D % 128 == 0.        */
int mdir_pack_q_i8(const float* q32, int n_q, int D, const float* stats, int8_t* q8, float* q_scale,
                   float* q_eps, void* stream);

/* Exact fp32 re-scoring of a shortlist: out[q, j] = <db32[idx[q,j]-idx_base], q32[q]>
 * (idx < 0 or outside this shard -> -inf); then callers re-finalize.             */
int mdir_rescore_f32(const float* db32, int64_t n_db, uint32_t idx_base, const float* q32, int n_q, int D,
                     const int32_t* idx, int kk, uint64_t* out_keys, void* stream);

/* alpha query expansion / database-side augmentation.  NOT in the reference (SURVEY.md
 * App. E; parity unpinned): acc[q, :] = sum_j max(scores[q,j], 0)^alpha * db32[idx[q,j] -
 * idx_base, :] over the shortlist entries this shard owns (others contribute 0, so shards
 * combine with an all-reduce);  mdir_add_l2n: out = (a + b) / ||a + b||, b may be NULL.   */
int mdir_qe_accumulate(const float* db32, int64_t n_db, uint32_t idx_base, int D, const int32_t* idx,
                       const float* scores, int n_q, int n_qe, float alpha, float* acc, void* stream);
int mdir_add_l2n(const float* a, const float* b, int n, int D, float* out, void* stream);

/* Full per-query ranking of a score matrix given in the REFERENCE layout
 * scores (n_db, n_q) fp32 C-order -> ranks (n_db, n_q) int64 C-order, identical to
 * np.argsort(-scores, axis=0, kind='stable') (cirscore.py:70; ties by ascending
 * index).  query_major != 0 means scores is already (n_q, n_db).  ranks_ld >= n_q is
 * the row pitch of ranks in elements (lets callers fill a column block of a wider array).
 * ws: mdir_rank_workspace_bytes() bytes.                                         */
size_t mdir_rank_workspace_bytes(int64_t n_db, int n_q);
int mdir_rank_scores(const float* scores, int64_t n_db, int n_q, int query_major,
                     int64_t* ranks, int64_t ranks_ld, void* ws, void* stream);

/* The same result through a sample sort: per query ONE data-adaptive partition pass into buckets of <= 2048 pairs
 * (splitters = every 32nd of a sorted systematic sample of (score key, row) composites, so ties cannot unbalance
 * them; every bucket owns a 2048-slot region, so no counting pass) and one shared-memory interpolation counting sort per
 * bucket -- ~36 B of HBM traffic per pair instead of ~100 B for the four radix passes.  *status (device int32) is
 * cleared first and set non-zero when a bucket overflowed its region: ranks is then incomplete and the caller re-runs
 * mdir_rank_scores.  Segments longer than 196,608 rows take the radix path directly.
 * ws: mdir_rank_fast_workspace_bytes() bytes.                                                                      */
size_t mdir_rank_fast_workspace_bytes(int64_t n_db, int n_q);
int mdir_rank_scores_fast(const float* scores, int64_t n_db, int n_q, int query_major,
                          int64_t* ranks, int64_t ranks_ld, void* ws, int32_t* status, void* stream);

/* The same result through a histogram sort, the fastest route for smooth score populations (1,025 .. 131,072 rows per
 * query; other lengths are forwarded to mdir_rank_scores_fast): per query an exact 4096-cell histogram linear in the
 * score over mean +- 4 sigma gives a cell -> bucket table and the exact offset of every bucket (runs of whole cells of
 * ~2,048 rows); one scatter pass (bucket = one table lookup per row) fills a compact pair array; one CTA per bucket
 * finishes with an interpolation counting sort in shared memory; a 64 x 64 tiled transpose writes the int64 ranks.
 * *status (device int32) is cleared first; bit 1 (value 2) is set when some query has a bucket of more than 4,096 rows
 * (massive ties, spikes): ranks is then incomplete and the caller re-runs mdir_rank_scores_fast (bit 0, value 1, keeps
 * its meaning when the call was forwarded).  ws: mdir_rank_hist_workspace_bytes() bytes.                            */
size_t mdir_rank_hist_workspace_bytes(int64_t n_db, int n_q);
int mdir_rank_scores_hist(const float* scores, int64_t n_db, int n_q, int query_major,
                          int64_t* ranks, int64_t ranks_ld, void* ws, int32_t* status, void* stream);

/* ------------------------------------------------------------------- mAP ---
 * Average precision and precision@kappa per query from the ranks array, on the device.
 * Replaces compute_ap / compute_map (mdir/external/cirtorch/utils/evaluate.py:3-111).
 * ranks: (n_db, n_q) int64 C-order.  The ground truth arrives flattened: items[i] is a db index
 * that is positive (item_class 0, "ok") or junk (item_class 1) for query item_query[i];
 * n_pos[q] = len(gnd[q]['ok']) (0 -> AP = NaN, excluded by the caller as in evaluate.py:68-72).
 * aps: (n_q) fp64; prs: (n_q, n_kappa) fp64 (n_kappa <= 16).  ws: mdir_map_workspace_bytes().   */
size_t mdir_map_workspace_bytes(int64_t n_db, int n_q);
int mdir_compute_ap(const int64_t* ranks, int64_t n_db, int n_q, const int64_t* items, const int32_t* item_query,
                    const int32_t* item_class, int64_t n_items, const int32_t* n_pos, const int32_t* kappas,
                    int n_kappa, double* aps, double* prs, void* ws, void* stream);

/* ------------------------------------------------------------- composites ---
 * One call per stage for hosts that do not want to chain the component launchers themselves
 * (SURVEY.md section 8b).  Pure host-side planning + the launchers above on the caller's stream.
 *
 * mdir_sim_topk_bf16: the k best database rows for n_q <= 128 queries -- the first k rows of
 * np.argsort(-np.dot(vecs.T, qvecs), axis=0) (cirscore.py:69-70) without materialising scores.
 *   db16 (n_db, D) bf16 rows (mdir_pack_bf16); db32 (n_db, D) fp32 master or NULL;
 *   q32 (n_q, D) fp32 queries.  db32 != NULL: bf16 shortlist of `shortlist` rows (0 = 1.25k rounded
 *   up to a multiple of 64) re-scored exactly in fp32 (fp32-faithful ranking), certified when
 *   db_stats (mdir_pack_stats) is given -- see mdir_topk_finalize_rescore; NULL: exact top-k of the
 *   bf16 scores.
 *   route 0 = automatic (one-launch threshold+filter scan, three-launch scan, or dense for small
 *   databases), 1 = dense (every score; the exact recovery after overflow[q] != 0; n_db <= 131072).
 *   out_scores / out_idx (n_q, k), out_keys (n_q, k) or NULL, overflow (n_q) int32 status words
 *   (MDIR_STATUS_*).  k <= n_db.
 *   ws: mdir_sim_topk_workspace_bytes(D) bytes (~115 MB), contents irrelevant.
 *   mdir_topk_plan exposes the route choice (0 dense / 1 one-launch / 2 three-launch + its sampling plan).
 * mdir_gem_head: pooling -> L2N -> multi-scale aggregation -> [Lw centre, project, renormalise] for
 *   n_img images x S scales (maps image-major, scale-minor; off/hw as in mdir_pool).  P (>= dims, C)
 *   and/or Px3 = mdir_split_tf32x3(P, role 0) select the projection (both NULL: out is (n_img, C));
 *   msp = the GeM p when the reference's msp rule applies (wrapper.py:122-124), else 1.
 *   out (n_img, dims).  ws: mdir_gem_head_workspace_bytes(n_img, S, C, dims) bytes.            */
int mdir_topk_plan(int64_t n_db, int kth, int sm_count, int* route, int* n_sample, int* stride);   /* host-only planner */
size_t mdir_sim_topk_workspace_bytes(int D);
int mdir_sim_topk_bf16(const uint16_t* db16, const float* db32, const float* db_stats, int64_t n_db,
                       const float* q32, int n_q, int D, int k, int shortlist, uint32_t idx_base, int route,
                       float* out_scores, int32_t* out_idx, uint64_t* out_keys, int32_t* overflow,
                       void* ws, void* stream);
size_t mdir_gem_head_workspace_bytes(int n_img, int S, int C, int dims);
int mdir_gem_head(int kind, const float* x, const int64_t* off, const int32_t* hw, int n_img, int S, int C,
                  int hw_uniform, float p, float eps, float msp, const float* m, const float* P,
                  const float* Px3, int dims, float* out, void* ws, void* stream);

/* ------------------------------------ shard merge over NVLink peer memory ---
 * Multi-GPU top-k (SURVEY.md section 8e): every rank holds a row shard and its local top-k as sorted
 * 64-bit keys (n_q, k).  mdir_shard_exchange_merge is the exchange AND the merge in one kernel: it
 * stores the local keys into every rank's mailbox (peer-mapped device memory), publishes
 * per-(rank, query) sequence flags with system-scope release, waits (bounded) for the world's flags
 * and merges the world * k keys per query -> out_scores / out_idx (n_q, k), identical on every rank.
 * No collective-library call; every rank must issue the same sequence of calls.
 * Setup: each rank mdir_p2p_alloc()s a mailbox of mdir_shard_mailbox_bytes(world, max_q, max_k)
 * bytes (zeroed), ships the 64-byte handle to its peers (any transport), and mdir_p2p_open()s theirs;
 * mailboxes = host array of `world` device pointers, entry `rank` being the own allocation.
 * mdir_shard_status: non-zero once a peer failed to arrive within the bounded wait (~2 s).      */
size_t mdir_shard_mailbox_bytes(int world, int max_q, int max_k);
int mdir_p2p_alloc(size_t bytes, void** ptr, void* handle64);
int mdir_p2p_open(const void* handle64, void** ptr);
int mdir_p2p_close(void* ptr);
int mdir_p2p_free(void* ptr);
#define MDIR_EXCHANGE_SYNC 0      /* push this step's keys, wait for the world's, merge them               */
#define MDIR_EXCHANGE_DEFERRED 1  /* push this step's keys, merge the PREVIOUS step's (arrived a step ago):  */
                                  /* exchange latency and rank skew hide behind the next scan                */
#define MDIR_EXCHANGE_FLUSH 2     /* no push; merge the last pushed step (drain after deferred calls)        */
/* local_status (n_q) int32 or NULL: this rank's MDIR_STATUS_* word per query of the step being pushed (it rides in
 * the flag word); out_status (n_q) int32 or NULL: OR of the world's status words for the step being MERGED, plus
 * bit 2 (value 4) when a peer did not arrive -- identical on every rank except for that last bit.               */
int mdir_shard_exchange_merge(const uint64_t* local_keys, int n_q, int k, int rank, int world,
                              int max_q, int max_k, int mode, void* const* mailboxes,
                              float* out_scores, int32_t* out_idx,
                              const int32_t* local_status, int32_t* out_status, void* stream);
int mdir_shard_status(const void* own_mailbox, int* status);

/* ---------------------------------------------- hard-negative mining (f4) ---
 * The consumer of a full ranking inside TuplesDataset.create_epoch_tuples
 * (mdir/external/cirtorch/datasets/traindataset.py:250-267): for query q walk ranks[:, q]
 * (ranks (n_pool, n_q) int64 C-order, pitch ranks_ld, as mdir_rank_scores writes them) from the
 * best score down and keep the first nnum pool positions whose cluster differs from
 * q_cluster[q] and from every cluster already kept.  out_pos (n_q, nnum) pool positions (-1
 * where the pool ran out), out_found (n_q) how many were found.  nnum <= 63.
 * mdir_pair_l2dist: out[q, j] = sqrt(sum_d (q[q, d] - pool[pos[q, j], d] + eps)^2), the
 * reference's torch.pow(q - p + 1e-6, 2).sum().sqrt() (traindataset.py:263); q (n_q, D) and
 * pool (n_pool, D) row-major fp32; NaN where pos < 0.                                        */
int mdir_mine_negatives(const int64_t* ranks, int64_t ranks_ld, int64_t n_pool, int n_q,
                        const int32_t* pool_cluster, const int32_t* q_cluster, int nnum,
                        int64_t* out_pos, int32_t* out_found, void* stream);
int mdir_pair_l2dist(const float* q, const float* pool, const int64_t* pos, int n_q, int nnum, int D,
                     float eps, float* out, void* stream);

/* --------------------------------------------- learning the whitening (f4) ---
 * The O(D^2 N) fp64 contractions of whitenlearn / pcawhitenlearn
 * (mdir/external/cirtorch/utils/whiten.py:14-53) on (D, N) matrices whose columns are images.
 * mdir_gemm_f64: C (M, N) = alpha * (A - a_sub) * op(B - b_sub); A (M, K) row-major pitch lda;
 * b_is_kxn == 0: B (N, K) row-major (np.dot(A, B.T), the covariance shape), else B (K, N)
 * row-major (np.dot(A, B)); a_sub / b_sub: optional per-row constants of A / B in their own
 * storage (the fused "X - m").  Deterministic (split-K partial planes summed in order);
 * ws: mdir_gemm_f64_workspace_bytes(M, N, K) bytes (may be 0 -> NULL).
 * mdir_pair_diff_f64: out (D, n_pairs) = X[:, qidx] - X[:, pidx] (whiten.py:41).
 * mdir_cols_mean_f64: mean[d] = mean_j X[d, idx[j]]  (idx NULL: the first n_idx columns).    */
size_t mdir_gemm_f64_workspace_bytes(int M, int N, int64_t K);
int mdir_gemm_f64(const double* A, int64_t lda, const double* a_sub, const double* B, int64_t ldb,
                  const double* b_sub, int b_is_kxn, int M, int N, int64_t K, double alpha,
                  double* C, int64_t ldc, void* ws, void* stream);
int mdir_pair_diff_f64(const double* X, int64_t ldx, int D, int64_t n_cols, const int64_t* qidx,
                       const int64_t* pidx, int64_t n_pairs, double* out, void* stream);
int mdir_cols_mean_f64(const double* X, int64_t ldx, int D, int64_t n_cols, const int64_t* idx,
                       int64_t n_idx, double* mean, void* stream);
int mdir_f32_to_f64(const float* src, int64_t n, double* dst, void* stream);

#ifdef __cplusplus
}
#endif
#endif
