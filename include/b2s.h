/* b2s.h — C ABI of libb2s.so: B200 (sm_100a) kernels for the ORB front-end hot path.
 *
 * Drop-in boundary (SURVEY.md §8b).  Each entry point names the reference
 * interface (file:line under /root/reference) whose arithmetic it replaces.
 * Plain pointers and sizes only; no torch types.  All device pointers must be
 * CUDA device memory on the current device; `stream` is a cudaStream_t passed
 * as void*.  Every function returns 0 on success, non-zero on error
 * (b2s_last_error() has the text); nothing throws across the ABI.  All work is
 * enqueued asynchronously on `stream`; nothing here synchronises the device.
 *
 * Batching: a "pair" is one (query frame, train frame) match problem.  Rows of
 * all pairs are concatenated; `*_off` arrays (device, n_pairs+1 int32) are CSR
 * offsets into the concatenation.  Descriptors are 32 bytes (ORB), row-major,
 * buffers 16-byte aligned.
 *
 * Packed key: key = (distance << 22) | index, distance in [0,256], index < 2^22.
 * min(key) == lexicographic (distance, index) minimum == OpenCV's tie rule.
 * Any key >= 0x80000000 means "none"; outputs use B2S_NONE_KEY for it.
 */
#ifndef B2S_H_
#define B2S_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2S_ABI_VERSION 5
#define B2S_IDX_BITS 22
#define B2S_IDX_MASK ((1u << B2S_IDX_BITS) - 1u)
#define B2S_NONE_KEY 0xFFFFFFFFu
#define B2S_DESC_BYTES 32
#define B2S_MAX_ROWS_PER_PAIR (1 << B2S_IDX_BITS)
#define B2S_SELECT_MAX_QUERIES 32768 /* per pair, b2s_select_matches */

/* error codes */
#define B2S_OK 0
#define B2S_ERR_INVALID 1   /* bad argument */
#define B2S_ERR_CUDA 2      /* CUDA runtime error (text in b2s_last_error) */
#define B2S_ERR_UNSUPPORTED 3

/* Hamming kernel variants */
#define B2S_VARIANT_POPC 0  /* LOP3/POPC integer-pipe kernel (K1) */
#define B2S_VARIANT_I8MMA 1 /* tcgen05.mma kind::i8 +-8 contraction, two products D and D^T (K2) */
#define B2S_VARIANT_I8MMA1 2 /* same contraction, ONE product; column minima by warp butterfly (K2s) */
/* OR-ed into `variant` (K2s only; the other kernels ignore it): the per-row SECOND neighbour is not needed —
 * fwd_second is left "none".  That is BFMatcher(crossCheck=True).match (feature_pipeline.py.bak:82,
 * persistent_map.py:266, keyframe_manager.py:126,141), the reference's default matcher; only knnMatch + ratio
 * (.bak:84-91) and match_orb_descriptors (homography.py:9-26) read the second neighbour. */
#define B2S_HAMMING_BEST_ONLY 0x100

int b2s_abi_version(void);
/* Number of kernels this library has launched in this process (bench.py gpu_launches). */
unsigned long long b2s_launch_count(void);
const char* b2s_last_error(void);
/* sm_count / cc_major / cc_minor / sm clock kHz of the current device. */
int b2s_device_info(int* sm_count, int* cc_major, int* cc_minor, int* clock_khz);

/* Optional record sink of the winner kernels (HOST struct, passed by pointer; NULL or records == NULL = none): the
 * kernel that picks the winner also writes the pair's result record (layout: b2s_pack_records below) — no extra
 * launch at the end of a step.  out_q / out_t / out_d: the selection outputs in the compact layout (pair p at
 * p * stride); R | t in the record header stay zero (use b2s_pack_records after the pose kernels for those). */
typedef struct b2s_record_sink {
  uint8_t* records;      /* device, n_pairs records of record_bytes each */
  size_t record_bytes;   /* >= b2s_record_bytes(stride), multiple of 16 */
  const int32_t* out_q;
  const int32_t* out_t;
  const int32_t* out_d;
  int stride;
  int pair_id0;          /* header pair id = pair_id0 + p */
} b2s_record_sink;

/* ---- K1/K2: brute-force Hamming kNN-2 + column minimum ------------------------
 * Replaces cv::BFMatcher(NORM_HAMMING).knnMatch(k=2) and the two batchDistance
 * passes of BFMatcher(crossCheck=True).match (feature_pipeline.py.bak:68,82,84;
 * persistent_map.py:266; keyframe_manager.py:126,141) and the NumPy matcher's
 * distance loops (homography.py:12-15, :21-23) — one distance matrix serves both
 * directions.
 *   fwd_best[i], fwd_second[i]  (total_nq)  two smallest (dist, trainIdx) keys of query row i
 *   bwd_best[j]                 (total_nt)  smallest (dist, queryIdx) key of train row j
 * Indices inside keys are pair-local.  q_src_row/t_src_row (device, n_pairs int32,
 * or NULL): row in q_desc/t_desc where pair p's descriptors start, when that differs
 * from the CSR offset — lets many pairs share one descriptor block (relocalization:
 * every keyframe against the same current frame, persistent_map.py:244-266) while the
 * outputs stay CSR-addressed.  max_nq/max_nt: upper bounds on any pair's
 * row counts (host-known; sizes the grid).  t_split: CTAs per query tile along the
 * train axis (0 = choose automatically); workspace must hold
 * b2s_hamming_workspace_bytes(total_nq, t_split_max) bytes when t_split != 1. */
size_t b2s_hamming_workspace_bytes(int total_nq, int t_split);
/* Workspace of either variant.  The I8MMA variants stage every descriptor as 256 int8 (+8/-8)
 * in 36 KB operand tiles (128 rows x 18 k-chunks of 16 B): n_pairs * (ceil(max_nq/128) +
 * ceil(max_nt/128)) * 36 KB, 128-byte aligned.  The single-product variant (I8MMA1) also honours
 * t_split (0 = automatic: a batch with fewer (pair, query block) work items than SMs — one
 * 10 000 x 10 000 pair, a lone 2000 x 2000 drop-in call — is cut along the train axis and the
 * partial top-2 merged on the packed keys) and adds total_nq * t_split * 8 bytes for it. */
size_t b2s_hamming_workspace_bytes_v(int variant, int n_pairs, int total_nq, int max_nq, int max_nt,
                                     int t_split);
int b2s_hamming_knn2_batched(const uint8_t* q_desc, const uint8_t* t_desc,
                             const int32_t* q_off, const int32_t* t_off,
                             const int32_t* q_src_row, const int32_t* t_src_row, int n_pairs,
                             int total_nq, int total_nt, int max_nq, int max_nt,
                             uint32_t* fwd_best, uint32_t* fwd_second, uint32_t* bwd_best,
                             int variant, int t_split, void* workspace, size_t workspace_bytes,
                             void* stream);
/* Tuning of the POPC kernel (bench sweeps): csa_level 0..3 (8/6/5/4 POPC per
 * descriptor pair), rows_per_thread in {2,4}, warps in {4,8}.  -1 keeps a field. */
int b2s_hamming_set_config(int csa_level, int rows_per_thread, int warps);
int b2s_hamming_get_config(int* csa_level, int* rows_per_thread, int* warps);

/* ---- selection: ratio LUT, cross-check, stable sort, truncate -----------------
 * Replaces the Python post-processing of ORBFeaturePipeline.match
 * (feature_pipeline.py.bak:85-94), the emit rule of BFMatcher(crossCheck=True)
 * and match_orb_descriptors' ratio + symmetry tests (homography.py:16-25).
 *   use_ratio: keep iff a second neighbour exists and d1 < ratio_lut[d2]
 *              (ratio_lut: HOST pointer, 257 int32, = ceil(ratio*d2) in float64)
 *   use_cross: keep iff index(bwd_best[j]) == i
 *   sort_by_distance: stable sort by distance (ties ascending queryIdx), else ascending queryIdx
 *   max_matches: > 0 truncates, 0 = keep all
 *   kp_q/kp_t: optional (rows, 2) float32 keypoint coordinates; when both given,
 *              out_corr[(base+k)*4 .. +3] = (x1, y1, x2, y2) of match k
 *              (matches_to_points, feature_pipeline.py.bak:104-111).  kp_*_src_row
 *              (device, n_pairs int32, or NULL): first keypoint row of pair p when it is
 *              not the CSR offset (shared frames, as q_src_row/t_src_row above).
 *   out_stride: 0 -> pair p's outputs live at [q_off[p], q_off[p] + out_count[p]);
 *              > 0 -> at [p*out_stride, p*out_stride + out_count[p]) (compact layout for
 *              truncated selections; a pair that does not fit gets out_count = -1).
 *   out_total: optional (n_pairs int32): matches that passed the tests BEFORE truncation to max_matches
 *              (the relocalization sweep ranks keyframes by it). */
int b2s_select_matches(const uint32_t* fwd_best, const uint32_t* fwd_second,
                       const uint32_t* bwd_best, const int32_t* q_off, const int32_t* t_off,
                       int n_pairs, int max_nq, int use_ratio, int use_cross,
                       const int32_t* ratio_lut_host, int sort_by_distance, int max_matches,
                       const float* kp_q, const float* kp_t, const int32_t* kp_q_src_row,
                       const int32_t* kp_t_src_row, int out_stride, int32_t* out_q, int32_t* out_t,
                       int32_t* out_d, float* out_corr, int32_t* out_count, int32_t* out_total, void* stream);

/* ---- K4: batched 8-point minimal solver ---------------------------------------
 * Replaces the per-iteration body of ransac_essential up to the hypothesis
 * (homography.py:325-326 -> eight_point_E, :222-248, K^T F K quirk included).
 * corr: float32 (x1,y1,x2,y2) per correspondence; pair p owns
 * [c_off[p], c_off[p]+c_count[p]).  For every pair, H hypotheses:
 *   samples_in != NULL: use samples_in[(p*H+h)*8 .. +7] (seeded host draws, parity mode)
 *   samples_in == NULL: draw 8 distinct indices on device from (seed, id(p), h), id(p) = pair_ids[p]
 *                       (device int32, optional) or pair_id0 + p: the pair's GLOBAL id, so that a pair
 *                       draws the same samples on whichever rank / batch position it is processed
 * samples_out (optional) receives the indices used.  K_host / Kinv_host: HOST
 * pointers to 9 doubles, row-major (NULL = identity).  E_out: (n_pairs*H*9) doubles.
 * Pairs with fewer than 8 correspondences get all-zero hypotheses. */
int b2s_eight_point_batched(const float* corr, const int32_t* c_off, const int32_t* c_count,
                            int n_pairs, int H, const int32_t* samples_in, uint64_t seed,
                            const int32_t* pair_ids, int pair_id0, int32_t* samples_out,
                            const double* K_host, const double* Kinv_host, double* E_out, void* stream);

/* ---- K3: batched Sampson-error hypothesis scoring ------------------------------
 * Replaces homography.py:328-333 for all hypotheses at once.
 * counts[p*H+h] = #{m : (x2^T E x1)^2 < th2 * (Ex1_x^2+Ex1_y^2+Etx2_x^2+Etx2_y^2)}
 * th2_per_pair: optional device array (n_pairs doubles) overriding th2.
 * precision: 64 = float64 decisions (float32 screening with a rigorous rounding bound, the
 * undecidable band re-evaluated in float64 — counts identical to 6464 at ~0.6x the time),
 * 6464 = every evaluation in float64 (the reference's arithmetic, kept for validation),
 * 32 = float32 only (within the north-star flip tolerance, not bit-identical).
 * max_m: host-known upper bound of any c_count[p], or 0 = unknown; with precision 64 a batch of few
 * pairs with thousands of correspondences each is then also cut along the correspondences (partial
 * counts summed with atomicAdd) so that it fills the machine. */
int b2s_ransac_score_batched(const float* corr, const int32_t* c_off, const int32_t* c_count,
                             int n_pairs, const double* E, int H, double th2,
                             const double* th2_per_pair, int precision, int max_m, int32_t* counts,
                             void* stream);

/* K5 / K6 — batched RANSAC homography (next-row #3).  Same conventions as the essential-matrix
 * entry points: corr = (src.x, src.y, dst.x, dst.y) float32 per correspondence, CSR c_off /
 * c_count per pair, H hypotheses per pair, H_out / Hm = [pair][H][9] float64 row-major with
 * H[2][2] = 1 (all zero for a pair with fewer than 4 correspondences).
 * b2s_homography_dlt_batched   replaces dlt_homography on 4-samples, homography.py:193-194 / :131-142
 *                              (samples_in [pair][H][4] = the host's rng.choice draws, or NULL = device RNG);
 * b2s_homography_score_batched replaces the symmetric transfer error + threshold, homography.py:196-206
 *                              (th in the units of the points; th_per_pair optional);
 * b2s_homography_select        replaces the strict-improvement / 0.8 n early-exit bookkeeping, :207-211,
 *                              and writes the winner's inlier mask. */
/* samples_in == NULL: the device draws 4 distinct indices from (seed, id(p), h) with id(p) = pair_ids[p] (device int32,
 * optional) or pair_id0 + p, the pair's GLOBAL id, as b2s_eight_point_batched does: a pair draws the same samples on
 * whichever rank / batch position it is processed (pair_ids = NULL, pair_id0 = 0: id(p) = p). */
int b2s_homography_dlt_batched(const float* corr, const int32_t* c_off, const int32_t* c_count, int n_pairs, int H,
                               const int32_t* samples_in, uint64_t seed, const int32_t* pair_ids, int pair_id0,
                               int32_t* samples_out, double* H_out, void* stream);
int b2s_homography_score_batched(const float* corr, const int32_t* c_off, const int32_t* c_count, int n_pairs,
                                 const double* Hm, int H, double th, const double* th_per_pair, int32_t* counts,
                                 void* stream);
int b2s_homography_select(const int32_t* counts, const float* corr, const int32_t* c_off, const int32_t* c_count,
                          int n_pairs, const double* Hm, int H, double th, const double* th_per_pair, int32_t* best_h,
                          int32_t* best_count, uint8_t* inlier_mask, void* stream);

/* K7 — batched decompose_essential (homography.py:251-299, next-row #2): per pair the SVD of E,
 * the four (R, t) candidates in the reference's order (U W V^T, +u3), (U W V^T, -u3),
 * (U W^T V^T, +u3), (U W^T V^T, -u3), and for each candidate the number of correspondences
 * (restricted to inlier_mask != 0 when given) whose DLT triangulation lies in front of both
 * cameras.  candidates = [pair][4][12] float64 (R row-major, then t), votes = [pair][4] int32.
 * The caller takes the first maximum of votes (np.argmax semantics, :296-298).  K_host = 3x3
 * row-major intrinsics on the HOST (NULL = identity); max_m >= every c_count[p]. */
int b2s_decompose_essential_batched(const double* E, const float* corr, const int32_t* c_off, const int32_t* c_count,
                                    const uint8_t* inlier_mask, int n_pairs, int max_m, const double* K_host,
                                    double* candidates, int32_t* votes, void* stream);

/* The (R, t) of the first candidate with the most votes (np.argmax semantics of homography.py:296-298):
 * R_out [pair][9], t_out [pair][3] float64. */
int b2s_pose_pick(const double* candidates, const int32_t* votes, int n_pairs, double* R_out, double* t_out, void* stream);

/* Refit of E on a pair's inliers (homography.py:344 -> eight_point_E, :222-248, K^T F K quirk
 * included): E_out [pair][9] float64 (zeros when fewer than 8 correspondences take part),
 * n_used [pair] (optional) = correspondences that took part.  inlier_mask NULL = all. */
int b2s_refit_essential_batched(const float* corr, const int32_t* c_off, const int32_t* c_count, const uint8_t* inlier_mask,
                                int n_pairs, const double* K_host, const double* Kinv_host, double* E_out, int32_t* n_used,
                                void* stream);

/* K8 — batched 5-point minimal solver (Nister): S samples per pair, up to 10 real essential
 * matrices per sample.  corr must hold CALIBRATED (K^-1-normalised) points, as cv2.findEssentialMat
 * normalises them before its solver (call sites slam_viewer.py:195, web_dashboard_server.py:145,
 * visual_slam_offline_entry_point.py:51).  E_out = [pair][S][10][9] float64, unit Frobenius norm,
 * unused slots zero (a zero E scores zero inliers, so E_out can go to the scoring entry points as
 * H = 10 S hypotheses); n_sol [pair][S] (optional) = real solutions found; samples_in [pair][S][5]
 * = host-drawn indices or NULL = device RNG. */
int b2s_five_point_batched(const float* corr, const int32_t* c_off, const int32_t* c_count, int n_pairs, int S,
                           const int32_t* samples_in, uint64_t seed, int32_t* samples_out, double* E_out, int32_t* n_sol,
                           void* stream);

/* b2s_hamming_knn2_batched (variant B2S_VARIANT_I8MMA1) for batches whose pairs SHARE descriptor blocks:
 * consecutive-frame tracking (frame k+1 is the train side of pair k and the query side of pair k+1,
 * slam_api.py:352-353) and relocalization (one query frame against every keyframe,
 * persistent_map.py:244-309).  Every distinct block is expanded to tensor-core operand tiles ONCE.
 * desc = the one descriptor buffer; block b = blk_rows[b] rows starting at row blk_row0[b], its
 * tiles start at tile blk_tile0[b] (prefix sum of ceil(rows / 128); total_tiles in all);
 * q_xtile[p] / t_xtile[p] = first tile of pair p's query / train block; q_off / t_off = CSR of the
 * OUTPUT rows (q_off[p+1] - q_off[p] must equal the query block's rows).  All index arrays int32 on
 * the device.  Outputs and t_split as b2s_hamming_knn2_batched; need_second = 0 is B2S_HAMMING_BEST_ONLY.  workspace: b2s_hamming_shared_workspace_bytes
 * (same n_pairs / total_nq / max_nq / max_nt / t_split as the call). */
size_t b2s_hamming_shared_workspace_bytes(int total_tiles, int n_pairs, int total_nq, int max_nq, int max_nt,
                                          int t_split);
int b2s_hamming_knn2_shared(const uint8_t* desc, const int32_t* blk_row0, const int32_t* blk_rows,
                            const int32_t* blk_tile0, int n_blocks, int total_tiles, int max_block_rows,
                            const int32_t* q_xtile, const int32_t* t_xtile, const int32_t* q_off, const int32_t* t_off,
                            int n_pairs, int total_nq, int total_nt, int max_nq, int max_nt, uint32_t* fwd_best,
                            uint32_t* fwd_second, uint32_t* bwd_best, int t_split, int need_second, void* workspace,
                            size_t workspace_bytes, void* stream);
/* Diagnostics: work decomposition of the most recent single-product launch — query sub-tiles per
 * work item (always 2), train-axis split, CTAs. */
void b2s_hamming_last_plan(int* subs, int* t_split, int* grid);

/* K9 — bag-of-words candidate ranking, the step in front of the relocalizer's matching (next-row #4).
 * b2s_bow_histogram_batched  replaces compute_bow_histogram (persistent_map.py:82-96) and
 *                            BoWDatabase._compute_hist (loop_closure.py:36-48) for n_frames frames at
 *                            once: desc = concatenated (N, 32) uint8 ORB descriptors read as 32 float
 *                            values, f_off = CSR offsets (n_frames + 1), vocab = [k][32] float32
 *                            centroids; nearest centroid by squared Euclidean distance in float64
 *                            (sklearn pairwise_distances_argmin_min; first index on ties);
 *                            words [total] (optional) = word of every descriptor, counts
 *                            [n_frames][k] int32 (zeroed here), hist [n_frames][k] float32 =
 *                            counts / n (float32 division, all zero for an empty frame).
 * b2s_bow_cosine             replaces sklearn cosine_similarity([hist], hists)[0]
 *                            (persistent_map.py:235, loop_closure.py:63): scores [n] float32, float64
 *                            accumulation, zero rows score 0. */
int b2s_bow_histogram_batched(const uint8_t* desc, const int32_t* f_off, int n_frames, int max_n, const float* vocab,
                              int k, int32_t* words, int32_t* counts, float* hist, void* stream);
int b2s_bow_cosine(const float* hist_q, const float* hists, int n, int k, float* scores, void* stream);

/* K3t — the same counts as b2s_ransac_score_batched(precision 64 / 6464) from the tensor cores:
 * both bilinear forms of the Sampson test as tcgen05.mma kind::tf32 products of hi/lo-split
 * operands, float32 decision with a rigorous error bound, float64 re-evaluation inside the band
 * (csrc/ransac_tc.cu).  max_m >= every c_count[p].  workspace: b2s_ransac_score_tc_workspace_bytes,
 * 128-byte aligned.  dbg_num / dbg_den (both or neither, [pair][H][dbg_ld] float) receive the raw
 * accumulators, dbg_band (two ints) the number of float64 re-evaluations and the work-list
 * overflow flag; NULL in production.  Replaces the scoring lines of ransac_essential, homography.py:328-333. */
size_t b2s_ransac_score_tc_workspace_bytes(int n_pairs, int H, int max_m);
int b2s_ransac_score_tc(const float* corr, const int32_t* c_off, const int32_t* c_count, int n_pairs, int max_m,
                        const double* E, int H, double th2, const double* th2_per_pair, int32_t* counts,
                        void* workspace, size_t workspace_bytes, float* dbg_num, float* dbg_den, int dbg_ld,
                        int32_t* dbg_band, void* stream);

/* ---- winner selection + inlier mask --------------------------------------------
 * Replaces the sequential best/early-exit bookkeeping of homography.py:335-339:
 * best_h = first h with count > 0.8*M if any, else the lowest h among the
 * maximum count; -1 when every count is 0.  inlier_mask[c_off[p]+m] = 1 iff
 * correspondence m is an inlier of hypothesis best_h (float64 arithmetic).  mask_stride > 0: the kernel also
 * zeroes inlier_mask[c_off[p] + c_count[p] .. c_off[p] + mask_stride) (the unused tail of a compact slot), so the
 * caller need not clear the array; sink: see b2s_record_sink. */
int b2s_ransac_select(const int32_t* counts, const float* corr, const int32_t* c_off,
                      const int32_t* c_count, int n_pairs, const double* E, int H, double th2,
                      const double* th2_per_pair, int32_t* best_h, int32_t* best_count,
                      uint8_t* inlier_mask, const b2s_record_sink* sink, int mask_stride, void* stream);

/* ---- result records: what leaves the GPU ------------------------------------------
 * One fixed-size record per pair, written by ONE kernel straight into the buffer that is all-gathered over
 * NCCL when pairs are sharded across GPUs (SURVEY.md 8e) or copied to the host in one transfer.  Replaces
 * the Python result objects of the reference: list[cv2.DMatch] (feature_pipeline.py.bak:78-95) and
 * (R, t, inliers, match_count) (homography.py:423-438).
 *   record = int32 header[16] { n_matches, best_h, inlier_count, pair_id, R[9] as float32 bits, t[3] as float32 bits }
 *            | uint16 queryIdx[S] | uint16 trainIdx[S] | uint16 distance[S] | uint8 inlier[S] | pad to 64 bytes
 * S = stride = the compact selection stride (max_matches; rows per frame must be < 65536).
 * count / out_q / out_t / out_d / inlier_mask: the selection and winner outputs (compact layout, pair p at
 * p * stride); count_total (optional): header n_matches when it differs from the selected count (matches
 * before truncation); R / t (optional, float64 [.][9] / [.][3]); pair_ids (optional) overrides
 * pair_id0 + p; src_pair (optional, n_records int32): record r describes pair src_pair[r] (-1 = empty
 * slot) and best_h / best_count / R / t are then indexed by r (ranked candidates, b2s_rank_pairs). */
size_t b2s_record_bytes(int max_matches);
/* Pose record: the answer of the robust pose estimator (b2s_robust_pose_decide with a record sink) appended to a result
 * record, so that every offset of the record above stays where it is:
 *   pose record = record of b2s_record_bytes(S) bytes | b2s_pose_result (B2S_POSE_RESULT_BYTES = 200) | 56 zero bytes
 * b2s_pose_record_bytes(S) = b2s_record_bytes(S) + B2S_POSE_BLOCK_BYTES (S = 500: 3584 + 256 = 3840 bytes).  The
 * header of a pose record: n_matches = the selection count (-1 on overflow), best_h = the SELECTED model's RANSAC winner
 * (e_best_h or h_best_h of the result; -1 for an error outcome), inlier_count = result.inliers, pair_id = pair_id0 + p,
 * R | t = the result's R and normalised t as float32 (zero for an error outcome); inlier[S] = the selected model's
 * flags (zero past n_matches, and all zero for an error outcome).  A record slot that holds no pair (the padding of a
 * sharded gather buffer) has pair_id -1 and, in a pose record, outcome -1. */
#define B2S_POSE_BLOCK_BYTES 256
size_t b2s_pose_record_bytes(int max_matches);
int b2s_pack_records(const int32_t* count, const int32_t* count_total, const int32_t* best_h, const int32_t* best_count,
                     const int32_t* out_q, const int32_t* out_t, const int32_t* out_d, const uint8_t* inlier_mask,
                     const double* R, const double* t, const int32_t* pair_ids, const int32_t* src_pair, int n_records,
                     int stride, int pair_id0, uint8_t* records, size_t record_bytes, void* stream);

/* The k (<= 32) pairs with the largest score, ties to the lower id then the lower position — the candidate
 * ranking of MapRelocalizer.relocalize (persistent_map.py:236-242: sorted by (-score, frame_id), first
 * max_candidates) on the device, for the whole-map sweep (BASELINE config #5: score = cross-check match
 * count).  score < 0 excludes a pair.  top_idx [k] = pair index or -1; top_id [k] (optional) = its id (-1);
 * c_off / c_count (optional, [k]) =
 * CSR view of the winners' compact correspondences (top_idx * stride, sel_count[top_idx]) for the RANSAC
 * entry points. */
int b2s_rank_pairs(const int32_t* score, const int32_t* ids, const int32_t* sel_count, int n, int k, int stride,
                   int32_t* top_idx, int32_t* top_id, int32_t* c_off, int32_t* c_count, void* stream);

/* ---- winner only: the reference's answer without scoring every hypothesis to the end ----------------
 * best_h / best_count / inlier_mask exactly as b2s_ransac_score_batched(precision 64) + b2s_ransac_select
 * return them, but a hypothesis is abandoned as soon as it can neither exceed 0.8 * M nor reach the largest
 * complete count (homography.py:335-339): all H hypotheses are scored on the first ~3/8 of the correspondences,
 * the 8 most promising are finished to get a lower bound of the maximum, and only the hypotheses whose upper
 * bound reaches it are finished.  counts_out (optional, [pair][H]) receives complete counts for the finished
 * hypotheses and lower bounds for the abandoned ones; n_finished_out (optional, [pair]) the number finished in
 * the last pass.  workspace: b2s_ransac_winner_workspace_bytes, 16-byte aligned. */
size_t b2s_ransac_winner_workspace_bytes(int n_pairs, int H);
int b2s_ransac_winner_batched(const float* corr, const int32_t* c_off, const int32_t* c_count, int n_pairs, const double* E,
                              int H, double th2, const double* th2_per_pair, int32_t* best_h, int32_t* best_count,
                              uint8_t* inlier_mask, void* workspace, size_t workspace_bytes, int32_t* counts_out,
                              int32_t* n_finished_out, const b2s_record_sink* sink, int mask_stride, void* stream);

/* ---- robust pose: essential / homography model selection with stability gates ------------------------
 * The batched form of RobustPoseEstimator.estimate_pose (robust_pose_estimator.py:89-251): adaptive threshold,
 * both RANSAC branches, per-branch inlier ratio, median parallax, cheirality and score, model selection (the
 * essential model wins ties) and the five stability gates.  The RANSAC stages are the existing entry points
 * (K4 / K3 / select with th2_per_pair, K7 refit + decomposition, K5 / K6 / select at th = 3); the three
 * entry points below are the pieces around them.
 *
 * Configuration: the fields of RobustPoseEstimatorConfig (robust_pose_estimator.py:42-70).  Passed as a DEVICE
 * array of n_cfg entries; pair p uses cfg[n_cfg == 1 ? 0 : p]. */
typedef struct b2s_robust_pose_config {
  int32_t min_matches;
  int32_t min_inliers;
  int32_t min_cheirality_inliers;
  int32_t reserved;
  double base_ransac_threshold;
  double min_ransac_threshold;
  double max_ransac_threshold;
  double min_inlier_ratio;
  double homography_bias;
  double essential_bias;
  double min_parallax;
  double min_cheirality_ratio;
} b2s_robust_pose_config;
#define B2S_ROBUST_POSE_CONFIG_BYTES 80

/* outcome of one pair: what estimate_pose returns or raises */
#define B2S_POSE_ESTIMATE 0           /* PoseEstimate */
#define B2S_POSE_GATE_FAILED 1        /* PoseEstimationFailure(gate reason, "relocalize", metrics) */
#define B2S_POSE_ERR_MATCHES 2        /* ValueError: fewer than min_matches correspondences */
#define B2S_POSE_ERR_EIGHT 3          /* ValueError: fewer than eight correspondences (ransac_essential) */
#define B2S_POSE_ERR_ESSENTIAL 4      /* RuntimeError: essential branch (< 8 RANSAC inliers / decomposition) */
#define B2S_POSE_ERR_HOMOGRAPHY 5     /* RuntimeError: homography branch (< 4 RANSAC inliers / decomposition) */
#define B2S_POSE_ERR_TRANSLATION 6    /* ValueError: zero translation; `method` names the branch */
/* method */
#define B2S_POSE_METHOD_ESSENTIAL 0
#define B2S_POSE_METHOD_HOMOGRAPHY 1
/* gate: the first failed stability gate, in the reference's order */
#define B2S_GATE_NONE 0
#define B2S_GATE_LOW_INLIER_COUNT 1
#define B2S_GATE_LOW_INLIER_RATIO 2
#define B2S_GATE_LOW_PARALLAX 3
#define B2S_GATE_CHEIRALITY_INLIERS 4
#define B2S_GATE_CHEIRALITY_RATIO 5

/* One fixed-size result per pair.  The diagnostics are those of the selected model (of the failing branch for
 * an error); e_* / h_* are the two RANSAC winners (hypothesis index, inlier count; -1 when the branch did not
 * run), which is what a caller needs to leave seeded generators where the reference leaves them.
 * median_parallax is the float32 median widened to float64; t is normalised. */
typedef struct b2s_pose_result {
  int32_t outcome;
  int32_t method;
  int32_t gate;
  int32_t match_count;
  int32_t inliers;
  int32_t cheirality_inliers;
  int32_t e_best_h;
  int32_t e_inliers;
  int32_t h_best_h;
  int32_t h_inliers;
  int32_t reserved[2];
  double inlier_ratio;
  double median_parallax;
  double cheirality_ratio;
  double score;
  double score_essential;
  double score_homography;
  double threshold;
  double R[9];
  double t[3];
} b2s_pose_result;
#define B2S_POSE_RESULT_BYTES 200
#ifdef __cplusplus
static_assert(sizeof(b2s_robust_pose_config) == B2S_ROBUST_POSE_CONFIG_BYTES, "b2s_robust_pose_config layout");
static_assert(sizeof(b2s_pose_result) == B2S_POSE_RESULT_BYTES, "b2s_pose_result layout");
static_assert(offsetof(b2s_pose_result, inlier_ratio) == 48 && offsetof(b2s_pose_result, threshold) == 96 &&
              offsetof(b2s_pose_result, R) == 104 && offsetof(b2s_pose_result, t) == 176, "b2s_pose_result offsets");
static_assert(B2S_POSE_BLOCK_BYTES >= B2S_POSE_RESULT_BYTES && B2S_POSE_BLOCK_BYTES % 64 == 0, "pose block");
#else
_Static_assert(sizeof(b2s_robust_pose_config) == B2S_ROBUST_POSE_CONFIG_BYTES, "b2s_robust_pose_config layout");
_Static_assert(sizeof(b2s_pose_result) == B2S_POSE_RESULT_BYTES, "b2s_pose_result layout");
_Static_assert(offsetof(b2s_pose_result, inlier_ratio) == 48 && offsetof(b2s_pose_result, threshold) == 96 &&
               offsetof(b2s_pose_result, R) == 104 && offsetof(b2s_pose_result, t) == 176, "b2s_pose_result offsets");
_Static_assert(B2S_POSE_BLOCK_BYTES >= B2S_POSE_RESULT_BYTES && B2S_POSE_BLOCK_BYTES % 64 == 0, "pose block");
#endif

/* Median displacement per pair: np.median(np.linalg.norm(pts2[sel] - pts1[sel], axis=1)) on the float32
 * correspondences, bit for bit (float32 norm without contraction, exact radix select on the bit patterns,
 * float32(a + b) / 2 for an even count, 0 for an empty selection; a NaN displacement gives NaN).  mask NULL =
 * all correspondences.  cfg (device, n_cfg entries) non-NULL: also the adaptive threshold of
 * adaptive_ransac_threshold (feature_pipeline.py.bak:114-129) in float64, th_out and th2_out = th * th
 * (either may be NULL).  One CTA per pair; any count. */
int b2s_displacement_median_batched(const float* corr, const int32_t* c_off, const int32_t* c_count, const uint8_t* mask,
                                    int n_pairs, const b2s_robust_pose_config* cfg, int n_cfg, float* median_out,
                                    double* th_out, double* th2_out, void* stream);

/* n-point normalised DLT of each pair's masked correspondences (dlt_homography, homography.py:118-142, the
 * final refit of ransac_homography :216): Hartley normalisation, Gram matrix in float64 reduced in a fixed order,
 * eigenvector of its smallest eigenvalue, de-normalised with H[2][2] = 1.  H_out [pair][9] (zeros when fewer
 * than 4 correspondences take part); n_used (optional) = correspondences that took part. */
int b2s_refit_homography_batched(const float* corr, const int32_t* c_off, const int32_t* c_count, const uint8_t* mask,
                                 int n_pairs, double* H_out, int32_t* n_used, void* stream);

/* Decision stage: per pair the essential branch (e_best_h / e_inliers from b2s_ransac_select, e_R / e_t from
 * b2s_pose_pick, e_votes from b2s_decompose_essential_batched, e_median = inlier median), the homography branch
 * (h_best_h / h_inliers from b2s_homography_select, H_fit from b2s_refit_homography_batched, decompose_homography
 * homography.py:59-78), all_median / th from b2s_displacement_median_batched; model selection and gates.
 * results [n_pairs]; out_mask [c_off[p] .. + c_count[p]) = the selected model's inlier flags (also for a gate
 * failure; zero for an error outcome); mask_stride > 0: out_mask[c_off[p] + c_count[p] .. c_off[p] + mask_stride)
 * is zeroed too (the unused tail of a compact slot).  Kinv_host: HOST 3x3 row-major (NULL = identity). */
int b2s_robust_pose_decide(const int32_t* c_off, const int32_t* c_count, int n_pairs, const int32_t* e_best_h,
                           const int32_t* e_inliers, const uint8_t* e_mask, const double* e_R, const double* e_t,
                           const int32_t* e_votes, const float* e_median, const float* all_median, const double* th,
                           const int32_t* h_best_h, const int32_t* h_inliers, const uint8_t* h_mask, const double* H_fit,
                           const double* Kinv_host, const b2s_robust_pose_config* cfg, int n_cfg,
                           b2s_pose_result* results, uint8_t* out_mask, int mask_stride, void* stream);
/* The same decision, and the same kernel launch, that also writes every pair's POSE record (b2s_pose_record_bytes
 * above) from the sink's selection outputs and its own result and flags: no extra launch at the end of a robust step.
 * sink NULL (or records NULL) = b2s_robust_pose_decide.  The sink needs record_bytes >= b2s_pose_record_bytes(stride),
 * a multiple of 16, 16-byte aligned records, and the compact selection layout (pair p at p * stride). */
int b2s_robust_pose_decide_records(const int32_t* c_off, const int32_t* c_count, int n_pairs, const int32_t* e_best_h,
                                   const int32_t* e_inliers, const uint8_t* e_mask, const double* e_R, const double* e_t,
                                   const int32_t* e_votes, const float* e_median, const float* all_median, const double* th,
                                   const int32_t* h_best_h, const int32_t* h_inliers, const uint8_t* h_mask,
                                   const double* H_fit, const double* Kinv_host, const b2s_robust_pose_config* cfg, int n_cfg,
                                   b2s_pose_result* results, uint8_t* out_mask, int mask_stride, const b2s_record_sink* sink,
                                   void* stream);

/* ---- measurement helper ----------------------------------------------------------
 * Saturates one SM pipe with independent instructions to measure its rate:
 * which = 0 POPC, 1 LOP3, 2 IADD3, 3 IMNMX, 4 DFMA, 5 FFMA, 6 IMAD, 7 REDUX.MIN, 8 SHFL, 9-13 packed 16-bit min/max,
 * SEL, PRMT, 14 FFMA2 (fma.rn.f32x2), 15-19 FFMA2 mixed with FFMA / IADD3 (one group counts as one instruction).
 * Launches ctas_per_sm*SMs CTAs of 256 threads doing `iters` x 64 instructions per
 * thread; *ops_out = total thread-level instructions executed (the caller times it). */
int b2s_pipe_microbench(int which, int iters, int ctas_per_sm, double* ops_out, uint32_t* sink,
                        void* stream);

/* Measurement: enable = 1 / 0 switches a CUDA-event pair around the tcgen05 Hamming kernel
 * proper (without the operand pre-pass) on and off, enable < 0 leaves it as it is; if last_ms
 * != NULL it receives the duration of the most recent timed launch (waits for it), -1 if none. */
int b2s_hamming_kernel_timing(int enable, float* last_ms);

/* Raw tcgen05.mma kind::i8 rate: every SM issues iters x 8 MMAs (M=128, N=n_dim in
 * {128,256}, K=32) from shared memory with no epilogue; *macs_out = int8 MACs issued. */
int b2s_mma_microbench(int iters, int n_dim, double* macs_out, void* stream);
/* TMEM -> register read bandwidth: every SM reads its 128 x 512 x 4 B of TMEM `iters` times
 * with `warps` (4, 8 or 16) warps issuing tcgen05.ld 32x32b.x32; *bytes_out = bytes read. */
int b2s_tmem_microbench(int iters, int warps, double* bytes_out, uint32_t* sink, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B2S_H_ */
