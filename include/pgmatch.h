/*
 * pgmatch.h -- C ABI of libpgmatch.so: B200 (sm_100a) descriptor matching for
 * Takatsuka-Mark/Photogrammetry.
 *
 * This is the drop-in boundary for ONE reference path:
 *
 *   List<KeypointPair> KeypointMatching.MatchKeypoints(List<Keypoint>, List<Keypoint>)
 *       dotnet_src/ImageProcessing/KeypointMatching.cs:14-69   (+ CountOnes :71-82)
 *   called from dotnet_src/Photogrammetry/TestService.cs:96
 *
 * The reference has no native code and no FFI; the entry points below are
 * what a P/Invoke ([LibraryImport]) binding of that method would bind (see
 * INTEGRATION.md and dotnet/GpuKeypointMatching.cs).  Everything is
 * `extern "C"`, blittable: plain pointers, sizes, no C++/torch types.
 *
 * Conventions
 *  - Descriptors: uint8[n][stride_bytes], the little-endian bytes of the
 *    non-negative BigInteger `Keypoint.BriefDescriptor`
 *    (dotnet_src/ImageProcessing.Abstractions/Keypoint.cs:14,29-57), i.e.
 *    BigInteger.ToByteArray(isUnsigned: true, isBigEndian: false) copied into
 *    a zero-filled slot.  stride_bytes is a multiple of 16 and
 *    8*stride_bytes >= desc_bits; 1 <= desc_bits <= 512; bits at positions
 *    >= desc_bits must be zero.
 *  - Matches: SoA int32 arrays (query index, train index, distance) standing
 *    for KeypointPair {Keypoint1, Keypoint2, Distance}
 *    (dotnet_src/ImageProcessing.Abstractions/KeypointPair.cs:3-8); the caller
 *    rebuilds object references by indexing its own input lists.
 *  - Every function returns PGM_OK (0) or a negative pgm_status; no exception
 *    crosses the ABI.  pgm_last_error(h) gives the text for the last failure.
 *  - The caller owns every buffer it passes.  Host-buffer entry points copy
 *    H2D/D2H synchronously with respect to the call and retain no caller
 *    pointer after return.  `_dev` entry points take device pointers on the
 *    handle's device and enqueue on the handle's stream WITHOUT a final
 *    synchronize unless stated otherwise.
 *  - One handle = one device + one stream; calls on one handle are serialised
 *    by an internal mutex; different handles may be used concurrently.
 *  - n1, n2 < 2^20 (1 048 576) per pair: match keys pack (distance, index)
 *    into 32 bits so that an integer min implements the reference's
 *    (distance, query index, train index) tie-break (KeypointMatching.cs:44-54).
 */
#ifndef PGMATCH_H
#define PGMATCH_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PGM_VERSION 100 /* 0.1.0 */

typedef enum pgm_status {
    PGM_OK = 0,
    PGM_E_INVALID_ARG = -1,
    PGM_E_CAPACITY = -2,    /* output buffer too small */
    PGM_E_CUDA = -3,        /* a CUDA runtime call failed; see pgm_last_error */
    PGM_E_NCCL = -4,        /* pgm_multi_*: NCCL could not be loaded, or a collective / communicator call failed */
    PGM_E_EMPTY_TRAIN = -5, /* n1 > 0 and n2 == 0: the reference throws
                               ArgumentOutOfRangeException at KeypointMatching.cs:61 */
    PGM_E_NOMEM = -6,
    PGM_E_NO_DEVICE = -7    /* no usable sm_100 device: there is NO CPU fallback */
} pgm_status;

/* pgm_match_* flags */
#define PGM_FLAG_REFERENCE_COMPAT_TAIL 0x1u /* when n1 > n2 append the reference's n1-n2
                                               (0, 0, int.MaxValue) triples
                                               (KeypointMatching.cs:38-42,57-62) */
#define PGM_TAIL_DISTANCE 2147483647

typedef struct pgm_handle pgm_handle;

/* Counters of the last match call on a handle (diagnostics / bench). */
typedef struct pgm_stats {
    int32_t rounds;            /* mutual-nearest-neighbour rounds run on the grid */
    int32_t kernel_launches;   /* kernels launched by the call */
    int32_t host_syncs;        /* stream synchronisations inside the call */
    int32_t pairs;             /* image pairs processed */
    int64_t distance_evals;    /* sum over pairs of n1*n2 (each (i,j) counted once) */
    int64_t evals_computed;    /* XOR+popcount evaluations actually executed (all rounds) */
    int64_t matched;           /* real (non-tail) triples produced */
    int64_t h2d_bytes;
    int64_t d2h_bytes;
} pgm_stats;

int pgm_version(void);
const char *pgm_status_string(int status);

/* Creates a matcher bound to CUDA device `device_ordinal` (own stream, own
 * scratch).  Fails with PGM_E_NO_DEVICE when the device is absent or is not
 * compute capability 10.x -- there is no fallback path. */
int pgm_create(int device_ordinal, pgm_handle **out);
int pgm_destroy(pgm_handle *h);
const char *pgm_last_error(pgm_handle *h);
/* Borrow a caller-owned cudaStream_t (e.g. a torch stream) for all subsequent
 * work of this handle; NULL restores the handle's own stream.  To run on the legacy default
 * stream pass cudaStreamLegacy ((cudaStream_t)0x1), not 0. */
int pgm_set_stream(pgm_handle *h, void *cuda_stream);
/* Page-locked host memory for callers that want the host-buffer entry points to DMA straight out of /
 * into their arrays (a C# caller pins with `fixed` only against the GC, not against paging): buffers
 * from pgm_host_alloc (or any cudaHostAlloc / cudaHostRegister memory) are recognised and copied
 * without the internal staging pass; pageable buffers keep working and are staged. */
int pgm_host_alloc(size_t bytes, void **out);
int pgm_host_free(void *p);
int pgm_synchronize(pgm_handle *h);
/* Statistics of the last call.  After an asynchronous (_dev) call on a few pairs the round / evaluation counts still sit
 * on the device: the function then synchronises the handle's stream and fetches them (nothing is copied per call). */
int pgm_get_stats(pgm_handle *h, pgm_stats *out);

/* ---- MatchKeypoints (KeypointMatching.cs:14-69) -------------------------
 * Full Hamming matrix + greedy global one-to-one assignment, bit-exact with
 * the reference including output order ((distance, i, j) ascending) and, with
 * PGM_FLAG_REFERENCE_COMPAT_TAIL, the degenerate tail.
 * Writes *out_count triples: n1 with the tail flag, min(n1,n2) without.
 * capacity must be >= that count.  n1 == 0 -> 0 triples.  n2 == 0 < n1 ->
 * PGM_E_EMPTY_TRAIN. */
int pgm_match_hamming_greedy(pgm_handle *h,
                             const uint8_t *q, int32_t n1,
                             const uint8_t *t, int32_t n2,
                             int32_t desc_bits, int32_t stride_bytes,
                             int32_t *out_qi, int32_t *out_tj, int32_t *out_dist,
                             int32_t capacity, int32_t *out_count, uint32_t flags);

/* Same, every pointer except out_count is DEVICE memory; out_count (host) is
 * computed from n1/n2/flags.  Asynchronous on the handle's stream except for
 * the rare internal synchronisations counted in pgm_stats.host_syncs. */
int pgm_match_hamming_greedy_dev(pgm_handle *h,
                                 const uint8_t *d_q, int32_t n1,
                                 const uint8_t *d_t, int32_t n2,
                                 int32_t desc_bits, int32_t stride_bytes,
                                 int32_t *d_out_qi, int32_t *d_out_tj, int32_t *d_out_dist,
                                 int32_t capacity, int32_t *out_count, uint32_t flags);

/* ---- many image pairs in one call (all-pairs / consecutive-frame modes) --
 * all_desc: uint8[image_offsets[n_images]][stride_bytes], image k owning rows
 * [image_offsets[k], image_offsets[k+1]).  pair_list: int32[n_pairs][2] =
 * (query image, train image).  Outputs are packed in pair order: pair p's
 * triples start at  sum_{p' < p} n1(p')  (the exclusive prefix sum of the
 * query-image sizes) and out_counts[p] of them are valid (n1(p) with the tail
 * flag, min(n1,n2) without; unused slots are filled with -1).  capacity (in
 * triples) must be >= sum_p n1(p).  A pair with an empty train image and a
 * non-empty query image fails the call with PGM_E_EMPTY_TRAIN.  Each pair is
 * matched exactly as pgm_match_hamming_greedy would match it. */
int pgm_match_pairs_batch(pgm_handle *h,
                          const uint8_t *all_desc, const int64_t *image_offsets, int32_t n_images,
                          const int32_t *pair_list, int32_t n_pairs,
                          int32_t desc_bits, int32_t stride_bytes,
                          int32_t *out_qi, int32_t *out_tj, int32_t *out_dist,
                          int64_t capacity, int32_t *out_counts, uint32_t flags);

/* Same with all_desc and the three output arrays in DEVICE memory;
 * image_offsets, pair_list and out_counts stay on the host. */
int pgm_match_pairs_batch_dev(pgm_handle *h,
                              const uint8_t *d_all_desc, const int64_t *image_offsets, int32_t n_images,
                              const int32_t *pair_list, int32_t n_pairs,
                              int32_t desc_bits, int32_t stride_bytes,
                              int32_t *d_out_qi, int32_t *d_out_tj, int32_t *d_out_dist,
                              int64_t capacity, int32_t *out_counts, uint32_t flags);

/* ---- nearest / second-nearest neighbour (north_star extension) ----------
 * Per query i: the best and second-best train index under the (distance, j)
 * order, -1 where absent.  Column 0/1 of the rows that
 * python_src/photogrammetry/image_processing/keypoint_matching.py:7-33
 * returns (up to its unspecified tie order). */
int pgm_knn2_hamming(pgm_handle *h,
                     const uint8_t *q, int32_t n1, const uint8_t *t, int32_t n2,
                     int32_t desc_bits, int32_t stride_bytes,
                     int32_t *best_j, int32_t *best_d, int32_t *second_j, int32_t *second_d);
int pgm_knn2_hamming_dev(pgm_handle *h,
                         const uint8_t *d_q, int32_t n1, const uint8_t *d_t, int32_t n2,
                         int32_t desc_bits, int32_t stride_bytes,
                         int32_t *d_best_j, int32_t *d_best_d, int32_t *d_second_j, int32_t *d_second_d);

/* ---- train-sharded nearest neighbours: the "top-2 merge" (north_star; SURVEY.md 8e) ----
 * A single huge pair whose train set is split over G ranks: every rank runs
 * pgm_knn2_hamming_dev on (all queries x its train slice), packs the result with
 * pgm_pack_top2_keys_dev (key = distance << 20 | (local j + index_offset), 0x7F7F7F7F where
 * absent: integer order == the (distance, j) order, positive as int32), exchanges the
 * [2][n] key arrays with ONE all-gather (NCCL over NVLink, done by the caller), and
 * pgm_merge_top2_dev picks the two smallest of the 2G keys of every query: the result is
 * bit-identical to pgm_knn2_hamming_dev on the unsharded train set.
 * d_keys of pgm_merge_top2_dev: int32[n_shards][2][n]. */
int pgm_pack_top2_keys_dev(pgm_handle *h, const int32_t *d_best_j, const int32_t *d_best_d,
                           const int32_t *d_second_j, const int32_t *d_second_d, int32_t n,
                           int32_t index_offset, int32_t *d_keys);
int pgm_merge_top2_dev(pgm_handle *h, const int32_t *d_keys, int32_t n_shards, int32_t n,
                       int32_t *d_best_j, int32_t *d_best_d, int32_t *d_second_j, int32_t *d_second_d);

/* The filter of pgm_match_ratio_crosscheck on device-resident knn2 results (all pointers
 * device memory except out_count): d_col_best_i[n2] = best query of every train row under
 * (distance, i) (ignored unless cross_check).  Writes the kept (i, j1, d1) triples in
 * ascending i and their number. */
int pgm_ratio_crosscheck_filter_dev(pgm_handle *h, int32_t n1, int32_t n2,
                                    const int32_t *d_best_j, const int32_t *d_best_d, const int32_t *d_second_d,
                                    const int32_t *d_col_best_i, float ratio, int32_t cross_check, int32_t max_dist,
                                    int32_t *d_out_qi, int32_t *d_out_tj, int32_t *d_out_dist, int32_t *out_count);

/* ---- match_keypoints of the Python generation (keypoint_matching.py:7-33) ---
 * out: int64[n1][n2][2] = (idx2, dist) with every row sorted by dist -- the array
 * `match_keypoints(keypoints1, keypoints2, hamming_threshold)` returns (the
 * threshold argument is unused upstream).  numpy's default argsort is not stable,
 * so the order among equal distances is unspecified upstream; this library
 * returns the stable (dist, idx2) order. */
int pgm_match_keypoints_sorted(pgm_handle *h,
                               const uint8_t *q, int32_t n1, const uint8_t *t, int32_t n2,
                               int32_t desc_bits, int32_t stride_bytes, int64_t *out);
int pgm_match_keypoints_sorted_dev(pgm_handle *h,
                                   const uint8_t *d_q, int32_t n1, const uint8_t *d_t, int32_t n2,
                                   int32_t desc_bits, int32_t stride_bytes, int64_t *d_out);

/* Ratio test + mutual cross-check (north_star extension; not in the
 * reference).  Keep (i, j1, d1) iff
 *   [n2 < 2 or ratio <= 0 or (float)d1 < ratio * (float)d2]  and
 *   [!cross_check or the best query of train j1 under (distance, i) is i] and
 *   [max_dist < 0 or d1 <= max_dist]     (python_src/scripts/match_keypoints.py:126-128)
 * Output ordered by i ascending. */
int pgm_match_ratio_crosscheck(pgm_handle *h,
                               const uint8_t *q, int32_t n1, const uint8_t *t, int32_t n2,
                               int32_t desc_bits, int32_t stride_bytes,
                               float ratio, int32_t cross_check, int32_t max_dist,
                               int32_t *out_qi, int32_t *out_tj, int32_t *out_dist,
                               int32_t capacity, int32_t *out_count);

/* ---- float descriptors: squared-L2 nearest / second nearest (north_star extension) --
 * q: float[n1][dim], t: float[n2][dim], 1 <= dim <= 128.  The reference has no float
 * descriptor; semantics are those of oracle/pgm_oracle.c orc_l2_knn2: exact squared
 * Euclidean distance, best and second-best train index under (distance, index), -1 where
 * absent.  Computed as ||q||^2 + ||t||^2 - 2 q.t on the tcgen05 tensor cores (fp32
 * accumulation in TMEM) to RANK candidates, then every candidate inside the error band of the
 * ranking is re-evaluated exactly in fp32: distances are exact to fp32 rounding (<= 1e-5
 * relative); indices equal the oracle's except where two candidates' exact fp32 distances
 * differ only by summation order (near-ties).  Ranking operands: one fp16 term per component
 * under a global power-of-two scale (band 2^-9 (3|q|^2 + 2d)); a query whose band could hide a
 * train row that the kernel's per-column-group top-8 lists dropped is recomputed exhaustively on
 * the device, so the guarantee does not depend on the data (pgm_l2_last_fallback_rows counts
 * them).  n1 <= 128 ranks with a three-term bf16 split (three GEMM passes) instead.
 * d_debug_dist (optional, device float[n1][n2]) receives the
 * approximate GEMM distances. */
int pgm_knn2_l2(pgm_handle *h, const float *q, int32_t n1, const float *t, int32_t n2, int32_t dim,
                int32_t *best_j, float *best_d, int32_t *second_j, float *second_d);
int pgm_knn2_l2_dev(pgm_handle *h, const float *d_q, int32_t n1, const float *d_t, int32_t n2, int32_t dim,
                    int32_t *d_best_j, float *d_best_d, int32_t *d_second_j, float *d_second_d,
                    float *d_debug_dist);
/* Rows of the handle's last float call that took the exhaustive fallback (synchronises the stream);
 * -1 if that call did not run in the fp16 ranking mode.  After a batch call below: the call's
 * total over all chunks and, with cross-check, both directions. */
int pgm_l2_last_fallback_rows(pgm_handle *h);

/* ---- float descriptors, many image pairs per call ---------------------------------------
 * Layout as pgm_match_ratio_crosscheck_pairs_batch_dev: d_all_desc is device float[rows][dim],
 * 1 <= dim <= 128; image_offsets[n_images + 1] and pair_list[n_pairs][2] (query image, train
 * image) are host arrays; pair p's rows start at the sum of the query-image sizes n1 of the pairs
 * before it.  0 <= n1, n2 < 2^20 per pair.  PGM_E_INVALID_ARG: bad dim, pair index, image size or
 * null pointer; PGM_E_CAPACITY: capacity < sum of n1.
 *
 * pgm_knn2_l2_pairs_batch_dev: per pair the contract of pgm_knn2_l2_dev (squared L2, best and
 * second best under (distance, train index), index -1 and distance -1.0 where absent); a pair
 * with n1 = 0 writes nothing.  Every pair, n1 <= 128 included, ranks on the CTA-pair fp16 path
 * (certified band + exhaustive fallback), so a pair with n1 > 128 gets bit-identically the
 * pgm_knn2_l2_dev result.  The fp16 operands use one power-of-two scale per chunk of pairs, from
 * max |x| over the images the chunk references: results do not depend on it, but an image far
 * smaller in magnitude than the chunk's largest goes subnormal in fp16 and its rows take the
 * exhaustive fallback -- correct, slower.
 *
 * pgm_match_l2_ratio_crosscheck_pairs_batch_dev: keeps (i, j1, d1) of a pair iff
 *   n2 < 2 || ratio <= 0 || d1 < (ratio * ratio) * d2   (fp32, ratio * ratio rounded to fp32 first:
 *                                                        Lowe's ratio on Euclidean distances),
 *   !cross_check || the best query of train row j1 under (distance, query index) is i,
 *   max_sq_dist < 0 || d1 <= max_sq_dist,
 * on the squared distances knn2 reports.  Output in ascending i at the pair's rows; out_counts[p]
 * = kept triples, no slot beyond a pair's count is written.  Every exact distance is a per-lane
 * sum of fmaf((q - t), (q - t), .) and a butterfly, bit-symmetric in q and t, so the column best
 * of pair (a, b) is the row best of (b, a): with cross_check the library runs the top-2 pass of
 * the reversed pairs too, in the same chunk -- twice the GEMM work (pgm_stats.evals_computed =
 * 2 distance_evals). */
int pgm_knn2_l2_pairs_batch_dev(pgm_handle *h, const float *d_all_desc, const int64_t *image_offsets, int32_t n_images,
                                const int32_t *pair_list, int32_t n_pairs, int32_t dim,
                                int32_t *d_best_j, float *d_best_d, int32_t *d_second_j, float *d_second_d,
                                int64_t capacity);
int pgm_match_l2_ratio_crosscheck_pairs_batch_dev(pgm_handle *h, const float *d_all_desc, const int64_t *image_offsets,
                                int32_t n_images, const int32_t *pair_list, int32_t n_pairs, int32_t dim,
                                float ratio, int32_t cross_check, float max_sq_dist,
                                int32_t *d_out_qi, int32_t *d_out_tj, float *d_out_dist,
                                int64_t capacity, int32_t *out_counts);

/* ---- the producer of the matcher's inputs (SURVEY.md section 8, rows f1/f2) ----------
 * gray: float[height][width] = Grayscale.K (Images.Abstractions/Pixels/Grayscale.cs:19-23),
 * pixel (x, y) at gray[y*width + x].
 *
 * pgm_fast_detect    KeypointDetection.Detect (KeypointDetection.cs:42-133): FAST-12 on the
 *                    reference's ring table (typo in its last entry included); keypoints in the
 *                    reference's row-major order, out_xy[k] = (x, y), out_score[k] = FastScore.
 *                    *out_count always receives the number found; PGM_E_CAPACITY if > capacity.
 * pgm_brief_describe Keypoint.GetBriefDescriptor (Keypoint.cs:29-57): pairs int32[n_pairs][4] =
 *                    (dx1, dy1, dx2, dy2); first pair = most significant bit; descriptors in the
 *                    matcher's row layout (desc_bits = n_pairs).
 * pgm_nms            RedundantKeypointEliminator.EliminateRedundantKeypoints
 *                    (RedundantKeypointEliminator.cs:16-39): out_kept = indices of the survivors in
 *                    the reference's output order (stable by FastScore descending).
 *
 * flags: 0 = the C# generation.  PGM_FLAG_PYTHON_GENERATION selects the older Python generation's
 * variants of the same two steps, which the reference tree can execute and therefore pins with golden
 * vectors: FASTKeypointDetector (python_src/photogrammetry/image_processing/keypoint_detection.py:12-115,
 * correct ring entry 15, same segment test) and KeyPoint._brief_descriptor
 * (python_src/photogrammetry/models/keypoint.py:32-50: pair idx sets bit idx, LSB first). */
#define PGM_FLAG_PYTHON_GENERATION 0x2u
int pgm_fast_detect(pgm_handle *h, const float *gray, int32_t width, int32_t height, float threshold,
                    uint32_t flags, int32_t *out_xy, int32_t *out_score, int32_t capacity, int32_t *out_count);
int pgm_brief_describe(pgm_handle *h, const float *gray, int32_t width, int32_t height, const int32_t *xy,
                       int32_t n, const int32_t *pairs, int32_t n_pairs, int32_t stride_bytes, uint32_t flags,
                       uint8_t *out_desc);
int pgm_nms(pgm_handle *h, const int32_t *xy, const int32_t *score, int32_t n, int32_t radius,
            int32_t *out_kept, int32_t *out_count);

/* The same chain on a DEVICE-resident image, descriptors never leaving the GPU: FAST-12
 * (KeypointDetection.Detect) -> optionally RedundantKeypointEliminator (nms_radius >= 0; < 0 skips it) -> BRIEF
 * of the survivors, in the reference's output order.  d_gray, d_out_xy[capacity][2], d_out_score[capacity],
 * d_out_desc[capacity][stride_bytes] are device memory (d_out_desc is directly a matcher operand for
 * pgm_match_hamming_greedy_dev / pgm_match_pairs_batch_dev); `pairs` (int32[n_pairs][4]) and out_count are host
 * memory.  PGM_E_CAPACITY with *out_count = the number of keypoints when they do not fit. */
int pgm_detect_describe_dev(pgm_handle *h, const float *d_gray, int32_t width, int32_t height, float threshold,
                            int32_t nms_radius, const int32_t *pairs, int32_t n_pairs, int32_t stride_bytes,
                            uint32_t flags, int32_t *d_out_xy, int32_t *d_out_score, uint8_t *d_out_desc,
                            int32_t capacity, int32_t *out_count);

/* The batched form for a frame sequence (BASELINE configs[2]; the step the reference runs per frame,
 * TestService.cs:85-91, KeypointDetection.Detect KeypointDetection.cs:42-63): n_images device-resident images of one
 * size, d_gray[n_images][height][width].  Image k's keypoints go to its own `capacity` slots --
 * d_out_xy[n_images][capacity][2], d_out_score[n_images][capacity], d_out_desc[n_images][capacity][stride_bytes] --
 * and its keypoint count to d_out_counts[k] (device); a count above `capacity` means the list was truncated.
 * Nothing is read back between the images: the call enqueues six kernels for the whole batch.  out_counts
 * (host, int32[n_images]) may be NULL, in which case the call does not synchronise at all.  No NMS in this form:
 * pgm_detect_nms_describe_batch_dev below is the batched chain with it. */
int pgm_detect_describe_batch_dev(pgm_handle *h, const float *d_gray, int32_t n_images, int32_t width, int32_t height,
                                  float threshold, const int32_t *pairs, int32_t n_pairs, int32_t stride_bytes,
                                  uint32_t flags, int32_t *d_out_xy, int32_t *d_out_score, uint8_t *d_out_desc,
                                  int32_t capacity, int32_t *d_out_counts, int32_t *out_counts);

/* The batched form WITH non-maximum suppression: FAST-12 -> RedundantKeypointEliminator (radius nms_radius >= 0)
 * -> BRIEF of the survivors, for n_images device-resident images of one size (the C# pipeline's per-frame chain,
 * BuildKeypointDetectorPipeline, whose denoised keypoints TestService.cs:94-95 matches).  Arguments and output layout
 * are those of pgm_detect_describe_batch_dev, plus nms_radius.
 *  - For every image k and both generations the result equals pgm_detect_describe_dev(image k, threshold,
 *    nms_radius, ...) bit for bit: survivors' (x, y), FastScore and descriptor bytes, in the reference's output
 *    order (stable by FastScore descending).  NMS always runs over the image's full FAST list.
 *  - d_out_counts[k] (device) = the number of survivors of image k.  A count above `capacity` means only the first
 *    `capacity` survivors were written.  No slot at or beyond min(count, capacity) of an image is written.
 *    out_counts (host, int32[n_images]) may be NULL.
 *  - Synchronisation: one, the read-back of the per-image FAST totals that sizes the scratch (host_syncs = 1, 2 with
 *    out_counts).  Every NMS round of every image runs on the device; the number of kernel launches depends neither
 *    on the rounds nor on n_images.
 *  - Refusals: PGM_E_INVALID_ARG for nms_radius < 0 (use pgm_detect_describe_batch_dev without NMS) and for every
 *    argument pgm_detect_describe_batch_dev refuses; PGM_E_CAPACITY when the batch's FAST keypoints together exceed
 *    2^31 - 1, after the read-back and before any later kernel runs.  n_images == 0 does nothing. */
int pgm_detect_nms_describe_batch_dev(pgm_handle *h, const float *d_gray, int32_t n_images, int32_t width,
                                      int32_t height, float threshold, int32_t nms_radius, const int32_t *pairs,
                                      int32_t n_pairs, int32_t stride_bytes, uint32_t flags, int32_t *d_out_xy,
                                      int32_t *d_out_score, uint8_t *d_out_desc, int32_t capacity,
                                      int32_t *d_out_counts, int32_t *out_counts);

/* The batched chain for images of ANY sizes, with or without NMS: a photogrammetry capture is an unordered set of
 * photos (portrait next to landscape, mixed cameras and crops), and upstream detects each at its own size
 * (KeypointDetection.Detect takes a Matrix<Grayscale> of any dimensions).  Image k is row-major widths[k] x
 * heights[k] at d_gray + pixel_offsets[k] (device memory); pixel_offsets (int64[n_images + 1], the delimiter
 * convention of the matchers' image_offsets), widths and heights (int32[n_images]) are host memory.  Only the declared
 * pixels are read: gaps between the images may hold anything.  nms_radius < 0 skips NMS.
 *  - Output layout, flags (both generations) and counts are those of pgm_detect_describe_batch_dev (nms_radius < 0)
 *    and pgm_detect_nms_describe_batch_dev (nms_radius >= 0): image k owns `capacity` slots, d_out_counts[k] (device)
 *    can be above `capacity`, and no slot at or beyond min(count, capacity) of an image is written.
 *  - For every image k the result equals pgm_detect_describe_dev(image k, widths[k], heights[k], threshold,
 *    nms_radius, ...) bit for bit: (x, y), FastScore, descriptor bytes and order.  Images below 7 pixels on a side
 *    have no FAST interior and count 0.
 *  - Synchronisation and launches are those of the uniform forms, whatever n_images and the mix of sizes:
 *    host_syncs 0 without NMS and 1 with it, plus 1 with out_counts; 6 kernel launches without NMS, 11 with it.
 *  - Refusals: PGM_E_INVALID_ARG for a null pointer, n_images outside 0..65535, a width or height outside
 *    1..65535, pixel_offsets[0] < 0, pixel_offsets[k + 1] < pixel_offsets[k] + widths[k] * heights[k],
 *    capacity < 1 and every descriptor format pgm_detect_describe_batch_dev refuses; PGM_E_CAPACITY when the set's
 *    FAST keypoints together exceed 2^31 - 1 (NMS only; after the read-back and before any later kernel runs).
 *    n_images == 0 does nothing. */
int pgm_detect_describe_images_batch_dev(pgm_handle *h, const float *d_gray, const int64_t *pixel_offsets,
                                         const int32_t *widths, const int32_t *heights, int32_t n_images,
                                         float threshold, int32_t nms_radius, const int32_t *pairs, int32_t n_pairs,
                                         int32_t stride_bytes, uint32_t flags, int32_t *d_out_xy, int32_t *d_out_score,
                                         uint8_t *d_out_desc, int32_t capacity, int32_t *d_out_counts,
                                         int32_t *out_counts);

/* ---- the consumer of the match list (SURVEY.md section 8, row f3) --------------------
 * pgm_ransac_score: the scoring loops of CameraPoseEstimation.GetFundamentalMatrix
 * (ImageProcessing/CameraPoseEstimation.cs:41-88).  F: n_hyp row-major 3x3 float matrices (the estimates of the
 * sampled subsets, :44); valid[k] == 0 skips hypothesis k like upstream's rank test (:46-51), NULL = all valid;
 * xy1 / xy2: int32[n][2] = Keypoint1 / Keypoint2 coordinates of every pair.  A pair is an inlier of F when
 * (F . (x2, y2, 1)) . (x1, y1, 1) <= threshold (:66-73, signed as upstream).  out_counts[k] = inliers of
 * hypothesis k (-1 if skipped); *out_best = the first hypothesis with the largest positive count (:79-84), -1
 * if none (upstream throws, :87-88); out_best_mask[p] = 1 for the winner's inliers (its bestSample).  Any
 * output pointer may be NULL. */
int pgm_ransac_score(pgm_handle *h, const float *F, const uint8_t *valid, int32_t n_hyp, const int32_t *xy1,
                     const int32_t *xy2, int32_t n, float threshold, int32_t *out_counts, int32_t *out_best,
                     uint8_t *out_best_mask);

/* pgm_ransac_fundamental_pairs_batch_dev: GetFundamentalMatrix(list, n_samples, pairs_per_sample, threshold)
 * (CameraPoseEstimation.cs:26-94, as the host mirror camera_pose_estimation.py restates it) for MANY match lists in one
 * call, on the device, with no read-back (pgm_stats.host_syncs == 0).
 *  - Inputs: d_all_xy device int32[rows][2] = (x, y) of every keypoint, image k at rows [image_offsets[k],
 *    image_offsets[k + 1]) (host int64[n_images + 1]); pair_list host int32[n_pairs][2] = (image a, image b); pair p owns
 *    the match slots [match_starts[p], match_starts[p] + match_counts[p]) (host arrays) of d_match_qi / d_match_tj
 *    (device int32[capacity]): Keypoint1 = row image_offsets[a] + qi of d_all_xy, Keypoint2 = row image_offsets[b] + tj.
 *    That is the output layout of the batch matchers (greedy tail triples included).  The indices must lie inside their
 *    images (a precondition; the -DPGM_CHECKED build asserts it).
 *  - Per pair, with P = pairs_per_sample (8..64) and S = n_samples (>= 1):
 *    count < P: out_best = -2 (upstream throws, :29-32), inliers 0, F zeros, mask slots 0.
 *    Hypothesis s draws P distinct indices in [0, count) with Floyd's algorithm, sorted ascending afterwards.  Draw t
 *    (t = 0..P-1, j = count - P + t) is r = (u * (j + 1)) >> 32 with the 32-bit
 *        u = splitmix64(key ^ ((uint64)s << 32 | t)) >> 32,   key = splitmix64(seed ^ splitmix64((uint64)(uint32)a << 32 | (uint32)b)),
 *        splitmix64(z): z += 0x9E3779B97F4A7C15; z = (z ^ z >> 30) * 0xBF58476D1CE4E5B9; z = (z ^ z >> 27) * 0x94D049BB133111EB;
 *                       return z ^ z >> 31;
 *    Floyd: if r is already drawn, j is taken instead.  The key depends on the image pair, not on its position in the list.
 *    Estimate: centroids in double rounded to float32, c = fl32(x - cx), rows of A = float32 (c1x c2x, c1x c2y, c1x,
 *    c1y c2x, c1y c2y, c1y, c2x, c2y, 1); the null vector v of A in fp64 (Givens QR, one-sided Jacobi), its largest-
 *    magnitude component positive (lowest index on exact ties; components equal up to rounding, as in the skew-symmetric
 *    F of a pure translation, are ordered by the fp64 result); F0[i][j] = v[3 j + i]; F = T2^T F0 T1 in fp64, rounded once to
 *    float32 (row-major).  With PGM_FLAG_RANSAC_RANK_TEST a hypothesis is skipped (count -1) unless #{sigma_k > 3
 *    ulp_f32(sigma_0)} == 2, sigma the fp64 singular values of the float32 F (:46-51).  Scoring as pgm_ransac_score.
 *    out_best = the first s with the largest positive count, else -1 (upstream throws, :87-88); out_inliers and
 *    out_F (float32[n_pairs][9]) are the winner's (0 and zeros without one); d_out_mask = 1 at the winner's inlier slots,
 *    0 at the pair's other slots.  No slot outside a pair's [start, start + count) is written.
 *  - d_hyp_F (float[n_pairs][S][9]) and d_hyp_counts (int32[n_pairs][S]) are optional diagnostics (NULL in production):
 *    every hypothesis' F and count (-1 if skipped); a pair with count < P leaves its rows unwritten.
 *  - PGM_E_INVALID_ARG: P outside 8..64, S < 1, unknown flags, a bad pair or image index, a null pointer, a negative
 *    count, start < 0, start + count > capacity, matches of an empty image. */
#define PGM_FLAG_RANSAC_RANK_TEST 0x4u   /* apply upstream's rank gate (CameraPoseEstimation.cs:46-51) */
int pgm_ransac_fundamental_pairs_batch_dev(pgm_handle *h,
        const int32_t *d_all_xy, const int64_t *image_offsets, int32_t n_images,
        const int32_t *pair_list, int32_t n_pairs,
        const int32_t *d_match_qi, const int32_t *d_match_tj,
        const int64_t *match_starts, const int32_t *match_counts,
        int32_t n_samples, int32_t pairs_per_sample, float threshold, uint64_t seed, uint32_t flags,
        int32_t *d_out_best, int32_t *d_out_inliers, float *d_out_F,
        uint8_t *d_out_mask, int64_t capacity,
        float *d_hyp_F, int32_t *d_hyp_counts);

/* Nearest neighbour + ratio test + mutual cross-check (+ optional distance bound) for MANY small pairs in one launch --
 * the consecutive frames of a sequence (BASELINE configs[2]; per pair the same result as pgm_match_ratio_crosscheck, which
 * extends the nearest-neighbour-within-a-threshold use of python_src/scripts/match_keypoints.py:112-134).  Layout as for
 * pgm_match_pairs_batch_dev: d_all_desc holds every image's descriptors, image_offsets[n_images + 1] (host) delimits
 * them, pair_list[n_pairs][2] (host) names the pairs; pair p's kept triples (ascending query index) start at the sum
 * of the query sizes of the pairs before it, out_counts[p] (host) says how many.  One CTA per pair with both descriptor
 * sets in shared memory: (n1 + n2) * stride_bytes + 4 * n2 + 16 must not exceed 200 KB (204 800 bytes), else
 * PGM_E_INVALID_ARG.  Larger pairs: pgm_match_ratio_crosscheck_pairs_batch_dev, same arguments. */
int pgm_match_ratio_crosscheck_batch_dev(pgm_handle *h, const uint8_t *d_all_desc, const int64_t *image_offsets,
                                         int32_t n_images, const int32_t *pair_list, int32_t n_pairs, int32_t desc_bits,
                                         int32_t stride_bytes, float ratio, int32_t cross_check, int32_t max_dist,
                                         int32_t *d_out_qi, int32_t *d_out_tj, int32_t *d_out_dist, int64_t capacity,
                                         int32_t *out_counts);

/* The same filter for many pairs of ANY size (0 <= n1, n2 < 2^20; e.g. all pairs of an image set, BASELINE configs[4]),
 * with the arguments, output layout and status codes of pgm_match_ratio_crosscheck_batch_dev.  Per pair the result is
 * bit-identical to pgm_match_ratio_crosscheck on that pair; a pair with n1 == 0 or n2 == 0 keeps nothing.  One fused
 * distance pass gives every query's best and second best train row under (distance, j) and, with cross_check, every
 * train row's best query under (distance, i), so pgm_stats.evals_computed == distance_evals.  The pair list is processed
 * in chunks of at most 4096 pairs and 24 M query + train rows, whose scratch is reused; the call reads back the counts
 * once at the end (pgm_stats.host_syncs == 2) and writes no slot beyond a pair's count. */
int pgm_match_ratio_crosscheck_pairs_batch_dev(pgm_handle *h, const uint8_t *d_all_desc, const int64_t *image_offsets,
                                               int32_t n_images, const int32_t *pair_list, int32_t n_pairs,
                                               int32_t desc_bits, int32_t stride_bytes, float ratio, int32_t cross_check,
                                               int32_t max_dist, int32_t *d_out_qi, int32_t *d_out_tj,
                                               int32_t *d_out_dist, int64_t capacity, int32_t *out_counts);

/* ---- train-sharded single pair (multi-GPU, SURVEY.md section 8e) ----------
 * For ONE huge pair (BASELINE configs[3]: 200k x 200k; the call it shards is MatchKeypoints,
 * KeypointMatching.cs:14-69) every rank holds all n1 queries and a contiguous slice
 * [col_offset, col_offset + n2_local) of the n2_total train descriptors.  Two surfaces:
 *
 * (1) pgm_multi_*: the library owns the communicator -- one pgm_multi per rank (= per handle = per GPU; one process
 *     per GPU, or one thread per GPU inside a process), NCCL over NVLink.  The host distributes the 128-byte id of
 *     pgm_multi_unique_id (made on rank 0) by whatever channel it has; nothing else crosses the ABI.  NCCL is loaded
 *     at run time (dlopen "libnccl.so.2"), so single-GPU users need no NCCL; failures return PGM_E_NCCL.
 *       pgm_multi_match_train_sharded_dev   the greedy matcher; per round ONE min all-reduce of 2 x bound 32-bit keys
 *                                           (bound = live rows, rounded up) and ONE all-gather of the ranks' candidate
 *                                           edges, no host synchronisation per round
 *       pgm_multi_knn2_train_sharded_dev    nearest / second nearest with the top-2 merge: one all-gather of [2][n1]
 *     Both are collective calls: every rank calls them with the same sizes / format / flags.
 *
 * (2) pgm_shard_*: the same steps with the exchanges left to the caller (another transport, or several emulated ranks
 *     on one GPU in the tests):
 *       pgm_shard_create;  pgm_shard_edge_capacity(n1, n2_total, n_ranks, &cap)      (same cap on every rank)
 *       repeat:
 *         pgm_shard_round(shard, x, bound)         local distances + row/column argmin; x[2 * bound] = [R | P]:
 *                                                  R[pos] best key of live row pos over this rank's columns,
 *                                                  P[pos] best key among this rank's columns that chose row pos
 *         x = element-wise MIN of x over the ranks (as int32 or uint32)
 *         pgm_shard_commit(shard, x, bound, edges, cap)    row pos is matched iff R[pos] == P[pos]; edges[1 + cap] (uint64,
 *                                                  count first) = this rank's candidate edges (distance <= the pass's
 *                                                  bound T) whose row and column are still unmatched
 *         edges_all[n_ranks][1 + cap] = all-gather of edges
 *         pgm_shard_finish_round(shard, edges_all, n_ranks, cap, &live_rows, &done)   mutual-best sub-rounds on the sparse
 *                                                  edge list (every rank identically), compaction, next round's plan
 *       until done
 *       pgm_shard_finish                           reference-ordered triples on every rank
 *     bound >= the number of live rows (n1 always works; the value pgm_shard_finish_round returned is the tight one).
 *     Passing NULL for edges / edges_all gives the plain one-accept-per-round behaviour (no second exchange).
 *
 * Exchange keys are (distance << 20 | global train index); "none" is 0x7F7F7F7F, so a signed 32-bit MIN orders them
 * like the reference's (distance, i, j) tie-break.  The result is bit-identical to pgm_match_hamming_greedy on the
 * unsharded pair.  All data pointers are device memory on the handle's device. */
typedef struct pgm_shard pgm_shard;
int pgm_shard_create(pgm_handle *h, const uint8_t *d_q, int32_t n1, const uint8_t *d_t_local, int32_t n2_local,
                     int32_t col_offset, int32_t n2_total, int32_t desc_bits, int32_t stride_bytes, pgm_shard **out);
int pgm_shard_edge_capacity(int32_t n1, int32_t n2_total, int32_t n_ranks, int32_t *out_cap);
int pgm_shard_round(pgm_shard *s, uint32_t *d_x, int32_t bound);
int pgm_shard_commit(pgm_shard *s, const uint32_t *d_x, int32_t bound, uint64_t *d_edges, int32_t edge_cap);
int pgm_shard_finish_round(pgm_shard *s, const uint64_t *d_edges_all, int32_t n_ranks, int32_t edge_cap,
                           int32_t *live_rows, int32_t *done);
int pgm_shard_finish(pgm_shard *s, int32_t *d_out_qi, int32_t *d_out_tj, int32_t *d_out_dist, uint32_t flags,
                     int32_t *out_count, int32_t *out_rounds);
int pgm_shard_destroy(pgm_shard *s);

typedef struct pgm_multi pgm_multi;
int pgm_multi_unique_id(uint8_t *out_id128);
int pgm_multi_create(pgm_handle *h, const uint8_t *id128, int32_t rank, int32_t world, pgm_multi **out);
int pgm_multi_destroy(pgm_multi *m);
int pgm_multi_match_train_sharded_dev(pgm_multi *m, const uint8_t *d_q, int32_t n1, const uint8_t *d_t_local,
                                      int32_t n2_local, int32_t col_offset, int32_t n2_total, int32_t desc_bits,
                                      int32_t stride_bytes, int32_t *d_out_qi, int32_t *d_out_tj, int32_t *d_out_dist,
                                      int32_t capacity, int32_t *out_count, uint32_t flags, int32_t *out_rounds);
int pgm_multi_knn2_train_sharded_dev(pgm_multi *m, const uint8_t *d_q, int32_t n1, const uint8_t *d_t_local,
                                     int32_t n2_local, int32_t col_offset, int32_t desc_bits, int32_t stride_bytes,
                                     int32_t *d_best_j, int32_t *d_best_d, int32_t *d_second_j, int32_t *d_second_d);
/* bytes this rank contributed to collectives, and their number, in the last pgm_multi_* call */
int pgm_multi_get_exchange(pgm_multi *m, int64_t *bytes, int32_t *collectives);

/* ---- measurement helpers -------------------------------------------------
 * Profiling mode brackets every launch of the dominant kernel (the round
 * kernel) with CUDA events on the handle's stream and records how many
 * XOR+popcount evaluations each launch executed.  It adds event records to
 * the stream, so bench.py uses it in a separate pass from the timed steps. */
int pgm_set_profiling(pgm_handle *h, int32_t enabled);
/* Per round-kernel launch of the last greedy call: duration in ms and
 * evaluations executed.  Synchronises the stream. */
int pgm_get_round_profile(pgm_handle *h, float *ms, int64_t *evals, int32_t capacity, int32_t *out_n);

/*
 * Register-only POPC.32 throughput of the device (the roofline denominator
 * for this path: one 256-bit distance = 8 POPC.32).  Runs a saturating
 * micro-benchmark for roughly `millis` ms and reports popc32 results / s. */
int pgm_measure_popc_peak(pgm_handle *h, int32_t millis, double *popc32_per_s,
                          double *lop3_per_s);

#ifdef __cplusplus
}
#endif
#endif /* PGMATCH_H */
