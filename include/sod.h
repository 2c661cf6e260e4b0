/* sod.h — C ABI of libsod_b200.so, the B200 (sm_100a) implementation of the SIFT object-detection
 * hot path of torn8to/sift-based-OD: 2-NN descriptor matching + ratio test, 4-D Hough pose-bin
 * voting, per-bin affine verification.
 *
 * The reference has no FFI: its boundary is the Python call surface (SURVEY.md §8b).  Each entry
 * point below names the reference code it replaces; INTEGRATION.md shows the ctypes binding.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in _host;
 *   - all work is enqueued on `stream` (a cudaStream_t) and is asynchronous; no entry point
 *     synchronises, allocates or frees caller-visible memory;
 *   - return value: 0 = SOD_OK, negative = error; sod_last_error() gives a thread-local message;
 *   - descriptors are unsigned 8-bit, 128 per row, row-major (OpenCV SIFT descriptors are
 *     integer-valued 0..255 stored as float32; sod_pack_u8_from_f32 converts and verifies).
 */
#ifndef SOD_H_
#define SOD_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SOD_OK 0
#define SOD_ERR_INVALID_ARGUMENT (-1)
#define SOD_ERR_CUDA (-2)
#define SOD_ERR_UNSUPPORTED (-3)

#define SOD_DESC_DIM 128  /* bytes per descriptor row */
#define SOD_TILE_ROWS 128 /* database rows per MMA tile */
#define SOD_CQ_TILE_INTS 260 /* int32 per tile in `cq`: 128 norms + 4 chunk minima + 128 original rows */

typedef void* sod_stream_t; /* cudaStream_t */

/* ABI version (major*1000 + minor). */
int sod_version(void);
/* Message for the last error raised on the calling thread ("" if none). */
const char* sod_last_error(void);
/* Number of SMs of the current device (grid sizing; 148 on B200). Negative on error. */
int sod_device_sm_count(void);

/* Measurement hook (bench.py's roofline figures; nothing in the reference): while enabled on the
 * calling thread, every entry point brackets the launches of the stages below with CUDA events on the
 * caller's stream (up to 128 calls per stage between reads; no synchronisation, two event records per
 * stage).  sod_timing_read waits for the recorded events of one stage, writes their durations in
 * milliseconds to ms_host (HOST pointer, oldest first, at most cap), forgets them and returns how many
 * it wrote (negative = error). */
#define SOD_STAGE_MATCH 0        /* match_top2_kernel alone (without the list merge that follows it) */
#define SOD_STAGE_HOUGH_PREP 1   /* pose + counting sort by Hough space */
#define SOD_STAGE_HOUGH_VOTE 2   /* hough_vote_kernel alone */
#define SOD_STAGE_HOUGH_FINISH 3 /* member order, running means, insertion keys */
#define SOD_STAGE_AFFINE 4       /* select + verify kernels */
#define SOD_STAGE_COUNT 5
int sod_timing_enable(int32_t on);
int32_t sod_timing_read(int32_t stage, float* ms_host, int32_t cap);

/* Number of int32 elements of the prepared per-row constants `cq` for a database of n_rows:
 * ceil(n_rows / SOD_TILE_ROWS) * SOD_CQ_TILE_INTS. */
int64_t sod_cq_ints(int64_t n_rows);

/* float32 [n_rows,128] -> u8 [n_rows,128].  *nonint_flag (device int32, caller zeroes it) is set
 * to 1 if any value is not an integer in 0..255 (such a set needs the bf16 path, not built yet).
 * Replaces nothing in the reference; it is the packing step in front of main.py:71. */
int sod_pack_u8_from_f32(const float* src, int64_t n_rows, uint8_t* dst, int32_t* nonint_flag,
                         sod_stream_t stream);

/* K1 (database side): one-time preparation of a database shard for the matcher.
 *   db_sorted [ceil(n/128)*128][128]  the rows re-ordered and zero-padded to whole tiles: every
 *                            tile of 128 rows holds rows of adjacent sum of squares |t|^2 (tiles are
 *                            stored in a scattered order), rows inside a tile by original index;
 *   cq [sod_cq_ints(n_rows)] per tile: (|t|^2 << 8 | column) of its 128 rows (|t|^2 = 0x7FFFFF for
 *                            padding), the minimum |t|^2 of each 32-row chunk (prunes the
 *                            matcher's epilogue) and the original row of every stored row (-1 for
 *                            padding).
 * |t|^2 is the per-row term of |q-t|^2 = |q|^2 + |t|^2 - 2 q.t that OpenCV recomputes per pair in
 * cv::batchDistance (called from main.py:71).  Matching results are reported in ORIGINAL indices;
 * the re-ordering is invisible to callers.  workspace: sod_db_prepare_workspace_bytes(n_rows),
 * 256-byte aligned.  Uses cub::DeviceRadixSort for the one-time sort. */
size_t sod_db_prepare_workspace_bytes(int64_t n_rows);
int sod_db_prepare(const uint8_t* db, int64_t n_rows, uint8_t* db_sorted, int32_t* cq, void* workspace,
                   size_t workspace_bytes, sod_stream_t stream);

/* K1 (query side).  qn[i] = sum_k q[i][k]^2. */
int sod_query_prepare(const uint8_t* q, int64_t n_rows, int32_t* qn, sod_stream_t stream);

/* Bytes of scratch sod_match_top2 needs for these sizes on the current device. */
size_t sod_match_workspace_bytes(int64_t n_query, int64_t n_db);

/* K2.  For every query row the two database rows with the smallest squared L2 distance, ascending,
 * ties -> lowest index: the result of cv2.BFMatcher().knnMatch(des_query, des, k=2)
 * (main.py:70-71) with exact integer distances.  db_sorted / cq come from sod_db_prepare.
 * out_idx[i][j] = db_index_base + ORIGINAL row (or -1 when the database has fewer than j+1 rows), out_d2[i][j] = squared distance (0xFFFFFFFF when idx = -1).
 * tcgen05 kind::i8 MMA, TMA-fed, top-2 selection fused in the TMEM epilogue. */
int sod_match_top2(const uint8_t* q, const int32_t* qn, int64_t n_query, const uint8_t* db_sorted,
                   const int32_t* cq, int64_t n_db, int32_t db_index_base, int32_t* out_idx,
                   uint32_t* out_d2, void* workspace, size_t workspace_bytes, sod_stream_t stream);

/* sod_match_top2 over the stored tiles [tile_begin, tile_end) only (tile_end < 0: to the end; a tile is
 * SOD_TILE_ROWS stored rows, in the order sod_db_prepare wrote them: an even sample of the norm range),
 * with an optional caller-held threshold array row_thr: int32 [sod_row_thr_ints(n_query)], in units of
 * d^2 - |q|^2, 0x7F7F7F7F = none.  The sweep prunes with it from the start and leaves
 * min(input, the row's 2nd best of this sweep) in it.  Any such value is an upper bound of the row's final
 * 2nd best, so results stay exact when the array is carried to another launch, or min-reduced across the
 * GPUs that hold other shards before each sweeps the rest of its shard: candidates that cannot be in the
 * GLOBAL top-2 are then never collected.  Lists of several ranges are combined with sod_top2_merge. */
int64_t sod_row_thr_ints(int64_t n_query);
int sod_match_top2_range(const uint8_t* q, const int32_t* qn, int64_t n_query, const uint8_t* db_sorted,
                         const int32_t* cq, int64_t n_db, int32_t db_index_base, int64_t tile_begin,
                         int64_t tile_end, int32_t* row_thr, int32_t* out_idx, uint32_t* out_d2,
                         void* workspace, size_t workspace_bytes, sod_stream_t stream);

/* sod_match_top2_range for a database sharded over several GPUs of one node, with the thresholds travelling
 * over peer memory instead of a collective: row_thr is this rank's threshold array (read when a query block's
 * sweep starts), peer_thr_host a HOST array of n_peers DEVICE pointers to the arrays of all ranks (own one
 * included; peers mapped with sod_ipc_open).  When a query block's sweep ends, the 2nd best of each of its rows
 * is min-ed into every rank's array (reductions over NVLink).  block_rotation (in query blocks of 256 rows)
 * rotates the order in which this rank visits the blocks - rank r of G passes r * n_blocks / G - so that the
 * ranks reach a block at different times and each prunes with what the earlier visitors found in THEIR shards:
 * no all-reduce, no stage boundary, and on average 7/16 of the database is known to a block's sweep.  Values are
 * 2nd-best distances of real rows, so results stay exact whatever the timing; the caller resets the array
 * (0x7F7F7F7F) before each batch and alternates between two arrays from batch to batch (a peer may run a
 * little ahead, never a whole batch: the exchange of the merged lists separates batches).  Applies to
 * single-segment sweeps (large batches); n_peers = 0 is sod_match_top2_range. */
int sod_match_top2_peer(const uint8_t* q, const int32_t* qn, int64_t n_query, const uint8_t* db_sorted,
                        const int32_t* cq, int64_t n_db, int32_t db_index_base, int64_t tile_begin,
                        int64_t tile_end, int32_t* row_thr, int32_t* const* peer_thr_host, int32_t n_peers,
                        int64_t block_rotation, int32_t* out_idx, uint32_t* out_d2, void* workspace,
                        size_t workspace_bytes, sod_stream_t stream);

/* K3.  Merge n_parts candidate lists (parts_idx/parts_d2 are [n_parts][n_query][2], e.g. the
 * all-gathered shard-local results) into the global top-2 by (d2, idx) lexicographic order and
 * apply Lowe's ratio test exactly as the reference evaluates it (main.py:81-82):
 *   distance = sqrtf(d2) as float32 (OpenCV), pass = (double)dist1 < ratio * (double)dist2.
 * out_dist (float32 [n_query][2]) and out_pass (u8 [n_query]) may be NULL. */
int sod_top2_merge(const int32_t* parts_idx, const uint32_t* parts_d2, int32_t n_parts,
                   int64_t n_query, int32_t* out_idx, uint32_t* out_d2, float* out_dist,
                   uint8_t* out_pass, double ratio, sod_stream_t stream);

/* K3 in exchange form, for a database sharded over G GPUs (SURVEY.md 8e; the shard merge the north
 * star describes as "an NCCL all-gather over NVLink merges them").  A candidate is one signed 64-bit
 * key (d2 << 32 | global row; INT64_MAX = none) whose order is the merge order (distance, then lowest
 * index - cv2's tie rule); keys travel as [row][2] pairs.  Instead of gathering every rank's lists onto
 * every rank (G x 16 B per query row received), rank r merges only rows [r*S, (r+1)*S), S = rows / G:
 *   sod_top2_keys        idx/d2 [n_query][2] of this rank -> keys int64 [n_rows][2]; rows n_query..n_rows
 *                        (padding up to G whole slices) are "none"
 *   (caller)             all-to-all: slice r of every rank's keys goes to rank r (16 B per row and peer)
 *   sod_top2_merge_keys  parts int64 [n_parts][n_rows][2] -> the two smallest keys per row, [n_rows][2]
 *   (caller)             all-gather of the merged slices (16 B per query row)
 *   sod_top2_from_keys   keys [n_query][2] -> out_idx/out_d2/out_dist/out_pass exactly as
 *                        sod_top2_merge writes them (ratio test included).
 * Key arrays must be 16-byte aligned. */
int sod_top2_keys(const int32_t* idx, const uint32_t* d2, int64_t n_query, int64_t n_rows, int64_t* keys,
                  sod_stream_t stream);
int sod_top2_merge_keys(const int64_t* parts, int32_t n_parts, int64_t n_rows, int64_t* out, sod_stream_t stream);
int sod_top2_from_keys(const int64_t* keys, int64_t n_query, int32_t* out_idx, uint32_t* out_d2, float* out_dist,
                       uint8_t* out_pass, double ratio, sod_stream_t stream);

/* K3 over peer memory: the same merge for query batches small enough that two NCCL calls would cost more
 * than the matching itself (BASELINE configs[2]: 10k query descriptors against a 1M-row database on 8 GPUs).
 * Every rank owns one exchange buffer of sod_exchange_bytes(max_query, world) bytes, allocated by
 * sod_exchange_alloc (cudaMalloc memory, zeroed; the one place this library allocates: IPC export needs a
 * whole allocation), exported with sod_ipc_export (a 64-byte cudaIpcMemHandle_t the caller passes to the
 * other processes of the node by any means) and mapped by every peer with sod_ipc_open.
 * sod_top2_exchange_peer(idx, d2, ...) stores this rank's lists as packed keys into slot `rank` of EVERY
 * rank's buffer (peer stores over NVLink), publishes a call counter there, waits until the counters of all
 * ranks have arrived in its own buffer, merges the G candidates per row and writes out_idx / out_d2 /
 * out_dist / out_pass exactly as sod_top2_merge does - two kernels on the caller's stream, no host
 * synchronisation, capturable in a CUDA graph (the call counter lives in the buffer).  Every rank must make
 * the same sequence of calls; peer_buffers_host is a HOST array of `world` device pointers (entry `rank` =
 * the own buffer).  A rank that waits ~4 s for a peer traps (launch error) instead of hanging. */
#define SOD_EXCHANGE_MAX_RANKS 16
#define SOD_IPC_HANDLE_BYTES 64
size_t sod_exchange_bytes(int64_t max_query, int32_t world);
int sod_exchange_alloc(size_t bytes, void** buffer_out);
int sod_exchange_free(void* buffer);
int sod_ipc_export(const void* buffer, uint8_t* handle_host);
int sod_ipc_open(const uint8_t* handle_host, void** buffer_out);
int sod_ipc_close(void* buffer);
int sod_top2_exchange_peer(const int32_t* idx, const uint32_t* d2, int64_t n_query, int32_t rank, int32_t world,
                           void* const* peer_buffers_host, int64_t max_query, int32_t* out_idx, uint32_t* out_d2,
                           float* out_dist, uint8_t* out_pass, double ratio, sod_stream_t stream);

/* ---- bf16 fallback for descriptors that are NOT integer-valued 0..255 (non-OpenCV extractors,
 * normalised float descriptors).  Same reference call as sod_match_top2 (main.py:70-73), approximate
 * distances: d^2 = |q|^2 + |t|^2 - 2 q.t with fp32 norms and the dot product on tcgen05 kind::f16
 * (bf16 x bf16 -> f32).  split = 1 (recommended) multiplies bf16 hi/lo halves of both sides
 * (K = 384); split = 0 is plain bf16 (K = 128).  Stated tolerance on d^2 relative to
 * |q|^2 + |t|^2: 2e-5 (split) / 4e-3 (plain); indices are those of the two smallest approximate
 * distances, ties -> lowest index. */

/* Operand row length in bf16 elements: 128 (split = 0) or 384 (split = 1). */
int64_t sod_bf16_operand_cols(int32_t split);
/* Rows of the database-side operand / norm arrays: n_rows rounded up to whole 128-row tiles. */
int64_t sod_bf16_db_rows(int64_t n_rows);

/* float32 [n_rows][128] -> bf16 operand and fp32 squared norms.
 * side = 0 (query):    dst [n_rows][cols],                   norms [n_rows]
 * side = 1 (database): dst [sod_bf16_db_rows(n_rows)][cols], norms [sod_bf16_db_rows(n_rows)]
 *                      (values pre-multiplied by -2, padding rows zero with norm +inf)
 * *nonfinite_flag (device, may be NULL) is OR-ed with 1 if any input is NaN or infinite. */
int sod_bf16_prepare(const float* src, int64_t n_rows, int32_t side, int32_t split, uint16_t* dst,
                     float* norms, int32_t* nonfinite_flag, sod_stream_t stream);

size_t sod_match_bf16_workspace_bytes(int64_t n_query, int64_t n_db);

/* out_idx int32 [n_query][2] (-1 = no such neighbour), out_d2 float32 [n_query][2] (+inf then). */
int sod_match_top2_bf16(const uint16_t* q_op, const float* qn, int64_t n_query, const uint16_t* db_op,
                        const float* dn, int64_t n_db, int32_t split, int32_t db_index_base,
                        int32_t* out_idx, float* out_d2, void* workspace, size_t workspace_bytes,
                        sod_stream_t stream);

/* sod_top2_merge for float distances (shard merge + ratio test of the bf16 path). */
int sod_top2_merge_f32(const int32_t* parts_idx, const float* parts_d2, int32_t n_parts,
                       int64_t n_query, int32_t* out_idx, float* out_d2, float* out_dist,
                       uint8_t* out_pass, double ratio, sod_stream_t stream);


/* ------------------------------------------------------------------------------------------------
 * Hough voting and affine verification
 * ---------------------------------------------------------------------------------------------- */

/* Keypoints as structure-of-arrays: exactly the fields the path reads from cv2.KeyPoint
 * (.pt, .angle, .octave; SURVEY.md §8b). */
typedef struct {
  const float* xy;       /* [n][2] KeyPoint.pt */
  const float* angle;    /* [n] KeyPoint.angle, degrees in [0,360) */
  const int32_t* octave; /* [n] KeyPoint.octave as packed by OpenCV SIFT (low byte = octave) */
  int64_t n;
} sod_keypoints;

/* Everything Main holds about the query image(s) and the model database that the Hough and affine
 * stages read (main.py:20-28).  A "frame" is one query image; a "group" is one Hough space.
 * The reference has one frame and one space for all model images (groups_per_frame = 1,
 * image_group = NULL); multi-object configurations give every object its own space. */
typedef struct {
  sod_keypoints query;          /* kp_query (all frames concatenated) */
  const int32_t* query_frame;   /* [query.n] frame of each query keypoint; NULL = all frame 0 */
  const int32_t* frame_wh;      /* [n_frames][2] (W,H) of each query image (image_query_size) */
  int32_t n_frames;
  sod_keypoints model;          /* kp (whole database, indexed by global descriptor row) */
  const int32_t* model_image;   /* [model.n] model image each keypoint came from */
  const double* image_centroid; /* [n_images][2] img_centroid_list entries */
  const double* image_size;     /* [n_images][2] (w,h) img_size_list entries */
  const int32_t* image_group;   /* [n_images] Hough space of the image inside a frame; NULL = 0 */
  int32_t n_images;
  int32_t groups_per_frame;
} sod_scene;

#define SOD_SIGMA_LUT_MIN (-24)
#define SOD_SIGMA_LUT_LEN 49
#define SOD_MAX_BINS 15 /* bins^4 uint32 counters must fit one SM's shared memory */
#define SOD_MAX_CLUSTER_BINS 65536 /* sod_pose_adjacency / sod_angle_adjacency: n x n/8 bytes of bit matrix */

/* Outputs of sod_hough_vote (device).  Bin records are compact and in no particular order;
 * `bin_order` reproduces the reference's dict insertion order when sorted ascending. */
typedef struct {
  double* pose;        /* [M][4] x, y, alpha, scale per match (estimate_object_pose) */
  uint32_t* base_bin;  /* [M] ix | iy<<8 | itheta<<16 | isigma<<24 (calculate_bin_index) */
  uint8_t* near_edge;  /* [M] 0; 1 = x*bins/W or y*bins/H lies within 1e-9 of an integer and the bin was
                          confirmed for every admissible libm (cos / sin moved by +-4 ulp give the same
                          bin, or the angle is exactly 0); 2 = those evaluations disagree (DESIGN.md 2) */
  int32_t* counters;   /* [8] n_bins, n_votes, n_near_edge (flags 1 and 2), overflow flag, n_unresolved
                          (flag 2), 3 reserved; zeroed by the call */
  int32_t* bin_group;  /* [cap_bins] frame * groups_per_frame + image_group */
  int32_t* bin_code;   /* [cap_bins] ((ix*bins + iy)*bins + itheta)*bins + isigma */
  int32_t* bin_count;  /* [cap_bins] votes */
  int32_t* bin_offset; /* [cap_bins] start of the bin's members */
  int64_t* bin_order;  /* [cap_bins] first member * 16 + its vote offset (w*8+x*4+y*2+z) */
  double* bin_mean;    /* [cap_bins][6] running means cx, cy, angle, scale, img_w, img_h (PoseBin) */
  int32_t* members;    /* [cap_votes] match ids, ascending inside every bin */
  int64_t cap_bins;    /* 16*M always suffices */
  int64_t cap_votes;
} sod_hough_out;

/* Stable compaction of the ratio survivors: match_q = query rows with pass != 0 in ascending
 * order, match_t = their nearest database row (main.py:81-86 builds the same list).  Only matches
 * whose database row lies in [t_lo, t_hi) are kept: a rank of a sharded database keeps the matches
 * of its own model objects (use 0, INT32_MAX for everything).  n_out is a device int32.
 * scratch: sod_compact_scratch_bytes(n_query). */
size_t sod_compact_scratch_bytes(int64_t n_query);
int sod_compact_matches(const int32_t* idx, const uint8_t* pass, int64_t n_query, int32_t t_lo,
                        int32_t t_hi, int32_t* match_q, int32_t* match_t, int32_t* n_out,
                        void* scratch, sod_stream_t stream);

/* estimate_object_pose + calculate_bin_index only (HoughTransformHelperFunctions.py:4-72), no voting:
 * pose [n][4] and base_bin [n] as in sod_hough_out; near_edge may be NULL. */
int sod_estimate_pose(const sod_scene* scene, const int32_t* match_q, const int32_t* match_t,
                      int64_t n_matches, int32_t bins, const int32_t* sigma_lut, double* pose,
                      uint32_t* base_bin, uint8_t* near_edge, sod_stream_t stream);

/* calculate_bin_index (HoughTransformHelperFunctions.py:39-72) for caller-supplied poses
 * (x, y, theta, scale) [n][4] -> packed base bins.  Scales that are not powers of two take
 * log(s)/log(2) on the device (last-bit differences from the host libm are possible there). */
int sod_pose_bin_index(const double* pose, int64_t n, int32_t bins, int32_t width, int32_t height,
                       const int32_t* sigma_lut, uint32_t* base_bin, sod_stream_t stream);

/* Bytes of scratch for sod_hough_vote. */
size_t sod_hough_workspace_bytes(int64_t n_matches, int64_t n_groups);

/* K4.  Main.apply_hough_transform (main.py:89-119) with estimate_object_pose and
 * calculate_bin_index (HoughTransformHelperFunctions.py:4-72) and the PoseBin bookkeeping
 * (PoseBin.py:19-54): every match votes into the <=16 bins (ix+w, iy+x, itheta+y, isigma+z) whose
 * coordinates are all < bins.  n_matches is the capacity of match_q/match_t; if n_matches_dev is
 * not NULL the actual count is read from it on the device.  sigma_lut[k - SOD_SIGMA_LUT_MIN] is
 * the isigma of scale factor 2^k (device int32[SOD_SIGMA_LUT_LEN]).  Every non-empty bin gets a
 * record (group, code, count, offset); bins with at least detail_min_count votes also get their
 * member list sorted, the running means and the insertion-order key (1 = all bins, as the
 * reference's dict; a caller that only goes on to sod_affine_verify passes its vote threshold and
 * skips that work for the bins it will never look at). */
int sod_hough_vote(const sod_scene* scene, const int32_t* match_q, const int32_t* match_t,
                   int64_t n_matches, const int32_t* n_matches_dev, int32_t bins,
                   const int32_t* sigma_lut, int32_t detail_min_count, const sod_hough_out* out,
                   void* workspace, size_t workspace_bytes, sod_stream_t stream);

/* sod_hough_vote with one bin count per pose dimension, as the legacy perform_hough_transform takes
 * them (HoughTransform.py:8: bin_x, bin_y, bin_theta, bin_sigma).  Bin codes are
 * ((ix * bins_y + iy) * bins_theta + itheta) * bins_sigma + isigma; sigma_lut must be built for
 * bins_sigma.  Each count <= 255 and their product <= SOD_MAX_BINS^4 (one SM's shared memory). */
int sod_hough_vote_dims(const sod_scene* scene, const int32_t* match_q, const int32_t* match_t,
                        int64_t n_matches, const int32_t* n_matches_dev, int32_t bins_x, int32_t bins_y,
                        int32_t bins_theta, int32_t bins_sigma, const int32_t* sigma_lut,
                        int32_t detail_min_count, const sod_hough_out* out, void* workspace,
                        size_t workspace_bytes, sod_stream_t stream);

/* Outputs of sod_affine_verify (device), one entry per bin that entered with >= vote_threshold. */
typedef struct {
  int32_t* counters;    /* [4] n_valid, overflow, bins with a near-singular normal matrix, residual tests
                           decided within 1e-9 relative + 1e-7 px of their limit; zeroed by the call */
  int32_t* valid_bin;   /* [cap_valid] index of the bin record */
  double* params;       /* [cap_valid][6] m1 m2 m3 m4 tx ty of the last fit */
  int32_t* votes;       /* [cap_valid] members left */
  int32_t* status;      /* [cap_valid] bit0 live (votes >= affine_threshold at the fixed point),
                           bit1 near-singular normal matrix (smallest |eigenvalue| <= 1e-10 x largest) in
                           some pass, bit2 a residual test of the bin was decided on the edge of its
                           limit, bits 8.. number of passes */
  uint8_t* member_keep; /* [cap_votes] aligned with sod_hough_out.members: 1 = still in its bin */
  int64_t cap_valid;
  int64_t cap_votes;    /* elements of member_keep: a bin whose members end past it is not verified and
                           sets the overflow counter (the array was sized for another Hough result) */
} sod_affine_out;

/* K5.  Main.get_valid_bins + Main.apply_affine_parameters (main.py:121-157) with AffineParameters
 * and remove_outliers (AffineParameters.py:89-160): per bin, fit u = m1 x + m2 y + tx,
 * v = m3 x + m4 y + ty by the pseudo-inverse of the normal matrix (rcond 1e-15), drop pairs whose
 * residual exceeds W*isigma/factor_x or H*isigma/factor_y, repeat until nothing is dropped or fewer
 * than affine_threshold pairs remain.  max_passes > 0 stops after that many fit/prune passes
 * (1 = one AffineParameters + remove_outliers call); factor <= 0 disables pruning on that axis
 * (a pure fit). */
int sod_affine_verify(const sod_scene* scene, const int32_t* match_q, const int32_t* match_t,
                      const sod_hough_out* hough, int32_t bins, int32_t vote_threshold,
                      int32_t affine_threshold, double factor_x, double factor_y, int32_t max_passes,
                      const sod_affine_out* out, sod_stream_t stream);

/* The Hough records (space, bin code, insertion-order key, six running means) of the bins listed in
 * affine->valid_bin, in that order: out_* hold affine->cap_valid entries, the first counters[0] are written.
 * What Main.post_process (main.py:159-168) reads of the surviving bins, gathered on the device so that the
 * caller's read-back is plain copies. */
int sod_valid_bin_records(const sod_hough_out* hough, const sod_affine_out* affine, int32_t* out_group,
                          int32_t* out_code, int64_t* out_order, double* out_mean, sod_stream_t stream);

/* remove_outliers' decision for caller-supplied parameters (AffineParameters.py:128-155):
 * keep[i] = !(|m1 x + m2 y + tx - u| > x_ref || |m3 x + m4 y + ty - v| > y_ref), params on the device. */
int sod_affine_residual_keep(const float* model_xy, const float* query_xy, int64_t n,
                             const double* params, double x_ref, double y_ref, uint8_t* keep,
                             sod_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Pose clustering after the path (SURVEY.md §8f N1)
 * ---------------------------------------------------------------------------------------------- */

/* Neighbour graph of group_position (PostProcessing.py:14-37) over n surviving bins: bins a, b are
 * adjacent iff |cx_a - cx_b| <= reach_x_a, reach_x_b and |cy_a - cy_b| <= reach_y_a, reach_y_b, with
 * reach_x = img_w * scale / 4 and reach_y = img_h * scale / 4 evaluated by the caller (fp64, the
 * reference's expression).  segment (may be NULL) restricts edges to bins of equal segment id
 * (e.g. the frame of a batch).  adj: uint32 [n][ceil(n/32)] bit matrix, bit j of row i (no self
 * loops); label[i] = lowest bin index of i's connected component.  n <= SOD_MAX_CLUSTER_BINS. */
int sod_pose_adjacency(const double* cx, const double* cy, const double* reach_x, const double* reach_y,
                       const int32_t* segment, int64_t n, uint32_t* adj, int32_t* label,
                       sod_stream_t stream);

/* Neighbour graph of group_orientation (PostProcessing.py:39-63): bins of equal segment (the
 * position cluster) are adjacent iff abs(math.degrees(angle_a - angle_b)) <= max_degrees (1 in the
 * reference).  Same outputs as sod_pose_adjacency. */
int sod_angle_adjacency(const double* angle, const int32_t* segment, int64_t n, double max_degrees,
                        uint32_t* adj, int32_t* label, sod_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * SIFT extraction (in front of the path)
 * ---------------------------------------------------------------------------------------------- */

/* cv2.SIFT_create() with its default parameters (3 layers per octave, contrast threshold 0.04, edge
 * threshold 10, sigma 1.6, image doubled first, all features kept) on a u8 gray image (device memory,
 * rows `pitch` bytes apart, 1..32768 pixels a side).  Keypoints follow cv2's conventions (KeyPoint.pt,
 * .size, .angle, .response, .octave packed with first octave -1, so unpack_sift_octave applies) and come
 * sorted and de-duplicated as cv2 returns them; descriptors are u8 rows ready for the matcher.  Not bit-exact:
 * DESIGN.md 2 states the measured agreement with cv2. */
#define SOD_SIFT_MAX_OCTAVES 16
#define SOD_SIFT_MAX_CAP (1 << 24)

typedef struct {
  float* xy;          /* [cap][2] KeyPoint.pt */
  float* size;        /* [cap] */
  float* angle;       /* [cap] degrees in [0,360) */
  float* response;    /* [cap] */
  int32_t* octave;    /* [cap] */
  uint8_t* des;       /* [cap][128] */
  int32_t* counters;  /* [2] number of keypoints, overflow flag (1 = more than cap keypoints before duplicate
                         removal: the output is incomplete and must not be used); written by the call */
  int64_t cap;        /* 1..SOD_SIFT_MAX_CAP */
} sod_sift_out;

/* Bytes of workspace (256-byte aligned) for an image of this size and max_keypoints = out.cap; 0 if the size or
 * the capacity is out of range.  max_keypoints = 0 is enough for sod_sift_describe. */
size_t sod_sift_workspace_bytes(int32_t width, int32_t height, int64_t max_keypoints);

/* Replaces cv2.SIFT_create().detectAndCompute(gray, None) of Main.get_query_features (main.py:43-46) and of
 * stream.sift_features.  The Gaussian pyramid is left in the workspace (sod_sift_level_offset). */
int sod_sift_extract(const uint8_t* gray, int32_t width, int32_t height, int64_t pitch, const sod_sift_out* out,
                     void* workspace, size_t workspace_bytes, sod_stream_t stream);

/* cv2.SIFT.compute(gray, keypoints) for n caller-supplied keypoints (device arrays in the layout of
 * sod_sift_out): des [n][128].  The pyramid is the one detectAndCompute builds (image doubled, so a keypoint set
 * that contains octave -1, as every set cv2 detects does).  A keypoint whose octave and layer name no pyramid
 * level gets a zero row and adds 1 to *n_invalid (device int32, caller zeroes it; may be NULL). */
int sod_sift_describe(const uint8_t* gray, int32_t width, int32_t height, int64_t pitch, const float* xy,
                      const float* size, const float* angle, const int32_t* octave, int64_t n, uint8_t* des,
                      int32_t* n_invalid, void* workspace, size_t workspace_bytes, sod_stream_t stream);

/* Byte offset in the workspace of Gaussian level `level` (0..5) of `octave` (-1 = the doubled image) after
 * sod_sift_extract / sod_sift_describe, f32 rows of wh_host[0] (HOST, may be NULL) values, wh_host[1] rows.
 * -1 if the image has no such level.  Lets a caller check the pyramid against cv2.  After
 * sod_sift_extract_batch the same level of frame f lies f x sod_sift_batch_workspace_bytes(w, h, 1, 0) bytes
 * further on (one frame's pyramid, 256-byte aligned). */
int64_t sod_sift_level_offset(int32_t width, int32_t height, int32_t octave, int32_t level, int32_t* wh_host);

/* ---- SIFT over a batch of same-size frames in one pass.  Every stage runs once for all frames (one launch per
 * pyramid level), and the rows come out packed frame after frame, already in the layout the detection path
 * takes (des, xy, angle, octave and the frame of each row). */
#define SOD_SIFT_MAX_FRAMES 4096

typedef struct {
  float* xy;              /* [cap_rows][2] KeyPoint.pt */
  float* size;            /* [cap_rows] */
  float* angle;           /* [cap_rows] degrees in [0,360) */
  float* response;        /* [cap_rows] */
  int32_t* octave;        /* [cap_rows] */
  uint8_t* des;           /* [cap_rows][128] */
  int32_t* frame;         /* [cap_rows] frame (0..frames-1) of each row */
  int32_t* count;         /* [frames] keypoints of each frame (after max_per_frame) */
  int32_t* offset;        /* [frames] first row of each frame: frame f is rows [offset[f], offset[f] + count[f]) */
  int32_t* overflow;      /* [frames] 1 = the frame had more than cap_per_frame keypoints before duplicate removal:
                             its rows are incomplete and must not be used */
  int32_t* rows_overflow; /* [1] 1 = the packed rows exceed cap_rows: rows from cap_rows on were dropped */
  int64_t cap_rows;       /* 1..SOD_SIFT_MAX_CAP */
  int64_t cap_per_frame;  /* keypoints one frame may produce before duplicate removal; frames x cap_per_frame
                             <= SOD_SIFT_MAX_CAP */
} sod_sift_batch_out;

/* Bytes of workspace (256-byte aligned) for `frames` images of this size and cap_per_frame = out.cap_per_frame;
 * 0 if an argument is out of range.  At least frames x the pyramid of one frame. */
size_t sod_sift_batch_workspace_bytes(int32_t width, int32_t height, int32_t frames, int64_t cap_per_frame);

/* sod_sift_extract of `frames` u8 gray images of one size (image f at gray + f x frame_stride, rows `pitch`
 * bytes apart, frame_stride >= pitch x height).  Frame f's rows are the first max_per_frame (0 = all) keypoints
 * sod_sift_extract gives for that image alone, in the same order; count, offset and every row are written on
 * the device, so the call never synchronises and can be captured in a CUDA graph.  Nothing is truncated
 * silently: overflow[f] and rows_overflow say when rows are missing. */
int sod_sift_extract_batch(const uint8_t* gray, int32_t width, int32_t height, int64_t pitch, int64_t frame_stride,
                           int32_t frames, int64_t max_per_frame, const sod_sift_batch_out* out, void* workspace,
                           size_t workspace_bytes, sod_stream_t stream);

/* ---- SIFT over a batch of frames of different sizes in one pass (training images of one width and many heights,
 * say).  Each (octave, level) is still one launch for all frames, sized for the largest frame that has it. */
#define SOD_SIFT_MAX_MIXED_FRAMES 64

/* Bytes of workspace (256-byte aligned) for `frames` images of the sizes wh_host[2f], wh_host[2f+1] (HOST) and
 * cap_per_frame; 0 if an argument is out of range.  Frame f's pyramid lies at the sum of
 * sod_sift_batch_workspace_bytes(w, h, 1, 0) of frames 0..f-1, so sod_sift_level_offset reads any frame's levels;
 * after the pyramids come the slabs of sod_sift_batch_workspace_bytes and a 160-byte geometry record a frame. */
size_t sod_sift_mixed_workspace_bytes(const int32_t* wh_host, int32_t frames, int64_t cap_per_frame);

/* sod_sift_extract_batch of `frames` u8 gray images of any sizes: image f at images_host[f] (a HOST array of
 * device pointers), wh_host[2f] x wh_host[2f+1] pixels (1..32768 a side), rows pitch_host[f] >= width bytes apart.
 * Frame f's rows are the first max_per_frame (0 = all) keypoints sod_sift_extract gives for that image alone, in
 * the same order, with out as in sod_sift_extract_batch.  The geometry reaches the device as a kernel argument, so
 * the call never synchronises and can be captured in a CUDA graph. */
int sod_sift_extract_mixed(const uint8_t* const* images_host, const int32_t* wh_host, const int64_t* pitch_host,
                           int32_t frames, int64_t max_per_frame, const sod_sift_batch_out* out, void* workspace,
                           size_t workspace_bytes, sod_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* SOD_H_ */
