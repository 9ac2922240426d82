/*
 * klt_b200.h -- C ABI of libklt_b200.so: B200 (sm_100a) pyramid build + pyramidal Lucas-Kanade.
 *
 * Drop-in boundary for the one hot path of JonasFrey96/Visual-Odom-Pipeline that this project
 * replaces: the four `cv2.calcOpticalFlowPyrLK(im0, im1, p, None, winSize, maxLevel, criteria)`
 * calls per frame at reference src/extractor/extractor.py:44,45 (extend_tracks) and :65,66
 * (extend_landmarks), with parameters from src/extractor/extractor.py:16-19.  The reference has no
 * plugin API for this path -- the interface *is* the OpenCV function -- so the entry points below
 * are what a ctypes binding of that function (and of cv2.buildOpticalFlowPyramid, which OpenCV
 * runs inside it) binds.  INTEGRATION.md shows the reference-side stub.
 *
 * Conventions: plain C, no exceptions / STL / torch types across the ABI.  Every function returns
 * a klt_status (0 = ok, <0 = KLT_ERR_*, >0 = cudaError_t passed through).  `stream` is a
 * cudaStream_t passed as void* (NULL = legacy default stream).  Device pointers are owned by the
 * caller.  Functions named *_host take HOST pointers, do their own H2D/D2H and are synchronous on
 * return (like the cv2 call); all others are asynchronous on `stream`.
 *
 * There is no CPU fallback anywhere in this library.
 */
#ifndef KLT_B200_H
#define KLT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KLT_B200_VERSION 120 /* 0.1.2: + bilateral pre-filter; thread-safe contexts; pageable inputs staged in the library */

#define KLT_MAX_LEVELS 16   /* pyramid levels incl. level 0 (cv2 stops when a level <= winSize) */
#define KLT_MAX_WIN_AREA 4096 /* win_w * win_h supported by the LK kernel (cv2 default 21x21) */
#define KLT_MAX_WIN_SIDE 504  /* win_w and win_h supported by the LK kernel */
/* Every LK window with win_w * win_h <= KLT_MAX_WIN_AREA and both sides <= KLT_MAX_WIN_SIDE is supported (win_w, win_h
 * >= 3, as for cv2).  A wider, taller or larger window returns KLT_ERR_UNSUPPORTED. */

/* cv2.TERM_CRITERIA_* and cv2.OPTFLOW_* values (same numbers as OpenCV) */
#define KLT_TERM_COUNT 1
#define KLT_TERM_EPS 2
#define KLT_OPTFLOW_USE_INITIAL_FLOW 4
#define KLT_OPTFLOW_LK_GET_MIN_EIGENVALS 8

typedef int klt_status;
#define KLT_OK 0
#define KLT_ERR_INVALID_ARG (-1)   /* cv2 would raise error -215 (assertion) */
#define KLT_ERR_UNSUPPORTED (-2)   /* valid for cv2, outside this library's limits */
#define KLT_ERR_NO_DEVICE (-3)     /* no CUDA device / wrong architecture: never falls back */
#define KLT_ERR_OUT_OF_MEMORY (-4)
#define KLT_ERR_INTERNAL (-5)

/* Opaque context: device id, two streams, device workspace, pinned staging, helper threads for pageable inputs.
 * Threads: a context may be shared.  The *_host entry points use the context's workspaces and streams and are
 * serialised by a mutex inside the context (concurrent callers queue up; one context per thread avoids that).  The
 * device-pointer entry points keep no per-call state in the context and may run concurrently on different streams.
 * Every entry point makes the context's device current for the duration of the call and restores the caller's. */
typedef struct klt_ctx klt_ctx;

/* One pyramid level as the kernels see it (row `y` of batch item `b` starts at
 * data + b*batch_stride + y*pitch). */
typedef struct klt_level {
    int32_t w, h;
    int64_t pitch;        /* bytes between rows */
    int64_t batch_stride; /* bytes between batch items */
    int64_t offset;       /* byte offset of this level inside the pyramid buffer (levels >= 1) */
} klt_level;

/* Geometry of a pyramid: level 0 is the caller's image batch (never copied), levels 1..top live
 * in ONE caller-provided buffer of `bytes` bytes.  Mirrors what cv2.buildOpticalFlowPyramid
 * returns (retval = top, list of levels) -- SURVEY.md s8b / A.2. */
typedef struct klt_pyr_layout {
    int32_t top;    /* index of the last level built (cv2's retval; may be < max_level) */
    int32_t batch;
    klt_level level[KLT_MAX_LEVELS]; /* level[0].pitch/batch_stride are filled by the caller */
    int64_t bytes;  /* size of the levels>=1 buffer for the whole batch */
} klt_pyr_layout;

/* ---- context -------------------------------------------------------------------------------- */
klt_status klt_create(int device, klt_ctx** out);
klt_status klt_destroy(klt_ctx* ctx);
int klt_version(void);
const char* klt_status_string(klt_status s);
/* number of SMs / name of the device the context is bound to (for bench & grid sizing) */
klt_status klt_device_info(klt_ctx* ctx, int* sm_count, int* cc_major, int* cc_minor, char* name, int name_len);

/* ---- pinned host memory (so numpy inputs can be DMA'd without a staging copy) ---------------- */
klt_status klt_host_alloc(void** ptr, int64_t bytes);
klt_status klt_host_free(void* ptr);

/* ---- pyramid (replaces cv2.buildOpticalFlowPyramid / pyrDown; SURVEY.md A.2) ----------------- */
/* Fills `out` for a w x h image batch: number of levels per cv2's rule (stop before a level whose
 * width <= win_w or height <= win_h), per-level size / pitch / offset.  Host-only, no CUDA call. */
klt_status klt_pyr_plan(int w, int h, int win_w, int win_h, int max_level, int batch, klt_pyr_layout* out);

/* Builds levels 1..top of batch items [first_item, first_item + n_items) (n_items <= 0: all of
 * them).  d_img: level 0 of item 0 (u8, pitch/batch_stride from layout->level[0]); d_pyr: buffer of
 * layout->bytes.  One kernel launch per level for the whole item range. */
klt_status klt_pyr_build(klt_ctx* ctx, const uint8_t* d_img, const klt_pyr_layout* layout,
                         uint8_t* d_pyr, int first_item, int n_items, void* stream);

/* Single pyrDown step (cv2.pyrDown on 1-channel u8, BORDER_REFLECT_101), device pointers. */
klt_status klt_pyr_down(klt_ctx* ctx, const uint8_t* d_src, int w, int h, int64_t src_pitch,
                        int64_t src_batch_stride, uint8_t* d_dst, int64_t dst_pitch,
                        int64_t dst_batch_stride, int batch, void* stream);

/* ---- Lucas-Kanade (replaces the per-level Scharr + LKTrackerInvoker loop; SURVEY.md A.3-A.6) -- */
typedef struct klt_lk_params {
    int32_t win_w, win_h;
    int32_t crit_type;      /* KLT_TERM_COUNT | KLT_TERM_EPS, as in cv2's criteria[0] */
    int32_t crit_max_count; /* criteria[1] */
    double crit_eps;        /* criteria[2] */
    int32_t flags;          /* KLT_OPTFLOW_*; every other bit must be 0 (0x100 / 0x200 are used by diagnostics and the launcher) */
    double min_eig_threshold; /* cv2 default 1e-4 */
} klt_lk_params;

/* Tracks n_per_pair points in each of n_pairs frame pairs, all pyramid levels in ONE launch.
 * `layout` describes both pyramid buffers (they may be the same buffer): pair i uses batch item
 * prev_first + i*pair_stride of (d_prev_img, d_prev_pyr) and item next_first + i*pair_stride of
 * (d_next_img, d_next_pyr), so one batched pyramid build can hold previous and next frames side by
 * side (interleaved: prev_first 0, next_first 1, pair_stride 2; a frame ring: 0, 1, 1).
 * d_prev_pts / d_next_pts: float2 [n_pairs][n_per_pair]; d_status: u8; d_err: float;
 * d_iters (optional, may be NULL): int32 LK iterations executed per point over all levels.
 * d_next_pts is read only with KLT_OPTFLOW_USE_INITIAL_FLOW.  Points whose err cv2 leaves
 * uninitialised (SURVEY.md A.6) get err = 0. */
klt_status klt_lk_track(klt_ctx* ctx,
                        const uint8_t* d_prev_img, const uint8_t* d_prev_pyr,
                        const uint8_t* d_next_img, const uint8_t* d_next_pyr,
                        const klt_pyr_layout* layout, int prev_first, int next_first, int pair_stride, int n_pairs,
                        const float* d_prev_pts, float* d_next_pts, uint8_t* d_status, float* d_err,
                        int32_t* d_iters, int n_per_pair, const klt_lk_params* params, void* stream);

/* ---- host-pointer entry points: exactly what a binding of the cv2 functions needs ------------ */
/* cv2.calcOpticalFlowPyrLK(prevImg, nextImg, prevPts, nextPts, winSize, maxLevel, criteria[, flags,
 * minEigThreshold]) -> nextPts, status, err.  HOST buffers (pinned or pageable); images u8 with
 * arbitrary row pitch; points float32 [n][2].  Synchronous.  top_level_out (optional) receives the
 * last pyramid level used.  Pinned images are DMA'd in place; pageable ones (numpy arrays of the un-edited
 * reference) are staged through a pinned landing zone by the calling thread and three helper threads of the
 * context while the DMA of the first image already runs. */
klt_status klt_calc_optical_flow_pyr_lk_host(klt_ctx* ctx,
                        const uint8_t* prev_img, int64_t prev_pitch,
                        const uint8_t* next_img, int64_t next_pitch, int w, int h,
                        const float* prev_pts, float* next_pts, uint8_t* status, float* err, int n,
                        int max_level, const klt_lk_params* params, int* top_level_out);

/* ---- the reference's tracking step, fused (SURVEY.md s8f rank 1) ------------------------------ */
/* Bidirectional-error / bounds filter, device pointers: reference src/extractor/extractor.py:46-47,53 (extend_tracks)
 * and :67-68,75 (extend_landmarks):  bidir = max(|p0 - p0r|) over x, y;  keep = bidir < max_bidir_error and
 * 0 <= p1.x <= w and 0 <= p1.y <= h (inclusive, as in the reference; NaN fails).  d_bidir_err may be NULL. */
klt_status klt_track_filter(klt_ctx* ctx, const float* d_p0, const float* d_p1, const float* d_p0r, int64_t n,
                            float max_bidir_error, int w, int h, uint8_t* d_keep, float* d_bidir_err, void* stream);

/* One call for what extend_tracks / extend_landmarks do with cv2 (extractor.py:43-53, 64-75): p1 = LK(im0, im1, p0),
 * p0r = LK(im0, im1, p1) (the reference's second call runs in the same direction, started from the forward result),
 * then the filter above.  HOST buffers, synchronous.  One upload and ONE pyramid build per image instead of the four
 * OpenCV builds two cv2 calls make.  next_pts / status / err are those of the first call (bit-identical to cv2's). */
klt_status klt_track_bidirectional_host(klt_ctx* ctx,
                        const uint8_t* prev_img, int64_t prev_pitch,
                        const uint8_t* next_img, int64_t next_pitch, int w, int h,
                        const float* prev_pts, int n, int max_level, const klt_lk_params* params,
                        float max_bidir_error, float* next_pts, uint8_t* status, float* err,
                        uint8_t* keep, float* bidir_err);

/* klt_track_bidirectional_host with a forward-backward check (Kalal et al., 2010) instead of the reference's second call:
 * p0r = LK(im1, im0, p1), p1 tracked from the new image back into the old one (started at p1, no flag), then the same
 * filter.  On a correct track d is the tracking error, not about twice the frame's motion, so a useful max_bidir_error is
 * about 1 px.  Arguments, outputs and errors as klt_track_bidirectional_host. */
klt_status klt_track_fb_host(klt_ctx* ctx,
                        const uint8_t* prev_img, int64_t prev_pitch,
                        const uint8_t* next_img, int64_t next_pitch, int w, int h,
                        const float* prev_pts, int n, int max_level, const klt_lk_params* params,
                        float max_bidir_error, float* next_pts, uint8_t* status, float* err,
                        uint8_t* keep, float* bidir_err);

/* cv2.buildOpticalFlowPyramid(img, winSize, maxLevel) without derivatives / borders: writes level
 * l (l = 0..top) tightly packed (pitch = level width) at out + level_offsets[l].  Pass out = NULL
 * to query `top` and the offsets / total size only. */
klt_status klt_build_optical_flow_pyramid_host(klt_ctx* ctx, const uint8_t* img, int64_t pitch, int w, int h,
                        int win_w, int win_h, int max_level, uint8_t* out, int64_t* level_offsets /*[KLT_MAX_LEVELS+1]*/,
                        int* top_out);

/* ---- Shi-Tomasi corner detection (SURVEY.md s8f rank 2) -------------------------------------------------------
 * Replaces cv2.goodFeaturesToTrack(img, mask=mask, maxCorners=1000, qualityLevel=0.03, minDistance, blockSize=31)
 * as called at reference src/extractor/extractor.py:110-111 (parameters :21-24; once per frame from
 * src/pipeline/pipeline.py:159-163) and the cv2.cornerMinEigenVal it runs inside (gradient size 3, no Harris).
 * Arithmetic: oracle/gftt_oracle.c G.1-G.8, bit-exact with the cv2 wheel of the image. */

/* Bytes of device scratch klt_corner_min_eigen_val needs for a batch of w x h images. */
int64_t klt_corner_ws_bytes(int w, int h, int batch);

/* cv2.cornerMinEigenVal(src, blockSize, ksize=3), device pointers, batched, asynchronous.  d_img: u8, any pitch;
 * d_eig: float32, eig_pitch / eig_batch_stride in ELEMENTS.  d_max (optional): one uint32 per batch item, zeroed by
 * the caller, receives the order-preserving encoding of the maximum eigenvalue over mask != 0 (d_mask optional =
 * everywhere); it is the input of klt_corner_candidates.  d_ws: klt_corner_ws_bytes() bytes, 256-byte aligned. */
klt_status klt_corner_min_eigen_val(klt_ctx* ctx, const uint8_t* d_img, int w, int h, int64_t pitch, int64_t batch_stride,
                        int batch, int block_size, float* d_eig, int64_t eig_pitch, int64_t eig_batch_stride,
                        const uint8_t* d_mask, int64_t mask_pitch, int64_t mask_batch_stride, uint32_t* d_max,
                        void* d_ws, int64_t ws_bytes, void* stream);

/* Threshold (max * quality_level), 3x3 dilation and local-maximum test of goodFeaturesToTrack fused: appends one
 * 64-bit key per candidate, (order-preserving float encoding << 32) | (y << 16) | x, in arbitrary order, to d_keys
 * (capacity keys per batch item, keys_batch_stride in ELEMENTS).  d_count: one uint32 per batch item, zeroed by the
 * caller, receives the number of candidates (may exceed capacity: the excess is dropped). */
klt_status klt_corner_candidates(klt_ctx* ctx, const float* d_eig, int64_t eig_pitch, int64_t eig_batch_stride, int w, int h,
                        int batch, const uint8_t* d_mask, int64_t mask_pitch, int64_t mask_batch_stride,
                        const uint32_t* d_max, double quality_level, uint64_t* d_keys, int64_t keys_batch_stride,
                        int capacity, uint32_t* d_count, void* stream);

/* The detection mask of reference src/extractor/extractor.py:102-107, built on the device: 255 everywhere, then a
 * filled cv2.circle(mask, np.int32((x, y)), radius, 0, -1) around each of the n points (float32 x, y pairs, device).
 * Bit-identical to OpenCV's filled circle (midpoint circle), centres outside the image included.  radius <= 127. */
klt_status klt_corner_mask_from_points(klt_ctx* ctx, const float* d_points, int n, int radius, int w, int h,
                        uint8_t* d_mask, int64_t mask_pitch, void* stream);

/* The sequential tail of goodFeaturesToTrack on the HOST: sorts the keys of klt_corner_candidates in place (strongest
 * first, equal values: the later pixel in raster order first, like OpenCV) and runs the greedy minimum-distance
 * selection.  corners: capacity x (x, y) floats; *n_out = corners found (<= max_corners if max_corners > 0). */
klt_status klt_select_corners_host(uint64_t* keys, int64_t n_keys, int w, int h, int max_corners, double min_distance,
                        float* corners, int capacity, int* n_out);

/* cv2.cornerMinEigenVal(img, blockSize, ksize=3) with HOST buffers, synchronous.  eig: h x w float32, packed. */
klt_status klt_corner_min_eigen_val_host(klt_ctx* ctx, const uint8_t* img, int64_t pitch, int w, int h, int block_size,
                        float* eig);

/* cv2.goodFeaturesToTrack(img, maxCorners, qualityLevel, minDistance, mask, blockSize) with HOST buffers, synchronous.
 * mask may be NULL.  corners: capacity x (x, y) float32, strongest first; *n_out = number found (cv2 returns None for
 * 0).  KLT_ERR_INVALID_ARG where cv2 asserts (quality_level <= 0, min_distance < 0, max_corners < 0). */
klt_status klt_good_features_to_track_host(klt_ctx* ctx, const uint8_t* img, int64_t pitch, int w, int h,
                        const uint8_t* mask, int64_t mask_pitch, int max_corners, double quality_level,
                        double min_distance, int block_size, float* corners, int capacity, int* n_out);

/* Caller-side fusion of the reference's extract() step (src/extractor/extractor.py:102-111): instead of a host mask the
 * caller passes the keypoints it tracks (HOST float32 x, y pairs) and mask_radius; the mask is rasterised on the device
 * (klt_corner_mask_from_points), so the call uploads n_points * 8 bytes instead of a w x h mask.  Same result as
 * building the mask with cv2.circle and calling klt_good_features_to_track_host. */
klt_status klt_good_features_to_track_points_host(klt_ctx* ctx, const uint8_t* img, int64_t pitch, int w, int h,
                        const float* points, int n_points, int mask_radius, int max_corners, double quality_level,
                        double min_distance, int block_size, float* corners, int capacity, int* n_out);

/* ---- the per-frame step for a batch of sequences --------------------------------------------------------------------
 * What KLTTracker.step does for one sequence (reference src/pipeline/pipeline.py:98-103,159-163 with
 * src/extractor/extractor.py:38-88,102-111), for n_seqs independent sequences with a different point count each, chained on
 * the device: forward LK pass and the reference's second pass, bidirectional-error / bounds filter, detection mask around
 * the survivors, goodFeaturesToTrack with that mask on the next frame.  Per sequence the result is that of the
 * single-sequence step, bit for bit. */

/* Bytes of device workspace klt_frame_step_batch and klt_frame_step_batch_async need for n_seqs w x h frames and n_per_seq point slots per sequence. */
int64_t klt_frame_step_ws_bytes(int w, int h, int n_seqs, int n_per_seq);

/* Pyramids as in klt_lk_track (sequence i: item prev_first + i*pair_stride of the previous pyramid, item
 * next_first + i*pair_stride of the next one; detection runs on level 0 of the next item).  d_pts: float32 x, y pairs,
 * [n_seqs][n_per_seq]; sequence i owns its first d_counts[i] points (device int32, 0 <= count <= n_per_seq; the slots
 * behind them are never read).  params: as klt_lk_track, without KLT_OPTFLOW_USE_INITIAL_FLOW.  Filter, mask and detection
 * parameters as klt_track_filter and klt_good_features_to_track_points_host, except max_corners >= 1
 * (KLT_ERR_UNSUPPORTED for 0: the output width must be bounded).
 * Outputs, device: row i of d_out_pts (float32 x, y pairs, out_stride >= n_per_seq + max_corners pairs per row) holds the
 * survivors in input order, then the new corners strongest first; d_keep [n_seqs][n_per_seq] (0 behind the count);
 * d_next_counts and d_n_new: int32 per sequence.  next_counts (host) receives d_next_counts.  d_ws: klt_frame_step_ws_bytes()
 * bytes, 256-byte aligned.
 * Runs on `stream` (the same kernels as klt_frame_step_batch_async; every frame is selected on the device) and
 * synchronises it once, to read back the next counts.  The device outputs are complete in stream order when the call
 * returns.  A count outside [0, n_per_seq] returns KLT_ERR_INVALID_ARG after that synchronisation, with the outputs
 * undefined.  Calls on one context that use this entry point are serialised (they share a pinned landing buffer). */
klt_status klt_frame_step_batch(klt_ctx* ctx,
                        const uint8_t* d_prev_img, const uint8_t* d_prev_pyr,
                        const uint8_t* d_next_img, const uint8_t* d_next_pyr,
                        const klt_pyr_layout* layout, int prev_first, int next_first, int pair_stride, int n_seqs,
                        const float* d_pts, const int32_t* d_counts, int n_per_seq, const klt_lk_params* params,
                        float max_bidir_error, int mask_radius, int max_corners, double quality_level, double min_distance,
                        int block_size, float* d_out_pts, int64_t out_stride, uint8_t* d_keep, int32_t* d_next_counts,
                        int32_t* d_n_new, int32_t* next_counts, void* d_ws, int64_t ws_bytes, void* stream);

/* The same step with no host involvement: every argument is a device pointer or a value, nothing is synchronised,
 * allocated or copied through the host, and everything runs on `stream`.  Frames can therefore be chained without
 * waiting (pass n_per_seq == out_stride == C and swap two point buffers), and the call can be captured into a CUDA graph
 * once one call has run eagerly on the same stream and device (that first call sets kernel attributes per device; the
 * pyramid builds the caller enqueues before it need the same first eager call).
 * Differences from klt_frame_step_batch:
 *  - out_stride >= n_per_seq is the capacity C of a row: sequence i gets at most min(max_corners, C - s_i) new corners,
 *    s_i its survivors (none when that is 0).  With that cap, the corners are the first ones cv2.goodFeaturesToTrack(...,
 *    maxCorners = min(max_corners, C - s_i)) returns, so d_next_counts[i] = s_i + d_n_new[i] <= C.
 *  - Track ids, optional (all three NULL or all given; d_ids_in may be NULL when n_per_seq == 0): d_ids_in
 *    [n_seqs][n_per_seq] and d_ids_out [n_seqs][out_stride] int32 ids of the points; d_next_id [n_seqs] int32, read and
 *    written.  A survivor's id moves with it; new corner j of sequence i gets id d_next_id[i] + j (strongest first), and
 *    d_next_id[i] grows by d_n_new[i].
 *  - d_flags (device uint32, not NULL): a count outside [0, n_per_seq] is clamped and sets *d_flags to 1 (bit 0); the
 *    caller clears it.  Nothing is read or written out of bounds. */
klt_status klt_frame_step_batch_async(klt_ctx* ctx,
                        const uint8_t* d_prev_img, const uint8_t* d_prev_pyr,
                        const uint8_t* d_next_img, const uint8_t* d_next_pyr,
                        const klt_pyr_layout* layout, int prev_first, int next_first, int pair_stride, int n_seqs,
                        const float* d_pts, const int32_t* d_counts, int n_per_seq, const klt_lk_params* params,
                        float max_bidir_error, int mask_radius, int max_corners, double quality_level, double min_distance,
                        int block_size, float* d_out_pts, int64_t out_stride, uint8_t* d_keep, int32_t* d_next_counts,
                        int32_t* d_n_new, const int32_t* d_ids_in, int32_t* d_ids_out, int32_t* d_next_id, uint32_t* d_flags,
                        void* d_ws, int64_t ws_bytes, void* stream);

/* ---- steering the chained step from a back end ------------------------------------------------------------------------
 * Device pointers a caller writes between two steps to end chosen tracks and to start sequences over.  The step reads
 * them in stream order, so they may be computed on the device, and a captured graph reads them at every replay.
 *   d_drop          [n_seqs][n_per_seq] uint8, or NULL (no drops): a nonzero entry ends the track in that input slot.
 *                   It is not a survivor, its d_keep is 0, and it does not enter the detection mask.  Entries at or behind
 *                   the sequence's count are ignored.  The step zeroes the whole array.
 *   d_restart       [n_seqs] uint8, or NULL (no restarts): nonzero starts sequence i over at this step, whose next frame
 *                   is frame 0 of the new sequence.  None of the old points survives (d_keep all 0; LK may still run on
 *                   them, its results are discarded); the output row starts with the staged points, and new corners are
 *                   appended behind them as in every step.  A restart takes precedence over drops in the same
 *                   sequence.  The step zeroes the array.
 *   d_restart_pts   [n_seqs][n_per_seq][2] float32 and d_restart_counts [n_seqs] int32: the staged points of sequence i
 *                   are its first d_restart_counts[i].  A count outside [0, n_per_seq] is clamped and sets *d_flags.
 *   d_restart_ids   [n_seqs][n_per_seq] int32 and d_restart_next_id [n_seqs] int32: ids of the staged points, and the
 *                   value d_next_id[i] takes before the new corners are numbered.  Given exactly when the step has ids.
 *   d_restarted     [n_seqs] uint8, written by every step: 1 where the sequence started over at this step.
 * The staged arrays are read only for sequences marked in d_restart and may be NULL when d_restart is. */
typedef struct klt_step_control {
    uint8_t* d_drop;
    uint8_t* d_restart;
    const float* d_restart_pts;
    const int32_t* d_restart_counts;
    const int32_t* d_restart_ids;
    const int32_t* d_restart_next_id;
    uint8_t* d_restarted;
} klt_step_control;

/* klt_frame_step_batch_async, steered by *control (not NULL; read when the call is made, so a graph keeps its
 * pointers).  KLT_ERR_INVALID_ARG as klt_frame_step_batch_async, and for a null control, a null d_restarted, d_restart
 * without staged points and counts, or staged ids / next id given without ids on the step, or the reverse. */
klt_status klt_frame_step_batch_control_async(klt_ctx* ctx,
                        const uint8_t* d_prev_img, const uint8_t* d_prev_pyr,
                        const uint8_t* d_next_img, const uint8_t* d_next_pyr,
                        const klt_pyr_layout* layout, int prev_first, int next_first, int pair_stride, int n_seqs,
                        const float* d_pts, const int32_t* d_counts, int n_per_seq, const klt_lk_params* params,
                        float max_bidir_error, int mask_radius, int max_corners, double quality_level, double min_distance,
                        int block_size, float* d_out_pts, int64_t out_stride, uint8_t* d_keep, int32_t* d_next_counts,
                        int32_t* d_n_new, const int32_t* d_ids_in, int32_t* d_ids_out, int32_t* d_next_id, uint32_t* d_flags,
                        void* d_ws, int64_t ws_bytes, const klt_step_control* control, void* stream);

/* ---- start positions of the chained step's forward pass ---------------------------------------------------------------
 * A back end that predicts where its tracks will be in the next frame hands the step those positions, and the forward LK
 * pass starts there instead of at the old position (cv2.calcOpticalFlowPyrLK(prev, next, p0, s,
 * flags=OPTFLOW_USE_INITIAL_FLOW)).  Nothing else of the step changes: the second pass still starts from the forward
 * result without the flag, and the two-pass border dispatch of the LK kernels still classifies a point by p0.
 *
 * klt_frame_step_batch_control_async (control may be NULL: no steering) with one more argument, d_init_pts
 * [n_seqs][n_per_seq][2] float32, in/out (not NULL when n_per_seq > 0): on entry slot j of sequence i holds the forward
 * pass's start position s[i][j] (read in stream order, so an earlier kernel may write it; entries at or behind the count
 * are not read); on return it holds the forward pass's result p1, which the step filters and compacts.  params must not
 * carry KLT_OPTFLOW_USE_INITIAL_FLOW itself: the call sets it for the forward pass.  KLT_ERR_INVALID_ARG as
 * klt_frame_step_batch_control_async, and for a null d_init_pts with n_per_seq > 0. */
klt_status klt_frame_step_batch_init_async(klt_ctx* ctx,
                        const uint8_t* d_prev_img, const uint8_t* d_prev_pyr,
                        const uint8_t* d_next_img, const uint8_t* d_next_pyr,
                        const klt_pyr_layout* layout, int prev_first, int next_first, int pair_stride, int n_seqs,
                        const float* d_pts, const int32_t* d_counts, int n_per_seq, const klt_lk_params* params,
                        float max_bidir_error, int mask_radius, int max_corners, double quality_level, double min_distance,
                        int block_size, float* d_out_pts, int64_t out_stride, uint8_t* d_keep, int32_t* d_next_counts,
                        int32_t* d_n_new, const int32_t* d_ids_in, int32_t* d_ids_out, int32_t* d_next_id, uint32_t* d_flags,
                        void* d_ws, int64_t ws_bytes, float* d_init_pts, const klt_step_control* control, void* stream);

/* ---- forward-backward check of the chained step ----------------------------------------------------------------------
 * klt_frame_step_batch_init_async with the second LK pass run from the new frame back into the old one (Kalal et al.,
 * 2010) instead of the reference's same-direction pass: per slot, with s the start positions (p0 when d_init_pts is NULL)
 *   p1  = LK(prev, next, p0)  started at s (OPTFLOW_USE_INITIAL_FLOW when d_init_pts is given)
 *   p0r = LK(next, prev, p1)  started at b = p1 - (s - p0) (float32, each operation rounded once) with the flag when
 *                             d_init_pts is given, else at p1 without it
 *   d   = max(|p0 - p0r|) over x, y; keep = d < max_bidir_error and p1 inside the image, as in every step.
 * On a correct track d is the tracking error rather than about twice the frame's motion, so a useful max_bidir_error is
 * about 1 px.  The reverse pass has the same size and launch shape as the same-direction pass it replaces; with start
 * positions the call adds one device-to-device copy of s and one small kernel that writes b.  The filter, compaction,
 * detection, ids and control are unchanged.
 * d_init_pts may be NULL (no start positions; otherwise as klt_frame_step_batch_init_async), control may be NULL (no
 * steering).  d_bidir_err [n_seqs][n_per_seq] float32 (may be NULL): d for every slot below the count, NaN behind it and
 * for a sequence restarted at this step.  KLT_ERR_INVALID_ARG as klt_frame_step_batch_control_async. */
klt_status klt_frame_step_batch_fb_async(klt_ctx* ctx,
                        const uint8_t* d_prev_img, const uint8_t* d_prev_pyr,
                        const uint8_t* d_next_img, const uint8_t* d_next_pyr,
                        const klt_pyr_layout* layout, int prev_first, int next_first, int pair_stride, int n_seqs,
                        const float* d_pts, const int32_t* d_counts, int n_per_seq, const klt_lk_params* params,
                        float max_bidir_error, int mask_radius, int max_corners, double quality_level, double min_distance,
                        int block_size, float* d_out_pts, int64_t out_stride, uint8_t* d_keep, int32_t* d_next_counts,
                        int32_t* d_n_new, const int32_t* d_ids_in, int32_t* d_ids_out, int32_t* d_next_id, uint32_t* d_flags,
                        void* d_ws, int64_t ws_bytes, float* d_init_pts, const klt_step_control* control, float* d_bidir_err,
                        void* stream);

/* ---- minimum distance between the chained step's tracks ---------------------------------------------------------------
 * Tracks that drift together (contracting image motion) fill a row with redundant tracks until the capacity stops
 * detection.  The step can end a survivor that comes closer than min_track_distance = d to an older one, as VINS-Mono's
 * setMask does before each detection, with Euclidean distance on the float positions:
 *   candidates  the input slots j < counts[i] that pass the filter (the bidirectional error and the inclusive bounds) and
 *               are not dropped by control;
 *   rule        candidates are visited in slot order; slot j is thinned when an earlier candidate i < j that was not
 *               thinned has dx * dx + dy * dy < d * d, with dx = double(x_j) - double(x_i) (dy alike) on the float32 p1
 *               positions, in float64, each subtraction, product and sum rounded once (no FMA: numpy float64 gives the
 *               same bits), and d * d rounded once; a distance of exactly d is not thinned;
 *   effect      a thinned slot gets d_keep 0 and d_thinned 1, is not written to the output row, does not enter the
 *               detection mask, and its track ends in the records like a dropped one; its d_bidir_err is still written.
 * Slot order is birth order: every row the step writes holds its survivors in input order, then the new corners strongest
 * first, so an older track wins, and within one birth frame the stronger corner.  For the initial rows and the staged
 * rows of a restart this holds only as far as the caller orders them.  A sequence restarted at this step thins nothing:
 * its staged points are taken as given.  The LK passes, the filter, the mask (discs of mask_radius around the kept
 * survivors), detection, ids, the capacity cap, drops and restarts are unchanged.  The step launches the same kernels:
 * the compaction does the thinning, with scratch taken from the workspace (klt_frame_step_ws_bytes is unchanged).
 *
 * klt_frame_step_batch_thin_async takes the arguments of klt_frame_step_batch_fb_async (d_init_pts, control and
 * d_bidir_err may be NULL) plus
 *   reverse             0: the reference's second pass (as klt_frame_step_batch_init_async), 1: the forward-backward check;
 *   min_track_distance  d, in (0, KLT_MAX_TRACK_DISTANCE] (a larger d thins exactly as that one does on any image the step
 *                       accepts, whose diagonal is shorter); NaN, infinite or <= 0: KLT_ERR_INVALID_ARG, larger:
 *                       KLT_ERR_UNSUPPORTED;
 *   d_thinned           [n_seqs][n_per_seq] uint8, may be NULL: 1 for a thinned slot, 0 elsewhere, behind the count and
 *                       for a restarted sequence.
 * KLT_ERR_INVALID_ARG as klt_frame_step_batch_fb_async, and for reverse outside {0, 1}.  These checks run before any
 * device work. */
#define KLT_MAX_TRACK_DISTANCE 131072.0
klt_status klt_frame_step_batch_thin_async(klt_ctx* ctx,
                        const uint8_t* d_prev_img, const uint8_t* d_prev_pyr,
                        const uint8_t* d_next_img, const uint8_t* d_next_pyr,
                        const klt_pyr_layout* layout, int prev_first, int next_first, int pair_stride, int n_seqs,
                        const float* d_pts, const int32_t* d_counts, int n_per_seq, const klt_lk_params* params,
                        float max_bidir_error, int mask_radius, int max_corners, double quality_level, double min_distance,
                        int block_size, float* d_out_pts, int64_t out_stride, uint8_t* d_keep, int32_t* d_next_counts,
                        int32_t* d_n_new, const int32_t* d_ids_in, int32_t* d_ids_out, int32_t* d_next_id, uint32_t* d_flags,
                        void* d_ws, int64_t ws_bytes, float* d_init_pts, const klt_step_control* control, float* d_bidir_err,
                        int reverse, double min_track_distance, uint8_t* d_thinned, void* stream);

/* ---- grid detection in the chained step -------------------------------------------------------------------------------
 * goodFeaturesToTrack on the whole frame takes the strongest corners first, so where contrast is uneven (shadow, sky, a
 * dark side of the street) every new track goes to the textured part and the pose solver sees tracks in part of the field
 * of view only.  Grid detection tops up each cell of a cols x rows grid to tracks_per_cell = q tracks instead, with the
 * cell's own quality threshold:
 *   cells       column edges X_i = floor(i * w / cols), row edges Y_j = floor(j * h / rows) (integer arithmetic); cell
 *               k = j * cols + i covers X_i <= u < X_(i+1), Y_j <= v < Y_(j+1).  1 <= cols <= w, 1 <= rows <= h.
 *   s_k         the points of the output row before detection (the kept survivors, or a restarted sequence's staged
 *               points) in cell k.  A point (x, y) counts in column max{i : X_i <= x} clamped to [0, cols - 1] (so x == w
 *               is in the last column, x < 0 in the first), rows alike; NaN counts nowhere.
 *   quota       n_k = max(0, q - s_k).
 *   L_k         cv2.goodFeaturesToTrack(frame, maxCorners = n_k, qualityLevel, minDistance, mask = M & R_k, blockSize),
 *               M the step's mask (255 with discs around the survivors), R_k the cell's rectangle: the threshold is the
 *               cell's masked maximum times qualityLevel, the 3x3 local-maximum test reads pixels across the cell edge,
 *               minDistance applies within a cell; empty when n_k == 0.
 *   row         the survivors, then L_0[0], L_1[0], ..., L_(G-1)[0], L_0[1], ... (exhausted cells skipped), cut to
 *               min(max_corners, C - survivors): a binding cap drops the weakest ranks of every cell evenly.  Ids follow
 *               the row, so within one birth frame the slot order is rank, then cell.
 * cols = rows = 1 with q = C is the step without the option (goodFeaturesToTrack is prefix-stable in maxCorners).
 * Per (sequence, cell): one block finds the cell's threshold, one block sorts its candidates, one block selects them; one
 * warp per sequence interleaves.  The kernels run on the stream with no synchronisation, allocation or host copy.
 *
 * klt_frame_step_batch_grid_async takes the arguments of klt_frame_step_batch_thin_async, with min_track_distance = 0
 * for no thinning (d_thinned is then unused), plus cols, rows and tracks_per_cell >= 1, in a workspace of
 * klt_frame_step_grid_ws_bytes() bytes.  KLT_ERR_INVALID_ARG as klt_frame_step_batch_thin_async, and for cols, rows or
 * tracks_per_cell < 1, cols > w or rows > h; KLT_ERR_UNSUPPORTED for cols * rows > KLT_MAX_GRID_CELLS.  These checks run
 * before any device work.
 * KLT_MAX_GRID_CELLS: the interleave runs one warp per sequence, whose lane c holds the largest count of cells
 * 32c .. 32c + 31, so 32 x 32 cells. */
#define KLT_MAX_GRID_CELLS 1024
int64_t klt_frame_step_grid_ws_bytes(int w, int h, int n_seqs, int n_per_seq, int cols, int rows);
klt_status klt_frame_step_batch_grid_async(klt_ctx* ctx,
                        const uint8_t* d_prev_img, const uint8_t* d_prev_pyr,
                        const uint8_t* d_next_img, const uint8_t* d_next_pyr,
                        const klt_pyr_layout* layout, int prev_first, int next_first, int pair_stride, int n_seqs,
                        const float* d_pts, const int32_t* d_counts, int n_per_seq, const klt_lk_params* params,
                        float max_bidir_error, int mask_radius, int max_corners, double quality_level, double min_distance,
                        int block_size, float* d_out_pts, int64_t out_stride, uint8_t* d_keep, int32_t* d_next_counts,
                        int32_t* d_n_new, const int32_t* d_ids_in, int32_t* d_ids_out, int32_t* d_next_id, uint32_t* d_flags,
                        void* d_ws, int64_t ws_bytes, float* d_init_pts, const klt_step_control* control, float* d_bidir_err,
                        int reverse, double min_track_distance, uint8_t* d_thinned, int cols, int rows, int tracks_per_cell,
                        void* stream);

/* Batched grid detection on device images: per image b and cell k (the cells above),
 * cv2.goodFeaturesToTrack(img_b, maxCorners = max_corners_per_cell, quality_level, min_distance, mask = mask_b & R_k,
 * block_size) -> d_corners [batch][cols * rows][max_corners_per_cell][2] float32 (strongest first; entries behind the
 * count undefined) and d_counts [batch][cols * rows] int32.  d_mask may be NULL (the cell alone).  d_ws:
 * klt_good_features_to_track_grid_ws_bytes() bytes, 256-byte aligned.  Asynchronous on `stream`. */
int64_t klt_good_features_to_track_grid_ws_bytes(int w, int h, int batch, int cols, int rows);
klt_status klt_good_features_to_track_grid(klt_ctx* ctx, const uint8_t* d_img, int w, int h, int64_t pitch, int64_t batch_stride,
                        int batch, int cols, int rows, int max_corners_per_cell, double quality_level, double min_distance,
                        int block_size, const uint8_t* d_mask, int64_t mask_pitch, int64_t mask_batch_stride, float* d_corners,
                        int32_t* d_counts, void* d_ws, int64_t ws_bytes, void* stream);

/* Writes the start positions d_init_pts [n_seqs][n_per_seq][2] float32 of the next klt_frame_step_batch_init_async from
 * the current rows d_pts / d_counts (those of that step).  Slot j < d_counts[i] of sequence i starts at
 *   1. d_guess_pts[i][j] when d_guess_mask[i][j] is nonzero (used as given: NaN, inf and positions outside the image too);
 *   2. else, with a ring (depth >= 2, the ring of klt_track_records_step below, of width W = n_per_seq, and d_frame), at
 *      p + (p - q) when the track has a position q one frame ago (klt_track_window with k = 2: its older entry is not NaN;
 *      false for new corners and at a sequence's frame 0), p = d_pts[i][j]; float32, each operation rounded once, no FMA;
 *   3. else at p, which gives the result of a step without start positions.
 * Slots behind the count get p.  d_guess_pts / d_guess_mask ([n_seqs][n_per_seq] uint8): both or neither (NULL: no
 * given positions); the call zeroes the whole mask, so a captured graph consumes each request once.  depth = 0: no
 * velocity, and the ring pointers may be NULL.  Asynchronous on `stream`, device pointers only, can be captured.
 * KLT_ERR_INVALID_ARG: a null context or required pointer, n_seqs < 1, n_per_seq < 0, depth < 0 or depth == 1. */
klt_status klt_track_predict(klt_ctx* ctx, int n_seqs, int n_per_seq, const float* d_pts, const int32_t* d_counts,
                        const float* d_guess_pts, uint8_t* d_guess_mask, int depth, const float* d_ring_pts,
                        const int32_t* d_ring_src, const int32_t* d_ring_counts, const int32_t* d_frame, float* d_init_pts,
                        void* stream);

/* ---- per-track records of the chained step ----------------------------------------------------------------------------
 * What a VO back end reads about each track (the reference's Keypoint.t_first / uv_first / uv_history), kept on the device
 * next to klt_frame_step_batch_async with track ids.  Both calls are asynchronous on `stream`, take device pointers and
 * values only, synchronise nothing and can be captured into a CUDA graph.
 *
 * Frame counters: d_frame [n_seqs] int32, the index of the frame sequence i's current row belongs to (0 for the first).
 * Per-slot state, moved with the points like the ids: first_pts (float32 x, y pairs) and first_frames (int32), the
 * position and frame at which the track in that slot was first seen.  Rows of width n_per_seq (input) and out_stride (output).
 *
 * Observation ring of depth R >= 1, width W = out_stride of the step (all int32 / float32, row-major):
 *   ring_pts    [R][n_seqs][W][2]  positions of the tracks in frame f, in slot order
 *   ring_ids    [R][n_seqs][W]     their track ids
 *   ring_src    [R][n_seqs][W]     each one's slot in frame f - 1's row, or -1 if the track was born at frame f
 *   ring_counts [R][n_seqs]        number of valid entries (the count of frame f's row)
 *   ring_frames [R][n_seqs]        f
 * Ring slot f mod R holds frame f; entries behind the count are never written or read.  A caller initialises frame 0
 * itself: d_frame[i] = 0, ring slot 0 = the initial points, ids, src = -1, their count and frame 0, and first_frames /
 * first_pts of the initial rows (0 and the initial points, or older values for tracks that predate the batch). */

/* Run after klt_frame_step_batch_async, on the same stream, with that step's d_keep [n_seqs][n_per_seq], d_out_pts /
 * d_ids_out [n_seqs][out_stride] and d_next_counts.  Survivor i of sequence s moves first_pts / first_frames from slot i of
 * the input rows to its output slot (the step keeps survivors in input order); the new corners (the slots behind the
 * survivors up to d_next_counts[s]) get their own position and frame d_frame[s] + 1.  Writes ring slot
 * (d_frame[s] + 1) mod R for the slots [0, d_next_counts[s]) (src of a survivor = its input index i), then increments
 * d_frame[s].  The input and output rows must not alias.  KLT_ERR_INVALID_ARG: a null required pointer (d_keep and the
 * input rows may be NULL only when n_per_seq == 0), R < 1, n_per_seq < 0 or out_stride < n_per_seq. */
klt_status klt_track_records_step(klt_ctx* ctx, int n_seqs, int n_per_seq, int64_t out_stride, const uint8_t* d_keep,
                        const float* d_out_pts, const int32_t* d_ids_out, const int32_t* d_next_counts,
                        const float* d_first_pts_in, const int32_t* d_first_frames_in, float* d_first_pts_out,
                        int32_t* d_first_frames_out, int32_t* d_frame, int depth, float* d_ring_pts, int32_t* d_ring_ids,
                        int32_t* d_ring_src, int32_t* d_ring_counts, int32_t* d_ring_frames, void* stream);

/* klt_track_records_step after klt_frame_step_batch_control_async, with that step's d_restarted and the staged
 * d_restart_counts (both not NULL).  A sequence that started over gets frame 0 instead of d_frame[s] + 1: its staged
 * slots [0, count) take the first positions d_restart_first_pts and first frames d_restart_first_frames ([n_seqs]
 * [n_per_seq], each NULL for "their position" and "0"), the new corners behind them frame 0, every entry of its ring row
 * src = -1, and d_frame[s] becomes 0.  After a restart, the ring rows of sequence s are valid only for frames in
 * [max(0, f - R + 1), f], f = d_frame[s]: the other rows belong to the previous sequence, which klt_track_window never
 * reaches (the src links of frame 0 are all -1).  KLT_ERR_INVALID_ARG as klt_track_records_step, and for a null
 * d_restarted or d_restart_counts. */
klt_status klt_track_records_step_control(klt_ctx* ctx, int n_seqs, int n_per_seq, int64_t out_stride, const uint8_t* d_keep,
                        const float* d_out_pts, const int32_t* d_ids_out, const int32_t* d_next_counts,
                        const float* d_first_pts_in, const int32_t* d_first_frames_in, float* d_first_pts_out,
                        int32_t* d_first_frames_out, int32_t* d_frame, int depth, float* d_ring_pts, int32_t* d_ring_ids,
                        int32_t* d_ring_src, int32_t* d_ring_counts, int32_t* d_ring_frames, const uint8_t* d_restarted,
                        const int32_t* d_restart_counts, const float* d_restart_first_pts, const int32_t* d_restart_first_frames,
                        void* stream);

/* The last k positions (1 <= k <= R) of every slot of the current rows, following the src links back through the ring:
 * d_out [n_seqs][width][k][2] float32, entry [s][j][k - 1 - d] = slot j's position d frames ago.  NaN before the track was
 * born, before frame 0, and for j >= the current count.  width: the ring's W.  KLT_ERR_INVALID_ARG: a null pointer,
 * R < 1, k outside [1, R], width < 0. */
klt_status klt_track_window(klt_ctx* ctx, int n_seqs, int64_t width, int depth, const float* d_ring_pts, const int32_t* d_ring_src,
                        const int32_t* d_ring_counts, const int32_t* d_frame, int k, float* d_out, void* stream);

/* ---- bilateral pre-filter (SURVEY.md s8f rank 3) ------------------------------------------------------------------
 * Replaces cv2.bilateralFilter(img, d=5, sigmaColor=1.5, sigmaSpace=1.5) as the reference's loader applies it to every
 * frame (src/loader/loader.py:16-20,86): 8-bit single channel, BORDER_REFLECT_101 (cv2's default), d <= 15.
 * Arithmetic: oracle/bilateral_oracle.c B.1-B.6 = OpenCV's own code path (an OpenCV build without IPP); differs from
 * it only on exact rounding ties (< 1e-5 of the pixels, by 1), and by at most 1 from the IPP-enabled wheel. */

/* Device pointers, batched, asynchronous on `stream`.  d_dst must not alias d_src. */
klt_status klt_bilateral_filter(klt_ctx* ctx, const uint8_t* d_src, int w, int h, int64_t src_pitch, int64_t src_batch_stride,
                        uint8_t* d_dst, int64_t dst_pitch, int64_t dst_batch_stride, int batch, int d, double sigma_color,
                        double sigma_space, void* stream);

/* HOST buffers, synchronous. */
klt_status klt_bilateral_filter_host(klt_ctx* ctx, const uint8_t* img, int64_t pitch, int w, int h, int d, double sigma_color,
                        double sigma_space, uint8_t* out, int64_t out_pitch);

/* ---- sub-pixel corner refinement ---------------------------------------------------------------------------------
 * cv2.cornerSubPix(img, corners, winSize = (win_w, win_h), zeroZone = (zero_w, zero_h), criteria = (crit_type, max_count,
 * eps)) on 8-bit single-channel images.  Arithmetic: oracle/subpix_oracle.c S.1-S.6 = OpenCV's own code path (an OpenCV
 * build without IPP, or cv2.ipp.setUseIPP(False)), bit for bit; the weight mask is computed on the host with the C
 * library's expf and passed to the kernel by value.  The IPP-enabled wheel computes the patch differently in the last
 * bits, so its results differ slightly (DESIGN.md).
 * KLT_MAX_SUBPIX_WIN: win_w and win_h supported.  One warp keeps (2 win_w + 1)(2 win_h + 1) x 5 double terms and the
 * float patch in shared memory, which at 15 x 15 (42.8 KB) still fits the 48 KB a block gets without an opt-in; the
 * by-value mask is then 3.8 KB of kernel parameters. */
#define KLT_MAX_SUBPIX_WIN 15

/* Device pointers, batched, asynchronous on `stream`, graph-capturable (no allocation, copy or synchronisation).
 * Image b is d_img + b * batch_stride (rows `pitch` bytes apart).  Row b of d_pts holds row_stride float32 (x, y) pairs
 * starting at d_pts + 2 * b * row_stride; the call refines, in place, the slots [e - n, e) with e = clamp(d_end[b], 0,
 * row_stride) and n = clamp(d_n[b], 0, e) (device int32 arrays, read in stream order).  A frame step passes its
 * d_next_counts and d_n_new (its new corners); a plain batch passes its counts twice.  A slot whose point is NaN or
 * outside [0, w) x [0, h) is left unchanged (cv2 raises there).  Criteria as cv2: max_iters = clamp(max_count, 1, 100)
 * with KLT_TERM_COUNT, else 100; eps = max(eps, 0) with KLT_TERM_EPS, else 0.  Checked before any device work:
 * KLT_ERR_INVALID_ARG for a null pointer, batch < 1, win_w or win_h < 1, w < 2 win_w + 5, h < 2 win_h + 5, pitch < w or
 * row_stride < 0; KLT_ERR_UNSUPPORTED for win_w or win_h > KLT_MAX_SUBPIX_WIN or batch > 65535. */
klt_status klt_corner_sub_pix(klt_ctx* ctx, const uint8_t* d_img, int w, int h, int64_t pitch, int64_t batch_stride, int batch,
                        float* d_pts, int64_t row_stride, const int32_t* d_end, const int32_t* d_n, int win_w, int win_h,
                        int zero_w, int zero_h, int crit_type, int max_count, double eps, void* stream);

/* HOST image and points, synchronous: refines pts[n][2] in place, like cv2.cornerSubPix.  Errors as above (no device
 * work is done then); points that are NaN or outside the image are left unchanged (the Python drop-in raises first). */
klt_status klt_corner_sub_pix_host(klt_ctx* ctx, const uint8_t* img, int64_t pitch, int w, int h, float* pts, int n, int win_w,
                        int win_h, int zero_w, int zero_h, int crit_type, int max_count, double eps);

/* ---- contrast-limited adaptive histogram equalisation -------------------------------------------------------------
 * cv2.createCLAHE(clip_limit, (tiles_x, tiles_y)).apply(img) on 8-bit single-channel images, bit for bit as OpenCV 4.13's
 * CLAHE_Impl::apply computes it (oracle/clahe_oracle.py C.1-C.5; IPP does not change this function):
 *   C.1 padding: none when w % tiles_x == 0 and h % tiles_y == 0; otherwise BORDER_REFLECT_101 on the right by
 *       tiles_x - w % tiles_x and at the bottom by tiles_y - h % tiles_y (an axis that divides still gets a whole tile).
 *   C.2 tile tw x th = padded size / tiles, total = tw * th, lut_scale = 255.0f / (float)total.
 *   C.3 clip = max((int)(clip_limit * total / 256), 1) in double when clip_limit > 0, else 0 (no clipping).
 *   C.4 per tile: 256-bin histogram; with clip > 0 every bin cut at clip, the excess e spread as e / 256 to every bin and
 *       one more to bins 0, s, 2s, ... (s = max(256 / r, 1), the first r = e % 256 of them); then
 *       lut[v] = saturate_u8(rint((float)cumsum[v] * lut_scale)).
 *   C.5 per pixel: tyf = y * (1.0f / th) - 0.5f, ty1 = floor(tyf), ya = tyf - ty1, ty2 = min(ty1 + 1, tiles_y - 1),
 *       ty1 = max(ty1, 0), the same along x, and dst = saturate_u8(rint((L11 * xa1 + L12 * xa) * ya1 + (L21 * xa1 + L22 * xa)
 *       * ya)) in float32, each operation rounded once.
 * Differences from cv2: arguments on which cv2 crashes or overflows are rejected (below), and only 8-bit images are
 * taken (cv2 also equalises 16-bit ones).
 * KLT_MAX_CLAHE_TILES: tiles_x * tiles_y supported.  At that many tiles a KITTI frame has tiles of a few pixels each,
 * far past any grid that equalises usefully, and one image's LUTs already take 16 MB of workspace. */
#define KLT_MAX_CLAHE_TILES 65536

/* Workspace of klt_clahe: batch * tiles_x * tiles_y * 256 bytes (the LUTs); 0 for batch, tiles_x or tiles_y < 1. */
int64_t klt_clahe_ws_bytes(int batch, int tiles_x, int tiles_y);

/* Device pointers, batched, asynchronous on `stream`, graph-capturable (two launches; no allocation, copy or
 * synchronisation).  Image b is d_src + b * src_batch_stride, written to d_dst + b * dst_batch_stride.  d_dst may equal
 * d_src (in place; then with the same pitch and batch stride); any other overlap is undefined.  d_ws: ws_bytes >=
 * klt_clahe_ws_bytes(batch, tiles_x, tiles_y), 8-byte aligned.  Checked before any device work: KLT_ERR_INVALID_ARG for a
 * null pointer, w, h or batch < 1, a pitch < w, tiles_x or tiles_y < 1 (cv2 dies of SIGFPE on a 0 and asserts on a
 * negative), a non-finite clip_limit, a clip_limit whose clip_limit * total / 256 does not fit an int32 (undefined
 * behaviour in cv2), d_dst == d_src with another pitch or batch stride, or a workspace too small or misaligned;
 * KLT_ERR_UNSUPPORTED for tiles_x * tiles_y > KLT_MAX_CLAHE_TILES, a tile of more than 2^31 - 1 pixels, batch > 65535 or
 * h > 524280. */
klt_status klt_clahe(klt_ctx* ctx, const uint8_t* d_src, int w, int h, int64_t src_pitch, int64_t src_batch_stride, uint8_t* d_dst,
                        int64_t dst_pitch, int64_t dst_batch_stride, int batch, double clip_limit, int tiles_x, int tiles_y, void* d_ws,
                        int64_t ws_bytes, void* stream);

/* HOST buffers, synchronous (the context's workspace and stream).  out may equal img.  Errors as above. */
klt_status klt_clahe_host(klt_ctx* ctx, const uint8_t* img, int64_t pitch, int w, int h, double clip_limit, int tiles_x, int tiles_y,
                        uint8_t* out, int64_t out_pitch);

#ifdef __cplusplus
}
#endif
#endif /* KLT_B200_H */
