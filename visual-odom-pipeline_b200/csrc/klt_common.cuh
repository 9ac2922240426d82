// Shared device/host helpers for the KLT kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "klt_b200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libklt_b200 is written for sm_100a (B200) only"
#endif

namespace klt {

// One pyramid level as kernel argument (device pointer already offset to batch item 0).
struct LevelView {
    const uint8_t* data;
    long long batch_stride;
    int pitch;
    int w, h;
    int aligned4;  // data, pitch and batch_stride are multiples of 4: rows may be read with 32-bit loads
};

struct PyrView {
    LevelView lv[KLT_MAX_LEVELS];
    int top;
};

// BORDER_REFLECT_101 for any distance (SURVEY.md A.2).  len >= 1.
__host__ __device__ __forceinline__ int reflect101(int p, int len)
{
    if ((unsigned)p < (unsigned)len) return p;
    if (len == 1) return 0;
    do {
        p = (p < 0) ? -p : 2 * len - 2 - p;
    } while ((unsigned)p >= (unsigned)len);
    return p;
}

// cudaFuncSetAttribute is per device: a process that drives several GPUs must opt each of them in to the large
// dynamic shared memory of a kernel.  Returns true when the current device still needs it for this call site.
struct PerDeviceOnce {
    bool done[64] = {};
    bool needed()
    {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return true;   // unknown: just set it again
        if (done[dev]) return false;
        done[dev] = true;
        return true;
    }
};

// Programmatic dependent launch.  A kernel launched with launch_pdl may start while the kernel before it in the stream is
// still running.  Before pdl_wait it does parameter and index work only: no global read of anything an earlier kernel may
// have written, no global write.  pdl_wait returns once every earlier kernel has completed and its writes are visible.
// pdl_launch_dependents, called after pdl_wait, lets the next kernel's CTAs be dispatched; since that kernel waits in turn,
// a kernel that follows with or without this attribute still sees all of this kernel's writes.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// Launches `kernel` with the programmatic-stream-serialization attribute and, when cluster > 1, clusters of `cluster` CTAs
// along x.
template <typename... KArgs, typename... Args>
cudaError_t launch_pdl(void (*kernel)(KArgs...), unsigned grid, unsigned block, size_t smem, cudaStream_t stream, unsigned cluster,
                       Args&&... args)
{
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    attr[1].id = cudaLaunchAttributeClusterDimension;
    attr[1].val.clusterDim.x = cluster;
    attr[1].val.clusterDim.y = 1;
    attr[1].val.clusterDim.z = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(block);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cfg.attrs = attr;
    cfg.numAttrs = cluster > 1 ? 2 : 1;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, static_cast<Args&&>(args)...);
    if (e != cudaSuccess) cudaGetLastError();   // reported here; not left for the next cudaGetLastError of the caller
    return e;
}

// u / d for small operands via a 12.20 reciprocal: exact for u < 4096, 1 <= d <= 64
// (u*magic < 2^32 and the rounding excess u*e/2^20 stays below 1/d).
__host__ __device__ __forceinline__ unsigned fastdiv_magic(unsigned d) { return ((1u << 20) + d - 1u) / d; }
__host__ __device__ __forceinline__ unsigned fastdiv(unsigned u, unsigned magic) { return (u * magic) >> 20; }

klt_status pyr_down_launch(const uint8_t* src, int w, int h, long long spitch, long long sbatch,
                           uint8_t* dst, long long dpitch, long long dbatch, int batch, int sm_count,
                           cudaStream_t stream);

// Whole pyramid in one launch (klt_pyramid.cu: pyr_build_fused_kernel)
struct PyrStep {
    const uint8_t* src;
    uint8_t* dst;
    long long spitch, sbatch, dpitch, dbatch;
    int w, h, dw, dh;
    int rows, tiles_x, n8, rem_nout, strips_y;   // warp tasks of the step: tiles_x x strips_y x batch
    int cnt_off;                                 // first completion counter of the step ([image][strip])
    long long task_begin;
};
struct PyrFused {
    PyrStep s[KLT_MAX_LEVELS - 1];
    int n_steps, batch;
    long long n_tasks;
    unsigned* cnt;      // completion counters, monotonic: a strip of launch number `gen` is complete at gen * tiles_x
    unsigned gen;               // launch number on the counter array, from the host (ordinary launches)
    unsigned long long* done;   // graph-safe form: CTAs finished in all launches on this counter array so far (gen - 1 = done / grid size)
    // Reuse of pyramids across calls of the host entry points (klt_capi.cu: track_host): item b is left as it is when
    // bit b of reuse_mask is set and the content hash of its freshly uploaded level 0 (hash_new, 2 words per item) equals
    // the hash of the image its levels were built from (hash_old).  hash_clear: 4 words zeroed for the call after next.
    // skipped: statistics counter (items skipped).  All null / 0 for ordinary builds.
    const unsigned* hash_new;
    const unsigned* hash_old;
    unsigned* hash_clear;
    unsigned long long* skipped;
    unsigned reuse_mask;
};
klt_status pyr_fused_plan(PyrFused& P, int n_steps, const uint8_t* const* src, uint8_t* const* dst, const int* w, const int* h,
                          const long long* spitch, const long long* sbatch, const long long* dpitch, const long long* dbatch,
                          int batch, int sm_count, long long* n_counters);
klt_status pyr_fused_launch(const PyrFused& P, bool device_gen, cudaStream_t stream);

// Small batch: one thread-block cluster per image builds all levels (klt_pyramid.cu: pyr_build_cluster_kernel).  Level l
// (1..top) is split into bands of rows[l] rows, band k held by CTA k of the cluster in shared memory.
struct PyrCluster {
    const uint8_t* src;                 // level 0 of item 0
    long long spitch, sbatch;
    uint8_t* dst[KLT_MAX_LEVELS];       // level l of item 0 (l >= 1)
    long long dpitch[KLT_MAX_LEVELS], dbatch[KLT_MAX_LEVELS];
    int w[KLT_MAX_LEVELS], h[KLT_MAX_LEVELS];
    int rows[KLT_MAX_LEVELS];           // band height of level l
    int stride[KLT_MAX_LEVELS];         // shared-memory row stride of level l (l = 0: the staged level-0 rows)
    int buf1;                           // byte offset of the second band buffer (odd levels)
    int top, ctas, batch;
    int smem;                           // dynamic shared memory of a CTA
    // pyramid reuse, as in PyrFused
    const unsigned* hash_new;
    const unsigned* hash_old;
    unsigned* hash_clear;
    unsigned long long* skipped;
    unsigned reuse_mask;
};
// KLT_ERR_UNSUPPORTED: not a small batch, a level 0 band does not fit the shared-memory budget, or a level cannot take
// the ring kernel's loads and stores (the caller then takes pyr_fused_plan or one launch per level).
klt_status pyr_cluster_plan(PyrCluster& P, int n_steps, const uint8_t* const* src, uint8_t* const* dst, const int* w, const int* h,
                            const long long* spitch, const long long* sbatch, const long long* dpitch, const long long* dbatch,
                            int batch);
klt_status pyr_cluster_launch(const PyrCluster& P, cudaStream_t stream);

// Copies n_img tightly/oddly pitched u8 images (image i at src + i * sbatch, rows spitch apart, any alignment) into
// 16-byte-aligned pitched storage.  The source buffer must be readable up to 16 bytes past the last pixel.
// hash (optional): 2 words per image, zero on entry, receive a 64-bit content hash of the w x h pixels (position-dependent
// mix of every 16-byte chunk, summed).
klt_status repitch_launch(const uint8_t* src, long long spitch, long long sbatch, uint8_t* dst, long long dpitch,
                          long long dbatch, int w, int h, int n_img, cudaStream_t stream, unsigned* hash = nullptr);

struct LKLaunch {
    PyrView prev, next;
    const float* prev_pts;
    float* next_pts;
    uint8_t* status;
    float* err;
    int* iters;
    int n_per_pair;
    int batch;
    int win_w, win_h;
    int max_count;
    double eps2;
    // float brackets of eps2 for the termination test: dx*dx + dy*dy evaluated in float32 is within 2^-22 (relative) of
    // the double value OpenCV compares, so  s <= eps2_lo  decides "<= eps2" and  s >= eps2_hi  decides "> eps2"; only
    // values in between (practically never) take the double-precision path.  lo < 0 / hi = inf disable the shortcut.
    float eps2_lo, eps2_hi;
    int flags;
    float min_eig_thr;
    // optional, device: points per pair (<= n_per_pair), written by earlier kernels.  Point i of pair b is skipped (nothing
    // read or written) when i >= counts[b].  Null: every pair has n_per_pair points.
    const int* counts = nullptr;
};

klt_status lk_launch(const LKLaunch& L, int sm_count, cudaStream_t stream);
klt_status track_filter_launch(const float* p0, const float* p1, const float* p0r, long long n, float max_bidir_error,
                               int w, int h, uint8_t* keep, float* bidir, cudaStream_t stream);
// Filter plus stable compaction for a batch of padded point sets (one CTA per sequence): sequence b owns points
// [0, counts[b]) of row b (n_per_seq points per row of p0 / p1 / p0r).  keep[b][i] as in track_filter_launch (0 for
// i >= counts[b]); the survivors of p1 go in input order to out[b * out_stride + 0 .. s_b - 1] (float2), s_b to n_keep[b].
// A count outside [0, n_per_seq] is clamped and sets *bad_counts to 1.  ids_in [batch][n_per_seq] / ids_out
// [batch][out_stride] (both or neither): the track id of each survivor goes to the same slot of ids_out as its point.
// control (may be NULL): drops and restarts as klt_step_control describes (checked by the caller); a restart sets
// next_id[b] (may be NULL) to the staged counter.  bidir [batch][n_per_seq] (may be NULL): each slot's error d, NaN
// behind the count and for a restarted sequence.  thin (may be NULL): the minimum track distance of
// klt_frame_step_batch_thin_async, with its scratch.
struct TrackThin {
    double min_dist;            // d, in (0, KLT_MAX_TRACK_DISTANCE]
    uint8_t* thinned;           // [batch][n_per_seq], may be NULL
    int* heads;                 // scratch: heads_stride ints per sequence, at least the grid's cells (w * h suffices)
    long long heads_stride;
    unsigned* links;            // scratch: [batch][n_per_seq]
};
klt_status track_compact_launch(const float* p0, const float* p1, const float* p0r, const int* counts, int batch, int n_per_seq,
                                float max_bidir_error, int w, int h, uint8_t* keep, float* out, long long out_stride, int* n_keep,
                                unsigned* bad_counts, const int* ids_in, int* ids_out, const klt_step_control* control, int* next_id,
                                float* bidir, const TrackThin* thin, cudaStream_t stream);
// Per-track records of one step (klt_track_records_step; one CTA per sequence, run after the step on the same stream).
// keep [batch][n_per_seq], out / ids_out [batch][out_stride] and next_counts are the step's; first_pts / first_frames
// rows have the widths of the step's input and output rows; the ring is laid out as include/klt_b200.h describes.
// restarted (NULL: the step had no control) / restart_counts [batch] and the optional restart_first_pts /
// restart_first_frames [batch][n_per_seq]: the restarts of klt_frame_step_batch_control_async (klt_track_records_step_control).
klt_status track_records_launch(const uint8_t* keep, int batch, int n_per_seq, const float* out, const int* ids_out, long long out_stride,
                                const int* next_counts, const float* first_pts_in, const int* first_frames_in, float* first_pts_out,
                                int* first_frames_out, int* frame, int depth, float* ring_pts, int* ring_ids, int* ring_src,
                                int* ring_counts, int* ring_frames, const uint8_t* restarted, const int* restart_counts,
                                const float* restart_first_pts, const int* restart_first_frames, cudaStream_t stream);
// The last k positions of every slot, followed back through the ring (klt_track_window): out [batch][width][k] float2.
klt_status track_window_launch(const float* ring_pts, const int* ring_src, const int* ring_counts, const int* frame, int depth, int batch,
                               long long width, int k, float* out, cudaStream_t stream);
// Start positions of the next step's forward LK pass (klt_track_predict): init [batch][n_per_seq] float2 from the given
// positions (guess_pts / guess_mask, both or neither; the mask is cleared), the velocity of the ring of width n_per_seq
// (depth >= 2; 0: none) or the current points.
klt_status track_predict_launch(const float* pts, const int* counts, int batch, int n_per_seq, const float* guess_pts, uint8_t* guess_mask,
                                int depth, const float* ring_pts, const int* ring_src, const int* ring_counts, const int* frame,
                                float* init, cudaStream_t stream);
// Start of the reverse second pass after a forward pass from start positions: start [batch][n_per_seq] float2 holds the
// starts s on entry and b = p1 - (s - p0) on return, for the slots below each sequence's count.
klt_status track_mirror_start_launch(const float* p0, const float* p1, const int* counts, int batch, int n_per_seq, float* start,
                                     cudaStream_t stream);
klt_status lk_launch_fast(const LKLaunch& L, int sm_count, cudaStream_t stream);
klt_status lk_init(int device);

// Bilateral pre-filter (klt_bilateral.cu)
int bilateral_radius(int d, double sigma_space);
int bilateral_table_capacity();
int bilateral_tables(int d, double sigma_color, double sigma_space, float* tab, int capacity);
klt_status bilateral_launch(const uint8_t* src, int w, int h, long long spitch, long long sbatch, uint8_t* dst, long long dpitch,
                            long long dbatch, int batch, int radius, int n_taps, const float* d_tab, cudaStream_t stream);

// Contrast-limited histogram equalisation (klt_clahe.cu)
struct ClahePlan {
    int tiles_x, tiles_y, tw, th, clip;   // tw x th: the padded tile; clip 0: no clipping
    float lut_scale, inv_tw, inv_th;
};
klt_status clahe_plan(int w, int h, double clip_limit, int tiles_x, int tiles_y, ClahePlan* p);
long long clahe_lut_bytes(int batch, int tiles_x, int tiles_y);
klt_status clahe_launch(const uint8_t* src, int w, int h, long long spitch, long long sbatch, uint8_t* dst, long long dpitch,
                        long long dbatch, int batch, const ClahePlan& p, uint8_t* lut, cudaStream_t stream);

// Sub-pixel corner refinement (klt_subpix.cu)
void subpix_mask(int win_w, int win_h, int zero_w, int zero_h, float* mask);
klt_status subpix_launch(const uint8_t* imgs, int w, int h, long long pitch, long long batch_stride, int batch, float* pts,
                         long long row_stride, const int* d_end, const int* d_n, int win_w, int win_h, int zero_w, int zero_h,
                         int crit_type, int max_count, double eps, cudaStream_t stream);

// Shi-Tomasi detection (klt_corners.cu)
long long corners_ws_bytes(int w, int h, int batch);
klt_status corner_min_eig_launch(const uint8_t* img, long long pitch, long long batch_stride, int w, int h, int batch,
                                 int block, float* eig, long long eig_pitch, long long eig_batch_stride,
                                 const uint8_t* mask, long long mask_pitch, long long mask_batch_stride,
                                 unsigned* max_out, void* ws, cudaStream_t stream);
klt_status corner_candidates_launch(const float* eig, long long eig_pitch, long long eig_batch_stride, int w, int h, int batch,
                                    const uint8_t* mask, long long mask_pitch, long long mask_batch_stride,
                                    const unsigned* max_in, double quality, unsigned long long* keys,
                                    long long keys_batch_stride, int capacity, unsigned* count, cudaStream_t stream);
// sorts each item's keys (descending) when there are at most 8192 (rank: batch * 8192 zeroed words of scratch);
// out[0] = count | sorted << 32, keys from out[1]
klt_status corner_sort_launch(const unsigned long long* keys, long long keys_batch_stride, const unsigned* count, int batch,
                              unsigned* rank, unsigned long long* out, long long out_batch_stride, int out_capacity,
                              cudaStream_t stream);
// 255 everywhere, filled cv2.circle(radius) of 0 around np.int32 of every point (reference extractor.py:102-107), for a
// batch: item b's points are pts[b * pts_stride + 0 .. n_b - 1] (float2), n_b = counts[b] (device, clamped to [0, n]) or n
// when counts is null; its mask starts at mask + b * mask_batch_stride.
klt_status corner_mask_from_points_launch(const float* pts, long long pts_stride, const int* counts, int n, int batch, int radius,
                                          int w, int h, uint8_t* mask, long long pitch, long long mask_batch_stride,
                                          cudaStream_t stream);
// Descending radix sort, in place, of the items with more than 8192 keys (count[b] keys at keys + b * keys_batch_stride;
// alt: scratch of the same layout).  One launch whatever the counts: the other items return at once.
klt_status corner_radix_sort_launch(unsigned long long* keys, long long keys_batch_stride, const unsigned* count, int batch,
                                    unsigned long long* alt, long long alt_batch_stride, cudaStream_t stream);
// Greedy minimum-distance selection on the device, one CTA per image: every image, any min_distance >= 0.  Keys: the
// sorted lists of corner_sort_launch (sorted, header first) for images with at most 8192 of them, else the list
// corner_radix_sort_launch sorted in `keys`.  Item b's corners go to out[b * out_stride + first[b] ..] (float2), at most
// min(max_corners, cap - first[b]) of them (max_corners >= 1); next_counts[b] = first[b] + n_new[b].  ids_out / next_id
// (both or neither): corner j of item b gets id next_id[b] + j in the same slot of ids_out; next_id[b] += n_new[b].
// gbitmap: scratch of batch x gbitmap_stride words, used (and zeroed on the stream) when an image's bitmap exceeds the
// shared memory budget (180 KB, e.g. 3840 x 2160).
klt_status corner_select_launch(const unsigned long long* sorted, long long sorted_batch_stride, const unsigned long long* keys,
                                long long keys_batch_stride, int w, int h, int batch, double min_distance, int max_corners,
                                long long cap, const int* first, float* out, long long out_stride, int* next_counts, int* n_new,
                                int* ids_out, int* next_id, unsigned* gbitmap, long long gbitmap_stride, cudaStream_t stream);

// Grid detection (klt_corners.cu): cols x rows cells, column edges floor(i * w / cols), row edges floor(j * h / rows),
// cols * rows <= KLT_MAX_GRID_CELLS.  Per-cell arrays are [batch][cols * rows].
// quota[b][k] = max(0, q - s_k), s_k the first first[b] (clamped to [0, n_max]) points of item b (float2 at pts +
// b * pts_stride) in cell k (a point counts in the last column / row with a position <= its own, clamped; NaN nowhere).
klt_status corner_grid_quota_launch(const float* pts, long long pts_stride, const int* first, int n_max, int batch, int w, int h, int cols,
                                    int rows, int q, int* quota, cudaStream_t stream);
// Per (item, cell): cv2.goodFeaturesToTrack(maxCorners = k_max, qualityLevel, minDistance, mask & cell) on the eigenvalue
// map, k_max = min(max_corners, cap - first[b], quota[b][k]) (first / quota may be null: no such bound).  The cell's
// corners end at the front of its segment of keys (item stride keys_batch_stride >= w * h; cell k's segment at
// Y_j * w + X_i * (Y_(j+1) - Y_j)) as (y << 16) | x, strongest first, and n_sel[b][k] counts them.  thr, seg_count:
// per-cell scratch; alt: scratch shaped like keys; gbitmap: batch x gbitmap_stride (>= w * h) words, used (and zeroed on
// the stream) when a cell's bitmap exceeds the shared memory budget.  The eigenvalue map may be gbitmap.
klt_status corner_grid_detect_launch(const float* eig, long long eig_pitch, long long eig_batch_stride, int w, int h, int batch,
                                     const uint8_t* mask, long long mask_pitch, long long mask_batch_stride, int cols, int rows,
                                     double quality, double min_distance, int max_corners, long long cap, const int* first,
                                     const int* quota, float* thr, unsigned* seg_count, int* n_sel, unsigned long long* keys,
                                     long long keys_batch_stride, unsigned long long* alt, long long alt_batch_stride, unsigned* gbitmap,
                                     long long gbitmap_stride, cudaStream_t stream);
// Writes the cells' corners behind the first[b] points of out's row b, interleaved by rank and cut to
// min(max_corners, cap - first[b]); next_counts, n_new, ids_out / next_id as corner_select_launch.
klt_status corner_grid_interleave_launch(const unsigned long long* keys, long long keys_batch_stride, const int* n_sel, int w, int h, int batch,
                                         int cols, int rows, int max_corners, long long cap, const int* first, float* out,
                                         long long out_stride, int* next_counts, int* n_new, int* ids_out, int* next_id,
                                         cudaStream_t stream);
// out[b][k][0 .. n_sel[b][k]) (q pairs per cell, float32 x, y) and counts[b][k] = n_sel[b][k].
klt_status corner_grid_out_launch(const unsigned long long* keys, long long keys_batch_stride, const int* n_sel, int w, int h, int batch,
                                  int cols, int rows, int q, float* out, int* counts, cudaStream_t stream);

}  // namespace klt
