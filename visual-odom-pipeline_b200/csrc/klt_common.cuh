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
};

klt_status lk_launch(const LKLaunch& L, int sm_count, cudaStream_t stream);
klt_status track_filter_launch(const float* p0, const float* p1, const float* p0r, long long n, float max_bidir_error,
                               int w, int h, uint8_t* keep, float* bidir, cudaStream_t stream);
klt_status lk_launch_fast(const LKLaunch& L, int sm_count, int forced_wpp, cudaStream_t stream);
klt_status lk_init(int device);

// Bilateral pre-filter (klt_bilateral.cu)
int bilateral_radius(int d, double sigma_space);
int bilateral_table_capacity();
int bilateral_tables(int d, double sigma_color, double sigma_space, float* tab, int capacity);
klt_status bilateral_launch(const uint8_t* src, int w, int h, long long spitch, long long sbatch, uint8_t* dst, long long dpitch,
                            long long dbatch, int batch, int radius, int n_taps, const float* d_tab, cudaStream_t stream);

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
// 255 everywhere, filled cv2.circle(radius) of 0 around np.int32 of every point (reference extractor.py:102-107)
klt_status corner_mask_from_points_launch(const float* pts, int n, int radius, int w, int h, uint8_t* mask, long long pitch,
                                          cudaStream_t stream);

}  // namespace klt
