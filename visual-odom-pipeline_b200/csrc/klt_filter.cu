// Bidirectional-error / bounds filter of the reference's tracking step on the device.
//
// Replaces, per point, reference src/extractor/extractor.py:46-47,53 (extend_tracks) and :67-68,75 (extend_landmarks):
//     d = abs(p0 - p0r).reshape(-1, 2).max(-1);  good = d < max_bidir_error
//     keep = good and 0 <= x <= W and 0 <= y <= H          (x, y) = p1, inclusive bounds
// where p1 = LK(im0, im1, p0) and p0r = LK(im0, im1, p1) -- the reference's second call runs in the SAME direction,
// started from the forward result; it is reproduced as is.  float32 arithmetic like numpy's: |a - b| rounds once,
// max() and the comparisons are exact, NaN fails every test.  track_compact_kernel applies the same test to a batch of
// padded point sets and compacts the survivors (the batched frame step, klt_frame_step_batch).
#include "klt_common.cuh"

namespace klt {

namespace {

// The reference's test for one point; `d` receives the bidirectional error.
__device__ __forceinline__ bool track_keep(float2 a, float2 q, float2 b, float max_bidir_error, float w, float h, float& d)
{
    const float dx = fabsf(__fsub_rn(a.x, b.x)), dy = fabsf(__fsub_rn(a.y, b.y));
    // numpy's max propagates NaN; fmaxf would drop it
    d = (dx != dx || dy != dy) ? __int_as_float(0x7fc00000) : fmaxf(dx, dy);
    const bool good = d < max_bidir_error;
    const bool inside = (0.f <= q.x) && (q.x <= w) && (0.f <= q.y) && (q.y <= h);
    return good && inside;
}

__global__ void __launch_bounds__(256)
track_filter_kernel(const float2* __restrict__ p0, const float2* __restrict__ p1, const float2* __restrict__ p0r,
                    long long n, float max_bidir_error, float w, float h, uint8_t* __restrict__ keep,
                    float* __restrict__ bidir)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float d;
    keep[i] = track_keep(p0[i], p1[i], p0r[i], max_bidir_error, w, h, d) ? 1 : 0;
    if (bidir) bidir[i] = d;
}

// One CTA per sequence walks its points in chunks of kCompactThreads; a block-wide prefix count of the kept flags gives
// each survivor its slot, so the survivors keep their input order.  kIds: each survivor's track id moves with it (a
// template parameter, so that the launch without ids runs the same code as before ids existed).
constexpr int kCompactThreads = 1024;

template <bool kIds>
__global__ void __launch_bounds__(kCompactThreads)
track_compact_kernel(const float2* __restrict__ p0, const float2* __restrict__ p1, const float2* __restrict__ p0r,
                     const int* __restrict__ counts, int n_per_seq, float max_bidir_error, float w, float h,
                     uint8_t* __restrict__ keep, float2* __restrict__ out, long long out_stride, int* __restrict__ n_keep,
                     unsigned* __restrict__ bad_counts, const int* __restrict__ ids_in, int* __restrict__ ids_out)
{
    __shared__ int s_warp[kCompactThreads / 32];
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wrp = tid >> 5;
    const int c = counts[b];
    if (c < 0 || c > n_per_seq) {
        if (tid == 0) *bad_counts = 1u;
    }
    const int n = min(max(c, 0), n_per_seq);
    const long long row = (long long)b * n_per_seq;
    float2* __restrict__ dst = out + (long long)b * out_stride;
    int base = 0;
    for (int i0 = 0; i0 < n_per_seq; i0 += kCompactThreads) {
        const int i = i0 + tid;
        bool k = false;
        float2 q = make_float2(0.f, 0.f);
        if (i < n) {
            float d;
            q = p1[row + i];
            k = track_keep(p0[row + i], q, p0r[row + i], max_bidir_error, w, h, d);
        }
        if (i < n_per_seq) keep[row + i] = k ? 1 : 0;
        if (i0 >= n) continue;   // uniform: the rest of the row is padding
        const unsigned m = __ballot_sync(0xffffffffu, k);
        if (lane == 0) s_warp[wrp] = __popc(m);
        __syncthreads();
        int before = __popc(m & ((1u << lane) - 1u)), total = 0;
#pragma unroll
        for (int j = 0; j < kCompactThreads / 32; ++j) {
            const int t = s_warp[j];
            before += j < wrp ? t : 0;
            total += t;
        }
        if (k) {
            dst[base + before] = q;
            if (kIds) ids_out[(long long)b * out_stride + base + before] = ids_in[row + i];
        }
        base += total;
        __syncthreads();   // s_warp is rewritten by the next chunk
    }
    if (tid == 0) n_keep[b] = base;
}

}  // namespace

klt_status track_filter_launch(const float* p0, const float* p1, const float* p0r, long long n, float max_bidir_error,
                               int w, int h, uint8_t* keep, float* bidir, cudaStream_t stream)
{
    if (n < 0 || w <= 0 || h <= 0) return KLT_ERR_INVALID_ARG;
    if (n == 0) return KLT_OK;
    if (!p0 || !p1 || !p0r || !keep) return KLT_ERR_INVALID_ARG;
    const long long blocks = (n + 255) / 256;
    if (blocks > 0x7fffffffLL) return KLT_ERR_UNSUPPORTED;
    track_filter_kernel<<<(unsigned)blocks, 256, 0, stream>>>(reinterpret_cast<const float2*>(p0), reinterpret_cast<const float2*>(p1),
                                                               reinterpret_cast<const float2*>(p0r), n, max_bidir_error, (float)w, (float)h,
                                                               keep, bidir);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KLT_OK : (klt_status)e;
}

klt_status track_compact_launch(const float* p0, const float* p1, const float* p0r, const int* counts, int batch, int n_per_seq,
                                float max_bidir_error, int w, int h, uint8_t* keep, float* out, long long out_stride, int* n_keep,
                                unsigned* bad_counts, const int* ids_in, int* ids_out, cudaStream_t stream)
{
    if (batch < 1 || n_per_seq < 0 || w <= 0 || h <= 0 || out_stride < n_per_seq || !counts || !out || !n_keep || !bad_counts)
        return KLT_ERR_INVALID_ARG;
    if (n_per_seq > 0 && (!p0 || !p1 || !p0r || !keep)) return KLT_ERR_INVALID_ARG;
    if (!ids_in != !ids_out) return KLT_ERR_INVALID_ARG;
    auto kernel = ids_in ? track_compact_kernel<true> : track_compact_kernel<false>;
    kernel<<<batch, kCompactThreads, 0, stream>>>(
        reinterpret_cast<const float2*>(p0), reinterpret_cast<const float2*>(p1), reinterpret_cast<const float2*>(p0r), counts, n_per_seq,
        max_bidir_error, (float)w, (float)h, keep, reinterpret_cast<float2*>(out), out_stride, n_keep, bad_counts, ids_in, ids_out);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KLT_OK : (klt_status)e;
}

}  // namespace klt
