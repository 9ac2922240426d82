// Bidirectional-error / bounds filter of the reference's tracking step on the device.
//
// Replaces, per point, reference src/extractor/extractor.py:46-47,53 (extend_tracks) and :67-68,75 (extend_landmarks):
//     d = abs(p0 - p0r).reshape(-1, 2).max(-1);  good = d < max_bidir_error
//     keep = good and 0 <= x <= W and 0 <= y <= H          (x, y) = p1, inclusive bounds
// where p1 = LK(im0, im1, p0) and p0r = LK(im0, im1, p1) -- the reference's second call runs in the SAME direction,
// started from the forward result; it is reproduced as is.  float32 arithmetic like numpy's: |a - b| rounds once,
// max() and the comparisons are exact, NaN fails every test.  track_compact_kernel applies the same test to a batch of
// padded point sets and compacts the survivors (the batched frame step, klt_frame_step_batch).  The forward-backward
// check (klt_frame_step_batch_fb_async, klt_track_fb_host) runs the same test on p0r = LK(im1, im0, p1), the second pass
// in the reverse direction; only p0r changes.
#include <algorithm>
#include <cmath>

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
// template parameter, so that the launch without ids runs the same code as before ids existed).  kControl: the step is
// steered by a klt_step_control (another instance, for the same reason): dropped slots are not kept, a restarted
// sequence keeps nothing and starts its output row with the staged points, and both requests are cleared.
// kBidir: also store each input slot's error d (NaN behind the count and for a restarted sequence).  It is one instance,
// launched with kIds and kControl set, that finds out at run time whether the step has ids and control.
// kThin: the minimum track distance (klt_frame_step_batch_thin_async; ThinGrid below).  One more instance, launched with
// the other three set, that finds out at run time whether the step has ids, control and an error output.
constexpr int kCompactThreads = 1024;

// The minimum track distance of one step.  The candidates (slots that pass the filter and are not dropped) are visited in
// slot order, and a candidate is thinned when an earlier candidate that was not thinned lies closer than d:
// dx * dx + dy * dy < d * d in float64 on the float32 positions, each operation rounded once.  Each CTA keeps a uniform
// grid of cell side s >= d over its image, so a conflict lies in the 3 x 3 cells around a candidate.  Every candidate
// is pushed onto the singly linked list of its cell (heads: one int per cell, -1 = empty; links: per slot, the next
// slot + 1 in bits 0..30 and "thinned" in bit 31), so the grid is exact at any density, exact duplicates included.  A
// chunk's candidates are resolved as in select_corners_kernel: a candidate is thinned as soon as a conflicting earlier
// one is kept, and kept as soon as every conflicting earlier one is thinned; the earliest undecided candidate always
// decides, so the rounds end.  Slots of earlier chunks are final, read from bit 31 of their link.
struct ThinGrid {
    double md2;                 // d * d
    double inv_s;               // 1 / s
    int gw, gh;                 // cells per row and per column
    uint8_t* thinned;           // may be null
    int* heads;
    long long heads_stride;
    unsigned* links;
};

// kThin: one CTA per SM is enough, so ptxas may use 64 registers (50, no spills, against 32 and spills by default); the
// other instances keep the bounds they had (0: unspecified).
template <bool kIds, bool kControl, bool kBidir, bool kThin>
__global__ void __launch_bounds__(kCompactThreads, kThin ? 1 : 0)
track_compact_kernel(const float2* __restrict__ p0, const float2* __restrict__ p1, const float2* __restrict__ p0r,
                     const int* __restrict__ counts, int n_per_seq, float max_bidir_error, float w, float h,
                     uint8_t* __restrict__ keep, float2* __restrict__ out, long long out_stride, int* __restrict__ n_keep,
                     unsigned* __restrict__ bad_counts, const int* __restrict__ ids_in, int* __restrict__ ids_out,
                     const klt_step_control ctl, int* __restrict__ next_id, float* __restrict__ bidir, const ThinGrid thin)
{
    __shared__ int s_warp[kCompactThreads / 32];
    __shared__ uint8_t s_state[kThin ? kCompactThreads : 1];   // this chunk's candidates: 0 undecided, 1 kept, 2 thinned
    const bool has_ids = kIds && (!kBidir || ids_in != nullptr);
    const bool has_ctl = kControl && (!kBidir || ctl.d_restarted != nullptr);
    const bool has_bidir = kBidir && (!kThin || bidir != nullptr);
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wrp = tid >> 5;
    const int c = counts[b];
    if (c < 0 || c > n_per_seq) {
        if (tid == 0) *bad_counts = 1u;
    }
    const bool restart = has_ctl && ctl.d_restart && ctl.d_restart[b] != 0;
    const int n = restart ? 0 : min(max(c, 0), n_per_seq);
    const long long row = (long long)b * n_per_seq;
    uint8_t* __restrict__ drop = has_ctl && ctl.d_drop ? ctl.d_drop + row : nullptr;
    float2* __restrict__ dst = out + (long long)b * out_stride;
    int* heads = nullptr;
    unsigned* links = nullptr;
    if (kThin && n > 0) {   // uniform
        heads = thin.heads + (long long)b * thin.heads_stride;
        links = thin.links + row;
        for (int j = tid; j < thin.gw * thin.gh; j += kCompactThreads) heads[j] = -1;
        __syncthreads();
    }
    int base = 0;
    for (int i0 = 0; i0 < n_per_seq; i0 += kCompactThreads) {
        const int i = i0 + tid;
        bool k = false;
        float2 q = make_float2(0.f, 0.f);
        float d = __int_as_float(0x7fc00000);
        if (i < n) {
            q = p1[row + i];
            k = track_keep(p0[row + i], q, p0r[row + i], max_bidir_error, w, h, d);
            if (has_ctl && drop) k = k && drop[i] == 0;
        }
        bool t = false;
        if (kThin && i0 < n) {   // uniform
            // a candidate lies inside [0, w] x [0, h] (the filter's bounds), so its cell is in the grid
            int cx = 0, cy = 0;
            if (k) {
                cx = min((int)__dmul_rn((double)q.x, thin.inv_s), thin.gw - 1);
                cy = min((int)__dmul_rn((double)q.y, thin.inv_s), thin.gh - 1);
                links[i] = (unsigned)(atomicExch(heads + (long long)cy * thin.gw + cx, i) + 1);
            }
            s_state[tid] = 0;
            __syncthreads();   // every candidate of the chunk is in the grid
            const double qx = (double)q.x, qy = (double)q.y;
            bool decided = !k;
            while (true) {
                uint8_t verdict = 0;
                if (!decided) {
                    bool hit = false, pending = false;
                    for (int gy = max(cy - 1, 0); gy <= min(cy + 1, thin.gh - 1) && !hit; ++gy) {
                        for (int gx = max(cx - 1, 0); gx <= min(cx + 1, thin.gw - 1) && !hit; ++gx) {
                            int e = heads[(long long)gy * thin.gw + gx];
                            while (e >= 0 && !hit) {
                                const unsigned l = links[e];
                                if (e < i) {
                                    const uint8_t st = e < i0 ? ((l >> 31) ? 2 : 1) : s_state[e - i0];
                                    if (st != 2) {
                                        const float2 r = p1[row + e];
                                        const double dx = __dsub_rn(qx, (double)r.x), dy = __dsub_rn(qy, (double)r.y);
                                        if (__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)) < thin.md2) {
                                            if (st == 1) hit = true;
                                            else pending = true;
                                        }
                                    }
                                }
                                e = (int)(l & 0x7fffffffu) - 1;
                            }
                        }
                    }
                    verdict = hit ? 2 : pending ? 0 : 1;
                }
                __syncthreads();   // everyone has read the previous state
                if (verdict) {
                    s_state[tid] = verdict;
                    decided = true;
                }
                if (!__syncthreads_or(!decided)) break;
            }
            t = k && s_state[tid] == 2;
            if (t) {
                links[i] |= 0x80000000u;   // read by the next chunks' walks, after the __syncthreads below
                k = false;
            }
        }
        if (i < n_per_seq) {
            keep[row + i] = k ? 1 : 0;
            if (has_ctl && drop) drop[i] = 0;
            if (has_bidir) bidir[row + i] = d;
            if (kThin && thin.thinned) thin.thinned[row + i] = t ? 1 : 0;
        }
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
            if (has_ids) ids_out[(long long)b * out_stride + base + before] = ids_in[row + i];
        }
        base += total;
        __syncthreads();   // s_warp is rewritten by the next chunk
    }
    if (has_ctl) {
        if (restart) {
            const int sc = ctl.d_restart_counts[b];
            if ((sc < 0 || sc > n_per_seq) && tid == 0) *bad_counts = 1u;
            base = min(max(sc, 0), n_per_seq);
            const float2* __restrict__ src = reinterpret_cast<const float2*>(ctl.d_restart_pts) + row;
            for (int j = tid; j < base; j += kCompactThreads) {
                dst[j] = src[j];
                if (has_ids) ids_out[(long long)b * out_stride + j] = ctl.d_restart_ids[row + j];
            }
        }
        __syncthreads();   // every thread has read the restart flag
        if (tid == 0) {
            if (restart && next_id) next_id[b] = ctl.d_restart_next_id[b];
            if (ctl.d_restart) ctl.d_restart[b] = 0;
            ctl.d_restarted[b] = restart ? 1 : 0;
        }
    }
    if (tid == 0) n_keep[b] = base;
}

// Per-track records of the step that track_compact_kernel and select_corners_kernel just finished (one CTA per sequence).
// Survivor i of sequence b goes to the slot track_compact_kernel gave it: the same block-wide prefix count over keep,
// which is 0 behind the count, so the slots match.  Slots [s_b, next_counts[b]) hold the new corners.
// kRestart: after a steered step.  A restarted sequence has no survivors (keep is all 0), its frame becomes 0, and its
// staged slots [0, count) take the staged first positions / frames when they are given.
struct RestartRecords {
    const uint8_t* restarted;
    const int* counts;
    const float2* first_pts;
    const int* first_frames;
};

template <bool kRestart>
__global__ void __launch_bounds__(kCompactThreads, 1)
track_records_kernel(const uint8_t* __restrict__ keep, int n_per_seq, const float2* __restrict__ out, const int* __restrict__ ids_out,
                     long long out_stride, const int* __restrict__ next_counts, const float2* __restrict__ first_pts_in,
                     const int* __restrict__ first_frames_in, float2* __restrict__ first_pts_out, int* __restrict__ first_frames_out,
                     int* __restrict__ frame, int depth, int n_seqs, float2* __restrict__ ring_pts, int* __restrict__ ring_ids,
                     int* __restrict__ ring_src, int* __restrict__ ring_counts, int* __restrict__ ring_frames, const RestartRecords rs)
{
    __shared__ int s_warp[kCompactThreads / 32];
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wrp = tid >> 5;
    const bool restarted = kRestart && rs.restarted[b] != 0;
    const int f1 = restarted ? 0 : frame[b] + 1;                   // the frame this step produced
    const int n_staged = restarted ? min(max(rs.counts[b], 0), n_per_seq) : 0;
    const int r = ((f1 % depth) + depth) % depth;
    const long long row_in = (long long)b * n_per_seq, row_out = (long long)b * out_stride;
    const long long ring_row = ((long long)r * n_seqs + b) * out_stride;
    keep += row_in; first_pts_in += row_in; first_frames_in += row_in;
    out += row_out; ids_out += row_out; first_pts_out += row_out; first_frames_out += row_out;
    ring_pts += ring_row; ring_ids += ring_row; ring_src += ring_row;
    int base = 0;
    for (int i0 = 0; i0 < n_per_seq; i0 += kCompactThreads) {
        const int i = i0 + tid;
        const bool k = i < n_per_seq && keep[i] != 0;
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
            const int o = base + before;
            first_pts_out[o] = first_pts_in[i];
            first_frames_out[o] = first_frames_in[i];
            ring_pts[o] = out[o];
            ring_ids[o] = ids_out[o];
            ring_src[o] = i;
        }
        base += total;
        __syncthreads();   // s_warp is rewritten by the next chunk
    }
    const int n = (int)min((long long)max(next_counts[b], base), out_stride);
    for (int j = base + tid; j < n; j += kCompactThreads) {
        const float2 q = out[j];
        if (kRestart && j < n_staged) {
            first_pts_out[j] = rs.first_pts ? rs.first_pts[row_in + j] : q;
            first_frames_out[j] = rs.first_frames ? rs.first_frames[row_in + j] : 0;
        } else {
            first_pts_out[j] = q;
            first_frames_out[j] = f1;
        }
        ring_pts[j] = q;
        ring_ids[j] = ids_out[j];
        ring_src[j] = -1;
    }
    __syncthreads();   // every thread has read frame[b]
    if (tid == 0) {
        ring_counts[(long long)r * n_seqs + b] = n;
        ring_frames[(long long)r * n_seqs + b] = f1;
        frame[b] = f1;
    }
}

// The last k positions of slot j of sequence b, whose current frame is f: dst[k - 1 - d] is the slot's position d frames
// ago, found by following d src links back through the ring; NaN before the track was born, before frame 0 and behind
// the count.  Shared by track_window_kernel and track_predict_kernel.
__device__ __forceinline__ void track_window_walk(const float2* __restrict__ ring_pts, const int* __restrict__ ring_src,
                                                  const int* __restrict__ ring_counts, int f, int depth, int n_seqs, int b,
                                                  long long width, long long j, int k, float2* __restrict__ dst)
{
    const float nan = __int_as_float(0x7fc00000);
    long long pos = j < ring_counts[(long long)(((f % depth) + depth) % depth) * n_seqs + b] ? j : -1;
    for (int d = 0; d < k; ++d) {
        const int fd = f - d;
        float2 v = make_float2(nan, nan);
        if (fd >= 0 && pos >= 0 && pos < width) {
            const long long row = ((long long)(fd % depth) * n_seqs + b) * width;
            v = ring_pts[row + pos];
            pos = ring_src[row + pos];
        } else {
            pos = -1;
        }
        dst[k - 1 - d] = v;
    }
}

// Window of the last k positions of every slot (one thread per sequence and slot): out[b][j] = track_window_walk.
__global__ void __launch_bounds__(256)
track_window_kernel(const float2* __restrict__ ring_pts, const int* __restrict__ ring_src, const int* __restrict__ ring_counts,
                    const int* __restrict__ frame, int depth, int n_seqs, long long width, int k, float2* __restrict__ out)
{
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (long long)n_seqs * width) return;
    const int b = (int)(t / width);
    const long long j = t - (long long)b * width;
    track_window_walk(ring_pts, ring_src, ring_counts, frame[b], depth, n_seqs, b, width, j, k, out + t * k);
}

// Start positions of the next step's forward LK pass (klt_track_predict; one thread per sequence and slot).  Slot j of
// sequence b, j < counts[b], starts at the given position when guess_mask marks it; otherwise, with a ring (depth >= 2),
// at p + (p - q) when the track has a position q one frame ago (a window of k = 2 whose older entry is not NaN), p its
// current position; otherwise at p.  Each coordinate is rounded once per operation, as numpy's float32 would.  Slots
// behind the count start at p (the step never reads them).  The whole mask is cleared, so each request is used once.
__global__ void __launch_bounds__(256)
track_predict_kernel(const float2* __restrict__ pts, const int* __restrict__ counts, int n_per_seq, int n_seqs,
                     const float2* __restrict__ guess_pts, uint8_t* __restrict__ guess_mask, int depth,
                     const float2* __restrict__ ring_pts, const int* __restrict__ ring_src, const int* __restrict__ ring_counts,
                     const int* __restrict__ frame, float2* __restrict__ init)
{
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (long long)n_seqs * n_per_seq) return;
    const int b = (int)(t / n_per_seq);
    const int j = (int)(t - (long long)b * n_per_seq);
    float2 s = pts[t];
    if (j < min(max(counts[b], 0), n_per_seq)) {
        if (guess_mask && guess_mask[t] != 0) {
            s = guess_pts[t];
        } else if (depth > 0) {
            float2 w[2];
            track_window_walk(ring_pts, ring_src, ring_counts, frame[b], depth, n_seqs, b, n_per_seq, j, 2, w);
            const float2 q = w[0];
            if (q.x == q.x) s = make_float2(__fadd_rn(s.x, __fsub_rn(s.x, q.x)), __fadd_rn(s.y, __fsub_rn(s.y, q.y)));
        }
    }
    if (guess_mask) guess_mask[t] = 0;
    init[t] = s;
}

// Start of the reverse second pass when the forward pass had start positions s (klt_frame_step_batch_fb_async; one thread
// per sequence and slot): the forward pass started s - p0 away from p0, so the reverse pass starts as far from p1 in the
// other direction, b = p1 - (s - p0), each subtraction rounded once, as numpy's float32 would.  `start` holds s on entry
// and b on return; slots behind the count are not touched (the LK pass does not read them).
__global__ void __launch_bounds__(256)
track_mirror_start_kernel(const float2* __restrict__ p0, const float2* __restrict__ p1, const int* __restrict__ counts, int n_per_seq,
                          int n_seqs, float2* __restrict__ start)
{
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (long long)n_seqs * n_per_seq) return;
    const int b = (int)(t / n_per_seq);
    const int j = (int)(t - (long long)b * n_per_seq);
    if (j >= min(max(counts[b], 0), n_per_seq)) return;
    const float2 a = p0[t], q = p1[t], s = start[t];
    start[t] = make_float2(__fsub_rn(q.x, __fsub_rn(s.x, a.x)), __fsub_rn(q.y, __fsub_rn(s.y, a.y)));
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
                                unsigned* bad_counts, const int* ids_in, int* ids_out, const klt_step_control* control, int* next_id,
                                float* bidir, const TrackThin* thin, cudaStream_t stream)
{
    if (batch < 1 || n_per_seq < 0 || w <= 0 || h <= 0 || out_stride < n_per_seq || !counts || !out || !n_keep || !bad_counts)
        return KLT_ERR_INVALID_ARG;
    if (n_per_seq > 0 && (!p0 || !p1 || !p0r || !keep)) return KLT_ERR_INVALID_ARG;
    if (!ids_in != !ids_out) return KLT_ERR_INVALID_ARG;
    const klt_step_control ctl = control ? *control : klt_step_control{};
    ThinGrid g{};
    if (thin) {
        if (!(thin->min_dist > 0.0 && thin->min_dist <= KLT_MAX_TRACK_DISTANCE)) return KLT_ERR_INVALID_ARG;
        if (n_per_seq > 0 && (!thin->heads || !thin->links)) return KLT_ERR_INVALID_ARG;
        // cell side s: at least d (a conflict lies in the 3 x 3 cells), at least 2 (then the cells number at most w * h),
        // and large enough for about one cell per slot (fewer cells to clear per step); the factor keeps two positions
        // closer than d in adjacent cells whatever the rounding of x * (1 / s)
        const double s = std::max(std::max(thin->min_dist, 2.0), std::sqrt((double)w * h / std::max(n_per_seq, 1024))) * (1.0 + 0x1p-20);
        g.md2 = thin->min_dist * thin->min_dist;
        g.inv_s = 1.0 / s;
        g.gw = (int)((double)w * g.inv_s) + 1;
        g.gh = (int)((double)h * g.inv_s) + 1;
        if ((long long)g.gw * g.gh > thin->heads_stride) return KLT_ERR_INVALID_ARG;
        g.thinned = thin->thinned;
        g.heads = thin->heads;
        g.heads_stride = thin->heads_stride;
        g.links = thin->links;
    }
    auto kernel = thin ? track_compact_kernel<true, true, true, true>
                : bidir ? track_compact_kernel<true, true, true, false>
                : control ? (ids_in ? track_compact_kernel<true, true, false, false> : track_compact_kernel<false, true, false, false>)
                          : (ids_in ? track_compact_kernel<true, false, false, false> : track_compact_kernel<false, false, false, false>);
    kernel<<<batch, kCompactThreads, 0, stream>>>(
        reinterpret_cast<const float2*>(p0), reinterpret_cast<const float2*>(p1), reinterpret_cast<const float2*>(p0r), counts, n_per_seq,
        max_bidir_error, (float)w, (float)h, keep, reinterpret_cast<float2*>(out), out_stride, n_keep, bad_counts, ids_in, ids_out, ctl,
        next_id, bidir, g);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KLT_OK : (klt_status)e;
}

klt_status track_records_launch(const uint8_t* keep, int batch, int n_per_seq, const float* out, const int* ids_out, long long out_stride,
                                const int* next_counts, const float* first_pts_in, const int* first_frames_in, float* first_pts_out,
                                int* first_frames_out, int* frame, int depth, float* ring_pts, int* ring_ids, int* ring_src,
                                int* ring_counts, int* ring_frames, const uint8_t* restarted, const int* restart_counts,
                                const float* restart_first_pts, const int* restart_first_frames, cudaStream_t stream)
{
    if (batch < 1 || n_per_seq < 0 || out_stride < n_per_seq || out_stride > 0x7fffffff || depth < 1) return KLT_ERR_INVALID_ARG;
    if (!out || !ids_out || !next_counts || !first_pts_out || !first_frames_out || !frame || !ring_pts || !ring_ids || !ring_src ||
        !ring_counts || !ring_frames)
        return KLT_ERR_INVALID_ARG;
    if (n_per_seq > 0 && (!keep || !first_pts_in || !first_frames_in)) return KLT_ERR_INVALID_ARG;
    if (restarted && !restart_counts) return KLT_ERR_INVALID_ARG;
    const RestartRecords rs{restarted, restart_counts, reinterpret_cast<const float2*>(restart_first_pts), restart_first_frames};
    auto kernel = restarted ? track_records_kernel<true> : track_records_kernel<false>;
    kernel<<<batch, kCompactThreads, 0, stream>>>(
        keep, n_per_seq, reinterpret_cast<const float2*>(out), ids_out, out_stride, next_counts, reinterpret_cast<const float2*>(first_pts_in),
        first_frames_in, reinterpret_cast<float2*>(first_pts_out), first_frames_out, frame, depth, batch, reinterpret_cast<float2*>(ring_pts),
        ring_ids, ring_src, ring_counts, ring_frames, rs);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KLT_OK : (klt_status)e;
}

klt_status track_window_launch(const float* ring_pts, const int* ring_src, const int* ring_counts, const int* frame, int depth, int batch,
                               long long width, int k, float* out, cudaStream_t stream)
{
    if (batch < 1 || width < 0 || width > 0x7fffffff || depth < 1 || k < 1 || k > depth) return KLT_ERR_INVALID_ARG;
    if (!ring_pts || !ring_src || !ring_counts || !frame || !out) return KLT_ERR_INVALID_ARG;
    const long long blocks = ((long long)batch * width + 255) / 256;
    if (blocks == 0) return KLT_OK;
    if (blocks > 0x7fffffffLL) return KLT_ERR_UNSUPPORTED;
    track_window_kernel<<<(unsigned)blocks, 256, 0, stream>>>(reinterpret_cast<const float2*>(ring_pts), ring_src, ring_counts, frame, depth,
                                                               batch, width, k, reinterpret_cast<float2*>(out));
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KLT_OK : (klt_status)e;
}

klt_status track_predict_launch(const float* pts, const int* counts, int batch, int n_per_seq, const float* guess_pts, uint8_t* guess_mask,
                                int depth, const float* ring_pts, const int* ring_src, const int* ring_counts, const int* frame,
                                float* init, cudaStream_t stream)
{
    if (batch < 1 || n_per_seq < 0 || depth < 0 || depth == 1 || !counts) return KLT_ERR_INVALID_ARG;
    if (n_per_seq > 0 && (!pts || !init)) return KLT_ERR_INVALID_ARG;
    if (!guess_pts != !guess_mask) return KLT_ERR_INVALID_ARG;
    if (depth > 0 && (!ring_pts || !ring_src || !ring_counts || !frame)) return KLT_ERR_INVALID_ARG;
    const long long blocks = ((long long)batch * n_per_seq + 255) / 256;
    if (blocks == 0) return KLT_OK;
    if (blocks > 0x7fffffffLL) return KLT_ERR_UNSUPPORTED;
    track_predict_kernel<<<(unsigned)blocks, 256, 0, stream>>>(reinterpret_cast<const float2*>(pts), counts, n_per_seq, batch,
                                                                reinterpret_cast<const float2*>(guess_pts), guess_mask, depth,
                                                                reinterpret_cast<const float2*>(ring_pts), ring_src, ring_counts, frame,
                                                                reinterpret_cast<float2*>(init));
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KLT_OK : (klt_status)e;
}

klt_status track_mirror_start_launch(const float* p0, const float* p1, const int* counts, int batch, int n_per_seq, float* start,
                                     cudaStream_t stream)
{
    if (batch < 1 || n_per_seq < 0 || !counts) return KLT_ERR_INVALID_ARG;
    if (n_per_seq > 0 && (!p0 || !p1 || !start)) return KLT_ERR_INVALID_ARG;
    const long long blocks = ((long long)batch * n_per_seq + 255) / 256;
    if (blocks == 0) return KLT_OK;
    if (blocks > 0x7fffffffLL) return KLT_ERR_UNSUPPORTED;
    track_mirror_start_kernel<<<(unsigned)blocks, 256, 0, stream>>>(reinterpret_cast<const float2*>(p0), reinterpret_cast<const float2*>(p1),
                                                                     counts, n_per_seq, batch, reinterpret_cast<float2*>(start));
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KLT_OK : (klt_status)e;
}

}  // namespace klt
