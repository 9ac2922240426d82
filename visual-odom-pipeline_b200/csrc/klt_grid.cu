// Grid detection (include/klt_b200.h: klt_frame_step_batch_grid_async, klt_good_features_to_track_grid): the
// goodFeaturesToTrack of klt_corners.cu run per cell of a cols x rows grid, with the cell's own quality threshold and
// quota, for a batch of images.  The per-pixel and per-candidate arithmetic is that of klt_corners.cu (G.7, G.8); the
// eigenvalue map comes from corner_min_eig_launch.  Kept in a file of its own so that the kernels of klt_corners.cu
// compile exactly as before.
//   cell_quota_kernel       per image: the points of the row in each cell, and the quota max(0, q - s_k);
//   cell_threshold_kernel   per (cell, image): the cell's masked maximum eigenvalue times qualityLevel;
//   cell_candidates_kernel  candidates_kernel with the threshold of each pixel's cell, into per-cell segments;
//   cell_rank_sort_kernel, cell_radix_sort_kernel   per (cell, image): descending sort of the segment (shared memory up
//                           to kCellSortSmem keys, else the radix sort of klt_corners.cu);
//   cell_select_kernel      per (cell, image): the greedy minimum-distance selection of select_corners_kernel, with a
//                           bitmap of the cell only, up to the cell's quota;
//   cell_interleave_kernel  per image (one warp): the cells' corners by rank behind the survivors, under the cap;
//   cell_corners_out_kernel per (cell, image): the standalone detector's (B, G, q, 2) output.
#include "klt_common.cuh"

namespace klt {

namespace {

// as klt_corners.cu
constexpr unsigned kFullMask = 0xffffffffu;
constexpr int kRadixThreads = 1024;
constexpr int kRadixWarps = kRadixThreads / 32;
constexpr int kSelThreads = 128;
constexpr int kSelMaxRadius = 63;
constexpr int kSelMaxBitmapWords = 45 * 1024;   // 180 KB

__device__ __forceinline__ unsigned ordered_from_float(float f)
{
    const unsigned b = __float_as_uint(f);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float float_from_ordered(unsigned u)
{
    return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

// largest dx with dx^2 + dy^2 < md2 (-1: none)
__device__ __forceinline__ int sel_halfwidth(long long md2, int dy)
{
    const long long rem = md2 - (long long)dy * dy;
    if (rem <= 0) return -1;
    int hx = (int)sqrt((double)(rem - 1));
    while ((long long)hx * hx >= rem) --hx;
    while ((long long)(hx + 1) * (hx + 1) < rem) ++hx;
    return hx;
}

// The image is split into cols x rows cells, column edges X_i = floor(i * w / cols), row edges Y_j = floor(j * h / rows);
// cell k = j * cols + i.  Per (image, cell) the kernels below reproduce cv2.goodFeaturesToTrack(img, maxCorners = n_k,
// qualityLevel, minDistance, mask = M & R_k): the threshold comes from the cell's own masked maximum, the 3x3
// local-maximum test reads pixels across the cell edge (thresholded with the cell's threshold), and minDistance applies
// within the cell.  The candidates of cell k go to their own segment of the image's key list, at the pixel offset of the
// cell in a cell-major layout (Y_j * w + X_i * (Y_(j+1) - Y_j)), whose size is the cell's area: no segment can overflow.
struct CellGrid {
    int cols, rows, w, h;
    __host__ __device__ int x_edge(int i) const { return (int)((long long)i * w / cols); }
    __host__ __device__ int y_edge(int j) const { return (int)((long long)j * h / rows); }
    __device__ int col_of(int x) const { return (int)(((long long)(x + 1) * cols - 1) / w); }   // max{i : X_i <= x}, 0 <= x < w
    __device__ int row_of(int y) const { return (int)(((long long)(y + 1) * rows - 1) / h); }
    __host__ __device__ long long seg_off(int k) const
    {
        const int i = k % cols, j = k / cols, y0 = y_edge(j);
        return (long long)y0 * w + (long long)x_edge(i) * (y_edge(j + 1) - y0);
    }
};

// column of a float coordinate: max{i : X_i <= x} clamped to [0, cols - 1] (x == w is in the last column); NaN: -1
__device__ __forceinline__ int cell_index_f(float v, int n_cells, int len)
{
    if (v != v) return -1;
    if (!(v >= 0.f)) return 0;
    if (v >= (float)len) return n_cells - 1;
    const int p = (int)floorf(v);
    return min((int)(((long long)(p + 1) * n_cells - 1) / len), n_cells - 1);
}

// quota[b][k] = max(0, q - s_k), s_k the points of first[b] points at pts + b * pts_stride (float2) that lie in cell k.
// One block per image, one shared counter per cell.
__global__ void __launch_bounds__(256)
cell_quota_kernel(const float2* __restrict__ pts, long long pts_stride, const int* __restrict__ first, int n_max, CellGrid cg, int q,
                  int* __restrict__ quota)
{
    __shared__ int s_cnt[KLT_MAX_GRID_CELLS];
    const int b = blockIdx.x, G = cg.cols * cg.rows;
    for (int k = threadIdx.x; k < G; k += 256) s_cnt[k] = 0;
    __syncthreads();
    const int n = min(max(first[b], 0), n_max);
    const float2* __restrict__ p = pts + (long long)b * pts_stride;
    for (int t = threadIdx.x; t < n; t += 256) {
        const float2 v = p[t];
        const int i = cell_index_f(v.x, cg.cols, cg.w), j = cell_index_f(v.y, cg.rows, cg.h);
        if (i >= 0 && j >= 0) atomicAdd(&s_cnt[j * cg.cols + i], 1);
    }
    __syncthreads();
    for (int k = threadIdx.x; k < G; k += 256) quota[(long long)b * G + k] = max(0, q - s_cnt[k]);
}

// Per (cell, image) block: the cell's threshold maxVal * qualityLevel (G.7), maxVal the largest eigenvalue over the
// cell's pixels where mask != 0 (0 when there is none, as minMaxLoc); and the cell's candidate count zeroed.
__global__ void __launch_bounds__(256)
cell_threshold_kernel(const float* __restrict__ eig, long long eig_pitch, long long eig_batch_stride, const uint8_t* __restrict__ mask,
                      long long mask_pitch, long long mask_batch_stride, CellGrid cg, double quality, float* __restrict__ thr,
                      unsigned* __restrict__ seg_count)
{
    __shared__ unsigned s_best[8];
    const int k = blockIdx.x, b = blockIdx.y, G = cg.cols * cg.rows;
    const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
    const int i = k % cg.cols, j = k / cg.cols;
    const int x0 = cg.x_edge(i), x1 = cg.x_edge(i + 1), y0 = cg.y_edge(j), y1 = cg.y_edge(j + 1);
    const float* __restrict__ E = eig + (long long)b * eig_batch_stride;
    const uint8_t* __restrict__ M = mask ? mask + (long long)b * mask_batch_stride : nullptr;
    unsigned best = 0;   // 0 = nothing seen
    for (int y = y0 + wrp; y < y1; y += 8)
        for (int x = x0 + lane; x < x1; x += 32)
            if (!M || M[(long long)y * mask_pitch + x]) best = max(best, ordered_from_float(E[(long long)y * eig_pitch + x]));
    best = __reduce_max_sync(kFullMask, best);
    if (lane == 0) s_best[wrp] = best;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w_ = 1; w_ < 8; ++w_) best = max(best, s_best[w_]);
        const float max_val = best ? float_from_ordered(best) : 0.f;
        thr[(long long)b * G + k] = __double2float_rn(__dmul_rn((double)max_val, quality));
        seg_count[(long long)b * G + k] = 0u;
    }
}

// candidates_kernel with the threshold of each pixel's own cell; a candidate is appended to its cell's segment.
__global__ void __launch_bounds__(256)
cell_candidates_kernel(const float* __restrict__ eig, long long eig_pitch, long long eig_batch_stride, const uint8_t* __restrict__ mask,
                       long long mask_pitch, long long mask_batch_stride, CellGrid cg, const float* __restrict__ thr_in,
                       unsigned long long* __restrict__ keys, long long keys_batch_stride, unsigned* __restrict__ seg_count)
{
    const int lane = threadIdx.x, wrp = threadIdx.y;
    const int x = blockIdx.x * 32 + lane;
    const int b = blockIdx.z, G = cg.cols * cg.rows, w = cg.w, h = cg.h;
    const int ci = x < w ? cg.col_of(x) : 0;
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
        const int y = blockIdx.y * 32 + wrp * 4 + kk;
        if (x >= 1 && x < w - 1 && y >= 1 && y < h - 1) {
            const int k = cg.row_of(y) * cg.cols + ci;
            const float thr = thr_in[(long long)b * G + k];
            const float* __restrict__ E = eig + (long long)b * eig_batch_stride + (long long)y * eig_pitch + x;
            float v = E[0];
            v = v > thr ? v : 0.f;
            if (v != 0.f && (!mask || mask[(long long)b * mask_batch_stride + (long long)y * mask_pitch + x])) {
                float m = v;
#pragma unroll
                for (int dy = -1; dy <= 1; ++dy)
#pragma unroll
                    for (int dx = -1; dx <= 1; ++dx) {
                        float u = E[(long long)dy * eig_pitch + dx];
                        u = u > thr ? u : 0.f;
                        m = fmaxf(m, u);
                    }
                if (v == m) {
                    const unsigned slot = atomicAdd(seg_count + (long long)b * G + k, 1u);   // < the cell's area
                    keys[(long long)b * keys_batch_stride + cg.seg_off(k) + slot] =
                        ((unsigned long long)ordered_from_float(v) << 32) | ((unsigned)y << 16) | (unsigned)x;
                }
            }
        }
    }
}

// Descending sort of the segments with at most kCellSortSmem keys, in place, one block per (cell, image): keys are
// distinct, so a key's position is the number of keys above it (counted in shared memory).  cell_radix_sort_kernel
// sorts the larger segments.
constexpr int kCellSortSmem = 4096;
constexpr int kCellRankThreads = 512;

__global__ void __launch_bounds__(kCellRankThreads)
cell_rank_sort_kernel(unsigned long long* __restrict__ keys, long long keys_batch_stride, const unsigned* __restrict__ seg_count,
                      CellGrid cg)
{
    __shared__ unsigned long long s_k[kCellSortSmem];
    const int k = blockIdx.x, b = blockIdx.y, G = cg.cols * cg.rows;
    const int n = (int)seg_count[(long long)b * G + k];
    if (n <= 1 || n > kCellSortSmem) return;
    unsigned long long* __restrict__ list = keys + (long long)b * keys_batch_stride + cg.seg_off(k);
    for (int t = threadIdx.x; t < n; t += kCellRankThreads) s_k[t] = list[t];
    __syncthreads();
    for (int t = threadIdx.x; t < n; t += kCellRankThreads) {
        const unsigned long long v = s_k[t];
        int above = 0;
        for (int u = 0; u < n; ++u) above += s_k[u] > v ? 1 : 0;
        list[above] = v;
    }
}

// radix_sort_keys_kernel for one segment with more than kCellSortSmem keys per (cell, image) block; alt: scratch of the
// keys' layout.  The sorted segment ends in `keys`.
__global__ void __launch_bounds__(kRadixThreads)
cell_radix_sort_kernel(unsigned long long* __restrict__ keys, long long keys_batch_stride, const unsigned* __restrict__ seg_count,
                       unsigned long long* __restrict__ alt, long long alt_batch_stride, CellGrid cg)
{
    __shared__ unsigned s_off[kRadixWarps][256];
    __shared__ unsigned s_wsum[8];
    __shared__ int s_skip;
    const int k = blockIdx.x, b = blockIdx.y, G = cg.cols * cg.rows;
    const int tid = threadIdx.x, lane = tid & 31, wrp = tid >> 5;
    const unsigned n = seg_count[(long long)b * G + k];
    if (n <= (unsigned)kCellSortSmem) return;
    unsigned long long* const home = keys + (long long)b * keys_batch_stride + cg.seg_off(k);
    unsigned long long* src = home;
    unsigned long long* dst = alt + (long long)b * alt_batch_stride + cg.seg_off(k);
    const unsigned chunk = (n + kRadixWarps - 1) / kRadixWarps;
    const unsigned lo = min(n, chunk * wrp), hi = min(n, lo + chunk);
    for (int shift = 0; shift < 64; shift += 8) {
        for (int i = tid; i < kRadixWarps * 256; i += kRadixThreads) (&s_off[0][0])[i] = 0u;
        if (tid == 0) s_skip = 0;
        __syncthreads();
        for (unsigned i = lo + lane; i < hi; i += 32) atomicAdd(&s_off[wrp][255u - (unsigned)((src[i] >> shift) & 0xffu)], 1u);
        __syncthreads();
        unsigned tot = 0, incl = 0;
        if (tid < 256) {
#pragma unroll 8
            for (int w = 0; w < kRadixWarps; ++w) tot += s_off[w][tid];
            if (tot == n) s_skip = 1;
            incl = tot;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned t = __shfl_up_sync(kFullMask, incl, o);
                if (lane >= o) incl += t;
            }
            if (lane == 31) s_wsum[wrp] = incl;
        }
        __syncthreads();
        const bool skip = s_skip;
        if (!skip && tid < 256) {
            unsigned run = incl - tot;
            for (int w = 0; w < wrp; ++w) run += s_wsum[w];
#pragma unroll 8
            for (int w = 0; w < kRadixWarps; ++w) {
                const unsigned c = s_off[w][tid];
                s_off[w][tid] = run;
                run += c;
            }
        }
        __syncthreads();
        for (unsigned i0 = lo; !skip && i0 < hi; i0 += 32) {
            const unsigned i = i0 + lane;
            const bool valid = i < hi;
            const unsigned long long key = valid ? src[i] : 0ull;
            const unsigned d = valid ? 255u - (unsigned)((key >> shift) & 0xffu) : 256u + lane;
            const unsigned peers = __match_any_sync(kFullMask, d);
            if (valid) dst[s_off[wrp][d] + __popc(peers & ((1u << lane) - 1u))] = key;
            __syncwarp();
            if (valid && lane == __ffs(peers) - 1) s_off[wrp][d] += __popc(peers);
            __syncwarp();
        }
        __syncthreads();
        if (!skip) { unsigned long long* t = src; src = dst; dst = t; }
    }
    if (src != home)
        for (unsigned i = tid; i < n; i += kRadixThreads) dst[i] = src[i];
}

// select_corners_kernel for one (cell, image) block: the cell's sorted segment, a bitmap of the cell only (positions
// relative to its corner), at most k_max = min(max_corners, cap - first[b], quota[b][k]) corners (first / quota may be
// null: no such bound).  The accepted corners overwrite the front of the segment as (y << 16) | x; n_sel[b][k] counts
// them.  gbitmap: the cell's bitmap at its segment offset (in words) of image b's region, zeroed by the launcher.
template <bool kGlobalBitmap, bool kAnyRadius>
__global__ void __launch_bounds__(kSelThreads)
cell_select_kernel(unsigned long long* __restrict__ keys, long long keys_batch_stride, const unsigned* __restrict__ seg_count,
                   CellGrid cg, long long md2, int radius, int max_corners, long long cap, const int* __restrict__ first,
                   const int* __restrict__ quota, int* __restrict__ n_sel, unsigned* __restrict__ gbitmap, long long gbitmap_stride)
{
    extern __shared__ __align__(16) unsigned sel_smem[];
    __shared__ unsigned short sx[kSelThreads], sy[kSelThreads];
    __shared__ unsigned s_alive[4], s_acc[4], s_rej[4];
    __shared__ short s_halfw[kSelMaxRadius + 1];
    __shared__ unsigned short s_ax[kSelThreads], s_ay[kSelThreads];
    const int tid = threadIdx.x, lane = tid & 31, wrp = tid >> 5;
    const int kc = blockIdx.x, b = blockIdx.y, G = cg.cols * cg.rows;
    const long long bk = (long long)b * G + kc;
    const int n = (int)seg_count[bk];
    long long lim = first ? min((long long)max_corners, cap - first[b]) : (long long)max_corners;
    if (quota) lim = min(lim, (long long)quota[bk]);
    const int k_max = (int)max(lim, 0LL);
    if (k_max <= 0 || n == 0) {
        if (tid == 0) n_sel[bk] = 0;
        return;
    }
    const int ci = kc % cg.cols, cj = kc / cg.cols;
    const int x0 = cg.x_edge(ci), y0 = cg.y_edge(cj);
    const int w = cg.x_edge(ci + 1) - x0, h = cg.y_edge(cj + 1) - y0;
    const long long off = cg.seg_off(kc);
    unsigned long long* list = keys + (long long)b * keys_batch_stride + off;
    const int wpr = (w + 31) >> 5;
    const int nwords = wpr * h;
    unsigned* bitmap = kGlobalBitmap ? gbitmap + (long long)b * gbitmap_stride + off : sel_smem;
    if (!kGlobalBitmap)
        for (int i = tid; i < nwords; i += kSelThreads) bitmap[i] = 0u;
    if (!kAnyRadius && tid <= radius) s_halfw[tid] = (short)sel_halfwidth(md2, tid);
    __syncthreads();
    int accepted_total = 0;
    for (int base = 0; base < n && accepted_total < k_max; base += kSelThreads) {
        const int t = base + tid;
        int x = 0, y = 0;
        bool alive = false;
        if (t < n) {
            const unsigned long long key = list[t];
            x = (int)(key & 0xffffu) - x0; y = (int)((key >> 16) & 0xffffu) - y0;
            alive = !((bitmap[y * wpr + (x >> 5)] >> (x & 31)) & 1u);
        }
        sx[tid] = (unsigned short)x; sy[tid] = (unsigned short)y;
        const unsigned am = __ballot_sync(kFullMask, alive);
        if (lane == 0) { s_alive[wrp] = am; s_acc[wrp] = 0u; s_rej[wrp] = ~am; }
        __syncthreads();
        // stronger alive window members within minDistance: the coordinates of one predecessor warp at a time in
        // registers, broadcast by shuffle (a data-dependent loop over shared memory paid one load latency per test)
        unsigned conf[4] = {0u, 0u, 0u, 0u};
#pragma unroll
        for (int wi = 0; wi < 4; ++wi) {
            if (wi > wrp) break;                      // uniform per warp
            unsigned bits = s_alive[wi];
            if (wi == wrp) bits &= (1u << lane) - 1u;
            if (__ballot_sync(kFullMask, alive && bits != 0u) == 0u) continue;   // nothing to test for this warp
            const int px = sx[wi * 32 + lane], py = sy[wi * 32 + lane];
            unsigned c = 0u;
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                const int dx = x - __shfl_sync(kFullMask, px, j), dy = y - __shfl_sync(kFullMask, py, j);
                const bool close = kAnyRadius ? ((long long)dx * dx + (long long)dy * dy < md2)
                                              : ((unsigned)dx * (unsigned)dx + (unsigned)dy * (unsigned)dy < (unsigned)md2);
                const bool near = (abs(dx) <= radius) && (abs(dy) <= radius) && close;
                c |= near ? (1u << j) : 0u;
            }
            conf[wi] = alive ? (c & bits) : 0u;
        }
        // fixpoint of "accepted iff no accepted conflicting predecessor"
        bool decided = !alive, acc = false;
        while (true) {
            bool now_acc = false, now_rej = false;
            if (!decided) {
                const unsigned a0 = s_acc[0], a1 = s_acc[1], a2 = s_acc[2], a3 = s_acc[3];
                const unsigned r0 = s_rej[0], r1 = s_rej[1], r2 = s_rej[2], r3 = s_rej[3];
                if ((conf[0] & a0) | (conf[1] & a1) | (conf[2] & a2) | (conf[3] & a3)) now_rej = true;
                else if (!((conf[0] & ~r0) | (conf[1] & ~r1) | (conf[2] & ~r2) | (conf[3] & ~r3))) now_acc = true;
            }
            __syncthreads();   // everyone has read the previous state
            const unsigned ba = __ballot_sync(kFullMask, now_acc), br = __ballot_sync(kFullMask, now_rej);
            if (lane == 0) { s_acc[wrp] |= ba; s_rej[wrp] |= br; }
            if (now_acc) { acc = true; decided = true; }
            if (now_rej) decided = true;
            if (!__syncthreads_or(!decided)) break;
        }
        // positions in the output: accepted members in window order
        const unsigned a0 = s_acc[0], a1 = s_acc[1], a2 = s_acc[2], a3 = s_acc[3];
        int before = __popc(s_acc[wrp] & ((1u << lane) - 1u));
        if (wrp > 0) before += __popc(a0);
        if (wrp > 1) before += __popc(a1);
        if (wrp > 2) before += __popc(a2);
        const int nacc_win = __popc(a0) + __popc(a1) + __popc(a2) + __popc(a3);
        int nkeep = nacc_win;
        nkeep = min(nkeep, k_max - accepted_total);
        if (acc && before < nkeep) {
            s_ax[before] = (unsigned short)x; s_ay[before] = (unsigned short)y;
            list[accepted_total + before] = ((unsigned long long)(y + y0) << 16) | (unsigned)(x + x0);   // read in an earlier window
        }
        __syncthreads();
        // paint the discs of the corners just accepted (rows outside the image are skipped)
        const int rows_per = 2 * radius + 1;
        for (int sidx = tid; sidx < nkeep * rows_per; sidx += kSelThreads) {
            const int a = sidx / rows_per, dy = sidx - a * rows_per - radius;
            const int yy = (int)s_ay[a] + dy;
            if (yy < 0 || yy >= h) continue;
            const int ady = dy < 0 ? -dy : dy;
            const int hx = kAnyRadius ? sel_halfwidth(md2, ady) : s_halfw[ady];
            if (hx < 0) continue;
            const int xa = max((int)s_ax[a] - hx, 0), xb = min((int)s_ax[a] + hx, w - 1);
            for (int wd_ = xa >> 5; wd_ <= (xb >> 5); ++wd_) {
                const int lo = max(xa - (wd_ << 5), 0), hi = min(xb - (wd_ << 5), 31);
                const unsigned m = (hi == 31 ? 0xffffffffu : ((1u << (hi + 1)) - 1u)) & ~((1u << lo) - 1u);
                atomicOr(&bitmap[yy * wpr + wd_], m);
            }
        }
        accepted_total += nkeep;
        __syncthreads();
    }
    if (tid == 0) n_sel[bk] = accepted_total;
}

// Behind the first[b] points of row b: the cells' corners interleaved by rank (L_0[0], L_1[0], ..., L_0[1], ...,
// exhausted cells skipped), cut to min(max_corners, cap - first[b]); ids as select_corners_kernel.  One warp per image:
// lane c holds the largest count of cells 32c .. 32c + 31 (G <= 32 * 32), so a rank visits only the chunks that still
// have corners, and each visit writes at least one.
__global__ void __launch_bounds__(32)
cell_interleave_kernel(const unsigned long long* __restrict__ keys, long long keys_batch_stride, const int* __restrict__ n_sel,
                       CellGrid cg, int max_corners, long long cap, const int* __restrict__ first, float2* __restrict__ out,
                       long long out_stride, int* __restrict__ next_counts, int* __restrict__ n_new, int* __restrict__ ids_out,
                       int* __restrict__ next_id)
{
    const int b = blockIdx.x, lane = threadIdx.x, G = cg.cols * cg.rows;
    const int fb = first[b];
    const int cut = (int)max(min((long long)max_corners, cap - fb), 0LL);
    const int id0 = ids_out ? next_id[b] : 0;
    const int* __restrict__ ns = n_sel + (long long)b * G;
    int cmax = 0;
    if (lane * 32 < G)
        for (int t = 0; t < 32 && lane * 32 + t < G; ++t) cmax = max(cmax, ns[lane * 32 + t]);
    const unsigned long long* __restrict__ K = keys + (long long)b * keys_batch_stride;
    int pos = 0;
    for (int r = 0; pos < cut; ++r) {
        unsigned act = __ballot_sync(kFullMask, cmax > r);
        if (!act) break;
        while (act && pos < cut) {
            const int c = __ffs(act) - 1;
            act &= act - 1;
            const int k = c * 32 + lane;
            const bool has = k < G && ns[k] > r;
            const unsigned bal = __ballot_sync(kFullMask, has);
            const int p = pos + __popc(bal & ((1u << lane) - 1u));
            if (has && p < cut) {
                const unsigned long long v = K[cg.seg_off(k) + r];
                out[(long long)b * out_stride + fb + p] = make_float2((float)(v & 0xffffu), (float)((v >> 16) & 0xffffu));
                if (ids_out) ids_out[(long long)b * out_stride + fb + p] = id0 + p;
            }
            pos += __popc(bal);
        }
    }
    const int nn = min(pos, cut);
    __syncwarp();
    if (lane == 0) {
        n_new[b] = nn;
        next_counts[b] = fb + nn;
        if (ids_out) next_id[b] = id0 + nn;
    }
}

// The cells' corners as float (x, y) pairs: out[b][k][0 .. n_sel[b][k]) (q per cell), counts[b][k] = n_sel[b][k].
__global__ void __launch_bounds__(128)
cell_corners_out_kernel(const unsigned long long* __restrict__ keys, long long keys_batch_stride, const int* __restrict__ n_sel,
                        CellGrid cg, int q, float2* __restrict__ out, int* __restrict__ counts)
{
    const int k = blockIdx.x, b = blockIdx.y, G = cg.cols * cg.rows;
    const long long bk = (long long)b * G + k;
    const int n = n_sel[bk];
    const unsigned long long* __restrict__ K = keys + (long long)b * keys_batch_stride + cg.seg_off(k);
    for (int t = threadIdx.x; t < n; t += 128)
        out[bk * q + t] = make_float2((float)(K[t] & 0xffffu), (float)((K[t] >> 16) & 0xffffu));
    if (threadIdx.x == 0) counts[bk] = n;
}

bool grid_ok(int w, int h, int batch, int cols, int rows)
{
    return w >= 1 && h >= 1 && w <= 65535 && h <= 65535 && batch >= 1 && batch <= 65535 && cols >= 1 && rows >= 1 && cols <= w &&
           rows <= h && (long long)cols * rows <= KLT_MAX_GRID_CELLS;
}

// selection radius as corner_select_launch: squared distances are integers, d2 < md2 <=> d2 < ceil(md2); -1: no conflicts
void sel_radius(double min_distance, int w, int h, long long* md2, int* radius)
{
    *md2 = 0;
    *radius = -1;
    if (min_distance >= 1) {
        const double md2d = ceil(min_distance * min_distance);
        *md2 = md2d < 4.0e18 ? (long long)md2d : (long long)4.0e18;
        const int rmax = w > h ? w : h;
        int r = 0;
        while (r < rmax && (long long)(r + 1) * (r + 1) < *md2) ++r;
        *radius = r;
    }
}

}  // namespace

klt_status corner_grid_quota_launch(const float* pts, long long pts_stride, const int* first, int n_max, int batch, int w, int h, int cols,
                                    int rows, int q, int* quota, cudaStream_t stream)
{
    if (!grid_ok(w, h, batch, cols, rows) || n_max < 0 || q < 0 || !first || !quota || (n_max > 0 && !pts)) return KLT_ERR_INVALID_ARG;
    cell_quota_kernel<<<batch, 256, 0, stream>>>(reinterpret_cast<const float2*>(pts), pts_stride, first, n_max, CellGrid{cols, rows, w, h}, q,
                                                 quota);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KLT_OK : (klt_status)e;
}

klt_status corner_grid_detect_launch(const float* eig, long long eig_pitch, long long eig_batch_stride, int w, int h, int batch,
                                     const uint8_t* mask, long long mask_pitch, long long mask_batch_stride, int cols, int rows,
                                     double quality, double min_distance, int max_corners, long long cap, const int* first,
                                     const int* quota, float* thr, unsigned* seg_count, int* n_sel, unsigned long long* keys,
                                     long long keys_batch_stride, unsigned long long* alt, long long alt_batch_stride, unsigned* gbitmap,
                                     long long gbitmap_stride, cudaStream_t stream)
{
    const long long px = (long long)w * h;
    if (!grid_ok(w, h, batch, cols, rows) || !eig || !thr || !seg_count || !n_sel || !keys || !alt || !gbitmap || !(quality > 0) ||
        !(min_distance >= 0) || max_corners < 1 || keys_batch_stride < px || alt_batch_stride < px || gbitmap_stride < px)
        return KLT_ERR_INVALID_ARG;
    const CellGrid cg{cols, rows, w, h};
    const int G = cols * rows;
    long long md2;
    int radius;
    sel_radius(min_distance, w, h, &md2, &radius);
    int cw = 0, ch = 0;   // the largest cell
    for (int i = 0; i < cols; ++i) cw = max(cw, cg.x_edge(i + 1) - cg.x_edge(i));
    for (int j = 0; j < rows; ++j) ch = max(ch, cg.y_edge(j + 1) - cg.y_edge(j));
    const long long nwords = (long long)((cw + 31) / 32) * ch;
    const bool in_smem = nwords <= kSelMaxBitmapWords, any_radius = radius > kSelMaxRadius;
    auto sel = in_smem ? (any_radius ? cell_select_kernel<false, true> : cell_select_kernel<false, false>)
                       : (any_radius ? cell_select_kernel<true, true> : cell_select_kernel<true, false>);
    cudaError_t e = cudaSuccess;
    if (in_smem) {
        static PerDeviceOnce configured;
        if (configured.needed()) {
            e = cudaFuncSetAttribute(cell_select_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSelMaxBitmapWords * 4);
            if (e == cudaSuccess)
                e = cudaFuncSetAttribute(cell_select_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSelMaxBitmapWords * 4);
            if (e != cudaSuccess) return (klt_status)e;
        }
    }
    const dim3 cells(G, batch);
    cell_threshold_kernel<<<cells, 256, 0, stream>>>(eig, eig_pitch, eig_batch_stride, mask, mask_pitch, mask_batch_stride, cg, quality, thr,
                                                     seg_count);
    cell_candidates_kernel<<<dim3((w + 31) / 32, (h + 31) / 32, batch), dim3(32, 8), 0, stream>>>(
        eig, eig_pitch, eig_batch_stride, mask, mask_pitch, mask_batch_stride, cg, thr, keys, keys_batch_stride, seg_count);
    cell_rank_sort_kernel<<<cells, kCellRankThreads, 0, stream>>>(keys, keys_batch_stride, seg_count, cg);
    cell_radix_sort_kernel<<<cells, kRadixThreads, 0, stream>>>(keys, keys_batch_stride, seg_count, alt, alt_batch_stride, cg);
    if (!in_smem) {
        e = cudaMemset2DAsync(gbitmap, (size_t)gbitmap_stride * 4, 0, (size_t)px * 4, (size_t)batch, stream);
        if (e != cudaSuccess) return (klt_status)e;
    }
    sel<<<cells, kSelThreads, in_smem ? (size_t)nwords * 4 : 0, stream>>>(keys, keys_batch_stride, seg_count, cg, md2, radius, max_corners,
                                                                         cap, first, quota, n_sel, gbitmap, gbitmap_stride);
    e = cudaGetLastError();
    return e == cudaSuccess ? KLT_OK : (klt_status)e;
}

klt_status corner_grid_interleave_launch(const unsigned long long* keys, long long keys_batch_stride, const int* n_sel, int w, int h, int batch,
                                         int cols, int rows, int max_corners, long long cap, const int* first, float* out,
                                         long long out_stride, int* next_counts, int* n_new, int* ids_out, int* next_id,
                                         cudaStream_t stream)
{
    if (!grid_ok(w, h, batch, cols, rows) || !keys || !n_sel || !first || !out || !next_counts || !n_new || (!ids_out != !next_id) ||
        max_corners < 1)
        return KLT_ERR_INVALID_ARG;
    cell_interleave_kernel<<<batch, 32, 0, stream>>>(keys, keys_batch_stride, n_sel, CellGrid{cols, rows, w, h}, max_corners, cap, first,
                                                     reinterpret_cast<float2*>(out), out_stride, next_counts, n_new, ids_out, next_id);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KLT_OK : (klt_status)e;
}

klt_status corner_grid_out_launch(const unsigned long long* keys, long long keys_batch_stride, const int* n_sel, int w, int h, int batch,
                                  int cols, int rows, int q, float* out, int* counts, cudaStream_t stream)
{
    if (!grid_ok(w, h, batch, cols, rows) || !keys || !n_sel || q < 1 || !out || !counts) return KLT_ERR_INVALID_ARG;
    cell_corners_out_kernel<<<dim3(cols * rows, batch), 128, 0, stream>>>(keys, keys_batch_stride, n_sel, CellGrid{cols, rows, w, h}, q,
                                                                         reinterpret_cast<float2*>(out), counts);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KLT_OK : (klt_status)e;
}

}  // namespace klt
