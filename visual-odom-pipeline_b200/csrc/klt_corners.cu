// K5: Shi-Tomasi corner detection (SURVEY.md s8f rank 2) -- what the reference delegates to
// cv2.goodFeaturesToTrack(img, mask=mask, maxCorners=1000, qualityLevel=0.03, minDistance, blockSize=31) at
// reference src/extractor/extractor.py:21-24,110-111 (called once per frame from src/pipeline/pipeline.py:159-163).
//
// Arithmetic: oracle/gftt_oracle.c G.1-G.7 (float32 Sobel with OpenCV's AVX2 fused-multiply-add pattern, float32
// products, DOUBLE running box sums in OpenCV's order, non-fused eigenvalue formula) -- bit-exact with the cv2 wheel.
// Kernels per image batch:
//   cov_kernel        32x32 pixel tiles: u8 tile + halo in shared memory -> Dx, Dy -> (Dx^2, DxDy, Dy^2), written
//                     TRANSPOSED ([channel][x][y]) so that the row scan reads it coalesced;
//   row_scan_kernel   one lane per image row (a block = 32 rows of one channel): the serial double-precision running
//                     sum along x (the order is part of the result: the sums are not exact) on a "chain" warp that has
//                     a warp scheduler to itself; helper warps fetch the operands two chunks ahead, form the per-step
//                     differences and write the sums out; named-barrier signals over rings of chunks;
//   col_scan_kernel   one lane per image column, three chain warps (one per channel) on one scheduler: running sum along
//                     y (operand rows staged by helper warps with cp.async), float32 conversion, eigenvalue, masked
//                     maximum (REDUX + one atomicMax per warp);
//   candidates_kernel threshold (maxVal * qualityLevel), 3x3 dilation and local-maximum test fused; survivors are
//                     appended as 64-bit keys (ordered float << 32 | y << 16 | x) with one atomicAdd per 32x32 tile;
//   rank_keys_kernel, scatter_keys_kernel   chip-wide rank sort of the (<= 8192) keys, written with their count into
//                     page-locked host memory mapped into the device address space.
//   radix_sort_keys_kernel   descending radix sort of the frames with more than 8192 keys, one block per frame: only
//                     for the batched frame step, so that the selection below takes every frame.
//   select_corners_kernel   greedy minimum-distance selection (G.8), one block per image: only for batches of frames
//                     (klt_frame_step_batch[_async]), where B blocks run side by side.  On one frame it takes about 165 us
//                     per KITTI frame against about 75 us for the host loop, so single-frame detection selects on the host
//                     (klt_capi.cu), like the tail of cv::cuda::GoodFeaturesToTrackDetector.
// DESIGN.md s4 K5 has the measurements behind each of these choices.
#include "klt_common.cuh"

namespace klt {

namespace {

constexpr unsigned kFullMask = 0xffffffffu;

__device__ __forceinline__ unsigned ordered_from_float(float f)
{
    const unsigned b = __float_as_uint(f);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float float_from_ordered(unsigned u)
{
    return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

// ---- cov_kernel -----------------------------------------------------------------------------------------------
constexpr int kTile = 32;

__global__ void __launch_bounds__(256)
cov_kernel(const uint8_t* __restrict__ img, long long pitch, long long batch_stride, int w, int h,
           float* __restrict__ covT, int hp, float k1, float k0)
{
    __shared__ uint8_t sI[kTile + 2][kTile + 4];
    __shared__ float sT[kTile + 2][kTile + 1];   // smoothed rows (for Dy)
    __shared__ int sR[kTile + 2][kTile + 1];     // horizontal differences (for Dx)
    __shared__ float sC[3][kTile][kTile + 1];    // [channel][x][y]
    const int tx = threadIdx.x, ty = threadIdx.y;
    const int x0 = blockIdx.x * kTile, y0 = blockIdx.y * kTile;
    const uint8_t* __restrict__ src = img + (long long)blockIdx.z * batch_stride;
    for (int i = ty * 32 + tx; i < (kTile + 2) * (kTile + 2); i += 256) {
        const int r = i / (kTile + 2), c = i - r * (kTile + 2);
        const int yy = reflect101(min(y0 + r - 1, h), h), xx = reflect101(min(x0 + c - 1, w), w);
        sI[r][c] = __ldg(src + (long long)yy * pitch + xx);
    }
    __syncthreads();
    const int nv = 32 * (w / 32);
    for (int r = ty; r < kTile + 2; r += 8) {
        const float L = (float)sI[r][tx], C = (float)sI[r][tx + 1], R = (float)sI[r][tx + 2];
        sR[r][tx] = (int)sI[r][tx + 2] - (int)sI[r][tx];
        float t;
        if (x0 + tx < nv) t = __fmaf_rn(k1, R, __fmaf_rn(k0, C, __fmul_rn(k1, L)));                       // G.3, SIMD part
        else t = __fadd_rn(__fadd_rn(__fmul_rn(k1, L), __fmul_rn(k0, C)), __fmul_rn(k1, R));             // scalar tail
        sT[r][tx] = t;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int y = ty + 8 * k;
        const float dx = __fmaf_rn(k1, (float)(sR[y][tx] + sR[y + 2][tx]), __fmul_rn(k0, (float)sR[y + 1][tx]));   // G.2
        const float dy = __fsub_rn(sT[y + 2][tx], sT[y][tx]);
        sC[0][tx][y] = __fmul_rn(dx, dx);
        sC[1][tx][y] = __fmul_rn(dx, dy);
        sC[2][tx][y] = __fmul_rn(dy, dy);
    }
    __syncthreads();
    float* __restrict__ dst = covT + (long long)blockIdx.z * 3 * w * hp;
    if (y0 + tx < h) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int x = ty + 8 * k;
            if (x0 + x < w) {
#pragma unroll
                for (int c = 0; c < 3; ++c) dst[((long long)c * w + (x0 + x)) * hp + (y0 + tx)] = sC[c][x][tx];
            }
        }
    }
}

// ---- cp.async helpers (LDGSTS: global -> shared without registers in flight) ------------------------------------
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc)
{
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
// named barriers as producer / consumer signals (PTX bar.arrive / bar.sync pairs): the producer warps arrive after
// their shared-memory writes, the consumer warps sync before reading; `n` counts the threads of both sides
__device__ __forceinline__ void bar_sync(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ void bar_arrive(int id, int n) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(n) : "memory"); }

// profiling aid (KLT_CORNER_TIMELINE=1, scripts/corner_timeline.py): clock64 stamps of the chain warp of block (0,0,0)
__device__ long long g_timeline[4 * 256 + 6 * 256];   // chain warp: 4 stamps per chunk; helper warp 0: 6 per chunk from word 1024
__device__ int g_timeline_on;

// ---- row_scan_kernel ------------------------------------------------------------------------------------------
// Serves block sizes >= 6, the ones OpenCV sums with a running sum (smaller ones: row_sum_small_kernel).
// The running sum along x is a serial chain of one DADD per pixel and row, and with so little parallelism (H rows x 3
// channels) the launch time IS the time of one chain.  So the block is specialised: warp 0 ("chain", lane = row) does
// nothing but  d = smem, s += d, smem = s;  the helper warps keep everything else off that warp: lane = row for them as
// well, so a column of the transposed product image is one coalesced 128-byte load; they fetch the entering and the
// leaving column of each step a chunk ahead (registers), form d = (double)new - (double)old exactly as OpenCV does, and
// write the finished sums row-major in 256-byte runs.  The two sides are coupled only by named-barrier signals over
// rings of kRowRing chunks (d full / s full / s empty), and the chain warp has a warp scheduler to itself (warps are
// dealt to the four schedulers round-robin; the other warps whose index is a multiple of 4 idle).
// Shared-memory traffic is the budget that matters (chain-warp timeline, scripts/corner_timeline.py): per 64-step chunk
// the d and s rings cost 4 x 128 wavefronts, the same order as the 512 cycles of the DADD chain; an earlier version
// that also staged the operands through shared memory (cp.async) and wrote d with a 4-way bank conflict needed ~1150
// wavefronts and ran at 22 cycles per step.  Rings are lane-major with a row stride of 65 doubles: conflict-free for
// "32 rows, one column" and for "one row, 32 columns".
constexpr int kRowChunk = 64;     // x steps per chunk
constexpr int kRowRing = 4;       // chunks of d / s between the chain warp and the helpers
constexpr int kRowLag = 2;        // helpers write out chunk c - kRowLag while the chain works on chunk c (< kRowRing)
constexpr int kRowHelperWarps = 23;
constexpr int kRowHelpers = 32 * kRowHelperWarps;
constexpr int kRowThreads = 32 + kRowHelpers;            // threads that take part in the named barriers
constexpr int kRowBlock = 32 * (1 + kRowHelperWarps + (kRowHelperWarps + 2) / 3);   // + idle warps
constexpr int kRowCPW = (kRowChunk + kRowHelperWarps - 1) / kRowHelperWarps;        // columns per helper warp and chunk
struct RowSmem {
    double d[kRowRing][32][kRowChunk + 1];
    double s[kRowRing][32][kRowChunk + 1];
};
enum { kBarRowDFull = 1, kBarRowSFull = 1 + kRowRing, kBarRowSEmpty = 1 + 2 * kRowRing };

// padded column i (0 <= i < w + block - 1) -> source column (reflect-101 of i - anchor)
__device__ __forceinline__ int src_col(int i, int an, int w) { return reflect101(i - an, w); }

__global__ void __launch_bounds__(kRowBlock)
row_scan_kernel(const float* __restrict__ covT, int w, int h, int hp, int block, double* __restrict__ rows, int wd)
{
    extern __shared__ __align__(16) uint8_t smem_raw[];
    RowSmem& sm = *reinterpret_cast<RowSmem*>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, wrp = tid >> 5;
    const int y0 = blockIdx.x * 32, c = blockIdx.y;
    const int an = block / 2;
    const float* __restrict__ S = covT + ((long long)blockIdx.z * 3 + c) * w * hp + y0 + lane;   // column x, this lane's row: S[x * hp]
    double* __restrict__ D = rows + (((long long)blockIdx.z * 3 + c) * h + y0) * wd;              // row r at D + r * wd
    const int nrows = min(32, h - y0);
    const int nck = (w + kRowChunk - 1) / kRowChunk;
    // output o = 0 is the sum of the first `block` padded columns; output o >= 1 adds column o-1+block and drops o-1

    if (wrp == 0) {
        // ---- chain warp ----
        double s = 0.0;
        for (int i0 = 0; i0 < block; i0 += 16) {
            float v[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = S[(long long)src_col(min(i0 + i, block - 1), an, w) * hp];
#pragma unroll
            for (int i = 0; i < 16; ++i)
                if (i0 + i < block) s = __dadd_rn(s, (double)v[i]);
        }
        const bool tl_on = g_timeline_on == 1 && lane == 0 && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0;
        for (int k = 0; k < nck; ++k) {
            const int slot = k % kRowRing;
            const bool tl = tl_on && k < 256;
            if (tl) g_timeline[4 * k] = clock64();
            bar_sync(kBarRowDFull + slot, kRowThreads);                       // d[slot] holds chunk k
            if (tl) g_timeline[4 * k + 1] = clock64();
            if (k >= kRowRing) bar_sync(kBarRowSEmpty + slot, kRowThreads);   // chunk k - kRowRing has been written out
            if (tl) g_timeline[4 * k + 2] = clock64();
            const double* __restrict__ pd = &sm.d[slot][lane][0];
            double* __restrict__ ps = &sm.s[slot][lane][0];
#pragma unroll
            for (int q = 0; q < kRowChunk / 16; ++q) {
                double v[16];
#pragma unroll
                for (int j = 0; j < 16; ++j) v[j] = pd[16 * q + j];
                if (k == 0 && q == 0) v[0] = 0.0;   // output 0 is the initial sum itself (s + 0.0 == s: s is never -0)
#pragma unroll
                for (int j = 0; j < 16; ++j) { s = __dadd_rn(s, v[j]); v[j] = s; }
#pragma unroll
                for (int j = 0; j < 16; ++j) ps[16 * q + j] = v[j];
            }
            bar_arrive(kBarRowSFull + slot, kRowThreads);
            if (tl) g_timeline[4 * k + 3] = clock64();
        }
        return;
    }
    if ((wrp & 3) == 0) return;                       // leave the chain's scheduler alone
    const int hw = wrp - 1 - (wrp >> 2);              // helper warp index
    if (hw >= kRowHelperWarps) return;
    // ---- helper warps: lane = row; helper warp hw owns columns hw, hw + kRowHelperWarps, ... of every chunk ----
    float leadA[kRowCPW], trailA[kRowCPW], leadB[kRowCPW], trailB[kRowCPW];   // two chunks of operands in flight
    auto fetch = [&](int k, float (&lead)[kRowCPW], float (&trail)[kRowCPW]) {   // operands of outputs k * kRowChunk + j
        const int t0 = k * kRowChunk + hw - 1 - an;            // leaving column of this warp's first step (unreflected)
        if (t0 >= 0 && k * kRowChunk + hw >= 1 && t0 + block + kRowHelperWarps * (kRowCPW - 1) < w) {
            // interior chunk (all but the first and the last one or two): plain strides, no reflection
            const float* __restrict__ p = S + (long long)t0 * hp;
            const long long lead_off = (long long)block * hp, step = (long long)kRowHelperWarps * hp;
#pragma unroll
            for (int i = 0; i < kRowCPW; ++i) {
                trail[i] = p[i * step];
                lead[i] = p[i * step + lead_off];
            }
            return;
        }
#pragma unroll
        for (int i = 0; i < kRowCPW; ++i) {
            const int j = hw + kRowHelperWarps * i;
            const int o = min(max(k * kRowChunk + j, 1), w - 1 > 1 ? w - 1 : 1);
            lead[i] = S[(long long)src_col(o - 1 + block, an, w) * hp];
            trail[i] = S[(long long)src_col(o - 1, an, w) * hp];
        }
    };
    auto convert = [&](int k, const float (&lead)[kRowCPW], const float (&trail)[kRowCPW]) {
        double* __restrict__ dst = &sm.d[k % kRowRing][lane][0];
#pragma unroll
        for (int i = 0; i < kRowCPW; ++i) {
            const int j = hw + kRowHelperWarps * i;
            if (j < kRowChunk) dst[j] = __dsub_rn((double)lead[i], (double)trail[i]);
        }
    };
    // the (row, 32-column half) pairs this warp writes out are the same for every chunk: offsets computed once
    constexpr int NT = 32 * (kRowChunk / 32), NR = (NT + kRowHelperWarps - 1) / kRowHelperWarps;
    int f_soff[NR], f_c0[NR];
    long long f_goff[NR];
#pragma unroll
    for (int i = 0; i < NR; ++i) {
        const int t = hw + kRowHelperWarps * i;
        const int r = min(t, NT - 1) / (kRowChunk / 32), c0 = 32 * (min(t, NT - 1) % (kRowChunk / 32)) + lane;
        f_soff[i] = r * (kRowChunk + 1) + c0;
        f_c0[i] = (t < NT && r < nrows) ? c0 : kRowChunk;      // kRowChunk = never below n: nothing to write
        f_goff[i] = (long long)r * wd + c0;
    }
    auto flush = [&](int k, long long* tl) {     // outputs of chunk k, lane = column: 256-byte runs
        const int xbase = k * kRowChunk, n = min(kRowChunk, w - xbase);
        bar_sync(kBarRowSFull + k % kRowRing, kRowThreads);
        if (tl) tl[3] = clock64();
        // all loads first, then all stores: a load into the register a store has just read waits for that store
        const double* __restrict__ sp = &sm.s[k % kRowRing][0][0];
        double* __restrict__ gp = D + xbase;
        double v[NR];
#pragma unroll
        for (int i = 0; i < NR; ++i) v[i] = sp[f_soff[i]];
#pragma unroll
        for (int i = 0; i < NR; ++i)
            if (f_c0[i] < n) gp[f_goff[i]] = v[i];
        if (tl) tl[4] = clock64();
        if (k + kRowRing < nck) bar_arrive(kBarRowSEmpty + k % kRowRing, kRowThreads);   // the slot may be rewritten
    };
    static_assert(kRowLag + 1 <= kRowRing, "d[slot] is rewritten only after the chain finished the chunk that was in it");
    fetch(0, leadA, trailA);
    fetch(1, leadB, trailB);
    const bool htl = g_timeline_on == 1 && hw == 0 && lane == 0 && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0;
    auto step = [&](int k, float (&lead)[kRowCPW], float (&trail)[kRowCPW]) {
        // feed the chain first: d[k % ring] is free because this warp has already seen "s full" of chunk k - 1 - lag
        long long* tl = (htl && k < 256) ? g_timeline + 1024 + 6 * k : nullptr;
        if (tl) tl[0] = clock64();
        convert(k, lead, trail);
        if (tl) tl[1] = clock64();
        bar_arrive(kBarRowDFull + k % kRowRing, kRowThreads);
        if (k + 2 < nck) fetch(k + 2, lead, trail);   // two chunks ahead: the load latency hides behind a whole iteration
        if (tl) tl[2] = clock64();
        if (k >= kRowLag) flush(k - kRowLag, tl);
        if (tl) tl[5] = clock64();
    };
    for (int k = 0; k < nck; k += 2) {
        step(k, leadA, trailA);
        if (k + 1 < nck) step(k + 1, leadB, trailB);
    }
    for (int k = max(nck - kRowLag, 0); k < nck; ++k) flush(k, nullptr);
}

// OpenCV's box filter forms fresh left-to-right row sums for kernel sizes up to 5 (G.5): no chain, one thread per output.
__global__ void __launch_bounds__(256)
row_sum_small_kernel(const float* __restrict__ covT, int w, int h, int hp, int block, double* __restrict__ rows, int wd)
{
    const int y = blockIdx.x * 32 + threadIdx.x, x = blockIdx.y * 8 + threadIdx.y;
    const int c = blockIdx.z % 3, b = blockIdx.z / 3;
    if (x >= w || y >= h) return;
    const int an = block / 2;
    const float* __restrict__ S = covT + ((long long)b * 3 + c) * w * hp + y;
    double s = (double)S[(long long)src_col(x, an, w) * hp];
    for (int k = 1; k < block; ++k) s = __dadd_rn(s, (double)S[(long long)src_col(x + k, an, w) * hp]);
    rows[(((long long)b * 3 + c) * h + y) * wd + x] = s;
}

// ---- col_scan_kernel ------------------------------------------------------------------------------------------
// Same specialisation along y: warps 0..2 are the chains of the three channels (lane = column; two dependent DADDs
// per pixel:  t = SUM + entering row,  SUM = t - leaving row), twenty-four helper warps stage the entering / leaving
// row-sum rows with cp.async kColStages-1 chunks ahead and turn the finished box sums of the previous chunk into the
// eigenvalue (G.6), the masked maximum and the coalesced float32 output.  Coupling by named-barrier signals only
// (stage full / t full / t empty).
constexpr int kColChunk = 16;     // y steps per chunk
constexpr int kColStages = 6;     // stages of operand rows (ring between the loaders and the chains)
constexpr int kColRing = 4;       // chunks of box sums between the chains and the helpers
constexpr int kColThreads = 96 + 768, kColHelpers = kColThreads - 96;   // threads that take part in the named barriers
constexpr int kColBlock = 1024;   // chains = warps 0, 4, 8 (one scheduler to themselves), helpers = the warps of the other three schedulers
struct ColSmem {
    double st[kColStages][2][3][kColChunk][32];   // [stage][entering / leaving][channel][row][column]
    float t[kColRing][3][kColChunk][32];
};
enum { kBarColStFull = 1, kBarColTFull = 1 + kColStages, kBarColTEmpty = 1 + kColStages + kColRing };

__global__ void __launch_bounds__(kColBlock)
col_scan_kernel(const double* __restrict__ rows, int w, int h, int wd, int block, float* __restrict__ eig, long long eig_pitch,
                long long eig_batch_stride, const uint8_t* __restrict__ mask, long long mask_pitch, long long mask_batch_stride,
                unsigned* __restrict__ max_out)
{
    extern __shared__ __align__(16) uint8_t smem_raw[];
    ColSmem& sm = *reinterpret_cast<ColSmem*>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, wrp = tid >> 5;
    const int x0 = blockIdx.x * 32;
    const int an = block / 2;
    const long long plane = (long long)h * wd;
    const double* __restrict__ R = rows + (long long)blockIdx.z * 3 * plane + x0;
    const int nck = (h + kColChunk - 1) / kColChunk;

    if ((wrp & 3) == 0) {
        // ---- chain warps: 0, 4, 8 (all on the first warp scheduler, which no helper shares); the rest of that scheduler idles
        if (wrp > 8) return;
        const int ch = wrp >> 2;
        const double* __restrict__ Rx = R + ch * plane + lane;
        double s = 0.0;
        for (int i0 = 0; i0 < block - 1; i0 += 16) {
            double v[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = Rx[(long long)reflect101(min(i0 + i, block - 2) - an, h) * wd];
#pragma unroll
            for (int i = 0; i < 16; ++i)
                if (i0 + i < block - 1) s = __dadd_rn(s, v[i]);
        }
        const bool tl_on = g_timeline_on == 2 && wrp == 0 && lane == 0 && blockIdx.x == 0 && blockIdx.z == 0;
        for (int k = 0; k < nck; ++k) {
            const bool tl = tl_on && k < 256;
            if (tl) g_timeline[4 * k] = clock64();
            bar_sync(kBarColStFull + k % kColStages, kColThreads);                        // operand rows of chunk k staged
            if (tl) g_timeline[4 * k + 1] = clock64();
            if (k >= kColRing) bar_sync(kBarColTEmpty + k % kColRing, kColThreads);       // chunk k - kColRing turned into eigenvalues
            if (tl) g_timeline[4 * k + 2] = clock64();
            const double* __restrict__ pe = &sm.st[k % kColStages][0][ch][0][lane];
            const double* __restrict__ pl = &sm.st[k % kColStages][1][ch][0][lane];
            float* __restrict__ pt = &sm.t[k % kColRing][ch][0][lane];
            // 8 steps at a time: the block has 1024 threads, i.e. 64 registers per thread -- with all 32 operands of a chunk
            // "in registers first" ptxas had to reload just in time and every step paid a shared-memory latency (timeline: 52
            // cycles per step for two dependent DADDs)
#pragma unroll
            for (int g = 0; g < kColChunk / 8; ++g) {
                double ve[8], vl[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) { ve[j] = pe[(8 * g + j) * 32]; vl[j] = pl[(8 * g + j) * 32]; }
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    ve[j] = __dadd_rn(s, ve[j]);
                    s = __dsub_rn(ve[j], vl[j]);
                }
#pragma unroll
                for (int j = 0; j < 8; ++j) pt[(8 * g + j) * 32] = __double2float_rn(ve[j]);
            }
            bar_arrive(kBarColTFull + k % kColRing, kColThreads);   // also: this chain is done with the stage
            if (tl) g_timeline[4 * k + 3] = clock64();
        }
        return;
    }
    // ---- helper warps: every thread owns 4 fixed 16-byte pieces of each stage and up to 2 pixels of each chunk ----
    const int ht = (wrp - 1 - (wrp >> 2)) * 32 + lane;
    float* __restrict__ E = eig + (long long)blockIdx.z * eig_batch_stride;
    const uint8_t* __restrict__ M = mask ? mask + (long long)blockIdx.z * mask_batch_stride : nullptr;
    constexpr int NRG = kColHelpers / 96;               // row groups: 16 pieces x 6 planes per row
    static_assert(kColHelpers % 96 == 0 && kColChunk % NRG == 0, "whole rows per helper thread");
    const int part2 = (ht & 15) * 2;                   // piece = 2 doubles of a 32-column row
    const int pp = (ht >> 4) % 6, prg = (ht >> 4) / 6;  // plane (entering / leaving x channel), row group 0..NRG-1
    const int plt = pp / 3, pc = pp - 3 * plt;
    const double* __restrict__ Rp = R + pc * plane + part2;
    auto issue = [&](int k) {   // rows entering (y + block - 1 - an) and leaving (y - an) for y in chunk k
        if (k < nck) {
            double* st = &sm.st[k % kColStages][plt][pc][0][part2];
#pragma unroll
            for (int i = 0; i < kColChunk / NRG; ++i) {
                const int r = prg + NRG * i;
                const int y = min(k * kColChunk + r, h - 1);
                const int sy = reflect101(plt ? y - an : y + block - 1 - an, h);
                cp_async16(st + r * 32, Rp + (long long)sy * wd);
            }
        }
        cp_async_commit();
    };
    unsigned best = 0;   // 0 = nothing seen (every real float maps above it)
    const int fj0 = ht >> 5, fx = ht & 31;   // pixels (row fj0, column fx) and (row fj0 + kColHelpers / 32, column fx) of a chunk
    auto load_mask = [&](int k, unsigned& m0, unsigned& m1) {
        m0 = 1u; m1 = 1u;
        if (M && k >= 0 && k < nck) {
            const int x = x0 + fx, ya = k * kColChunk + fj0, yb = ya + kColHelpers / 32;
            if (x < w && ya < h && fj0 < kColChunk) m0 = M[(long long)ya * mask_pitch + x];
            if (x < w && yb < h && fj0 + kColHelpers / 32 < kColChunk) m1 = M[(long long)yb * mask_pitch + x];
        }
    };
    auto finish_px = [&](int k, int j, unsigned m) {
        const int y = k * kColChunk + j, x = x0 + fx;
        const float a = __fmul_rn(sm.t[k % kColRing][0][j][fx], 0.5f), b = sm.t[k % kColRing][1][j][fx], c = __fmul_rn(sm.t[k % kColRing][2][j][fx], 0.5f);
        const float d = __fsub_rn(a, c);
        const float e = __fsub_rn(__fadd_rn(a, c), __fsqrt_rn(__fadd_rn(__fmul_rn(d, d), __fmul_rn(b, b))));   // G.6
        if (x < w && y < h) {
            E[(long long)y * eig_pitch + x] = e;
            if (max_out && m) best = max(best, ordered_from_float(e));
        }
    };
    auto finish = [&](int k, unsigned m0, unsigned m1) {  // eigenvalues of chunk k, once all three chains have delivered it
        bar_sync(kBarColTFull + k % kColRing, kColThreads);
        if (fj0 < kColChunk) finish_px(k, fj0, m0);
        if (fj0 + kColHelpers / 32 < kColChunk) finish_px(k, fj0 + kColHelpers / 32, m1);
        if (k + kColRing < nck) bar_arrive(kBarColTEmpty + k % kColRing, kColThreads);
    };
#pragma unroll
    for (int k = 0; k < kColStages - 2; ++k) issue(k);
    unsigned mc0 = 1u, mc1 = 1u;
    const bool htl = g_timeline_on == 2 && ht == 0 && blockIdx.x == 0 && blockIdx.z == 0;
    for (int k = 0; k < nck; ++k) {
        // feed the chains first, then finish chunk k - 2 (two chunks of slack before they could starve)
        long long* tl = (htl && k < 256) ? g_timeline + 1024 + 6 * k : nullptr;
        if (tl) tl[0] = clock64();
        cp_async_wait<kColStages - 3>();       // chunk k has landed (this thread's pieces)
        if (tl) tl[1] = clock64();
        bar_arrive(kBarColStFull + k % kColStages, kColThreads);
        unsigned mn0, mn1;
        load_mask(k - 1, mn0, mn1);            // consumed one iteration later: the load latency hides behind the waits
        if (tl) tl[2] = clock64();
        if (k >= 2) finish(k - 2, mc0, mc1);   // implies: the chains are done with the stage of chunk k - 2 ...
        if (tl) tl[3] = clock64();
        issue(k + kColStages - 2);             // ... which is the stage this refills
        if (tl) { tl[4] = clock64(); tl[5] = tl[4]; }
        mc0 = mn0; mc1 = mn1;
    }
    if (nck >= 2) {
        finish(nck - 2, mc0, mc1);
        load_mask(nck - 1, mc0, mc1);
    } else {
        load_mask(0, mc0, mc1);
    }
    finish(nck - 1, mc0, mc1);
    if (max_out) {
        best = __reduce_max_sync(kFullMask, best);
        if (lane == 0 && best) atomicMax(max_out + blockIdx.z, best);
    }
}

// ---- candidates_kernel ----------------------------------------------------------------------------------------
// 32 x 32 pixel tile per block (4 rows per thread); the tile's candidates are counted first so that the block takes
// its slots in the output list with ONE atomicAdd.
__global__ void __launch_bounds__(256)
candidates_kernel(const float* __restrict__ eig, long long eig_pitch, long long eig_batch_stride, int w, int h,
                  const uint8_t* __restrict__ mask, long long mask_pitch, long long mask_batch_stride,
                  const unsigned* __restrict__ max_in, double quality, unsigned long long* __restrict__ keys,
                  long long keys_batch_stride, int capacity, unsigned* __restrict__ count)
{
    __shared__ unsigned sWarp[8];
    __shared__ unsigned sBase;
    const int lane = threadIdx.x, wrp = threadIdx.y;
    const int x = blockIdx.x * 32 + lane;
    const int b = blockIdx.z;
    const unsigned mo = max_in[b];
    const float max_val = mo ? float_from_ordered(mo) : 0.f;                    // minMaxLoc over an empty mask gives 0
    const float thr = __double2float_rn(__dmul_rn((double)max_val, quality));   // G.7
    float val[4];
    unsigned cand = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int y = blockIdx.y * 32 + wrp * 4 + k;
        val[k] = 0.f;
        if (x >= 1 && x < w - 1 && y >= 1 && y < h - 1) {
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
                if (v == m) { cand |= 1u << k; val[k] = v; }
            }
        }
    }
    const int mine = __popc(cand);
    // exclusive prefix of `mine` over the block: warp scan + 8 warp totals
    int incl = mine;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const int t = __shfl_up_sync(kFullMask, incl, off);
        if (lane >= off) incl += t;
    }
    if (lane == 31) sWarp[wrp] = (unsigned)incl;
    __syncthreads();
    unsigned before = 0, total = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const unsigned t = sWarp[i];
        before += (i < wrp) ? t : 0u;
        total += t;
    }
    if (total == 0) return;
    if (lane == 0 && wrp == 0) sBase = atomicAdd(count + b, total);
    __syncthreads();
    unsigned slot = sBase + before + (unsigned)(incl - mine);
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (cand & (1u << k)) {
            const int y = blockIdx.y * 32 + wrp * 4 + k;
            if (slot < (unsigned)capacity)
                keys[(long long)b * keys_batch_stride + slot] = ((unsigned long long)ordered_from_float(val[k]) << 32) | ((unsigned)y << 16) | (unsigned)x;
            ++slot;
        }
}

// ---- rank_keys_kernel / scatter_keys_kernel ------------------------------------------------------------------
// Sorting a few thousand 64-bit keys on ONE SM is issue-bound (a shared-memory bitonic sort of 8192 keys measured
// 82 us); the whole chip does it by brute force in a few microseconds: the keys are distinct, so the position of key i
// in the descending order is the number of keys greater than it.  Block (bi, bj) counts, for 256 keys i, how many of
// the 1024 keys of chunk bj are greater (chunk in shared memory, broadcast reads) and adds the partial count to
// rank[i]; a second small kernel writes every key to its position -- straight into page-locked host memory mapped into
// the device address space when `out` points there, together with a one-word header (count | sorted << 32).  More
// than kSortMax candidates (plateaus of equal eigenvalues, 4K frames) are passed through unsorted (sorted = 0): the
// host sorts them, or radix_sort_keys_kernel does in the batched frame step.
constexpr int kSortMax = 8192;
constexpr int kRankI = 256, kRankJ = 256;

__global__ void __launch_bounds__(kRankI / 2)
rank_keys_kernel(const unsigned long long* __restrict__ keys, long long keys_batch_stride, const unsigned* __restrict__ count,
                 unsigned* __restrict__ rank)
{
    __shared__ unsigned long long sj[kRankJ];
    const int b = blockIdx.z;
    const int n = (int)count[b];
    const int i0 = blockIdx.x * kRankI, j0 = blockIdx.y * kRankJ;
    if (n > kSortMax || i0 >= n || j0 >= n) return;
    const unsigned long long* __restrict__ src = keys + (long long)b * keys_batch_stride;
    for (int j = threadIdx.x; j < kRankJ; j += kRankI / 2) sj[j] = (j0 + j < n) ? src[j0 + j] : 0ull;   // 0 is below every key
    __syncthreads();
    // two keys per thread: one broadcast shared-memory load feeds two comparisons
    const int ia = i0 + threadIdx.x, ib = ia + kRankI / 2;
    const unsigned long long ka = (ia < n) ? src[ia] : ~0ull, kb = (ib < n) ? src[ib] : ~0ull;
    unsigned above_a = 0, above_b = 0;
#pragma unroll 16
    for (int j = 0; j < kRankJ; ++j) {
        const unsigned long long v = sj[j];
        above_a += (v > ka) ? 1u : 0u;
        above_b += (v > kb) ? 1u : 0u;
    }
    if (ia < n && above_a) atomicAdd(rank + (long long)b * kSortMax + ia, above_a);
    if (ib < n && above_b) atomicAdd(rank + (long long)b * kSortMax + ib, above_b);
}

// one block per image: keys to their positions in shared memory, then out in contiguous runs
__global__ void __launch_bounds__(1024)
scatter_keys_kernel(const unsigned long long* __restrict__ keys, long long keys_batch_stride, const unsigned* __restrict__ count,
                    const unsigned* __restrict__ rank, unsigned long long* __restrict__ out, long long out_batch_stride, int out_capacity)
{
    extern __shared__ __align__(16) unsigned long long sk[];
    const int b = blockIdx.x, tid = threadIdx.x;
    const unsigned total = count[b];
    const unsigned long long* __restrict__ src = keys + (long long)b * keys_batch_stride;
    unsigned long long* __restrict__ dst = out + (long long)b * out_batch_stride;   // dst[0] = header, keys from dst[1]
    const bool sorted = total <= (unsigned)kSortMax;
    const int n_out = (int)min(total, (unsigned)out_capacity);
    if (tid == 0) dst[0] = (unsigned long long)total | (sorted ? (1ull << 32) : 0ull);
    if (sorted) {
        for (int i = tid; i < (int)total; i += 1024) sk[rank[(long long)b * kSortMax + i]] = src[i];
        __syncthreads();
        for (int i = tid; i < n_out; i += 1024) dst[1 + i] = sk[i];
    } else {
        for (int i = tid; i < n_out; i += 1024) dst[1 + i] = src[i];
    }
}

// ---- radix_sort_keys_kernel ------------------------------------------------------------------------------------
// Descending sort of the frames with more than kSortMax candidates (textured frames at a low qualityLevel, 4K frames),
// one CTA per frame: LSD radix sort of the whole 64-bit key, 8 passes of 8 bits, between the key list and a scratch
// list of the same size.  The other frames return at once, so the launch is the same whatever the counts are (a CUDA
// graph can hold it).  Each warp owns one contiguous slice of the list: its per-digit histogram, the scan over
// (digit, warp) and an in-order scatter (warp match on the digit for the rank among equal digits) keep every pass stable.
// A pass whose digit is the same for every key of the frame is skipped.  Keys are distinct, so the result is the
// descending order of the key, i.e. OpenCV's order including its tie rule.  The sorted list ends in `keys`.
constexpr int kRadixThreads = 1024;
constexpr int kRadixWarps = kRadixThreads / 32;

__global__ void __launch_bounds__(kRadixThreads)
radix_sort_keys_kernel(unsigned long long* __restrict__ keys, long long keys_batch_stride, const unsigned* __restrict__ count,
                       unsigned long long* __restrict__ alt, long long alt_batch_stride)
{
    __shared__ unsigned s_off[kRadixWarps][256];   // per warp and (inverted) digit: count, then the next output slot
    __shared__ unsigned s_wsum[8];
    __shared__ int s_skip;
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wrp = tid >> 5;
    const unsigned n = count[b];
    if (n <= (unsigned)kSortMax) return;
    unsigned long long* src = keys + (long long)b * keys_batch_stride;
    unsigned long long* dst = alt + (long long)b * alt_batch_stride;
    const unsigned chunk = (n + kRadixWarps - 1) / kRadixWarps;
    const unsigned lo = min(n, chunk * wrp), hi = min(n, lo + chunk);
    for (int shift = 0; shift < 64; shift += 8) {
        for (int i = tid; i < kRadixWarps * 256; i += kRadixThreads) (&s_off[0][0])[i] = 0u;
        if (tid == 0) s_skip = 0;
        __syncthreads();
        for (unsigned i = lo + lane; i < hi; i += 32) atomicAdd(&s_off[wrp][255u - (unsigned)((src[i] >> shift) & 0xffu)], 1u);
        __syncthreads();
        // digit totals, their exclusive scan (ascending inverted digit = descending digit), then the slot of every warp
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
        const bool skip = s_skip;   // every key has the same digit: the pass would not move anything
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
            const unsigned long long k = valid ? src[i] : 0ull;
            const unsigned d = valid ? 255u - (unsigned)((k >> shift) & 0xffu) : 256u + lane;   // padding lanes match nobody
            const unsigned peers = __match_any_sync(kFullMask, d);
            if (valid) dst[s_off[wrp][d] + __popc(peers & ((1u << lane) - 1u))] = k;
            __syncwarp();
            if (valid && lane == __ffs(peers) - 1) s_off[wrp][d] += __popc(peers);
            __syncwarp();
        }
        __syncthreads();
        if (!skip) { unsigned long long* t = src; src = dst; dst = t; }
    }
    if (src != keys + (long long)b * keys_batch_stride)
        for (unsigned i = tid; i < n; i += kRadixThreads) dst[i] = src[i];
}

// ---- select_corners_kernel ------------------------------------------------------------------------------------
// The greedy minimum-distance selection of goodFeaturesToTrack (G.8) on the device, one block per image.  The
// candidates arrive sorted (strongest first); a candidate is accepted iff no ACCEPTED stronger candidate lies closer
// than minDistance.  Accepted corners paint their disc (dx^2 + dy^2 < minDistance^2) into a bitmap of the image, so "is
// there an accepted corner from an earlier window nearby" is one bit test.  The candidates are processed in windows of
// 128 (one per thread); inside a window every thread builds the 128-bit mask of stronger window members within
// minDistance, and the sequential rule is resolved as a fixpoint (accepted if all conflicting predecessors are rejected,
// rejected if one is accepted; the first undecided one always decides, typically 2-4 rounds).  Identical to the
// sequential result by construction.  minDistance < 1 (radius -1): nothing conflicts, the first candidates are taken, as
// OpenCV does without its grid.
// kGlobalBitmap: the bitmap is in global memory (zeroed by the launcher), for images whose bitmap exceeds the 180 KB of
// shared memory (3840 x 2160); otherwise it is in shared memory.  kAnyRadius: a selection radius over kSelMaxRadius;
// the half widths of the disc are computed per row and the distances in 64 bits (dx^2 + dy^2 reaches 2 * 65535^2).
// Without it the radius is at most 63: a table, and 32-bit distances.
// The keys of image b are the first 8192 of sorted[b] (rank sort; sorted[b][0] is the header, the count in its low word)
// when it has at most 8192, else keys[b] (radix sort).  Its corners are appended to its row of `out` after the first[b]
// points already there (the survivors of the frame step): at most k_b = min(max_corners, cap - first[b]) of them, the
// greedy result with maxCorners = k_b.  next_counts[b] = first[b] + n_new[b].  ids_out / next_id (optional): corner j of
// image b gets id next_id[b] + j in the same slot of ids_out, and next_id[b] grows by n_new[b].
constexpr int kSelThreads = 128;
constexpr int kSelMaxRadius = 63;               // radii up to this take the half widths from a table
constexpr int kSelMaxBitmapWords = 45 * 1024;   // 180 KB

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

template <bool kGlobalBitmap, bool kAnyRadius>
__global__ void __launch_bounds__(kSelThreads)
select_corners_kernel(const unsigned long long* __restrict__ sorted, long long sorted_batch_stride,
                      const unsigned long long* __restrict__ keys, long long keys_batch_stride, int w, int h,
                      long long md2, int radius, int max_corners, long long cap, const int* __restrict__ first,
                      float2* __restrict__ out, long long out_stride, int* __restrict__ next_counts, int* __restrict__ n_new,
                      int* __restrict__ ids_out, int* __restrict__ next_id, unsigned* __restrict__ gbitmap, long long gbitmap_stride)
{
    extern __shared__ __align__(16) unsigned sel_smem[];
    __shared__ unsigned short sx[kSelThreads], sy[kSelThreads];
    __shared__ unsigned s_alive[4], s_acc[4], s_rej[4];
    __shared__ short s_halfw[kSelMaxRadius + 1];
    __shared__ unsigned short s_ax[kSelThreads], s_ay[kSelThreads];
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wrp = tid >> 5;
    const unsigned long long* __restrict__ src = sorted + (long long)b * sorted_batch_stride;   // src[0] = header
    const int n = (int)(src[0] & 0xffffffffu);
    const unsigned long long* __restrict__ list = n <= kSortMax ? src + 1 : keys + (long long)b * keys_batch_stride;
    const int fb = first[b];
    const int k_max = (int)min((long long)max_corners, cap - fb);
    const int id0 = ids_out ? next_id[b] : 0;
    if (k_max <= 0) {
        if (tid == 0) { n_new[b] = 0; next_counts[b] = fb; }
        return;
    }
    const int wpr = (w + 31) >> 5;
    const int nwords = wpr * h;
    unsigned* bitmap = kGlobalBitmap ? gbitmap + (long long)b * gbitmap_stride : sel_smem;
    if (!kGlobalBitmap)
        for (int i = tid; i < nwords; i += kSelThreads) bitmap[i] = 0u;
    if (!kAnyRadius && tid <= radius) s_halfw[tid] = (short)sel_halfwidth(md2, tid);
    __syncthreads();
    int accepted_total = 0;
    float2* corners = out + (long long)b * out_stride + fb;
    for (int base = 0; base < n && accepted_total < k_max; base += kSelThreads) {
        const int t = base + tid;
        int x = 0, y = 0;
        bool alive = false;
        if (t < n) {
            const unsigned long long key = list[t];
            x = (int)(key & 0xffffu); y = (int)((key >> 16) & 0xffffu);
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
            corners[accepted_total + before] = make_float2((float)x, (float)y);   // < k_max: nkeep is capped
            if (ids_out) ids_out[(long long)b * out_stride + fb + accepted_total + before] = id0 + accepted_total + before;
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
    if (tid == 0) {
        n_new[b] = accepted_total;
        next_counts[b] = fb + accepted_total;
        if (ids_out) next_id[b] = id0 + accepted_total;
    }
}

// ---- mask_from_points_kernel ----------------------------------------------------------------------------------
// The detection mask of reference src/extractor/extractor.py:102-107 on the device: 255 everywhere, then a filled
// cv2.circle of value 0 around np.int32(x, y) of every tracked keypoint.  OpenCV's filled circle is the midpoint circle:
// row cy +- d is filled over [cx - half[d], cx + half[d]] (table computed by the launcher with OpenCV's octant walk).
// Batched: blockIdx.y / blockIdx.z is the image; image b has counts[b] points (or n without counts) at pts + b * pts_stride.
struct CircleTable { short half[128]; };

__global__ void __launch_bounds__(256)
mask_fill_kernel(uint8_t* __restrict__ mask, long long pitch, long long batch_stride, int w, int h)
{
    const int x = (blockIdx.x * 256 + threadIdx.x) * 4, y = blockIdx.y;
    if (x >= w) return;
    uint8_t* p = mask + (long long)blockIdx.z * batch_stride + (long long)y * pitch + x;
    if (x + 3 < w && ((reinterpret_cast<uintptr_t>(p) & 3) == 0)) *reinterpret_cast<unsigned*>(p) = 0xffffffffu;
    else for (int i = 0; i < 4 && x + i < w; ++i) p[i] = 255;
}

__global__ void __launch_bounds__(256)
mask_from_points_kernel(const float* __restrict__ pts, long long pts_stride, const int* __restrict__ counts, int n, int radius, int w,
                        int h, uint8_t* __restrict__ mask, long long pitch, long long mask_batch_stride,
                        const __grid_constant__ CircleTable tab)
{
    const int rows_per = 2 * radius + 1;
    const long long t = (long long)blockIdx.x * 256 + threadIdx.x;
    const int b = blockIdx.y;
    const int nb = counts ? min(max(counts[b], 0), n) : n;
    if (t >= (long long)nb * rows_per) return;
    const int i = (int)(t / rows_per), d = (int)(t - (long long)i * rows_per) - radius;
    const float* __restrict__ pt = pts + 2 * ((long long)b * pts_stride + i);
    const float fx = pt[0], fy = pt[1];
    if (!(fabsf(fx) < 1.0e9f) || !(fabsf(fy) < 1.0e9f)) return;         // NaN / out of int range: np.int32 is undefined there
    const int cx = (int)fx, cy = (int)fy;                                 // truncation toward zero, like np.int32
    const int y = cy + d, hw = tab.half[d < 0 ? -d : d];
    if (y < 0 || y >= h || hw < 0) return;
    const int x1 = max(cx - hw, 0), x2 = min(cx + hw, w - 1);
    uint8_t* __restrict__ row = mask + (long long)b * mask_batch_stride + (long long)y * pitch;
    for (int x = x1; x <= x2; ++x) row[x] = 0;
}

}  // namespace

long long corners_ws_bytes(int w, int h, int batch)
{
    const long long hp = (h + 31) / 32 * 32, wd = (w + 31) / 32 * 32;
    const long long cov = 3LL * w * hp * 4, rows = 3LL * h * wd * 8;
    return ((cov + 255) / 256 * 256 + (rows + 255) / 256 * 256) * batch;
}

klt_status corner_min_eig_launch(const uint8_t* img, long long pitch, long long batch_stride, int w, int h, int batch,
                                 int block, float* eig, long long eig_pitch, long long eig_batch_stride,
                                 const uint8_t* mask, long long mask_pitch, long long mask_batch_stride,
                                 unsigned* max_out, void* ws, cudaStream_t stream)
{
    if (w < 1 || h < 1 || batch < 1 || block < 1) return KLT_ERR_INVALID_ARG;
    if (block / 2 >= w || block / 2 >= h || batch > 21845 || (w + 7) / 8 > 65535) return KLT_ERR_UNSUPPORTED;
    const int hp = (h + 31) / 32 * 32, wd = (w + 31) / 32 * 32;
    const long long cov_bytes = (3LL * w * hp * 4 * batch + 255) / 256 * 256;
    float* covT = static_cast<float*>(ws);
    double* rows = reinterpret_cast<double*>(static_cast<uint8_t*>(ws) + cov_bytes);
    const float k1 = (float)(1.0 / (4.0 * (double)block * 255.0));   // G.1
    const float k0 = (float)(2.0 / (4.0 * (double)block * 255.0));
    cov_kernel<<<dim3((w + kTile - 1) / kTile, (h + kTile - 1) / kTile, batch), dim3(32, 8), 0, stream>>>(
        img, pitch, batch_stride, w, h, covT, hp, k1, k0);
    static PerDeviceOnce configured;
    if (configured.needed()) {
        cudaError_t ce = cudaFuncSetAttribute(row_scan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(RowSmem));
        if (ce == cudaSuccess) ce = cudaFuncSetAttribute(col_scan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(ColSmem));
        if (ce != cudaSuccess) return (klt_status)ce;
    }
    if (block <= 5)
        row_sum_small_kernel<<<dim3((h + 31) / 32, (w + 7) / 8, 3 * batch), dim3(32, 8), 0, stream>>>(covT, w, h, hp, block, rows, wd);
    else
        row_scan_kernel<<<dim3((h + 31) / 32, 3, batch), kRowBlock, sizeof(RowSmem), stream>>>(covT, w, h, hp, block, rows, wd);
    col_scan_kernel<<<dim3((w + 31) / 32, 1, batch), kColBlock, sizeof(ColSmem), stream>>>(rows, w, h, wd, block, eig, eig_pitch, eig_batch_stride,
                                                                                         mask, mask_pitch, mask_batch_stride, max_out);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KLT_OK : (klt_status)e;
}

klt_status corner_candidates_launch(const float* eig, long long eig_pitch, long long eig_batch_stride, int w, int h, int batch,
                                    const uint8_t* mask, long long mask_pitch, long long mask_batch_stride,
                                    const unsigned* max_in, double quality, unsigned long long* keys,
                                    long long keys_batch_stride, int capacity, unsigned* count, cudaStream_t stream)
{
    if (w < 1 || h < 1 || batch < 1 || capacity < 0 || !(quality > 0)) return KLT_ERR_INVALID_ARG;
    if (batch > 65535 || w > 65535 || h > 65535) return KLT_ERR_UNSUPPORTED;
    candidates_kernel<<<dim3((w + 31) / 32, (h + 31) / 32, batch), dim3(32, 8), 0, stream>>>(
        eig, eig_pitch, eig_batch_stride, w, h, mask, mask_pitch, mask_batch_stride, max_in, quality, keys, keys_batch_stride,
        capacity, count);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KLT_OK : (klt_status)e;
}

klt_status corner_sort_launch(const unsigned long long* keys, long long keys_batch_stride, const unsigned* count, int batch,
                              unsigned* rank, unsigned long long* out, long long out_batch_stride, int out_capacity,
                              cudaStream_t stream)
{
    if (batch < 1 || batch > 65535 || out_capacity < 0) return KLT_ERR_INVALID_ARG;
    // rank: batch * 8192 words, zeroed by the caller
    static PerDeviceOnce configured;
    if (configured.needed()) {
        cudaError_t ce = cudaFuncSetAttribute(scatter_keys_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSortMax * 8);
        if (ce != cudaSuccess) return (klt_status)ce;
    }
    rank_keys_kernel<<<dim3(kSortMax / kRankI, kSortMax / kRankJ, batch), kRankI / 2, 0, stream>>>(keys, keys_batch_stride, count, rank);
    scatter_keys_kernel<<<batch, 1024, kSortMax * 8, stream>>>(keys, keys_batch_stride, count, rank, out, out_batch_stride, out_capacity);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KLT_OK : (klt_status)e;
}

klt_status corner_radix_sort_launch(unsigned long long* keys, long long keys_batch_stride, const unsigned* count, int batch,
                                    unsigned long long* alt, long long alt_batch_stride, cudaStream_t stream)
{
    if (batch < 1 || batch > 0x7fffffff || !keys || !count || !alt) return KLT_ERR_INVALID_ARG;
    radix_sort_keys_kernel<<<batch, kRadixThreads, 0, stream>>>(keys, keys_batch_stride, count, alt, alt_batch_stride);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KLT_OK : (klt_status)e;
}

klt_status corner_select_launch(const unsigned long long* sorted, long long sorted_batch_stride, const unsigned long long* keys,
                                long long keys_batch_stride, int w, int h, int batch, double min_distance, int max_corners,
                                long long cap, const int* first, float* out, long long out_stride, int* next_counts, int* n_new,
                                int* ids_out, int* next_id, unsigned* gbitmap, long long gbitmap_stride, cudaStream_t stream)
{
    if (batch < 1 || w < 1 || h < 1 || w > 65535 || h > 65535 || !(min_distance >= 0) || max_corners < 1 || !sorted || !keys ||
        !first || !out || !next_counts || !n_new || (!ids_out != !next_id))
        return KLT_ERR_INVALID_ARG;
    long long md2 = 0;
    int radius = -1;   // minDistance < 1: no conflicts (OpenCV takes the first candidates without a grid there)
    if (min_distance >= 1) {
        const double md2d = ceil(min_distance * min_distance);   // squared pixel distances are integers: d2 < md2 <=> d2 < ceil(md2)
        md2 = md2d < 4.0e18 ? (long long)md2d : (long long)4.0e18;
        // largest r with r^2 < md2, at most max(w, h): every offset inside the image is within that
        const int rmax = w > h ? w : h;
        radius = 0;
        while (radius < rmax && (long long)(radius + 1) * (radius + 1) < md2) ++radius;
    }
    const long long nwords = (long long)((w + 31) / 32) * h;
    const bool in_smem = nwords <= kSelMaxBitmapWords, any_radius = radius > kSelMaxRadius;
    auto kernel = in_smem ? (any_radius ? select_corners_kernel<false, true> : select_corners_kernel<false, false>)
                          : (any_radius ? select_corners_kernel<true, true> : select_corners_kernel<true, false>);
    cudaError_t e = cudaSuccess;
    if (in_smem) {
        static PerDeviceOnce configured;
        if (configured.needed()) {
            e = cudaFuncSetAttribute(select_corners_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSelMaxBitmapWords * 4);
            if (e == cudaSuccess)
                e = cudaFuncSetAttribute(select_corners_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSelMaxBitmapWords * 4);
            if (e != cudaSuccess) return (klt_status)e;
        }
    } else {
        if (!gbitmap || gbitmap_stride < nwords) return KLT_ERR_INVALID_ARG;
        e = cudaMemset2DAsync(gbitmap, (size_t)gbitmap_stride * 4, 0, (size_t)nwords * 4, (size_t)batch, stream);
        if (e != cudaSuccess) return (klt_status)e;
    }
    kernel<<<batch, kSelThreads, in_smem ? (size_t)nwords * 4 : 0, stream>>>(
        sorted, sorted_batch_stride, keys, keys_batch_stride, w, h, md2, radius, max_corners, cap, first, reinterpret_cast<float2*>(out),
        out_stride, next_counts, n_new, ids_out, next_id, gbitmap, gbitmap_stride);
    e = cudaGetLastError();
    return e == cudaSuccess ? KLT_OK : (klt_status)e;
}

klt_status corner_mask_from_points_launch(const float* pts, long long pts_stride, const int* counts, int n, int batch, int radius,
                                          int w, int h, uint8_t* mask, long long pitch, long long mask_batch_stride,
                                          cudaStream_t stream)
{
    if (n < 0 || batch < 1 || radius < 0 || w < 1 || h < 1 || !mask || pitch < w || (n > 0 && !pts)) return KLT_ERR_INVALID_ARG;
    if (batch > 1 && (pts_stride < n || mask_batch_stride < pitch * (long long)(h - 1) + w)) return KLT_ERR_INVALID_ARG;
    if (radius > 127 || h > 65535 || batch > 65535) return KLT_ERR_UNSUPPORTED;
    CircleTable tab;
    for (int i = 0; i < 128; ++i) tab.half[i] = -1;
    {   // OpenCV's Circle() octant walk (drawing.cpp): rows cy -+ dy get [cx - dx, cx + dx], rows cy -+ dx get [cx - dy, cx + dy]
        int err = 0, dx = radius, dy = 0, plus = 1, minus = (radius << 1) - 1;
        while (dx >= dy) {
            if (dx > tab.half[dy]) tab.half[dy] = (short)dx;
            if (dy > tab.half[dx]) tab.half[dx] = (short)dy;
            dy++;
            err += plus;
            plus += 2;
            const int m = (err <= 0) - 1;
            err -= minus & m;
            dx += m;
            minus -= m & 2;
        }
    }
    mask_fill_kernel<<<dim3((w + 1023) / 1024, h, batch), 256, 0, stream>>>(mask, pitch, mask_batch_stride, w, h);
    const long long total = (long long)n * (2 * radius + 1);   // threads per image (the most points an image may have)
    if (total > 0) {
        if ((total + 255) / 256 > 0x7fffffffLL) return KLT_ERR_UNSUPPORTED;
        mask_from_points_kernel<<<dim3((unsigned)((total + 255) / 256), batch), 256, 0, stream>>>(pts, pts_stride, counts, n, radius, w, h,
                                                                                                   mask, pitch, mask_batch_stride, tab);
    }
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KLT_OK : (klt_status)e;
}

}  // namespace klt

// profiling aid, not part of the ABI of include/klt_b200.h: switch the chain-warp timeline on / read it back
extern "C" int klt_debug_corner_timeline(int enable, long long* out, int n_words)
{
    cudaError_t e = cudaMemcpyToSymbol(klt::g_timeline_on, &enable, sizeof(int));
    if (e == cudaSuccess && out && n_words > 0)
        e = cudaMemcpyFromSymbol(out, klt::g_timeline, sizeof(long long) * (size_t)(n_words < 2560 ? n_words : 2560));
    return (int)e;
}
