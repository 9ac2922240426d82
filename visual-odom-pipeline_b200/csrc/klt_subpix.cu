// Sub-pixel corner refinement: cv2.cornerSubPix(image, corners, winSize, zeroZone, criteria) on 8-bit single-channel
// images, batched, on the device, in place.
//
// Arithmetic = OpenCV's own code path (oracle/subpix_oracle.c S.1-S.6): per iteration a float32 getRectSubPix patch of
// (2wx + 3) x (2wy + 3) (interior recurrence or the adjustRect border path), central differences in float, five double
// sums in row-major order, a 2 x 2 solve in double, the float32 update.  The weight mask is computed on the host with the
// C library's expf (CUDA's expf is another function) and passed by value.
//
// One warp per corner.  The lanes build the patch and the per-pixel double terms gxx, gxy, gyy, gxx px + gxy py and
// gxy px + gyy py (each independent of the others, so the parallel build is exact) in shared memory; lane 0 then runs the
// five dependent sums in cv2's order and broadcasts them, and every lane takes the same branch.  The serial part is one
// DADD chain of W * H additions per sum per iteration.
#include "klt_common.cuh"

#include <cfloat>
#include <cmath>

namespace klt {

namespace {

constexpr int kMaxSide = 2 * KLT_MAX_SUBPIX_WIN + 1;
constexpr int kMaxWarps = 4;
constexpr size_t kSmemBudget = 48 * 1024;   // default dynamic shared memory of a block, no opt-in

struct SubpixMask { float w[kMaxSide * kMaxSide]; };

struct SubpixGeom {
    int win_w, win_h;
    int max_iters;
    double eps2;
};

// bytes of one warp's shared memory: the W * H x 5 double terms, then the (W + 2) x (H + 2) float patch
__host__ __device__ inline size_t subpix_warp_bytes(int win_w, int win_h)
{
    const int W = 2 * win_w + 1, H = 2 * win_h + 1;
    return (size_t)W * H * 5 * sizeof(double) + (((size_t)(W + 2) * (H + 2) * sizeof(float) + 15) & ~(size_t)15);
}

// getRectSubPix(img, (pw, ph), (cx, cy), CV_32F) into out[ph][pw], lanes over pixels (S.5 / S.6)
__device__ void rect_patch(const uint8_t* __restrict__ img, int w, int h, long long pitch, int pw, int ph, float cx, float cy,
                           float* out, int lane)
{
    cx = __fsub_rn(cx, __fmul_rn((float)(pw - 1), 0.5f));
    cy = __fsub_rn(cy, __fmul_rn((float)(ph - 1), 0.5f));
    const int ix = (int)floorf(cx), iy = (int)floorf(cy);
    const int n = pw * ph;
    if (0 <= ix && ix + pw < w && 0 <= iy && iy + ph < h) {
        const float a = fmaxf(__fsub_rn(cx, (float)ix), 0.0001f);
        const float b = __fsub_rn(cy, (float)iy);
        const float b1 = __fsub_rn(1.f, b), b2 = b;
        const float a12 = __fmul_rn(a, b1), a22 = __fmul_rn(a, b);
        const double s = __ddiv_rn(__dsub_rn(1.0, (double)a), (double)a);
        for (int p = lane; p < n; p += 32) {
            const int r = p / pw, j = p - r * pw;
            const uint8_t* p0 = img + (long long)(iy + r) * pitch + ix;
            const uint8_t* p1 = p0 + pitch;
            const float t = __fadd_rn(__fmul_rn(a12, (float)p0[j + 1]), __fmul_rn(a22, (float)p1[j + 1]));
            float prev;
            if (j == 0) {
                prev = __fmul_rn(__fsub_rn(1.f, a), __fadd_rn(__fmul_rn(b1, (float)p0[0]), __fmul_rn(b2, (float)p1[0])));
            } else {
                const float tp = __fadd_rn(__fmul_rn(a12, (float)p0[j]), __fmul_rn(a22, (float)p1[j]));
                prev = __double2float_rn(__dmul_rn((double)tp, s));
            }
            out[p] = __fadd_rn(prev, t);
        }
        return;
    }
    const float a = __fsub_rn(cx, (float)ix), b = __fsub_rn(cy, (float)iy);
    const float a1 = __fsub_rn(1.f, a), b1 = __fsub_rn(1.f, b), b2 = b;
    const float a11 = __fmul_rn(a1, b1), a12 = __fmul_rn(a, b1), a21 = __fmul_rn(a1, b), a22 = __fmul_rn(a, b);
    // adjustRect: `col` / `row` are the image column and row of the patch's source origin
    int col, row, rx, rw, ry, rh;
    if (ix >= 0) { col = ix; rx = 0; }
    else { col = 0; rx = min(-ix, pw); }
    if (ix < w - pw) rw = pw;
    else { rw = w - ix - 1; if (rw < 0) { col += rw; rw = 0; } }
    if (iy >= 0) { row = iy; ry = 0; }
    else { row = 0; ry = -iy; }
    if (iy < h - ph) rh = ph;
    else { rh = h - iy - 1; if (rh < 0) { row += rh; rh = 0; } }
    col -= rx;
    for (int p = lane; p < n; p += 32) {
        const int r = p / pw, j = p - r * pw;
        // OpenCV steps the source row once per patch row in [ry, rh); rows outside read one row twice
        const int r0 = row + max(0, min(r, rh) - ry);
        const int r1 = (r >= ry && r < rh) ? r0 + 1 : r0;
        const uint8_t* s1 = img + (long long)r0 * pitch + col;
        const uint8_t* s2 = img + (long long)r1 * pitch + col;
        float v;
        if (j >= rw) v = __fadd_rn(__fmul_rn((float)s1[rw], b1), __fmul_rn((float)s2[rw], b2));
        else if (j < rx) v = __fadd_rn(__fmul_rn((float)s1[rx], b1), __fmul_rn((float)s2[rx], b2));
        else v = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn((float)s1[j], a11), __fmul_rn((float)s1[j + 1], a12)),
                                     __fmul_rn((float)s2[j], a21)), __fmul_rn((float)s2[j + 1], a22));
        out[p] = v;
    }
}

__global__ void __launch_bounds__(32 * kMaxWarps)
subpix_kernel(const uint8_t* __restrict__ imgs, int w, int h, long long pitch, long long batch_stride, float* __restrict__ pts,
              long long row_stride, const int* __restrict__ d_end, const int* __restrict__ d_n, SubpixGeom g, SubpixMask mask)
{
    extern __shared__ __align__(16) uint8_t smem_raw[];
    const int W = 2 * g.win_w + 1, H = 2 * g.win_h + 1, pw = W + 2, ph = H + 2, n_px = W * H;
    float* s_mask = reinterpret_cast<float*>(smem_raw);
    uint8_t* warp_base = smem_raw + ((n_px * sizeof(float) + 15) & ~(size_t)15);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double* s_terms = reinterpret_cast<double*>(warp_base + (size_t)warp * subpix_warp_bytes(g.win_w, g.win_h));
    float* s_patch = reinterpret_cast<float*>(s_terms + (size_t)n_px * 5);
    for (int k = threadIdx.x; k < n_px; k += blockDim.x) s_mask[k] = mask.w[k];
    __syncthreads();

    const int b = blockIdx.y;
    const long long end = min((long long)max(d_end[b], 0), row_stride);
    const long long first = end - min((long long)max(d_n[b], 0), end);
    const uint8_t* img = imgs + (long long)b * batch_stride;
    float* row = pts + (long long)b * row_stride * 2;
    const long long stride = (long long)gridDim.x * (blockDim.x >> 5);
    for (long long slot = first + (long long)blockIdx.x * (blockDim.x >> 5) + warp; slot < end; slot += stride) {
        const float tx = row[2 * slot], ty = row[2 * slot + 1];
        if (!(0.f <= tx && tx < (float)w && 0.f <= ty && ty < (float)h)) continue;   // cv2 raises; NaN too
        float cx = tx, cy = ty;
        int iter = 0;
        float err = 0.f;
        do {
            rect_patch(img, w, h, pitch, pw, ph, cx, cy, s_patch, lane);
            __syncwarp();
            for (int k = lane; k < n_px; k += 32) {
                const int i = k / W, j = k - i * W;
                const float* s = s_patch + (i + 1) * pw + j + 1;
                const double m = (double)s_mask[k];
                const double tgx = (double)__fsub_rn(s[1], s[-1]);
                const double tgy = (double)__fsub_rn(s[pw], s[-pw]);
                const double gxx = __dmul_rn(__dmul_rn(tgx, tgx), m);
                const double gxy = __dmul_rn(__dmul_rn(tgx, tgy), m);
                const double gyy = __dmul_rn(__dmul_rn(tgy, tgy), m);
                const double px = (double)(j - g.win_w), py = (double)(i - g.win_h);
                double* t = s_terms + (size_t)k * 5;
                t[0] = gxx;
                t[1] = gxy;
                t[2] = gyy;
                t[3] = __dadd_rn(__dmul_rn(gxx, px), __dmul_rn(gxy, py));
                t[4] = __dadd_rn(__dmul_rn(gxy, px), __dmul_rn(gyy, py));
            }
            __syncwarp();
            double A = 0, B = 0, C = 0, bb1 = 0, bb2 = 0;
            if (lane == 0) {
#pragma unroll 4
                for (int k = 0; k < n_px; ++k) {
                    const double* t = s_terms + (size_t)k * 5;
                    A = __dadd_rn(A, t[0]);
                    B = __dadd_rn(B, t[1]);
                    C = __dadd_rn(C, t[2]);
                    bb1 = __dadd_rn(bb1, t[3]);
                    bb2 = __dadd_rn(bb2, t[4]);
                }
            }
            A = __shfl_sync(0xffffffffu, A, 0);
            B = __shfl_sync(0xffffffffu, B, 0);
            C = __shfl_sync(0xffffffffu, C, 0);
            bb1 = __shfl_sync(0xffffffffu, bb1, 0);
            bb2 = __shfl_sync(0xffffffffu, bb2, 0);
            const double det = __dsub_rn(__dmul_rn(A, C), __dmul_rn(B, B));
            if (fabs(det) <= DBL_EPSILON * DBL_EPSILON) break;
            const double scale = __ddiv_rn(1.0, det);
            const float nx = __double2float_rn(__dsub_rn(__dadd_rn((double)cx, __dmul_rn(__dmul_rn(C, scale), bb1)),
                                                         __dmul_rn(__dmul_rn(B, scale), bb2)));
            const float ny = __double2float_rn(__dadd_rn(__dsub_rn((double)cy, __dmul_rn(__dmul_rn(B, scale), bb1)),
                                                         __dmul_rn(__dmul_rn(A, scale), bb2)));
            const float dx = __fsub_rn(nx, cx), dy = __fsub_rn(ny, cy);
            err = __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
            if (nx < 0.f || nx >= (float)w || ny < 0.f || ny >= (float)h) break;   // a step out of the image is not taken
            cx = nx;
            cy = ny;
        } while (++iter < g.max_iters && (double)err > g.eps2);
        if (fabsf(__fsub_rn(cx, tx)) > (float)g.win_w || fabsf(__fsub_rn(cy, ty)) > (float)g.win_h) { cx = tx; cy = ty; }
        if (lane == 0) {
            row[2 * slot] = cx;
            row[2 * slot + 1] = cy;
        }
        __syncwarp();
    }
}

}  // namespace

// S.2 on the host: the C library's expf, float32, then the zero zone
void subpix_mask(int win_w, int win_h, int zero_w, int zero_h, float* mask)
{
    const int W = 2 * win_w + 1, H = 2 * win_h + 1;
    for (int i = 0; i < H; ++i) {
        const float y = (float)(i - win_h) / (float)win_h;
        const float vy = ::expf(-y * y);
        for (int j = 0; j < W; ++j) {
            const float x = (float)(j - win_w) / (float)win_w;
            mask[i * W + j] = vy * ::expf(-x * x);
        }
    }
    if (zero_w >= 0 && zero_h >= 0 && 2 * zero_w + 1 < W && 2 * zero_h + 1 < H)
        for (int i = win_h - zero_h; i <= win_h + zero_h; ++i)
            for (int j = win_w - zero_w; j <= win_w + zero_w; ++j) mask[i * W + j] = 0.f;
}

klt_status subpix_launch(const uint8_t* imgs, int w, int h, long long pitch, long long batch_stride, int batch, float* pts,
                         long long row_stride, const int* d_end, const int* d_n, int win_w, int win_h, int zero_w, int zero_h,
                         int crit_type, int max_count, double eps, cudaStream_t stream)
{
    SubpixGeom g;
    g.win_w = win_w;
    g.win_h = win_h;
    g.max_iters = (crit_type & KLT_TERM_COUNT) ? std::min(std::max(max_count, 1), 100) : 100;
    const double e = (crit_type & KLT_TERM_EPS) ? std::max(eps, 0.) : 0.;
    g.eps2 = e * e;
    SubpixMask mask;
    subpix_mask(win_w, win_h, zero_w, zero_h, mask.w);
    const int n_px = (2 * win_w + 1) * (2 * win_h + 1);
    const size_t mask_bytes = ((size_t)n_px * sizeof(float) + 15) & ~(size_t)15;
    const size_t per_warp = subpix_warp_bytes(win_w, win_h);
    const int warps = (int)std::max<size_t>(1, std::min<size_t>(kMaxWarps, (kSmemBudget - mask_bytes) / per_warp));
    const size_t smem = mask_bytes + per_warp * warps;
    if (smem > kSmemBudget) return KLT_ERR_UNSUPPORTED;
    const long long blocks = std::min<long long>((row_stride + warps - 1) / warps, 256);
    if (blocks < 1) return KLT_OK;
    subpix_kernel<<<dim3((unsigned)blocks, (unsigned)batch), 32 * warps, smem, stream>>>(imgs, w, h, pitch, batch_stride, pts, row_stride,
                                                                                       d_end, d_n, g, mask);
    const cudaError_t err = cudaGetLastError();
    return err == cudaSuccess ? KLT_OK : (klt_status)err;
}

}  // namespace klt
