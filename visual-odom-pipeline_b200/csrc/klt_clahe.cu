// Contrast-limited adaptive histogram equalisation of 8-bit single-channel frames, batched, on the device:
// cv2.createCLAHE(clipLimit, tileGridSize).apply(img), bit for bit as OpenCV 4.13's CLAHE_Impl::apply computes it
// (oracle/clahe_oracle.py C.1-C.5, DESIGN.md "CLAHE").
//
// Two launches on the caller's stream, no allocation, no host read, no synchronisation (graph-capturable):
//   clahe_lut_kernel    one CTA per (tile, image): 256-bin histogram of the padded tile in shared memory (the padding,
//                       right and bottom only, is read through reflect101 and never stored), then one warp clips,
//                       redistributes, scans and writes the tile's 256-entry LUT to the workspace.
//   clahe_apply_kernel  one thread per 4 horizontally adjacent pixels (one 32-bit load and store): the bilinear blend of
//                       the four surrounding tiles' LUT entries, in float32, each operation rounded once.
// Each pixel is read and written by the same thread after the LUT pass has finished, so dst may equal src.
#include "klt_common.cuh"

#include <cmath>

namespace klt {

namespace {

constexpr int kHistWarps = 8;                 // one private histogram per warp of the LUT CTA
constexpr int kLutThreads = 32 * kHistWarps;
constexpr int kBX = 32, kBY = 8;              // apply: 128 x 8 pixels per CTA

__device__ __forceinline__ void count4(int* hist, uint32_t v)
{
    atomicAdd(&hist[v & 0xff], 1);
    atomicAdd(&hist[(v >> 8) & 0xff], 1);
    atomicAdd(&hist[(v >> 16) & 0xff], 1);
    atomicAdd(&hist[v >> 24], 1);
}

__global__ void __launch_bounds__(kLutThreads)
clahe_lut_kernel(const uint8_t* __restrict__ src, int w, int h, long long spitch, long long sbatch, int tiles_x, int tw, int th,
                 int clip, float lut_scale, uint8_t* __restrict__ lut)
{
    __shared__ int hist[kHistWarps][256];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int i = tid; i < kHistWarps * 256; i += kLutThreads) (&hist[0][0])[i] = 0;
    __syncthreads();
    const int k = blockIdx.x;
    const int x0 = (k % tiles_x) * tw, y0 = (k / tiles_x) * th;
    const uint8_t* __restrict__ img = src + (long long)blockIdx.y * sbatch;
    int* my = hist[warp];
    // a warp per row, lanes along it; rows past the image bottom are reflected (C.1)
    const bool words = ((x0 | tw) & 3) == 0 && x0 + tw <= w && (spitch & 3) == 0 && (reinterpret_cast<uintptr_t>(img) & 3) == 0;
    for (int r = warp; r < th; r += kHistWarps) {
        const uint8_t* row = img + (long long)reflect101(y0 + r, h) * spitch;
        if (words) {
            const uint32_t* row4 = reinterpret_cast<const uint32_t*>(row + x0);
            for (int c = lane; c < (tw >> 2); c += 32) count4(my, __ldg(row4 + c));
        } else {
            for (int c = lane; c < tw; c += 32) atomicAdd(&my[__ldg(row + reflect101(x0 + c, w))], 1);
        }
    }
    __syncthreads();
    if (warp != 0) return;
    // C.3: lane l owns bins 8l .. 8l + 7
    int cnt[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        int s = 0;
#pragma unroll
        for (int q = 0; q < kHistWarps; ++q) s += hist[q][8 * lane + j];
        cnt[j] = s;
    }
    if (clip > 0) {
        int excess = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j)
            if (cnt[j] > clip) { excess += cnt[j] - clip; cnt[j] = clip; }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) excess += __shfl_xor_sync(0xffffffffu, excess, o);
        const int batch = excess / 256, residual = excess - batch * 256;
        // cv2 adds one to bins 0, s, 2s, ... (s = max(256 / residual, 1)), to the first `residual` of them
        const int step = residual ? max(256 / residual, 1) : 1;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int i = 8 * lane + j;
            cnt[j] += batch + ((residual && i % step == 0 && i / step < residual) ? 1 : 0);
        }
    }
    // C.4: inclusive scan, lut = saturate_u8(rint(float(cumsum) * lut_scale))
#pragma unroll
    for (int j = 1; j < 8; ++j) cnt[j] += cnt[j - 1];
    int incl = cnt[7];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    const int base = incl - cnt[7];
    uint32_t lo = 0, hi = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int v = min(max(__float2int_rn(__fmul_rn(__int2float_rn(base + cnt[j]), lut_scale)), 0), 255);
        if (j < 4) lo |= (uint32_t)v << (8 * j);
        else hi |= (uint32_t)v << (8 * (j - 4));
    }
    uint8_t* out = lut + ((long long)blockIdx.y * gridDim.x + k) * 256;
    reinterpret_cast<uint2*>(out)[lane] = make_uint2(lo, hi);
}

__device__ __forceinline__ float lut_at(const uint8_t* __restrict__ row, int t, int v)
{
    return __int2float_rn(__ldg(row + t * 256 + v));
}

__global__ void __launch_bounds__(kBX * kBY)
clahe_apply_kernel(const uint8_t* src, int w, int h, long long spitch, long long sbatch, uint8_t* dst, long long dpitch,
                   long long dbatch, int tiles_x, int tiles_y, float inv_tw, float inv_th, const uint8_t* __restrict__ lut)
{
    const int y = blockIdx.y * kBY + threadIdx.y;
    const int xb = (blockIdx.x * kBX + threadIdx.x) * 4;
    if (y >= h || xb >= w) return;
    const uint8_t* srow = src + (long long)blockIdx.z * sbatch + (long long)y * spitch + xb;
    uint8_t* drow = dst + (long long)blockIdx.z * dbatch + (long long)y * dpitch + xb;
    const bool full = xb + 4 <= w;
    uint32_t in = 0;
    if (full && (reinterpret_cast<uintptr_t>(srow) & 3) == 0) {
        in = *reinterpret_cast<const uint32_t*>(srow);
    } else {
        for (int px = 0; px < 4 && xb + px < w; ++px) in |= (uint32_t)srow[px] << (8 * px);
    }
    // C.5, rows: tyf = y / th - 0.5, the tile rows above and below, and the weights
    const float tyf = __fsub_rn(__fmul_rn(__int2float_rn(y), inv_th), 0.5f);
    int ty1 = (int)floorf(tyf);
    const float ya = __fsub_rn(tyf, __int2float_rn(ty1)), ya1 = __fsub_rn(1.0f, ya);
    const int ty2 = min(ty1 + 1, tiles_y - 1);
    ty1 = max(ty1, 0);
    const uint8_t* L = lut + (long long)blockIdx.z * tiles_x * tiles_y * 256;
    const uint8_t* row1 = L + (long long)ty1 * tiles_x * 256;
    const uint8_t* row2 = L + (long long)ty2 * tiles_x * 256;
    uint32_t out = 0;
#pragma unroll
    for (int px = 0; px < 4; ++px) {
        const int x = xb + px;
        // past the row's end the tile index can exceed tiles_x - 1 (unpadded tiles of <= 4 pixels): load nothing there
        if (x >= w) break;
        const float txf = __fsub_rn(__fmul_rn(__int2float_rn(x), inv_tw), 0.5f);
        int tx1 = (int)floorf(txf);
        const float xa = __fsub_rn(txf, __int2float_rn(tx1)), xa1 = __fsub_rn(1.0f, xa);
        const int tx2 = min(tx1 + 1, tiles_x - 1);
        tx1 = max(tx1, 0);
        const int v = (in >> (8 * px)) & 0xff;
        const float top = __fadd_rn(__fmul_rn(lut_at(row1, tx1, v), xa1), __fmul_rn(lut_at(row1, tx2, v), xa));
        const float bot = __fadd_rn(__fmul_rn(lut_at(row2, tx1, v), xa1), __fmul_rn(lut_at(row2, tx2, v), xa));
        const float res = __fadd_rn(__fmul_rn(top, ya1), __fmul_rn(bot, ya));
        out |= (uint32_t)min(max(__float2int_rn(res), 0), 255) << (8 * px);
    }
    if (full && (reinterpret_cast<uintptr_t>(drow) & 3) == 0) {
        *reinterpret_cast<uint32_t*>(drow) = out;
    } else {
        for (int px = 0; px < 4 && xb + px < w; ++px) drow[px] = (uint8_t)(out >> (8 * px));
    }
}

}  // namespace

// C.1-C.3 on the host: padding, tile size, clip count and the float constants, with the checks of include/klt_b200.h.
klt_status clahe_plan(int w, int h, double clip_limit, int tiles_x, int tiles_y, ClahePlan* p)
{
    if (w < 1 || h < 1 || tiles_x < 1 || tiles_y < 1 || !std::isfinite(clip_limit)) return KLT_ERR_INVALID_ARG;
    if ((long long)tiles_x * tiles_y > KLT_MAX_CLAHE_TILES) return KLT_ERR_UNSUPPORTED;
    // OpenCV pads both axes when either does not divide: an axis that divides gets a whole extra tile then
    const bool pad = w % tiles_x != 0 || h % tiles_y != 0;
    const long long wext = pad ? (long long)w + tiles_x - w % tiles_x : w;
    const long long hext = pad ? (long long)h + tiles_y - h % tiles_y : h;
    const long long tw = wext / tiles_x, th = hext / tiles_y, total = tw * th;
    if (total > 2147483647LL) return KLT_ERR_UNSUPPORTED;   // cv2 counts a tile's pixels in an int
    int clip = 0;
    if (clip_limit > 0) {
        const double c = clip_limit * (double)total / 256;
        if (c >= 2147483648.0) return KLT_ERR_INVALID_ARG;   // int overflow in cv2 (undefined behaviour)
        clip = c < 1 ? 1 : (int)c;
    }
    p->tiles_x = tiles_x;
    p->tiles_y = tiles_y;
    p->tw = (int)tw;
    p->th = (int)th;
    p->clip = clip;
    p->lut_scale = 255.0f / (float)total;
    p->inv_tw = 1.0f / (float)tw;
    p->inv_th = 1.0f / (float)th;
    return KLT_OK;
}

long long clahe_lut_bytes(int batch, int tiles_x, int tiles_y) { return (long long)batch * tiles_x * tiles_y * 256; }

klt_status clahe_launch(const uint8_t* src, int w, int h, long long spitch, long long sbatch, uint8_t* dst, long long dpitch,
                        long long dbatch, int batch, const ClahePlan& p, uint8_t* lut, cudaStream_t stream)
{
    if (batch < 1 || (reinterpret_cast<uintptr_t>(lut) & 7) != 0) return KLT_ERR_INVALID_ARG;
    const dim3 agrid((w + 4 * kBX - 1) / (4 * kBX), (h + kBY - 1) / kBY, batch);
    if (batch > 65535 || agrid.y > 65535) return KLT_ERR_UNSUPPORTED;
    clahe_lut_kernel<<<dim3(p.tiles_x * p.tiles_y, batch), kLutThreads, 0, stream>>>(src, w, h, spitch, sbatch, p.tiles_x, p.tw, p.th,
                                                                                     p.clip, p.lut_scale, lut);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return (klt_status)e;
    clahe_apply_kernel<<<agrid, dim3(kBX, kBY), 0, stream>>>(src, w, h, spitch, sbatch, dst, dpitch, dbatch, p.tiles_x, p.tiles_y,
                                                             p.inv_tw, p.inv_th, lut);
    e = cudaGetLastError();
    return e == cudaSuccess ? KLT_OK : (klt_status)e;
}

}  // namespace klt
