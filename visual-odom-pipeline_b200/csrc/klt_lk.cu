// K4: fused Scharr-derivative + pyramidal Lucas-Kanade solver for sm_100a, one warp per keypoint.
//
// Replaces, per point, everything cv2.calcOpticalFlowPyrLK does after the pyramids exist
// (calcScharrDeriv + LKTrackerInvoker for every level), i.e. what the reference runs at
// src/extractor/extractor.py:44,45,65,66.  Arithmetic follows SURVEY.md Appendix A.3-A.6 exactly:
// int16 Scharr derivatives (zero outside the image), Q14 bilinear weights, Q5 intensity patch,
// float32 G / b sums in OpenCV's SIMD128 accumulation order (A.5), float32 2x2 solve without FMA
// contraction, double eps test, min-eigenvalue gate, level-0 status / err semantics.
//
// Design:
//  * ONE launch for all pyramid levels: a warp walks its point coarse -> fine, so there is no
//    inter-level launch or global round trip (cv2 runs a parallel_for per level).
//  * Per level the warp stages the (win+3)^2 u8 neighbourhood of the previous image and a
//    (win+1+2M)^2 neighbourhood of the next image in shared memory (REFLECT_101 resolved during
//    staging, so pyramid levels need no border copies and the inner loops have no bounds checks);
//    the next-image region is re-staged only when the iterate leaves its margin M.
//  * Scharr derivatives are computed on the fly from the staged u8 patch (never materialised in
//    HBM), masked to zero outside the image.
//  * The patch / G / mismatch passes are split into "units" of 8 consecutive window pixels of one
//    row, matching OpenCV's 8-pixel SIMD step, so a lane's pixels fall into fixed accumulation
//    classes (4 SIMD lanes + scalar tail).  Class sums are accumulated as exact integers and
//    reduced with warp shuffles; if every class satisfies sum|v| <= 2^24 the float32 accumulation
//    OpenCV performs is exact and equals the integer sum, otherwise (rare: <1% of mismatch passes
//    on textured frames) the warp replays that sum serially in OpenCV's order (bit-exactness).
//  * The per-point scalar arithmetic is shared with the specialised kernel (klt_lk_point.cuh).
#include "klt_lk_point.cuh"

#include <math_constants.h>

namespace klt {

namespace {

constexpr int kLKWarps = 4;   // warps (= points) per CTA, fewer when kLKWarps slices of the window's footprint do not fit
constexpr int kMargin = 3;    // extra pixels staged around the next-image window

struct LKGeom {
    int win_w, win_h;
    int g8;        // 8-pixel units per window row (last one may be the scalar tail)
    int nv;        // 8 * (win_w / 8): width handled by OpenCV's SIMD loop
    int tl;        // win_w - nv: scalar tail length
    int pw;        // 8 * g8: padded patch row width (pixels)
    int nu;        // win_h * g8 units
    unsigned g8_magic;
    int r8;        // 8-position runs per derivative row
    int nruns;     // (win_h + 1) * r8
    unsigned r8_magic;
    int si;        // I-region row stride (bytes)
    int sd;        // derivative-region row stride (words)
    int sj;        // J-region row stride (bytes)
    int jr_w, jr_h;  // J-region logical size
    int off_ipatch, off_dpatch, off_jreg, off_scratch, off_dreg;  // byte offsets in the warp slice
    int warp_bytes;
};

__host__ inline int round_up(int v, int a) { return (v + a - 1) / a * a; }

__host__ LKGeom make_geom(int win_w, int win_h)
{
    LKGeom g{};
    g.win_w = win_w; g.win_h = win_h;
    g.g8 = (win_w + 7) / 8;
    g.nv = 8 * (win_w / 8);
    g.tl = win_w - g.nv;
    g.pw = 8 * g.g8;
    g.nu = win_h * g.g8;
    g.g8_magic = fastdiv_magic((unsigned)g.g8);
    g.r8 = (win_w + 1 + 7) / 8;
    g.nruns = (win_h + 1) * g.r8;
    g.r8_magic = fastdiv_magic((unsigned)g.r8);
    g.si = g.pw + 12;
    g.sd = g.pw + 1;
    g.jr_w = win_w + 1 + 2 * kMargin;
    g.jr_h = win_h + 1 + 2 * kMargin;
    g.sj = round_up(g.pw + 2 * kMargin + 2, 4);
    int off = 0;
    g.off_ipatch = off; off += round_up(2 * g.pw * win_h, 16);
    g.off_dpatch = off; off += round_up(4 * g.pw * win_h, 16);
    g.off_jreg = off;   off += round_up(g.sj * g.jr_h, 16);
    g.off_scratch = off;
    const int ireg = round_up(g.si * (win_h + 3), 16);
    const int dreg = round_up(4 * g.sd * (win_h + 1), 16);
    const int diff = round_up(2 * g.pw * win_h, 16);
    g.off_dreg = off + ireg;
    off += (ireg + dreg > diff) ? ireg + dreg : diff;
    g.warp_bytes = round_up(off, 128);
    return g;
}

// Stage a rows x cols u8 region whose top-left image coordinate is (x0, y0) into smem (row stride
// `stride`), resolving REFLECT_101.  8 columns x 4 rows per warp instruction.
__device__ __forceinline__ void stage_region(uint8_t* __restrict__ dst, int stride, const LevelView& lv,
                                             const uint8_t* __restrict__ img, int x0, int y0, int rows,
                                             int cols, int lane)
{
    const int lc = lane & 7, lr = lane >> 3;
    const bool inside = (x0 >= 0) && (y0 >= 0) && (x0 + cols <= lv.w) && (y0 + rows <= lv.h);
    if (inside) {  // warp-uniform fast path: no reflection
        const uint8_t* __restrict__ base = img + (long long)y0 * lv.pitch + x0;
        for (int r = lr; r < rows; r += 4) {
            const uint8_t* __restrict__ rp = base + (long long)r * lv.pitch;
            for (int c = lc; c < cols; c += 8) dst[r * stride + c] = __ldg(rp + c);
        }
    } else {
        for (int r = lr; r < rows; r += 4) {
            const uint8_t* __restrict__ rp = img + (long long)reflect101(y0 + r, lv.h) * lv.pitch;
            for (int c = lc; c < cols; c += 8) dst[r * stride + c] = __ldg(rp + reflect101(x0 + c, lv.w));
        }
    }
}

// Reduce 16 per-lane integers over the warp; afterwards every lane holds all 16 totals.
__device__ __forceinline__ void warp_sum16(int (&v)[16], int lane)
{
#pragma unroll
    for (int half = 8, m = 16; half >= 1; half >>= 1, m >>= 1) {
        const bool up = (lane & m) != 0;
#pragma unroll
        for (int i = 0; i < half; ++i) {
            const int send = up ? v[i] : v[i + half];
            const int keep = up ? v[i + half] : v[i];
            v[i] = keep + __shfl_xor_sync(kFull, send, m);
        }
    }
    v[0] += __shfl_xor_sync(kFull, v[0], 1);
    const int mine = v[0];  // total of value index (lane >> 1)
#pragma unroll
    for (int k = 0; k < 16; ++k) v[k] = __shfl_sync(kFull, mine, 2 * k);
}

struct WarpCtx {
    const LKGeom* g;
    short* ipatch;        // [win_h][pw] Q5 intensity of the prev window
    uint32_t* dpatch;     // [win_h][pw] packed (gx | gy << 16)
    uint8_t* jreg;        // staged next-image region
    uint8_t* ireg;        // staged prev-image region (scratch)
    uint32_t* dreg;       // derivative at the (win+1)^2 integer positions (scratch)
    short* diff;          // [win_h][pw] last mismatch image (scratch, aliases ireg/dreg)
    int lane;
};

// ---- derivative pass: Scharr at every integer position the bilinear patch touches --------------
__device__ __forceinline__ void scharr_pass(const WarpCtx& c, int ipx, int ipy, int lw, int lh)
{
    const LKGeom& g = *c.g;
    for (int u = c.lane; u < g.nruns; u += 32) {
        const int dy = (int)fastdiv((unsigned)u, g.r8_magic);
        const int dx0 = 8 * (u - dy * g.r8);
        const uint8_t* r0 = c.ireg + dy * g.si + dx0;
        const uint8_t* r1 = r0 + g.si;
        const uint8_t* r2 = r1 + g.si;
        int t0[10], t1[10];
#pragma unroll
        for (int k = 0; k < 10; ++k) {
            const int a = r0[k], b = r1[k], cc = r2[k];
            t0[k] = 3 * (a + cc) + 10 * b;
            t1[k] = cc - a;
        }
        const bool yin = (unsigned)(ipy + dy) < (unsigned)lh;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int dx = dx0 + k;
            const int gx = t0[k + 2] - t0[k];
            const int gy = 3 * (t1[k] + t1[k + 2]) + 10 * t1[k + 1];
            const bool in = yin && ((unsigned)(ipx + dx) < (unsigned)lw);
            const uint32_t packed = in ? (((uint32_t)gx & 0xffffu) | ((uint32_t)gy << 16)) : 0u;
            if (dx < g.sd) c.dreg[dy * g.sd + dx] = packed;
        }
    }
}

// ---- patch pass: Q5 intensity + Q14 derivative patch, integer class sums of G -------------------
// vals[0..4] = sum gx*gx per class (4 SIMD lanes, tail), [5..9] = gx*gy, [10..14] = gy*gy
__device__ __forceinline__ void patch_pass(const WarpCtx& c, int w00, int w01, int w10, int w11, int (&vals)[16])
{
    const LKGeom& g = *c.g;
    unsigned q11[4] = {0, 0, 0, 0}, q22[4] = {0, 0, 0, 0}, t11 = 0, t22 = 0;
    int q12[4] = {0, 0, 0, 0}, t12 = 0;
    for (int u = c.lane; u < g.nu; u += 32) {
        const int y = (int)fastdiv((unsigned)u, g.g8_magic);
        const int gi = u - y * g.g8;
        const int x0 = 8 * gi;
        const uint8_t* i0 = c.ireg + (y + 1) * g.si + x0 + 1;
        const uint8_t* i1 = i0 + g.si;
        const uint32_t* d0 = c.dreg + y * g.sd + x0;
        const uint32_t* d1 = d0 + g.sd;
        int pa0 = i0[0], pa1 = i1[0];
        uint32_t pd0 = d0[0], pd1 = d1[0];
        unsigned u11[4] = {0, 0, 0, 0}, u22[4] = {0, 0, 0, 0};
        int u12[4] = {0, 0, 0, 0};
        uint32_t ip[4], dp[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int a0 = i0[j + 1], a1 = i1[j + 1];
            const uint32_t e0 = d0[j + 1], e1 = d1[j + 1];
            int iv = (pa0 * w00 + a0 * w01 + pa1 * w10 + a1 * w11 + (1 << 8)) >> 9;
            int gx = (lo16(pd0) * w00 + lo16(e0) * w01 + lo16(pd1) * w10 + lo16(e1) * w11 + (1 << 13)) >> 14;
            int gy = (hi16(pd0) * w00 + hi16(e0) * w01 + hi16(pd1) * w10 + hi16(e1) * w11 + (1 << 13)) >> 14;
            const bool valid = (x0 + j) < g.win_w;
            iv = valid ? iv : 0; gx = valid ? gx : 0; gy = valid ? gy : 0;
            u11[j & 3] += (unsigned)(gx * gx);
            u12[j & 3] += gx * gy;
            u22[j & 3] += (unsigned)(gy * gy);
            if (j & 1) ip[j >> 1] |= (uint32_t)iv << 16; else ip[j >> 1] = (uint32_t)iv & 0xffffu;
            dp[j] = ((uint32_t)gx & 0xffffu) | ((uint32_t)gy << 16);
            pa0 = a0; pa1 = a1; pd0 = e0; pd1 = e1;
        }
        *reinterpret_cast<uint4*>(c.ipatch + y * g.pw + x0) = make_uint4(ip[0], ip[1], ip[2], ip[3]);
        uint4* dpp = reinterpret_cast<uint4*>(c.dpatch + y * g.pw + x0);
        dpp[0] = make_uint4(dp[0], dp[1], dp[2], dp[3]);
        dpp[1] = make_uint4(dp[4], dp[5], dp[6], dp[7]);
        const bool tail = (x0 >= g.nv);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            q11[k] += tail ? 0u : u11[k];
            q12[k] += tail ? 0 : u12[k];
            q22[k] += tail ? 0u : u22[k];
        }
        t11 += tail ? (u11[0] + u11[1] + u11[2] + u11[3]) : 0u;
        t12 += tail ? (u12[0] + u12[1] + u12[2] + u12[3]) : 0;
        t22 += tail ? (u22[0] + u22[1] + u22[2] + u22[3]) : 0u;
    }
    // clamp so that 32-lane totals cannot wrap; any clamped value already proves "inexact"
    const unsigned cap = 1u << 25;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        vals[k] = (int)min(q11[k], cap);
        vals[5 + k] = max(min(q12[k], (int)cap), -(int)cap);
        vals[10 + k] = (int)min(q22[k], cap);
    }
    vals[4] = (int)min(t11, cap);
    vals[9] = max(min(t12, (int)cap), -(int)cap);
    vals[14] = (int)min(t22, cap);
    vals[15] = 0;
}

// serial replay of the G sums in OpenCV's accumulation order (A.5); lanes 0..14 = 3 sums x 5 chains
__device__ __forceinline__ void g_chain_fallback(const WarpCtx& c, float& A11, float& A12, float& A22)
{
    const LKGeom& g = *c.g;
    const int s = c.lane / 5, k = c.lane - 5 * s;
    const int per_row = (k < 4) ? g.nv / 4 : g.tl;
    const int steps = max(g.nv / 4, g.tl);
    float acc = 0.f;
    for (int y = 0; y < g.win_h; ++y) {
        const uint32_t* row = c.dpatch + y * g.pw;
        for (int st = 0; st < steps; ++st) {
            if (c.lane < 15 && st < per_row) {
                const int x = (k < 4) ? (k + 4 * st) : (g.nv + st);
                const uint32_t wd = row[x];
                const int gx = lo16(wd), gy = hi16(wd);
                const int prod = (s == 0) ? gx * gx : ((s == 1) ? gx * gy : gy * gy);
                acc = __fadd_rn(acc, (float)prod);
            }
        }
    }
    float r[3];
#pragma unroll
    for (int ss = 0; ss < 3; ++ss) {
        const float q0 = __shfl_sync(kFull, acc, 5 * ss + 0), q1 = __shfl_sync(kFull, acc, 5 * ss + 1);
        const float q2 = __shfl_sync(kFull, acc, 5 * ss + 2), q3 = __shfl_sync(kFull, acc, 5 * ss + 3);
        const float t = __shfl_sync(kFull, acc, 5 * ss + 4);
        r[ss] = combine5(q0, q1, q2, q3, t);
    }
    A11 = r[0]; A12 = r[1]; A22 = r[2];
}

// ---- mismatch pass: diff = bilinear(J) - Ipatch; integer class sums of diff*gx, diff*gy ----------
// vals[0..4] = sum d*gx per class, [5..9] = d*gy, [10..14] = ceil-ish(sum |d|(|gx|+|gy|) / 16)
// ERR mode: vals[0] = sum |d| only.
template <bool ERR>
__device__ __forceinline__ void mismatch_pass(const WarpCtx& c, int ry0, int cx0, int w00, int w01, int w10,
                                              int w11, int (&vals)[16])
{
    const LKGeom& g = *c.g;
    int s1[4] = {0, 0, 0, 0}, s2[4] = {0, 0, 0, 0}, t1 = 0, t2 = 0;
    unsigned bq[4] = {0, 0, 0, 0}, bt = 0;
    int esum = 0;
    for (int u = c.lane; u < g.nu; u += 32) {
        const int y = (int)fastdiv((unsigned)u, g.g8_magic);
        const int gi = u - y * g.g8;
        const int x0 = 8 * gi;
        const uint8_t* j0 = c.jreg + (ry0 + y) * g.sj + cx0 + x0;
        const uint8_t* j1 = j0 + g.sj;
        const uint4 iq = *reinterpret_cast<const uint4*>(c.ipatch + y * g.pw + x0);
        const uint32_t ipk[4] = {iq.x, iq.y, iq.z, iq.w};
        uint32_t dpk[8];
        if (!ERR) {
            const uint4* dpp = reinterpret_cast<const uint4*>(c.dpatch + y * g.pw + x0);
            const uint4 da = dpp[0], db = dpp[1];
            dpk[0] = da.x; dpk[1] = da.y; dpk[2] = da.z; dpk[3] = da.w;
            dpk[4] = db.x; dpk[5] = db.y; dpk[6] = db.z; dpk[7] = db.w;
        }
        int pb0 = j0[0], pb1 = j1[0];
        int v1[4] = {0, 0, 0, 0}, v2[4] = {0, 0, 0, 0};
        unsigned vb[4] = {0, 0, 0, 0};
        uint32_t dk[4];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int b0 = j0[j + 1], b1 = j1[j + 1];
            const int jv = (pb0 * w00 + b0 * w01 + pb1 * w10 + b1 * w11 + (1 << 8)) >> 9;
            const int iv = (j & 1) ? hi16(ipk[j >> 1]) : lo16(ipk[j >> 1]);
            int d = jv - iv;
            d = ((x0 + j) < g.win_w) ? d : 0;
            if (ERR) {
                esum += abs(d);
            } else {
                const int gx = lo16(dpk[j]), gy = hi16(dpk[j]);
                v1[j & 3] += d * gx;
                v2[j & 3] += d * gy;
                vb[j & 3] += ((unsigned)(abs(d) * (abs(gx) + abs(gy))) + 15u) >> 4;
                if (j & 1) dk[j >> 1] |= (uint32_t)d << 16; else dk[j >> 1] = (uint32_t)d & 0xffffu;
            }
            pb0 = b0; pb1 = b1;
        }
        if (!ERR) {
            *reinterpret_cast<uint4*>(c.diff + y * g.pw + x0) = make_uint4(dk[0], dk[1], dk[2], dk[3]);
            const bool tail = (x0 >= g.nv);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                s1[k] += tail ? 0 : v1[k];
                s2[k] += tail ? 0 : v2[k];
                bq[k] += tail ? 0u : vb[k];
            }
            t1 += tail ? (v1[0] + v1[1] + v1[2] + v1[3]) : 0;
            t2 += tail ? (v2[0] + v2[1] + v2[2] + v2[3]) : 0;
            bt += tail ? (vb[0] + vb[1] + vb[2] + vb[3]) : 0u;
        }
    }
    if (ERR) {
        vals[0] = esum;
    } else {
        const unsigned cap = 1u << 22;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            vals[k] = s1[k];
            vals[5 + k] = s2[k];
            vals[10 + k] = (int)min(bq[k], cap);
        }
        vals[4] = t1; vals[9] = t2; vals[14] = (int)min(bt, cap);
        vals[15] = 0;
    }
}

// serial replay of the b sums in OpenCV's order (pairs (l, l+4) summed in int32 first; A.5)
__device__ __forceinline__ void b_chain_fallback(const WarpCtx& c, float& b1, float& b2)
{
    const LKGeom& g = *c.g;
    const int s = c.lane / 5, k = c.lane - 5 * s;
    const int per_row = (k < 4) ? g.nv / 8 : g.tl;
    const int steps = max(g.nv / 8, g.tl);
    float acc = 0.f;
    for (int y = 0; y < g.win_h; ++y) {
        const uint32_t* drow = c.dpatch + y * g.pw;
        const short* frow = c.diff + y * g.pw;
        for (int st = 0; st < steps; ++st) {
            if (c.lane < 10 && st < per_row) {
                int v;
                if (k < 4) {
                    const int xa = 8 * st + k, xb = xa + 4;
                    const uint32_t wa = drow[xa], wb = drow[xb];
                    const int ga = s ? hi16(wa) : lo16(wa), gb = s ? hi16(wb) : lo16(wb);
                    v = (int)frow[xa] * ga + (int)frow[xb] * gb;
                } else {
                    const int x = g.nv + st;
                    const uint32_t wa = drow[x];
                    v = (int)frow[x] * (s ? hi16(wa) : lo16(wa));
                }
                acc = __fadd_rn(acc, (float)v);
            }
        }
    }
    float r[2];
#pragma unroll
    for (int ss = 0; ss < 2; ++ss) {
        const float q0 = __shfl_sync(kFull, acc, 5 * ss + 0), q1 = __shfl_sync(kFull, acc, 5 * ss + 1);
        const float q2 = __shfl_sync(kFull, acc, 5 * ss + 2), q3 = __shfl_sync(kFull, acc, 5 * ss + 3);
        const float t = __shfl_sync(kFull, acc, 5 * ss + 4);
        r[ss] = combine5(q0, q1, q2, q3, t);
    }
    b1 = r[0]; b2 = r[1];
}

// kFullCTA: the CTA has kLKWarps warps, else the warp count is read from the launch.  A run-time warp count in every
// launch would cost spills (36 bytes instead of 12 at 72 registers), so the common launch keeps the constant.
template <bool kFullCTA>
__global__ void __launch_bounds__(kLKWarps * 32)
lk_kernel(const __grid_constant__ LKLaunch L, const __grid_constant__ LKGeom G)
{
    extern __shared__ __align__(128) uint8_t smem[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const long long gid = (long long)blockIdx.x * (kFullCTA ? kLKWarps : (int)(blockDim.x >> 5)) + warp;
    const long long total = (long long)L.n_per_pair * L.batch;
    if (gid >= total) return;  // warp-uniform; no block-level barriers below
    const int b = (int)(gid / L.n_per_pair);
    // past this pair's point count (warp-uniform); the index within the pair is exact in 32-bit unsigned arithmetic
    if (L.counts && (int)((unsigned)gid - (unsigned)b * (unsigned)L.n_per_pair) >= __ldg(L.counts + b)) return;

    uint8_t* ws = smem + warp * G.warp_bytes;
    WarpCtx c;
    c.g = &G;
    c.ipatch = reinterpret_cast<short*>(ws + G.off_ipatch);
    c.dpatch = reinterpret_cast<uint32_t*>(ws + G.off_dpatch);
    c.jreg = ws + G.off_jreg;
    c.ireg = ws + G.off_scratch;
    c.dreg = reinterpret_cast<uint32_t*>(ws + G.off_dreg);
    c.diff = reinterpret_cast<short*>(ws + G.off_scratch);
    c.lane = lane;

    const float2 p0 = reinterpret_cast<const float2*>(L.prev_pts)[gid];
    float2 outp = make_float2(0.f, 0.f);
    if (L.flags & KLT_OPTFLOW_USE_INITIAL_FLOW) outp = reinterpret_cast<const float2*>(L.next_pts)[gid];
    int status = 1;
    float err = 0.f;
    int iters = 0;

    const float hwx = (float)(G.win_w - 1) * 0.5f, hwy = (float)(G.win_h - 1) * 0.5f;
    const int top = L.prev.top;

    for (int level = top; level >= 0; --level) {
        const LevelView lvI = L.prev.lv[level];
        const LevelView lvJ = L.next.lv[level];
        const uint8_t* __restrict__ imgI = lvI.data + (long long)b * lvI.batch_stride;
        const uint8_t* __restrict__ imgJ = lvJ.data + (long long)b * lvJ.batch_stride;
        const int lw = lvI.w, lh = lvI.h;

        // A.4 step 1
        float px, py, nx, ny;
        level_start(p0, outp, level, top, L.flags, px, py, nx, ny);

        // step 2
        px = __fsub_rn(px, hwx); py = __fsub_rn(py, hwy);
        int ipx, ipy;
        if (!floor_in_range(px, py, G.win_w, G.win_h, lw, lh, ipx, ipy)) {
            if (level == 0) { status = 0; err = 0.f; }
            continue;
        }
        int w00, w01, w10, w11;
        q14_weights(__fsub_rn(px, (float)ipx), __fsub_rn(py, (float)ipy), w00, w01, w10, w11);

        // stage both neighbourhoods (the next-image one speculatively at the initial guess)
        nx = __fsub_rn(nx, hwx); ny = __fsub_rn(ny, hwy);
        int jx0 = 0, jy0 = 0;
        bool jvalid = false;
        {
            int inx, iny;
            if (floor_in_range(nx, ny, G.win_w, G.win_h, lw, lh, inx, iny)) {
                jx0 = inx - kMargin; jy0 = iny - kMargin; jvalid = true;
                stage_region(c.jreg, G.sj, lvJ, imgJ, jx0, jy0, G.jr_h, G.jr_w, lane);
            }
        }
        stage_region(c.ireg, G.si, lvI, imgI, ipx - 1, ipy - 1, G.win_h + 3, G.win_w + 3, lane);
        __syncwarp();
        scharr_pass(c, ipx, ipy, lw, lh);
        __syncwarp();

        // steps 4 + 5
        int vals[16];
        patch_pass(c, w00, w01, w10, w11, vals);
        warp_sum16(vals, lane);
        __syncwarp();  // patches visible; ireg/dreg are dead from here (diff aliases them)
        float A11, A12, A22;
        {
            bool exact = true;
#pragma unroll
            for (int k = 0; k < 5; ++k) exact = exact && ((unsigned)vals[k] + (unsigned)vals[10 + k] <= (unsigned)kExact);
            if (exact) {
                A11 = combine5((float)vals[0], (float)vals[1], (float)vals[2], (float)vals[3], (float)vals[4]);
                A12 = combine5((float)vals[5], (float)vals[6], (float)vals[7], (float)vals[8], (float)vals[9]);
                A22 = combine5((float)vals[10], (float)vals[11], (float)vals[12], (float)vals[13], (float)vals[14]);
            } else {
                g_chain_fallback(c, A11, A12, A22);
            }
        }
        float D;
        if (!eig_gate(A11, A12, A22, G.win_w, G.win_h, L.flags, L.min_eig_thr, err, D)) {
            if (level == 0) status = 0;
            continue;
        }

        // step 6
        float pdx = 0.f, pdy = 0.f;
        for (int j = 0; j < L.max_count; ++j) {
            int inx, iny;
            if (!floor_in_range(nx, ny, G.win_w, G.win_h, lw, lh, inx, iny)) {
                if (level == 0) status = 0;
                break;
            }
            ++iters;
            if (!jvalid || inx < jx0 || iny < jy0 || inx + G.win_w + 1 > jx0 + G.jr_w || iny + G.win_h + 1 > jy0 + G.jr_h) {
                __syncwarp();
                jx0 = inx - kMargin; jy0 = iny - kMargin; jvalid = true;
                stage_region(c.jreg, G.sj, lvJ, imgJ, jx0, jy0, G.jr_h, G.jr_w, lane);
                __syncwarp();
            }
            q14_weights(__fsub_rn(nx, (float)inx), __fsub_rn(ny, (float)iny), w00, w01, w10, w11);
            mismatch_pass<false>(c, iny - jy0, inx - jx0, w00, w01, w10, w11, vals);
            warp_sum16(vals, lane);
            float b1, b2;
            {
                bool exact = true;
#pragma unroll
                for (int k = 0; k < 5; ++k) exact = exact && (vals[10 + k] <= (kExact >> 4));
                if (exact) {
                    b1 = combine5((float)vals[0], (float)vals[1], (float)vals[2], (float)vals[3], (float)vals[4]);
                    b2 = combine5((float)vals[5], (float)vals[6], (float)vals[7], (float)vals[8], (float)vals[9]);
                } else {
                    __syncwarp();
                    b_chain_fallback(c, b1, b2);
                    __syncwarp();
                }
            }
            if (newton_step(A11, A12, A22, D, b1, b2, j, L.eps2_lo, L.eps2_hi, L.eps2, hwx, hwy, nx, ny, pdx, pdy, outp)) break;
        }

        // step 7
        if (status && level == 0 && (L.flags & KLT_OPTFLOW_LK_GET_MIN_EIGENVALS) == 0) {
            const float qx = __fsub_rn(outp.x, hwx), qy = __fsub_rn(outp.y, hwy);
            int iqx, iqy;
            if (!floor_in_range(qx, qy, G.win_w, G.win_h, lw, lh, iqx, iqy)) {
                status = 0;
                continue;
            }
            if (!jvalid || iqx < jx0 || iqy < jy0 || iqx + G.win_w + 1 > jx0 + G.jr_w || iqy + G.win_h + 1 > jy0 + G.jr_h) {
                __syncwarp();
                jx0 = iqx - kMargin; jy0 = iqy - kMargin; jvalid = true;
                stage_region(c.jreg, G.sj, lvJ, imgJ, jx0, jy0, G.jr_h, G.jr_w, lane);
                __syncwarp();
            }
            q14_weights(__fsub_rn(qx, (float)iqx), __fsub_rn(qy, (float)iqy), w00, w01, w10, w11);
            mismatch_pass<true>(c, iqy - jy0, iqx - jx0, w00, w01, w10, w11, vals);
            int e = vals[0];
#pragma unroll
            for (int m = 16; m >= 1; m >>= 1) e += __shfl_xor_sync(kFull, e, m);
            // |diff| <= 8160 and win area <= 4096: e < 2^25 fits; the float32 running sum OpenCV keeps is
            // exact (hence order-free) while e <= 2^24, i.e. always for win area <= 2056.
            float ef;
            if (e <= kExact) {
                ef = (float)e;
            } else {  // replay row-major in float32 (never reached for win <= 45x45)
                __syncwarp();
                // recompute diffs into the scratch buffer through the non-ERR pass, then sum serially
                int tmp[16];
                mismatch_pass<false>(c, iqy - jy0, iqx - jx0, w00, w01, w10, w11, tmp);
                __syncwarp();
                ef = 0.f;
                for (int y = 0; y < G.win_h; ++y)
                    for (int x = 0; x < G.win_w; ++x) ef = __fadd_rn(ef, fabsf((float)c.diff[y * G.pw + x]));
                __syncwarp();
            }
            err = lk_err(ef, G.win_w, G.win_h);
        }
        __syncwarp();
    }

    if (lane == 0) {
        reinterpret_cast<float2*>(L.next_pts)[gid] = outp;
        L.status[gid] = (uint8_t)status;
        L.err[gid] = err;
        if (L.iters) L.iters[gid] = iters;
    }
}

int g_max_smem_optin = 0;

}  // namespace

klt_status lk_init(int device)
{
    int v = 0;
    cudaError_t e = cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
    if (e != cudaSuccess) return (klt_status)e;
    g_max_smem_optin = v;
    e = cudaFuncSetAttribute(lk_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, v);
    if (e != cudaSuccess) return (klt_status)e;
    e = cudaFuncSetAttribute(lk_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, v);
    if (e != cudaSuccess) return (klt_status)e;
    // the 12.20 reciprocal must be exact over the ranges the kernel uses
    for (unsigned d = 1; d <= 64; ++d)
        for (unsigned u = 0; u < 4096; ++u)
            if (fastdiv(u, fastdiv_magic(d)) != u / d) return KLT_ERR_INTERNAL;
    return KLT_OK;
}

klt_status lk_launch(const LKLaunch& L, int sm_count, cudaStream_t stream)
{
    if (L.win_w <= 2 || L.win_h <= 2) return KLT_ERR_INVALID_ARG;
    {   // specialised kernels for the common windows
        const klt_status s = lk_launch_fast(L, sm_count, stream);
        if (s != KLT_ERR_UNSUPPORTED) return s;
    }
    if ((long long)L.win_w * L.win_h > KLT_MAX_WIN_AREA || L.win_w > KLT_MAX_WIN_SIDE || L.win_h > KLT_MAX_WIN_SIDE)
        return KLT_ERR_UNSUPPORTED;
    const LKGeom G = make_geom(L.win_w, L.win_h);
    if (G.nu >= 4096 || G.nruns >= 4096 || G.g8 > 64 || G.r8 > 64) return KLT_ERR_UNSUPPORTED;
    const long long total = (long long)L.n_per_pair * L.batch;
    if (total <= 0) return KLT_OK;
    // as many warps per CTA as the opt-in shared memory holds: a large window's slice (up to 114 KB) leaves room for fewer
    // than kLKWarps (on a B200, with 227 KB, every supported window fits at least two)
    int warps = kLKWarps;
    while (warps > 1 && (long long)G.warp_bytes * warps > g_max_smem_optin) --warps;
    const size_t smem = (size_t)G.warp_bytes * warps;
    if ((long long)smem > g_max_smem_optin) return KLT_ERR_UNSUPPORTED;
    const long long blocks = (total + warps - 1) / warps;
    if (blocks > 0x7fffffffLL) return KLT_ERR_UNSUPPORTED;
    if (warps == kLKWarps) lk_kernel<true><<<(unsigned)blocks, warps * 32, smem, stream>>>(L, G);
    else lk_kernel<false><<<(unsigned)blocks, warps * 32, smem, stream>>>(L, G);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KLT_OK : (klt_status)e;
}

}  // namespace klt
