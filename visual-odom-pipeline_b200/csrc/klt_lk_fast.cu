// K4 (specialised): fused Scharr + pyramidal LK for compile-time window sizes, WPP warps per point.
//
// Same arithmetic as klt_lk.cu (klt_lk_point.cuh; SURVEY.md A.3-A.6, bit-exact with cv2.calcOpticalFlowPyrLK as called
// at reference src/extractor/extractor.py:44,45,65,66); this variant is what the BASELINE configs
// (winSize 21 and 31) run.  Differences in structure:
//  * WPP in {2,4} warps cooperate on one keypoint (named barriers), so a 2000-point frame pair fills
//    the chip and the per-iteration latency of the slowest point -- which bounds the launch -- drops;
//    the launcher picks 4, or 2 for 21x21 launches that fill the chip more than once (lk_launch_fast).
//  * the window is cut into 4-pixel units; each thread keeps the Q5 intensity / Q14 derivative patch of
//    its units in registers for the whole level, only the next-image region lives in shared memory;
//  * bilinear taps use dp2a (two 14-bit weights x two u8 pixels per instruction, exact);
//  * neighbourhoods are staged with 32-bit loads (all loads in flight before the first store);
//  * the mismatch sums are reduced in three tiers: (0) if sum|d|*max(|gx|,|gy|) over the WHOLE window
//    is <= 2^24 every float32 partial sum OpenCV forms is an exact integer, so b = float(sum) and only
//    3 values cross the warp(s); (1) otherwise per-accumulation-class sums (4 SIMD lanes + tail) with
//    the same test per class; (2) otherwise a serial float32 replay in OpenCV's order.
#include "klt_lk_point.cuh"

namespace klt {

namespace {

constexpr int kThreads = 128;
constexpr int kM = 3;  // margin of the staged next-image region
constexpr int kTwoPass = 0x200;   // internal launch flag (klt_b200.h: the public flag bits end at 0x8)

#ifdef KLT_LK_PHASES
// diagnostics build (build.py --variant phases --extra -DKLT_LK_PHASES; scripts/lk_phases.py): cycles per phase of the
// iteration loop of ONE selected point, stamped by its warp 0
__device__ unsigned long long g_ph[16];
__device__ long long g_ph_gid = -1;
// ph_on is uniform over the warp (a per-lane condition makes the compiler split the lane's path off the warp's)
#define PH(i) do { if (ph_on) { const long long c_ = clock64(); if (lane == 0) atomicAdd(&g_ph[i], (unsigned long long)(c_ - ph_t)); ph_t = clock64(); } } while (0)
#define PH_COUNT(i) do { if (ph_on && lane == 0) atomicAdd(&g_ph[i], 1ull); } while (0)
#else
#define PH(i) do { } while (0)
#define PH_COUNT(i) do { } while (0)
#endif

__host__ __device__ constexpr int r4(int v) { return (v + 3) / 4 * 4; }
__host__ __device__ constexpr int r16(int v) { return (v + 15) / 16 * 16; }

// ---- serial float32 replay in OpenCV's accumulation order (SURVEY.md A.5) -------------------------------
// Scratch layout: one zero-padded row per accumulation chain (4 SIMD lanes with x % 4 == l, x < NV, then the scalar
// tail x >= NV), elements in OpenCV's visiting order.  Padding with zeros makes every chain the same length, so the
// replay loop has no bounds checks: adding +0.0f is an exact no-op (the accumulator is never -0).
template <int WW, int WH>
struct Chains {
    static constexpr int NV = 8 * (WW / 8), TL = WW - NV;
    static constexpr int OVER = 16;   // the chain loops request up to 4 groups of 4 words past the end of a chain (never used)
    // G scratch: 12 SIMD chains (3 sums x 4 lanes, one float product per pixel) of GQ4 floats, then 3 tail chains of
    // GT4 floats (zero padded to multiples of 4), OVER words, then 16 result words
    static constexpr int GQ = WH * (NV / 4), GT = WH * TL;
    static constexpr int GQ4 = (GQ + 3) / 4 * 4, GT4 = (GT + 3) / 4 * 4;
    static constexpr int G_RES = 12 * GQ4 + 3 * GT4 + OVER;
    static constexpr int G_WORDS = G_RES + 16;
    // b scratch: 8 SIMD chains (2 sums x 4 lanes) of int pairs (x, x+4) in visiting order, then 2 tail chains of floats
    // (zero padded), OVER words, then 12 result words: q[0..3] of b1, of b2, t of b1, of b2
    static constexpr int NS = NV / 8;                                // 8-pixel SIMD steps per window row
    static constexpr int SLEN = 2 * WH * NS;                         // ints per SIMD chain
    static constexpr int SLEN4 = (SLEN + 3) / 4 * 4;                 // chain stride (the odd pair of an odd chain is zero padded)
    static constexpr int TLEN = (WH * TL + 3) / 4 * 4;               // floats per tail chain (zero padded)
    static constexpr int B_RES = 8 * SLEN4 + 2 * TLEN + OVER;
    static constexpr int B_WORDS = (B_RES + 12 + 3) / 4 * 4;
};

template <int WW, int WH, int WPP>
struct Cfg {
    static constexpr int UPR = (WW + 3) / 4;          // 4-pixel units per window row
    static constexpr int NV = 8 * (WW / 8);           // width of OpenCV's SIMD part (A.5)
    static constexpr int TL = WW - NV;                // scalar tail
    static constexpr int NU = WH * UPR;
    static constexpr int NT = 32 * WPP;               // threads per point
    static constexpr int UPT = (NU + NT - 1) / NT;    // units per thread
    static constexpr int PPC = kThreads / NT;         // points per CTA
    static constexpr int SI = r4(WW + 6);             // prev-image region: row stride (bytes)
    static constexpr int IR = WH + 3;                 //                    rows
    static constexpr int SD = r4(WW + 2);             // derivative region: row stride (words)
    static constexpr int DR = WH + 1;
    static constexpr int JW = WW + 1 + 2 * kM;        // next-image region: logical size
    static constexpr int JR = WH + 1 + 2 * kM;
    static constexpr int SJ = r4(JW + 3);             //                    row stride (bytes)
    static constexpr int RPR = (WW + 1 + 3) / 4;      // Scharr: 4-position runs per row
    static constexpr int NRUN = DR * RPR;
    // shared-memory slice of one point (bytes)
    static constexpr int OFF_J = 0;
    static constexpr int OFF_D = OFF_J + r16(SJ * JR);        // dreg; fallback: packed derivative patch
    static constexpr int CHAIN_WORDS = r4(Chains<WW, WH>::B_WORDS > Chains<WW, WH>::G_WORDS ? Chains<WW, WH>::B_WORDS : Chains<WW, WH>::G_WORDS);   // replay scratch
    static constexpr int D_BYTES = r16(4 * (SD * DR > CHAIN_WORDS ? SD * DR : CHAIN_WORDS));  // dreg, or the replay chains
    static constexpr int OFF_I = OFF_D + D_BYTES;             // ireg
    static constexpr int I_BYTES = r16(SI * IR);
    static constexpr int NS = NV / 8;                         // 8-pixel SIMD steps per window row
    static constexpr int OFF_R3 = OFF_I + I_BYTES;            // [2][WPP] int4
    static constexpr int OFF_R16 = OFF_R3 + 2 * WPP * 16;     // [2][16 values][4 warps] int
    static constexpr int POINT_BYTES = (OFF_R16 + 2 * 256 + 127) / 128 * 128;
};

__device__ __forceinline__ int dp2a_lo(uint32_t w, uint32_t b, int c)
{
    int d;
    asm("dp2a.lo.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(w), "r"(b), "r"(c));
    return d;
}
__device__ __forceinline__ int dp2a_hi(uint32_t w, uint32_t b, int c)
{
    int d;
    asm("dp2a.hi.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(w), "r"(b), "r"(c));
    return d;
}
// Patch state of one window pixel, in registers for the whole level: Q5 intensity, Q14 derivative, gm = max(|gx|,|gy|)
struct Px {
    int iv, gx, gy, gm;
};

template <int WPP>
__device__ __forceinline__ void point_sync(int bar)
{
    asm volatile("bar.sync %0, %1;" ::"r"(bar), "n"(32 * WPP) : "memory");
}

// Stage ROWS x STRIDE bytes whose top-left image coordinate is (ax, y0) (ax % 4 == 0) into smem.  Columns
// [c0, c0 + need) of every row are the ones later read; the rest may hold anything.
template <int ROWS, int STRIDE, int NT>
__device__ __forceinline__ void stage(uint8_t* __restrict__ dst, const LevelView& lv, const uint8_t* __restrict__ img,
                                      int ax, int y0, int c0, int need, int tid)
{
    constexpr int NWR = STRIDE / 4;
    constexpr int NWORDS = ROWS * NWR;
    constexpr int PER = (NWORDS + NT - 1) / NT;
    // 32-bit loads whenever the staged columns lie inside the image; rows are reflected per row (REFLECT_101), which
    // is the common border case on the small coarse levels.  Only horizontal crossings take the byte path.
    const bool fast = lv.aligned4 && ax >= 0 && (ax + STRIDE <= lv.w);
    if (fast) {  // uniform over the point's threads
        const uint8_t* __restrict__ base = img + ax;
        const bool rows_inside = (y0 >= 0) && (y0 + ROWS <= lv.h);
        uint32_t v[PER];
#pragma unroll
        for (int k = 0; k < PER; ++k) {
            const int i = tid + k * NT;
            const int r = i / NWR, c = i - r * NWR;
            const int yy = rows_inside ? (y0 + r) : reflect101(y0 + r, lv.h);
            v[k] = (i < NWORDS) ? __ldg(reinterpret_cast<const uint32_t*>(base + (long long)yy * lv.pitch) + c) : 0u;
        }
#pragma unroll
        for (int k = 0; k < PER; ++k) {
            const int i = tid + k * NT;
            if (i < NWORDS) reinterpret_cast<uint32_t*>(dst)[i] = v[k];
        }
    } else {
        for (int i = tid; i < ROWS * need; i += NT) {
            const int r = i / need, c = c0 + (i - r * need);
            dst[r * STRIDE + c] = __ldg(img + (long long)reflect101(y0 + r, lv.h) * lv.pitch + reflect101(ax + c, lv.w));
        }
    }
}

// two words holding bytes [o, o+4) and [o+1, o+5) of an smem row (o = arbitrary byte offset)
__device__ __forceinline__ void load5(const uint8_t* row, int o, uint32_t& a, uint32_t& b)
{
    const uint32_t* wp = reinterpret_cast<const uint32_t*>(row) + (o >> 2);
    const uint32_t w0 = wp[0], w1 = wp[1];
    const int s = (o & 3) * 8;
    a = __funnelshift_r(w0, w1, s);
    b = __funnelshift_rc(w0, w1, s + 8);
}

// sum 3 values over all threads of the point; every thread gets the totals (REDUX + one smem exchange)
template <int WPP>
__device__ __forceinline__ void point_sum3(int& a, int& b, int& c, int4* red3, int& par3, int wip, int lane, int bar)
{
    a = __reduce_add_sync(kFull, a);
    b = __reduce_add_sync(kFull, b);
    c = __reduce_add_sync(kFull, c);
    int4* slot = red3 + par3 * WPP;
    if (lane == 0) slot[wip] = make_int4(a, b, c, 0);
    point_sync<WPP>(bar);
    a = 0; b = 0; c = 0;
#pragma unroll
    for (int w = 0; w < WPP; ++w) {
        const int4 v = slot[w];
        a += v.x; b += v.y; c += v.z;
    }
    par3 ^= 1;
}

// Sum 15 values over all threads of the point.  Returns, in lane L < 15 of EVERY warp, the point-wide total of
// value L (one REDUX per value, then one value-major smem exchange so a lane fetches its partials with one load).
template <int WPP>
__device__ __forceinline__ int point_sum15_lane(const int (&v)[16], int* red16, int& par16, int wip, int lane, int bar)
{
    int mine = 0;
#pragma unroll
    for (int i = 0; i < 15; ++i) {
        const int t = __reduce_add_sync(kFull, v[i]);
        mine = (lane == i) ? t : mine;
    }
    int* slot = red16 + par16 * 64;
    if (lane < 15) slot[lane * 4 + wip] = mine;
    point_sync<WPP>(bar);
    const int4 t = reinterpret_cast<const int4*>(slot)[lane & 15];
    mine = t.x + t.y + (WPP > 2 ? t.z + t.w : 0);
    par16 ^= 1;
    return mine;
}

// Serial float32 sum, in order, of one zero-padded chain of 4 * N4 floats.  The adds are one dependent chain (4 cycles
// each), so the loads must never be waited for: three groups of 4 are always in flight in rotating registers (the last
// requests read up to 3 groups past the chain -- the next chain or the OVER words -- and are dropped).
__device__ __forceinline__ float add4(float acc, const float4 v)
{
    return __fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(acc, v.x), v.y), v.z), v.w);
}
template <int N4>
__device__ __forceinline__ float chain_sum(const float* __restrict__ p)
{
    const float4* __restrict__ src = reinterpret_cast<const float4*>(p);
    constexpr int R = N4 / 3 * 3;
    float acc = 0.f;
    float4 a = src[0], b = src[1], c = src[2];
#pragma unroll 1
    for (int e = 0; e < R; e += 3) {
        acc = add4(acc, a); a = src[e + 3];
        acc = add4(acc, b); b = src[e + 4];
        acc = add4(acc, c); c = src[e + 5];
    }
    if constexpr (N4 - R >= 1) acc = add4(acc, a);
    if constexpr (N4 - R >= 2) acc = add4(acc, b);
    return acc;
}

// The same for a chain of 2 * N4 int pairs: each pair is summed in int32 and converted (off the dependent chain) before
// it is added; four groups of two pairs in flight.
__device__ __forceinline__ float add2p(float acc, const int4 v)
{
    return __fadd_rn(__fadd_rn(acc, (float)(v.x + v.y)), (float)(v.z + v.w));
}
template <int N4>
__device__ __forceinline__ float chain_sum_pairs(const int* __restrict__ p)
{
    const int4* __restrict__ src = reinterpret_cast<const int4*>(p);
    constexpr int R = N4 / 4 * 4;
    float acc = 0.f;
    int4 a = src[0], b = src[1], c = src[2], d = src[3];
#pragma unroll 1
    for (int e = 0; e < R; e += 4) {
        acc = add2p(acc, a); a = src[e + 4];
        acc = add2p(acc, b); b = src[e + 5];
        acc = add2p(acc, c); c = src[e + 6];
        acc = add2p(acc, d); d = src[e + 7];
    }
    if constexpr (N4 - R >= 1) acc = add2p(acc, a);
    if constexpr (N4 - R >= 2) acc = add2p(acc, b);
    if constexpr (N4 - R >= 3) acc = add2p(acc, c);
    return acc;
}

// G replay, split over the point's warps: warp 0 runs the 12 SIMD chains (lane = chain), warp 1 the 3 tail chains.
// The products were converted to float by the threads that own the pixels (|gx*gy| < 2^24: exact).
template <int WW, int WH>
__device__ __forceinline__ void replay_g(float* __restrict__ gf, int wip, int lane)
{
    using CH = Chains<WW, WH>;
    if (wip == 0) {
        const float acc = chain_sum<CH::GQ4 / 4>(gf + (lane < 12 ? lane : 0) * CH::GQ4);
        if (lane < 12) gf[CH::G_RES + (lane >> 2) * 5 + (lane & 3)] = acc;   // result layout: [sum][q0 q1 q2 q3 t]
    }
    if (wip == 1) {
        const float acc = chain_sum<CH::GT4 / 4>(gf + 12 * CH::GQ4 + (lane < 3 ? lane : 0) * CH::GT4);
        if (lane < 3) gf[CH::G_RES + lane * 5 + 4] = acc;
    }
}

// zero the padding of the chains of one b scratch buffer
template <int WW, int WH, int NT>
__device__ __forceinline__ void zero_pad_b(int* buf, int tid)
{
    using CH = Chains<WW, WH>;
    constexpr int PQ = CH::SLEN4 - CH::SLEN, PT = CH::TLEN - WH * CH::TL;
    static_assert(8 * PQ + 2 * PT <= NT, "one pad word per thread");
    if (tid < 8 * PQ) buf[(tid / (PQ > 0 ? PQ : 1)) * CH::SLEN4 + CH::SLEN + tid % (PQ > 0 ? PQ : 1)] = 0;
    else if (tid < 8 * PQ + 2 * PT) {
        const int t = tid - 8 * PQ;
        buf[8 * CH::SLEN4 + (t / (PT > 0 ? PT : 1)) * CH::TLEN + WH * CH::TL + t % (PT > 0 ? PT : 1)] = 0;
    }
}

// b replay, split over the point's warps: warp 0 runs the 8 SIMD chains (lane = chain; int pair -> float -> add), warp
// 1 the 2 tail chains (floats, converted by the threads that own the pixels).  Results go to buf[B_RES ..].
template <int WW, int WH>
__device__ __forceinline__ void replay_b(int* __restrict__ buf, int wip, int lane)
{
    using CH = Chains<WW, WH>;
    if (wip == 0) {
        const float acc = chain_sum_pairs<CH::SLEN4 / 4>(buf + (lane & 7) * CH::SLEN4);
        if (lane < 8) reinterpret_cast<float*>(buf)[CH::B_RES + lane] = acc;
    }
    if (wip == 1) {
        const float acc = chain_sum<CH::TLEN / 4>(reinterpret_cast<const float*>(buf) + 8 * CH::SLEN4 + (lane & 1) * CH::TLEN);
        if (lane < 2) reinterpret_cast<float*>(buf)[CH::B_RES + 8 + lane] = acc;
    }
}

// COUNTS: the launch carries per-pair point counts (LKLaunch::counts, the batched frame step).  A template parameter, so
// that the launches without counts run exactly the code they ran before the counts existed.
template <int WW, int WH, int WPP, bool COUNTS>
// CTAs per SM.  4-warp shape, 21x21: 7 (72 registers, no spills) -- with the launch no longer ending in a tail of long
// points the bulk is issue-bound and more resident warps fill more slots (single pair 65.1 -> 64.5 us, four streams
// 50.1 -> 44.6 us per pair; 8 CTAs spill: 72.1 us); 31x31: 5 (6 spill: 98 -> 106 us).  2-warp shape (21x21): 4.
__global__ void __launch_bounds__(kThreads, (WPP == 4 ? (WW * WH <= 21 * 21 ? 7 : 5) : 4))
lk_fast_kernel(const __grid_constant__ LKLaunch L)
{
    using C = Cfg<WW, WH, WPP>;
    extern __shared__ __align__(128) uint8_t smem[];
    const int lane = threadIdx.x & 31;
    const int pic = threadIdx.x / C::NT;        // point within the CTA
    const int tid = threadIdx.x - pic * C::NT;  // thread within the point
    const int wip = tid >> 5;                   // warp within the point
    const int bar = 1 + pic;
    const long long total = (long long)L.n_per_pair * L.batch;
    // Two-pass grid (flag kTwoPass, set by the launcher for launches that fit the chip a few times): the grid holds every
    // point twice; the first copy runs the points close to the image border, the second copy the others.  Points that
    // drift along the border for the full iteration count on two levels are the ones that end a launch, and they are all
    // within win + 8 px of the border; CTAs are dispatched in index order, so they now start at t = 0.
    long long blk = blockIdx.x;
    int pass = 0;
    if (L.flags & kTwoPass) {
        const long long nb = (total + C::PPC - 1) / C::PPC;
        pass = blk >= nb;
        blk -= pass ? nb : 0;
    }
    const long long gid = blk * C::PPC + pic;
    if (gid >= total) return;  // uniform over the point's warps: its named barrier is never used
    pdl_wait();                // points, pyramids and initial flow come from earlier kernels
    if (COUNTS) {              // past this pair's point count; the index within the pair is exact in 32-bit unsigned arithmetic
        const unsigned pair = (unsigned)(gid / L.n_per_pair);
        if ((int)((unsigned)gid - pair * (unsigned)L.n_per_pair) >= __ldg(L.counts + pair)) return;
    }
    pdl_launch_dependents();
    if (L.flags & kTwoPass) {
        const float2 p = reinterpret_cast<const float2*>(L.prev_pts)[gid];
        const float m = fminf(fminf(p.x, (float)(L.prev.lv[0].w - 1) - p.x), fminf(p.y, (float)(L.prev.lv[0].h - 1) - p.y));
        const bool near_border = !(m >= (float)(WW + 8));   // NaN: first pass
        if (near_border == (pass != 0)) return;
    }
    const int bidx = (int)(gid / L.n_per_pair);

    uint8_t* ws = smem + pic * C::POINT_BYTES;
    uint8_t* jreg = ws + C::OFF_J;
    uint32_t* dreg = reinterpret_cast<uint32_t*>(ws + C::OFF_D);
    uint8_t* ireg = ws + C::OFF_I;
    int4* red3 = reinterpret_cast<int4*>(ws + C::OFF_R3);
    int* red16 = reinterpret_cast<int*>(ws + C::OFF_R16);
    int par3 = 0, par16 = 0;

    // units of this thread: unit u = tid + k*NT covers window pixels (y, x0..x0+3).  Only jw[k] = y * (SJ/4) + x0/4, the word
    // offset inside the staged next-image region, is kept; y and x0 are decoded from it where needed (shift / mask when
    // SJ/4 is a power of two -- the 21x21 window, where the division of u by UPR = 6 that this replaces was 5-8 % of all
    // executed instructions -- else from u as before: UPR = 8 for the 31x31 window).
    auto unit_ok = [&](int k) { return tid + k * C::NT < C::NU; };
    int jw[C::UPT];
#pragma unroll
    for (int k = 0; k < C::UPT; ++k) {
        const int u = tid + k * C::NT, uu = (u < C::NU ? u : 0), y = uu / C::UPR;
        jw[k] = y * (C::SJ / 4) + (uu - y * C::UPR);
    }
    static_assert(C::UPR <= C::SJ / 4, "x0/4 must fit below the row stride");
    constexpr bool kDecodeJw = ((C::SJ / 4) & (C::SJ / 4 - 1)) == 0;
    auto unit_y = [&](int k) {
        if constexpr (kDecodeJw) return jw[k] / (C::SJ / 4);
        else { const int u = tid + k * C::NT; return (u < C::NU ? u : 0) / C::UPR; }
    };
    auto unit_x0 = [&](int k) {
        if constexpr (kDecodeJw) return 4 * (jw[k] % (C::SJ / 4));
        else { const int u = tid + k * C::NT; const int uu = (u < C::NU ? u : 0); return 4 * (uu - (uu / C::UPR) * C::UPR); }
    };

    const long long t_start = clock64();
    int n_t1 = 0, n_t2 = 0;
#ifdef KLT_LK_PHASES
    const bool ph_on = (wip == 0) && (gid == g_ph_gid);
    long long ph_t = 0;
#endif
    const float2 p0 = reinterpret_cast<const float2*>(L.prev_pts)[gid];
    float2 outp = make_float2(0.f, 0.f);
    if (L.flags & KLT_OPTFLOW_USE_INITIAL_FLOW) outp = reinterpret_cast<const float2*>(L.next_pts)[gid];
    int status = 1;
    float err = 0.f;
    int iters = 0;
    const float hwx = (float)(WW - 1) * 0.5f, hwy = (float)(WH - 1) * 0.5f;
    const int top = L.prev.top;

    for (int level = top; level >= 0; --level) {
        const LevelView lvI = L.prev.lv[level];
        const LevelView lvJ = L.next.lv[level];
        const uint8_t* __restrict__ imgI = lvI.data + (long long)bidx * lvI.batch_stride;
        const uint8_t* __restrict__ imgJ = lvJ.data + (long long)bidx * lvJ.batch_stride;
        const int lw = lvI.w, lh = lvI.h;

        float px, py, nx, ny;
        level_start(p0, outp, level, top, L.flags, px, py, nx, ny);
        px = __fsub_rn(px, hwx); py = __fsub_rn(py, hwy);
        int ipx, ipy;
        if (!floor_in_range(px, py, WW, WH, lw, lh, ipx, ipy)) {
            if (level == 0) { status = 0; err = 0.f; }
            continue;
        }
        int w00, w01, w10, w11;
        q14_weights(__fsub_rn(px, (float)ipx), __fsub_rn(py, (float)ipy), w00, w01, w10, w11);

        nx = __fsub_rn(nx, hwx); ny = __fsub_rn(ny, hwy);
        // ---- stage both neighbourhoods; the previous level's readers are done (barrier below) -------------
        point_sync<WPP>(bar);
        // region origin: smem col 0 <-> image x = jax; window columns start at jx0.  Nothing staged: an origin that no
        // window position is near (window positions lie in (-2^30, 2^30))
        int jax = 0, jy0 = INT_MIN / 2, jx0 = INT_MIN / 2;
        {
            int inx, iny;
            if (floor_in_range(nx, ny, WW, WH, lw, lh, inx, iny)) {
                jx0 = inx - kM; jy0 = iny - kM; jax = jx0 & ~3;
                stage<C::JR, C::SJ, C::NT>(jreg, lvJ, imgJ, jax, jy0, jx0 - jax, C::JW, tid);
            }
        }
        const int iax = (ipx - 1) & ~3;
        const int oi = (ipx - 1) - iax;
        stage<C::IR, C::SI, C::NT>(ireg, lvI, imgI, iax, ipy - 1, oi, WW + 3, tid);
        point_sync<WPP>(bar);

        // ---- patch pass: Q5 intensity + Q14 derivative patch into registers, integer class sums of G ------------
        const uint32_t W0 = (uint32_t)(w00 & 0xffff) | ((uint32_t)w01 << 16);
        const uint32_t W1 = (uint32_t)(w10 & 0xffff) | ((uint32_t)w11 << 16);
        Px pxs[C::UPT][4];
        int vals[16];
        unsigned q11[4] = {0, 0, 0, 0}, q22[4] = {0, 0, 0, 0}, t11 = 0, t22 = 0;
        int q12[4] = {0, 0, 0, 0}, t12 = 0;
        // all (WW+1) x (WH+1) derivative positions inside the image <=> no zero-masking of the derivative
        const bool interior = (ipx >= 0) && (ipy >= 0) && (ipx + WW < lw) && (ipy + WH < lh);
        if (interior) {
            // Scharr is linear and so is the Q14 bilinear tap, so  sum_c w_c * Scharr(I)(p + c)  ==  Scharr(T)(p)  with
            // T(q) = sum_c w_c * I(q + c) the UNROUNDED bilinear sum (<= 255 * 2^14); exact in int32 (|.| < 2^27).
            const int sh = (oi & 3) * 8;
#pragma unroll
            for (int k = 0; k < C::UPT; ++k) {
                const int y = unit_y(k), x0 = unit_x0(k);
                const bool ok = unit_ok(k);
                uint32_t pa[4], pb[4], pc[4], pd[4];   // byte pairs (c,c+1) of 4 region rows: see pair() below
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    const uint32_t* wp = reinterpret_cast<const uint32_t*>(ireg + (y + r) * C::SI) + ((oi + x0) >> 2);
                    const uint32_t w0 = wp[0], w1 = wp[1], w2 = wp[2];
                    pa[r] = __funnelshift_r(w0, w1, sh);        // bytes c0 .. c0+3   (c0 = column of window x0-1)
                    pb[r] = __funnelshift_rc(w0, w1, sh + 8);   // bytes c0+1 .. c0+4
                    pc[r] = __funnelshift_r(w1, w2, sh);        // bytes c0+4 .. c0+7
                    pd[r] = __funnelshift_rc(w1, w2, sh + 8);   // bytes c0+5 .. c0+8
                }
                int T[3][6];
#pragma unroll
                for (int r = 0; r < 3; ++r) {
                    T[r][0] = dp2a_lo(W1, pa[r + 1], dp2a_lo(W0, pa[r], 0));
                    T[r][1] = dp2a_lo(W1, pb[r + 1], dp2a_lo(W0, pb[r], 0));
                    T[r][2] = dp2a_hi(W1, pa[r + 1], dp2a_hi(W0, pa[r], 0));
                    T[r][3] = dp2a_hi(W1, pb[r + 1], dp2a_hi(W0, pb[r], 0));
                    T[r][4] = dp2a_lo(W1, pc[r + 1], dp2a_lo(W0, pc[r], 0));
                    T[r][5] = dp2a_lo(W1, pd[r + 1], dp2a_lo(W0, pd[r], 0));
                }
                int t0[6], t1[6];
#pragma unroll
                for (int c = 0; c < 6; ++c) {
                    t0[c] = 3 * (T[0][c] + T[2][c]) + 10 * T[1][c];
                    t1[c] = T[2][c] - T[0][c];
                }
                unsigned u11[4], u22[4];
                int u12[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const bool valid = ok && (x0 + j) < WW;
                    const int iv = (T[1][j + 1] + (1 << 8)) >> 9;
                    int gx = (t0[j + 2] - t0[j] + (1 << 13)) >> 14;
                    int gy = (3 * (t1[j] + t1[j + 2]) + 10 * t1[j + 1] + (1 << 13)) >> 14;
                    gx = valid ? gx : 0; gy = valid ? gy : 0;
                    pxs[k][j] = {valid ? iv : 0, gx, gy, max(abs(gx), abs(gy))};
                    u11[j] = (unsigned)(gx * gx); u12[j] = gx * gy; u22[j] = (unsigned)(gy * gy);
                }
                const bool tail = x0 >= C::NV;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    q11[j] += tail ? 0u : u11[j];
                    q12[j] += tail ? 0 : u12[j];
                    q22[j] += tail ? 0u : u22[j];
                }
                t11 += tail ? (u11[0] + u11[1] + u11[2] + u11[3]) : 0u;
                t12 += tail ? (u12[0] + u12[1] + u12[2] + u12[3]) : 0;
                t22 += tail ? (u22[0] + u22[1] + u22[2] + u22[3]) : 0u;
            }
        } else {
            // border window: Scharr at the (WW+1) x (WH+1) integer positions, zero outside the image, then bilinear
            for (int u = tid; u < C::NRUN; u += C::NT) {
                const int dy = u / C::RPR;
                const int dx0 = 4 * (u - dy * C::RPR);
                const uint8_t* r0 = ireg + dy * C::SI + oi + dx0;
                const uint8_t* r1 = r0 + C::SI;
                const uint8_t* r2 = r1 + C::SI;
                int t0[6], t1[6];
#pragma unroll
                for (int k = 0; k < 6; ++k) {
                    const int a = r0[k], b = r1[k], cc = r2[k];
                    t0[k] = 3 * (a + cc) + 10 * b;
                    t1[k] = cc - a;
                }
                const bool yin = (unsigned)(ipy + dy) < (unsigned)lh;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int dx = dx0 + k;
                    const int gx = t0[k + 2] - t0[k];
                    const int gy = 3 * (t1[k] + t1[k + 2]) + 10 * t1[k + 1];
                    const bool in = yin && ((unsigned)(ipx + dx) < (unsigned)lw);
                    if (dx < C::SD) dreg[dy * C::SD + dx] = in ? (((uint32_t)gx & 0xffffu) | ((uint32_t)gy << 16)) : 0u;
                }
            }
            point_sync<WPP>(bar);
#pragma unroll
            for (int k = 0; k < C::UPT; ++k) {
                const int y = unit_y(k), x0 = unit_x0(k);
                const bool ok = unit_ok(k);
                uint32_t a0, b0, a1, b1;
                load5(ireg + (y + 1) * C::SI, oi + 1 + x0, a0, b0);
                load5(ireg + (y + 2) * C::SI, oi + 1 + x0, a1, b1);
                int iv[4];
                iv[0] = dp2a_lo(W1, a1, dp2a_lo(W0, a0, 256)) >> 9;
                iv[1] = dp2a_lo(W1, b1, dp2a_lo(W0, b0, 256)) >> 9;
                iv[2] = dp2a_hi(W1, a1, dp2a_hi(W0, a0, 256)) >> 9;
                iv[3] = dp2a_hi(W1, b1, dp2a_hi(W0, b0, 256)) >> 9;
                const uint32_t* d0 = dreg + y * C::SD + x0;
                const uint32_t* d1 = d0 + C::SD;
                const uint4 e0 = *reinterpret_cast<const uint4*>(d0);
                const uint4 e1 = *reinterpret_cast<const uint4*>(d1);
                const uint32_t r0w[5] = {e0.x, e0.y, e0.z, e0.w, d0[4]};
                const uint32_t r1w[5] = {e1.x, e1.y, e1.z, e1.w, d1[4]};
                unsigned u11[4], u22[4];
                int u12[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    int gx = (lo16(r0w[j]) * w00 + lo16(r0w[j + 1]) * w01 + lo16(r1w[j]) * w10 + lo16(r1w[j + 1]) * w11 + (1 << 13)) >> 14;
                    int gy = (hi16(r0w[j]) * w00 + hi16(r0w[j + 1]) * w01 + hi16(r1w[j]) * w10 + hi16(r1w[j + 1]) * w11 + (1 << 13)) >> 14;
                    const bool valid = ok && (x0 + j) < WW;
                    gx = valid ? gx : 0; gy = valid ? gy : 0;
                    pxs[k][j] = {valid ? iv[j] : 0, gx, gy, max(abs(gx), abs(gy))};
                    u11[j] = (unsigned)(gx * gx); u12[j] = gx * gy; u22[j] = (unsigned)(gy * gy);
                }
                const bool tail = x0 >= C::NV;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    q11[j] += tail ? 0u : u11[j];
                    q12[j] += tail ? 0 : u12[j];
                    q22[j] += tail ? 0u : u22[j];
                }
                t11 += tail ? (u11[0] + u11[1] + u11[2] + u11[3]) : 0u;
                t12 += tail ? (u12[0] + u12[1] + u12[2] + u12[3]) : 0;
                t22 += tail ? (u22[0] + u22[1] + u22[2] + u22[3]) : 0u;
            }
        }
        {
            // A clamped value must still prove "not exact": the clamp is kExact + 1 whatever the team size (a smaller one
            // -- round 1 used 2^25 / WPP -- let a window whose whole gradient energy sits in one thread pass the test:
            // found by tests/test_gpu_random.py on a 12 x 12 image).  Totals stay below 2^32: compared as unsigned.
            const unsigned cap = (unsigned)kExact + 1u;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                vals[j] = (int)min(q11[j], cap);
                vals[5 + j] = max(min(q12[j], (int)cap), -(int)cap);
                vals[10 + j] = (int)min(q22[j], cap);
            }
            vals[4] = (int)min(t11, cap);
            vals[9] = max(min(t12, (int)cap), -(int)cap);
            vals[14] = (int)min(t22, cap);
            vals[15] = 0;
        }
        // lane L < 15 now holds class total L: [0..4] = gx*gx (4 SIMD lanes, tail), [5..9] = gx*gy, [10..14] = gy*gy
        const int gtot = point_sum15_lane<WPP>(vals, red16, par16, wip, lane, bar);

        float A11, A12, A22;
        {
            // A11 / A22: non-negative terms, exact iff every class total <= 2^24; A12: |gx gy| <= (gx^2 + gy^2) / 2
            const unsigned partner = (unsigned)__shfl_sync(kFull, gtot, (lane + 10) & 31);
            const bool ok = (lane >= 5) || ((unsigned)gtot <= (unsigned)kExact && partner <= (unsigned)kExact &&
                                            (unsigned)gtot + partner <= 2u * (unsigned)kExact);
            if (__all_sync(kFull, ok)) {
                const float f = (float)gtot;
                A11 = combine5(__shfl_sync(kFull, f, 0), __shfl_sync(kFull, f, 1), __shfl_sync(kFull, f, 2), __shfl_sync(kFull, f, 3),
                               __shfl_sync(kFull, f, 4));
                A12 = combine5(__shfl_sync(kFull, f, 5), __shfl_sync(kFull, f, 6), __shfl_sync(kFull, f, 7), __shfl_sync(kFull, f, 8),
                               __shfl_sync(kFull, f, 9));
                A22 = combine5(__shfl_sync(kFull, f, 10), __shfl_sync(kFull, f, 11), __shfl_sync(kFull, f, 12), __shfl_sync(kFull, f, 13),
                               __shfl_sync(kFull, f, 14));
            } else {
                // serial replay in OpenCV's order (A.5): every thread stores the float products of its pixels in chain
                // order; all scratch is dead here (every warp passed the exchange barrier above)
                using CH = Chains<WW, WH>;
                float* gf = reinterpret_cast<float*>(dreg);
#pragma unroll
                for (int k = 0; k < C::UPT; ++k)
                    if (unit_ok(k)) {
                        const int y = unit_y(k), x0 = unit_x0(k);
                        const bool tail = x0 >= C::NV;
                        float* g0 = tail ? gf + 12 * CH::GQ4 + y * CH::TL + (x0 - C::NV) : gf + y * (C::NV / 4) + (x0 >> 2);
                        const int sj = tail ? 1 : CH::GQ4;            // next pixel: next element of the tail / next lane chain
                        const int ss = tail ? CH::GT4 : 4 * CH::GQ4;  // next sum
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            if (x0 + j < WW) {
                                const int gx = pxs[k][j].gx, gy = pxs[k][j].gy;
                                g0[j * sj] = (float)(gx * gx);
                                g0[j * sj + ss] = (float)(gx * gy);
                                g0[j * sj + 2 * ss] = (float)(gy * gy);
                            }
                    }
                {   // zero pads
                    constexpr int PQ = CH::GQ4 - CH::GQ, PT = CH::GT4 - CH::GT;
                    if (tid < 12 * PQ) gf[(tid / (PQ > 0 ? PQ : 1)) * CH::GQ4 + CH::GQ + tid % (PQ > 0 ? PQ : 1)] = 0.f;
                    if (tid < 3 * PT) gf[12 * CH::GQ4 + (tid / (PT > 0 ? PT : 1)) * CH::GT4 + CH::GT + tid % (PT > 0 ? PT : 1)] = 0.f;
                }
                point_sync<WPP>(bar);
                replay_g<WW, WH>(gf, wip, lane);
                point_sync<WPP>(bar);
                const float* r = gf + CH::G_RES;
                A11 = combine5(r[0], r[1], r[2], r[3], r[4]);
                A12 = combine5(r[5], r[6], r[7], r[8], r[9]);
                A22 = combine5(r[10], r[11], r[12], r[13], r[14]);
            }
        }
        float D;
        if (!eig_gate(A11, A12, A22, WW, WH, L.flags, L.min_eig_thr, err, D)) {
            if (level == 0) status = 0;
            continue;
        }

        // ---- iterations ------------------------------------------------------------------------------------
        // make sure the staged next-image region covers the window at (inx, iny)
        auto ensure_j = [&](int inx, int iny) {
            // covered <=> 0 <= inx - jx0 <= 2 kM and the same in y (the region is the window + 1 plus kM on every side)
            if ((unsigned)(inx - jx0) > 2u * kM || (unsigned)(iny - jy0) > 2u * kM) {
                point_sync<WPP>(bar);
                jx0 = inx - kM; jy0 = iny - kM; jax = jx0 & ~3;
                stage<C::JR, C::SJ, C::NT>(jreg, lvJ, imgJ, jax, jy0, jx0 - jax, C::JW, tid);
                point_sync<WPP>(bar);
            }
        };

        float pdx = 0.f, pdy = 0.f;
        bool sticky = false, pads_zeroed = false;
#ifdef KLT_LK_PHASES
        ph_t = clock64();
#endif
        // The position is tested for NaN / inf once: inside the loop it is a position that passed the range test plus a
        // finite step (|A| < 2^14, |b| < 2^15, 1/D <= 2^23), so it stays finite.
        if (L.max_count > 0 && !((fabsf(nx) < 1.0e9f) && (fabsf(ny) < 1.0e9f))) {
            if (level == 0) status = 0;
            continue;
        }
        for (int j = 0; j < L.max_count; ++j) {
            int inx, iny;
            if (!floor_in_range_finite(nx, ny, WW, WH, lw, lh, inx, iny)) {
                if (level == 0) status = 0;
                break;
            }
            ++iters;
            PH_COUNT(15);
            ensure_j(inx, iny);
            int v00, v01, v10, v11;
            q14_weights(__fsub_rn(nx, (float)inx), __fsub_rn(ny, (float)iny), v00, v01, v10, v11);
            const uint32_t W0 = (uint32_t)(v00 & 0xffff) | ((uint32_t)v01 << 16);
            const uint32_t W1 = (uint32_t)(v10 & 0xffff) | ((uint32_t)v11 << 16);
            int dd[C::UPT][4];
            int s1, s2, bnd;
            PH(0);   // loop top: range test, region test, weights
            {
                // invalid pixels carry gx = gy = gm = 0, so they drop out of all three sums without a select
                const int cb = (iny - jy0) * C::SJ + (inx - jax);
                const uint32_t* __restrict__ jbase = reinterpret_cast<const uint32_t*>(jreg) + (cb >> 2);
                const int sh = (cb & 3) * 8;
                s1 = 0; s2 = 0; bnd = 0;
#pragma unroll
                for (int k = 0; k < C::UPT; ++k) {
                    const uint32_t* __restrict__ r0 = jbase + jw[k];
                    const uint32_t* __restrict__ r1 = r0 + C::SJ / 4;
                    const uint32_t p0 = r0[0], p1 = r0[1], q0 = r1[0], q1 = r1[1];
                    const uint32_t a0 = __funnelshift_r(p0, p1, sh), b0 = __funnelshift_rc(p0, p1, sh + 8);
                    const uint32_t a1 = __funnelshift_r(q0, q1, sh), b1 = __funnelshift_rc(q0, q1, sh + 8);
                    int jv[4];
                    jv[0] = dp2a_lo(W1, a1, dp2a_lo(W0, a0, 256)) >> 9;
                    jv[1] = dp2a_lo(W1, b1, dp2a_lo(W0, b0, 256)) >> 9;
                    jv[2] = dp2a_hi(W1, a1, dp2a_hi(W0, a0, 256)) >> 9;
                    jv[3] = dp2a_hi(W1, b1, dp2a_hi(W0, b0, 256)) >> 9;
#pragma unroll
                    for (int jj = 0; jj < 4; ++jj) {
                        const int d = jv[jj] - pxs[k][jj].iv;
                        dd[k][jj] = d;
                        s1 += d * pxs[k][jj].gx;
                        s2 += d * pxs[k][jj].gy;
                        bnd += abs(d) * pxs[k][jj].gm;
                    }
                }
            }
            // Tier 0 (whole-window bound) unless the previous iteration of this point already failed it ("sticky"):
            // diverging points fail it every time, and they are the ones that bound the launch latency.
            float b1 = 0.f, b2 = 0.f;
            bool classes = sticky;
            PH(1);   // per-pixel pass
            if (!sticky) {
                // per-thread |bound| <= UPT*4*8160*4080 < 2^31 for UPT <= 2; clamped to kExact + 1 so that the point total
                // (<= 128 * (2^24 + 1) < 2^32, compared as unsigned) cannot wrap and a clamped thread alone fails the test
                bnd = min(bnd, kExact + 1);
                point_sum3<WPP>(s1, s2, bnd, red3, par3, wip, lane, bar);
                if ((unsigned)bnd <= (unsigned)kExact) {
                    // every float32 partial sum OpenCV forms (lanes, tail, final combine) is an exact integer
                    b1 = __fmul_rn((float)s1, 9.5367431640625e-07f);
                    b2 = __fmul_rn((float)s2, 9.5367431640625e-07f);
                } else {
                    sticky = true;
                    classes = true;
                }
            }
            PH(2);   // tier 0
            if (classes) {
                // tier 1: per accumulation class (4 SIMD lanes + tail), bound in units of 16 (rounded up per pixel)
                ++n_t1;
                int cv[16];
#pragma unroll
                for (int i = 0; i < 16; ++i) cv[i] = 0;
#pragma unroll
                for (int k = 0; k < C::UPT; ++k) {
                    int u1[4], u2[4], ub[4];
#pragma unroll
                    for (int jj = 0; jj < 4; ++jj) {
                        const int d = dd[k][jj];
                        u1[jj] = d * pxs[k][jj].gx;
                        u2[jj] = d * pxs[k][jj].gy;
                        ub[jj] = (abs(d) * pxs[k][jj].gm + 15) >> 4;
                    }
                    const bool tail = unit_x0(k) >= C::NV;
#pragma unroll
                    for (int jj = 0; jj < 4; ++jj) {
                        cv[jj] += tail ? 0 : u1[jj];
                        cv[5 + jj] += tail ? 0 : u2[jj];
                        cv[10 + jj] += tail ? 0 : ub[jj];
                    }
                    cv[4] += tail ? (u1[0] + u1[1] + u1[2] + u1[3]) : 0;
                    cv[9] += tail ? (u2[0] + u2[1] + u2[2] + u2[3]) : 0;
                    cv[14] += tail ? (ub[0] + ub[1] + ub[2] + ub[3]) : 0;
                }
#pragma unroll
                for (int i = 10; i < 15; ++i) cv[i] = min(cv[i], (kExact >> 4) + 1);   // clamped => not exact (see the G sums)
                const int ctot = point_sum15_lane<WPP>(cv, red16, par16, wip, lane, bar);
                const bool is_bound = (lane >= 10) && (lane < 15);
                const bool exact = __all_sync(kFull, !is_bound || ctot <= (kExact >> 4));
                // leave sticky mode once the whole-window bound would pass again (converging point)
                sticky = __reduce_add_sync(kFull, is_bound ? ctot : 0) > (kExact >> 4);
                PH(3);   // tier 1 sums + tests
                if (exact) {
                    const float f = (float)ctot;
                    b1 = combine5(__shfl_sync(kFull, f, 0), __shfl_sync(kFull, f, 1), __shfl_sync(kFull, f, 2), __shfl_sync(kFull, f, 3),
                                  __shfl_sync(kFull, f, 4));
                    b2 = combine5(__shfl_sync(kFull, f, 5), __shfl_sync(kFull, f, 6), __shfl_sync(kFull, f, 7), __shfl_sync(kFull, f, 8),
                                  __shfl_sync(kFull, f, 9));
                } else {
                    // tier 2: serial replay (pairs (l, l+4) summed in int32 first; A.5).  The scratch is rewritten by the
                    // next replay only after every warp has passed that replay's first barrier, i.e. after it has read
                    // these results.
                    ++n_t2;
                    using CH = Chains<WW, WH>;
                    int* buf = reinterpret_cast<int*>(dreg);
                    if (!pads_zeroed) { zero_pad_b<WW, WH, C::NT>(buf, tid); pads_zeroed = true; }  // pads survive until the next level
#pragma unroll
                    for (int k = 0; k < C::UPT; ++k)
                        if (unit_ok(k)) {
                            const int y = unit_y(k), x0 = unit_x0(k);
                            if (x0 >= C::NV) {
                                float* tf = reinterpret_cast<float*>(buf) + 8 * CH::SLEN4 + y * CH::TL + (x0 - C::NV);
#pragma unroll
                                for (int jj = 0; jj < 4; ++jj)
                                    if (x0 + jj < WW) {
                                        const int d = dd[k][jj];
                                        tf[jj] = (float)(d * pxs[k][jj].gx);
                                        tf[CH::TLEN + jj] = (float)(d * pxs[k][jj].gy);
                                    }
                            } else {
                                int* si = buf + (y * CH::NS + (x0 >> 3)) * 2 + ((x0 >> 2) & 1);
#pragma unroll
                                for (int jj = 0; jj < 4; ++jj) {
                                    const int d = dd[k][jj];
                                    si[jj * CH::SLEN4] = d * pxs[k][jj].gx;
                                    si[(4 + jj) * CH::SLEN4] = d * pxs[k][jj].gy;
                                }
                            }
                        }
                    PH(4);   // replay stores
                    point_sync<WPP>(bar);
                    PH(5);   // barrier before the replay
                    replay_b<WW, WH>(buf, wip, lane);
                    PH(6);   // warp 0's chains
                    point_sync<WPP>(bar);
                    PH(7);   // barrier after the replay (= the tail chains of warp 1)
                    PH_COUNT(14);
                    static_assert(CH::B_RES % 4 == 0, "results are read with 128-bit loads");
                    const float4 r1 = *reinterpret_cast<const float4*>(buf + CH::B_RES);
                    const float4 r2 = *reinterpret_cast<const float4*>(buf + CH::B_RES + 4);
                    const float2 rt = *reinterpret_cast<const float2*>(buf + CH::B_RES + 8);
                    b1 = combine5(r1.x, r1.y, r1.z, r1.w, rt.x);
                    b2 = combine5(r2.x, r2.y, r2.z, r2.w, rt.y);
                }
            }
            PH(8);   // combine
            if (newton_step(A11, A12, A22, D, b1, b2, j, L.eps2_lo, L.eps2_hi, L.eps2, hwx, hwy, nx, ny, pdx, pdy, outp)) break;
            PH(9);   // solve + termination tests
        }

        // ---- err at level 0 ------------------------------------------------------------------------------------
        if (status && level == 0 && (L.flags & KLT_OPTFLOW_LK_GET_MIN_EIGENVALS) == 0) {
            const float qx = __fsub_rn(outp.x, hwx), qy = __fsub_rn(outp.y, hwy);
            int iqx, iqy;
            if (!floor_in_range(qx, qy, WW, WH, lw, lh, iqx, iqy)) {
                status = 0;
                continue;
            }
            ensure_j(iqx, iqy);
            int v00, v01, v10, v11;
            q14_weights(__fsub_rn(qx, (float)iqx), __fsub_rn(qy, (float)iqy), v00, v01, v10, v11);
            const uint32_t W0 = (uint32_t)(v00 & 0xffff) | ((uint32_t)v01 << 16);
            const uint32_t W1 = (uint32_t)(v10 & 0xffff) | ((uint32_t)v11 << 16);
            int e = 0, z1 = 0, z2 = 0;
            {
                const int cb = (iqy - jy0) * C::SJ + (iqx - jax);
                const uint32_t* __restrict__ jbase = reinterpret_cast<const uint32_t*>(jreg) + (cb >> 2);
                const int sh = (cb & 3) * 8;
#pragma unroll
                for (int k = 0; k < C::UPT; ++k) {
                    const uint32_t* __restrict__ r0 = jbase + jw[k];
                    const uint32_t* __restrict__ r1 = r0 + C::SJ / 4;
                    const uint32_t p0 = r0[0], p1 = r0[1], q0 = r1[0], q1 = r1[1];
                    const uint32_t a0 = __funnelshift_r(p0, p1, sh), b0 = __funnelshift_rc(p0, p1, sh + 8);
                    const uint32_t a1 = __funnelshift_r(q0, q1, sh), b1 = __funnelshift_rc(q0, q1, sh + 8);
                    int jv[4];
                    jv[0] = dp2a_lo(W1, a1, dp2a_lo(W0, a0, 256)) >> 9;
                    jv[1] = dp2a_lo(W1, b1, dp2a_lo(W0, b0, 256)) >> 9;
                    jv[2] = dp2a_hi(W1, a1, dp2a_hi(W0, a0, 256)) >> 9;
                    jv[3] = dp2a_hi(W1, b1, dp2a_hi(W0, b0, 256)) >> 9;
                    const bool ok = unit_ok(k);
                    const int x0 = unit_x0(k);
#pragma unroll
                    for (int jj = 0; jj < 4; ++jj) e += (ok && (x0 + jj) < WW) ? abs(jv[jj] - pxs[k][jj].iv) : 0;
                }
            }
            point_sum3<WPP>(e, z1, z2, red3, par3, wip, lane, bar);
            // |d| <= 8160 and WW*WH <= 2056 for the instantiated windows: e <= 2^24, so OpenCV's float32 running sum is exact
            err = lk_err((float)e, WW, WH);
        }
    }

    if (tid == 0) {
        reinterpret_cast<float2*>(L.next_pts)[gid] = outp;
        L.status[gid] = (uint8_t)status;
        L.err[gid] = err;
        if (L.iters) {
            // debug flag 0x100: cycles / 64 in the low 20 bits, tier-1 and tier-2 counts above (profiling aid)
            L.iters[gid] = (L.flags & 0x100) ? (int)(((clock64() - t_start) >> 6) & 0xfffff) | (min(n_t1, 63) << 20) | (min(n_t2, 63) << 26) : iters;
        }
    }
}

template <int WW, int WH, int WPP, bool COUNTS>
klt_status launch_fast_as(const LKLaunch& L, cudaStream_t stream)
{
    using C = Cfg<WW, WH, WPP>;
    static_assert(WW * WH <= 2056, "err pass assumes an exact float32 sum");
    static_assert(C::UPT <= 2, "per-pixel state of at most 8 pixels per thread in registers; bound accumulators must not overflow");
    static PerDeviceOnce configured;
    const size_t smem = (size_t)C::POINT_BYTES * C::PPC;
    if (configured.needed()) {
        cudaError_t e = cudaFuncSetAttribute(lk_fast_kernel<WW, WH, WPP, COUNTS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (klt_status)e;
    }
    const long long total = (long long)L.n_per_pair * L.batch;
    long long blocks = (total + C::PPC - 1) / C::PPC;
    if (L.flags & kTwoPass) blocks *= 2;
    if (blocks > 0x7fffffffLL) return KLT_ERR_UNSUPPORTED;
    const cudaError_t e = launch_pdl(lk_fast_kernel<WW, WH, WPP, COUNTS>, (unsigned)blocks, kThreads, smem, stream, 1, L);
    return e == cudaSuccess ? KLT_OK : (klt_status)e;
}

template <int WW, int WH, int WPP>
klt_status launch_fast(const LKLaunch& L, cudaStream_t stream)
{
    return L.counts ? launch_fast_as<WW, WH, WPP, true>(L, stream) : launch_fast_as<WW, WH, WPP, false>(L, stream);
}

}  // namespace

// Returns KLT_ERR_UNSUPPORTED when no specialisation exists (the caller then uses the generic kernel).
klt_status lk_launch_fast(const LKLaunch& L, int sm_count, cudaStream_t stream)
{
    const long long total = (long long)L.n_per_pair * L.batch;
    // warps per point, from measurements on B200 (profiles/): the kernel is latency-bound, so more warps per point win
    // until the per-iteration overhead replicated in every warp dominates: 31x31 -> always 4; 21x21 -> 4 while the
    // points fit the chip about once, else 2.  One warp per point never wins (register-limited occupancy).
    const bool two_warps = L.win_w * L.win_h <= 21 * 21 && total > (long long)sm_count * 32;
    // Two-pass grid (see the kernel): only for one point per CTA (with two, a CTA whose points fall into different passes
    // would run half empty twice) and for launches whose end is a tail of a few points rather than a last full wave.
    // Measured on the KITTI bench (155 pairs, 2000 points each): 77.8 -> 65.2 us per launch at win 21, 115.7 -> 98.0 us at
    // win 31; a launch without any border point pays for 2000 CTAs that exit at once (< 2 us).
    LKLaunch L2 = L;
    L2.flags &= ~kTwoPass;
    if (!two_warps && total <= (long long)sm_count * 128) L2.flags |= kTwoPass;
    if (L.win_w == 21 && L.win_h == 21) return two_warps ? launch_fast<21, 21, 2>(L2, stream) : launch_fast<21, 21, 4>(L2, stream);
    if (L.win_w == 31 && L.win_h == 31) return launch_fast<31, 31, 4>(L2, stream);
    return KLT_ERR_UNSUPPORTED;
}

}  // namespace klt

#ifdef KLT_LK_PHASES
extern "C" int klt_debug_lk_phase_select(long long gid)
{
    unsigned long long zero[16] = {};
    cudaError_t e = cudaMemcpyToSymbol(klt::g_ph, zero, sizeof(zero));
    if (e == cudaSuccess) e = cudaMemcpyToSymbol(klt::g_ph_gid, &gid, sizeof(gid));
    return (int)e;
}
extern "C" int klt_debug_lk_phase_read(unsigned long long* out16)
{
    return (int)cudaMemcpyFromSymbol(out16, klt::g_ph, 16 * sizeof(unsigned long long));
}
#endif
