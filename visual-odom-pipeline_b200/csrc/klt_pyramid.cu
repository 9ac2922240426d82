// K1: batched 5-tap separable pyrDown for u8 images on sm_100a.
//
// Replaces cv2.pyrDown as run inside cv2.buildOpticalFlowPyramid / calcOpticalFlowPyrLK, which the
// reference reaches from src/extractor/extractor.py:44,45,65,66.  Arithmetic (SURVEY.md A.2):
//   dst(x,y) = ( sum_{i,j in [-2,2]} k_i k_j src(R(2x+i), R(2y+j)) + 128 ) >> 8,  k = [1 4 6 4 1],
//   R = BORDER_REFLECT_101, dst size ((w+1)/2, (h+1)/2).  Integer, bit-exact.
//
// Design (HBM-bound byte work, no tensor cores):
//  * one warp owns a strip of 64*NOUT input columns x (2R+3) input rows and produces 32*NOUT x R
//    outputs.  Main kernel (16-byte aligned rows): every lane streams its 2*NOUT contiguous bytes of
//    each input row into a per-warp shared-memory ring with ONE 128/64-bit cp.async (LDGSTS: no
//    registers held while in flight, 4 rows = 2 KB per warp of lookahead, no block-level barriers);
//    the 2+1 halo columns are the neighbouring lanes' bytes in the same ring slot, so the consumer
//    reads them with plain LDS -- REFLECT_101 at the image edges is patched in the slot (2 byte
//    copies per row, edge warps only).  Fallback kernel (unaligned pitches / tiny images): direct
//    loads + warp shuffles + byte gathers.
//  * bytes are widened to packed u16x2 lanes (PRMT) so one 32-bit op filters two columns; the
//    vertical pass is a sliding window (T_y = r[2y] + 4 r[2y+1] + r[2y+2]; V_y = T_{y-1} + T_y +
//    4 r[2y]) so each input row is loaded and unpacked once per strip; the horizontal pass works
//    on funnel-shifted packed pairs; max partial sum 255*256 = 65280 fits the 16-bit lanes;
//  * next strip rows are prefetched into registers while the current output row is computed;
//  * image borders (REFLECT_101) and unaligned pitches take a byte-gather path in the edge lanes
//    only; interior lanes never branch on coordinates;
//  * pyr_build_fused_kernel runs the ring kernel's warp tasks for every level of a pyramid in one launch.
// Measured on B200 and removed (DESIGN.md s4 K1, s7): a TMA (UTMALDG) fill of the ring reached 36-51 % of the copy peak
// against 55-66 %, and a tile kernel that builds two levels per launch took 187 us for the pyramids of 310 KITTI frames
// against 69 us for one ring launch per level.
#include "klt_common.cuh"

#include <cstdlib>

namespace klt {

namespace {

constexpr int kWarpsPerBlock = 8;

__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel)
{
    uint32_t r;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(sel));
    return r;
}
__device__ __forceinline__ uint32_t dp4a_uu(uint32_t a, uint32_t b, uint32_t c)
{
    uint32_t d;
    asm("dp4a.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
// (b0, 0, b2, 0) and (b1, 0, b3, 0) of a word: even / odd columns as packed u16x2
__device__ __forceinline__ uint32_t even_bytes(uint32_t w) { return prmt(w, 0u, 0x4240u); }
__device__ __forceinline__ uint32_t odd_bytes(uint32_t w) { return prmt(w, 0u, 0x4341u); }

template <int NOUT>
struct RawRow {
    uint32_t w[NOUT / 2];  // own 2*NOUT bytes
    uint32_t l, r;         // word left of / right of the own bytes (from neighbours)
};

// Load the raw bytes one lane needs from one (already row-reflected) input row.
template <int NOUT, bool ALIGNED>
__device__ __forceinline__ void load_row(const uint8_t* __restrict__ row, int cb, int w, bool fast,
                                         int lane, RawRow<NOUT>& out)
{
    constexpr int NW = NOUT / 2;
    if (ALIGNED && fast) {
        if constexpr (NOUT == 8) {
            uint4 v = __ldg(reinterpret_cast<const uint4*>(row + cb));
            out.w[0] = v.x; out.w[1] = v.y; out.w[2] = v.z; out.w[3] = v.w;
        } else {
            uint2 v = __ldg(reinterpret_cast<const uint2*>(row + cb));
            out.w[0] = v.x; out.w[1] = v.y;
        }
    } else {
#pragma unroll
        for (int i = 0; i < NW; ++i) {
            uint32_t v = 0;
#pragma unroll
            for (int j = 0; j < 4; ++j)
                v |= (uint32_t)__ldg(row + reflect101(cb + 4 * i + j, w)) << (8 * j);
            out.w[i] = v;
        }
    }
    out.l = __shfl_up_sync(0xffffffffu, out.w[NW - 1], 1);
    out.r = __shfl_down_sync(0xffffffffu, out.w[0], 1);
    if (lane == 0) {
        out.l = ((uint32_t)__ldg(row + reflect101(cb - 2, w)) << 16) |
                ((uint32_t)__ldg(row + reflect101(cb - 1, w)) << 24);
    }
    if (lane == 31) out.r = (uint32_t)__ldg(row + reflect101(cb + 2 * NOUT, w));
}

// packed u16x2 columns of one row: [0]=(cb-4,cb-2) [1]=(cb-3,cb-1) then per own word i:
// [2+2i]=(cb+4i, cb+4i+2) [3+2i]=(cb+4i+1, cb+4i+3), last = (cb+2NOUT, junk)
template <int NOUT>
__device__ __forceinline__ void unpack_row(const RawRow<NOUT>& raw, uint32_t (&p)[NOUT + 3])
{
    constexpr int NW = NOUT / 2;
    p[0] = even_bytes(raw.l);
    p[1] = odd_bytes(raw.l);
#pragma unroll
    for (int i = 0; i < NW; ++i) {
        p[2 + 2 * i] = even_bytes(raw.w[i]);
        p[3 + 2 * i] = odd_bytes(raw.w[i]);
    }
    p[NOUT + 2] = even_bytes(raw.r);
}

template <int NOUT, bool ALIGNED>
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
pyr_down_kernel(const uint8_t* __restrict__ src, int w, int h, long long spitch, long long sbatch,
                uint8_t* __restrict__ dst, int dw, int dh, long long dpitch, long long dbatch,
                int rows_per_strip, int tiles_x, int strips_y, long long n_tasks)
{
    constexpr int NW = NOUT / 2;
    constexpr int NP = NOUT + 3;
    const int lane = threadIdx.x & 31;
    const long long task = (long long)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
    if (task >= n_tasks) return;  // warp-uniform

    const int tx = (int)(task % tiles_x);
    const long long t2 = task / tiles_x;
    const int sy = (int)(t2 % strips_y);
    const int b = (int)(t2 / strips_y);

    const uint8_t* __restrict__ simg = src + (long long)b * sbatch;
    uint8_t* __restrict__ dimg = dst + (long long)b * dbatch;

    const int cb = tx * (64 * NOUT) + 2 * NOUT * lane;  // first own input column
    const bool fast = (cb + 2 * NOUT <= w);             // all own columns inside the image
    const int y0 = sy * rows_per_strip;
    const int y1 = min(y0 + rows_per_strip, dh);

    uint32_t tprev[NP], rc[NP];
    {
        RawRow<NOUT> a, bq, c;
        load_row<NOUT, ALIGNED>(simg + (long long)reflect101(2 * y0 - 2, h) * spitch, cb, w, fast, lane, a);
        load_row<NOUT, ALIGNED>(simg + (long long)reflect101(2 * y0 - 1, h) * spitch, cb, w, fast, lane, bq);
        load_row<NOUT, ALIGNED>(simg + (long long)reflect101(2 * y0, h) * spitch, cb, w, fast, lane, c);
        uint32_t pa[NP], pb[NP];
        unpack_row<NOUT>(a, pa);
        unpack_row<NOUT>(bq, pb);
        unpack_row<NOUT>(c, rc);
#pragma unroll
        for (int i = 0; i < NP; ++i) tprev[i] = pa[i] + 4u * pb[i] + rc[i];
    }

    RawRow<NOUT> nxt_o, nxt_e;  // prefetched rows 2y+1, 2y+2
    load_row<NOUT, ALIGNED>(simg + (long long)reflect101(2 * y0 + 1, h) * spitch, cb, w, fast, lane, nxt_o);
    load_row<NOUT, ALIGNED>(simg + (long long)reflect101(2 * y0 + 2, h) * spitch, cb, w, fast, lane, nxt_e);

    const int xo = cb >> 1;  // first output column of this lane
    for (int y = y0; y < y1; ++y) {
        uint32_t ro[NP], re[NP];
        unpack_row<NOUT>(nxt_o, ro);
        unpack_row<NOUT>(nxt_e, re);
        if (y + 1 < y1) {  // warp-uniform: prefetch the next output row's inputs
            load_row<NOUT, ALIGNED>(simg + (long long)reflect101(2 * y + 3, h) * spitch, cb, w, fast, lane, nxt_o);
            load_row<NOUT, ALIGNED>(simg + (long long)reflect101(2 * y + 4, h) * spitch, cb, w, fast, lane, nxt_e);
        }
        uint32_t v[NP];
#pragma unroll
        for (int i = 0; i < NP; ++i) {
            uint32_t t = rc[i] + 4u * ro[i] + re[i];
            v[i] = tprev[i] + t + 4u * rc[i];
            tprev[i] = t;
            rc[i] = re[i];
        }
        // horizontal pass: own word i gives outputs 2i (centre col cb+4i) and 2i+1 (cb+4i+2)
        uint32_t s[NW];
#pragma unroll
        for (int i = 0; i < NW; ++i) {
            const uint32_t e_m = v[2 * i], o_m = v[2 * i + 1];      // (c-4,c-2) (c-3,c-1)
            const uint32_t e_c = v[2 * i + 2], o_c = v[2 * i + 3];  // (c,c+2)   (c+1,c+3)
            const uint32_t e_p = v[2 * i + 4];                      // (c+4, .)
            const uint32_t a = __funnelshift_r(e_m, e_c, 16);       // (c-2, c)
            const uint32_t c = __funnelshift_r(e_c, e_p, 16);       // (c+2, c+4)
            const uint32_t oa = __funnelshift_r(o_m, o_c, 16);      // (c-1, c+1)
            s[i] = a + c + 6u * e_c + 4u * (oa + o_c) + 0x00800080u;  // +128 per lane; >>8 below
        }
        uint8_t* drow = dimg + (long long)y * dpitch + xo;
        if (ALIGNED && xo + NOUT <= dw) {
            if constexpr (NOUT == 8) {
                uint2 o;
                o.x = prmt(s[0], s[1], 0x7531u);
                o.y = prmt(s[2], s[3], 0x7531u);
                *reinterpret_cast<uint2*>(drow) = o;
            } else {
                *reinterpret_cast<uint32_t*>(drow) = prmt(s[0], s[1], 0x7531u);
            }
        } else {
#pragma unroll
            for (int i = 0; i < NW; ++i) {
                if (xo + 2 * i < dw) drow[2 * i] = (uint8_t)(s[i] >> 8);
                if (xo + 2 * i + 1 < dw) drow[2 * i + 1] = (uint8_t)(s[i] >> 24);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// Main kernel: cp.async ring.  Requires 16-byte aligned src rows, 8-byte aligned dst rows, w >= 3.
constexpr int kRing = 8;  // ring slots (input rows) per warp
constexpr int kRingCtasPerSm = 3;   // resident CTAs of kWarpsPerBlock warps per SM (80 registers a thread)

template <int NOUT>
struct RingCfg {
    static constexpr int BODY = 64 * NOUT;              // bytes of one input row owned by the warp
    static constexpr int SLOT = BODY + 32;              // [12 pad][4 left halo][BODY][4 right halo][12 pad]
    static constexpr int WARP_BYTES = kRing * SLOT;
};

__device__ __forceinline__ void cp_async_16(uint32_t dst, const void* src)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_8(uint32_t dst, const void* src)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_4(uint32_t dst, const void* src)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__device__ __forceinline__ uint32_t lds_u32(uint32_t a)
{
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ uint2 lds_v2(uint32_t a)
{
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a));
    return v;
}
__device__ __forceinline__ uint4 lds_v4(uint32_t a)
{
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ uint32_t lds_u8(uint32_t a)
{
    uint32_t v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts_u8(uint32_t a, uint32_t v) { asm volatile("st.shared.u8 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }

// One warp task: output rows [y0, y1) of the tile whose first input column is X0 (NOUT outputs per lane).
template <int NOUT>
__device__ __forceinline__ void ring_task(const uint8_t* __restrict__ simg, int w, int h, long long spitch,
                                          uint8_t* __restrict__ dimg, int dw, long long dpitch, int X0, int y0, int y1,
                                          uint32_t ring_s, int lane)
{
    using RC = RingCfg<NOUT>;
    constexpr int NW = NOUT / 2;
    const int cb = X0 + 2 * NOUT * lane;          // first own input column
    const int n_rows = 2 * (y1 - y0) + 3;         // input rows 2*y0-2 .. 2*y1
    const uint32_t my_s = ring_s + 16 + 2 * NOUT * lane;   // own bytes inside slot 0
    const uint8_t* __restrict__ gown = simg + cb;
    // one extra 4-byte halo copy per row: lane 0 fetches columns X0-4..X0-1, lane 31 columns X0+BODY..X0+BODY+3
    const bool has_x = (lane == 0 && X0 > 0) || (lane == 31 && X0 + RC::BODY < w);
    const uint32_t x_s = ring_s + ((lane == 0) ? 12u : (uint32_t)(16 + RC::BODY));
    const uint8_t* __restrict__ gx = simg + ((lane == 0) ? (X0 - 4) : (X0 + RC::BODY));
    const int hm2 = 2 * h - 2;
    const unsigned pitch32 = (unsigned)spitch;   // h * pitch < 2^31 is checked by the launcher

    // input row i of the strip = image row 2*y0-2+i under REFLECT_101; for -h < r < 2h-1 that is
    // min(|r|, 2h-2-|r|), branch-free.  SO_ = compile-time ring slot offset.  One commit group per row, always.
    // Copies are whole 16/8/4-byte granules: a granule that holds at least one pixel lies inside the 16-byte-pitched
    // row, and the bytes past column w-1 it may bring along are never used (columns w, w+1 are patched below).
    const int r_first = 2 * y0 - 2;
    const bool do_own = cb < w;
#define KLT_ISSUE(i_, SO_)                                                                              \
    do {                                                                                                \
        if ((i_) < n_rows) { /* warp-uniform */                                                         \
            const int ra_ = abs(r_first + (i_));                                                        \
            const unsigned long long off_ = (unsigned long long)(unsigned)min(ra_, hm2 - ra_) * pitch32; \
            if (do_own) {                                                                               \
                if constexpr (NOUT == 8) cp_async_16(my_s + (SO_), gown + off_);                        \
                else cp_async_8(my_s + (SO_), gown + off_);                                             \
            }                                                                                           \
            if (has_x) cp_async_4(x_s + (SO_), gx + off_);                                              \
        }                                                                                               \
        cp_async_commit();                                                                              \
    } while (0)

    // REFLECT_101 at the right image edge: columns w, w+1 mirror w-2, w-3; patched inside the landed slot by two
    // lanes (the sources are always inside the slot: body or left halo).  The left edge is fixed in registers.
    const bool fix_right = (w < X0 + RC::BODY + 4);
    const int fr_c = w - X0 + lane;                  // lane 0: column w (mirror: -2), lane 1: column w+1 (mirror: -4)
    const bool fr_on = (lane < 2) && (fr_c < RC::BODY + 4);
    const uint32_t fr_dst = ring_s + 16 + fr_c, fr_src = fr_dst - 2 - 2 * lane;
#define KLT_FIX_RIGHT(SO_)                                                                              \
    do {                                                                                                \
        if (fr_on) sts_u8(fr_dst + (SO_), lds_u8(fr_src + (SO_)));                                      \
    } while (0)

    const bool fix_left = (X0 == 0) && (lane == 0);
    // Words of one landed row: W[0] = the 4 bytes left of the own bytes, W[1..NW] = own bytes, W[NW+1] = the 4 bytes right.
#define KLT_LOAD_ROW(SO_, W_)                                                                           \
    do {                                                                                                \
        const uint32_t a_ = my_s + (SO_);                                                               \
        if constexpr (NOUT == 8) {                                                                      \
            const uint4 v_ = lds_v4(a_);                                                                \
            (W_)[1] = v_.x; (W_)[2] = v_.y; (W_)[3] = v_.z; (W_)[4] = v_.w;                             \
        } else {                                                                                        \
            const uint2 v_ = lds_v2(a_);                                                                \
            (W_)[1] = v_.x; (W_)[2] = v_.y;                                                             \
        }                                                                                               \
        (W_)[0] = lds_u32(a_ - 4);                                                                      \
        (W_)[NW + 1] = lds_u32(a_ + 2 * NOUT);                                                          \
        if (fix_left) (W_)[0] = prmt((W_)[1], (W_)[1], 0x1200u); /* columns -2,-1 mirror 2,1 */         \
    } while (0)
    // Horizontal 5-tap [1 4 6 4 1] * M_ on raw bytes with two dp4a per output: output 2k is centred on byte 0 of own
    // word k (taps: bytes 2,3 of the word before, bytes 0..2 of the word), output 2k+1 on byte 2 (bytes 0..3 of the
    // word, byte 0 of the next).  INIT_[j] seeds the accumulators, so vertical weights and sums ride along for free.
#define KLT_HORIZ(W_, M_, INIT_, OUT_)                                                                  \
    _Pragma("unroll") for (int k_ = 0; k_ < NW; ++k_) {                                                 \
        (OUT_)[2 * k_] = dp4a_uu((W_)[k_], 0x04010000u * (M_), dp4a_uu((W_)[k_ + 1], 0x00010406u * (M_), (INIT_)[2 * k_]));          \
        (OUT_)[2 * k_ + 1] = dp4a_uu((W_)[k_ + 1], 0x04060401u * (M_), dp4a_uu((W_)[k_ + 2], 0x00000001u * (M_), (INIT_)[2 * k_ + 1])); \
    }
#define KLT_SLOT(i_) ((uint32_t)((((i_) % kRing + kRing) % kRing) * RC::SLOT))

    KLT_ISSUE(0, KLT_SLOT(0)); KLT_ISSUE(1, KLT_SLOT(1)); KLT_ISSUE(2, KLT_SLOT(2)); KLT_ISSUE(3, KLT_SLOT(3));
    KLT_ISSUE(4, KLT_SLOT(4)); KLT_ISSUE(5, KLT_SLOT(5)); KLT_ISSUE(6, KLT_SLOT(6));
    cp_async_wait<4>();   // rows 0, 1, 2 have landed
    __syncwarp();
    if (fix_right) {      // warp-uniform
        KLT_FIX_RIGHT(KLT_SLOT(0)); KLT_FIX_RIGHT(KLT_SLOT(1)); KLT_FIX_RIGHT(KLT_SLOT(2));
        __syncwarp();
    }
    // Vertical pass as a recurrence over output rows y (h_r = horizontal sum of input row r):
    //   E_y = h_{2y} + 16,  P_y = E_y + 4 h_{2y+1},  V_y = P_{y-1} + P_y + 5 E_y + E_{y+1}
    //       = h_{2y-2} + 4 h_{2y-1} + 6 h_{2y} + 4 h_{2y+1} + h_{2y+2} + 128;   dst = V_y >> 8   (V_y <= 65408)
    // Every input row gets exactly one horizontal pass; the x4 of the odd rows is folded into the dp4a coefficients.
    uint32_t e_cur[NOUT], p_prev[NOUT], k16[NOUT];
#pragma unroll
    for (int i = 0; i < NOUT; ++i) k16[i] = 16u;
    {
        uint32_t wa[NW + 2], wb[NW + 2], wc[NW + 2], e_m1[NOUT];
        KLT_LOAD_ROW(KLT_SLOT(0), wa);
        KLT_LOAD_ROW(KLT_SLOT(1), wb);
        KLT_LOAD_ROW(KLT_SLOT(2), wc);
        KLT_HORIZ(wa, 1u, k16, e_m1);
        KLT_HORIZ(wb, 4u, e_m1, p_prev);
        KLT_HORIZ(wc, 1u, k16, e_cur);
    }
    const int xo = cb >> 1;
    uint8_t* __restrict__ drow = dimg + (long long)y0 * dpitch + xo;
    const bool full_store = (xo + NOUT <= dw);
    const int n_out = y1 - y0;

    // one output row; K_ = t % 4 fixes every ring slot offset at compile time (rows 2t+3, 2t+4 are consumed, rows
    // 2t+7, 2t+8 are issued into the slots of rows 2t-1, 2t, last read two iterations ago)
#define KLT_STEP(K_, FIX_)                                                                                \
    do {                                                                                                \
        cp_async_wait<2>(); /* rows <= 2t+4 have landed; the two newest groups may still be in flight */ \
        __syncwarp();                                                                                   \
        if (FIX_) {                                                                                     \
            KLT_FIX_RIGHT(KLT_SLOT(2 * (K_) + 3)); KLT_FIX_RIGHT(KLT_SLOT(2 * (K_) + 4));               \
            __syncwarp();                                                                               \
        }                                                                                               \
        uint32_t wo[NW + 2], we[NW + 2];                                                                \
        KLT_LOAD_ROW(KLT_SLOT(2 * (K_) + 3), wo);                                                       \
        KLT_LOAD_ROW(KLT_SLOT(2 * (K_) + 4), we);                                                       \
        KLT_ISSUE(2 * t + 7, KLT_SLOT(2 * (K_) + 7));                                                   \
        KLT_ISSUE(2 * t + 8, KLT_SLOT(2 * (K_) + 8));                                                   \
        uint32_t p_cur[NOUT], e_nxt[NOUT], v_[NOUT];                                                    \
        KLT_HORIZ(wo, 4u, e_cur, p_cur);                                                                \
        KLT_HORIZ(we, 1u, k16, e_nxt);                                                                  \
        _Pragma("unroll") for (int i = 0; i < NOUT; ++i) {                                              \
            v_[i] = (5u * e_cur[i] + p_cur[i]) + (p_prev[i] + e_nxt[i]);                                \
            p_prev[i] = p_cur[i];                                                                       \
            e_cur[i] = e_nxt[i];                                                                        \
        }                                                                                               \
        if (full_store) {                                                                               \
            /* byte 1 of every V: pair two V's into one word (V < 2^16), then one PRMT per 4 outputs */ \
            if constexpr (NOUT == 8) {                                                                  \
                uint2 o;                                                                                \
                o.x = prmt(v_[1] * 65536u + v_[0], v_[3] * 65536u + v_[2], 0x7531u);                    \
                o.y = prmt(v_[5] * 65536u + v_[4], v_[7] * 65536u + v_[6], 0x7531u);                    \
                *reinterpret_cast<uint2*>(drow) = o;                                                    \
            } else {                                                                                    \
                *reinterpret_cast<uint32_t*>(drow) = prmt(v_[1] * 65536u + v_[0], v_[3] * 65536u + v_[2], 0x7531u); \
            }                                                                                           \
        } else {                                                                                        \
            _Pragma("unroll") for (int i = 0; i < NOUT; ++i)                                            \
                if (xo + i < dw) drow[i] = (uint8_t)(v_[i] >> 8);                                       \
        }                                                                                               \
        drow += dpitch;                                                                                 \
        ++t;                                                                                            \
    } while (0)

#define KLT_LOOP(FIX_)                                                                                  \
    for (int t = 0; t < n_out;) {                                                                       \
        KLT_STEP(0, FIX_);                                                                              \
        if (t >= n_out) break;                                                                          \
        KLT_STEP(1, FIX_);                                                                              \
        if (t >= n_out) break;                                                                          \
        KLT_STEP(2, FIX_);                                                                              \
        if (t >= n_out) break;                                                                          \
        KLT_STEP(3, FIX_);                                                                              \
    }
    // the right-edge patch is needed by the last tile of a row only: keep it (and its warp barrier) out of the others
    if (fix_right) { KLT_LOOP(true) } else { KLT_LOOP(false) }
#undef KLT_LOOP
    cp_async_wait<0>();
#undef KLT_STEP
#undef KLT_SLOT
#undef KLT_ISSUE
#undef KLT_FIX_RIGHT
#undef KLT_LOAD_ROW
#undef KLT_HORIZ
}

// Tiles of one image row: n8 full 512-column tiles (8 outputs per lane), then at most one remainder tile that uses
// 4 outputs per lane when the remainder fits 256 columns (KITTI: 1241 = 2 x 512 + 217 -> 97 % of the lanes busy
// instead of 81 % with three 512-column tiles).
__global__ void __launch_bounds__(kWarpsPerBlock * 32, kRingCtasPerSm)
pyr_down_ring_kernel(const uint8_t* __restrict__ src, int w, int h, long long spitch, long long sbatch,
                     uint8_t* __restrict__ dst, int dw, int dh, long long dpitch, long long dbatch,
                     int rows_per_strip, int tiles_x, int n8, int rem_nout, int strips_y, long long n_tasks)
{
    extern __shared__ __align__(128) uint8_t ring_smem[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const long long task = (long long)blockIdx.x * kWarpsPerBlock + warp;
    if (task >= n_tasks) return;  // warp-uniform; no block-level barriers in this kernel
    const int tx = (int)(task % tiles_x);
    const long long t2 = task / tiles_x;
    const int sy = (int)(t2 % strips_y);
    const int b = (int)(t2 / strips_y);
    const uint8_t* __restrict__ simg = src + (long long)b * sbatch;
    uint8_t* __restrict__ dimg = dst + (long long)b * dbatch;
    const uint32_t ring_s = (uint32_t)__cvta_generic_to_shared(ring_smem) + (uint32_t)(warp * RingCfg<8>::WARP_BYTES);
    const int X0 = tx * RingCfg<8>::BODY;
    const int y0 = sy * rows_per_strip;
    const int y1 = min(y0 + rows_per_strip, dh);
    if (tx < n8 || rem_nout == 8) ring_task<8>(simg, w, h, spitch, dimg, dw, dpitch, X0, y0, y1, ring_s, lane);
    else ring_task<4>(simg, w, h, spitch, dimg, dw, dpitch, X0, y0, y1, ring_s, lane);
}

// Strip height: every warp task costs about (2*rows + 3 input rows + pipeline fill); tasks run in rounds of `resident`
// warps.  Pick the height that minimises rounds x task cost -- tall strips amortise the 3 halo rows, but a nearly empty
// last round is pure loss.
int ring_rows(int dh, int tiles_x, int batch, long long resident)
{
    int rows = 2;
    double best = 1e300;
    for (int r = 2; r <= 48; ++r) {
        const int strips = (dh + r - 1) / r;
        const int rr = (dh + strips - 1) / strips;   // balanced strips of that count
        const long long tasks = (long long)tiles_x * strips * batch;
        const long long rounds = (tasks + resident - 1) / resident;
        const double cost = (double)rounds * (2.0 * rr + 3.0 + 6.0);
        if (cost < best) { best = cost; rows = rr; }
    }
    return rows;
}

klt_status launch_ring(const uint8_t* src, int w, int h, long long spitch, long long sbatch, uint8_t* dst,
                       int dw, int dh, long long dpitch, long long dbatch, int batch, int sm_count, cudaStream_t stream)
{
    using RC = RingCfg<8>;
    static PerDeviceOnce configured;
    const int smem = RC::WARP_BYTES * kWarpsPerBlock;
    if (configured.needed()) {
        cudaError_t e = cudaFuncSetAttribute(pyr_down_ring_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return (klt_status)e;
    }
    const int n8 = w / RC::BODY, rem = w - n8 * RC::BODY;
    const int rem_nout = (rem == 0) ? 0 : (rem <= RingCfg<4>::BODY ? 4 : 8);
    const int tiles_x = n8 + (rem > 0);
    const int rows = ring_rows(dh, tiles_x, batch, (long long)sm_count * kRingCtasPerSm * kWarpsPerBlock);
    const int strips_y = (dh + rows - 1) / rows;
    const long long n_tasks = (long long)tiles_x * strips_y * batch;
    const long long blocks = (n_tasks + kWarpsPerBlock - 1) / kWarpsPerBlock;
    if (blocks <= 0 || blocks > 0x7fffffffLL) return KLT_ERR_UNSUPPORTED;
    pyr_down_ring_kernel<<<(unsigned)blocks, kWarpsPerBlock * 32, smem, stream>>>(
        src, w, h, spitch, sbatch, dst, dw, dh, dpitch, dbatch, rows, tiles_x, n8, rem_nout, strips_y, n_tasks);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KLT_OK : (klt_status)e;
}

// ---------------------------------------------------------------------------------------------------
// Whole pyramid in ONE launch.  The task list is [all tasks of level 0 -> 1 | all of 1 -> 2 | ...] over the same warp
// tasks as pyr_down_ring_kernel; a task of step l >= 1 first waits until the strips of level l that hold its input rows
// are complete: every producer task ends with fence + one atomicAdd on its (image, strip) counter, and a counter is
// complete at gen * tiles_x (gen = launches so far on this counter array, so nothing is zeroed between launches).
// gen comes from the host, or -- for launches recorded into a CUDA graph -- from a device-side count (see DEVGEN below).
// Producers always have lower task indices than their consumers and CTAs are dispatched in index order, and a waiting
// warp holds no resource a producer needs, so the wait cannot deadlock; it is bounded anyway.
// Why: the small levels are launch- and tail-bound on their own (level 1 -> 2: 40 %, 2 -> 3: 18 % of the copy peak for
// 310 KITTI frames, 3 x 4 us of launch latency for a single pair); in one grid they run in the shadow of level 0 -> 1.
template <bool DEVGEN>
__global__ void __launch_bounds__(kWarpsPerBlock * 32, kRingCtasPerSm)
pyr_build_fused_kernel(const __grid_constant__ PyrFused P)
{
    extern __shared__ __align__(128) uint8_t ring_smem[];
    __shared__ unsigned cta_done;   // finished tasks of this CTA (see sign_off)
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const long long task = (long long)blockIdx.x * kWarpsPerBlock + warp;
    if constexpr (DEVGEN) {
        if (threadIdx.x == 0) cta_done = 0u;
        __syncthreads();            // the only block-level barrier of the kernel: before any warp leaves
    }
    if (task >= P.n_tasks) return;  // warp-uniform
    int l = 0;
    while (l + 1 < P.n_steps && task >= P.s[l + 1].task_begin) ++l;
    const PyrStep& S = P.s[l];
    const long long local = task - S.task_begin;
    const int tx = (int)(local % S.tiles_x);
    const long long t2 = local / S.tiles_x;
    const int sy = (int)(t2 % S.strips_y);
    const int b = (int)(t2 / S.strips_y);
    const int y0 = sy * S.rows;
    const int y1 = min(y0 + S.rows, S.dh);
    // Number of this launch on the counter array.  Ordinary launches get it from the host (P.gen).  Launches recorded into a
    // CUDA graph (DEVGEN) must not carry host-side state: they derive it from P.done, which counts the CTAs that have
    // finished in ALL launches so far (64 bits: never wraps) -- every launch on this array has the same grid, the previous
    // launches are complete when this one starts, and the count cannot reach the next multiple of the grid size while a task
    // is still running, so done / gridDim.x is the number of completed launches for every task of this launch.  (Costs 3 %
    // on the 310-image build, hence the two forms; they use separate counter arrays.)
    unsigned gen = P.gen;
    if constexpr (DEVGEN) {
        if (l > 0) gen = (unsigned)(*reinterpret_cast<const volatile unsigned long long*>(P.done) / gridDim.x) + 1u;
    }
    // DEVGEN: tasks are counted per CTA in shared memory; the last warp of a CTA adds the CTA to the global count
    auto sign_off = [&]() {
        if constexpr (DEVGEN) {
            if (lane == 0) {
                const long long first = (long long)blockIdx.x * kWarpsPerBlock;
                const unsigned cta_tasks = (unsigned)min((long long)kWarpsPerBlock, P.n_tasks - first);
                if (atomicAdd(&cta_done, 1u) == cta_tasks - 1u) atomicAdd(P.done, 1ull);   // (only counted: the kernel boundary orders the data)
            }
        }
    };
    if (P.hash_new != nullptr) {
        if (task == 0 && lane == 0) { P.hash_clear[0] = 0u; P.hash_clear[1] = 0u; P.hash_clear[2] = 0u; P.hash_clear[3] = 0u; }
        // unchanged image (same content hash as the one this item's levels were built from): leave the item alone.  All
        // tasks of the item take the same decision; the completion counter still advances so that later launches agree.
        if (b < 32 && ((P.reuse_mask >> b) & 1u) && P.hash_new[2 * b] == P.hash_old[2 * b] && P.hash_new[2 * b + 1] == P.hash_old[2 * b + 1]) {
            if (lane == 0) {
                if (l + 1 < P.n_steps) atomicAdd(P.cnt + S.cnt_off + (long long)b * S.strips_y + sy, 1u);
                if (l == 0 && tx == 0 && sy == 0 && P.skipped) atomicAdd(P.skipped, 1ull);
            }
            sign_off();
            return;
        }
    }
    if (l > 0) {
        const PyrStep& Q = P.s[l - 1];              // produced this step's source level
        const int s_lo = max(2 * y0 - 2, 0) / Q.rows;
        const int s_hi = min(min(2 * y1, S.h - 1) / Q.rows, Q.strips_y - 1);
        const unsigned target = gen * (unsigned)Q.tiles_x;
        const volatile unsigned* c = P.cnt + Q.cnt_off + (long long)b * Q.strips_y;
        for (int k = s_lo + lane; k <= s_hi; k += 32) {
            int spins = 0;
            while ((int)(c[k] - target) < 0 && ++spins < (1 << 24)) __nanosleep(64);
        }
        __threadfence();
        __syncwarp();
    }
    const uint8_t* __restrict__ simg = S.src + (long long)b * S.sbatch;
    uint8_t* __restrict__ dimg = S.dst + (long long)b * S.dbatch;
    const uint32_t ring_s = (uint32_t)__cvta_generic_to_shared(ring_smem) + (uint32_t)(warp * RingCfg<8>::WARP_BYTES);
    const int X0 = tx * RingCfg<8>::BODY;
    if (tx < S.n8 || S.rem_nout == 8) ring_task<8>(simg, S.w, S.h, S.spitch, dimg, S.dw, S.dpitch, X0, y0, y1, ring_s, lane);
    else ring_task<4>(simg, S.w, S.h, S.spitch, dimg, S.dw, S.dpitch, X0, y0, y1, ring_s, lane);
    if (l + 1 < P.n_steps) {
        __threadfence();                             // this lane's output bytes before the counter
        __syncwarp();
        if (lane == 0) atomicAdd(P.cnt + S.cnt_off + (long long)b * S.strips_y + sy, 1u);
    }
    sign_off();
}

template <int NOUT, bool ALIGNED>
klt_status launch_t(const uint8_t* src, int w, int h, long long spitch, long long sbatch, uint8_t* dst,
                    int dw, int dh, long long dpitch, long long dbatch, int batch, int sm_count,
                    cudaStream_t stream)
{
    const int tiles_x = (dw + 32 * NOUT - 1) / (32 * NOUT);
    // strip height: tall strips amortise the 3 halo rows; shrink them until the grid can fill the chip
    int rows = 16;
    const long long want = (long long)sm_count * kWarpsPerBlock * 4;
    while (rows > 2 && (long long)tiles_x * ((dh + rows - 1) / rows) * batch < want) rows >>= 1;
    const int strips_y = (dh + rows - 1) / rows;
    const long long n_tasks = (long long)tiles_x * strips_y * batch;
    const long long blocks = (n_tasks + kWarpsPerBlock - 1) / kWarpsPerBlock;
    if (blocks <= 0 || blocks > 0x7fffffffLL) return KLT_ERR_UNSUPPORTED;
    pyr_down_kernel<NOUT, ALIGNED><<<(unsigned)blocks, kWarpsPerBlock * 32, 0, stream>>>(
        src, w, h, spitch, sbatch, dst, dw, dh, dpitch, dbatch, rows, tiles_x, strips_y, n_tasks);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KLT_OK : (klt_status)e;
}

// Row repitch: every thread produces 16 destination bytes from 5 aligned source words (funnel shift by the
// source row's byte misalignment).  Used by the host entry points so the H2D transfer can be ONE contiguous DMA per
// image (a pitched 2-D copy of 1241-byte rows runs at a fraction of PCIe speed).
__device__ __forceinline__ unsigned long long mix64(unsigned long long x)
{
    x ^= x >> 30; x *= 0xbf58476d1ce4e5b9ull;
    x ^= x >> 27; x *= 0x94d049bb133111ebull;
    x ^= x >> 31;
    return x;
}

template <bool HASH>
__global__ void __launch_bounds__(256)
repitch_kernel(const uint8_t* __restrict__ src, long long spitch, long long sbatch, uint8_t* __restrict__ dst,
               long long dpitch, long long dbatch, int w, int chunks, int h, unsigned* __restrict__ hash)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int i = blockIdx.y;
    const bool live = t < chunks * h;
    unsigned long long hv = 0ull;
    if (live) {
        const int y = t / chunks, c = t - y * chunks;
        const uint8_t* s = src + (long long)i * sbatch + (long long)y * spitch + 16 * c;
        const uintptr_t a = reinterpret_cast<uintptr_t>(s);
        const uint32_t* wp = reinterpret_cast<const uint32_t*>(a & ~(uintptr_t)3);
        const int sh = (int)(a & 3) * 8;
        const uint32_t w0 = __ldg(wp), w1 = __ldg(wp + 1), w2 = __ldg(wp + 2), w3 = __ldg(wp + 3), w4 = __ldg(wp + 4);
        uint4 o;
        o.x = __funnelshift_r(w0, w1, sh);
        o.y = __funnelshift_r(w1, w2, sh);
        o.z = __funnelshift_r(w2, w3, sh);
        o.w = __funnelshift_r(w3, w4, sh);
        *reinterpret_cast<uint4*>(dst + (long long)i * dbatch + (long long)y * dpitch + 16 * c) = o;
        if constexpr (HASH) {
            // only the w pixels of the row count: the bytes a chunk carries past column w - 1 belong to whatever lies
            // behind the row in the landing zone
            const int valid = min(16, w - 16 * c);
            uint32_t q[4] = {o.x, o.y, o.z, o.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int nb = valid - 4 * k;
                q[k] = nb >= 4 ? q[k] : (nb <= 0 ? 0u : (q[k] & (0xffffffffu >> (8 * (4 - nb)))));
            }
            const unsigned long long pos = (unsigned long long)(unsigned)t + 1ull;
            hv = mix64((((unsigned long long)q[1] << 32) | q[0]) + pos * 0x9e3779b97f4a7c15ull) +
                 mix64((((unsigned long long)q[3] << 32) | q[2]) ^ (pos * 0xc2b2ae3d27d4eb4full + 0x165667b19e3779f9ull));
        }
    }
    if constexpr (HASH) {
        // two independent 32-bit sums (the halves of the 64-bit terms): one REDUX each per warp, combined per block, ONE
        // pair of atomics per block (1800 warps hitting the same two words cost 4.5 us per call; 230 blocks do not)
        __shared__ unsigned s_lo[8], s_hi[8];
        const unsigned lo = __reduce_add_sync(0xffffffffu, (unsigned)(hv & 0xffffffffull));
        const unsigned hi = __reduce_add_sync(0xffffffffu, (unsigned)(hv >> 32));
        if ((threadIdx.x & 31) == 0) { s_lo[threadIdx.x >> 5] = lo; s_hi[threadIdx.x >> 5] = hi; }
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned a = 0, b = 0;
#pragma unroll
            for (int k = 0; k < 8; ++k) { a += s_lo[k]; b += s_hi[k]; }
            if (a | b) {
                atomicAdd(hash + 2 * i, a);
                atomicAdd(hash + 2 * i + 1, b);
            }
        }
    }
}

}  // namespace

klt_status repitch_launch(const uint8_t* src, long long spitch, long long sbatch, uint8_t* dst, long long dpitch,
                          long long dbatch, int w, int h, int n_img, cudaStream_t stream, unsigned* hash)
{
    if (!src || !dst || w <= 0 || h <= 0 || n_img <= 0 || n_img > 65535) return KLT_ERR_INVALID_ARG;
    if ((((uintptr_t)dst | (uintptr_t)dpitch | (uintptr_t)dbatch) & 15) != 0 || dpitch < (w + 15) / 16 * 16) return KLT_ERR_INVALID_ARG;
    const int chunks = (w + 15) / 16;
    if ((long long)chunks * h > 0x7fffff00LL) return KLT_ERR_UNSUPPORTED;
    dim3 grid((unsigned)(((long long)chunks * h + 255) / 256), n_img, 1);
    if (hash) repitch_kernel<true><<<grid, 256, 0, stream>>>(src, spitch, sbatch, dst, dpitch, dbatch, w, chunks, h, hash);
    else repitch_kernel<false><<<grid, 256, 0, stream>>>(src, spitch, sbatch, dst, dpitch, dbatch, w, chunks, h, nullptr);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KLT_OK : (klt_status)e;
}

klt_status pyr_down_launch(const uint8_t* src, int w, int h, long long spitch, long long sbatch,
                           uint8_t* dst, long long dpitch, long long dbatch, int batch, int sm_count,
                           cudaStream_t stream)
{
    if (!src || !dst || w <= 0 || h <= 0 || batch <= 0 || spitch < w) return KLT_ERR_INVALID_ARG;
    const int dw = (w + 1) / 2, dh = (h + 1) / 2;
    if (dpitch < dw) return KLT_ERR_INVALID_ARG;
    const bool aligned = (((uintptr_t)src | (uintptr_t)spitch | (uintptr_t)sbatch) % 16 == 0) &&
                         (((uintptr_t)dst | (uintptr_t)dpitch | (uintptr_t)dbatch) % 8 == 0);
    // 8 outputs per lane (128-bit loads) unless the 256-wide warp tile would waste > 1/4 of its lanes
    const int t8 = (dw + 255) / 256 * 256, t4 = (dw + 127) / 128 * 128;
    const bool use8 = (t8 * 3 <= dw * 4) || (t8 == t4);
    static const char* force_fallback = getenv("KLT_PYR_FALLBACK");   // tests: exercise the shuffle/gather kernel
    if (aligned && w >= 4 && h >= 3 && (long long)h * spitch < 0x7fffffffLL && !(force_fallback && force_fallback[0] == '1'))
        return launch_ring(src, w, h, spitch, sbatch, dst, dw, dh, dpitch, dbatch, batch, sm_count, stream);
    if (aligned) {
        return use8 ? launch_t<8, true>(src, w, h, spitch, sbatch, dst, dw, dh, dpitch, dbatch, batch, sm_count, stream)
                    : launch_t<4, true>(src, w, h, spitch, sbatch, dst, dw, dh, dpitch, dbatch, batch, sm_count, stream);
    }
    return launch_t<4, false>(src, w, h, spitch, sbatch, dst, dw, dh, dpitch, dbatch, batch, sm_count, stream);
}

// Plans the one-launch pyramid build (n_steps pyrDown steps; step i: src[i] -> dst[i], dst[i] == src[i + 1]).  Returns the
// number of counters the launch needs in *n_counters (layout valid for this geometry only), KLT_ERR_UNSUPPORTED when a
// level cannot take the ring kernel (unaligned rows, tiny images) -- the caller then launches level by level.
klt_status pyr_fused_plan(PyrFused& P, int n_steps, const uint8_t* const* src, uint8_t* const* dst, const int* w, const int* h,
                          const long long* spitch, const long long* sbatch, const long long* dpitch, const long long* dbatch,
                          int batch, int sm_count, long long* n_counters)
{
    if (n_steps < 1 || n_steps > KLT_MAX_LEVELS - 1 || batch <= 0) return KLT_ERR_UNSUPPORTED;
    using RC = RingCfg<8>;
    const long long resident = (long long)sm_count * kRingCtasPerSm * kWarpsPerBlock;
    long long tasks = 0, counters = 0;
    for (int i = 0; i < n_steps; ++i) {
        PyrStep& S = P.s[i];
        const bool aligned = (((uintptr_t)src[i] | (uintptr_t)spitch[i] | (uintptr_t)sbatch[i]) % 16 == 0) &&
                             (((uintptr_t)dst[i] | (uintptr_t)dpitch[i] | (uintptr_t)dbatch[i]) % 8 == 0);
        if (!aligned || w[i] < 4 || h[i] < 3 || (long long)h[i] * spitch[i] >= 0x7fffffffLL) return KLT_ERR_UNSUPPORTED;
        S.src = src[i]; S.dst = dst[i];
        S.spitch = spitch[i]; S.sbatch = sbatch[i]; S.dpitch = dpitch[i]; S.dbatch = dbatch[i];
        S.w = w[i]; S.h = h[i]; S.dw = (w[i] + 1) / 2; S.dh = (h[i] + 1) / 2;
        S.n8 = w[i] / RC::BODY;
        const int rem = w[i] - S.n8 * RC::BODY;
        S.rem_nout = (rem == 0) ? 0 : (rem <= RingCfg<4>::BODY ? 4 : 8);
        S.tiles_x = S.n8 + (rem > 0);
        S.rows = ring_rows(S.dh, S.tiles_x, batch, resident);
        S.strips_y = (S.dh + S.rows - 1) / S.rows;
        S.task_begin = tasks;
        S.cnt_off = (int)counters;
        tasks += (long long)S.tiles_x * S.strips_y * batch;
        if (i + 1 < n_steps) counters += (long long)S.strips_y * batch;
        if (counters > 0x7fffffffLL) return KLT_ERR_UNSUPPORTED;
    }
    P.n_steps = n_steps; P.batch = batch; P.n_tasks = tasks;
    P.hash_new = nullptr; P.hash_old = nullptr; P.hash_clear = nullptr; P.skipped = nullptr; P.reuse_mask = 0u;
    P.gen = 0u; P.done = nullptr;
    *n_counters = counters;
    return KLT_OK;
}

klt_status pyr_fused_launch(const PyrFused& P, bool device_gen, cudaStream_t stream)
{
    using RC = RingCfg<8>;
    static PerDeviceOnce configured;
    const int smem = RC::WARP_BYTES * kWarpsPerBlock;
    if (configured.needed()) {
        cudaError_t e = cudaFuncSetAttribute(pyr_build_fused_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(pyr_build_fused_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return (klt_status)e;
    }
    const long long blocks = (P.n_tasks + kWarpsPerBlock - 1) / kWarpsPerBlock;
    if (blocks <= 0 || blocks > 0x7fffffffLL) return KLT_ERR_UNSUPPORTED;
    if (device_gen) pyr_build_fused_kernel<true><<<(unsigned)blocks, kWarpsPerBlock * 32, smem, stream>>>(P);
    else pyr_build_fused_kernel<false><<<(unsigned)blocks, kWarpsPerBlock * 32, smem, stream>>>(P);
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KLT_OK : (klt_status)e;
}

}  // namespace klt
