// Per-point scalar arithmetic of pyramidal LK (SURVEY.md A.4), shared by the generic kernel (klt_lk.cu) and the
// specialised one (klt_lk_fast.cu).  Bit-exactness with cv2.calcOpticalFlowPyrLK rests on these lines: every float op
// rounds once (no FMA contraction: -fmad=false), in OpenCV's order.
#pragma once
#include "klt_common.cuh"

namespace klt {

constexpr unsigned kFull = 0xffffffffu;
// While every partial sum stays <= 2^24 in magnitude, OpenCV's float32 accumulation is exact and equals the integer sum.
constexpr int kExact = 1 << 24;

__device__ __forceinline__ int lo16(uint32_t w) { return (int)(short)(w & 0xffffu); }
__device__ __forceinline__ int hi16(uint32_t w) { return ((int)w) >> 16; }

// A.4 step 1: the point and the initial iterate at `level` (2^-level scaling is exact); outp becomes the iterate.
__device__ __forceinline__ void level_start(float2 p0, float2& outp, int level, int top, int flags, float& px, float& py,
                                            float& nx, float& ny)
{
    const float scale = __int_as_float((127 - level) << 23);
    px = __fmul_rn(p0.x, scale); py = __fmul_rn(p0.y, scale);
    if (level == top) {
        if (flags & KLT_OPTFLOW_USE_INITIAL_FLOW) { nx = __fmul_rn(outp.x, scale); ny = __fmul_rn(outp.y, scale); }
        else { nx = px; ny = py; }
    } else {
        nx = __fmul_rn(outp.x, 2.f); ny = __fmul_rn(outp.y, 2.f);
    }
    outp = make_float2(nx, ny);
}

// cvFloor + the window range test of A.4 step 2 (NaN / huge coordinates count as out of range)
__device__ __forceinline__ bool floor_in_range(float x, float y, int win_w, int win_h, int lw, int lh, int& ix, int& iy)
{
    const bool finite = (fabsf(x) < 1.0e9f) && (fabsf(y) < 1.0e9f);
    ix = finite ? __float2int_rd(x) : INT_MIN;
    iy = finite ? __float2int_rd(y) : INT_MIN;
    return finite && !(ix < -win_w || ix >= lw || iy < -win_h || iy >= lh);
}

// The same for coordinates known to be finite: a conversion that saturates (|x| >= 2^31) still lands outside the range.
__device__ __forceinline__ bool floor_in_range_finite(float x, float y, int win_w, int win_h, int lw, int lh, int& ix, int& iy)
{
    ix = __float2int_rd(x);
    iy = __float2int_rd(y);
    return !(ix < -win_w || ix >= lw || iy < -win_h || iy >= lh);
}

// A.4 step 3: Q14 bilinear weights from the fractional position.  OpenCV rounds (x * y) * 2^14; x * (y * 2^14) is the same
// bit for bit, since scaling by a power of two commutes with rounding (nothing here under- or overflows).
__device__ __forceinline__ void q14_weights(float a, float b, int& w00, int& w01, int& w10, int& w11)
{
    const float oa = __fsub_rn(1.f, a), ob = __fmul_rn(__fsub_rn(1.f, b), 16384.f), bb = __fmul_rn(b, 16384.f);
    w00 = __float2int_rn(__fmul_rn(oa, ob));
    w01 = __float2int_rn(__fmul_rn(a, ob));
    w10 = __float2int_rn(__fmul_rn(oa, bb));
    w11 = 16384 - w00 - w01 - w10;
}

// A.5 final combine: t + ((q0 + q2) + (q1 + q3)), then * 2^-20
__device__ __forceinline__ float combine5(float q0, float q1, float q2, float q3, float t)
{
    const float s = __fadd_rn(__fadd_rn(q0, q2), __fadd_rn(q1, q3));
    return __fmul_rn(__fadd_rn(t, s), 9.5367431640625e-07f);
}

// A.4 step 5: minimum-eigenvalue gate (its value is the err output under KLT_OPTFLOW_LK_GET_MIN_EIGENVALS) and the
// determinant test.  Returns false when OpenCV drops the point at this level, else sets inv_det = 1 / det(G).
__device__ __forceinline__ bool eig_gate(float A11, float A12, float A22, int win_w, int win_h, int flags, float min_eig_thr,
                                         float& err, float& inv_det)
{
    const float D = __fsub_rn(__fmul_rn(A11, A22), __fmul_rn(A12, A12));
    const float dA = __fsub_rn(A11, A22);
    const float rad = __fsqrt_rn(__fadd_rn(__fmul_rn(dA, dA), __fmul_rn(__fmul_rn(4.f, A12), A12)));
    const float min_eig = __fdiv_rn(__fsub_rn(__fadd_rn(A22, A11), rad), (float)(2 * win_w * win_h));
    if (flags & KLT_OPTFLOW_LK_GET_MIN_EIGENVALS) err = min_eig;
    if (min_eig < min_eig_thr || D < 1.1920929e-7f) return false;
    inv_det = __fdiv_rn(1.f, D);
    return true;
}

// A.4 step 6: one Newton step of the window-corner iterate (nx, ny) from the mismatch vector (b1, b2); outp is the centre.
// Returns true when the iteration ends: step below eps (LKLaunch::eps2 and its float brackets), or the step of iteration
// j > 0 undoes the previous one (then outp takes half of it back).  (pdx, pdy) carries the previous step.
// The launch fields are passed by value: a reference into the kernel's parameter block changes the code ptxas emits.
__device__ __forceinline__ bool newton_step(float A11, float A12, float A22, float inv_det, float b1, float b2, int j,
                                            float eps2_lo, float eps2_hi, double eps2, float hwx, float hwy, float& nx,
                                            float& ny, float& pdx, float& pdy, float2& outp)
{
    const float dx = __fmul_rn(__fsub_rn(__fmul_rn(A12, b2), __fmul_rn(A22, b1)), inv_det);
    const float dy = __fmul_rn(__fsub_rn(__fmul_rn(A12, b1), __fmul_rn(A11, b2)), inv_det);
    nx = __fadd_rn(nx, dx); ny = __fadd_rn(ny, dy);
    outp = make_float2(__fadd_rn(nx, hwx), __fadd_rn(ny, hwy));
    {   // termination tests of A.4 6f / 6g without double-precision instructions on the common path
        const float s2f = __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
        bool small = s2f <= eps2_lo;
        if (!small && !(s2f >= eps2_hi))
            small = __dadd_rn(__dmul_rn((double)dx, (double)dx), __dmul_rn((double)dy, (double)dy)) <= eps2;
        if (small) return true;
    }
    // (double)f < 0.01  <=>  f <= 0.01f: the float nearest to 0.01 lies below it, the next float above it
    if (j > 0 && fabsf(__fadd_rn(dx, pdx)) <= 0.01f && fabsf(__fadd_rn(dy, pdy)) <= 0.01f) {
        outp.x = __fsub_rn(outp.x, __fmul_rn(dx, 0.5f));
        outp.y = __fsub_rn(outp.y, __fmul_rn(dy, 0.5f));
        return true;
    }
    pdx = dx; pdy = dy;
    return false;
}

// A.4 step 7: err at level 0 from sum |J - I| over the window (Q5 intensities)
__device__ __forceinline__ float lk_err(float sum_abs, int win_w, int win_h)
{
    return __fdiv_rn(__fmul_rn(sum_abs, 1.f), (float)(32 * win_w * win_h));
}

}  // namespace klt
