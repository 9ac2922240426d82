/*
 * subpix_oracle.c -- CPU restatement of cv2.cornerSubPix(image, corners, winSize, zeroZone, criteria) for 8-bit
 * single-channel images.  TEST INFRASTRUCTURE, NOT PRODUCT CODE: only tests/ and scripts/ may load it.
 *
 * The arithmetic lives in OpenCV (imgproc/src/cornersubpix.cpp, imgproc/src/samplers.cpp).  Restated here, every float
 * operation rounded once (no FMA; oracle/subpix_oracle.py compiles it with -ffp-contract=off, as oracle/Makefile does the
 * other oracles):
 *   S.1  win = (wx, wy), patch W = 2wx + 1 by H = 2wy + 1.  Criteria: max_iters = clamp(maxCount, 1, 100) with
 *        TERM_COUNT, else 100; eps = max(epsilon, 0) with TERM_EPS, else 0; then eps = eps * eps (double).
 *   S.2  weight mask, float32, with the C library's expf:  y = (float)(i - wy) / wy,  vy = expf(-y * y),
 *        x = (float)(j - wx) / wx,  mask[i][j] = vy * expf(-x * x).  Zero zone (zx, zy): when zx >= 0, zy >= 0,
 *        2zx + 1 < W and 2zy + 1 < H, mask = 0 on rows wy - zy .. wy + zy, columns wx - zx .. wx + zx.
 *   S.3  per point cT (cv2 asserts 0 <= x < cols and 0 <= y < rows in float: NaN fails), cI = cT, iter = 0; loop:
 *        a. buf = getRectSubPix(img, (W + 2, H + 2), cI) as float32 (S.5 / S.6);
 *        b. for i < H (py = i - wy), j < W (px = j - wx), row-major, with v = buf[i + 1][j + 1]:
 *             tgx = (double)(buf[i+1][j+2] - buf[i+1][j])   (float subtraction, then widened)
 *             tgy = (double)(buf[i+2][j+1] - buf[i][j+1])
 *             m = mask[i][j];  gxx = tgx * tgx * m;  gxy = tgx * tgy * m;  gyy = tgy * tgy * m   (left to right)
 *             a += gxx;  b += gxy;  c += gyy;  bb1 += gxx * px + gxy * py;  bb2 += gxy * px + gyy * py   (double)
 *        c. det = a * c - b * b; |det| <= DBL_EPSILON^2: stop (cI unchanged);
 *        d. scale = 1.0 / det;  x' = (float)(cI.x + c * scale * bb1 - b * scale * bb2),
 *           y' = (float)(cI.y - b * scale * bb1 + a * scale * bb2)   (double, each product left to right);
 *        e. err = (x' - cI.x)^2 + (y' - cI.y)^2 in float;  stop if x' < 0 || x' >= cols || y' < 0 || y' >= rows
 *           (cI unchanged: a step out of the image is not taken);  cI = (x', y');
 *        f. ++iter; continue while iter < max_iters && err > eps.
 *   S.4  if |cI.x - cT.x| > wx or |cI.y - cT.y| > wy (float): the result is cT, else cI.
 *   S.5  getRectSubPix, (pw, ph) = (W + 2, H + 2), centre (cx, cy) float:  cx -= (pw - 1) * 0.5f, cy -= (ph - 1) * 0.5f,
 *        ix = floor(cx), iy = floor(cy), ax = cx - ix, by = cy - iy (float).  Interior when 0 <= ix, ix + pw < cols,
 *        0 <= iy, iy + ph < rows (getRectSubPix_8u32f):  a = max(ax, 0.0001f), a12 = a * (1 - by), a22 = a * by,
 *        b1 = 1 - by, b2 = by, s = (1.0 - a) / a (double); per row r with p0 = img[iy + r], p1 = img[iy + r + 1]:
 *          prev = (1 - a) * (b1 * p0[ix] + b2 * p1[ix]);  for j < pw:  t = a12 * p0[ix + j + 1] + a22 * p1[ix + j + 1],
 *          out[r][j] = prev + t,  prev = (float)(t * s).
 *   S.6  otherwise (getRectSubPix_Cn_ with adjustRect; no 0.0001 floor): a11 = (1 - ax)(1 - by), a12 = ax (1 - by),
 *        a21 = (1 - ax) by, a22 = ax by, b1 = 1 - by, b2 = by.  Columns: rx = min(-ix, pw) when ix < 0, else 0;
 *        rw = pw when ix < cols - pw, else cols - ix - 1 (when negative, the base moves left by it and rw = 0); the source
 *        column of patch column j is base + j.  Rows: ry = -iy when iy < 0, else 0; rh = ph when iy < rows - ph, else
 *        rows - iy - 1 (likewise); row r reads rows s and s2 = s + 1, or s2 = s when r < ry or r >= rh; after the row
 *        s = s2 when r < rh.  Per row: columns j < rx get src[rx] * b1 + src2[rx] * b2, columns j >= rw get
 *        src[rw] * b1 + src2[rw] * b2 (written after the first, so it wins where both apply), the rest
 *        src[j] * a11 + src[j + 1] * a12 + src2[j] * a21 + src2[j + 1] * a22 (left to right).
 * Pinned bit-for-bit against live cv2.cornerSubPix with cv2.ipp.setUseIPP(False), OpenCV's own code path; the default
 * wheel routes S.5 / S.6 through IPP, whose patch differs in the last bits (tolerance test in tests/test_subpix_cpu.py).
 */
#include <float.h>
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

/* S.5 + S.6: getRectSubPix(img, (pw, ph), (cx, cy), CV_32F) -> out[ph][pw] */
static void rect_sub_pix(const uint8_t* img, int w, int h, int64_t pitch, int pw, int ph, float cx, float cy, float* out)
{
    cx -= (pw - 1) * 0.5f;
    cy -= (ph - 1) * 0.5f;
    const int ix = (int)floorf(cx), iy = (int)floorf(cy);
    if (0 <= ix && ix + pw < w && 0 <= iy && iy + ph < h) {
        float a = cx - (float)ix;
        const float b = cy - (float)iy;
        if (a < 0.0001f) a = 0.0001f;
        const float a12 = a * (1.f - b), a22 = a * b, b1 = 1.f - b, b2 = b;
        const double s = (1. - a) / a;
        for (int r = 0; r < ph; ++r) {
            const uint8_t* p0 = img + (int64_t)(iy + r) * pitch + ix;
            const uint8_t* p1 = p0 + pitch;
            float prev = (1 - a) * (b1 * (float)p0[0] + b2 * (float)p1[0]);
            for (int j = 0; j < pw; ++j) {
                const float t = a12 * (float)p0[j + 1] + a22 * (float)p1[j + 1];
                out[r * pw + j] = prev + t;
                prev = (float)(t * s);
            }
        }
        return;
    }
    const float a = cx - (float)ix, b = cy - (float)iy;
    const float a11 = (1.f - a) * (1.f - b), a12 = a * (1.f - b), a21 = (1.f - a) * b, a22 = a * b;
    const float b1 = 1.f - b, b2 = b;
    /* adjustRect: `col` / `row` are the image column and row of src[0] */
    int col, row, rx, rw, ry, rh;
    if (ix >= 0) { col = ix; rx = 0; }
    else { col = 0; rx = -ix; if (rx > pw) rx = pw; }
    if (ix < w - pw) rw = pw;
    else { rw = w - ix - 1; if (rw < 0) { col += rw; rw = 0; } }
    if (iy >= 0) { row = iy; ry = 0; }
    else { row = 0; ry = -iy; }
    if (iy < h - ph) rh = ph;
    else { rh = h - iy - 1; if (rh < 0) { row += rh; rh = 0; } }
    col -= rx;
    for (int r = 0; r < ph; ++r) {
        const int row2 = (r < ry || r >= rh) ? row : row + 1;
        const uint8_t* s1 = img + (int64_t)row * pitch + col;
        const uint8_t* s2 = img + (int64_t)row2 * pitch + col;
        float* o = out + r * pw;
        float v = (float)s1[rx] * b1 + (float)s2[rx] * b2;
        for (int j = 0; j < rx; ++j) o[j] = v;
        v = (float)s1[rw] * b1 + (float)s2[rw] * b2;
        for (int j = rw; j < pw; ++j) o[j] = v;
        for (int j = rx; j < rw; ++j)
            o[j] = (float)s1[j] * a11 + (float)s1[j + 1] * a12 + (float)s2[j] * a21 + (float)s2[j + 1] * a22;
        if (r < rh) row = row2;
    }
}

/* getRectSubPix alone, for the tests: out[ph][pw] float32 */
int klt_oracle_rect_sub_pix(const uint8_t* img, int w, int h, int64_t pitch, int pw, int ph, float cx, float cy, float* out)
{
    if (!img || !out || w < 1 || h < 1 || pw < 1 || ph < 1 || pitch < w) return -1;
    rect_sub_pix(img, w, h, pitch, pw, ph, cx, cy, out);
    return 0;
}

/* S.2: mask[(2wy + 1)][(2wx + 1)] */
void klt_oracle_subpix_mask(int win_w, int win_h, int zero_w, int zero_h, float* mask)
{
    const int W = 2 * win_w + 1, H = 2 * win_h + 1;
    for (int i = 0; i < H; ++i) {
        const float y = (float)(i - win_h) / (float)win_h;
        const float vy = expf(-y * y);
        for (int j = 0; j < W; ++j) {
            const float x = (float)(j - win_w) / (float)win_w;
            mask[i * W + j] = vy * expf(-x * x);
        }
    }
    if (zero_w >= 0 && zero_h >= 0 && 2 * zero_w + 1 < W && 2 * zero_h + 1 < H)
        for (int i = win_h - zero_h; i <= win_h + zero_h; ++i)
            for (int j = win_w - zero_w; j <= win_w + zero_w; ++j) mask[i * W + j] = 0.f;
}

/* cv2.cornerSubPix on pts[n][2] in place.  Returns 0, -1 for invalid arguments (cv2's assertions on the window and the
 * image size), -2 when a point is outside the image or NaN (cv2 raises; that point and the later ones are left as they
 * are), -4 out of memory.  iters (NULL or [n]): iterations run per point (the number of S.3.a passes). */
int klt_oracle_corner_sub_pix(const uint8_t* img, int w, int h, int64_t pitch, float* pts, int n, int win_w, int win_h,
                              int zero_w, int zero_h, int crit_type, int max_count, double eps, int* iters)
{
    if (!img || (n > 0 && !pts) || n < 0 || pitch < w) return -1;
    if (n == 0) return 0;
    if (win_w < 1 || win_h < 1 || w < 2 * win_w + 5 || h < 2 * win_h + 5) return -1;
    const int max_iters = (crit_type & 1) ? (max_count < 1 ? 1 : max_count > 100 ? 100 : max_count) : 100;
    double eps2 = (crit_type & 2) ? (eps > 0 ? eps : 0.) : 0.;
    eps2 *= eps2;
    const int W = 2 * win_w + 1, H = 2 * win_h + 1, pw = W + 2, ph = H + 2;
    float* mask = (float*)malloc(sizeof(float) * (size_t)W * H);
    float* buf = (float*)malloc(sizeof(float) * (size_t)pw * ph);
    if (!mask || !buf) { free(mask); free(buf); return -4; }
    klt_oracle_subpix_mask(win_w, win_h, zero_w, zero_h, mask);
    int rc = 0;
    for (int p = 0; p < n; ++p) {
        const float tx = pts[2 * p], ty = pts[2 * p + 1];
        if (!(0.f <= tx && tx < (float)w && 0.f <= ty && ty < (float)h)) { rc = -2; break; }
        float cx = tx, cy = ty;
        int iter = 0, passes = 0;
        float err = 0.f;
        do {
            rect_sub_pix(img, w, h, pitch, pw, ph, cx, cy, buf);
            ++passes;
            double a = 0, b = 0, c = 0, bb1 = 0, bb2 = 0;
            for (int i = 0; i < H; ++i) {
                const double py = i - win_h;
                const float* s = buf + (i + 1) * pw + 1;
                for (int j = 0; j < W; ++j) {
                    const double m = mask[i * W + j];
                    const double tgx = s[j + 1] - s[j - 1];
                    const double tgy = s[j + pw] - s[j - pw];
                    const double gxx = tgx * tgx * m, gxy = tgx * tgy * m, gyy = tgy * tgy * m;
                    const double px = j - win_w;
                    a += gxx;
                    b += gxy;
                    c += gyy;
                    bb1 += gxx * px + gxy * py;
                    bb2 += gxy * px + gyy * py;
                }
            }
            const double det = a * c - b * b;
            if (fabs(det) <= DBL_EPSILON * DBL_EPSILON) break;
            const double scale = 1.0 / det;
            const float nx = (float)(cx + c * scale * bb1 - b * scale * bb2);
            const float ny = (float)(cy - b * scale * bb1 + a * scale * bb2);
            err = (nx - cx) * (nx - cx) + (ny - cy) * (ny - cy);
            if (nx < 0 || nx >= (float)w || ny < 0 || ny >= (float)h) break;
            cx = nx; cy = ny;
        } while (++iter < max_iters && err > eps2);
        if (fabsf(cx - tx) > (float)win_w || fabsf(cy - ty) > (float)win_h) { cx = tx; cy = ty; }
        pts[2 * p] = cx; pts[2 * p + 1] = cy;
        if (iters) iters[p] = passes;
    }
    free(mask); free(buf);
    return rc;
}
