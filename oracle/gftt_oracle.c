/*
 * gftt_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * Plain-C, single-threaded CPU restatement of the Shi-Tomasi detection step that the reference
 * (JonasFrey96/Visual-Odom-Pipeline) delegates to OpenCV at
 *     src/extractor/extractor.py:21-24     (maxCorners=1000, qualityLevel=0.03, minDistance, blockSize=31)
 *     src/extractor/extractor.py:102-112   (mask of circles around tracked keypoints, cv2.goodFeaturesToTrack call)
 *     src/pipeline/pipeline.py:159-163     (called once per frame)
 * (SURVEY.md s8f rank 2).  The arithmetic lives in a third-party dependency that is NOT vendored under
 * /root/reference: OpenCV (pinned `opencv=4.4.0`, setup/conda_env.yml:57,78,87): goodFeaturesToTrack
 * (modules/imgproc/src/featureselect.cpp), cornerMinEigenVal (corner.cpp), Sobel / sepFilter2D (deriv.cpp,
 * filter.simd.hpp), boxFilter (box_filter.simd.hpp).  This file restates the published algorithm with the
 * floating-point evaluation order of the x86-64 AVX2 dispatch of the `cv2` wheel in this image (4.13.0), which was
 * established by probing (DESIGN.md s9):
 *   G.1  k1 = (float)(1 / (4 * blockSize * 255)), k0 = 2 * k1; image reflect-101 extended by 1 pixel.
 *   G.2  Dx: r(x,y) = I(x+1,y) - I(x-1,y) (exact); Dx = fmaf(k1, r(x,y-1) + r(x,y+1), k0 * r(x,y)).
 *   G.3  Dy: t(x,y) = fmaf(k1, I(x+1,y), fmaf(k0, I(x,y), k1 * I(x-1,y)))      for x <  32 * (W / 32)   (SIMD part)
 *                   = ((k1 * I(x-1,y) + k0 * I(x,y)) + k1 * I(x+1,y))          for x >= 32 * (W / 32)   (scalar tail)
 *        Dy = t(x,y+1) - t(x,y-1), rows reflect-101.
 *   G.4  cov = (Dx*Dx, Dx*Dy, Dy*Dy), each product rounded to float32.
 *   G.5  boxFilter(blockSize x blockSize, normalize=false, anchor = blockSize/2, reflect-101 of cov) with DOUBLE
 *        running sums in OpenCV's order: per row, for blockSize <= 5 a fresh left-to-right sum of the blockSize values
 *        of every output; for blockSize >= 6  s = sum of the first blockSize values (left to right), then
 *        s += (double)new - (double)old  per step; per column
 *        SUM = sum of the first blockSize-1 row sums (top to bottom), then per output row  s0 = SUM + bottom,
 *        out = (float)s0, SUM = s0 - top.
 *   G.6  a = 0.5f * cxx, b = cxy, c = 0.5f * cyy;  eig = (a + c) - sqrtf((a - c) * (a - c) + b * b)  (no FMA).
 *   G.7  maxVal = max of eig over mask != 0 (0 if the mask is empty); thr = (float)((double)maxVal * qualityLevel);
 *        e = eig > thr ? eig : 0;  candidate at 1 <= x < W-1, 1 <= y < H-1  iff  e != 0, e == max of e over the
 *        3x3 neighbourhood, mask != 0;  candidates sorted by (e descending, y*W+x descending);
 *   G.8  greedy minimum-distance selection on a grid of cells of size cvRound(minDistance) (a candidate is dropped
 *        if an accepted corner in the 3x3 neighbouring cells is closer than minDistance), stop at maxCorners.
 *
 * Parity pinning: the reference has no tests / golden vectors for this path.  The oracle is pinned bit-for-bit
 * against the live `cv2` module (the reference's own implementation) in tests/test_oracle.py and against the
 * committed vectors tests/golden/gftt_*.npz (made by tests/golden/make_golden.py).
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg may load this library.
 * Build: oracle/Makefile (-ffp-contract=off: only the explicit fmaf calls fuse).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

static int refl101(int p, int len)
{
    if (len == 1) return 0;
    while (p < 0 || p >= len) {
        if (p < 0) p = -p;
        else p = 2 * len - 2 - p;
    }
    return p;
}

/* G.1 - G.6: eig must hold w*h floats.  Returns 0, or a negative error. */
int klt_oracle_corner_min_eigen_val(const uint8_t* img, int w, int h, int64_t pitch, int block, float* eig)
{
    if (!img || !eig || w < 1 || h < 1 || block < 1) return -1;
    const float k1 = (float)(1.0 / (4.0 * (double)block * 255.0));
    const float k0 = (float)(2.0 / (4.0 * (double)block * 255.0));
    const size_t n = (size_t)w * (size_t)h;
    float* cov = (float*)malloc(sizeof(float) * 3 * n);              /* planar: cxx, cxy, cyy */
    float* t = (float*)malloc(sizeof(float) * n);                    /* smoothed rows for Dy */
    int* r = (int*)malloc(sizeof(int) * n);                          /* horizontal differences for Dx */
    const int an = block / 2;
    const int pw = w + block - 1, ph = h + block - 1;
    double* rows = (double*)malloc(sizeof(double) * (size_t)h * (size_t)w);
    double* sum = (double*)malloc(sizeof(double) * (size_t)w);
    int* xs = (int*)malloc(sizeof(int) * (size_t)pw);
    int* ys = (int*)malloc(sizeof(int) * (size_t)ph);
    int rc = (cov && t && r && rows && sum && xs && ys) ? 0 : -2;
    if (rc) goto done;

    const int nv = 32 * (w / 32);
    for (int y = 0; y < h; ++y) {
        const uint8_t* s = img + (int64_t)y * pitch;
        for (int x = 0; x < w; ++x) {
            const float L = (float)s[refl101(x - 1, w)], C = (float)s[x], R = (float)s[refl101(x + 1, w)];
            r[(size_t)y * w + x] = (int)s[refl101(x + 1, w)] - (int)s[refl101(x - 1, w)];
            float v;
            if (x < nv) v = fmaf(k1, R, fmaf(k0, C, k1 * L));
            else { v = k1 * L + k0 * C; v = v + k1 * R; }
            t[(size_t)y * w + x] = v;
        }
    }
    for (int y = 0; y < h; ++y) {
        const size_t ym = (size_t)refl101(y - 1, h) * w, yp = (size_t)refl101(y + 1, h) * w, yc = (size_t)y * w;
        for (int x = 0; x < w; ++x) {
            const float dx = fmaf(k1, (float)(r[ym + x] + r[yp + x]), k0 * (float)r[yc + x]);
            const float dy = t[yp + x] - t[ym + x];
            cov[yc + x] = dx * dx;
            cov[n + yc + x] = dx * dy;
            cov[2 * n + yc + x] = dy * dy;
        }
    }
    for (int i = 0; i < pw; ++i) xs[i] = refl101(i - an, w);
    for (int i = 0; i < ph; ++i) ys[i] = refl101(i - an, h);
    for (int c = 0; c < 3; ++c) {
        const float* C = cov + (size_t)c * n;
        /* row sums of every source row (border rows are copies of source rows, so are their sums) */
        for (int y = 0; y < h; ++y) {
            const float* S = C + (size_t)y * w;
            double* D = rows + (size_t)y * w;
            if (block <= 5) {
                for (int x = 0; x < w; ++x) {
                    double s = (double)S[xs[x]];
                    for (int k = 1; k < block; ++k) s += (double)S[xs[x + k]];
                    D[x] = s;
                }
            } else {
                double s = 0;
                for (int i = 0; i < block; ++i) s += (double)S[xs[i]];
                D[0] = s;
                for (int x = 0; x < w - 1; ++x) {
                    s += (double)S[xs[x + block]] - (double)S[xs[x]];
                    D[x + 1] = s;
                }
            }
        }
        float* O = cov + (size_t)c * n;   /* in place: the row sums are complete */
        for (int x = 0; x < w; ++x) sum[x] = 0;
        for (int i = 0; i < block - 1; ++i) {
            const double* Sp = rows + (size_t)ys[i] * w;
            for (int x = 0; x < w; ++x) sum[x] += Sp[x];
        }
        for (int y = 0; y < h; ++y) {
            const double* Sp = rows + (size_t)ys[y + block - 1] * w;
            const double* Sm = rows + (size_t)ys[y] * w;
            for (int x = 0; x < w; ++x) {
                const double s0 = sum[x] + Sp[x];
                O[(size_t)y * w + x] = (float)s0;
                sum[x] = s0 - Sm[x];
            }
        }
    }
    for (size_t i = 0; i < n; ++i) {
        const float a = cov[i] * 0.5f, b = cov[n + i], c = cov[2 * n + i] * 0.5f;
        const float d = a - c;
        const float q = d * d, bb = b * b;
        eig[i] = (a + c) - sqrtf(q + bb);
    }
done:
    free(cov); free(t); free(r); free(rows); free(sum); free(xs); free(ys);
    return rc;
}

typedef struct { float v; int idx; } cand_t;

static int cand_cmp(const void* pa, const void* pb)
{
    const cand_t* a = (const cand_t*)pa;
    const cand_t* b = (const cand_t*)pb;
    if (a->v > b->v) return -1;
    if (a->v < b->v) return 1;
    return a->idx > b->idx ? -1 : (a->idx < b->idx ? 1 : 0);
}

/* G.7 + G.8 on a given eigenvalue map.  corners: capacity * 2 floats (x, y).  Returns the number of corners. */
int klt_oracle_select_corners(const float* eig, int w, int h, const uint8_t* mask, int64_t mask_pitch,
                              int max_corners, double quality, double min_distance, float* corners, int capacity)
{
    if (!eig || w < 1 || h < 1 || quality <= 0 || min_distance < 0 || !corners) return -1;
    const size_t n = (size_t)w * (size_t)h;
    float max_val = 0.f;
    int any = 0;
    for (int y = 0; y < h; ++y)
        for (int x = 0; x < w; ++x)
            if (!mask || mask[(int64_t)y * mask_pitch + x]) {
                const float v = eig[(size_t)y * w + x];
                if (!any || v > max_val) { max_val = v; any = 1; }
            }
    if (!any) max_val = 0.f;
    const float thr = (float)((double)max_val * quality);
    float* e = (float*)malloc(sizeof(float) * n);
    cand_t* cand = (cand_t*)malloc(sizeof(cand_t) * n);
    if (!e || !cand) { free(e); free(cand); return -2; }
    for (size_t i = 0; i < n; ++i) e[i] = eig[i] > thr ? eig[i] : 0.f;
    int total = 0;
    for (int y = 1; y < h - 1; ++y)
        for (int x = 1; x < w - 1; ++x) {
            const float v = e[(size_t)y * w + x];
            if (v == 0.f || (mask && !mask[(int64_t)y * mask_pitch + x])) continue;
            float m = v;
            for (int dy = -1; dy <= 1; ++dy)
                for (int dx = -1; dx <= 1; ++dx) {
                    const float u = e[(size_t)(y + dy) * w + (x + dx)];
                    if (u > m) m = u;
                }
            if (v == m) { cand[total].v = v; cand[total].idx = y * w + x; ++total; }
        }
    qsort(cand, (size_t)total, sizeof(cand_t), cand_cmp);
    int nc = 0;
    if (min_distance >= 1) {
        const int cell = (int)lrint(min_distance);
        const int gw = (w + cell - 1) / cell, gh = (h + cell - 1) / cell;
        const double md2 = min_distance * min_distance;   /* compared in double, like OpenCV */
        /* per-cell singly linked lists of accepted corners */
        int* head = (int*)malloc(sizeof(int) * (size_t)gw * (size_t)gh);
        int* next = (int*)malloc(sizeof(int) * (size_t)(total > 0 ? total : 1));
        float* acc = (float*)malloc(sizeof(float) * 2 * (size_t)(total > 0 ? total : 1));
        for (int i = 0; i < gw * gh; ++i) head[i] = -1;
        int nacc = 0;
        for (int i = 0; i < total; ++i) {
            const int y = cand[i].idx / w, x = cand[i].idx - y * w;
            const int xc = x / cell, yc = y / cell;
            int x1 = xc - 1, y1 = yc - 1, x2 = xc + 1, y2 = yc + 1;
            if (x1 < 0) x1 = 0;
            if (y1 < 0) y1 = 0;
            if (x2 > gw - 1) x2 = gw - 1;
            if (y2 > gh - 1) y2 = gh - 1;
            int good = 1;
            for (int yy = y1; yy <= y2 && good; ++yy)
                for (int xx = x1; xx <= x2 && good; ++xx)
                    for (int j = head[yy * gw + xx]; j >= 0; j = next[j]) {
                        const float dx = (float)x - acc[2 * j], dy = (float)y - acc[2 * j + 1];
                        if ((double)(dx * dx + dy * dy) < md2) { good = 0; break; }
                    }
            if (good) {
                acc[2 * nacc] = (float)x; acc[2 * nacc + 1] = (float)y;
                next[nacc] = head[yc * gw + xc]; head[yc * gw + xc] = nacc; ++nacc;
                if (nc < capacity) { corners[2 * nc] = (float)x; corners[2 * nc + 1] = (float)y; }
                ++nc;
                if (max_corners > 0 && nc == max_corners) break;
            }
        }
        free(head); free(next); free(acc);
    } else {
        for (int i = 0; i < total; ++i) {
            const int y = cand[i].idx / w, x = cand[i].idx - y * w;
            if (nc < capacity) { corners[2 * nc] = (float)x; corners[2 * nc + 1] = (float)y; }
            ++nc;
            if (max_corners > 0 && nc == max_corners) break;
        }
    }
    free(e); free(cand);
    return nc;
}

/* cv2.goodFeaturesToTrack(image, maxCorners, qualityLevel, minDistance, mask, blockSize) (gradientSize 3, no Harris) */
int klt_oracle_good_features_to_track(const uint8_t* img, int w, int h, int64_t pitch, const uint8_t* mask,
                                      int64_t mask_pitch, int max_corners, double quality, double min_distance,
                                      int block, float* corners, int capacity)
{
    float* eig = (float*)malloc(sizeof(float) * (size_t)w * (size_t)h);
    if (!eig) return -2;
    int rc = klt_oracle_corner_min_eigen_val(img, w, h, pitch, block, eig);
    if (!rc) rc = klt_oracle_select_corners(eig, w, h, mask, mask_pitch, max_corners, quality, min_distance, corners, capacity);
    free(eig);
    return rc;
}

/* ---- mask of filled circles (reference src/extractor/extractor.py:102-107) --------------------------------------
 * mask[:] = 255; for every tracked keypoint (x, y) = np.int32(kp.uv): cv2.circle(mask, (x, y), radius, 0, -1).
 * cv2.circle with thickness -1, LINE_8, shift 0 is OpenCV's midpoint circle (modules/imgproc/src/drawing.cpp, Circle()):
 * for every step (dx, dy) of the octant walk it fills rows cy -+ dy over [cx - dx, cx + dx] and rows cy -+ dx over
 * [cx - dy, cx + dy], clipped to the image.  half[d] below is the resulting half-width of row cy +- d. */
int klt_oracle_circle_half_widths(int radius, int* half /* radius + 1 entries */)
{
    if (radius < 0 || !half) return -1;
    for (int i = 0; i <= radius; ++i) half[i] = -1;
    int err = 0, dx = radius, dy = 0, plus = 1, minus = (radius << 1) - 1;
    while (dx >= dy) {
        if (dx > half[dy]) half[dy] = dx;     /* rows cy -+ dy: [cx - dx, cx + dx] */
        if (dy > half[dx]) half[dx] = dy;     /* rows cy -+ dx: [cx - dy, cx + dy] */
        dy++;
        err += plus;
        plus += 2;
        const int mask = (err <= 0) - 1;
        err -= minus & mask;
        dx += mask;
        minus -= mask & 2;
    }
    return 0;
}

int klt_oracle_mask_from_points(const float* pts /* n x (x, y) */, int n, int radius, int w, int h, uint8_t* mask, int64_t pitch)
{
    if (n < 0 || radius < 0 || w < 1 || h < 1 || !mask || (n > 0 && !pts)) return -1;
    int* half = (int*)malloc(sizeof(int) * (size_t)(radius + 1));
    if (!half) return -2;
    klt_oracle_circle_half_widths(radius, half);
    for (int y = 0; y < h; ++y) memset(mask + (int64_t)y * pitch, 255, (size_t)w);
    for (int i = 0; i < n; ++i) {
        const int cx = (int)pts[2 * i], cy = (int)pts[2 * i + 1];      /* np.int32(): truncation toward zero */
        for (int d = -radius; d <= radius; ++d) {
            const int y = cy + d, hw = half[d < 0 ? -d : d];
            if (y < 0 || y >= h || hw < 0) continue;
            int x1 = cx - hw, x2 = cx + hw;
            if (x1 < 0) x1 = 0;
            if (x2 > w - 1) x2 = w - 1;
            for (int x = x1; x <= x2; ++x) mask[(int64_t)y * pitch + x] = 0;
        }
    }
    free(half);
    return 0;
}
