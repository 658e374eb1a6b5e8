// Evaluation metrics on the device (reference: spnet/diagnostics.py).
//  * calc_errors (:13-60): ring-count / object-existence counters over every (image, predictor slot) and the
//    first predictor's centre error per image - exact (integer decisions on round-half-even, as Python's round).
//  * compute_iou (:85-120) for every (image, slot) in one launch: the reference draws two anti-aliased filled
//    ellipses with cv2 on a 512 x 384 canvas per pair and counts pixels on the CPU (calc_map does that for
//    2 x 72 x N masks x 10 thresholds). Here one CTA per pair rasterises both ellipses EXACTLY as cv2 does (integer
//    port of its polygon / anti-aliased line / convex fill code, pixel VALUES included: ellipse_iou_exact_kernel) and
//    writes the intersection and union pixel counts - intersection / union is the reference's IoU, bit for bit.
//    union = 0 where the reference returns -1.
#include "common.cuh"

namespace {

constexpr int VARS = 8;  // spnet/config.py:30

__global__ void __launch_bounds__(256) calc_errors_kernel(const float* __restrict__ yp, const float* __restrict__ yt,
                                                          int n, int ncols, int* __restrict__ counters,
                                                          float* __restrict__ pix_err) {
    const int slots = ncols / VARS;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    // counters: 0 ring_miscounts 1 ring_truecounts 2 total_obj 3 false_obj_pos 4 false_obj_neg 5 true_obj_pos 6 true_obj_neg
    int which = -1, ring = -1;
    if (idx < n * slots) {
        const int j = idx / slots, an = idx - j * slots;
        const float* p = yp + (size_t)j * ncols + an * VARS;
        const float* t = yt + (size_t)j * ncols + an * VARS;
        const int t_no = __float2int_rn(t[6]), p_no = __float2int_rn(p[6]);
        if (t_no == 0) {
            if (p_no == 0) { which = 5; ring = fabsf(__fsub_rn(t[7], p[7])) > 0.5f ? 0 : 1; }
            else which = 4;
        } else {
            which = p_no == 0 ? 3 : 6;
        }
        if (an == 0) {
            const float d0 = __fsub_rn(p[0], t[0]), d1 = __fsub_rn(p[1], t[1]);
            pix_err[j] = __fsqrt_rn(__fadd_rn(__fmul_rn(d0, d0), __fmul_rn(d1, d1)));
        }
    }
    // warp-aggregated atomics
#pragma unroll
    for (int c = 0; c < 7; ++c) {
        const bool hit = which == c || ring == c || (c == 2 && (which == 4 || which == 5));
        const unsigned m = __ballot_sync(0xffffffffu, hit);
        if ((threadIdx.x & 31) == 0 && m) atomicAdd(counters + c, __popc(m));
    }
}

// =================================================================================================
// EXACT rasterisation: the pixels cv2.ellipse(canvas, centre, axes, -angle, 0, 360, 255, thickness = -1, LINE_AA,
// shift = 10) leaves non-zero - what the reference's compute_iou counts (spnet/diagnostics.py:61-120 through
// utils.draw_ellipse, spnet/utils.py:35-53). Integer port of OpenCV's EllipseEx / ellipse2Poly / FillConvexPoly /
// LineAA (imgproc/src/drawing.cpp, third-party; restated and pinned pixel for pixel against cv2 4.13 by
// oracle/cv2_raster.py + tests/test_diagnostics.py). One CTA per (image, slot) pair: polygon vertices in parallel, the
// anti-aliased edges one thread per edge (atomicOr into a bit canvas in shared memory), the two scanline edge walkers
// by one thread (they share OpenCV's `edges` budget, so they are sequential by definition), the span fill and the
// population counts by everybody.
// =================================================================================================
constexpr int RX = 512, RY = 384;            // create_ellipse_image(nx = 512, ny = 384)
constexpr int RW = RX / 32;                  // 32-bit words per canvas row
constexpr int MAXV = 76;
constexpr int XYS = 16;
constexpr long long XY1 = 1LL << XYS;

__constant__ float c_sin[451] = {
#include "sin_table.inc"
};
__constant__ int c_slope_corr[32] = {181, 181, 181, 182, 182, 183, 184, 185, 187, 188, 190, 192, 194, 196, 198, 201,
                                     203, 206, 209, 211, 214, 218, 221, 224, 227, 231, 235, 238, 242, 246, 250, 254};
__constant__ int c_filter[64] = {168, 177, 185, 194, 202, 210, 218, 224, 231, 236, 241, 246, 249, 252, 254, 254,
                                 254, 254, 252, 249, 246, 241, 236, 231, 224, 218, 210, 202, 194, 185, 177, 168,
                                 158, 149, 140, 131, 122, 114, 105, 97,  89,  82,  75,  68,  62,  56,  50,  45,
                                 40,  36,  32,  28,  25,  22,  19,  16,  14,  12,  11,  9,   8,   7,   5,   5};

struct Poly { long long x[MAXV], y[MAXV]; int n; };

// Anti-aliased edge pixels keep their VALUE (the reference ANDs / ORs pixel values, and two partially covered pixels can
// AND to zero): a small open-addressing table per ellipse, entry = (pixel index + 1) << 8 | value. ONE thread per ellipse
// draws all its edges in order - the blends of cv2's ICV_PUT_POINT are order dependent - so no atomics are needed.
constexpr int HASH_BITS = 13, HASH_N = 1 << HASH_BITS;
struct AACanvas { unsigned* bits; unsigned* table; int* used; };

__device__ __forceinline__ int aa_slot(const unsigned* table, unsigned key) {
    unsigned h = (key * 2654435761u) >> (32 - HASH_BITS);
    for (int probe = 0; probe < HASH_N; ++probe) {
        const unsigned e = table[h];
        if (e == 0u || (e >> 8) == key + 1u) return (int)h;
        h = (h + 1u) & (HASH_N - 1);
    }
    return -1;
}
__device__ __forceinline__ void blend_px(const AACanvas& c, int yy, int xx, int a) {
    if (yy < 0 || yy >= RY || xx < 0 || xx >= RX) return;
    const unsigned key = (unsigned)(yy * RX + xx);
    c.bits[yy * RW + (xx >> 5)] |= 1u << (xx & 31);   // alpha >= 1 always makes a zero pixel non-zero
    if (*c.used >= HASH_N - 64) return;  // absurdly long outline: the pixel only counts as covered (mask exactness is kept)
    const int sl = aa_slot(c.table, key);
    const unsigned e = c.table[sl];
    int v = e ? (int)(e & 255u) : 0;
    if (!e) ++*c.used;
    v += ((255 - v) * a + 127) >> 8;   // ICV_PUT_POINT: two blend steps towards the colour
    v += ((255 - v) * a + 127) >> 8;
    c.table[sl] = ((key + 1u) << 8) | (unsigned)v;
}
__device__ __forceinline__ int aa_value(const unsigned* table, int yy, int xx) {
    const int sl = aa_slot(table, (unsigned)(yy * RX + xx));
    if (sl < 0) return 255;
    const unsigned e = table[sl];
    return e ? (int)(e & 255u) : 255;   // not in the table (overflow guard): treat as fully covered
}

// clipLine() of drawing.cpp on 16.16 coordinates
__device__ bool clip_line(long long w, long long h, long long& x1, long long& y1, long long& x2, long long& y2) {
    const long long right = w - 1, bottom = h - 1;
    int c1 = (x1 < 0) + (x1 > right) * 2 + (y1 < 0) * 4 + (y1 > bottom) * 8;
    int c2 = (x2 < 0) + (x2 > right) * 2 + (y2 < 0) * 4 + (y2 > bottom) * 8;
    if ((c1 & c2) == 0 && (c1 | c2) != 0) {
        long long a;
        if (c1 & 12) {
            a = c1 < 8 ? 0 : bottom;
            x1 += (long long)((double)(a - y1) * (double)(x2 - x1) / (double)(y2 - y1));
            y1 = a;
            c1 = (x1 < 0) + (x1 > right) * 2;
        }
        if (c2 & 12) {
            a = c2 < 8 ? 0 : bottom;
            x2 += (long long)((double)(a - y2) * (double)(x2 - x1) / (double)(y2 - y1));
            y2 = a;
            c2 = (x2 < 0) + (x2 > right) * 2;
        }
        if ((c1 & c2) == 0 && (c1 | c2) != 0) {
            if (c1) {
                a = c1 == 1 ? 0 : right;
                y1 += (long long)((double)(a - x1) * (double)(y2 - y1) / (double)(x2 - x1));
                x1 = a;
                c1 = 0;
            }
            if (c2) {
                a = c2 == 1 ? 0 : right;
                y2 += (long long)((double)(a - x2) * (double)(y2 - y1) / (double)(x2 - x1));
                x2 = a;
                c2 = 0;
            }
        }
    }
    return (c1 | c2) == 0;
}

// LineAA(): blends the three pixels across the line at every step along it
__device__ void line_aa(const AACanvas& canvas, long long x1, long long y1, long long x2, long long y2) {
    if (!clip_line((long long)RX << XYS, (long long)RY << XYS, x1, y1, x2, y2)) return;
    long long dx = x2 - x1, dy = y2 - y1;
    long long j = dx < 0 ? -1 : 0;
    const long long ax = (dx ^ j) - j;
    long long i = dy < 0 ? -1 : 0;
    const long long ay = (dy ^ i) - i;
    const bool steep = !(ax > ay);
    long long step;
    int ecount, slope;
    if (!steep) {
        dy = (dy ^ j) - j;
        if (j) { long long t = x1; x1 = x2; x2 = t; t = y1; y1 = y2; y2 = t; }
        step = (dy << XYS) / (ax | 1);
        x2 += XY1;
        ecount = (int)((x2 >> XYS) - (x1 >> XYS));
        j = -(x1 & (XY1 - 1));
        y1 += ((step * j) >> XYS) + (XY1 >> 1);
        slope = (int)((step >> (XYS - 5)) & 0x3f);
        slope ^= (step < 0 ? 0x3f : 0);
        i = (x1 >> (XYS - 7)) & 0x78;
        j = (x2 >> (XYS - 7)) & 0x78;
    } else {
        dx = (dx ^ i) - i;
        if (i) { long long t = x1; x1 = x2; x2 = t; t = y1; y1 = y2; y2 = t; }
        step = (dx << XYS) / (ay | 1);
        y2 += XY1;
        ecount = (int)((y2 >> XYS) - (y1 >> XYS));
        j = -(y1 & (XY1 - 1));
        x1 += ((step * j) >> XYS) + (XY1 >> 1);
        slope = (int)((step >> (XYS - 5)) & 0x3f);
        slope ^= (step < 0 ? 0x3f : 0);
        i = (y1 >> (XYS - 7)) & 0x78;
        j = (y2 >> (XYS - 7)) & 0x78;
    }
    slope = (slope & 0x20) ? 0x100 : c_slope_corr[slope];
    int ep[9];
    {
        const int ii = (int)i, jj = (int)j;
        const int t0 = slope << 7, t1 = ((0x78 - ii) | 4) * slope, t2 = (jj | 4) * slope;
        ep[0] = 0;
        ep[8] = slope;
        ep[1] = ep[3] = ((((jj - ii) & 0x78) | 4) * slope >> 8) & 0x1ff;
        ep[2] = (t1 >> 8) & 0x1ff;
        ep[4] = ((((jj - ii) + 0x80) | 4) * slope >> 8) & 0x1ff;
        ep[5] = ((t1 + t0) >> 8) & 0x1ff;
        ep[6] = (t2 >> 8) & 0x1ff;
        ep[7] = ((t2 + t0) >> 8) & 0x1ff;
    }
    int scount = 0;
    while (ecount >= 0) {
        const int ep_corr = ep[(((scount >= 2) + 1) & (scount | 2)) * 3 + (((ecount >= 2) + 1) & (ecount | 2))];
        const long long minor = steep ? x1 : y1, major = steep ? y1 : x1;
        const int m0 = (int)(minor >> XYS) - 1, mj = (int)(major >> XYS);
        const int dist = (int)((minor >> (XYS - 5)) & 31);
        const int f[3] = {c_filter[dist + 32], c_filter[dist], c_filter[63 - dist]};
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const int a = ((ep_corr * f[k]) >> 8) & 0xff;
            if (a) {
                if (steep) blend_px(canvas, mj, m0 + k, a);
                else blend_px(canvas, m0 + k, mj, a);
            }
        }
        if (steep) { x1 += step; y1 += XY1; }
        else { y1 += step; x1 += XY1; }
        ++scount;
        --ecount;
    }
}

// utils.draw_ellipse + cv2.ellipse + EllipseEx + ellipse2Poly: vertex `vi` (before the removal of consecutive
// duplicates) of the polygon; returns false past the last vertex
__device__ bool ellipse_vertex(const float* a, int vi, long long* px, long long* py, int* nverts) {
    // centre / axes: int(round(v * 2^10)) on float32 values (Python round = half to even), shifted to 16.16
    const long long cx = (long long)rintf(a[0] * 1024.0f) << 6, cy = (long long)rintf(a[1] * 1024.0f) << 6;
    long long aw = (long long)rintf(a[2] * 1024.0f) << 6, ah = (long long)rintf(a[3] * 1024.0f) << 6;
    aw = aw < 0 ? -aw : aw;
    ah = ah < 0 ? -ah : ah;
    // angle = rad2deg(arctan2(sin2t, cos2t) / 2) in float32 (create_ellipse_image), negated by draw_ellipse, cvRound
    const float ang32 = (atan2f(a[5], a[4]) / 2.0f) * 57.29577951308232f;
    int angle = (int)rint(-(double)ang32);
    int delta = (int)(((aw > ah ? aw : ah) + (XY1 >> 1)) >> XYS);
    delta = delta < 3 ? 90 : delta < 10 ? 30 : delta < 15 ? 18 : 5;
    *nverts = 360 / delta + 1;
    if (vi >= *nverts) return false;
    while (angle < 0) angle += 360;
    while (angle > 360) angle -= 360;
    const float alpha = c_sin[450 - angle], beta = c_sin[angle];
    const int ang = min(vi * delta, 360);
    const double x = (double)aw * (double)c_sin[450 - ang], y = (double)ah * (double)c_sin[ang];
    const double fx = (double)cx + x * (double)alpha - y * (double)beta, fy = (double)cy + x * (double)beta + y * (double)alpha;
    long long qx = (long long)rint(fx / 65536.0) << XYS, qy = (long long)rint(fy / 65536.0) << XYS;
    qx += (long long)rint(fx - (double)qx);
    qy += (long long)rint(fy - (double)qy);
    *px = qx;
    *py = qy;
    return true;
}

// FillConvexPoly(LINE_AA) scanline part, sequential (one thread): per row the span [xl, xr] it fills, -1 when empty
__device__ void fill_spans(const Poly& P, int* row_l, int* row_r, int* y_first, int* y_last) {
    const int n = P.n;
    const long long delta = XY1 >> 1, delta1 = XY1 - 1, delta2 = 0;
    long long xmin = P.x[0], xmax = P.x[0], ymin = P.y[0], ymax = P.y[0];
    int imin = 0;
    for (int i = 0; i < n; ++i) {
        if (P.y[i] < ymin) { ymin = P.y[i]; imin = i; }
        ymax = P.y[i] > ymax ? P.y[i] : ymax;
        xmax = P.x[i] > xmax ? P.x[i] : xmax;
        xmin = P.x[i] < xmin ? P.x[i] : xmin;
    }
    xmin = (xmin + delta) >> XYS; xmax = (xmax + delta) >> XYS;
    ymin = (ymin + delta) >> XYS; ymax = (ymax + delta) >> XYS;
    *y_first = 0; *y_last = -1;
    if (n < 3 || (int)xmax < 0 || (int)ymax < 0 || (int)xmin >= RX || (int)ymin >= RY) return;
    if (ymax > RY - 1) ymax = RY - 1;
    int e_idx[2] = {imin, imin}, e_di[2] = {1, n - 1}, e_ye[2] = {(int)ymin, (int)ymin};
    long long e_x[2] = {-XY1, -XY1}, e_dx[2] = {0, 0};
    int edges = n, y = (int)ymin;
    *y_first = y < 0 ? 0 : y;
    do {
        if (y < (int)ymax || y == (int)ymin) {
            for (int i = 0; i < 2; ++i) {
                if (y >= e_ye[i]) {
                    int idx0 = e_idx[i];
                    const int di = e_di[i];
                    int idx = idx0 + di;
                    if (idx >= n) idx -= n;
                    for (; edges-- > 0;) {
                        const int ty = (int)((P.y[idx] + delta) >> XYS);
                        if (ty > y) {
                            const long long xs = P.x[idx0], xe = P.x[idx];
                            e_ye[i] = ty;
                            e_dx[i] = ((xe - xs) * 2 + (ty - y)) / (2 * (ty - y));
                            e_x[i] = xs;
                            e_idx[i] = idx;
                            break;
                        }
                        idx0 = idx;
                        idx += di;
                        if (idx >= n) idx -= n;
                    }
                }
            }
        }
        if (edges < 0) break;
        if (y >= 0) {
            int left = 0, right = 1;
            if (e_x[0] > e_x[1]) { left = 1; right = 0; }
            int xx1 = (int)((e_x[left] + delta1) >> XYS), xx2 = (int)((e_x[right] + delta2) >> XYS);
            if (xx2 >= 0 && xx1 < RX) {
                if (xx1 < 0) xx1 = 0;
                if (xx2 >= RX) xx2 = RX - 1;
                row_l[y] = xx1;
                row_r[y] = xx2;
            } else {
                row_l[y] = 0; row_r[y] = -1;
            }
            *y_last = y;
        }
        e_x[0] += e_dx[0];
        e_x[1] += e_dx[1];
    } while (++y <= (int)ymax);
}

// dynamic shared memory: per ellipse a bit canvas of the filled spans (value 255), a bit canvas + value table of the
// anti-aliased edge pixels, the polygon and the spans
struct RasterSmem {
    unsigned fill[2][RY * RW];
    unsigned aa[2][RY * RW];
    unsigned table[2][HASH_N];
    int used[2];
    Poly poly[2];
    long long vx[2][MAXV], vy[2][MAXV];
    int row_l[2][RY], row_r[2][RY];
    int y_first[2], y_last[2];
    int red[2][8];
};

__global__ void __launch_bounds__(256) ellipse_iou_exact_kernel(const float* __restrict__ yp, const float* __restrict__ yt,
                                                                int ncols, int* __restrict__ counts) {
    extern __shared__ __align__(16) unsigned char raster_raw[];
    RasterSmem& S = *reinterpret_cast<RasterSmem*>(raster_raw);
    const int slots = ncols / VARS;
    const int pair = blockIdx.x, jimg = pair / slots, an = pair - jimg * slots;
    const float* pe[2] = {yp + (size_t)jimg * ncols + an * VARS, yt + (size_t)jimg * ncols + an * VARS};
    if (pe[1][6] > 0.99f) {  // empty true slot: the reference skips the pair (compute_iou :98-99)
        if (threadIdx.x == 0) { counts[2 * pair] = 0; counts[2 * pair + 1] = 0; }
        return;
    }
    const bool drawn[2] = {pe[0][6] < 0.5f, pe[1][6] < 0.5f};   // create_ellipse_image: noobj < 0.5
    for (int i = threadIdx.x; i < 2 * RY * RW; i += blockDim.x) { (&S.fill[0][0])[i] = 0u; (&S.aa[0][0])[i] = 0u; }
    for (int i = threadIdx.x; i < 2 * HASH_N; i += blockDim.x) (&S.table[0][0])[i] = 0u;
    if (threadIdx.x < 2) S.used[threadIdx.x] = 0;
    // ---- polygon vertices: threads 0..127 -> ellipse 0, 128..255 -> ellipse 1
    {
        const int e = threadIdx.x >> 7, vi = threadIdx.x & 127;
        int nv = 0;
        long long x = 0, y = 0;
        if (drawn[e] && vi < MAXV && ellipse_vertex(pe[e], vi, &x, &y, &nv)) { S.vx[e][vi] = x; S.vy[e][vi] = y; }
        if (vi == 0) S.poly[e].n = drawn[e] ? nv : 0;
    }
    __syncthreads();
    if ((threadIdx.x & 127) == 0) {  // drop consecutive duplicates (EllipseEx); a single point becomes a zero-size polygon
        const int e = threadIdx.x >> 7;
        Poly& P = S.poly[e];
        const int nv = P.n;
        int m = 0;
        for (int i = 0; i < nv; ++i)
            if (m == 0 || S.vx[e][i] != P.x[m - 1] || S.vy[e][i] != P.y[m - 1]) { P.x[m] = S.vx[e][i]; P.y[m] = S.vy[e][i]; ++m; }
        if (m == 1) {
            const long long cx = (long long)rintf(pe[e][0] * 1024.0f) << 6, cy = (long long)rintf(pe[e][1] * 1024.0f) << 6;
            P.x[0] = P.x[1] = cx; P.y[0] = P.y[1] = cy;
            m = 2;
        }
        P.n = m;
        S.y_first[e] = 0; S.y_last[e] = -1;
    }
    __syncthreads();
    // ---- per ellipse: one thread walks the scanline spans, another draws the anti-aliased edges IN ORDER (edge i runs
    //      from vertex i-1 to vertex i; the blends are order dependent where two edges touch the same pixel)
    {
        const int e = threadIdx.x >> 7, role = threadIdx.x & 127;
        const Poly& P = S.poly[e];
        if (role == 0 && P.n > 0) fill_spans(P, S.row_l[e], S.row_r[e], &S.y_first[e], &S.y_last[e]);
        if (role == 32 && P.n > 0) {
            const AACanvas c = {S.aa[e], S.table[e], &S.used[e]};
            for (int ei = 0; ei < P.n; ++ei) {
                const int p0 = ei == 0 ? P.n - 1 : ei - 1;
                line_aa(c, P.x[p0], P.y[p0], P.x[ei], P.y[ei]);
            }
        }
    }
    __syncthreads();
    // ---- span fill: one (row, word) item per thread step
    for (int e = 0; e < 2; ++e) {
        const int y0 = S.y_first[e], y1 = S.y_last[e];
        for (int i = threadIdx.x; i < (y1 - y0 + 1) * RW; i += blockDim.x) {
            const int y = y0 + i / RW, w = i % RW;
            const int l = S.row_l[e][y], r = S.row_r[e][y];
            const int lo = max(l, w * 32), hi = min(r, w * 32 + 31);
            if (hi >= lo) {
                const unsigned bits = (hi - lo == 31) ? 0xffffffffu : (((1u << (hi - lo + 1)) - 1u) << (lo & 31));
                atomicOr(&S.fill[e][y * RW + w], bits);
            }
        }
    }
    __syncthreads();
    // cv2.bitwise_and / bitwise_or of the pixel VALUES, then countNonZero (compute_iou :104-107): a pixel is in the
    // union when either canvas is non-zero; in the intersection when both are AND their values share a bit - always true
    // when one of them is a filled (255) pixel, looked up in the value tables where both are edge pixels
    int ni = 0, nu = 0;
    for (int i = threadIdx.x; i < RY * RW; i += blockDim.x) {
        const unsigned fp = S.fill[0][i], ft = S.fill[1][i], ap = S.aa[0][i], at = S.aa[1][i];
        const unsigned P = fp | ap, T = ft | at;
        ni += __popc(P & T);
        nu += __popc(P | T);
        unsigned both = ap & at & ~fp & ~ft;
        while (both) {
            const int b = __ffs(both) - 1;
            both &= both - 1;
            const int yy = i / RW, xx = (i % RW) * 32 + b;
            if ((aa_value(S.table[0], yy, xx) & aa_value(S.table[1], yy, xx)) == 0) --ni;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        ni += __shfl_xor_sync(0xffffffffu, ni, o);
        nu += __shfl_xor_sync(0xffffffffu, nu, o);
    }
    if ((threadIdx.x & 31) == 0) { S.red[0][threadIdx.x >> 5] = ni; S.red[1][threadIdx.x >> 5] = nu; }
    __syncthreads();
    if (threadIdx.x == 0) {
        int si = 0, su = 0;
        for (int w = 0; w < 8; ++w) { si += S.red[0][w]; su += S.red[1][w]; }
        counts[2 * pair] = si;
        counts[2 * pair + 1] = su;  // 0 when nothing is drawn at all: the reference returns -1
    }
}

}  // namespace

extern "C" {

// counters: int32 [7] (zeroed by the caller): ring_miscounts, ring_truecounts, total_obj, false_obj_pos,
// false_obj_neg, true_obj_pos, true_obj_neg; pix_err: fp32 [n]. yp / yt: denormalised [n, ncols] fp32.
int spnet_calc_errors(const float* yp, const float* yt, int n, int ncols, int* counters, float* pix_err,
                      cudaStream_t stream) {
    SPNET_REQUIRE(yp && yt && counters && pix_err && n > 0 && ncols > 0 && ncols % VARS == 0, "calc_errors: bad args");
    const int items = n * (ncols / VARS);
    calc_errors_kernel<<<ceil_div(items, 256), 256, 0, stream>>>(yp, yt, n, ncols, counters, pix_err);
    return spnet_check_launch("calc_errors");
}

// counts: int32 [n, ncols/8, 2] = (intersection, union) pixel counts of the reference's raster on its 512 x 384 canvas
int spnet_ellipse_iou(const float* yp, const float* yt, int n, int ncols, int* counts, cudaStream_t stream) {
    SPNET_REQUIRE(yp && yt && counts && n > 0 && ncols > 0 && ncols % VARS == 0, "ellipse_iou: bad args");
    static bool configured[64] = {};
    const int rc = spnet_smem_optin(configured, ellipse_iou_exact_kernel, sizeof(RasterSmem), "ellipse_iou");
    if (rc) return rc;
    ellipse_iou_exact_kernel<<<n * (ncols / VARS), 256, sizeof(RasterSmem), stream>>>(yp, yt, ncols, counts);
    return spnet_check_launch("ellipse_iou");
}

}  // extern "C"
