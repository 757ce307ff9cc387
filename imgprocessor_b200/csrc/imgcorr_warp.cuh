// imgcorr_warp.cuh — per-pixel arithmetic of cv2.warpPerspective as PerspectiveCorrection uses it
// (SURVEY §8 row f3; reference paths relative to /root/reference/imgProcessor/):
//   PerspectiveCorrection.correct     camera/PerspectiveCorrection.py:380-406   INTER_LANCZOS4
//   PerspectiveCorrection.uncorrect   camera/PerspectiveCorrection.py:374-378   INTER_CUBIC | WARP_INVERSE_MAP
//
// Like imgcorr_core.cuh this file is __host__ __device__ and free of memory staging, so that
// tests/host_emul compiles the same functions with g++ and checks them against the oracle
// (oracle/warp.py) where no GPU exists.  OpenCV semantics restated (imgwarp.cpp, 4.13.0 behaviour
// pinned by the tests): float64 blockwise coordinates with 5 fractional bits, float32 coefficient
// tables for the 32 phases, 2-D weight = float32(wy * wx), one left-to-right sum per tap row, row sums
// added top to bottom, no FMA; border pixels  cv + sum((S - cv) * w)  over the in-range taps.
#pragma once
#include "imgcorr_core.cuh"

namespace imgcorr {

enum : int { WARP_CUBIC = 2, WARP_LANCZOS4 = 4 };   // cv2.INTER_CUBIC, cv2.INTER_LANCZOS4

struct WarpConst {
    double m[9];   // dst -> src matrix (already inverted unless WARP_INVERSE_MAP)
    int bw0;       // OpenCV's block width: x coordinates are built as bx + x1 with bx = (x / bw0) * bw0
};

// ---- host-side setup --------------------------------------------------------------------
// cv::invert(DECOMP_LU) of a 3x3 double matrix: cofactors times 1/det; singular -> zeros.
inline void warp_invert3x3(const double* s, double* t) {
#define M_(r, c) s[(r) * 3 + (c)]
    double d = M_(0, 0) * (M_(1, 1) * M_(2, 2) - M_(1, 2) * M_(2, 1)) - M_(0, 1) * (M_(1, 0) * M_(2, 2) - M_(1, 2) * M_(2, 0)) +
               M_(0, 2) * (M_(1, 0) * M_(2, 1) - M_(1, 1) * M_(2, 0));
    if (d == 0) {
        for (int i = 0; i < 9; ++i) t[i] = 0;
        return;
    }
    d = 1. / d;
    t[0] = (M_(1, 1) * M_(2, 2) - M_(1, 2) * M_(2, 1)) * d;
    t[1] = (M_(0, 2) * M_(2, 1) - M_(0, 1) * M_(2, 2)) * d;
    t[2] = (M_(0, 1) * M_(1, 2) - M_(0, 2) * M_(1, 1)) * d;
    t[3] = (M_(1, 2) * M_(2, 0) - M_(1, 0) * M_(2, 2)) * d;
    t[4] = (M_(0, 0) * M_(2, 2) - M_(0, 2) * M_(2, 0)) * d;
    t[5] = (M_(0, 2) * M_(1, 0) - M_(0, 0) * M_(1, 2)) * d;
    t[6] = (M_(1, 0) * M_(2, 1) - M_(1, 1) * M_(2, 0)) * d;
    t[7] = (M_(0, 1) * M_(2, 0) - M_(0, 0) * M_(2, 1)) * d;
    t[8] = (M_(0, 0) * M_(1, 1) - M_(0, 1) * M_(1, 0)) * d;
#undef M_
}

inline WarpConst make_warp_const(const double M[9], int inverse_map, int dst_w, int dst_h) {
    WarpConst c;
    if (inverse_map)
        for (int i = 0; i < 9; ++i) c.m[i] = M[i];
    else
        warp_invert3x3(M, c.m);
    int bh0 = dst_h < 16 ? dst_h : 16;
    if (bh0 < 1) bh0 = 1;
    c.bw0 = 1024 / bh0 < dst_w ? 1024 / bh0 : dst_w;
    if (c.bw0 < 1) c.bw0 = 1;
    return c;
}

// cv::interpolateLanczos4 for phase k/32, float32 coefficients; tab is [32][8]
inline void warp_lanczos4_table(float* tab) {
    static const double s45 = 0.70710678118654752440084436210485;
    static const double cs[8][2] = {{1, 0}, {-s45, -s45}, {0, 1}, {s45, -s45}, {-1, 0}, {s45, s45}, {0, -1}, {-s45, s45}};
    const double pi = 3.1415926535897932384626433832795;
    for (int k = 0; k < 32; ++k) {
        float* co = tab + k * 8;
        const float x = (float)k * (1.0f / 32);
        if (x < FLT_EPSILON) {
            for (int i = 0; i < 8; ++i) co[i] = 0;
            co[3] = 1;
            continue;
        }
        float sum = 0;
        const double y0 = -(x + 3) * pi * 0.25, s0 = sin(y0), c0 = cos(y0);
        for (int i = 0; i < 8; ++i) {
            const double y = -(x + 3 - i) * pi * 0.25;
            co[i] = (float)((cs[i][0] * s0 + cs[i][1] * c0) / (y * y));
            sum += co[i];
        }
        sum = 1.f / sum;
        for (int i = 0; i < 8; ++i) co[i] *= sum;
    }
}

// cv::interpolateCubic (A = -0.75); tab is [32][4]
inline void warp_cubic_table(float* tab) {
    const float A = -0.75f;
    for (int k = 0; k < 32; ++k) {
        float* co = tab + k * 4;
        const float x = (float)k * (1.0f / 32);
        co[0] = ((A * (x + 1) - 5 * A) * (x + 1) + 8 * A) * (x + 1) - 4 * A;
        co[1] = ((A + 2) * x - (A + 3)) * x * x + 1;
        co[2] = ((A + 2) * (1 - x) - (A + 3)) * (1 - x) * (1 - x) + 1;
        co[3] = 1.f - co[0] - co[1] - co[2];
    }
}

// uint8 images: OpenCV's fixed-point branch of initInterTab2D — int16 weights [32][32][n*n] (phase fy, phase fx, tap
// row-major) = saturate_cast<short>(wy * wx * 2^15), the sum of each phase pair forced to 2^15 on one of the four
// central taps (the largest if the sum fell short, the smallest if it overshot).
inline void warp_fixed_table(const float* tab, int n, int16_t* out) {
    const int k2 = n / 2;
    for (int i = 0; i < 32; ++i)
        for (int j = 0; j < 32; ++j) {
            int16_t* it = out + ((size_t)i * 32 + j) * n * n;
            int isum = 0;
            for (int a = 0; a < n; ++a)
                for (int b = 0; b < n; ++b) {
                    const float v = tab[i * n + a] * tab[j * n + b];
                    float r = nearbyintf(v * 32768.0f);
                    r = r < -32768.0f ? -32768.0f : (r > 32767.0f ? 32767.0f : r);
                    it[a * n + b] = (int16_t)r;
                    isum += it[a * n + b];
                }
            if (isum != 32768) {
                const int diff = isum - 32768;
                int Mk1 = k2, Mk2 = k2, mk1 = k2, mk2 = k2;
                for (int a = k2; a < k2 + 2; ++a)
                    for (int b = k2; b < k2 + 2; ++b) {
                        if (it[a * n + b] < it[mk1 * n + mk2]) { mk1 = a; mk2 = b; }
                        else if (it[a * n + b] > it[Mk1 * n + Mk2]) { Mk1 = a; Mk2 = b; }
                    }
                if (diff < 0) it[Mk1 * n + Mk2] = (int16_t)(it[Mk1 * n + Mk2] - diff);
                else it[mk1 * n + mk2] = (int16_t)(it[mk1 * n + mk2] - diff);
            }
        }
}

// ---- coordinates (d2i_rn: imgcorr_core.cuh) --------------------------------------------------

// X = cvRound(max(INT_MIN, min(INT_MAX, (X0 + M0*x1) * W))); a NaN ends up as INT_MAX (std::min / std::max
// argument order in OpenCV, fmin / fmax here).  OpenCV additionally saturates X >> 5 to int16; for sources
// up to 32767 px per side a saturated coordinate is entirely outside on either side, so it is dropped.
IC_HD FixedCoord warp_coord(const WarpConst& c, int x, int y) {
    const double bx = (double)((x / c.bw0) * c.bw0), x1 = (double)(x % c.bw0), yd = (double)y;
    const double X0 = dadd(dadd(dmul(c.m[0], bx), dmul(c.m[1], yd)), c.m[2]);
    const double Y0 = dadd(dadd(dmul(c.m[3], bx), dmul(c.m[4], yd)), c.m[5]);
    const double W0 = dadd(dadd(dmul(c.m[6], bx), dmul(c.m[7], yd)), c.m[8]);
    double W = dadd(W0, dmul(c.m[6], x1));
    W = W != 0.0 ? ddiv(32.0, W) : 0.0;
    const double fX = fmax(-2147483648.0, fmin(2147483647.0, dmul(dadd(X0, dmul(c.m[0], x1)), W)));
    const double fY = fmax(-2147483648.0, fmin(2147483647.0, dmul(dadd(Y0, dmul(c.m[3], x1)), W)));
    const int X = d2i_rn(fX), Y = d2i_rn(fY);
    FixedCoord r;
    r.ix = X >> 5;
    r.iy = Y >> 5;
    r.fx = X & 31;
    r.fy = Y & 31;
    return r;
}

// ---- accumulation ---------------------------------------------------------------------------
IC_HD float wmul(float a, float b) { return fmul(a, b); }
IC_HD double wmul(double a, double b) { return dmul(a, b); }
IC_HD float wadd(float a, float b) { return fadd(a, b); }
IC_HD double wadd(double a, double b) { return dadd(a, b); }
IC_HD float wsub(float a, float b) { return fsub(a, b); }
IC_HD double wsub(double a, double b) { return dsub(a, b); }

// interior pixel: S points at the top-left tap, `pitch` in elements; wy / wx are the phase rows of the table
template <typename T, typename AT, int N>
IC_HD AT warp_sum_interior(const T* S, long long pitch, const float* wy, const float* wx) {
    AT total = (AT)0;
    for (int r = 0; r < N; ++r) {
        const T* R = S + r * pitch;
        AT acc = wmul((AT)R[0], (AT)fmul(wy[r], wx[0]));
        for (int c = 1; c < N; ++c) acc = wadd(acc, wmul((AT)R[c], (AT)fmul(wy[r], wx[c])));
        total = wadd(total, acc);
    }
    return total;
}

// border pixel (window partly outside): S0 = frame origin; taps outside [0,W) x [0,H) are skipped
template <typename T, typename AT, int N>
IC_HD AT warp_sum_border(const T* S0, int H, int W, int sx, int sy, const float* wy, const float* wx, AT cv) {
    AT sum = wmul(cv, (AT)1);
    for (int r = 0; r < N; ++r) {
        const int yy = sy + r;
        if (yy < 0 || yy >= H) continue;
        const T* R = S0 + (long long)yy * W;
        for (int c = 0; c < N; ++c) {
            const int xx = sx + c;
            if (xx < 0 || xx >= W) continue;
            sum = wadd(sum, wmul(wsub((AT)R[xx], cv), (AT)fmul(wy[r], wx[c])));
        }
    }
    return sum;
}

// whole pixel, any position (the kernels specialise the interior case; this is what host_emul checks)
template <typename T, typename AT, int N>
IC_HD AT warp_pixel(const T* S0, int H, int W, FixedCoord c, const float* tab, AT cv) {
    const int off = N / 2 - 1;
    const int sx = c.ix - off, sy = c.iy - off;
    const float* wy = tab + c.fy * N;
    const float* wx = tab + c.fx * N;
    const int w1 = W - (N - 1) > 0 ? W - (N - 1) : 0, h1 = H - (N - 1) > 0 ? H - (N - 1) : 0;
    if ((unsigned)sx < (unsigned)w1 && (unsigned)sy < (unsigned)h1)
        return warp_sum_interior<T, AT, N>(S0 + (long long)sy * W + sx, W, wy, wx);
    if (sx >= W || sx + N <= 0 || sy >= H || sy + N <= 0) return cv;
    return warp_sum_border<T, AT, N>(S0, H, W, sx, sy, wy, wx, cv);
}

// uint8 pixel: w = the n*n int16 weights of this pixel's phase pair; int32 accumulation, FixedPtCast = rounding shift by
// 15 bits + saturation.  The interior sum and OpenCV's border form  cv*2^15 + sum((S - cv) * w)  are both exact integers.
template <int N>
IC_HD uint8_t warp_pixel_u8(const uint8_t* S0, int H, int W, FixedCoord c, const int16_t* w, int cv) {
    const int off = N / 2 - 1;
    const int sx = c.ix - off, sy = c.iy - off;
    int sum;
    if (sx >= W || sx + N <= 0 || sy >= H || sy + N <= 0) {
        sum = cv << 15;
    } else {
        const int w1 = W - (N - 1) > 0 ? W - (N - 1) : 0, h1 = H - (N - 1) > 0 ? H - (N - 1) : 0;
        const bool interior = (unsigned)sx < (unsigned)w1 && (unsigned)sy < (unsigned)h1;
        sum = interior ? 0 : cv << 15;
        const int sub = interior ? 0 : cv;
        for (int r = 0; r < N; ++r) {
            const int yy = sy + r;
            if (yy < 0 || yy >= H) continue;
            const uint8_t* R = S0 + (long long)yy * W;
            for (int k = 0; k < N; ++k) {
                const int xx = sx + k;
                if (xx < 0 || xx >= W) continue;
                sum += ((int)R[xx] - sub) * (int)w[r * N + k];
            }
        }
    }
    const int v = (sum + (1 << 14)) >> 15;
    return (uint8_t)(v < 0 ? 0 : (v > 255 ? 255 : v));
}

}  // namespace imgcorr
