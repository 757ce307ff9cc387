// K2 — lens undistortion: per output pixel evaluate the lens model analytically (Brown-Conrady; with the EXT flag
// OpenCV's rational, thin-prism and tilted-sensor terms as well)
// (float64, one rounding to float32 — no map arrays are read), convert to OpenCV's 5-bit
// fixed-point coordinates and gather the bilinear blend from the K1 output through L1/L2.
//
// Replaces  LensDistortion.correct()  camera/LensDistortion.py:316-330:
//   cv2.getOptimalNewCameraMatrix (host, stays cv2)  ->  P           :350-353
//   cv2.initUndistortRectifyMap(K, d, None, P, CV_32FC1)              :355-357   (device, analytic)
//   cv2.remap(INTER_LINEAR, BORDER_CONSTANT, borderValue)             :323-326   (device)
//   optional crop to roi                                              :327-329   (output window)
// The same kernel also serves explicit float32 maps (distortImage, parity tests against
// cv2's own maps).  When n_frames > 1 the coordinates and weights of a pixel are computed once
// and applied to every frame of the launch.
//
// A thread owns one output column and four rows of a 32x32 tile (consecutive lanes = consecutive
// columns: coalesced stores, neighbouring gathers).  When P^-1 has no cross terms (what
// getOptimalNewCameraMatrix always produces) x depends on the column only and is hoisted.
#include "imgcorr_kernels.cuh"
#include "imgcorr_tma.cuh"
#include <stdlib.h>

namespace imgcorr {

#ifndef K2_ROWS_V
#define K2_ROWS_V 2
#endif
#ifndef K2_MINB_V
#define K2_MINB_V 5
#endif
constexpr int K2_BX = 32, K2_BY = 8, K2_ROWS = K2_ROWS_V;     // CTA = 32 x 8 threads, tile = 32 x (8 * K2_ROWS) outputs
constexpr int K2_MINB = K2_MINB_V;

template <typename SrcT> __device__ __forceinline__ SrcT border_cast(double b) { return (SrcT)b; }

// fixed_coord() without the two F2I conversions (the XU pipe is what bounds the coordinate phase of a one-frame launch:
// 7 conversions per pixel at 16 lanes per clock and SM): cvRound(m * 32) by the magic-number addition
//   s = m * 32 + 1.5 * 2^23   (one rounding to the integer grid, ties to even = cvRound / cvt.rni)
// whose bit pattern minus that of the constant is the integer.  The constant's low five bits are zero, so the 1/32-pixel
// phase is `bits & 31` and the pixel index `(bits - bits(1.5 * 2^23)) >> 5`.  Exact for |m * 32| < 2^22 (every coordinate
// of a frame up to 32767 pixels a side — larger frames are refused); beyond that, and for NaN / inf, the result is some
// index far outside the frame on either side, which is all fixed_coord() guarantees there too (border value).
__device__ __forceinline__ FixedCoord fixed_coord_fast(float mapx, float mapy) {
    constexpr int MAGIC = 0x4B400000;                               // bits of 12582912.0f = 1.5 * 2^23
    const int bx = __float_as_int(__fmaf_rn(mapx, 32.0f, 12582912.0f));
    const int by = __float_as_int(__fmaf_rn(mapy, 32.0f, 12582912.0f));
    FixedCoord c;
    c.ix = (bx - MAGIC) >> 5;
    c.iy = (by - MAGIC) >> 5;
    c.fx = bx & 31;
    c.fy = by & 31;
    return c;
}
// float(k) for 0 <= k < 2^23 without an I2F conversion
__device__ __forceinline__ float small_int_to_float(int k) { return __int_as_float(0x4B000000 | k) - 8388608.0f; }
__device__ __forceinline__ void bilinear_weights_fast(int fx, int fy, float& w00, float& w01, float& w10, float& w11) {
    const float tx = small_int_to_float(fx) * 0.03125f, ty = small_int_to_float(fy) * 0.03125f;     // exact
    const float ux = 1.0f - tx, uy = 1.0f - ty;                                                       // exact
    w00 = fmul(uy, ux); w01 = fmul(uy, tx); w10 = fmul(ty, ux); w11 = fmul(ty, tx);
}

// per-pixel interpolation weights, computed once and applied to every frame of the launch
template <typename SrcT> struct Weights {        // float32 / uint16 / float64 images: OpenCV's float32 table entry
    float w00, w01, w10, w11;
    __device__ __forceinline__ void set(const FixedCoord& c) { bilinear_weights_fast(c.fx, c.fy, w00, w01, w10, w11); }
    // the same four values from the 32 x 32 table OpenCV itself uses (BilinearTab_f), built once per context on the host:
    // one 16-byte load (L1-resident, 16 KB) instead of a dozen instructions
    __device__ __forceinline__ void lookup(unsigned fyfx, const float4* tab) {       // fyfx = fy * 32 + fx
        const float4 w = __ldg(tab + fyfx);
        w00 = w.x; w01 = w.y; w10 = w.z; w11 = w.w;
    }
};
template <> struct Weights<uint8_t> {            // uint8 images: int16 fixed-point weights
    int fx, fy;
    __device__ __forceinline__ void set(const FixedCoord& c) { fx = c.fx; fy = c.fy; }
    __device__ __forceinline__ void lookup(unsigned fyfx, const float4*) { fx = fyfx & 31; fy = fyfx >> 5; }
};

template <typename SrcT, typename DstT> struct Blend;
template <> struct Blend<float, float> {
    static __device__ __forceinline__ float run(float a, float b, float c, float d, const Weights<float>& w) {
        return blend_f32(a, b, c, d, w.w00, w.w01, w.w10, w.w11);
    }
};
template <> struct Blend<float, double> {
    static __device__ __forceinline__ double run(float a, float b, float c, float d, const Weights<float>& w) {
        return (double)blend_f32(a, b, c, d, w.w00, w.w01, w.w10, w.w11);
    }
};
template <> struct Blend<double, double> {
    static __device__ __forceinline__ double run(double a, double b, double c, double d, const Weights<double>& w) {
        return blend_f64(a, b, c, d, w.w00, w.w01, w.w10, w.w11);
    }
};
template <> struct Blend<uint16_t, uint16_t> {
    static __device__ __forceinline__ uint16_t run(uint16_t a, uint16_t b, uint16_t c, uint16_t d, const Weights<uint16_t>& w) {
        return sat_u16(blend_f32((float)a, (float)b, (float)c, (float)d, w.w00, w.w01, w.w10, w.w11));
    }
};
template <> struct Blend<uint8_t, uint8_t> {
    static __device__ __forceinline__ uint8_t run(uint8_t a, uint8_t b, uint8_t c, uint8_t d, const Weights<uint8_t>& w) {
        return (uint8_t)blend_u8(a, b, c, d, w.fx, w.fy);
    }
};

// F32 -> U16 / U8 (the batch chain's integer output): the float32 pair's result, then the quantiser.  These pairs read
// the float32 blend of Blend<float, float>, so their values are quantise(the F32 call's values) by construction.
template <typename SrcT, typename DstT> struct K2Quant { static constexpr bool value = sizeof(SrcT) == 4 && sizeof(DstT) <= 2; };
template <typename SrcT, typename DstT>
__device__ __forceinline__ DstT blend_out(SrcT a, SrcT b, SrcT c, SrcT d, const Weights<SrcT>& w, const OutScale& q) {
    if constexpr (K2Quant<SrcT, DstT>::value) return quantise<DstT>(Blend<float, float>::run(a, b, c, d, w), q);
    else return Blend<SrcT, DstT>::run(a, b, c, d, w);
}
template <typename SrcT, typename DstT> __device__ __forceinline__ DstT border_out(SrcT b, const OutScale& q) {
    if constexpr (K2Quant<SrcT, DstT>::value) return quantise<DstT>(b, q);
    else return (DstT)b;
}

// rim of the image: any neighbour outside [0,W)x[0,H) is the border value; a window entirely outside is the border
// value itself (OpenCV does not blend it).  Rare -> kept out of line so the hot path stays small.
template <typename SrcT, typename DstT>
__device__ __noinline__ DstT remap_rim(const SrcT* __restrict__ src, int H, int W, int ix, int iy, Weights<SrcT> w, SrcT bval) {
    if (ix >= W || ix + 1 < 0 || iy >= H || iy + 1 < 0) return (DstT)bval;
    const bool x0 = (unsigned)ix < (unsigned)W, x1 = (unsigned)(ix + 1) < (unsigned)W;
    const bool y0 = (unsigned)iy < (unsigned)H, y1 = (unsigned)(iy + 1) < (unsigned)H;
    const SrcT* p = src + (ptrdiff_t)iy * W + ix;
    const SrcT v00 = (x0 && y0) ? __ldg(p) : bval;
    const SrcT v01 = (x1 && y0) ? __ldg(p + 1) : bval;
    const SrcT v10 = (x0 && y1) ? __ldg(p + W) : bval;
    const SrcT v11 = (x1 && y1) ? __ldg(p + W + 1) : bval;
    return Blend<SrcT, DstT>::run(v00, v01, v10, v11, w);
}
template <typename SrcT, typename DstT>
__device__ __forceinline__ DstT rim_out(const SrcT* __restrict__ src, int H, int W, int ix, int iy, const Weights<SrcT>& w, SrcT bval,
                                        const OutScale& q) {
    if constexpr (K2Quant<SrcT, DstT>::value) return quantise<DstT>(remap_rim<float, float>(src, H, W, ix, iy, w, bval), q);
    else return remap_rim<SrcT, DstT>(src, H, W, ix, iy, w, bval);
}

// the extra terms of a lens (LensExt, packed after the LensPack slots): eight 16-byte loads
__device__ __forceinline__ void load_lens_ext(const double* lens_dev, LensExt& E) {
    const double2* lp = reinterpret_cast<const double2*>(lens_dev + LP_COUNT);
    double2 q;
    q = __ldg(lp + 0); E.k4 = q.x; E.k5 = q.y;
    q = __ldg(lp + 1); E.k6 = q.x; E.s1 = q.y;
    q = __ldg(lp + 2); E.s2 = q.x; E.s3 = q.y;
    q = __ldg(lp + 3); E.s4 = q.x; E.t[0] = q.y;
    q = __ldg(lp + 4); E.t[1] = q.x; E.t[2] = q.y;
    q = __ldg(lp + 5); E.t[3] = q.x; E.t[4] = q.y;
    q = __ldg(lp + 6); E.t[5] = q.x; E.t[6] = q.y;
    q = __ldg(lp + 7); E.t[7] = q.x; E.t[8] = q.y;
}

// MODE: 0 explicit maps, 1 analytic general P, 2 analytic separable P^-1 (x = x(u), y = y(v))
// EXT: the analytic map with OpenCV's rational, thin-prism and tilt terms (map_distort_ext); only MODE 1 and 2
//
// The kernel is bound by the latency of the four-neighbour gathers, not by the float64 map evaluation (with explicit
// maps it is no faster, see profiles/).  So a thread first computes the coordinates of all its K2_ROWS pixels, then
// issues all 4*K2_ROWS gathers unconditionally (pixels on the rim gather from offset 0 and are redone out of line),
// then blends and stores: 4*K2_ROWS loads in flight per thread instead of 4.
template <typename SrcT, typename DstT, int MODE, bool EXT>
__global__ void __launch_bounds__(K2_BX * K2_BY, K2_MINB) k2_remap_kernel(K2Args a) {
    static_assert(!EXT || MODE != 0, "explicit maps have no lens terms");
    const int ox = blockIdx.x * K2_BX + (threadIdx.x % K2_BX);
    const int ty = threadIdx.x / K2_BX;
    if (ox >= a.ow) return;
    const int u = ox + a.x0;
    const SrcT bval = border_cast<SrcT>(a.border);
    const int H = a.H, W = a.W, nf = a.n_frames, ow = a.ow, oh = a.oh;
    const int src_stride = H * W, dst_stride = oh * ow;      // elements; frames are < 2^31 pixels (32767^2)
    // lens constants live in registers for the whole thread.  They are read from a small device buffer, not from
    // the kernel parameters: ptxas re-materialises parameter loads at every use (one LDC per use, ~16 issue
    // slots per pixel); a global load it has to keep.
    LensConst L = a.lens;
    if (MODE == 2) {
        const double2* lp = reinterpret_cast<const double2*>(a.lens_dev);
        double2 q;
        q = __ldg(lp + 0); L.k1 = q.x; L.k2 = q.y;
        q = __ldg(lp + 1); L.k3 = q.x; L.p1 = q.y;
        q = __ldg(lp + 2); L.p2 = q.x; L.p1x2 = q.y;
        q = __ldg(lp + 3); L.p2x2 = q.x; L.fx = q.y;
        q = __ldg(lp + 4); L.fy = q.x; L.cx = q.y;
        q = __ldg(lp + 5); L.cy = q.x; L.ir[0] = q.y;
        q = __ldg(lp + 6); L.ir[2] = q.x; L.ir[4] = q.y;
        q = __ldg(lp + 7); L.ir[5] = q.x;
    }
    LensExt E;
    if constexpr (EXT) load_lens_ext(a.lens_dev, E);
    double xc = 0.0, xc2 = 0.0;
    if (MODE == 2) {
        xc = fma((double)u, L.ir[0], L.ir[2]);
        xc2 = dmul(xc, xc);
    }
    const int oy0 = blockIdx.y * (K2_BY * K2_ROWS) + ty;

    int off[K2_ROWS];            // element offset of the top-left neighbour; 0 for rim pixels (done in the second pass)
    int cix[K2_ROWS], ciy[K2_ROWS];
    Weights<SrcT> wt[K2_ROWS];
    unsigned rim = 0, live = 0;  // bit j: pixel j lies on the rim / row j exists
#pragma unroll
    for (int j = 0; j < K2_ROWS; ++j) {
        const int oy = oy0 + j * K2_BY;
        const int v = (oy < oh ? oy : oh - 1) + a.y0;
        float mx, my;
        if (MODE == 2) {
            const double y = fma((double)v, L.ir[4], L.ir[5]);
            if constexpr (EXT) map_distort_ext(L, E, xc, y, xc2, dmul(y, y), mx, my);
            else map_distort(L, xc, y, xc2, dmul(y, y), mx, my);
        } else if (MODE == 1) {
            if constexpr (EXT) undistort_map_ext(L, E, u, v, mx, my);
            else undistort_map(L, u, v, mx, my);
        } else {
            mx = __ldg(a.mapx + v * W + u);
            my = __ldg(a.mapy + v * W + u);
        }
        const FixedCoord c = fixed_coord_fast(mx, my);
        const bool inner = (unsigned)c.ix < (unsigned)(W - 1) && (unsigned)c.iy < (unsigned)(H - 1);
        off[j] = inner ? c.iy * W + c.ix : 0;
        cix[j] = c.ix; ciy[j] = c.iy;
        wt[j].set(c);
        if (oy < oh) { live |= 1u << j; if (!inner) rim |= 1u << j; }
    }

    const bool tiny = W < 2 || H < 2;                     // no interior 2x2 window exists: offset 0 + 1 + W would overrun
    if (!tiny) {
        const SrcT* src = (const SrcT*)a.src;
        DstT* dst = (DstT*)a.dst + (oy0 * ow + ox);
        const unsigned fast = live & ~rim;
#pragma unroll 1
        for (int f = 0; f < nf; ++f) {
            SrcT v00[K2_ROWS], v01[K2_ROWS], v10[K2_ROWS], v11[K2_ROWS];
#pragma unroll
            for (int j = 0; j < K2_ROWS; ++j) {
                const SrcT* p = src + off[j];
                v00[j] = __ldg(p); v01[j] = __ldg(p + 1); v10[j] = __ldg(p + W); v11[j] = __ldg(p + W + 1);
            }
#pragma unroll
            for (int j = 0; j < K2_ROWS; ++j)
                if (fast & (1u << j)) dst[j * K2_BY * ow] = blend_out<SrcT, DstT>(v00[j], v01[j], v10[j], v11[j], wt[j], a.q);
            src += src_stride;
            dst += dst_stride;
        }
    } else {
        rim = live;
    }
    // second pass, rare: pixels whose 2x2 window touches or leaves the frame
    if (rim) {
        const SrcT* src = (const SrcT*)a.src;
        DstT* dst = (DstT*)a.dst + (oy0 * ow + ox);
        for (int f = 0; f < nf; ++f) {
#pragma unroll
            for (int j = 0; j < K2_ROWS; ++j)
                if (rim & (1u << j)) dst[j * K2_BY * ow] = rim_out<SrcT, DstT>(src, H, W, cix[j], ciy[j], wt[j], bval, a.q);
            src += src_stride;
            dst += dst_stride;
        }
    }
}

// ------------------------------------------------------------------------------------------------------------
// Tiled variant (float32 sources — the chain; uint16 / uint8 batches): the source window of a 64x16 output tile is
// staged in shared memory by ONE TMA box per frame and the four neighbours are gathered from there.  The L1 path above
// spends ~8 L1 wavefronts per 32 pixels on the gather (unaligned, two rows) and is bound by them; shared memory serves the
// same gather in ~4-5 conflict-free wavefronts, TMA moves whole lines, and the frames of a launch are ring-buffered so the
// box of frame f+1 lands while frame f is blended.
//   * the box position is ESTIMATED by warp 0 from nine sample pixels of the tile (3 x 3; exact coordinates, a 3-pixel
//     margin, clamped to the frame) and the boxes of the first frames are issued at once: their DRAM latency overlaps the
//     coordinate phase of the other warps;
//   * coordinates / weights / shared offsets of the tile's pixels are then computed once (4 pixels per thread) and every
//     pixel is classified against that box: inside -> gathered from shared memory; window entirely outside the frame ->
//     the border value (written once per frame, no reads); anything else (frame rim, or outside the box: a fraction of a
//     percent) -> "slow": gathered from global memory with per-neighbour border handling.  A tile whose window does not fit
//     a box at all (stronger distortion than the launch geometry was chosen for) is all "slow": correct for any map;
//   * results leave by predicated per-pixel stores (full 128-byte lines per warp).
template <int TW_, int TH_, int BW_, int BH_, int NBUF_, int MINB_> struct KtGeom {
    static constexpr int TW = TW_, TH = TH_, BW = BW_, BH = BH_, NBUF = NBUF_, MINB = MINB_;
};
#ifndef KT_NBUF_V
#define KT_NBUF_V 5
#endif
#ifndef KT_MINB_V
#define KT_MINB_V 4
#endif
// 28 rows x 5 boxes in flight instead of 32 x 4 (same shared memory): the moderate 4096x3000 lens needs 27 rows, and the kernel
// waits on box arrival (19.6 vs 20.1 us per frame); lenses that need 29-32 rows take the 96x32 geometry
#ifndef KT_BH0
#define KT_BH0 28
#endif
typedef KtGeom<64, 16, 80, KT_BH0, KT_NBUF_V, KT_MINB_V> KtG0;       // every tile of a realistic lens (float32 frames)
typedef KtGeom<64, 16, 96, 32, 4, KT_MINB_V> KtG1;       // strong lenses (SURVEY's 8192^2 lens needs 84 columns), 16-bit / 8-bit frames
typedef KtGeom<64, 16, 112, 48, 2, 4> KtG2;                      // very strong distortion (window up to ~1.5 x the tile)
typedef KtGeom<32, 16, 112, 64, 2, 4> KtG3;                      // extreme distortion / large shear
constexpr int KT_THREADS = 256;
constexpr int KT_MARGIN = 3;                                     // pixels added around the estimated window
// box width per source type: 16-byte origin granularity costs up to 3 / 7 / 15 extra columns (float32 / uint16 / uint8)
template <typename SrcT, typename G> struct KtBox {
    static constexpr int BW = sizeof(SrcT) == 1 ? G::BW + 16 : G::BW, GRAN = 16 / (int)sizeof(SrcT), BYTES = BW * G::BH * (int)sizeof(SrcT);
};
template <typename SrcT, typename G> constexpr int kt_smem() { return G::NBUF * KtBox<SrcT, G>::BYTES + 128; }

// predicated global store: a plain `if (flag) *p = v` lets ptxas wrap the whole gather of that pixel in a branch.
// No "memory" clobber: these stores write output pixels that nothing in the kernel reads back, and a clobber would stop
// the compiler from hoisting the next pixel's shared-memory gathers above this pixel's store (serialised LDS latency).
__device__ __forceinline__ void st_if(float* p, float v, unsigned flag) {
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %2, 0;\n\t@q st.global.f32 [%0], %1;\n\t}" ::"l"(p), "f"(v), "r"(flag));
}
__device__ __forceinline__ void st_if(double* p, double v, unsigned flag) {
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %2, 0;\n\t@q st.global.f64 [%0], %1;\n\t}" ::"l"(p), "d"(v), "r"(flag));
}
__device__ __forceinline__ void st_if(uint16_t* p, uint16_t v, unsigned flag) {
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %2, 0;\n\t@q st.global.u16 [%0], %1;\n\t}" ::"l"(p), "h"(v), "r"(flag));
}
__device__ __forceinline__ void st_if(uint8_t* p, uint8_t v, unsigned flag) {
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %2, 0;\n\t@q st.global.u8 [%0], %1;\n\t}" ::"l"(p), "r"((unsigned)v), "r"(flag));
}
struct KtLens { LensConst L; };
template <int MODE> __device__ __forceinline__ void kt_load_lens(const K2Args& a, LensConst& L) {
    L = a.lens;
    if (MODE == 2) {
        const double2* lp = reinterpret_cast<const double2*>(a.lens_dev);
        double2 q;
        q = __ldg(lp + 0); L.k1 = q.x; L.k2 = q.y;
        q = __ldg(lp + 1); L.k3 = q.x; L.p1 = q.y;
        q = __ldg(lp + 2); L.p2 = q.x; L.p1x2 = q.y;
        q = __ldg(lp + 3); L.p2x2 = q.x; L.fx = q.y;
        q = __ldg(lp + 4); L.fy = q.x; L.cx = q.y;
        q = __ldg(lp + 5); L.cy = q.x; L.ir[0] = q.y;
        q = __ldg(lp + 6); L.ir[2] = q.x; L.ir[4] = q.y;
        q = __ldg(lp + 7); L.ir[5] = q.x;
    }
}
// fixed-point source coordinate of output pixel (u, v) (full-frame coordinates)
template <int MODE, bool EXT>
__device__ __forceinline__ FixedCoord kt_coord(const K2Args& a, const LensConst& L, const LensExt& E, int u, int v, double dv, double xc,
                                               double xc2) {
    float mx, my;
    if (MODE == 2) {
        const double y = fma(dv, L.ir[4], L.ir[5]);                 // dv == (double)v
        if constexpr (EXT) map_distort_ext(L, E, xc, y, xc2, dmul(y, y), mx, my);
        else map_distort(L, xc, y, xc2, dmul(y, y), mx, my);
    } else if (MODE == 1) {
        if constexpr (EXT) undistort_map_ext(L, E, u, v, mx, my);
        else undistort_map(L, u, v, mx, my);
    } else {
        mx = __ldg(a.mapx + v * a.W + u);
        my = __ldg(a.mapy + v * a.W + u);
    }
    return fixed_coord_fast(mx, my);
}

// packed per-pixel state of a tile (the coordinate cache, see below): bits 0..13 offset of the top-left neighbour inside
// the staged box, 14..18 fx, 19..23 fy (1/32-pixel phases), bit 31 = window entirely outside the frame (the border value
// itself, as OpenCV), bit 30 = "slow" pixel (window on the frame rim or not inside the box): redone from global memory.
constexpr unsigned KP_OUTSIDE = 0x80000000u, KP_SLOW = 0x40000000u;

// CMODE 0: coordinates computed, nothing cached (explicit maps; cache switched off)
//       1: coordinates computed and written to the context's coordinate cache (first launch for a lens / window)
//       2: coordinates read from the cache: 4 bytes per pixel instead of ~45 float64 operations and ~90 instructions.
// The lens is constant per context, so the analytic evaluation — what bounds a ONE-frame launch (119 instructions per pixel,
// 65 us per 4096x3000 frame, issue bound: profiles/r2_k2_single_analytic_ncu_full.txt) — is paid once, not once per call.
template <typename SrcT, typename DstT, int MODE, typename G, int CMODE, bool EXT>
__global__ void __launch_bounds__(KT_THREADS, G::MINB) k2_tiled_kernel(const __grid_constant__ CUtensorMap tm_src, K2Args a) {
    static_assert(!EXT || (MODE != 0 && CMODE != 2), "EXT: analytic maps that are evaluated");
    constexpr int KT_TW = G::TW, KT_TH = G::TH, KT_BH = G::BH, KT_NBUF = G::NBUF;
    constexpr int KT_PX = KT_TW * KT_TH / KT_THREADS, KT_RSTEP = KT_THREADS / KT_TW;
    constexpr int BW = KtBox<SrcT, G>::BW, KT_BOX_BYTES = KtBox<SrcT, G>::BYTES, GRAN = KtBox<SrcT, G>::GRAN;
    static_assert(BW * KT_BH <= (1 << 14), "box offset must fit 14 bits of the packed word");
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t* full = (uint64_t*)(smem + KT_NBUF * KT_BOX_BYTES);
    int* est = (int*)(smem + KT_NBUF * KT_BOX_BYTES + 64);      // bx, by (bx < 0: no box)
    const int tid = threadIdx.x;
    const int c = tid % KT_TW, r0 = tid / KT_TW;               // rows r0 + RSTEP * j
    const int tx0 = blockIdx.x * KT_TW, ty0 = blockIdx.y * KT_TH;
    const int tile = blockIdx.y * gridDim.x + blockIdx.x;
    const int ox = tx0 + c;
    const int oy0 = ty0 + r0;
    const int H = a.H, W = a.W, nf = a.n_frames, ow = a.ow, oh = a.oh;
    const int u = (ox < ow ? ox : ow - 1) + a.x0;

    auto issue = [&](int f, int bx, int by) {
        uint64_t* bar = &full[f % KT_NBUF];
        mbar_expect_tx(bar, KT_BOX_BYTES);
        tma_load_3d(smem + (f % KT_NBUF) * KT_BOX_BYTES, &tm_src, bar, bx, by, f);
    };
    unsigned pk[KT_PX];
    int bx, by;
    if (CMODE == 2) {
        // ---- cached coordinates: the box position comes with the tile, its boxes are issued before anything else ----
        const int2 hdr = __ldg(a.chdr + tile);
        bx = hdr.x; by = hdr.y;
        if (tid == 0) {
            for (int b = 0; b < KT_NBUF; ++b) mbar_init(&full[b], 1);
            mbar_init_fence();
            if (bx >= 0) for (int f = 0; f < KT_NBUF && f < nf; ++f) issue(f, bx, by);
        }
        const unsigned* cp = a.cpack + ((size_t)tile * KT_PX) * KT_THREADS + tid;
#pragma unroll
        for (int j = 0; j < KT_PX; ++j) pk[j] = __ldg(cp + j * KT_THREADS);
    } else {
        if (tid == 0) {
            for (int b = 0; b < KT_NBUF; ++b) mbar_init(&full[b], 1);
            mbar_init_fence();
        }
        LensConst L;
        kt_load_lens<MODE>(a, L);
        LensExt E;
        if constexpr (EXT) load_lens_ext(a.lens_dev, E);
        // ---- the staged box: position ESTIMATED by warp 0 from nine sample pixels of the tile (3 x 3: corners, edge
        // midpoints, centre; exact coordinates, KT_MARGIN pixels added all round) and clamped to the frame, so that
        // "inside the box" implies "all four neighbours exist".  Thread 0 issues the boxes of the first frames at once:
        // their DRAM latency overlaps the coordinate phase of the other warps.
        if (tid < 32) {
            const int x1 = (tx0 + KT_TW <= ow ? tx0 + KT_TW : ow) - 1, y1 = (ty0 + KT_TH <= oh ? ty0 + KT_TH : oh) - 1;
            const int kx = tid % 3, ky = (tid / 3) % 3;
            const int sx = kx == 0 ? tx0 : (kx == 1 ? x1 : (tx0 + x1) / 2);
            const int sy = ky == 0 ? ty0 : (ky == 1 ? y1 : (ty0 + y1) / 2);
            int ex0 = 0x7fffffff, ex1 = -1, ey0 = 0x7fffffff, ey1 = -1;
            if (tid < 9) {
                const int su = sx + a.x0, sv = sy + a.y0;
                const double sxc = MODE == 2 ? fma((double)su, L.ir[0], L.ir[2]) : 0.0;
                const FixedCoord fc = kt_coord<MODE, EXT>(a, L, E, su, sv, (double)sv, sxc, dmul(sxc, sxc));
                if (!(fc.ix < -1 || fc.ix > W - 1 || fc.iy < -1 || fc.iy > H - 1)) {       // outside the frame: nothing to stage
                    const int qx = fc.ix < 0 ? 0 : (fc.ix > W - 2 ? W - 2 : fc.ix), qy = fc.iy < 0 ? 0 : (fc.iy > H - 2 ? H - 2 : fc.iy);
                    ex0 = ex1 = qx; ey0 = ey1 = qy;
                }
            }
            ex0 = __reduce_min_sync(0xffffffffu, ex0); ex1 = __reduce_max_sync(0xffffffffu, ex1);
            ey0 = __reduce_min_sync(0xffffffffu, ey0); ey1 = __reduce_max_sync(0xffffffffu, ey1);
            int ebx = ex0 - KT_MARGIN, eby = ey0 - KT_MARGIN;
            ebx = (ebx < 0 ? 0 : ebx) & ~(GRAN - 1);
            eby = eby < 0 ? 0 : eby;
            const bool have = ex1 >= 0 && (ex1 + 1 + KT_MARGIN - ebx) < BW && (ey1 + 1 + KT_MARGIN - eby) < KT_BH && W >= 2 && H >= 2;
            if (tid == 0) {
                if (have) for (int f = 0; f < KT_NBUF && f < nf; ++f) issue(f, ebx, eby);
                est[0] = have ? ebx : -1; est[1] = eby;
                if (CMODE == 1) a.chdr_w[tile] = make_int2(have ? ebx : -1, eby);
            }
        }
        double xc = 0.0, xc2 = 0.0;
        if (MODE == 2) {
            xc = fma((double)u, L.ir[0], L.ir[2]);
            xc2 = dmul(xc, xc);
        }
        // (double)v of the thread's rows by exact additions: one I2F per thread instead of one per pixel.  Rows / columns
        // beyond the output window are not clamped for the analytic map: such pixels are never stored or gathered.
        const double dv0 = (double)(oy0 + a.y0);
        int cix[KT_PX], ciy[KT_PX];
#pragma unroll
        for (int j = 0; j < KT_PX; ++j) {
            const int oy = oy0 + j * KT_RSTEP;
            const int v = (MODE == 0 ? (oy < oh ? oy : oh - 1) : oy) + a.y0;
            const FixedCoord fc = kt_coord<MODE, EXT>(a, L, E, u, v, dadd(dv0, (double)(j * KT_RSTEP)), xc, xc2);
            cix[j] = fc.ix; ciy[j] = fc.iy;
            pk[j] = (unsigned)(fc.fx << 14) | (unsigned)(fc.fy << 19);
        }
        __syncthreads();                               // the estimate is published (and the barriers are initialised)
        bx = est[0]; by = est[1];
        // a pixel reads its 2 x 2 window from the box iff  bx <= ix < bx + limx  and  by <= iy < by + limy
        const unsigned limx = bx >= 0 ? (unsigned)((bx + BW - 1 < W - 1 ? bx + BW - 1 : W - 1) - bx) : 0u;
        const unsigned limy = bx >= 0 ? (unsigned)((by + KT_BH - 1 < H - 1 ? by + KT_BH - 1 : H - 1) - by) : 0u;
#pragma unroll
        for (int j = 0; j < KT_PX; ++j) {
            const int dx = cix[j] - bx, dy = ciy[j] - by;
            const bool inb = (unsigned)dx < limx && (unsigned)dy < limy;
            const bool outside = cix[j] >= W || cix[j] + 1 < 0 || ciy[j] >= H || ciy[j] + 1 < 0;
            pk[j] |= inb ? (unsigned)(dy * BW + dx) : (outside ? KP_OUTSIDE : KP_SLOW);
        }
        if (CMODE == 1) {
            unsigned* cp = a.cpack_w + ((size_t)tile * KT_PX) * KT_THREADS + tid;
#pragma unroll
            for (int j = 0; j < KT_PX; ++j) cp[j * KT_THREADS] = pk[j];
        }
    }
    const bool have_box = bx >= 0;
    // ---- unpack: shared-memory offset, the four weights (OpenCV's own 32 x 32 table, L1-resident), pixel classes ----
    int so[KT_PX];
    Weights<SrcT> wt[KT_PX];
    unsigned fast = 0, slow = 0, outm = 0;
    const bool col_live = ox < ow;
#pragma unroll
    for (int j = 0; j < KT_PX; ++j) {
        const bool live = col_live && oy0 + j * KT_RSTEP < oh;
        const unsigned w = pk[j];
        so[j] = (w & (KP_OUTSIDE | KP_SLOW)) ? 0 : (int)(w & 0x3fffu);
        wt[j].lookup((w >> 14) & 1023u, a.wtab);
        if (live) {
            if (w & KP_OUTSIDE) outm |= 1u << j;
            else if (w & KP_SLOW) slow |= 1u << j;
            else fast |= 1u << j;
        }
    }
    if (CMODE == 2) __syncthreads();                   // the barriers are initialised for everyone

    // "slow" pixels (window on the frame rim, or a tile the box does not cover): per-neighbour border handling from global
    // memory with coordinates recomputed — a fraction of a percent of the pixels, kept off the hot path
    auto slow_pixel = [&](const SrcT* src, int j) -> DstT {
        LensConst L2;
        kt_load_lens<MODE>(a, L2);
        LensExt E2;
        if constexpr (EXT) load_lens_ext(a.lens_dev, E2);
        const int oy = oy0 + j * KT_RSTEP;
        const int v = (MODE == 0 ? (oy < oh ? oy : oh - 1) : oy) + a.y0;
        const double sxc = MODE == 2 ? fma((double)u, L2.ir[0], L2.ir[2]) : 0.0;
        const FixedCoord fc = kt_coord<MODE, EXT>(a, L2, E2, u, v, (double)v, sxc, dmul(sxc, sxc));
        Weights<SrcT> w;
        w.set(fc);
        return rim_out<SrcT, DstT>(src, H, W, fc.ix, fc.iy, w, border_cast<SrcT>(a.border), a.q);
    };
    const DstT bout = border_out<SrcT, DstT>(border_cast<SrcT>(a.border), a.q);

    const int src_stride = H * W, dst_stride = oh * ow;
    const SrcT* src = (const SrcT*)a.src;
    DstT* dst = (DstT*)a.dst + (oy0 * ow + ox);
    const int dstep = KT_RSTEP * ow;
#pragma unroll 1
    for (int f = 0; f < nf; ++f) {
        if (have_box) {
            mbar_wait(&full[f % KT_NBUF], (f / KT_NBUF) & 1);
            const SrcT* box = (const SrcT*)(smem + (f % KT_NBUF) * KT_BOX_BYTES);
#pragma unroll
            for (int j = 0; j < KT_PX; ++j) {
                const SrcT* p = box + so[j];
                const DstT r = blend_out<SrcT, DstT>(p[0], p[1], p[BW], p[BW + 1], wt[j], a.q);
                st_if(dst + j * dstep, r, fast & (1u << j));            // predicated store, no branch around the gather
            }
        }
        if (outm) {
#pragma unroll
            for (int j = 0; j < KT_PX; ++j)
                if (outm & (1u << j)) dst[j * dstep] = bout;
        }
        if (slow) {
#pragma unroll 1
            for (int j = 0; j < KT_PX; ++j)
                if (slow & (1u << j)) dst[j * dstep] = slow_pixel(src, j);
        }
        src += src_stride;
        dst += dst_stride;
        if (have_box) {
            __syncthreads();                           // everyone is done with this buffer
            if (tid == 0 && f + KT_NBUF < nf) issue(f + KT_NBUF, bx, by);
        }
    }
}

template <typename T> static CUtensorMapDataType kt_dtype() {
    return sizeof(T) == 8 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT64 : sizeof(T) == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
         : sizeof(T) == 2 ? CU_TENSOR_MAP_DATA_TYPE_UINT16 : CU_TENSOR_MAP_DATA_TYPE_UINT8;
}

// ------------------------------------------------------------------------------------------------------------
// Cached-coordinate variant: a PERSISTENT kernel over the work items (tile, frame) of a launch, tile-major, each CTA a
// contiguous range.  Thread 0 keeps a ring of KC_NBUF items in flight — the source box of the item (one TMA box) and,
// for the first item of a tile, the tile's packed coordinates (one 4 KB bulk copy), both completing on the item's
// mbarrier — so DRAM latency is covered across tiles as well as across frames: a ONE-frame launch streams like a batch
// (the analytic kernel above serialises box latency -> blend -> store per CTA and is issue bound on top of that).
// Per item: wait, (new tile: unpack offsets, weights from OpenCV's table, pixel classes), four shared-memory gathers and
// the blend per pixel, predicated per-pixel stores.  No lens arithmetic except for "slow" pixels.
#ifndef KC_NBUF
#define KC_NBUF 3
#endif
template <typename G> struct KcGeom { static constexpr int NBUF = G::BW * G::BH * 4 > 16384 ? 2 : KC_NBUF; };
constexpr int KC_MAXT = 256;

#ifndef KC_MINB
#define KC_MINB 3           // 85 registers: 46 vs 51 us for one 4096x3000 frame with 4 CTAs of 64 registers
#endif
// EXT: the lens has extra terms, which the "slow" pixels' recomputed coordinates need
template <typename SrcT, typename DstT, typename G, bool EXT>
__global__ void __launch_bounds__(KT_THREADS, KC_MINB)
k2_cached_kernel(const __grid_constant__ CUtensorMap tm_src, K2Args a, int tiles_x, long long n_items) {
    constexpr int KT_TW = G::TW, KT_TH = G::TH, KT_BH = G::BH, NBUF = KcGeom<G>::NBUF;
    constexpr int KT_PX = KT_TW * KT_TH / KT_THREADS, KT_RSTEP = KT_THREADS / KT_TW;
    constexpr int BW = KtBox<SrcT, G>::BW, BOX_BYTES = KtBox<SrcT, G>::BYTES;
    constexpr int PK_BYTES = KT_TW * KT_TH * 4, SLOT = BOX_BYTES + PK_BYTES;
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t* full = (uint64_t*)(smem + NBUF * SLOT);
    int* meta = (int*)(smem + NBUF * SLOT + 64);               // per slot: the item's tile has a box
    int2* hdrs = (int2*)(smem + NBUF * SLOT + 128);             // box origins of this CTA's tiles (KC_MAXT of them)
    const int tid = threadIdx.x;
    const int c = tid % KT_TW, r0 = tid / KT_TW;
    const int H = a.H, W = a.W, nf = a.n_frames, ow = a.ow, oh = a.oh;
    // CTA b owns the tiles b, b + grid, b + 2 grid, ... (all frames of a tile back to back): the CTAs running at the same
    // time work on neighbouring tiles, whose source boxes overlap (a box is 2.5 x the tile's area) — the overlap is then
    // served by L2 instead of being read from DRAM again (contiguous ranges per CTA read 2.3 x the algorithmic bytes).
    const int n_tiles = (int)(n_items / nf);
    const int my_tiles = ((int)blockIdx.x < n_tiles) ? (n_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
    if (my_tiles == 0) return;
    const int n_mine = my_tiles * nf;                           // items of this CTA
    int p_t = 0, p_f = 0, p_k = 0;                              // thread 0: the next item to prefetch = (tile index p_t of this CTA, frame p_f)
    // the box origins of this CTA's tiles come to shared memory first: thread 0 must not wait for a global load per item
    for (int t = tid; t < KC_MAXT && t < my_tiles; t += KT_THREADS) hdrs[t] = __ldg(a.chdr + blockIdx.x + t * gridDim.x);
    __syncthreads();

    auto issue = [&]() {                                        // thread 0: prefetch item lo + p_k = (p_tile, p_f)
        const int slot = p_k % NBUF;
        const int p_tile = blockIdx.x + p_t * gridDim.x;
        const int2 hdr = p_t < KC_MAXT ? hdrs[p_t] : __ldg(a.chdr + p_tile);
        const bool carries = p_f == 0;
        const bool box = hdr.x >= 0;
        meta[slot] = box ? 1 : 0;
        if (box || carries) {
            uint8_t* base = smem + slot * SLOT;
            mbar_expect_tx(&full[slot], (box ? BOX_BYTES : 0) + (carries ? PK_BYTES : 0));
            if (box) tma_load_3d(base, &tm_src, &full[slot], hdr.x, hdr.y, p_f);
            if (carries) bulk_load_1d(base + BOX_BYTES, a.cpack + (size_t)p_tile * (KT_TW * KT_TH), PK_BYTES, &full[slot]);
        }
        ++p_k;
        if (++p_f == nf) { p_f = 0; ++p_t; }
    };
    if (tid == 0) {
        for (int b = 0; b < NBUF; ++b) mbar_init(&full[b], 1);
        mbar_init_fence();
        for (int k = 0; k < NBUF && k < n_mine; ++k) issue();
    }
    __syncthreads();

    int so[KT_PX];
    Weights<SrcT> wt[KT_PX];
    unsigned fast = 0, slow = 0, outm = 0, phases = 0;
    int tx0 = 0, ty0 = 0;
    const DstT bout = border_out<SrcT, DstT>(border_cast<SrcT>(a.border), a.q);
    const int src_stride = H * W, dst_stride = oh * ow;

    // "slow" pixels (window on the frame rim, or a tile the box does not cover): coordinates recomputed from the lens, per-
    // neighbour border handling from global memory — a fraction of a percent of the pixels
    auto slow_pixel = [&](const SrcT* src, int j) -> DstT {
        float mx, my;
        if constexpr (EXT) {
            LensExt E;
            load_lens_ext(a.lens_dev, E);
            undistort_map_ext(a.lens, E, tx0 + c + a.x0, ty0 + r0 + j * KT_RSTEP + a.y0, mx, my);
        } else {
            undistort_map(a.lens, tx0 + c + a.x0, ty0 + r0 + j * KT_RSTEP + a.y0, mx, my);
        }
        const FixedCoord fc = fixed_coord_fast(mx, my);
        Weights<SrcT> w;
        w.set(fc);
        return rim_out<SrcT, DstT>(src, H, W, fc.ix, fc.iy, w, border_cast<SrcT>(a.border), a.q);
    };

    int tile = blockIdx.x, f = 0, slot = 0;
#pragma unroll 1
    for (int k = 0; k < n_mine; ++k) {
        const bool carries = f == 0;
        const bool have_box = meta[slot] != 0;
        const uint8_t* base = smem + slot * SLOT;
        if (have_box || carries) {
            mbar_wait(&full[slot], (phases >> slot) & 1u);
            phases ^= 1u << slot;
        }
        if (carries) {
            // a new tile: unpack its coordinates
            const int tyi = tile / tiles_x;
            tx0 = (tile - tyi * tiles_x) * KT_TW;
            ty0 = tyi * KT_TH;
            const unsigned* pk = (const unsigned*)(base + BOX_BYTES) + tid;
            const bool col_live = tx0 + c < ow;
            fast = slow = outm = 0;
#pragma unroll
            for (int j = 0; j < KT_PX; ++j) {
                const unsigned w = pk[j * KT_THREADS];
                const bool live = col_live && ty0 + r0 + j * KT_RSTEP < oh;
                so[j] = (w & (KP_OUTSIDE | KP_SLOW)) ? 0 : (int)(w & 0x3fffu);
                wt[j].lookup((w >> 14) & 1023u, a.wtab);
                if (live) {
                    if (w & KP_OUTSIDE) outm |= 1u << j;
                    else if (w & KP_SLOW) slow |= 1u << j;
                    else fast |= 1u << j;
                }
            }
        }
        const SrcT* src = (const SrcT*)a.src + (size_t)f * src_stride;
        DstT* dst = (DstT*)a.dst + (size_t)f * dst_stride + ((ty0 + r0) * ow + tx0 + c);
        const int dstep = KT_RSTEP * ow;
        if (have_box) {
            const SrcT* box = (const SrcT*)base;
#pragma unroll
            for (int j = 0; j < KT_PX; ++j) {
                const SrcT* p = box + so[j];
                const DstT r = blend_out<SrcT, DstT>(p[0], p[1], p[BW], p[BW + 1], wt[j], a.q);
                st_if(dst + j * dstep, r, fast & (1u << j));
            }
        }
        if (outm) {
#pragma unroll
            for (int j = 0; j < KT_PX; ++j)
                if (outm & (1u << j)) dst[j * dstep] = bout;
        }
        if (slow) {
#pragma unroll 1
            for (int j = 0; j < KT_PX; ++j)
                if (slow & (1u << j)) dst[j * dstep] = slow_pixel(src, j);
        }
        __syncthreads();                               // everyone is done with this slot
        if (tid == 0 && p_k < n_mine) issue();
        if (++f == nf) { f = 0; tile += gridDim.x; }
        if (++slot == NBUF) slot = 0;
    }
}

template <typename SrcT, typename DstT, typename G, bool EXT>
static cudaError_t launch_cached_g(const K2Args& a, cudaStream_t st) {
    CUtensorMap tm;
    if (!make_tensor_map(&tm, kt_dtype<SrcT>(), sizeof(SrcT), a.src, a.W, a.H, a.n_frames, KtBox<SrcT, G>::BW, G::BH)) return cudaErrorInvalidValue;
    const int tiles_x = (a.ow + G::TW - 1) / G::TW, tiles_y = (a.oh + G::TH - 1) / G::TH;
    const long long n_items = (long long)tiles_x * tiles_y * a.n_frames;
    if (n_items > 0x7fffffffLL) return cudaErrorInvalidValue;
    constexpr int SMEM = KcGeom<G>::NBUF * (KtBox<SrcT, G>::BYTES + G::TW * G::TH * 4) + 128 + KC_MAXT * 8;
    auto kern = k2_cached_kernel<SrcT, DstT, G, EXT>;
    cudaError_t e = cudaSuccess;
    const int per_sm = blocks_per_sm_cached((const void*)kern, KT_THREADS, SMEM, &e);
    if (e != cudaSuccess) return e;
    long long grid = (long long)(a.sm_count > 0 ? a.sm_count : 148) * per_sm;
    if (grid > (long long)tiles_x * tiles_y) grid = (long long)tiles_x * tiles_y;
    kern<<<(unsigned)grid, KT_THREADS, SMEM, st>>>(tm, a, tiles_x, n_items);
    return cudaGetLastError();
}

static bool k2_tiled_eligible(const K2Args& a, int src_dtype, int dst_dtype) {
    const bool pair = (src_dtype == DT_F32 && dst_dtype >= DT_U8 && dst_dtype <= DT_F64) || (src_dtype == DT_U16 && dst_dtype == DT_U16) ||
                      (src_dtype == DT_U8 && dst_dtype == DT_U8);
    if (!pair) return false;
    if (a.W < 2 || a.H < 2) return false;
    if (((size_t)a.W * dtype_size(src_dtype)) % 16 || ((uintptr_t)a.src) % 16) return false;
    return tensor_map_encoder() != nullptr;
}

template <typename SrcT, typename DstT, typename G>
static cudaError_t launch_tiled_g(const K2Args& a, cudaStream_t st) {
    CUtensorMap tm;
    if (!make_tensor_map(&tm, kt_dtype<SrcT>(), sizeof(SrcT), a.src, a.W, a.H, a.n_frames, KtBox<SrcT, G>::BW, G::BH)) return cudaErrorInvalidValue;
    dim3 grid((a.ow + G::TW - 1) / G::TW, (a.oh + G::TH - 1) / G::TH);
    constexpr int SMEM = kt_smem<SrcT, G>();
    void (*kern)(const CUtensorMap, K2Args);
    const bool sep = a.lens.affine && a.lens.ir[1] == 0.0 && a.lens.ir[3] == 0.0;
    if (a.cpack && !a.mapx) return a.lens_ext ? launch_cached_g<SrcT, DstT, G, true>(a, st) : launch_cached_g<SrcT, DstT, G, false>(a, st);
    if constexpr (K2Quant<SrcT, DstT>::value) if (a.mapx) return cudaErrorNotSupported;    // the chain remaps with the analytic map only
    if (a.mapx) kern = k2_tiled_kernel<SrcT, DstT, 0, G, 0, false>;
    else if (a.lens_ext && a.cpack_w) kern = sep ? k2_tiled_kernel<SrcT, DstT, 2, G, 1, true> : k2_tiled_kernel<SrcT, DstT, 1, G, 1, true>;
    else if (a.lens_ext) kern = sep ? k2_tiled_kernel<SrcT, DstT, 2, G, 0, true> : k2_tiled_kernel<SrcT, DstT, 1, G, 0, true>;
    else if (a.cpack_w) kern = sep ? k2_tiled_kernel<SrcT, DstT, 2, G, 1, false> : k2_tiled_kernel<SrcT, DstT, 1, G, 1, false>;
    else kern = sep ? k2_tiled_kernel<SrcT, DstT, 2, G, 0, false> : k2_tiled_kernel<SrcT, DstT, 1, G, 0, false>;
    if (SMEM > 48 * 1024) {
        cudaError_t e = cudaSuccess;
        blocks_per_sm_cached((const void*)kern, KT_THREADS, SMEM, &e);       // opt-in to > 48 KB, once per (device, kernel)
        if (e != cudaSuccess) return e;
    }
    kern<<<grid, KT_THREADS, SMEM, st>>>(tm, a);
    return cudaGetLastError();
}

template <typename SrcT, typename DstT>
static cudaError_t launch_tiled_t(const K2Args& a, cudaStream_t st) {
    const int g = a.geometry;
    if (g == 3) return launch_tiled_g<SrcT, DstT, KtG3>(a, st);
    if (g == 2) return launch_tiled_g<SrcT, DstT, KtG2>(a, st);
    if (g == 1) return launch_tiled_g<SrcT, DstT, KtG1>(a, st);
    return launch_tiled_g<SrcT, DstT, KtG0>(a, st);
}

// words of the coordinate cache for an output window under geometry g (whole tiles) and the number of tiles
void k2_cache_size(int g, int ow, int oh, size_t* words, size_t* tiles) {
    const int TW = g == 3 ? KtG3::TW : 64, TH = 16;
    const size_t t = (size_t)((ow + TW - 1) / TW) * ((oh + TH - 1) / TH);
    *tiles = t;
    *words = t * (size_t)(TW * TH);
}

// Host: the staged-box geometry a lens needs for an output window — the largest source window (plus margins) over all
// 64x16 tiles, from the exact map at the very 3 x 3 sample points the kernel estimates from.
// 0: 80x32 box, 1: 96x32, 2: 112x48, 3: 32-wide tiles with a 112x64 box.  `src_elem_size` sets the column granularity of the
// box origin (16 bytes: 4 / 8 / 16 columns).  `ext`: the lens' extra terms, or null for the 5-term model.  Cached per window
// by the caller (imgcorr_api.cu).
int k2_pick_geometry(const LensConst& L, const LensExt* ext, int H, int W, int x0, int y0, int ow, int oh, int src_elem_size) {
    int need_w = 0, need_h = 0;
    const int TW = 64, TH = 16;
    for (int ty = 0; ty < oh; ty += TH)
        for (int tx = 0; tx < ow; tx += TW) {
            const int x1 = (tx + TW <= ow ? tx + TW : ow) - 1, y1 = (ty + TH <= oh ? ty + TH : oh) - 1;
            int ex0 = 0x7fffffff, ex1 = -1, ey0 = 0x7fffffff, ey1 = -1;
            for (int k = 0; k < 9; ++k) {
                const int sx = (k % 3) == 0 ? tx : ((k % 3) == 1 ? x1 : (tx + x1) / 2);
                const int sy = (k / 3) == 0 ? ty : ((k / 3) == 1 ? y1 : (ty + y1) / 2);
                float mx, my;
                if (ext) undistort_map_ext(L, *ext, sx + x0, sy + y0, mx, my);
                else undistort_map(L, sx + x0, sy + y0, mx, my);
                const FixedCoord fc = fixed_coord(mx, my);
                if (fc.ix < -1 || fc.ix > W - 1 || fc.iy < -1 || fc.iy > H - 1) continue;     // outside: nothing to stage
                const int qx = fc.ix < 0 ? 0 : (fc.ix > W - 2 ? W - 2 : fc.ix), qy = fc.iy < 0 ? 0 : (fc.iy > H - 2 ? H - 2 : fc.iy);
                ex0 = qx < ex0 ? qx : ex0; ex1 = qx > ex1 ? qx : ex1; ey0 = qy < ey0 ? qy : ey0; ey1 = qy > ey1 ? qy : ey1;
            }
            if (ex1 < 0) continue;
            const int w = ex1 - ex0 + 2 + 2 * KT_MARGIN + (16 / src_elem_size - 1), h = ey1 - ey0 + 2 + 2 * KT_MARGIN;   // + 16-byte origin
            if (w > need_w) need_w = w;
            if (h > need_h) need_h = h;
        }
    const int extra = src_elem_size == 1 ? 16 : 0;          // KtBox widens 8-bit boxes by 16 columns
    if (need_w <= KtG0::BW + extra && need_h <= KtG0::BH) return 0;
    if (need_w <= KtG1::BW + extra && need_h <= KtG1::BH) return 1;
    if (need_w <= KtG2::BW + extra && need_h <= KtG2::BH) return 2;
    return 3;
}

template <bool EXT>
__global__ void __launch_bounds__(256) k2_write_maps_kernel(LensConst lens, LensExt ext, float* mapx, float* mapy, int H, int W) {
    const int u = blockIdx.x * 32 + (threadIdx.x % 32);
    const int v = blockIdx.y * 8 + (threadIdx.x / 32);
    if (u >= W || v >= H) return;
    float mx, my;
    if constexpr (EXT) undistort_map_ext(lens, ext, u, v, mx, my);
    else undistort_map(lens, u, v, mx, my);
    mapx[(size_t)v * W + u] = mx;
    mapy[(size_t)v * W + u] = my;
}

static bool separable(const LensConst& L) { return L.affine && L.ir[1] == 0.0 && L.ir[3] == 0.0; }

template <typename SrcT, typename DstT>
static cudaError_t launch_t(const K2Args& a, cudaStream_t st) {
    dim3 grid((a.ow + K2_BX - 1) / K2_BX, (a.oh + K2_BY * K2_ROWS - 1) / (K2_BY * K2_ROWS));
    if constexpr (K2Quant<SrcT, DstT>::value) if (a.mapx) return cudaErrorNotSupported;
    if (a.mapx) k2_remap_kernel<SrcT, DstT, 0, false><<<grid, K2_BX * K2_BY, 0, st>>>(a);
    else if (a.lens_ext && separable(a.lens)) k2_remap_kernel<SrcT, DstT, 2, true><<<grid, K2_BX * K2_BY, 0, st>>>(a);
    else if (a.lens_ext) k2_remap_kernel<SrcT, DstT, 1, true><<<grid, K2_BX * K2_BY, 0, st>>>(a);
    else if (separable(a.lens)) k2_remap_kernel<SrcT, DstT, 2, false><<<grid, K2_BX * K2_BY, 0, st>>>(a);
    else k2_remap_kernel<SrcT, DstT, 1, false><<<grid, K2_BX * K2_BY, 0, st>>>(a);
    return cudaGetLastError();
}

bool k2_will_tile(const K2Args& a, int src_dtype, int dst_dtype, int variant) {
    if (a.H > 32767 || a.W > 32767) return false;
    const bool want_tiles = variant == 2 || (variant == 0 && (src_dtype == DT_F32 || a.n_frames >= 4));
    return want_tiles && k2_tiled_eligible(a, src_dtype, dst_dtype);
}

cudaError_t launch_k2(const K2Args& a, int src_dtype, int dst_dtype, int variant, cudaStream_t st, int* launches) {
    if (a.n_frames <= 0 || a.ow <= 0 || a.oh <= 0) return cudaSuccess;
    if (a.H > 32767 || a.W > 32767) return cudaErrorInvalidValue;      // OpenCV's remap itself is limited to short coordinates
    if (a.x0 < 0 || a.y0 < 0 || a.x0 + a.ow > a.W || a.y0 + a.oh > a.H) return cudaErrorInvalidValue;
    if ((a.mapx == nullptr) != (a.mapy == nullptr)) return cudaErrorInvalidValue;
    if (!a.mapx && !a.lens_dev) return cudaErrorInvalidValue;
    // variant: 0 auto, 1 gathers through L1, 2 shared-memory staged tiles (float32 sources)
    // integer sources: a single frame is faster through L1 (63 vs 69 us at 4096x3000 uint16), batches through the tiles (26 vs 31)
    const bool want_tiles = variant == 2 || (variant == 0 && (src_dtype == DT_F32 || a.n_frames >= 4));
    const bool tiled = want_tiles && k2_tiled_eligible(a, src_dtype, dst_dtype);
    if (variant == 2 && !tiled) return cudaErrorNotSupported;
    if (launches) ++*launches;
    if (tiled) {
        if (src_dtype == DT_U16) return launch_tiled_t<uint16_t, uint16_t>(a, st);
        if (src_dtype == DT_U8) return launch_tiled_t<uint8_t, uint8_t>(a, st);
        if (dst_dtype == DT_U16) return launch_tiled_t<float, uint16_t>(a, st);
        if (dst_dtype == DT_U8) return launch_tiled_t<float, uint8_t>(a, st);
        return dst_dtype == DT_F32 ? launch_tiled_t<float, float>(a, st) : launch_tiled_t<float, double>(a, st);
    }
    if (src_dtype == DT_F32 && dst_dtype == DT_F32) return launch_t<float, float>(a, st);
    if (src_dtype == DT_F32 && dst_dtype == DT_F64) return launch_t<float, double>(a, st);
    if (src_dtype == DT_F32 && dst_dtype == DT_U16) return launch_t<float, uint16_t>(a, st);
    if (src_dtype == DT_F32 && dst_dtype == DT_U8) return launch_t<float, uint8_t>(a, st);
    if (src_dtype == DT_F64 && dst_dtype == DT_F64) return launch_t<double, double>(a, st);
    if (src_dtype == DT_U16 && dst_dtype == DT_U16) return launch_t<uint16_t, uint16_t>(a, st);
    if (src_dtype == DT_U8 && dst_dtype == DT_U8) return launch_t<uint8_t, uint8_t>(a, st);
    if (launches) --*launches;
    return cudaErrorInvalidValue;
}

cudaError_t launch_write_maps(const LensConst& lens, const LensExt* ext, float* mapx, float* mapy, int H, int W, cudaStream_t st,
                              int* launches) {
    if (H <= 0 || W <= 0) return cudaSuccess;
    dim3 grid((W + 31) / 32, (H + 7) / 8);
    if (ext) k2_write_maps_kernel<true><<<grid, 256, 0, st>>>(lens, *ext, mapx, mapy, H, W);
    else k2_write_maps_kernel<false><<<grid, 256, 0, st>>>(lens, LensExt{}, mapx, mapy, H, W);
    if (launches) ++*launches;
    return cudaGetLastError();
}

}  // namespace imgcorr
