// imgcorr_kernels.cuh — launch-side declarations shared by the kernel translation units
// and the C-ABI layer (imgcorr_api.cu).  Not part of the public interface (include/imgcorr.h).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "imgcorr_core.cuh"
#include "imgcorr_warp.cuh"
#include "imgcorr_ste.cuh"

namespace imgcorr {

enum DType : int { DT_U8 = 0, DT_U16 = 1, DT_F32 = 2, DT_F64 = 3 };

inline size_t dtype_size(int dt) { return dt == DT_U8 ? 1 : dt == DT_U16 ? 2 : dt == DT_F32 ? 4 : 8; }

// K1: fused dark / flat / nan_to_num / NxN median-threshold --------------------------------
struct K1Args {
    const void* raw;        // [n_frames][H][W] of raw dtype
    const float* dark;      // [H][W] or null   (offset map when FLAG_DARK_LINEAR)
    const float* ascent;    // [H][W] or null   (FLAG_DARK_LINEAR only)
    const float* flat;      // [H][W] or null
    void* out;              // [n_frames][H][W] of out dtype
    uint8_t* mask;          // [n_frames][H][W] or null
    int H, W, n_frames;
    int raw_swap;           // raw samples are big-endian uint16 (reader/RAW.py default): bytes swapped in the load
    long long raw_gap;      // bytes between the end of one raw frame and the start of the next (reader/elbin.py: 20-byte headers)
    int ksize;              // 0 (pointwise only), 3, 5
    int maps_finite;        // dark / flat hold no NaN / inf (checked once at upload)
    const float* flat_nz;   // copy of flat with zeros replaced by 1.0 (unconditional division), or null
    void* dump;             // >= 2 * grid * threads * 8 bytes of scratch: lanes without an output pixel store here
    int out_streaming;      // the output is not consumed by a following kernel of the same call (K1-only entry point): L2 evict-first
    int no_overflow;        // the calibration proves |raw - dark| / |flat| < FLT_MAX for this raw dtype: nan_to_num is the identity
    PointwiseConst pw;
    PredicateConst pred;
    OutScale q;             // integer output (U16 / U8): quantise<OutT>(float32 result, q); the identity (0, 1) outside the chain
    const void* bg;         // [n_frames][H][W] of bg_dtype, dense and native-endian, or null: frame f subtracts float32(bg[f])
                            // in place of the dark map (FLAG_DARK set, dark / ascent null)
    int bg_dtype;           // the raw dtype or DT_F32
    const double* exposures;    // [n_frames] or null (FLAG_DARK_LINEAR only): frame f evaluates the line model with
                                // exposures[f] instead of pw.exposure_time
};

// variant: 0 = pick automatically, 1 = generic tiles (plain coalesced loads), 2 = TMA-staged tiles,
//          3 = TMA streaming pipeline (3x3 and 5x5).  seg_rows: rows per work unit of the streaming kernel (0 = default)
cudaError_t launch_k1(const K1Args& a, int raw_dtype, int out_dtype, int variant, int sm_count, int seg_rows,
                      cudaStream_t stream, int* launches);
bool k1_tma_eligible(const K1Args& a, int raw_dtype, int out_dtype);
bool k1_stream_eligible(const K1Args& a, int raw_dtype, int out_dtype);
cudaError_t launch_k1_stream(const K1Args& a, int raw_dtype, int out_dtype, int sm_count, int seg_rows, cudaStream_t stream);
bool k1_stream5_eligible(const K1Args& a, int raw_dtype, int out_dtype);     // 5x5 streaming pipeline
cudaError_t launch_k1_stream5(const K1Args& a, int raw_dtype, int out_dtype, int sm_count, int seg_rows, cudaStream_t stream);

// K2: undistortion remap ---------------------------------------------------------------------
struct K2Args {
    const void* src;        // [n_frames][H][W]
    void* dst;              // [n_frames][oh][ow]
    const float* mapx;      // explicit maps [H][W] (full frame) or null -> analytic Brown-Conrady
    const float* mapy;
    int H, W, n_frames;
    int x0, y0, ow, oh;     // output window in full-frame coordinates (keep_size=False crop)
    double border;
    LensConst lens;
    const double* lens_dev;  // device copy of the lens constants (see LensPack), loaded once per thread into registers
    int geometry;            // tiled variant: staged-box geometry (k2_pick_geometry), 0 = 80x32 box for 64x16 tiles
    const float4* wtab;      // device copy of OpenCV's 32 x 32 bilinear weight table [fy][fx] = (w00, w01, w10, w11)
    // coordinate cache of the tiled variant (k2_undistort.cu): packed per-pixel words [tile][px][256] + box origin per tile
    const unsigned* cpack;   // read the cache (it is complete)
    const int2* chdr;
    unsigned* cpack_w;       // write the cache while computing (first launch for this lens / window / geometry)
    int2* chdr_w;
    int sm_count;
    OutScale q;             // F32 -> U16 / U8: the float32 blend, then quantise<DstT>(blend, q)
    int lens_ext;           // the lens has rational / thin-prism / tilt terms (LensExt at lens_dev + LP_COUNT): the EXT kernels
};
void k2_cache_size(int geometry, int ow, int oh, size_t* words, size_t* tiles);
bool k2_will_tile(const K2Args& a, int src_dtype, int dst_dtype, int variant);    // launch_k2 takes the tiled variant
int k2_pick_geometry(const LensConst& lens, const LensExt* ext, int H, int W, int x0, int y0, int ow, int oh, int src_elem_size);

// order of the doubles in K2Args::lens_dev
enum LensPack : int { LP_K1, LP_K2, LP_K3, LP_P1, LP_P2, LP_P1X2, LP_P2X2, LP_FX, LP_FY, LP_CX, LP_CY, LP_IR0, LP_IR2, LP_IR4, LP_IR5, LP_PAD, LP_COUNT };
// followed by the LensExt of the lens (its 16 doubles in declaration order), read by the EXT kernels
constexpr int LP_EXT_COUNT = LP_COUNT + (int)(sizeof(LensExt) / sizeof(double));
static_assert(sizeof(LensExt) == 16 * sizeof(double), "LensExt is packed as 16 doubles");

cudaError_t launch_k2(const K2Args& a, int src_dtype, int dst_dtype, int variant, cudaStream_t stream,
                      int* launches);
cudaError_t launch_write_maps(const LensConst& lens, const LensExt* ext, float* mapx, float* mapy, int H, int W,
                              cudaStream_t stream, int* launches);

// K3: perspective warp (cv2.warpPerspective, Lanczos4 / bicubic) ------------------------------
struct K3Args {
    const void* src;        // [n_frames][H][W]
    void* dst;              // [n_frames][dh][dw] of dst_dtype
    int H, W, dh, dw, n_frames;
    double border;          // already converted to the image dtype's value range
    WarpConst wc;
    const float* tab;       // device coefficient table [32][N] of the interpolation
    const int16_t* itab;    // uint8 images: device fixed-point weights [32][32][N*N] (null otherwise)
    int dst_dtype;          // dtype of dst: the source dtype, or U16 / U8 for a float32 source (float32 warp, then quantise)
    OutScale q;             // the scale of that quantisation
    const WarpConst* wcs;   // device table [n_frames]: frame f of the launch is warped with wcs[f] (Lanczos4, float32 /
                            // float64 sources); null: every frame with wc
};
cudaError_t launch_k3(const K3Args& a, int dtype, int interp, int variant, cudaStream_t stream, int* launches);
cudaError_t launch_k3_divide(const void* src, int dtype, const double* div, double* dst, size_t npx, int n_frames,
                             int sm_count, cudaStream_t stream, int* launches);

// K4: single-time-effect-free average (SingleTimeEffectDetection) ------------------------------
struct K4Args {
    const void* img;        // [H][W] the image being added (FIRST: images[0])
    const void* img2;       // FIRST launch only: images[1]; null for the following images
    const double* avg_in;   // [H][W] running average (noSTE) before this image (unused by the FIRST launch)
    double* avg_out;        // [H][W] running average after it (a different buffer: neighbouring tiles read avg_in)
    const double* thr_in;   // FIRST launch: caller-supplied threshold map (already times nStd) instead of the boundedFunction model, or null
    double* thr;            // [H][W] threshold = nlf(avg after the first update) * nStd
    int* n;                 // [H][W] number of values averaged per pixel
    uint8_t* mask;          // [H][W] accumulated STE mask (save_ste_indices) or null
    int H, W;
    SteConst sc;
};
cudaError_t launch_k4(const K4Args& a, int dtype, cudaStream_t stream, int* launches);

// K5: calibration-map producers (k5_producers.cu, SURVEY §8 f4) -------------------------------------------
cudaError_t launch_k5_stack_mean(const void* frames, int dtype, int n, size_t elems, const double* minus, double minus_scalar,
                                 int has_scalar, int gray3, double* out, int sm_count, cudaStream_t stream, int* launches);
cudaError_t launch_k5_scale(double* data, size_t elems, double divisor, int sm_count, cudaStream_t stream, int* launches);
cudaError_t launch_k5_subsample(const double* src, int H, int W, int sy, int sx, double* dst, cudaStream_t stream, int* launches);
cudaError_t launch_k5_linear_fit(const void* frames, int dtype, int n, size_t px, const double* xs_dev, double max_intensity, double min_ascent,
                                 double x_mid, double* offset, double* ascent, double* rmse, int sm_count, cudaStream_t stream, int* launches);

// device self-test of the float64 division sequence (selftest.cu); dev2 = {mismatches, bits of the worst seed error}
cudaError_t launch_selftest_division(int nnum, uint64_t seed, unsigned long long* dev2, cudaStream_t stream);

}  // namespace imgcorr
