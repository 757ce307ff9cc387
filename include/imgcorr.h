/* imgcorr.h — C ABI of libimgcorr.so: the B200 (sm_100a) implementation of the per-frame
 * camera-correction path of radjkarl/imgProcessor,
 *
 *     imgProcessor.camera.CameraCalibration.correct()      camera/CameraCalibration.py:351-459
 *
 * The reference is pure Python and has no FFI of its own: this header is the boundary a
 * maintainer would bind (ctypes stub in INTEGRATION.md) to route that one path to the GPU.
 * Every entry point cites the reference lines it replaces (paths relative to
 * /root/reference/imgProcessor/).
 *
 * Conventions
 *   - plain C, no torch / C++ types; all images are dense row-major [n_frames][H][W].
 *   - "dev" pointers are device pointers owned by the caller (e.g. torch tensor data_ptr()),
 *     "host" pointers are host memory; the library owns only its per-context copies of the
 *     calibration maps, scratch frames and (for the *_host entry points) pinned staging rings.
 *   - `stream` is a cudaStream_t passed as void* (NULL = the legacy default stream). Calls are
 *     asynchronous with respect to the host unless stated otherwise.
 *   - every function returns IMGCORR_OK (0) or a negative imgcorr_status; the message of the
 *     last failure on the calling thread is returned by imgcorr_last_error().  Nothing aborts,
 *     nothing throws, and there is NO CPU fallback: without a CUDA device every compute call
 *     fails with IMGCORR_ERR_CUDA.
 */
#ifndef IMGCORR_H
#define IMGCORR_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IMGCORR_VERSION 200 /* 0.2.0: round 2 added imgcorr_ste_average_thr, imgcorr_stack_mean, imgcorr_scale_f64, imgcorr_subsample_f64,
                               imgcorr_linear_fit, imgcorr_host_fingerprint, imgcorr_selftest_division and the K2 options 11, 12;
                               later added imgcorr_set_perspective and IMGCORR_DO_PERSPECTIVE (the chain's perspective stage),
                               U16 / U8 output of the chain with imgcorr_set_output_scale, imgcorr_set_perspective_frames
                               (one homography per frame in the perspective stage), and imgcorr_correct_batch_bg /
                               imgcorr_correct_host_bg (one background image per frame in place of the dark map), and
                               imgcorr_set_dark_exposures (one exposure time per frame for the linear dark model), and
                               imgcorr_set_lens_model (OpenCV's 4-, 8-, 12- and 14-coefficient lens models in K2) */

#if defined(__GNUC__)
#define IMGCORR_API __attribute__((visibility("default")))
#else
#define IMGCORR_API
#endif

typedef struct imgcorr_ctx imgcorr_ctx;

typedef enum imgcorr_status {
    IMGCORR_OK = 0,
    IMGCORR_ERR_INVALID = -1, /* bad argument (shape, dtype combination, null pointer, ...) */
    IMGCORR_ERR_CUDA = -2,    /* a CUDA runtime / driver call failed (message has the detail) */
    IMGCORR_ERR_STATE = -3,   /* e.g. undistort requested but no lens set */
    IMGCORR_ERR_NOMEM = -4
} imgcorr_status;

typedef enum imgcorr_dtype { IMGCORR_U8 = 0, IMGCORR_U16 = 1, IMGCORR_F32 = 2, IMGCORR_F64 = 3 } imgcorr_dtype;

/* medianThreshold(condition=...)  filters/medianThreshold.py:21-24 */
typedef enum imgcorr_cond { IMGCORR_COND_GT = 0, IMGCORR_COND_LT = 1 } imgcorr_cond;

/* stage switches of the fused pointwise step */
enum {
    IMGCORR_DO_DARK = 1,       /* image -= bg                           CameraCalibration.py:502      */
    IMGCORR_DO_FLAT = 2,       /* image[flat != 0] /= flat[flat != 0]   CameraCalibration.py:525-526  */
    IMGCORR_DO_NAN_TO_NUM = 4, /* image = np.nan_to_num(image)          CameraCalibration.py:561      */
    IMGCORR_DO_PERSPECTIVE = 8 /* the context's perspective warp as the chain's last stage (imgcorr_set_perspective: one
                                  matrix for every frame, or imgcorr_set_perspective_frames: matrix i for frame i of the
                                  call); read by imgcorr_correct_batch and imgcorr_correct_host only */
};

/* imgcorr_set_option keys */
enum {
    IMGCORR_OPT_K1_VARIANT = 1, /* 0 auto, 1 generic tiles, 2 TMA-staged tiles, 3 TMA streaming pipeline (3x3 and 5x5) (2-3 fail if not eligible) */
    IMGCORR_OPT_K2_VARIANT = 2, /* 0 auto, 1 gathers through L1/L2, 2 shared-memory staged tiles (float32 / uint16 / uint8 sources; fails if not eligible) */
    IMGCORR_OPT_HOST_SLOTS = 3, /* depth of the pinned / device staging ring of the *_host calls (default 4) */
    IMGCORR_OPT_K1_SEG_ROWS = 4, /* rows per work unit of the streaming K1 kernel (0 = default) */
    IMGCORR_OPT_PROFILE = 5,     /* n > 0: bracket the K1 and K2 launch of every n-th frame group of the chain with CUDA
                                    events on the launching stream (read with imgcorr_profile_read); 0 = off */
    IMGCORR_OPT_CHAIN_GROUP = 6, /* frames per K1 / K2 launch inside imgcorr_correct_batch (default 16) */
    /* ingest formats, consumed as stored in the file (SURVEY §8 f2); they apply to every raw_dev of the context until reset: */
    IMGCORR_OPT_RAW_BIG_ENDIAN = 7, /* uint16 samples are big-endian: reader/RAW.py:19-20 (littleEndian=False is its default) */
    IMGCORR_OPT_RAW_FRAME_GAP = 8,  /* bytes between the end of one raw frame and the start of the next: reader/elbin.py:23-32
                                       (a 20-byte header precedes every frame).  Not available for the *_host entry point. */
    IMGCORR_OPT_CHAIN_OVERLAP = 10, /* imgcorr_correct_batch: run K1 of the next frame group on an internal high-priority stream while K2
                                       of the current group runs on the caller's stream (default 1; 0 = everything on the caller's stream) */
    IMGCORR_OPT_K2_COORD_CACHE = 11, /* 1 (default): the first tiled K2 launch for a lens / output window stores the packed fixed-point source
                                       coordinates it computed (4 bytes per pixel of device memory, at most two windows), later launches read them
                                       instead of re-evaluating the float64 lens model; 0: evaluate on every launch */
    /* key 12 is retired and not reused */
    IMGCORR_OPT_K3_VARIANT = 9      /* 0 auto, 1 gathers through L1/L2, 2 shared-memory staged tiles (uint16 / float32 sources; fails if not eligible;
                                       a launch with a per-frame table, as imgcorr_correct_batch's per-frame homographies, is never eligible) */
};

IMGCORR_API const char* imgcorr_last_error(void);
IMGCORR_API int imgcorr_version(void);

/* Number of CUDA devices visible, or a negative status. */
IMGCORR_API int imgcorr_device_count(void);

/* ---- context: one per (device, frame shape).  Holds the device copies of the calibration maps
 * that CameraCalibration keeps in self.coeffs (camera/CameraCalibration.py:63-81). -------------- */
IMGCORR_API int imgcorr_ctx_create(int device, int height, int width, imgcorr_ctx** out_ctx);
IMGCORR_API int imgcorr_ctx_destroy(imgcorr_ctx* ctx);
IMGCORR_API int imgcorr_set_option(imgcorr_ctx* ctx, int key, int value);
/* kernels launched by this context so far (bench.py's gpu_launches claim) */
IMGCORR_API long long imgcorr_launch_count(const imgcorr_ctx* ctx);
/* Sum the event-bracketed launch durations collected since the last call (IMGCORR_OPT_PROFILE):
 * out[0] = K1 milliseconds, out[1] = frames those K1 launches processed, out[2] = K2 milliseconds, out[3] = frames.
 * Synchronises on the recorded events. */
IMGCORR_API int imgcorr_profile_read(imgcorr_ctx* ctx, double out[4]);

/* Dark current (calcDarkCurrent, camera/CameraCalibration.py:504-518).
 *   ascent == NULL : bg = dark                                   (entry built by addDarkCurrent(arr), :516)
 *   ascent != NULL : bg = dark + ascent * exposure_time, clipped to 2**depth_bits - 1, evaluated in
 *                    float64 per pixel                           (legacy tuple entry, :507-513)
 * Maps are float32 [H][W]; `on_device` != 0 means the pointers are device pointers (copied D2D),
 * otherwise host pointers.  dark == NULL removes the calibration. Synchronous. */
IMGCORR_API int imgcorr_set_dark(imgcorr_ctx* ctx, const float* dark, const float* ascent, double exposure_time,
                     int depth_bits, int on_device);
/* One exposure time per frame for the linear dark model of imgcorr_set_dark: frame i of a call (i counts from the call's
 * first frame: raw_dev[i], raw_host[i], frame i of a framed file image) evaluates bg = dark + ascent * t[i], clipped to
 * 2**depth_bits - 1, bit for bit as the same call with exposure_time = t[i].  Read by imgcorr_pointwise_median,
 * imgcorr_correct_batch and imgcorr_correct_host; the _bg forms ignore it (their backgrounds replace the dark stage).
 *   t      host array [n] of exposure times, copied synchronously; NULL removes the table (n is ignored then)
 * IMGCORR_ERR_STATE if the context has no linear model (ascent), IMGCORR_ERR_INVALID for n <= 0 or a NaN entry.  A call
 * that evaluates the model (IMGCORR_DO_DARK, no per-frame backgrounds) over more frames than the table holds fails with
 * IMGCORR_ERR_INVALID before it enqueues anything.  imgcorr_set_dark drops the table.  Replacing or removing a table first
 * synchronises the device, since queued calls may still read it; a failed call leaves no table.  Synchronous. */
IMGCORR_API int imgcorr_set_dark_exposures(imgcorr_ctx* ctx, const double* t, int n);
/* Flat field (camera/CameraCalibration.py:520-526).  flat == NULL removes it. Synchronous. */
IMGCORR_API int imgcorr_set_flat(imgcorr_ctx* ctx, const float* flat, int on_device);
/* Lens (camera/LensDistortion.py:342-358): K = cameraMatrix (3x3 row-major), dist = [k1,k2,p1,p2,k3]
 * (camera/LensDistortion.py:370,380), P = newCameraMatrix from cv2.getOptimalNewCameraMatrix (:350-353,
 * computed by the host wrapper exactly as the reference does).  K == NULL removes the lens.
 * The same as imgcorr_set_lens_model(ctx, K, dist, 5, P). */
IMGCORR_API int imgcorr_set_lens(imgcorr_ctx* ctx, const double K[9], const double dist[5], const double P[9]);
/* Lens with any coefficient vector cv2.initUndistortRectifyMap takes: n_dist = 4, 5, 8, 12 or 14 coefficients in OpenCV's
 * order k1 k2 p1 p2 [k3 [k4 k5 k6 [s1 s2 s3 s4 [tau_x tau_y]]]] (rational model, thin prism, tilted sensor; missing
 * terms are zero).  K and P as for imgcorr_set_lens; the rectification is the identity.  K2 and imgcorr_undistort_maps
 * evaluate OpenCV's full model in float64 with correctly rounded divisions.  When every term after k3 is zero the
 * lens is the 5-term lens [k1, k2, p1, p2, k3] (k3 = 0 for n_dist = 4) and gives its results bit for bit.
 * IMGCORR_ERR_INVALID for another count, a null dist or P, or a singular P.  K == NULL removes the lens.
 * Setting the lens of the last call again (same K, coefficients, count and P) keeps K2's coordinate cache. */
IMGCORR_API int imgcorr_set_lens_model(imgcorr_ctx* ctx, const double K[9], const double* dist, int n_dist, const double P[9]);

/* ---- K1: fused dark / flat / nan_to_num / NxN median-threshold ---------------------------------
 * Replaces _correctDarkCurrent + _correctVignetting + _correctArtefacts
 * (camera/CameraCalibration.py:476-526, 556-563) and medianThreshold (filters/medianThreshold.py:7-30).
 *   raw_dev   [n][H][W] of raw_dtype (U8, U16, F32, F64)
 *   out_dev   [n][H][W] of out_dtype: F32 for U8/U16/F32 input, the input dtype itself (direct
 *             medianThreshold keeps the image dtype), F64 for F32/F64 input
 *   mask_dev  [n][H][W] uint8 `indices` of medianThreshold, or NULL
 *   ksize     0 (pointwise only), 3 or 5;  threshold <= 0 is treated as ksize 0 (medianThreshold.py:16)
 *   flags     IMGCORR_DO_* ; dark / flat are applied only if set in the context as well */
IMGCORR_API int imgcorr_pointwise_median(imgcorr_ctx* ctx, const void* raw_dev, int raw_dtype, void* out_dev, int out_dtype,
                             uint8_t* mask_dev, int n_frames, double threshold, int ksize, int cond, int flags,
                             void* stream);

/* ---- K2: undistortion ---------------------------------------------------------------------------
 * Replaces LensDistortion.correct (camera/LensDistortion.py:316-330): analytic Brown-Conrady map
 * (cv2.initUndistortRectifyMap semantics, float64 -> float32) + cv2.remap(INTER_LINEAR,
 * BORDER_CONSTANT, border_value) with OpenCV's 5-bit fixed-point coordinates and weight table.
 *   src_dev [n][H][W], dst_dev [n][oh][ow]; (x0,y0,ow,oh) = output window in full-frame coordinates:
 *   (0,0,W,H) for keepSize=True, the roi for keepSize=False (:327-329).
 *   dtype pairs: F32->F32, F32->F64 (widening for the float64 API), F64->F64, U16->U16, U8->U8. */
IMGCORR_API int imgcorr_undistort(imgcorr_ctx* ctx, const void* src_dev, int src_dtype, void* dst_dev, int dst_dtype,
                      int n_frames, double border_value, int x0, int y0, int ow, int oh, void* stream);
/* cv2.remap with caller-supplied float32 maps [H][W] (LensDistortion.distortImage, :332-340). */
IMGCORR_API int imgcorr_remap(imgcorr_ctx* ctx, const void* src_dev, int src_dtype, void* dst_dev, int dst_dtype, int n_frames,
                  const float* mapx_dev, const float* mapy_dev, double border_value, void* stream);
/* getUndistortRectifyMap (camera/LensDistortion.py:342-358): writes mapx, mapy float32 [H][W]. */
IMGCORR_API int imgcorr_undistort_maps(imgcorr_ctx* ctx, float* mapx_dev, float* mapy_dev, void* stream);

/* ---- the chain: K1 -> K2 per frame, device resident --------------------------------------------
 * CameraCalibration.correct() for n independent frames (camera/CameraCalibration.py:351-459, single
 * image branch; a stack of frames is a batch here, not the STE average of :385-406).
 *   threshold > 0 : median-threshold with ksize (3 in correct(), :556-563) after nan_to_num
 *   use_lens      : apply K2 if a lens is set (missing lens -> frames pass through, :570-575)
 *   out_dtype     : F32 or F64 (float64 is what the reference returns, :459), or U16 / U8: the F32 result v of every pixel
 *                   stored as an integer through the context's output scale (imgcorr_set_output_scale), fused into the
 *                   chain's last kernel (no extra pass):  t = ((double)v - offset) * gain (two roundings, no FMA);
 *                   0 if t is NaN or t <= 0, 65535 / 255 if t >= that, else t rounded half to even.  The default scale
 *                   (0, 1) is OpenCV's saturate_cast of the F32 result.
 *   flags         : IMGCORR_DO_* ; with IMGCORR_DO_PERSPECTIVE the frame described above (the K2 window [oh][ow], or the
 *                   K1 output [H][W] without a lens) is warped by the context's perspective stage and out_dev is
 *                   [n][dst_h][dst_w] (see imgcorr_set_perspective); IMGCORR_ERR_STATE if the context has none
 * Asynchronous on `stream`.  The context's chain scratch (the K1 output and, with the perspective stage, the warp source)
 * is shared by every chain call: a call on another stream than the previous chain call (imgcorr_correct_host included)
 * first waits for that call's work on the scratch, so calls of one context on several streams are correct and run one
 * after the other on the device. */
IMGCORR_API int imgcorr_correct_batch(imgcorr_ctx* ctx, const void* raw_dev, int raw_dtype, void* out_dev, int out_dtype,
                          int n_frames, double threshold, int ksize, int flags, int use_lens, double border_value,
                          int x0, int y0, int ow, int oh, void* stream);

/* Same chain with HOST buffers: frames are staged through a ring of pinned buffers, H2D copy,
 * kernels and D2H copy of consecutive frames (small frames: chunks of up to 16 frames) overlap on three streams.  Synchronous: returns
 * when out_host is complete.  Fastest when raw_host / out_host come from imgcorr_host_alloc
 * (or are otherwise page-locked).  Its kernels wait for an earlier imgcorr_correct_batch of the same context that is
 * still queued on another stream (they share the K1 scratch), so the call also waits for that batch to finish. */
IMGCORR_API int imgcorr_correct_host(imgcorr_ctx* ctx, const void* raw_host, int raw_dtype, void* out_host, int out_dtype,
                         int n_frames, double threshold, int ksize, int flags, int use_lens, double border_value,
                         int x0, int y0, int ow, int oh);

/* The chain with one background image per frame: correct(image, bgImages=bg) of the reference
 * (camera/CameraCalibration.py:484-502) for n (image, background) pairs.  Frame i of the call subtracts background i in
 * float64 (image -= bg) in place of the context's dark map, then the flat division rounds once to float32 and the rest of
 * the chain is unchanged; for U8 / U16 / F32 backgrounds the result equals imgcorr_correct_batch with the dark map set to
 * float32(bg[i]).
 *   bg_dev / bg_host  dense [n][H][W] of bg_dtype, native byte order; i counts from the call's first frame.  The ingest
 *                     options (IMGCORR_OPT_RAW_BIG_ENDIAN, IMGCORR_OPT_RAW_FRAME_GAP) apply to the raw frames only.
 *   bg_dtype          raw_dtype or F32; anything else, or flags without IMGCORR_DO_DARK, fails with IMGCORR_ERR_INVALID
 *                     before anything is enqueued
 * The context's dark map and linear dark model are neither read nor modified: a later call without backgrounds uses them
 * as before.  bg == NULL is imgcorr_correct_batch / imgcorr_correct_host.  Float32 backgrounds may hold NaN / inf; they
 * take the checked arithmetic of float32 frames.  The host call stages the backgrounds through its ring next to the raw
 * frames (a device buffer per slot, pinned staging for pageable input) and counts both against its chunk size.
 * Everything else (stream order, scratch, perspective stage, output scale) is as the calls without backgrounds. */
IMGCORR_API int imgcorr_correct_batch_bg(imgcorr_ctx* ctx, const void* raw_dev, int raw_dtype, const void* bg_dev, int bg_dtype,
                             void* out_dev, int out_dtype, int n_frames, double threshold, int ksize, int flags,
                             int use_lens, double border_value, int x0, int y0, int ow, int oh, void* stream);
IMGCORR_API int imgcorr_correct_host_bg(imgcorr_ctx* ctx, const void* raw_host, int raw_dtype, const void* bg_host, int bg_dtype,
                            void* out_host, int out_dtype, int n_frames, double threshold, int ksize, int flags,
                            int use_lens, double border_value, int x0, int y0, int ow, int oh);

/* Scale of the chain's integer output (out_dtype U16 / U8 of imgcorr_correct_batch / imgcorr_correct_host):
 * stored = quantise((F32 result - offset) * gain), see imgcorr_correct_batch.  Context state, read when a chain call is
 * enqueued; defaults offset 0, gain 1.  IMGCORR_ERR_INVALID for a non-finite offset or a gain that is not finite and > 0.
 * Other entry points (imgcorr_pointwise_median's integer output included) do not read it. */
IMGCORR_API int imgcorr_set_output_scale(imgcorr_ctx* ctx, double offset, double gain);

/* The chain's perspective stage: PerspectiveCorrection.correct (camera/PerspectiveCorrection.py:380-406) on every frame of
 * an imgcorr_correct_batch / imgcorr_correct_host call that sets IMGCORR_DO_PERSPECTIVE, without the intermediate frames
 * leaving the device.  Per frame group: K1 -> [K2] -> [tilt division] -> K3 (Lanczos4, forward map, BORDER_CONSTANT).
 *   M             3x3 row-major homography from the chain's frame (the K2 window, or the full frame without a lens) to
 *                 the destination; NULL removes the stage (and the tilt factor)
 *   dst_h, dst_w  destination frame, 1..32767 per side; border_value fills pixels that map outside the source
 *   tilt_factor   NULL: no intensity correction.  Otherwise float64 [tilt_h][tilt_w] (device pointer if on_device != 0,
 *                 host pointer otherwise), copied synchronously into the context; the chain frame is divided by it in
 *                 float64 before the warp (np.asfarray(img) / tf, :394-400)
 * Precision: with out_dtype F32 the float32 chain frame is warped in float32 (cv2.warpPerspective of that frame), with U16 / U8
 * that same float32 warp is quantised on store (imgcorr_set_output_scale); with F64
 * the float64 chain frame is warped in float64 (pc.correct(cal.correct(frame)) of the Python mirror).  A tilt factor needs
 * out_dtype F64 and the shape of the chain frame: either mismatch makes the chain call fail with IMGCORR_ERR_INVALID.
 * The stage adds one part to the chain scratch: a group of chain frames in out_dtype (float32 for U16 / U8).  Synchronous. */
IMGCORR_API int imgcorr_set_perspective(imgcorr_ctx* ctx, const double M[9], int dst_h, int dst_w, double border_value,
                            const double* tilt_factor, int tilt_h, int tilt_w, int on_device);
/* The same stage with one homography per frame: frame i of a chain call (raw_dev[i], raw_host[i]; i counts from the call's
 * first frame) is warped with matrix i.  Everything else is as imgcorr_set_perspective without a tilt factor: Lanczos4,
 * forward map, BORDER_CONSTANT, one destination size and border value, the same dtype rules.
 *   M             host array [n_matrices][9], row-major, each matrix mapping the chain frame to the destination; inverted
 *                 here with cv::invert's cofactor formula (a singular matrix becomes zeros) and uploaded synchronously.
 *                 NULL removes the stage.
 * A chain call with IMGCORR_DO_PERSPECTIVE and more than n_matrices frames fails with IMGCORR_ERR_INVALID before it
 * enqueues anything.  The two setters replace each other: imgcorr_set_perspective drops the table, this call drops a
 * single matrix and its tilt factor.  Replacing or removing a table first synchronises the device, since queued chain
 * calls may still read it.  A failed call leaves no stage.  Synchronous. */
IMGCORR_API int imgcorr_set_perspective_frames(imgcorr_ctx* ctx, const double* M, int n_matrices, int dst_h, int dst_w,
                                   double border_value);

/* ---- K3: perspective warp (SURVEY §8 row f3) -----------------------------------------------------
 * Replaces cv2.warpPerspective in PerspectiveCorrection.correct (flags=INTER_LANCZOS4,
 * camera/PerspectiveCorrection.py:401-405) and PerspectiveCorrection.uncorrect (INTER_CUBIC |
 * WARP_INVERSE_MAP, :374-378), bit-exact with OpenCV's arithmetic (BORDER_CONSTANT).
 *   src_dev [n][src_h][src_w], dst_dev [n][dst_h][dst_w], both of `dtype` (U8 with OpenCV's int16 fixed-point
 *   weights, U16, F32 or F64); frame sizes are free (<= 32767 per side), the context only supplies the device.
 *   M             3x3 row-major homography src -> dst (the matrix cv2.warpPerspective takes); inverted here
 *                 with cv::invert's cofactor formula unless inverse_map != 0
 *   interpolation IMGCORR_INTER_LANCZOS4 or IMGCORR_INTER_CUBIC (values of the cv2 flags) */
enum { IMGCORR_INTER_CUBIC = 2, IMGCORR_INTER_LANCZOS4 = 4 };
IMGCORR_API int imgcorr_warp_perspective(imgcorr_ctx* ctx, const void* src_dev, int dtype, int src_h, int src_w, void* dst_dev,
                             int dst_h, int dst_w, int n_frames, const double M[9], int interpolation, int inverse_map,
                             double border_value, void* stream);
/* dst[f][i] = (double)src[f][i] / divisor[i]: the tilt-factor division in front of the warp
 * (camera/PerspectiveCorrection.py:394-400, np.asfarray(img) / tf).  src of any dtype, divisor and dst float64;
 * dst_dev may equal src_dev for a float64 src (in place), other overlaps are not allowed. */
IMGCORR_API int imgcorr_divide_f64(imgcorr_ctx* ctx, const void* src_dev, int src_dtype, const double* divisor_dev, double* dst_dev,
                       size_t pixels_per_frame, int n_frames, void* stream);

/* ---- K4: single-time-effect-free average of several exposures (SURVEY §8 rows a11 / f1) --------------
 * Replaces SingleTimeEffectDetection(images, nStd, noise_level_function).noSTE in the multi-image branch of
 * CameraCalibration.correct() (camera/CameraCalibration.py:385-406; features/SingleTimeEffectDetection.py:23-75)
 * with noise_level_function = NoiseLevelFunction.boundedFunction(x, minY, ax, ay) (camera/NoiseLevelFunction.py:94-107;
 * nlf[3] = {minY, ax, ay}, the 'noise' calibration entry) and removeSinglePixels (filters/removeSinglePixels.py:4-33).
 *   frames_dev [n][H][W] of `dtype` (any), n >= 2;  avg_dev [H][W] float64 = noSTE;
 *   mask_dev   [H][W] uint8 accumulated STE mask (save_ste_indices=True) or NULL.
 * float64 arithmetic as in the reference; the running mean avg += (x - avg) / n restates fancytools'
 * MaskedMovingAverage (absent from the reference tree: that ingredient's parity is unpinned, see oracle/ste.py).
 * Asynchronous on `stream`.  The context's K4 scratch is shared by every K4 call (imgcorr_ste_average_thr included): a call
 * on another stream than the previous K4 call first waits for that call's work on the scratch, so calls of one context on
 * several streams are correct and run one after the other on the device. */
IMGCORR_API int imgcorr_ste_average(imgcorr_ctx* ctx, const void* frames_dev, int dtype, int n_frames, double* avg_dev,
                        uint8_t* mask_dev, const double nlf[3], double n_std, void* stream);
/* The same with a caller-supplied threshold map  threshold_dev[H][W] = noise_level_function(min(images[0], images[1])) * nStd
 * (float64) for noise level functions that are not boundedFunction: the one correct() ESTIMATES when no 'noise' calibration
 * exists may be a polynomial (oneImageNLF -> smooth, camera/NoiseLevelFunction.py:132-159), and a user may have assigned any
 * Python callable to CameraCalibration.noise_level_function.
 * Asynchronous on `stream`.  The context's K4 scratch is shared by every K4 call (imgcorr_ste_average included): a call on
 * another stream than the previous K4 call first waits for that call's work on the scratch, so calls of one context on
 * several streams are correct and run one after the other on the device. */
IMGCORR_API int imgcorr_ste_average_thr(imgcorr_ctx* ctx, const void* frames_dev, int dtype, int n_frames, double* avg_dev,
                            uint8_t* mask_dev, const double* threshold_dev, void* stream);

/* ---- K5: calibration-map producers (SURVEY §8 row f4) ---------------------------------------------------
 * Float64 streaming reductions over small stacks of frames; frame sizes are free (the context only supplies the device).
 *
 * imgcorr_stack_mean: imgAverage (transform/imgAverage.py:7-22) of n frames of `elems` samples each (H*W, or H*W*3 for colour
 *   frames), then optionally  img -= bg  (minus_dev: float64 [elems], or minus_scalar when use_scalar != 0) and, with gray3 != 0,
 *   toGray (transformations.py:126-135) over the 3 interleaved channels -> out_dev float64 [elems] or [elems / 3].  Together
 *   with imgcorr_subsample_f64 (img[::10, ::10]), the 3x3 median (imgcorr_pointwise_median) and imgcorr_scale_f64 (img /= mx)
 *   this is flatFieldFromCloseDistance (camera/flatField/flatFieldFromCloseDistance.py:16-38).
 * imgcorr_linear_fit: getLinearityFunction (camera/DarkCurrentMap.py:61-80): per-pixel line  image(t) = offset + ascent t
 *   through n frames taken at exposure times x[n], samples above max_intensity masked, NaN ascents set to 0 and ascents below
 *   min_ascent folded into the offset.  rmse_dev may be NULL.  The regression restates fancytools'
 *   linRegressUsingMasked2dArrays (absent from the reference tree: parity unpinned for that ingredient, see oracle/producers.py). */
IMGCORR_API int imgcorr_stack_mean(imgcorr_ctx* ctx, const void* frames_dev, int dtype, int n_frames, size_t elems, const double* minus_dev,
                       double minus_scalar, int use_scalar, int gray3, double* out_dev, void* stream);
IMGCORR_API int imgcorr_scale_f64(imgcorr_ctx* ctx, double* data_dev, size_t elems, double divisor, void* stream);
IMGCORR_API int imgcorr_subsample_f64(imgcorr_ctx* ctx, const double* src_dev, int height, int width, int step_y, int step_x, double* dst_dev,
                          void* stream);
IMGCORR_API int imgcorr_linear_fit(imgcorr_ctx* ctx, const void* frames_dev, int dtype, int n_frames, size_t pixels, const double* x_host,
                       double max_intensity, double min_ascent, double* offset_dev, double* ascent_dev, double* rmse_dev, void* stream);

/* ---- self-test ---------------------------------------------------------------------------------------
 * K1 and K4 divide in float64 with a shortened Newton sequence (MUFU.RCP64H seed, one refinement, residual correction:
 * csrc/imgcorr_core.cuh rcp_f32range / ddiv_rcp) that is exact only because the divisors are float32-derived or small
 * integers.  This runs the sequence on the device for every float32 significand pattern of the divisor (both signs,
 * exponents cycling over the float32 range), `numerators_per_divisor` numerators each, against IEEE division:
 *   out[0] = quotients that differ from IEEE a / b (must be 0), out[1] = largest |1 - b * seed| seen (seed quality).
 * Synchronous. */
IMGCORR_API int imgcorr_selftest_division(imgcorr_ctx* ctx, int numerators_per_divisor, unsigned long long seed, double out[2]);

/* 64-bit fingerprint of a host buffer (every byte contributes; several host threads).  The Python mirror keys its
 * "is this calibration map already on the device?" cache on it: the reference re-reads dark / flat arrays on every
 * correct() call (camera/CameraCalibration.py:500-502, 521-526), so an array edited in place must be uploaded again. */
IMGCORR_API int imgcorr_host_fingerprint(const void* host_ptr, size_t bytes, unsigned long long* out);

/* page-locked host memory for the *_host entry points */
IMGCORR_API int imgcorr_host_alloc(size_t bytes, void** out_ptr);
IMGCORR_API int imgcorr_host_free(void* ptr);

#ifdef __cplusplus
}
#endif
#endif /* IMGCORR_H */
