"""Engine: one libimgcorr context (device, frame shape) with torch tensors as the device buffers.

torch is plumbing only: it owns device memory and streams; every kernel that runs is one of the
hand-written sm_100a kernels in csrc/, reached through the C ABI of include/imgcorr.h.
"""
import ctypes
import os

import numpy as np

from . import _lib
from ._lib import DO_DARK, DO_FLAT, DO_NAN_TO_NUM, DO_PERSPECTIVE  # noqa: F401  (re-exported)

_TORCH = None


def torch():
    global _TORCH
    if _TORCH is None:
        import torch as _t
        _TORCH = _t
    return _TORCH


def _dtype_code(t):
    tt = torch()
    table = {tt.uint8: _lib.U8, tt.uint16: _lib.U16, tt.float32: _lib.F32, tt.float64: _lib.F64}
    if t not in table:
        raise TypeError('unsupported frame dtype %s (uint8, uint16, float32, float64)' % (t,))
    return table[t]


def _torch_dtype(code):
    tt = torch()
    return {_lib.U8: tt.uint8, _lib.U16: tt.uint16, _lib.F32: tt.float32, _lib.F64: tt.float64}[code]


NP_CODES = {np.dtype(np.uint8): _lib.U8, np.dtype(np.uint16): _lib.U16, np.dtype(np.float32): _lib.F32,
            np.dtype(np.float64): _lib.F64}
# coefficient counts of the lens models cv2.initUndistortRectifyMap takes (Engine.set_lens)
LENS_MODEL_SIZES = (4, 5, 8, 12, 14)


def require_cuda():
    tt = torch()
    if not tt.cuda.is_available():
        raise RuntimeError('imgprocessor_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback')
    return tt


class Engine(object):
    def __init__(self, height, width, device=None):
        tt = require_cuda()
        self.lib = _lib.lib()
        if device is None:
            device = tt.cuda.current_device()
        self.device_index = tt.device('cuda', device).index if not isinstance(device, int) else device
        self.device = tt.device('cuda', self.device_index)
        self.H, self.W = int(height), int(width)
        h = ctypes.c_void_p()
        _lib.check(self.lib.imgcorr_ctx_create(self.device_index, self.H, self.W, ctypes.byref(h)))
        self._h = h
        self.has_dark = self.has_flat = self.has_lens = self.has_exposures = False
        self.perspective_dsize = None          # (width, height) of the chain's perspective stage, if one is set
        self._tokens = {}

    # -- lifetime ---------------------------------------------------------------------------
    def close(self):
        if getattr(self, '_h', None):
            self.lib.imgcorr_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_option(self, key, value):
        _lib.check(self.lib.imgcorr_set_option(self._h, key, value))

    @property
    def launch_count(self):
        return int(self.lib.imgcorr_launch_count(self._h))

    def profile_read(self):
        """(k1_ms, k1_launches, k2_ms, k2_launches) of the event-bracketed launches since the last call"""
        buf = (ctypes.c_double * 4)()
        _lib.check(self.lib.imgcorr_profile_read(self._h, buf))
        return tuple(buf)

    def selftest_division(self, numerators_per_divisor=16, seed=1):
        """(mismatches, worst seed error) of the shortened float64 division sequence against IEEE division, run on the
        device for every float32 significand pattern of the divisor (imgcorr_selftest_division)"""
        buf = (ctypes.c_double * 2)()
        _lib.check(self.lib.imgcorr_selftest_division(self._h, int(numerators_per_divisor), int(seed), buf))
        return int(buf[0]), float(buf[1])

    def _check_out(self, out, shape, what='out'):
        """a caller-supplied output tensor goes to the kernels by pointer: refuse anything that is not exactly what they write"""
        tt = torch()
        if not isinstance(out, tt.Tensor) or not out.is_cuda or out.device != self.device:
            raise ValueError('%s must be a CUDA tensor on %s' % (what, self.device))
        if tuple(out.shape) != tuple(shape):
            raise ValueError('%s has shape %s, expected %s' % (what, tuple(out.shape), tuple(shape)))
        if not out.is_contiguous():
            raise ValueError('%s must be contiguous' % what)
        return out

    def _stream(self):
        return ctypes.c_void_p(torch().cuda.current_stream(self.device).cuda_stream)

    # -- calibration ------------------------------------------------------------------------
    def _map_arg(self, arr):
        """float32 [H][W] map as (pointer, on_device, keepalive)."""
        if arr is None:
            return None, 0, None
        tt = torch()
        if isinstance(arr, tt.Tensor):
            t = arr.to(device=self.device, dtype=tt.float32).contiguous()
            if tuple(t.shape) != (self.H, self.W):
                raise ValueError('map shape %s != frame shape %s' % (tuple(t.shape), (self.H, self.W)))
            return ctypes.c_void_p(t.data_ptr()), 1, t
        a = np.ascontiguousarray(arr, dtype=np.float32)
        if a.shape != (self.H, self.W):
            a = np.ascontiguousarray(np.broadcast_to(a, (self.H, self.W)))
        return a.ctypes.data_as(ctypes.c_void_p), 0, a

    def set_dark(self, dark, ascent=None, exposure_time=0.0, depth_bits=16, token=None):
        if token is not None and self._tokens.get('dark') == token:
            return
        p, dev, keep = self._map_arg(dark)
        p2, dev2, keep2 = self._map_arg(ascent)
        if keep is not None and keep2 is not None and dev != dev2:
            raise ValueError('dark and ascent must both be host arrays or both device tensors')
        self.has_exposures = False                       # imgcorr_set_dark drops the per-frame exposure times
        _lib.check(self.lib.imgcorr_set_dark(self._h, p, p2, float(exposure_time), int(depth_bits), dev))
        self.has_dark = dark is not None
        self._tokens['dark'] = token

    def set_dark_exposures(self, times):
        """One exposure time per frame for the linear dark model of set_dark(dark, ascent, ...)
        (imgcorr_set_dark_exposures): frame i of every later call evaluates dark + ascent * times[i], clipped, exactly as
        the same call with exposure_time=times[i]; a call with more frames than times is refused.  Calls with per-frame
        backgrounds ignore the table.  None removes it; set_dark removes it too."""
        self.has_exposures = False                       # a failed call leaves no table behind
        if times is None:
            _lib.check(self.lib.imgcorr_set_dark_exposures(self._h, None, 0))
            return
        t = np.ascontiguousarray(np.asarray(times, dtype=np.float64))
        if t.ndim != 1:
            raise ValueError('exposure times must be 1-D, got shape %s' % (t.shape,))
        _lib.check(self.lib.imgcorr_set_dark_exposures(self._h, t.ctypes.data_as(ctypes.c_void_p), int(t.size)))
        self.has_exposures = True

    def set_flat(self, flat, token=None):
        if token is not None and self._tokens.get('flat') == token:
            return
        p, dev, keep = self._map_arg(flat)
        _lib.check(self.lib.imgcorr_set_flat(self._h, p, dev))
        self.has_flat = flat is not None
        self._tokens['flat'] = token

    def set_lens(self, K, dist, P):
        if K is None:
            _lib.check(self.lib.imgcorr_set_lens(self._h, None, None, None))
            self.has_lens = False
            return
        K = np.ascontiguousarray(np.asarray(K, np.float64).reshape(3, 3))
        d = np.ascontiguousarray(np.asarray(dist, np.float64).ravel())     # (1, n), (n,) or (n, 1)
        if d.size not in LENS_MODEL_SIZES:
            raise ValueError('distortion coefficients: 4, 5, 8, 12 or 14 terms (OpenCV order k1 k2 p1 p2 k3 k4 k5 k6 '
                             's1 s2 s3 s4 tau_x tau_y), got %d' % d.size)
        P = np.ascontiguousarray(np.asarray(P, np.float64)[:3, :3])
        vp = lambda a: a.ctypes.data_as(ctypes.c_void_p)
        _lib.check(self.lib.imgcorr_set_lens_model(self._h, vp(K), vp(d), d.size, vp(P)))
        self.has_lens = True

    def set_perspective(self, M, dsize, border_value=0.0, tilt_factor=None, token=None):
        """the chain's perspective stage (imgcorr_set_perspective): chain calls with DO_PERSPECTIVE in their flags warp
        every frame they would return with cv2.warpPerspective(frame, M, dsize=(width, height), INTER_LANCZOS4,
        BORDER_CONSTANT, border_value), after dividing it by ``tilt_factor`` (float64, the chain frame's shape; needs
        float64 output) if one is given.  M None removes the stage.  ``token``: an identity of the tilt factor; a call
        with the same arguments and token as the last one uploads nothing.

        M of shape (n, 3, 3) is one matrix per frame (imgcorr_set_perspective_frames): frame i of every chain call is
        warped with M[i], and a call with more than n frames is refused.  Such a table takes no tilt factor."""
        if M is None:
            _lib.check(self.lib.imgcorr_set_perspective(self._h, None, 0, 0, 0.0, None, 0, 0, 0))
            self.perspective_dsize = None
            self._tokens['perspective'] = None
            return
        dw, dh = int(dsize[0]), int(dsize[1])
        Ma = np.asarray(M, np.float64)
        if Ma.ndim == 3:
            if Ma.shape[0] < 1 or Ma.shape[1:] != (3, 3):
                raise ValueError('a per-frame table has shape (n, 3, 3), got %s' % (Ma.shape,))
            if tilt_factor is not None:
                raise ValueError('a tilt factor needs a single matrix: the per-frame table has no tilt factor')
            Mt = np.ascontiguousarray(Ma)
            key = ('frames', Mt.tobytes(), dw, dh, float(border_value))
            if self._tokens.get('perspective') == key:
                return
            self._tokens['perspective'] = self.perspective_dsize = None      # a failed call leaves no stage behind
            _lib.check(self.lib.imgcorr_set_perspective_frames(self._h, Mt.ctypes.data_as(ctypes.c_void_p), Mt.shape[0], dh,
                                                               dw, float(border_value)))
            self.perspective_dsize = (dw, dh)
            self._tokens['perspective'] = key
            return
        Mh = np.ascontiguousarray(Ma.reshape(3, 3))
        key = (Mh.tobytes(), dw, dh, float(border_value), tilt_factor is None, token)
        if (tilt_factor is None or token is not None) and self._tokens.get('perspective') == key:
            return
        tp, th, tw, dev, keep = None, 0, 0, 0, None
        if tilt_factor is not None:
            tt = torch()
            if isinstance(tilt_factor, tt.Tensor):
                keep = tilt_factor.to(device=self.device, dtype=tt.float64).contiguous()
                tp, dev = ctypes.c_void_p(keep.data_ptr()), 1
            else:
                keep = np.ascontiguousarray(tilt_factor, dtype=np.float64)
                tp = keep.ctypes.data_as(ctypes.c_void_p)
            if keep.ndim != 2:
                raise ValueError('tilt_factor must be 2-D, got shape %s' % (tuple(keep.shape),))
            th, tw = (int(v) for v in keep.shape)
        self._tokens['perspective'] = self.perspective_dsize = None          # a failed call leaves no stage behind
        _lib.check(self.lib.imgcorr_set_perspective(self._h, Mh.ctypes.data_as(ctypes.c_void_p), dh, dw, float(border_value),
                                                    tp, th, tw, dev))
        self.perspective_dsize = (dw, dh)
        self._tokens['perspective'] = key

    def chain_shape(self, flags, use_lens=True, window=None):
        """(lens, (x0, y0, ow, oh), (h, w)) of a chain call: whether K2 runs, its output window and the shape of every
        frame the call returns (the perspective stage's destination with DO_PERSPECTIVE and a stage set; without a stage
        the library refuses the call)"""
        lens = bool(use_lens and self.has_lens)
        x0, y0, ow, oh = self._window(window if lens else None)
        if int(flags) & DO_PERSPECTIVE and self.perspective_dsize is not None:
            return lens, (x0, y0, ow, oh), self.perspective_dsize[::-1]
        return lens, (x0, y0, ow, oh), (oh, ow)

    # -- helpers ----------------------------------------------------------------------------
    def _frames(self, t):
        tt = torch()
        if not isinstance(t, tt.Tensor):
            raise TypeError('expected a torch tensor on %s' % self.device)
        if t.device != self.device:
            raise ValueError('tensor on %s, engine on %s' % (t.device, self.device))
        if t.dim() == 2:
            t = t.unsqueeze(0)
        if t.dim() != 3 or tuple(t.shape[1:]) != (self.H, self.W):
            raise ValueError('frames of shape %s do not match the engine (%d, %d)' % (tuple(t.shape), self.H, self.W))
        return t.contiguous()

    def _window(self, window):
        if window is None:
            return 0, 0, self.W, self.H
        x, y, w, h = (int(v) for v in window)
        return x, y, w, h

    class _Ingest(object):
        """context manager: raw frames of the enclosed calls are big-endian uint16 and / or separated by `gap` bytes"""

        def __init__(self, eng, big_endian, gap):
            self.eng, self.be, self.gap = eng, bool(big_endian), int(gap)

        def __enter__(self):
            if self.be:
                self.eng.set_option(_lib.OPT_RAW_BIG_ENDIAN, 1)
            if self.gap:
                self.eng.set_option(_lib.OPT_RAW_FRAME_GAP, self.gap)

        def __exit__(self, *a):
            if self.be:
                self.eng.set_option(_lib.OPT_RAW_BIG_ENDIAN, 0)
            if self.gap:
                self.eng.set_option(_lib.OPT_RAW_FRAME_GAP, 0)

    def ingest(self, big_endian=False, gap=0):
        return Engine._Ingest(self, big_endian, gap)

    def _set_out_scale(self, code, out_scale):
        """Integer output (U16 / U8): set the context's output scale (offset, gain) for the call that follows; None is the
        default (0, 1), OpenCV's saturate_cast of the float32 result.  Float output takes no scale."""
        if code in (_lib.U8, _lib.U16):
            offset, gain = (0.0, 1.0) if out_scale is None else out_scale
            _lib.check(self.lib.imgcorr_set_output_scale(self._h, float(offset), float(gain)))
        elif out_scale is not None:
            raise ValueError('out_scale applies to uint8 / uint16 output only')

    def correct_file_bytes(self, buf, offset, n_frames, gap=0, big_endian=False, dtype=None, **kw):
        """The chain on frames as they sit in a file image: ``buf`` is a uint8 CUDA tensor holding the file bytes,
        the first frame's pixels start at byte ``offset`` and consecutive frames are ``gap`` bytes apart
        (reader/elbin.py: 20-byte per-frame headers; reader/RAW.py: dense, big-endian by default).  No host-side
        byte swap or de-interleave: K1 does both in its load.  kw as correct_batch (out_scale included)."""
        tt = torch()
        dtype = dtype or tt.uint16
        esz = {tt.uint8: 1, tt.uint16: 2, tt.float32: 4}[dtype]
        need = offset + n_frames * self.H * self.W * esz + (n_frames - 1) * gap
        if buf.dtype != tt.uint8 or buf.device != self.device or buf.numel() < need:
            raise ValueError('buf must be a uint8 tensor on %s with at least %d bytes' % (self.device, need))
        if offset % esz or gap % esz:
            raise ValueError('offset and gap must be multiples of the sample size')
        flags = int(kw.get('flags', DO_DARK | DO_FLAT | DO_NAN_TO_NUM))
        lens, (x0, y0, ow, oh), (h, w) = self.chain_shape(flags, kw.get('use_lens', True), kw.get('window'))
        out = kw.get('out')
        if out is None:
            out = tt.empty((n_frames, h, w), dtype=kw.get('out_dtype') or tt.float32, device=self.device)
        else:
            self._check_out(out, (n_frames, h, w))
        self._set_out_scale(_dtype_code(out.dtype), kw.get('out_scale'))
        with self.ingest(big_endian, gap):
            _lib.check(self.lib.imgcorr_correct_batch(
                self._h, ctypes.c_void_p(buf.data_ptr() + offset), _dtype_code(dtype), ctypes.c_void_p(out.data_ptr()),
                _dtype_code(out.dtype), n_frames, float(kw.get('threshold', 0.1)), int(kw.get('ksize', 3)),
                flags, int(lens), float(kw.get('border_value', 0.0)), x0, y0, ow, oh, self._stream()))
        return out

    # -- kernels ----------------------------------------------------------------------------
    def pointwise_median(self, raw, threshold=0.1, ksize=3, cond='>', flags=DO_DARK | DO_FLAT | DO_NAN_TO_NUM,
                         out_dtype=None, want_mask=False, out=None):
        """K1.  raw: [n,H,W] or [H,W] device tensor.  Returns (out, mask-or-None)."""
        tt = torch()
        squeeze = raw.dim() == 2
        raw = self._frames(raw)
        n = raw.shape[0]
        rc = _dtype_code(raw.dtype)
        if out_dtype is None:
            out_dtype = tt.float64 if raw.dtype == tt.float64 else tt.float32
        if out is None:
            out = tt.empty((n, self.H, self.W), dtype=out_dtype, device=self.device)
        else:
            self._check_out(out, (n, self.H, self.W))
        mask = tt.zeros((n, self.H, self.W), dtype=tt.uint8, device=self.device) if want_mask else None
        _lib.check(self.lib.imgcorr_pointwise_median(
            self._h, ctypes.c_void_p(raw.data_ptr()), rc, ctypes.c_void_p(out.data_ptr()), _dtype_code(out.dtype),
            ctypes.c_void_p(mask.data_ptr()) if mask is not None else None, n, float(threshold), int(ksize),
            _lib.COND_GT if cond == '>' else _lib.COND_LT, int(flags), self._stream()))
        if squeeze:
            out = out[0]
            mask = mask[0] if mask is not None else None
        return out, mask

    def undistort(self, src, out_dtype=None, border_value=0.0, window=None, out=None):
        """K2 with the analytic map of the lens set by set_lens()."""
        tt = torch()
        squeeze = src.dim() == 2
        src = self._frames(src)
        n = src.shape[0]
        x0, y0, ow, oh = self._window(window)
        if out_dtype is None:
            out_dtype = src.dtype
        if out is None:
            out = tt.empty((n, oh, ow), dtype=out_dtype, device=self.device)
        else:
            self._check_out(out, (n, oh, ow))
        _lib.check(self.lib.imgcorr_undistort(
            self._h, ctypes.c_void_p(src.data_ptr()), _dtype_code(src.dtype), ctypes.c_void_p(out.data_ptr()),
            _dtype_code(out.dtype), n, float(border_value), x0, y0, ow, oh, self._stream()))
        return out[0] if squeeze else out

    def remap(self, src, mapx, mapy, border_value=0.0, out_dtype=None):
        """K2 with caller-supplied float32 maps [H,W] (device tensors)."""
        tt = torch()
        squeeze = src.dim() == 2
        src = self._frames(src)
        n = src.shape[0]
        mapx = mapx.to(device=self.device, dtype=tt.float32).contiguous()
        mapy = mapy.to(device=self.device, dtype=tt.float32).contiguous()
        if tuple(mapx.shape) != (self.H, self.W) or tuple(mapy.shape) != (self.H, self.W):
            raise ValueError('maps must be [H,W]')
        out = tt.empty((n, self.H, self.W), dtype=out_dtype or src.dtype, device=self.device)
        _lib.check(self.lib.imgcorr_remap(
            self._h, ctypes.c_void_p(src.data_ptr()), _dtype_code(src.dtype), ctypes.c_void_p(out.data_ptr()),
            _dtype_code(out.dtype), n, ctypes.c_void_p(mapx.data_ptr()), ctypes.c_void_p(mapy.data_ptr()),
            float(border_value), self._stream()))
        return out[0] if squeeze else out

    def warp_perspective(self, src, M, dsize, interpolation='lanczos4', inverse_map=False, border_value=0.0,
                         divide_by=None):
        """K3: cv2.warpPerspective(src, M, dsize=(width, height), flags=INTER_LANCZOS4 | INTER_CUBIC
        [| WARP_INVERSE_MAP], borderValue) for device frames [n,h,w] or [h,w] of uint8 / uint16 / float32 / float64
        (camera/PerspectiveCorrection.py:374-378, 401-405).  divide_by: float64 [h,w] tilt factor applied first
        in float64 (:394-400); the result is then float64.  The frame shape is free (not the engine's)."""
        tt = torch()
        squeeze = src.dim() == 2
        src = (src[None] if squeeze else src).to(self.device).contiguous()
        n, h, w = src.shape
        dw, dh = int(dsize[0]), int(dsize[1])
        if divide_by is not None:
            div = divide_by.to(device=self.device, dtype=tt.float64).contiguous()
            if tuple(div.shape) != (h, w):
                raise ValueError('divide_by must be [h,w]')
            q = tt.empty((n, h, w), dtype=tt.float64, device=self.device)
            _lib.check(self.lib.imgcorr_divide_f64(self._h, ctypes.c_void_p(src.data_ptr()), _dtype_code(src.dtype),
                                                   ctypes.c_void_p(div.data_ptr()), ctypes.c_void_p(q.data_ptr()),
                                                   h * w, n, self._stream()))
            src = q
        Mh = np.ascontiguousarray(np.asarray(M, np.float64).reshape(3, 3))
        out = tt.empty((n, dh, dw), dtype=src.dtype, device=self.device)
        _lib.check(self.lib.imgcorr_warp_perspective(
            self._h, ctypes.c_void_p(src.data_ptr()), _dtype_code(src.dtype), h, w, ctypes.c_void_p(out.data_ptr()),
            dh, dw, n, Mh.ctypes.data_as(ctypes.c_void_p), {'lanczos4': _lib.INTER_LANCZOS4, 'cubic': _lib.INTER_CUBIC}[interpolation],
            int(bool(inverse_map)), float(border_value), self._stream()))
        return out[0] if squeeze else out

    def ste_average(self, frames, nlf=None, n_std=4.0, want_mask=False, threshold=None):
        """K4: SingleTimeEffectDetection(frames, nStd=n_std, noise_level_function=boundedFunction(., *nlf)).noSTE
        for device frames [n,H,W] (n >= 2) -> float64 [H,W] (and the accumulated STE mask if asked)
        (features/SingleTimeEffectDetection.py:23-75).  ``threshold``: a float64 [H,W] map
        noise_level_function(min(frames[0], frames[1])) * nStd for noise level functions other than boundedFunction."""
        tt = torch()
        frames = self._frames(frames)
        n = frames.shape[0]
        avg = tt.empty((self.H, self.W), dtype=tt.float64, device=self.device)
        mask = tt.empty((self.H, self.W), dtype=tt.uint8, device=self.device) if want_mask else None
        mp = ctypes.c_void_p(mask.data_ptr()) if want_mask else None
        if threshold is not None:
            thr = threshold if isinstance(threshold, tt.Tensor) else tt.from_numpy(np.ascontiguousarray(threshold, dtype=np.float64))
            thr = thr.to(device=self.device, dtype=tt.float64).contiguous()
            if tuple(thr.shape) != (self.H, self.W):
                raise ValueError('threshold map shape %s != frame shape %s' % (tuple(thr.shape), (self.H, self.W)))
            _lib.check(self.lib.imgcorr_ste_average_thr(
                self._h, ctypes.c_void_p(frames.data_ptr()), _dtype_code(frames.dtype), n, ctypes.c_void_p(avg.data_ptr()),
                mp, ctypes.c_void_p(thr.data_ptr()), self._stream()))
        else:
            if nlf is None:
                raise ValueError('ste_average needs the boundedFunction parameters (nlf) or a threshold map')
            coeff = (ctypes.c_double * 3)(*[float(v) for v in nlf])
            _lib.check(self.lib.imgcorr_ste_average(
                self._h, ctypes.c_void_p(frames.data_ptr()), _dtype_code(frames.dtype), n, ctypes.c_void_p(avg.data_ptr()),
                mp, coeff, float(n_std), self._stream()))
        return (avg, mask.bool()) if want_mask else avg

    def median3x3(self, img):
        """scipy.ndimage.median_filter(img, 3) (mode='reflect') of a host float64 / float32 image through K1: a median-threshold
        whose threshold is so small that every pixel differing from its median is replaced by it (and a pixel equal to
        its median already is the median).  Used by the noise-level-function estimation (camera/NoiseLevelFunction.py)
        and flatFieldFromCloseDistance.

        Where the median is +inf or -inf, K1's predicate |(img - median) / median| > threshold is NaN for a finite pixel,
        so K1 keeps the pixel.  Those pixels are found by a second K1 run on the 0/1 image (img == inf): its median is 1
        exactly where at least 5 of the 9 window values are inf, which is where the true median is inf.  A 0/1 image has
        no infinite median, so K1 is an exact median on it.  Images without infinities take the single K1 run.
        Images with NaN are not matched to scipy, whose result next to a NaN depends on the order of its selection."""
        a = np.ascontiguousarray(img)
        if a.dtype not in (np.float64, np.float32):
            a = a.astype(np.float64)
        out = self._median3x3_k1(a)
        for inf in (np.inf, -np.inf):
            hit = a == inf
            if hit.any():
                out[self._median3x3_k1(hit.astype(a.dtype)) == 1] = inf
        return out

    def _median3x3_k1(self, a):
        dev = torch().from_numpy(a).to(self.device)
        out, _ = self.pointwise_median(dev, 1e-300, 3, flags=0, out_dtype=dev.dtype)
        return to_numpy(out)

    # -- K5: calibration-map producers (frame sizes are free; the engine only supplies the device) -----------
    def _k5_tensor(self, t, what, f64=False):
        """the K5 kernels take free shapes, so _frames() does not apply; they still need a tensor on this engine's device,
        and the float64-only ones a float64 tensor (anything narrower would be read or written past its end)"""
        tt = torch()
        if not isinstance(t, tt.Tensor):
            raise TypeError('%s must be a torch tensor on %s' % (what, self.device))
        if t.device != self.device:
            raise ValueError('%s on %s, engine on %s' % (what, t.device, self.device))
        if f64 and t.dtype != tt.float64:
            raise TypeError('%s must be float64 (got %s)' % (what, t.dtype))
        return t

    def stack_mean(self, frames, minus=None, gray3=False):
        """imgAverage(frames) [- minus] [-> toGray]: frames = device tensor [n, ...] (any supported dtype; colour frames
        [n,H,W,3] with gray3) -> float64 tensor of one frame's shape (without the channel axis if gray3)"""
        tt = torch()
        frames = self._k5_tensor(frames, 'frames').contiguous()
        if gray3 and (frames.dim() < 2 or frames.shape[-1] != 3):
            raise ValueError('gray3 needs colour frames [n, ..., 3], got %s' % (tuple(frames.shape),))
        n = frames.shape[0]
        elems = int(frames[0].numel())
        shape = tuple(frames.shape[1:-1]) if gray3 else tuple(frames.shape[1:])
        out = tt.empty(shape, dtype=tt.float64, device=self.device)
        mp, ms, use = None, 0.0, 0
        keep = None
        if minus is not None:
            if isinstance(minus, (int, float)):
                ms, use = float(minus), 1
            else:
                keep = (minus if isinstance(minus, tt.Tensor) else tt.from_numpy(np.ascontiguousarray(minus, dtype=np.float64)))
                keep = keep.to(device=self.device, dtype=tt.float64).contiguous()
                if keep.numel() != elems:
                    raise ValueError('background of %d samples for frames of %d' % (keep.numel(), elems))
                mp = ctypes.c_void_p(keep.data_ptr())
        _lib.check(self.lib.imgcorr_stack_mean(self._h, ctypes.c_void_p(frames.data_ptr()), _dtype_code(frames.dtype), n, elems,
                                               mp, ms, use, int(bool(gray3)), ctypes.c_void_p(out.data_ptr()), self._stream()))
        return out

    def scale_(self, data, divisor):
        """data /= divisor in place (contiguous float64 device tensor)"""
        self._k5_tensor(data, 'data', f64=True)
        if not data.is_contiguous():
            raise ValueError('scale_ works in place and needs a contiguous tensor')
        _lib.check(self.lib.imgcorr_scale_f64(self._h, ctypes.c_void_p(data.data_ptr()), int(data.numel()), float(divisor), self._stream()))
        return data

    def subsample(self, img, step_y, step_x):
        """img[::step_y, ::step_x] of a float64 device image"""
        tt = torch()
        img = self._k5_tensor(img, 'img', f64=True).contiguous()
        if img.dim() != 2:
            raise ValueError('subsample needs a 2-d image, got %s' % (tuple(img.shape),))
        step_y, step_x = int(step_y), int(step_x)
        if step_y < 1 or step_x < 1:
            raise ValueError('steps must be >= 1 (got %d, %d)' % (step_y, step_x))
        h, w = img.shape
        out = tt.empty(((h + step_y - 1) // step_y, (w + step_x - 1) // step_x), dtype=tt.float64, device=self.device)
        _lib.check(self.lib.imgcorr_subsample_f64(self._h, ctypes.c_void_p(img.data_ptr()), h, w, int(step_y), int(step_x),
                                                  ctypes.c_void_p(out.data_ptr()), self._stream()))
        return out

    def linear_fit(self, frames, x, max_intensity=65535, min_ascent=0.001, want_rmse=True):
        """per-pixel line frames[k] = offset + ascent * x[k] (getLinearityFunction): device tensor [n,H,W] -> float64 offset,
        ascent (, rmse)"""
        tt = torch()
        frames = self._k5_tensor(frames, 'frames').contiguous()
        n = frames.shape[0]
        px = int(frames[0].numel())
        x = [float(v) for v in x]
        if len(x) != n:
            raise ValueError('%d exposure times for %d frames' % (len(x), n))
        xs = (ctypes.c_double * n)(*x)
        offset = tt.empty(tuple(frames.shape[1:]), dtype=tt.float64, device=self.device)
        ascent = tt.empty_like(offset)
        rmse = tt.empty_like(offset) if want_rmse else None
        _lib.check(self.lib.imgcorr_linear_fit(self._h, ctypes.c_void_p(frames.data_ptr()), _dtype_code(frames.dtype), n, px, xs,
                                               float(max_intensity), float(min_ascent), ctypes.c_void_p(offset.data_ptr()),
                                               ctypes.c_void_p(ascent.data_ptr()), ctypes.c_void_p(rmse.data_ptr()) if want_rmse else None,
                                               self._stream()))
        return (offset, ascent, rmse) if want_rmse else (offset, ascent)

    def undistort_maps(self):
        tt = torch()
        mapx = tt.empty((self.H, self.W), dtype=tt.float32, device=self.device)
        mapy = tt.empty_like(mapx)
        _lib.check(self.lib.imgcorr_undistort_maps(self._h, ctypes.c_void_p(mapx.data_ptr()),
                                                   ctypes.c_void_p(mapy.data_ptr()), self._stream()))
        return mapx, mapy

    @staticmethod
    def _bg_code(bg_dtype, raw_code):
        """library dtype code of per-frame backgrounds: the frames' dtype or float32"""
        tt = torch()
        if isinstance(bg_dtype, tt.dtype):
            code = {tt.uint8: _lib.U8, tt.uint16: _lib.U16, tt.float32: _lib.F32}.get(bg_dtype)
        else:
            code = NP_CODES.get(np.dtype(bg_dtype))
        if code is None or code not in (raw_code, _lib.F32):
            raise ValueError("bg of dtype %s: the frames' dtype or float32" % (bg_dtype,))
        return code

    def correct_batch(self, raw, threshold=0.1, ksize=3, flags=DO_DARK | DO_FLAT | DO_NAN_TO_NUM, use_lens=True,
                      border_value=0.0, window=None, out_dtype=None, out=None, out_scale=None, bg=None):
        """K1 -> K2 [-> perspective stage with DO_PERSPECTIVE in flags] for every frame of a device-resident batch [n,H,W].
        uint16 / uint8 output stores the float32 result v as round_half_even(clip((v - offset) * gain)) with
        ``out_scale=(offset, gain)`` (default (0, 1)), inside the chain's last kernel.
        ``bg``: one background image per frame, a CUDA tensor [n,H,W] on this engine's device of the frames' dtype or
        float32: frame i subtracts bg[i] in place of the dark map (imgcorr_correct_batch_bg; flags must hold DO_DARK)."""
        tt = torch()
        squeeze = raw.dim() == 2
        raw = self._frames(raw)
        n = raw.shape[0]
        if bg is not None:
            if not isinstance(bg, tt.Tensor) or not bg.is_cuda or bg.device != self.device:
                raise ValueError('bg must be a CUDA tensor on %s' % self.device)
            if squeeze and bg.dim() == 2:
                bg = bg.unsqueeze(0)
            if tuple(bg.shape) != tuple(raw.shape):
                raise ValueError('bg has shape %s, frames %s' % (tuple(bg.shape), tuple(raw.shape)))
            bg_code = self._bg_code(bg.dtype, _dtype_code(raw.dtype))
            bg = bg.contiguous()
        lens, (x0, y0, ow, oh), (h, w) = self.chain_shape(flags, use_lens, window)
        if out is None:
            out = tt.empty((n, h, w), dtype=out_dtype or tt.float32, device=self.device)
        else:
            self._check_out(out, (h, w) if squeeze and out.dim() == 2 else (n, h, w))
        self._set_out_scale(_dtype_code(out.dtype), out_scale)
        if bg is not None:
            _lib.check(self.lib.imgcorr_correct_batch_bg(
                self._h, ctypes.c_void_p(raw.data_ptr()), _dtype_code(raw.dtype), ctypes.c_void_p(bg.data_ptr()), bg_code,
                ctypes.c_void_p(out.data_ptr()), _dtype_code(out.dtype), n, float(threshold), int(ksize), int(flags),
                int(lens), float(border_value), x0, y0, ow, oh, self._stream()))
            return out[0] if squeeze else out
        _lib.check(self.lib.imgcorr_correct_batch(
            self._h, ctypes.c_void_p(raw.data_ptr()), _dtype_code(raw.dtype), ctypes.c_void_p(out.data_ptr()),
            _dtype_code(out.dtype), n, float(threshold), int(ksize), int(flags), int(lens), float(border_value),
            x0, y0, ow, oh, self._stream()))
        return out[0] if squeeze else out

    def correct_host(self, raw, out=None, threshold=0.1, ksize=3, flags=DO_DARK | DO_FLAT | DO_NAN_TO_NUM,
                     use_lens=True, border_value=0.0, window=None, out_dtype=np.float32, out_scale=None, bg=None):
        """The chain on HOST numpy frames [n,H,W] (uint8/uint16/float32): pinned staging, H2D, kernels and
        D2H of consecutive frames overlap inside the library.  Synchronous.  flags, out_scale as correct_batch.
        ``bg``: one background image per frame, a numpy array [n,H,W] of the frames' dtype or float32, native byte order
        (imgcorr_correct_host_bg)."""
        squeeze = raw.ndim == 2
        raw = np.ascontiguousarray(raw)
        big_endian = raw.dtype.byteorder == '>' or (raw.dtype.byteorder == '=' and not np.little_endian)
        if big_endian:
            if raw.dtype.itemsize != 2 or raw.dtype.kind != 'u':
                raise TypeError('big-endian ingest is implemented for uint16 frames (got %s)' % raw.dtype)
            raw = raw.view(raw.dtype.newbyteorder('<'))          # same bytes; K1 swaps them in its load
        if squeeze:
            raw = raw[None]
        if raw.shape[1:] != (self.H, self.W):
            raise ValueError('frames of shape %s do not match the engine (%d, %d)' % (raw.shape, self.H, self.W))
        n = raw.shape[0]
        if bg is not None:
            if not isinstance(bg, np.ndarray):
                raise ValueError('bg must be a numpy array for host frames')
            if squeeze and bg.ndim == 2:
                bg = bg[None]
            if bg.shape != raw.shape:
                raise ValueError('bg has shape %s, frames %s' % (bg.shape, raw.shape))
            if not bg.dtype.isnative:
                raise ValueError('bg must be in native byte order')
            bg_code = self._bg_code(bg.dtype, NP_CODES.get(raw.dtype))
            bg = np.ascontiguousarray(bg)
        lens, (x0, y0, ow, oh), (h, w) = self.chain_shape(flags, use_lens, window)
        if out is None:
            out = np.empty((n, h, w), dtype=out_dtype)
        if not out.flags.c_contiguous or out.shape != (n, h, w):
            raise ValueError('out must be C-contiguous of shape %s' % ((n, h, w),))
        if out.dtype not in NP_CODES:
            raise TypeError('unsupported output dtype %s (uint8, uint16, float32, float64)' % out.dtype)
        self._set_out_scale(NP_CODES[out.dtype], out_scale)
        with self.ingest(big_endian, 0):
            if bg is not None:
                _lib.check(self.lib.imgcorr_correct_host_bg(
                    self._h, raw.ctypes.data_as(ctypes.c_void_p), NP_CODES[raw.dtype], bg.ctypes.data_as(ctypes.c_void_p),
                    bg_code, out.ctypes.data_as(ctypes.c_void_p), NP_CODES[out.dtype], n, float(threshold), int(ksize),
                    int(flags), int(lens), float(border_value), x0, y0, ow, oh))
            else:
                _lib.check(self.lib.imgcorr_correct_host(
                    self._h, raw.ctypes.data_as(ctypes.c_void_p), NP_CODES[raw.dtype], out.ctypes.data_as(ctypes.c_void_p),
                    NP_CODES[out.dtype], n, float(threshold), int(ksize), int(flags), int(lens), float(border_value),
                    x0, y0, ow, oh))
        return out[0] if squeeze else out


def host_fingerprint(arr):
    """64-bit fingerprint of a C-contiguous numpy array's bytes (imgcorr_host_fingerprint; no GPU involved)"""
    out = ctypes.c_ulonglong(0)
    _lib.check(_lib.lib().imgcorr_host_fingerprint(arr.ctypes.data_as(ctypes.c_void_p), arr.nbytes, ctypes.byref(out)))
    return int(out.value)


def pinned_empty(shape, dtype):
    """numpy array backed by page-locked memory from imgcorr_host_alloc (freed with the array)."""
    lib = _lib.lib()
    dtype = np.dtype(dtype)
    nbytes = int(np.prod(shape)) * dtype.itemsize
    p = ctypes.c_void_p()
    _lib.check(lib.imgcorr_host_alloc(nbytes, ctypes.byref(p)))

    class _Owner(object):
        def __init__(self, ptr):
            self.ptr = ptr

        def __del__(self):
            try:
                lib.imgcorr_host_free(self.ptr)
            except Exception:
                pass

    buf = (ctypes.c_char * max(nbytes, 1)).from_address(p.value)
    buf._owner = _Owner(p)
    arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
    return arr


_STAGE = {}


def to_numpy(t, threads=8):
    """device tensor -> new numpy array.  Large results go through a cached page-locked staging tensor and a
    multi-threaded copy into the fresh array: `tensor.cpu()` spends ~45 ms on the page faults of a 98 MB float64
    frame (4096x3000), this takes ~6 ms.  The array returned is ordinary pageable memory owned by the caller."""
    tt = torch()
    nbytes = t.numel() * t.element_size()
    if not t.is_cuda or nbytes < (16 << 20):
        return t.cpu().numpy()
    t = t.contiguous()
    key = (t.dtype, t.device.index)
    stage = _STAGE.get(key)
    if stage is None or stage.numel() < t.numel():
        stage = _STAGE[key] = tt.empty(t.numel(), dtype=t.dtype, pin_memory=True)
    view = stage[:t.numel()].view(t.shape)
    view.copy_(t)                                  # synchronous for a pinned destination
    src = view.numpy()
    out = np.empty(src.shape, src.dtype)
    flat_src, flat_out = src.reshape(-1), out.reshape(-1)
    import threading
    n = max(1, min(int(threads), os.cpu_count() or 1, nbytes >> 23))      # one thread per 8 MB
    cuts = np.linspace(0, flat_src.size, n + 1).astype(np.int64)
    workers = [threading.Thread(target=np.copyto, args=(flat_out[a:b], flat_src[a:b])) for a, b in zip(cuts[:-1], cuts[1:])]
    for w in workers:
        w.start()
    for w in workers:
        w.join()
    return out


_ENGINES = {}          # (device, H, W) -> Engine, least recently used first
MAX_CACHED_ENGINES = 16


def get_engine(height, width, device=None):
    """the cached engine (context: calibration copies, scratch, pinned rings) for a device and frame shape.  At most
    MAX_CACHED_ENGINES are kept; the least recently used one is dropped from the cache when a new shape arrives — its
    context (device memory) is freed as soon as nobody else holds the engine (Engine.__del__), never under a caller's feet."""
    tt = require_cuda()
    idx = tt.cuda.current_device() if device is None else tt.device('cuda', device).index
    key = (idx, int(height), int(width))
    e = _ENGINES.pop(key, None)
    if e is None or e._h is None:
        e = Engine(height, width, idx)
        while len(_ENGINES) >= MAX_CACHED_ENGINES:
            _ENGINES.pop(next(iter(_ENGINES)))
    _ENGINES[key] = e
    return e
