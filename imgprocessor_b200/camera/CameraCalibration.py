"""CameraCalibration: drop-in for imgProcessor.camera.CameraCalibration.CameraCalibration
(camera/CameraCalibration.py:52-636).

The calibration store (``coeffs`` schema :63-81, ``add*`` :187-285, date lookup :29-49, 590-611,
pickle persistence :300-322) is host code with the reference's behaviour.  ``correct()`` (:351-459)
resolves the calibration exactly as the reference does, prints the same progress lines, and then runs
the per-frame chain on the B200 through libimgcorr (K1 fused dark/flat/median-threshold, K2
undistortion) instead of numpy / scipy / OpenCV.  ``correct_batch()`` is the new entry point for
independent frames (a stack handed to ``correct()`` means "average these exposures" in the reference,
:385-406, not a batch).
"""
from __future__ import print_function

import pickle
import time

import numpy as np

from .. import _lib
from .. import engine as _engine
from ..imgIO import imread
from . import NoiseLevelFunction as _nlf
from .LensDistortion import LensDistortion

DATE_FORMAT = "%d %b %y - %H:%M"   # e.g. '30 Nov 15 - 13:20'


def _toDate(date):
    return time.localtime() if date is None else time.strptime(date, DATE_FORMAT)


def _insertDateIndex(date, entries):
    """position that keeps ``entries`` (items start with a struct_time) sorted newest first"""
    for i, e in enumerate(entries):
        if e[0] < date:
            return i
    return len(entries)


def _getFromDate(entries, date):
    """the calibration in force at ``date``: the entry just before the first one older than ``date``;
    the newest entry if date is None / unparsable or younger than everything."""
    try:
        i = _insertDateIndex(_toDate(date), entries) - 1
    except (ValueError, TypeError):
        return entries[0]
    return entries[0] if i == -1 else entries[i]


def _map_token(kind, arr):
    """identity of a calibration map for the engine's upload cache: shape, dtype and a fingerprint of EVERY byte of the
    array (imgcorr_host_fingerprint: a few host threads, ~1 ms for a 4096x3000 float32 map), so that an array modified in
    place between two calls — a patched hot pixel is enough — is uploaded again.  The reference reads the array on every
    call (camera/CameraCalibration.py:500-502, 521-526); `id()` is not part of the key (ids are recycled)."""
    if not isinstance(arr, np.ndarray):
        return None
    if not arr.flags.writeable and arr.base is None:
        # a read-only array that owns its memory cannot be edited in place: object identity + address + a sampled hash (in case
        # the id is recycled by a new array) is enough, and the ~1 ms full pass per map and call is saved.  Mark calibration
        # arrays read-only (arr.setflags(write=False)) to get this path.
        flat = arr.reshape(-1)
        step = max(1, flat.size // 4096)
        return (kind, 'ro', id(arr), arr.ctypes.data, arr.shape, arr.dtype.str, hash(flat[::step].tobytes()))
    a = arr if arr.flags.c_contiguous else np.ascontiguousarray(arr)
    return (kind, arr.shape, arr.dtype.str, _engine.host_fingerprint(a))


class _BoundedNLF(object):
    """NoiseLevelFunction.boundedFunction(x, minY, ax, ay) (camera/NoiseLevelFunction.py:94-107) with its parameters
    kept, so that kernel K4 can evaluate it per pixel; calling it evaluates the same expression with numpy."""

    def __init__(self, minY, ax, ay):
        self.coeff = (minY, ax, ay)

    def __call__(self, x):
        minY, ax, ay = self.coeff
        with np.errstate(invalid='ignore'):
            y = ay * (x - ax) ** 0.5
        return np.maximum(np.nan_to_num(y), minY)


class CameraCalibration(object):
    ftype = '.cal'

    def __init__(self):
        self.noise_level_function = None
        self.coeffs = {
            'name': 'no camera',
            'depth': 16,                  # bit depth of the sensor
            'light spectra': [],
            'dark current': [],           # [[date, info, bg | (slope, intercept), error], ...]
            'flat field': {},             # {light: [[date, info, array, error], ...]}
            'lens': {},                   # {light: [[date, info, LensDistortion.coeffs], ...]}
            'noise': [],
            'psf': {},
            'shape': None,
            'balance': {},
        }
        self.temp = {}
        self._last = None                 # (raw frame, bg, flat) of the last correct() for .last_img

    # ------------------------------------------------------------------ store (host)
    def _getDate(self, typ, light):
        d = self.coeffs[typ]
        if type(d) is dict:
            assert light is not None, 'need light spectrum given to access [%s]' % typ
            d = d[light]
        return d

    def dates(self, typ, light=None):
        try:
            return [self._toDateStr(c[0]) for c in self._getDate(typ, light)]
        except KeyError:
            return []

    def infos(self, typ, light=None, date=None):
        d = self._getDate(typ, light)
        if date is None:
            return [c[1] for c in d]
        return _getFromDate(d, date)[1]

    def overview(self):
        c = self.coeffs
        out = ['camera name: %s' % c['name'], 'max value: %s' % c['depth'], 'light spectra: %s' % c['light spectra'],
               'dark current:']
        for (date, info, data, error) in c['dark current']:
            shp = tuple(getattr(a, 'shape', None) for a in data) if isinstance(data, tuple) else getattr(data, 'shape', None)
            out.append('\t date: %s\n\t\t info: %s; shape:%s' % (self._toDateStr(date), info, shp))
        for title, key, fmt in (('flat field:', 'flat field', lambda v: 'array:%s' % (v[2].shape,)),
                                ('lens:', 'lens', lambda v: 'coeffs:%s' % (v[2],)),
                                ('Point spread function:', 'psf', lambda v: 'shape:%s' % (v[2].shape,))):
            out.append(title)
            for light, vals in c[key].items():
                out.append('\t light: %s' % light)
                for v in vals:
                    out.append('\t\t date: %s\n\t\t\t info: %s; %s' % (self._toDateStr(v[0]), v[1], fmt(v)))
        out.append('noise:')
        for (date, info, nlf_coeff, error) in c['noise']:
            out.append('\t date: %s\n\t\t info: %s; coeffs:%s' % (self._toDateStr(date), info, nlf_coeff))
        return '\n'.join(out)

    @staticmethod
    def _toDateStr(date_struct):
        return time.strftime(DATE_FORMAT, date_struct)

    @staticmethod
    def currentTime():
        return time.strftime(DATE_FORMAT)

    def _registerLight(self, light_spectrum):
        if light_spectrum not in self.coeffs['light spectra']:
            self.coeffs['light spectra'].append(light_spectrum)

    def setCamera(self, camera_name, bit_depth=16):
        self.coeffs['name'] = camera_name
        self.coeffs['depth'] = bit_depth

    def _checkShape(self, array):
        if not isinstance(array, np.ndarray):
            return
        s = self.coeffs['shape']
        if s is None:
            self.coeffs['shape'] = array.shape
        elif s[:2] != array.shape[:2]:
            raise Exception("""array shapes are different: stored(%s), given(%s)
if shapes are transposed, execute self.transpose() once """ % (s, array.shape))

    def _insert(self, entries, date, item):
        entries.insert(_insertDateIndex(date, entries), item)

    def _light_list(self, key, light_spectrum):
        self._registerLight(light_spectrum)
        return self.coeffs[key].setdefault(light_spectrum, [])

    def addDarkCurrent(self, slope, intercept=None, date=None, info='', error=None):
        """``addDarkCurrent(bg_array)`` stores a constant background image.  With ``intercept`` the pair is
        stored as the reference stores it (:203-207) — a list entry that calcDarkCurrent does not evaluate
        as a linear model (only legacy *tuple* entries are, :507-513)."""
        date = _toDate(date)
        self._checkShape(slope)
        self._checkShape(intercept)
        data = slope if intercept is None else (slope, intercept)
        self._insert(self.coeffs['dark current'], date, [date, info, data, error])

    def addNoise(self, nlf_coeff, date=None, info='', error=None):
        date = _toDate(date)
        self._insert(self.coeffs['noise'], date, [date, info, nlf_coeff, error])

    def addDeconvolutionBalance(self, balance, date=None, info='', light_spectrum='visible'):
        date = _toDate(date)
        self._insert(self._light_list('balance', light_spectrum), date, [date, info, balance])

    def addPSF(self, psf, date=None, info='', light_spectrum='visible'):
        date = _toDate(date)
        self._insert(self._light_list('psf', light_spectrum), date, [date, info, psf])

    def addFlatField(self, arr, date=None, info='', error=None, light_spectrum='visible'):
        self._registerLight(light_spectrum)
        self._checkShape(arr)
        date = _toDate(date)
        self._insert(self._light_list('flat field', light_spectrum), date, [date, info, arr, error])

    def addLens(self, lens, date=None, info='', light_spectrum='visible'):
        """lens: a LensDistortion instance (this package's or any object with ``.coeffs``) or a saved file"""
        self._registerLight(light_spectrum)
        date = _toDate(date)
        if not hasattr(lens, 'coeffs'):
            l = LensDistortion()
            l.readFromFile(lens)
            lens = l
        self._insert(self._light_list('lens', light_spectrum), date, [date, info, lens.coeffs])

    def clearOldCalibrations(self, date=None):
        self.coeffs['dark current'] = [self.coeffs['dark current'][-1]]
        self.coeffs['noise'] = [self.coeffs['noise'][-1]]
        for key in ('flat field', 'lens'):
            for light in self.coeffs[key]:
                self.coeffs[key][light] = [self.coeffs[key][light][-1]]

    def deleteCoeff(self, name, date, light=None):
        try:
            c = self.coeffs[name][light]
        except TypeError:
            c = self.coeffs[name]
        i = _insertDateIndex(_toDate(date), c) - 1
        if i == -1:
            raise Exception('no coeff %s for date %s' % (name, date))
        c.pop(i)

    def getCoeff(self, name, light=None, date=None):
        """calibration for the given light spectrum, or for any other one if there is none (:590-611)"""
        d = self.coeffs[name]
        try:
            c = d[light]
        except KeyError:
            try:
                k, c = next(iter(d.items()))
            except StopIteration:
                return None
            if light is not None:
                print('no calibration found for [%s] - using [%s] instead' % (light, k))
        except TypeError:
            c = d
        return _getFromDate(c, date)

    def _correctPath(self, path):
        return path if path.endswith(self.ftype) else path + self.ftype

    @staticmethod
    def loadFromFile(path):
        cal = CameraCalibration()
        path = cal._correctPath(path)
        with open(path, 'rb') as f:
            try:
                d = pickle.load(f)
            except UnicodeDecodeError:
                f.seek(0)
                d = pickle.load(f, encoding='latin1')
        cal.coeffs.update(d)
        return cal

    def saveToFile(self, path):
        with open(self._correctPath(path), 'wb') as f:
            pickle.dump(dict(self.coeffs), f, protocol=pickle.HIGHEST_PROTOCOL)

    def transpose(self):
        """transpose every stored calibration array (x,y) <-> (y,x)"""
        s = self.coeffs['shape']

        def walk(item):
            if type(item) == list:
                for n, it in enumerate(item):
                    if type(it) == tuple:
                        it = item[n] = list(it)
                    if type(it) == list:
                        walk(it)
                    if isinstance(it, np.ndarray) and it.shape == s:
                        item[n] = it.T

        for item in self.coeffs.values():
            if type(item) == dict:
                for sub in item.values():
                    walk(sub)
            else:
                walk(item)
        self.coeffs['shape'] = s[::-1]

    # ------------------------------------------------------------------ calibration lookup for one call
    def calcDarkCurrent(self, exposuretime, date=None):
        """host evaluation, as the reference (:504-518); correct() itself evaluates the linear model on
        the device and only calls this for the ``temp['bg']`` side effect of plain array entries."""
        d = _getFromDate(self.coeffs['dark current'], date)
        if type(d) == tuple:
            offs, ascent = d[2]
            bg = offs + ascent * exposuretime
            mx = 2 ** self.coeffs['depth'] - 1
            with np.errstate(invalid='ignore'):
                bg[bg > mx] = mx
            return bg
        return d[2]

    def getLens(self, light_spectrum, date):
        d = self.getCoeff('lens', light_spectrum, date)
        if d:
            return LensDistortion(d[2])

    def _normalise_args(self, date, light_spectrum):
        if isinstance(date, str) or date is None:
            date = dict.fromkeys(('dark current', 'flat field', 'lens', 'noise', 'psf'), date)
        if light_spectrum is None:
            try:
                light_spectrum = self.coeffs['light spectra'][0]
            except IndexError:
                pass
        return date, light_spectrum

    def _resolve_dark(self, shape, exposure_time, bgImages, date):
        """-> dict(dark=, ascent=, exposure=) for the engine, or None if the stage is skipped.
        Prints / swallows errors like the reference's try/except around _correctDarkCurrent (:418-422)."""
        print('... remove dark current')
        if bgImages is not None:
            if type(bgImages) in (list, tuple) or (isinstance(bgImages, np.ndarray) and bgImages.ndim == 3):
                if len(bgImages) > 1:
                    # several background images: STE-free average (:488-494), kernel K4
                    bg = self._ste_average(bgImages, self.noise_level_function)       # whatever it is, None included (:490-494)
                else:
                    bg = imread(bgImages[0])
            else:
                bg = imread(bgImages)
            entry = None
        else:
            entry = _getFromDate(self.coeffs['dark current'], date)
            bg = None
        if entry is not None and type(entry) == tuple:
            offs, ascent = entry[2]
            if exposure_time is None:
                raise TypeError("unsupported operand type(s) for *: 'float' and 'NoneType'")
            np.broadcast_to(offs, shape), np.broadcast_to(ascent, shape)
            self.temp['bg'] = None          # evaluated on the device; see calcDarkCurrent for a host copy
            return dict(dark=offs, ascent=ascent, exposure=float(exposure_time), token=None)
        if entry is not None:
            bg = entry[2]
        self.temp['bg'] = bg
        np.broadcast_to(np.asarray(bg), shape)           # same failure as `image -= bg` for a bad shape
        return dict(dark=bg, ascent=None, exposure=0.0, token=_map_token('dark', bg))

    def _configure_engine(self, eng, shape, bgImages, exposure_time, light_spectrum, date, use_dark=True):
        """upload whatever calibration applies; returns (flags, lens-or-None).  use_dark=False: the call brings one background
        image per frame (correct_batch(bg_frames=...)), which takes the dark stage's place like bgImages does in correct():
        the calibrated dark entry is not resolved and the engine's dark map is left as it is."""
        flags = 0
        if not use_dark:
            print('... remove dark current')
            flags |= _lib.DO_DARK
            self._last_bg = None
        else:
            try:
                d = self._resolve_dark(shape, exposure_time, bgImages, date['dark current'])
                eng.set_dark(d['dark'], d['ascent'], d['exposure'], self.coeffs['depth'], token=d['token'])
                flags |= _lib.DO_DARK
                self._last_bg = d
            except _lib.ImgcorrError:
                raise
            except Exception as errm:
                print('Error: %s' % errm)
                self._last_bg = None
        self._last_flat = None
        try:
            f = self.getCoeff('flat field', light_spectrum, date['flat field'])
            if f is not None:
                print('... remove vignetting and sensitivity')
                flat = f[2]
                np.broadcast_to(np.asarray(flat), shape)
                eng.set_flat(flat, token=_map_token('flat', flat))
                flags |= _lib.DO_FLAT
                self._last_flat = flat
        except _lib.ImgcorrError:
            raise
        except Exception as errm:
            print('Error: %s' % errm)
        return flags

    # ------------------------------------------------------------------ single-time-effect removal (K4)
    def _calibrated_nlf(self, date):
        """the 'noise' calibration entry becomes the noise level function on first use (:392-397); None if there is neither
        an entry nor a function from an earlier call — SingleTimeEffectDetection then estimates one from the images"""
        if self.noise_level_function is None:
            n = self.coeffs['noise']
            if len(n):
                coeff = tuple(float(v) for v in _getFromDate(n, date)[2])
                self.noise_level_function = _BoundedNLF(*coeff)
        return self.noise_level_function

    def _ste_average(self, images, nlf, n_std=4, keep_estimate=False):
        """SingleTimeEffectDetection(images, nStd=4, noise_level_function=nlf).noSTE (:401-403, 491-494) -> float64.
        ``nlf`` None: the function is estimated from min(images[0], images[1]) like the reference does
        (SingleTimeEffectDetection.py:43-45 -> NoiseLevelFunction.oneImageNLF) and, in the main branch of correct(), kept
        for later calls (:405-406).  boundedFunction-shaped functions are evaluated per pixel inside kernel K4; any other
        callable (the polynomial fallback of the estimate, a user's own function) is evaluated here on
        min(images[0], images[1]) and handed to K4 as a threshold map."""
        frames = [imread(i, 'gray') for i in images]
        if any(f.ndim != 2 or f.shape != frames[0].shape for f in frames):
            raise ValueError('single-time-effect removal needs 2-D frames of one shape')
        dt = np.result_type(*[f.dtype for f in frames])
        if dt.type not in (np.uint8, np.uint16, np.float32, np.float64):
            dt = np.dtype(np.float64)
        stack = np.stack([np.asarray(f, dtype=dt.newbyteorder('=')) for f in frames])
        first = None
        if nlf is None:
            first = np.min((stack[0].astype(np.float64), stack[1]), axis=0)
            nlf = _nlf.oneImageNLF(first)[0]
            if keep_estimate:
                self.noise_level_function = nlf
        params = getattr(nlf, 'coeff', None)
        if params is None:
            params = getattr(nlf, 'params', None)
        eng = _engine.get_engine(*stack.shape[1:])
        tt = _engine.torch()
        dev = tt.from_numpy(stack).to(eng.device)
        if params is not None:
            return _engine.to_numpy(eng.ste_average(dev, params, n_std))
        if first is None:
            first = np.min((stack[0].astype(np.float64), stack[1]), axis=0)
        thr = np.broadcast_to(np.asarray(nlf(first), dtype=np.float64) * n_std, first.shape)
        return _engine.to_numpy(eng.ste_average(dev, threshold=thr))

    # ------------------------------------------------------------------ THE hot path
    def correct(self, images, bgImages=None, exposure_time=None, light_spectrum=None, threshold=0.1, keep_size=True,
                date=None, deblur=False, denoise=False):
        """Correct one frame: dark current, flat field, 3x3 median-threshold artefact removal, lens
        distortion.  Same arguments and return value (a new float64 array; the input is never modified)
        as the reference.  Several exposures of one scene (list / 3-D array) are first merged into one
        single-time-effect-free average (kernel K4; the noise level function comes from the 'noise' calibration or is
        estimated from the exposures as in the reference).

        Precision: the chain computes in float32 between its stages (the north star's arithmetic).  For uint8 / uint16 /
        float32 frames and float32-representable calibration maps every pointwise value is the correctly rounded float32
        of the reference's float64 value (0 ulp) and the end-to-end deviation from the float64 reference stays below
        1e-5 of full scale; float64 frames, float64 calibration maps and the float64 average of several exposures are
        rounded to float32 once on entry (one extra half-ulp of float32), and the result is widened to float64 on the way out.
        Not supported on the GPU
        path: ``denoise``; ``deblur`` is reported and skipped like any other failing stage."""
        print('CORRECT CAMERA ...')
        date, light_spectrum = self._normalise_args(date, light_spectrum)
        if type(images) in (list, tuple) or (isinstance(images, np.ndarray) and images.ndim == 3
                                             and images.shape[-1] not in (3, 4)):
            if len(images) > 1:
                # several exposures of the same scene: one STE-free average (:390-406), kernel K4
                print('... remove single-time-effects from images ')
                images = self._ste_average(images, self._calibrated_nlf(date['noise']), keep_estimate=True)
            else:
                images = images[0]
        image = imread(images)
        if not isinstance(image, np.ndarray) or image.ndim != 2:
            raise ValueError('correct() expects one single-channel 2-D frame')
        self._checkShape(image)
        self.last_light_spectrum = light_spectrum
        H, W = image.shape
        big_endian = image.dtype.kind == 'u' and image.dtype.itemsize == 2 and image.dtype.byteorder == '>'
        if big_endian:
            raw = image.view(image.dtype.newbyteorder('<'))      # reader.RAW frames: same bytes, K1 swaps in its load
        else:
            raw = image if image.dtype.type in (np.uint8, np.uint16, np.float32) and image.dtype.isnative \
                else image.astype(np.float32)
        eng = _engine.get_engine(H, W)
        flags = self._configure_engine(eng, (H, W), bgImages, exposure_time, light_spectrum, date)
        self._last = (raw if not big_endian else image.astype(np.uint16), flags)
        if threshold > 0:
            print('... remove artefacts')
            flags |= _lib.DO_NAN_TO_NUM
        if deblur:
            print('... remove blur')
            print('Error: deblur (skimage Wiener deconvolution) is not available on the GPU path')
        lens = None
        try:
            lens = self.getLens(light_spectrum, date['lens'])
            if lens:
                print('... correct lens distortion')
                lens._lens_setup(W, H)
        except _lib.ImgcorrError:
            raise
        except TypeError:
            lens = None
        except Exception as errm:
            print('Error: %s' % errm)
            lens = None
        if denoise:
            raise NotImplementedError('denoise (skimage non-local means) is not available on the GPU path')
        tt = _engine.torch()
        dev = tt.from_numpy(np.ascontiguousarray(raw)).to(eng.device, non_blocking=False)
        window = None
        if lens and not keep_size:
            window = tuple(int(v) for v in lens.roi)
        with eng.ingest(big_endian, 0):
            out = eng.correct_batch(dev, threshold=threshold if threshold > 0 else 0.0, ksize=3, flags=flags,
                                    use_lens=bool(lens), window=window, out_dtype=tt.float64)
        result = _engine.to_numpy(out)
        print('DONE')
        return result

    @property
    def last_img(self):
        """dark- and flat-corrected (pre-median) float64 image of the last correct() call — the array the
        reference keeps in ``self.last_img`` (:414-415); computed on demand."""
        if self._last is None:
            raise AttributeError('last_img')
        raw, flags = self._last
        tt = _engine.torch()
        eng = _engine.get_engine(*raw.shape)
        dev = tt.from_numpy(np.ascontiguousarray(raw)).to(eng.device)
        out, _ = eng.pointwise_median(dev, 0.0, 0, flags=flags & ~_lib.DO_NAN_TO_NUM, out_dtype=tt.float64)
        return _engine.to_numpy(out)

    # ------------------------------------------------------------------ batches of independent frames
    @staticmethod
    def _perspective_stage(perspective, out, out_dtype, n):
        """(homography, dsize, border value, tilt factor) of a PerspectiveCorrection as the chain's last stage, or None.
        A sequence of n PerspectiveCorrection objects, one per frame, gives the homographies stacked to (n, 3, 3) and no
        tilt factor; they must agree on dsize and border value."""
        if perspective is None:
            return None
        if isinstance(perspective, (list, tuple)):
            if len(perspective) != n:
                raise ValueError('perspective: %d PerspectiveCorrection objects for %d frames' % (len(perspective), n))
            if n == 0:
                raise ValueError('perspective: an empty sequence')
            for i, pc in enumerate(perspective):
                if pc.opts['do_correctIntensity']:
                    raise ValueError('perspective[%d] has do_correctIntensity: per-frame tilt factors are not supported '
                                     'in the batch chain' % i)
            stages = [pc.correct_params() for pc in perspective]
            for i, s in enumerate(stages):
                if tuple(s[1]) != tuple(stages[0][1]) or s[2] != stages[0][2]:
                    raise ValueError('perspective[%d] has dsize %s and border value %r, perspective[0] %s and %r: the '
                                     'frames of one batch share both' % (i, tuple(s[1]), s[2], tuple(stages[0][1]),
                                                                         stages[0][2]))
            M = np.stack([np.asarray(s[0], np.float64).reshape(3, 3) for s in stages])
            return M, tuple(stages[0][1]), stages[0][2], None
        stage = perspective.correct_params()
        tt = _engine.torch()
        dt = out.dtype if out is not None else out_dtype
        f64 = dt is not None and (dt == tt.float64 if isinstance(dt, tt.dtype) else np.dtype(dt) == np.float64)
        if stage[3] is not None and not f64:
            raise ValueError('perspective with do_correctIntensity needs out_dtype=float64: the tilt-factor division and '
                             'the warp after it are computed in float64 (np.asfarray(img) / tf)')
        return stage

    @staticmethod
    def _set_perspective(eng, stage):
        M, dsize, border_value, tf = stage
        eng.set_perspective(M, dsize, border_value, tf, token=_map_token('tilt', tf))

    def correct_batch(self, frames, bgImages=None, exposure_time=None, light_spectrum=None, threshold=0.1,
                      keep_size=True, date=None, out=None, out_dtype=None, verbose=False, devices=None, perspective=None,
                      out_scale=None, bg_frames=None):
        """correct() for n INDEPENDENT frames with one calibration lookup.

        ``frames``: numpy [n,H,W] (uint8 / uint16 / float32, host) -> streamed through pinned buffers with
        H2D / kernels / D2H overlapped, result numpy [n,h,w]; or a CUDA torch tensor [n,H,W] -> result stays
        on the device.  ``out_dtype`` defaults to float32 (pass float64 for the reference's dtype).

        ``out_dtype`` uint16 / uint8 (torch.uint16 / torch.uint8 for tensors) returns the float32 result v of every pixel
        as an integer image, converted inside the chain's last kernel: t = (float64(v) - offset) * gain with
        ``out_scale=(offset, gain)`` (default (0, 1)), then 0 for NaN and t <= 0, the dtype's maximum for t >= it, else t
        rounded half to even (OpenCV's saturate_cast for the default scale).  Host frames then bring 2 (or 1) bytes per
        pixel back over PCIe instead of 4.

        ``devices``: CUDA device indices for host frames, e.g. ``range(8)``: the batch is split contiguously over them
        (sharding.shard_range), each device gets its own context with the calibration uploaded once and its own host
        thread driving the pinned H2D / kernels / D2H pipeline (the C ABI calls release the GIL); the shards land in one
        output array.  No collective is involved: frames are independent (SURVEY §8e).

        ``perspective``: a PerspectiveCorrection whose correct() becomes the chain's last stage on the device:
        ``correct_batch(frames, perspective=pc, out_dtype=np.float64)[i]`` equals ``pc.correct(correct(frames[i],
        keep_size=keep_size))``, and with float32 output the float32 chain frame is warped in float32.  The homography
        maps the frame the lens stage returns (the roi crop with keep_size=False).  A tilt factor
        (do_correctIntensity=True) needs float64 output.  The stage stays on the cached engine of the device and frame
        shape after the call, its tilt factor included (float64 on the device: 98 MB at 4096x3000), so that the next call
        with the same PerspectiveCorrection uploads nothing; calls without ``perspective=`` do not use it, and
        ``engine.get_engine(H, W, device).set_perspective(None, None)`` frees it.

        ``perspective`` may also be a list of n PerspectiveCorrection objects, one per frame (each module found at its own
        place, ``pc_i.setReference(quad_i)``): frame i is warped with ``perspective[i]``'s homography, so that
        ``correct_batch(frames, perspective=pcs)[i]`` equals ``pcs[i].correct(correct(frames[i]))``.  They must share the
        destination size and border value, and none may have do_correctIntensity; otherwise ValueError.  With
        ``devices=``, every device gets the matrices of its own shard.

        ``bg_frames``: one background image per frame (the same exposure with the module's current off), of the shape of
        ``frames``: a numpy array for host frames, a CUDA tensor on the frames' device for tensor frames.  Frame i is
        corrected as ``correct(frames[i], bgImages=bg_frames[i])``: ``bg_frames[i]`` takes the calibrated dark current's
        place (which is then not looked up), subtracted in float64 inside K1, so that
        ``correct_batch(frames, bg_frames=bgs, out_dtype=np.float64)[i]`` equals ``correct(frames[i], bgImages=bgs[i])``.
        Backgrounds of the frames' dtype or float32 go to the device as they are (a big-endian uint16 array is swapped on
        the host); any other dtype, float64 included, is rounded to float32 once, as correct() does with float64
        calibration maps.  It combines with ``devices=`` (every device gets its shard's backgrounds), ``perspective=``,
        ``out_dtype`` / ``out_scale`` and ``keep_size``.  ValueError, before any engine is created, for another shape, for
        ``bgImages`` given as well, for a numpy / tensor mismatch with ``frames`` and for a tensor on another device.

        ``exposure_time`` may be a 1-D sequence of n exposure times, one per frame (an .elbin stack's labels, frames taken
        at several exposures).  With a tuple dark-current entry (offset, ascent) frame i evaluates the line model with its
        own time, bit for bit as ``correct_batch(frames[i:i+1], exposure_time=t_i)``, inside K1: with float64 output
        ``correct_batch(frames, exposure_time=ts, out_dtype=np.float64)[i]`` equals ``correct(frames[i],
        exposure_time=ts[i])``.  With an array entry, ``bg_frames`` or ``bgImages`` the times are checked and then unused,
        as correct() does with its scalar.  It combines with host frames, CUDA tensors, ``devices=`` (every device gets
        its shard's times), ``perspective=``, ``keep_size``, ``out_dtype`` / ``out_scale`` and big-endian frames.
        ValueError, before any engine is created, for a length other than n, a sequence that is not 1-D, a non-numeric
        value or NaN."""
        import contextlib
        import io
        tt = _engine.torch()
        date, light_spectrum = self._normalise_args(date, light_spectrum)
        is_tensor = isinstance(frames, tt.Tensor)
        if frames.ndim != 3:
            raise ValueError('correct_batch() expects frames of shape [n,H,W]')
        n, H, W = frames.shape
        s = self.coeffs['shape']
        if s is not None and tuple(s[:2]) != (H, W):
            raise Exception('array shapes are different: stored(%s), given(%s)' % (s, (H, W)))
        if devices is not None:
            devices = [int(d) for d in devices]
            if is_tensor:
                raise ValueError('devices= shards HOST frames; a CUDA tensor is processed on its own device')
            if not devices:
                raise ValueError('devices is empty')
        stage = self._perspective_stage(perspective, out, out_dtype, n)
        if bg_frames is not None:
            bg_frames = self._bg_frames(frames, bg_frames, bgImages)
        times = self._exposure_times(exposure_time, n)
        if times is not None:
            exposure_time = float(times[0]) if n else 0.0       # resolves the dark entry; the table replaces it per frame
        if devices is not None and len(devices) > 1:
            return self._correct_batch_multi(frames, devices, bgImages, exposure_time, light_spectrum, threshold,
                                             keep_size, date, out, out_dtype, verbose, stage, out_scale, bg_frames, times)
        dev_index = frames.device.index if is_tensor else (devices[0] if devices else None)
        eng = _engine.get_engine(H, W, dev_index)
        sink = contextlib.nullcontext() if verbose else contextlib.redirect_stdout(io.StringIO())
        with sink:
            flags = self._configure_engine(eng, (H, W), bgImages, exposure_time, light_spectrum, date,
                                           use_dark=bg_frames is None)
            self._set_exposures(eng, times)
            lens = None
            try:
                lens = self.getLens(light_spectrum, date['lens'])
                if lens:
                    lens._lens_setup(W, H)
                    if eng is not _engine.get_engine(H, W):          # non-default device: set on that engine
                        eng.set_lens(lens.coeffs['cameraMatrix'], lens.coeffs['distortionCoeffs'],
                                     lens._new_camera_matrix)
            except _lib.ImgcorrError:
                raise
            except Exception as errm:
                print('Error: %s' % errm)
                lens = None
        if threshold > 0:
            flags |= _lib.DO_NAN_TO_NUM
        if stage is not None:
            self._set_perspective(eng, stage)
            flags |= _lib.DO_PERSPECTIVE
        window = tuple(int(v) for v in lens.roi) if (lens and not keep_size) else None
        thr = threshold if threshold > 0 else 0.0
        if is_tensor:
            if bg_frames is not None:
                bg_frames = self._bg_dtype(bg_frames, frames.dtype)
            return eng.correct_batch(frames, threshold=thr, ksize=3, flags=flags, use_lens=bool(lens), window=window,
                                     out_dtype=out_dtype or tt.float32, out=out, out_scale=out_scale, bg=bg_frames)
        be = frames.dtype.kind == 'u' and frames.dtype.itemsize == 2 and frames.dtype.byteorder == '>'
        if not be and (frames.dtype.type not in (np.uint8, np.uint16, np.float32) or not frames.dtype.isnative):
            frames = frames.astype(np.float32)
        if bg_frames is not None:
            bg_frames = self._bg_dtype(bg_frames, frames.dtype.newbyteorder('='))
        return eng.correct_host(frames, out=out, threshold=thr, ksize=3, flags=flags, use_lens=bool(lens),
                                window=window, out_dtype=out_dtype or np.float32, out_scale=out_scale, bg=bg_frames)

    @staticmethod
    def _exposure_times(exposure_time, n):
        """correct_batch's per-frame exposure times as a float64 array of n, or None for a scalar / None (used as
        today); ValueError for anything else that is not n numbers"""
        if np.ndim(exposure_time) == 0 and not isinstance(exposure_time, (list, tuple)):
            return None
        tt = _engine.torch()
        if isinstance(exposure_time, tt.Tensor):
            exposure_time = exposure_time.detach().cpu().numpy()
        t = np.asarray(exposure_time)
        if t.ndim != 1:
            raise ValueError('exposure_time: a scalar or a 1-D sequence of one time per frame, got shape %s' % (t.shape,))
        if t.size and t.dtype.kind not in 'iuf':
            raise ValueError('exposure_time: numbers expected, got %s' % t.dtype)
        if t.size != n:
            raise ValueError('exposure_time: %d times for %d frames' % (t.size, n))
        t = t.astype(np.float64)
        if np.isnan(t).any():
            raise ValueError('exposure_time[%d] is NaN' % int(np.flatnonzero(np.isnan(t))[0]))
        return t

    def _set_exposures(self, eng, times):
        """per-frame exposure times on the engine when the line model is in use (a tuple dark entry); otherwise no table"""
        linear = self._last_bg is not None and self._last_bg.get('ascent') is not None
        if times is not None and linear and times.size:
            eng.set_dark_exposures(times)
        elif eng.has_exposures:
            eng.set_dark_exposures(None)

    @staticmethod
    def _bg_frames(frames, bg_frames, bgImages):
        """the refusals of correct_batch(bg_frames=...), before any engine is created"""
        tt = _engine.torch()
        if bgImages is not None:
            raise ValueError('bg_frames and bgImages exclude each other: bg_frames gives every frame its own background')
        if isinstance(frames, tt.Tensor) != isinstance(bg_frames, tt.Tensor):
            raise ValueError('bg_frames must be a CUDA tensor for tensor frames and a numpy array for host frames')
        if not isinstance(bg_frames, tt.Tensor):
            bg_frames = np.asarray(bg_frames)
        elif not bg_frames.is_cuda or bg_frames.device != frames.device:
            raise ValueError('bg_frames on %s, frames on %s' % (bg_frames.device, frames.device))
        if tuple(bg_frames.shape) != tuple(frames.shape):
            raise ValueError('bg_frames of shape %s for frames of shape %s' % (tuple(bg_frames.shape), tuple(frames.shape)))
        return bg_frames

    @staticmethod
    def _bg_dtype(bg, frame_dtype):
        """backgrounds of the frames' dtype or float32 as they are (native byte order); anything else rounded to float32"""
        tt = _engine.torch()
        if isinstance(bg, tt.Tensor):
            return bg if bg.dtype in (frame_dtype, tt.float32) else bg.to(tt.float32)
        dt = bg.dtype.newbyteorder('=')
        if dt in (np.dtype(frame_dtype), np.dtype(np.float32)):
            return bg.astype(dt, copy=False)
        return bg.astype(np.float32)

    def _correct_batch_multi(self, frames, devices, bgImages, exposure_time, light_spectrum, threshold, keep_size, date,
                             out, out_dtype, verbose, stage, out_scale=None, bg_frames=None, times=None):
        """host frames [n,H,W] split over several devices of this process: one engine + one host thread per device"""
        import contextlib
        import io
        import threading
        from .. import sharding
        n, H, W = frames.shape
        be = frames.dtype.kind == 'u' and frames.dtype.itemsize == 2 and frames.dtype.byteorder == '>'
        if not be and (frames.dtype.type not in (np.uint8, np.uint16, np.float32) or not frames.dtype.isnative):
            frames = frames.astype(np.float32)
        if bg_frames is not None:
            bg_frames = self._bg_dtype(bg_frames, frames.dtype.newbyteorder('='))
        engines, own = [], []
        sink = contextlib.nullcontext() if verbose else contextlib.redirect_stdout(io.StringIO())
        lens = None
        try:
            with sink:
                for d in devices:
                    if d in [e.device_index for e in engines]:
                        e = _engine.Engine(H, W, d)           # the same device twice: a second context (closed below)
                        own.append(e)
                    else:
                        e = _engine.get_engine(H, W, d)
                    engines.append(e)
                flags = 0
                for i, e in enumerate(engines):               # calibration goes to every device once
                    with contextlib.nullcontext() if (verbose and i == 0) else contextlib.redirect_stdout(io.StringIO()):
                        flags = self._configure_engine(e, (H, W), bgImages, exposure_time, light_spectrum, date,
                                                       use_dark=bg_frames is None)
                    lo, hi = sharding.shard_range(n, len(engines), i)
                    self._set_exposures(e, None if times is None else times[lo:hi])
                try:
                    lens = self.getLens(light_spectrum, date['lens'])
                    if lens:
                        lens._lens_setup(W, H)
                        for e in engines:
                            e.set_lens(lens.coeffs['cameraMatrix'], lens.coeffs['distortionCoeffs'], lens._new_camera_matrix)
                except _lib.ImgcorrError:
                    raise
                except Exception as errm:
                    print('Error: %s' % errm)
                    lens = None
            if threshold > 0:
                flags |= _lib.DO_NAN_TO_NUM
            if stage is not None:
                for i, e in enumerate(engines):
                    lo, hi = sharding.shard_range(n, len(engines), i)
                    if np.ndim(stage[0]) == 3:                # a per-frame table: the matrices of this engine's shard
                        if hi <= lo:
                            continue
                        self._set_perspective(e, (stage[0][lo:hi],) + tuple(stage[1:]))
                    else:
                        self._set_perspective(e, stage)
                flags |= _lib.DO_PERSPECTIVE
            window = tuple(int(v) for v in lens.roi) if (lens and not keep_size) else None
            oh, ow = engines[0].chain_shape(flags, bool(lens), window)[2]
            odt = np.dtype(out_dtype or np.float32)
            if out is None:
                out = np.empty((n, oh, ow), dtype=odt)
            if out.shape != (n, oh, ow) or not out.flags.c_contiguous:
                raise ValueError('out must be C-contiguous of shape %s' % ((n, oh, ow),))
            thr = threshold if threshold > 0 else 0.0
            errors = [None] * len(engines)

            def work(i):
                lo, hi = sharding.shard_range(n, len(engines), i)
                if hi <= lo:
                    return
                try:
                    engines[i].correct_host(frames[lo:hi], out=out[lo:hi], threshold=thr, ksize=3, flags=flags,
                                            use_lens=bool(lens), window=window, out_dtype=out.dtype, out_scale=out_scale,
                                            bg=None if bg_frames is None else bg_frames[lo:hi])
                except BaseException as e:                    # noqa: BLE001 - re-raised in the caller's thread
                    errors[i] = e

            threads = [threading.Thread(target=work, args=(i,)) for i in range(1, len(engines))]
            for t in threads:
                t.start()
            work(0)
            for t in threads:
                t.join()
            for e in errors:
                if e is not None:
                    raise e
            return out
        finally:
            for e in own:
                e.close()
