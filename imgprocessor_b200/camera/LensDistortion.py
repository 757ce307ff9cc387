"""LensDistortion: drop-in for imgProcessor.camera.LensDistortion.LensDistortion
(camera/LensDistortion.py:16-402).

What moved to the GPU (kernel K2, csrc/k2_undistort.cu):
  * correct()                  :316-330   analytic lens map (OpenCV's 4-, 5-, 8-, 12- and 14-coefficient models)
                                          + OpenCV fixed-point bilinear remap
  * getUndistortRectifyMap()   :342-358   the float32 maps themselves (written by a map kernel)
  * distortImage()             :332-340   remap with explicit maps
What stays on the host, exactly as in the reference: cv2.getOptimalNewCameraMatrix (a 3x3, :350-353)
and the calibration half (pattern detection + cv2.calibrateCamera, :35-252) — calibration-time code,
not per-frame.
"""
from collections import OrderedDict

import numpy as np

from .. import engine as _engine
from ..imgIO import imread


class NothingFound(Exception):
    pass


class EnoughImages(Exception):
    pass


def _as_device_frame(eng, image):
    tt = _engine.torch()
    if isinstance(image, tt.Tensor):
        return image, True
    return tt.from_numpy(np.ascontiguousarray(image)).to(eng.device), False


class LensDistortion(object):
    ftype = 'npz'

    def __init__(self, coeffs=None):
        # the reference's default argument is a shared mutable dict (:26); a fresh one is the
        # behaviour callers rely on
        self._coeffs = {} if coeffs is None else coeffs
        self.opts = {}
        self.mapx, self.mapy = None, None
        self.roi = None
        self.findCount = 0
        self._new_camera_matrix = None

    # ------------------------------------------------------------------ parameters (:360-380)
    def setCameraParams(self, fx, fy, cx, cy, k1, k2, k3, p1, p2):
        cam = np.zeros((3, 3))
        cam[0, 0], cam[1, 1], cam[0, 2], cam[1, 2], cam[2, 2] = fx, fy, cx, cy, 1
        self._coeffs['cameraMatrix'] = cam
        self._coeffs['distortionCoeffs'] = np.array([[k1, k2, p1, p2, k3]])
        self.mapx = self.mapy = None

    def getCameraParams(self):
        cam = self.coeffs['cameraMatrix']
        k1, k2, p1, p2, k3 = tuple(np.asarray(self.coeffs['distortionCoeffs']).tolist()[0])
        return cam[0][0], cam[1][1], cam[0][2], cam[1][2], k1, k2, k3, p1, p2

    @property
    def coeffs(self):
        if not self._coeffs:
            self._coeffs = self._calibrate_from_points()
        return self._coeffs

    @coeffs.setter
    def coeffs(self, c):
        self._coeffs = c

    def getCoeffStr(self):
        return ''.join('%s = %s\n' % kv for kv in self.coeffs.items())

    # ------------------------------------------------------------------ the hot path
    def _lens_setup(self, imgWidth, imgHeight):
        """host part of getUndistortRectifyMap (:347-353): P and roi from OpenCV, then the lens
        constants go to the device context."""
        cam = np.asarray(self.coeffs['cameraMatrix'], np.float64)
        d = np.asarray(self.coeffs['distortionCoeffs'], np.float64)
        if d.size not in _engine.LENS_MODEL_SIZES:      # what cv2.initUndistortRectifyMap takes
            raise ValueError('distortionCoeffs: 4, 5, 8, 12 or 14 terms (k1 k2 p1 p2 k3 k4 k5 k6 s1 s2 s3 s4 tau_x tau_y), '
                             'got %d' % d.size)
        import cv2
        P, self.roi = cv2.getOptimalNewCameraMatrix(cam, d, (imgWidth, imgHeight), 1, (imgWidth, imgHeight))
        self._new_camera_matrix = P
        eng = _engine.get_engine(imgHeight, imgWidth)
        eng.set_lens(cam, d, P)
        return eng

    def getUndistortRectifyMap(self, imgWidth, imgHeight):
        if self.mapx is not None and self.mapx.shape == (imgHeight, imgWidth):
            return self.mapx, self.mapy
        eng = self._lens_setup(imgWidth, imgHeight)
        mx, my = eng.undistort_maps()
        self.mapx, self.mapy = mx.cpu().numpy(), my.cpu().numpy()
        return self.mapx, self.mapy

    def correct(self, image, keepSize=False, borderValue=0):
        """remove lens distortion from ``image`` (path, callable, 2-D numpy array of uint8 / uint16 /
        float32 / float64 — dtype preserved — or a CUDA torch tensor, which stays on the device)."""
        image = imread(image)
        tt = _engine.torch()
        is_tensor = isinstance(image, tt.Tensor)
        if image.ndim != 2:
            raise ValueError('LensDistortion.correct: single-channel 2-D frames only on the GPU path')
        h, w = image.shape[:2]
        eng = self._lens_setup(w, h)
        if not is_tensor and image.dtype.type not in (np.uint8, np.uint16, np.float32, np.float64):
            raise TypeError('unsupported image dtype %s (uint8, uint16, float32, float64)' % image.dtype)
        dev, _ = _as_device_frame(eng, image)
        window = None if keepSize else tuple(int(v) for v in self.roi)
        out = eng.undistort(dev, border_value=float(borderValue), window=window)
        self.img = out if is_tensor else _engine.to_numpy(out)
        return self.img

    def distortImage(self, image):
        """opposite of correct() (:332-340)."""
        image = imread(image)
        h, w = image.shape[:2]
        mapx, mapy = self.getDistortRectifyMap(w, h)
        eng = _engine.get_engine(h, w)
        tt = _engine.torch()
        dev, is_tensor = _as_device_frame(eng, image)
        out = eng.remap(dev, tt.from_numpy(mapx), tt.from_numpy(mapy), 0.0)
        return out if is_tensor else _engine.to_numpy(out)

    # ------------------------------------------------------------------ map-derived helpers (:382-418)
    def getDistortRectifyMap(self, sizex, sizey):
        posy, posx = np.mgrid[0:sizey, 0:sizex].astype(np.float32)
        mapx, mapy = self.getUndistortRectifyMap(sizex, sizey)
        posx += posx - mapx
        posy += posy - mapy
        return posx, posy

    def getShift(self, width, height):
        mapx, mapy = self.getUndistortRectifyMap(width, height)
        posy, posx = np.mgrid[0:height, 0:width].astype(np.float32)
        return ((mapx - posx) ** 2 + (mapy - posy) ** 2) ** 0.5

    def getDeflection(self, width, height):
        mapx, mapy = self.getUndistortRectifyMap(width, height)
        return 1 / np.abs(np.gradient(mapx)[1]), 1 / np.abs(np.gradient(mapy)[0])

    def standardUncertainties(self, sharpness=0.5):
        height, width = self.coeffs['shape']
        fx, fy = self.getDeflection(width, height)
        t = (sharpness ** 2 + self.coeffs['reprojectionError'] ** 2) ** 0.5
        return fx * t, fy * t

    def undistortPoints(self, points, keepSize=False):
        import cv2
        s = self.img.shape
        cam, d = self.coeffs['cameraMatrix'], self.coeffs['distortionCoeffs']
        pts = np.asarray(points, dtype=np.float32)
        if pts.ndim == 2:
            pts = pts[None]
        P, roi = cv2.getOptimalNewCameraMatrix(cam, d, s[::-1], 1, s[::-1])
        if not keepSize:
            pts[0, 0] -= roi[0]
            pts[0, 1] -= roi[1]
        return cv2.undistortPoints(pts, cam, d, P=P)

    # ------------------------------------------------------------------ persistence (:258-291)
    def writeToFile(self, filename, saveOpts=False):
        if not filename.endswith('.' + self.ftype):
            filename += '.' + self.ftype
        payload = {'coeffs': self.coeffs}
        if saveOpts:
            payload['opts'] = self.opts
        np.savez(filename, **payload)
        return filename

    def readFromFile(self, filename):
        s = dict(np.load(filename, allow_pickle=True))
        try:
            self.coeffs = s['coeffs'][()]
        except KeyError:
            self.coeffs = s
        try:
            self.opts = s['opts'][()]
        except KeyError:
            pass
        self.mapx = self.mapy = None
        return self.coeffs

    # ------------------------------------------------------------------ calibration, host / OpenCV (:35-252)
    def calibrate(self, board_size=(8, 6), method='Chessboard', images=(), max_images=100, sensorSize_mm=None,
                  detect_sensible=True):
        finders = {'Chessboard': self._findChessboard, 'Symmetric circles': self._findSymmetricCircles,
                   'Asymmetric circles': self._findAsymmetricCircles, 'Manual': None}
        self._coeffs = {}
        self.opts = {'foundPattern': [], 'size': board_size, 'imgs': [], 'imgPoints': []}
        self._detect_sensible = detect_sensible
        self.method = finders[method]
        self.max_images = max_images
        self.findCount = 0
        self.apertureSize = sensorSize_mm
        self.objp = self._mkObjPoints(board_size)
        if method == 'Asymmetric circles':
            odd = self.objp[:, 1] % 2 == 1
            self.objp[:, 0] *= 2
            self.objp[odd, 0] += 1
        self.objpoints = []
        self.mapx = self.mapy = None
        for n, im in enumerate(images):
            print('working on image %s' % n)
            if self.addImg(im):
                print('OK')

    @staticmethod
    def _mkObjPoints(board_size):
        s0, s1 = board_size
        o = np.zeros((s0 * s1, 3), np.float32)
        o[:, :2] = np.mgrid[0:s0, 0:s1].T.reshape(-1, 2)
        return o

    def addPoints(self, points, board_size=None):
        self.opts['foundPattern'].append(True)
        self.findCount += 1
        self.objpoints.append(self.objp if board_size is None else self._mkObjPoints(board_size))
        pts = np.asarray(points)
        self.opts['imgPoints'].append(pts.reshape(pts.shape[0], 1, 2).astype(np.float32))

    def setImgShape(self, shape):
        self.img = type('Dummy', (object,), {})
        self.img.shape = shape

    def addImgStream(self, img):
        if self.findCount > self.max_images:
            raise EnoughImages('have enough images')
        return self.addImg(img)

    def addImg(self, img):
        self.img = imread(img, 'gray', 'uint8')
        found, corners = self.method()
        self.opts['foundPattern'].append(found)
        if found:
            self.findCount += 1
            self.objpoints.append(self.objp)
            self.opts['imgPoints'].append(corners)
        return found

    def _findChessboard(self):
        import cv2
        flags = cv2.CALIB_CB_FAST_CHECK
        if self._detect_sensible:
            flags |= cv2.CALIB_CB_ADAPTIVE_THRESH | cv2.CALIB_CB_FILTER_QUADS | cv2.CALIB_CB_NORMALIZE_IMAGE
        found, corners = cv2.findChessboardCorners(self.img, self.opts['size'], flags=flags)
        if found:
            cv2.cornerSubPix(self.img, corners, (11, 11), (-1, -1),
                             (cv2.TERM_CRITERIA_EPS + cv2.TERM_CRITERIA_MAX_ITER, 30, 0.001))
        return found, corners

    def _findAsymmetricCircles(self):
        import cv2
        return self._findSymmetricCircles(flags=cv2.CALIB_CB_ASYMMETRIC_GRID)

    def _findSymmetricCircles(self, flags=None):
        import cv2
        if flags is None:
            flags = cv2.CALIB_CB_SYMMETRIC_GRID
        return cv2.findCirclesGrid(self.img, self.opts['size'], flags=flags | cv2.CALIB_CB_CLUSTERING)

    def _calibrate_from_points(self):
        import cv2
        if not self.findCount:
            raise NothingFound('can create camera calibration because no corners have been found')
        try:
            err, cam, dist, _, _ = cv2.calibrateCamera(self.objpoints, self.opts['imgPoints'], self.img.shape[::-1],
                                                       None, None)
            print('reprojectionError=%s' % err)
        except Exception as e:
            raise NothingFound(e)
        c = OrderedDict([('reprojectionError', err), ('apertureSize', self.apertureSize), ('cameraMatrix', cam),
                         ('distortionCoeffs', dist), ('shape', self.img.shape)])
        if self.apertureSize is not None:
            fovx, fovy, fl, pp, ar = cv2.calibrationMatrixValues(cam, self.img.shape, *self.apertureSize)
            c.update(OrderedDict([('fovx', fovx), ('fovy', fovy), ('focalLength', fl), ('principalPoint', pp),
                                  ('aspectRatio', ar)]))
        return c

    def drawChessboard(self, img=None):
        import cv2
        assert self.findCount > 0, 'cannot draw chessboard if nothing found'
        if img is None:
            img = self.img
        elif isinstance(img, bool) and not img:
            img = np.zeros(shape=self.img.shape, dtype=self.img.dtype)
        else:
            img = imread(img, dtype='uint8')
        gray = img.ndim == 2
        if gray:
            img = cv2.cvtColor(img, cv2.COLOR_GRAY2BGR)
        cv2.drawChessboardCorners(img, self.opts['size'], self.opts['imgPoints'][-1], self.opts['foundPattern'][-1])
        return cv2.cvtColor(img, cv2.COLOR_BGR2GRAY) if gray else img
