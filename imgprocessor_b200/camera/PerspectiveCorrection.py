"""PerspectiveCorrection: drop-in for the warp half of
imgProcessor.camera.PerspectiveCorrection.PerspectiveCorrection (camera/PerspectiveCorrection.py:38-406),
the step after lens correction in the EL workflow (SURVEY §8 row f3).

What moved to the GPU (kernel K3, csrc/k3_warp.cu), bit-exact with OpenCV's arithmetic:
  * correct()     :380-406   [img / tiltFactor in float64, then] cv2.warpPerspective(..., INTER_LANCZOS4)
  * uncorrect()   :374-378   cv2.warpPerspective(..., INTER_CUBIC | WARP_INVERSE_MAP)
What stays on the host exactly as in the reference: the 3x3 homography of a quad
(cv2.getPerspectiveTransform, :147-149), corner sorting (utils/sortCorners.py), correctPoints (:408-413).
Not reproduced (they need the absent `fancytools` / `transforms3d` packages or the proprietary
PROimgProcessor fallback, :8-30): reference-IMAGE homographies through PatternRecognition, pose
estimation and the tilt-factor MODEL (tiltFactor(), :514-540).  `do_correctIntensity=True` therefore needs
the factor map handed in with setTiltFactor(); the division and the warp then run on the GPU.
"""
import numpy as np

from .. import engine as _engine
from ..imgIO import imread

BL_ANGLE = 2.356194490192345  # = 135 degrees (utils/sortCorners.py:5)


def sortCorners(corners):
    """utils/sortCorners.py:8-47: order the corners of a quadrilateral counter-clockwise along its convex hull
    (clockwise on an image, where y grows downwards), starting with the one towards (-x, -y) of the centroid.
    The reference walks scipy's ConvexHull vertices; for four points that is the counter-clockwise angular
    order around an interior point, computed here directly."""
    corners = np.asarray(corners)
    if corners.shape != (4, 2):
        raise ValueError('a quad is four (x, y) points')
    c = corners.astype(float)

    def cross(o, a, b):
        return (a[0] - o[0]) * (b[1] - o[1]) - (a[1] - o[1]) * (b[0] - o[0])

    # a point inside the triangle of the other three is not a hull vertex; the reference then guesses a position
    # from ConvexHull's data-dependent start vertex (sortCorners.py:20-39) -- refused here
    for i in range(4):
        a, b, d = [c[j] for j in range(4) if j != i]
        s = (cross(a, b, c[i]), cross(b, d, c[i]), cross(d, a, c[i]))
        if all(v >= 0 for v in s) or all(v <= 0 for v in s):
            raise ValueError('quad is not convex')
    mid = c.mean(axis=0)
    ang = np.arctan2(c[:, 1] - mid[1], c[:, 0] - mid[0])
    corners2 = corners[np.argsort(ang, kind='stable')]
    mn = corners2.mean(axis=0)
    d = corners2 - mn
    ascent = np.arctan2(d[:, 1], d[:, 0])
    bl = int(np.abs(BL_ANGLE + ascent).argmin())
    i = list(range(bl, 4)) + list(range(0, bl))
    return corners2[i]


def genericCameraMatrix(shape, angularField=60):
    """utils/genericCameraMatrix.py:7-29"""
    cy = int(shape[0] / 2)
    cx = int(shape[1] / 2)
    fx = fy = cx / np.tan(angularField / 2 * np.pi / 180)
    return np.array([[fx, 0, cx], [0, fy, cy], [0, 0, 1]], dtype=np.float32)


class PerspectiveCorrection(object):

    def __init__(self, img_shape, cameraMatrix=None, distCoeffs=np.zeros((5, 1)), do_correctIntensity=False,
                 px_per_phys_unit=None, new_size=(None, None), in_plane=False, border=0, maxShear=0.05,
                 material='EL_Si_module', cv2_opts={}):
        self.opts = {'distCoeffs': distCoeffs.astype(np.float32),
                     'do_correctIntensity': do_correctIntensity,
                     'new_size': new_size,
                     'in_plane': in_plane,
                     'cv2_opts': cv2_opts,
                     'border': border,
                     'material': material,
                     'maxShear': maxShear,
                     'shape': img_shape[:2]}
        if cameraMatrix is None:
            cameraMatrix = genericCameraMatrix(img_shape)
        self.opts['cameraMatrix'] = cameraMatrix.astype(np.float32)
        self.refQuad = None
        self._obj_points = None
        self.px_per_phys_unit = px_per_phys_unit
        self._newBorders = self.opts['new_size']
        self._tilt_factor = None
        self.quad = None
        self._homography = None
        self._homography_is_fixed = True

    def setReferenceQuad(self, refQuad):
        self.refQuad = sortCorners(refQuad)

    def setTiltFactor(self, factor):
        """the map correct() divides by when do_correctIntensity is set (what tiltFactor() returns, :514-540)"""
        self._tilt_factor = None if factor is None else np.asarray(factor, np.float64)

    def tiltFactor(self, midpointdepth=None, printAvAngle=False):
        if self._tilt_factor is None:
            raise NotImplementedError('the tilt-factor model needs pose estimation through the absent fancytools / '
                                      'transforms3d packages; pass the factor map with setTiltFactor()')
        return self._tilt_factor

    def setReference(self, ref):
        """ref: 3x3 homography, or the four (x, y) image points of the quad to rectify (:98-133)."""
        self.quad = None
        self._camera_position = None
        self._homography = None
        self._homography_is_fixed = True
        self._pose = None
        if isinstance(ref, np.ndarray) and ref.shape == (3, 3):
            self._homography = ref
        elif len(ref) == 4:
            self.quad = sortCorners(ref)
            self.obj_points
        else:
            raise NotImplementedError('a reference IMAGE needs PatternRecognition (outside the GPU path); pass the '
                                      'homography or the quad')

    @property
    def obj_points(self):
        """:720-759 for a fully specified new_size"""
        if self._obj_points is None:
            sy, sx = self.opts['new_size']
            if sx is None or sy is None:
                raise NotImplementedError('new_size with None needs calcAspectRatioFromCorners (fancytools); give '
                                          'both sizes')
            self._obj_points = np.float32([[0, 0, 0], [sx, 0, 0], [sx, sy, 0], [0, sy, 0]])
        return self._obj_points

    @property
    def homography(self):
        if self._homography is None:
            import cv2
            b = self.opts['border']
            if self.quad is None:
                raise NotImplementedError('no quad and no homography set')
            if self.refQuad is not None:
                dst = self.refQuad.astype(np.float32)
            else:
                sy, sx = self._newBorders
                dst = np.float32([[b, b], [sx - b, b], [sx - b, sy - b], [b, sy - b]])
            self._homography = cv2.getPerspectiveTransform(self.quad.astype(np.float32), dst)
        return self._homography

    # ------------------------------------------------------------------ GPU part
    @staticmethod
    def _cv2_opts(opts):
        unknown = set(opts) - {'borderValue', 'borderMode'}
        if unknown:
            raise NotImplementedError('cv2_opts %s' % sorted(unknown))
        if opts.get('borderMode', 0) != 0:
            raise NotImplementedError('only BORDER_CONSTANT')
        bv = opts.get('borderValue', 0.0)
        return float(bv[0] if np.ndim(bv) else bv)

    def _warp(self, img, dsize, interpolation, inverse_map, border_value, divide_by=None):
        tt = _engine.torch()
        is_tensor = isinstance(img, tt.Tensor)
        if img.ndim != 2:
            raise ValueError('PerspectiveCorrection: single-channel 2-D frames only on the GPU path')
        h, w = img.shape
        eng = _engine.get_engine(h, w)
        if not is_tensor:
            if img.dtype.type not in (np.uint8, np.uint16, np.float32, np.float64):
                raise TypeError('unsupported image dtype %s (uint8, uint16, float32, float64)' % img.dtype)
            img = tt.from_numpy(np.ascontiguousarray(img)).to(eng.device)
        if divide_by is not None:
            divide_by = tt.from_numpy(np.ascontiguousarray(divide_by, np.float64))
        out = eng.warp_perspective(img, self.homography, dsize, interpolation, inverse_map, border_value, divide_by)
        return out if is_tensor else _engine.to_numpy(out)

    def correct_params(self):
        """(homography, dsize (width, height), border value, tilt factor or None) of correct(): the warp
        cv2.warpPerspective(img [/ tilt factor], homography, dsize, INTER_LANCZOS4, BORDER_CONSTANT, border value).
        CameraCalibration.correct_batch(perspective=...) runs the same warp as the chain's last stage."""
        if not self._homography_is_fixed:
            self._homography = None
        M = self.homography
        if None in tuple(self._newBorders):
            raise NotImplementedError('new_size must be given')
        tf = self.tiltFactor() if self.opts['do_correctIntensity'] else None
        return M, tuple(self._newBorders[::-1]), self._cv2_opts(self.opts['cv2_opts']), tf

    def correct(self, img):
        """perspective transformation [after the tilt-factor division] (:380-406)"""
        print("CORRECT PERSPECTIVE ...")
        self.img = imread(img)
        _, dsize, border_value, tf = self.correct_params()
        return self._warp(self.img, dsize, 'lanczos4', False, border_value, tf)

    def uncorrect(self, img):
        """:374-378"""
        img = imread(img)
        s = img.shape[:2]
        return self._warp(img, s[::-1], 'cubic', True, 0.0)

    def correctPoints(self, pts):
        import cv2
        if not self._homography_is_fixed:
            self._homography = None
        h = self._homography
        if pts.ndim == 2:
            pts = pts.reshape(1, *pts.shape)
        return cv2.perspectiveTransform(pts.astype(np.float32), h)

    @property
    def areaRatio(self):
        """:542-555 for a quad reference"""
        if self.quad is None:
            raise NotImplementedError('areaRatio without a quad needs the pattern homography')
        q = self.quad
        quad_size = 0.5 * abs((q[2, 0] - q[0, 0]) * (q[3, 1] - q[1, 1]) + (q[3, 0] - q[1, 0]) * (q[0, 1] - q[2, 1]))
        sx, sy = self._newBorders
        return (sx * sy) / quad_size
