"""References for OpenCV's full lens distortion model (4, 5, 8, 12 or 14 coefficients) in K2:

* undistort_map_model: float64 numpy evaluation of cv2.initUndistortRectifyMap(K, dist, None, P, size, CV_32FC1),
  oracle.models.undistort_map_model generalised to the rational, thin-prism and tilted-sensor terms;
* emul_maps: the core function the kernels call (imgcorr_core.cuh, undistort_map_ext), compiled with g++ from
  tests/host_emul/lens_emul.cpp;
* the test lenses shared by the CPU and the GPU tests."""
import ctypes
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, 'host_emul', 'lens_emul.cpp')
CORE = os.path.join(os.path.dirname(HERE), 'imgprocessor_b200', 'csrc', 'imgcorr_core.cuh')
OUT = os.path.join(HERE, '_build', 'libimgcorr_lens_emul.so')

# coefficients in OpenCV's order k1 k2 p1 p2 k3 k4 k5 k6 s1 s2 s3 s4 tau_x tau_y
_R8 = [-0.25, 0.06, 1e-3, -1e-3, -0.01, 0.05, 0.01, -0.004]
LENSES = {
    'moderate5': [-0.2, 0.05, 1e-3, -1e-3, 0.0],
    'four': [-0.2, 0.05, 1e-3, -1e-3],
    'rational8': _R8,
    'prism12': _R8 + [1e-3, -2e-4, 5e-4, 1e-4],
    'tilted14': _R8 + [1e-3, -2e-4, 5e-4, 1e-4, 0.01, -0.008],
}
# a strong wide-angle lens: shifts of up to 497 pixels at 4096x3000; its tiles need 104x48-pixel source windows, which
# sends K2 to the 112x48 staged boxes
WIDE = [-0.6, 0.3, 1e-3, -1e-3, -0.1, -0.2, 0.2, 0.02, 2e-3, -1e-3, 1e-3, 5e-4, 0.02, -0.015]
# a lens whose map folds over beyond the image (the distortion polynomial turns back): windows of hundreds of pixels,
# no staged box holds them, and K2's tiles take the all-slow path.  cv2 defines the map all the same.
FOLD = [-0.8, 0.5, 1e-3, -1e-3, -0.15, -0.2, 0.3, 0.03, 2e-3, -1e-3, 1e-3, 5e-4, 0.02, -0.015]


def camera(W, H):
    return np.array([[W, 0, W / 2.0], [0, W, H / 2.0], [0, 0, 1.0]])


def tilt_matrix(tau_x, tau_y):
    """cv::detail::computeTiltProjectionMatrix"""
    cx, sx, cy, sy = np.cos(tau_x), np.sin(tau_x), np.cos(tau_y), np.sin(tau_y)
    rx = np.array([[1, 0, 0], [0, cx, sx], [0, -sx, cx]])
    ry = np.array([[cy, 0, -sy], [0, 1, 0], [sy, 0, cy]])
    rxy = ry @ rx
    pz = np.array([[rxy[2, 2], 0, -rxy[0, 2]], [0, rxy[2, 2], -rxy[1, 2]], [0, 0, 1]])
    return pz @ rxy


def undistort_map_model(K, dist, P, width, height, T=None):
    """float32 (mapx, mapy) of cv2.initUndistortRectifyMap(K, dist, None, P, (width, height), CV_32FC1), R = I:

        [X Y W]^T = P^-1 [u v 1]^T ; x = X/W ; y = Y/W ; r2 = x^2 + y^2
        kr = (1 + ((k3 r2 + k2) r2 + k1) r2) / (1 + ((k6 r2 + k5) r2 + k4) r2)
        xd = x kr + p1 2xy + p2 (r2 + 2x^2) + s1 r2 + s2 r2^2 ; yd = y kr + p1 (r2 + 2y^2) + p2 2xy + s3 r2 + s4 r2^2
        [tx ty tz]^T = T [xd yd 1]^T ; ip = 1 / tz (1 if tz == 0)
        mapx = fx ip tx + cx ; mapy = fy ip ty + cy

    The 5-term part keeps oracle.models.undistort_map_model's expressions, and every extra term is an addition of a zero,
    a division by one or a product with one when it is zero: for a 4- or 5-term lens the result is that model's bit for bit.
    T defaults to tilt_matrix(tau_x, tau_y)."""
    K = np.asarray(K, np.float64).reshape(3, 3)
    d = np.asarray(dist, np.float64).ravel()
    assert d.size in (4, 5, 8, 12, 14), d.size
    d = np.concatenate([d, np.zeros(14 - d.size)])
    k1, k2, p1, p2, k3, k4, k5, k6, s1, s2, s3, s4, tau_x, tau_y = d
    T = tilt_matrix(tau_x, tau_y) if T is None else np.asarray(T, np.float64).reshape(3, 3)
    ir = np.linalg.inv(np.asarray(P, np.float64).reshape(3, 3)[:, :3])
    u = np.arange(width, dtype=np.float64)[None, :]
    v = np.arange(height, dtype=np.float64)[:, None]
    _x = u * ir[0, 0] + (v * ir[0, 1] + ir[0, 2])
    _y = u * ir[1, 0] + (v * ir[1, 1] + ir[1, 2])
    _w = u * ir[2, 0] + (v * ir[2, 1] + ir[2, 2])
    w = 1.0 / _w
    x = _x * w
    y = _y * w
    x2 = x * x
    y2 = y * y
    r2 = x2 + y2
    _2xy = 2 * x * y
    kr = (1 + ((k3 * r2 + k2) * r2 + k1) * r2) / (1 + ((k6 * r2 + k5) * r2 + k4) * r2)
    xd = x * kr + p1 * _2xy + p2 * (r2 + 2 * x2) + s1 * r2 + s2 * r2 * r2
    yd = y * kr + p1 * (r2 + 2 * y2) + p2 * _2xy + s3 * r2 + s4 * r2 * r2
    tx = T[0, 0] * xd + T[0, 1] * yd + T[0, 2]
    ty = T[1, 0] * xd + T[1, 1] * yd + T[1, 2]
    tz = T[2, 0] * xd + T[2, 1] * yd + T[2, 2]
    with np.errstate(divide='ignore'):
        ip = np.where(tz != 0, 1.0 / tz, 1.0)
    mapx = K[0, 0] * ip * tx + K[0, 2]
    mapy = K[1, 1] * ip * ty + K[1, 2]
    return mapx.astype(np.float32), mapy.astype(np.float32)


def fixed(m):
    """OpenCV remap's 5-bit fixed-point coordinate (cvRound(m * 32)) of a float32 map"""
    return np.rint(np.asarray(m, np.float32) * np.float32(32)).astype(np.int64)


_lib = None


def lib():
    global _lib
    if _lib is None:
        os.makedirs(os.path.dirname(OUT), exist_ok=True)
        if not os.path.exists(OUT) or os.path.getmtime(OUT) < max(os.path.getmtime(SRC), os.path.getmtime(CORE)):
            subprocess.check_call(['g++', '-O2', '-std=c++17', '-ffp-contract=off', '-fPIC', '-shared',
                                   '-fvisibility=hidden', '-o', OUT, SRC, '-lm'])
        _lib = ctypes.CDLL(OUT)
    return _lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def emul_maps(K, dist, P, H, W, force_ext=False):
    """(mapx, mapy, extended) from the core functions; `extended`: the extended model ran (not the 5-term one)"""
    K = np.ascontiguousarray(K, np.float64)
    d = np.ascontiguousarray(np.asarray(dist, np.float64).ravel())
    P = np.ascontiguousarray(np.asarray(P, np.float64)[:, :3])
    mx = np.empty((H, W), np.float32)
    my = np.empty((H, W), np.float32)
    r = lib().emul_maps_ext(_p(K), _p(d), d.size, _p(P), H, W, _p(mx), _p(my), int(bool(force_ext)))
    assert r >= 0
    return mx, my, bool(r)


def emul_tilt(tau_x, tau_y):
    t = np.empty(9, np.float64)
    lib().emul_tilt(ctypes.c_double(tau_x), ctypes.c_double(tau_y), _p(t))
    return t.reshape(3, 3)
