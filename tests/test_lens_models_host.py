"""OpenCV's 4-, 8-, 12- and 14-coefficient lens models on the CPU: the numpy reference (tests/lens_ref.py) and the host
build of the core function the K2 kernels evaluate (imgcorr_core.cuh undistort_map_ext) against
cv2.initUndistortRectifyMap, their reduction to the 5-term model, and the refusal of other coefficient counts."""
import sys

import numpy as np
import pytest

import emul
import lens_ref
from oracle import models

cv2 = pytest.importorskip('cv2')

SHAPES = [(3000, 4096), (501, 665)]
LENSES = dict(lens_ref.LENSES, wide=lens_ref.WIDE, fold=lens_ref.FOLD)


def _cv2_maps(d, H, W):
    K = lens_ref.camera(W, H)
    d = np.asarray(d, np.float64)
    P, _ = cv2.getOptimalNewCameraMatrix(K, d, (W, H), 1, (W, H))
    mx, my = cv2.initUndistortRectifyMap(K, d, None, P, (W, H), cv2.CV_32FC1)
    return K, P, mx, my


@pytest.mark.parametrize('shape', SHAPES, ids=['4096x3000', '665x501'])
@pytest.mark.parametrize('name', list(LENSES))
def test_fixed_point_coordinates_equal_cv2(name, shape):
    H, W = shape
    d = LENSES[name]
    K, P, cx, cy = _cv2_maps(d, H, W)
    fx, fy = lens_ref.fixed(cx), lens_ref.fixed(cy)
    mx, my = lens_ref.undistort_map_model(K, d, P, W, H)
    assert np.array_equal(lens_ref.fixed(mx), fx) and np.array_equal(lens_ref.fixed(my), fy)
    ex, ey, ext = lens_ref.emul_maps(K, d, P, H, W)
    assert ext == (len(d) > 5)
    assert np.array_equal(lens_ref.fixed(ex), fx) and np.array_equal(lens_ref.fixed(ey), fy)
    # the float32 maps themselves differ from cv2's in a handful of entries (last float64 bit, see DESIGN.md)
    assert (ex != cx).sum() + (ey != cy).sum() <= 16


@pytest.mark.parametrize('n', [4, 5, 8, 12, 14])
def test_zero_extra_terms_are_the_five_term_model(n):
    """an n-term vector whose terms after k3 are zero: both references and the extended core function give the current
    5-term model's maps bit for bit"""
    H, W = 501, 665
    d5 = np.array([-0.2, 0.05, 1e-3, -1e-3, 0.0 if n == 4 else 0.02])
    d = np.zeros(n)
    d[:min(n, 5)] = d5[:min(n, 5)]
    K, P, _, _ = _cv2_maps(d, H, W)
    ox, oy = models.undistort_map_model(K, d5, P, W, H)
    mx, my = lens_ref.undistort_map_model(K, d, P, W, H)
    assert np.array_equal(mx, ox) and np.array_equal(my, oy)
    e5x, e5y = emul.maps(K, d5, P, H, W)                     # the 5-term core function
    ex, ey, ext = lens_ref.emul_maps(K, d, P, H, W)
    assert not ext
    assert np.array_equal(ex, e5x) and np.array_equal(ey, e5y)
    fx, fy, ext = lens_ref.emul_maps(K, d, P, H, W, force_ext=True)
    assert ext
    assert np.array_equal(fx, e5x) and np.array_equal(fy, e5y)


def test_tilt_matrix():
    t = lens_ref.emul_tilt(0.01, -0.008)
    assert np.allclose(t, lens_ref.tilt_matrix(0.01, -0.008), rtol=0, atol=1e-15)
    assert np.array_equal(lens_ref.emul_tilt(0.0, 0.0), np.eye(3))


@pytest.mark.parametrize('n', [0, 3, 6, 7, 9, 13, 15])
def test_lens_setup_refuses_other_counts_before_an_engine_exists(n, monkeypatch):
    from imgprocessor_b200 import engine
    from imgprocessor_b200.camera import LensDistortion

    def no_engine(*a, **k):
        raise AssertionError('an engine was requested')
    monkeypatch.setattr(engine, 'get_engine', no_engine)
    monkeypatch.setitem(sys.modules, 'cv2', None)            # `import cv2` fails: cv2 must not be reached either
    lens = LensDistortion({'cameraMatrix': lens_ref.camera(64, 48), 'distortionCoeffs': np.full((1, n), 1e-3)})
    with pytest.raises(ValueError, match='4, 5, 8, 12 or 14'):
        lens._lens_setup(64, 48)


@pytest.mark.parametrize('n', [4, 5, 8, 12, 14])
@pytest.mark.parametrize('layout', ['row', 'flat', 'column'])
def test_lens_setup_accepts_model_counts(n, layout, monkeypatch):
    """every model count and coefficient layout reaches cv2 and the engine with the coefficients in OpenCV's order"""
    from imgprocessor_b200 import engine
    from imgprocessor_b200.camera import LensDistortion
    d = np.arange(1, n + 1) * 1e-3
    d = {'row': d[None, :], 'flat': d, 'column': d[:, None]}[layout]
    seen = {}

    class Eng:
        def set_lens(self, K, dist, P):
            seen['dist'] = np.asarray(dist, np.float64).ravel()
    monkeypatch.setattr(engine, 'get_engine', lambda h, w: Eng())
    lens = LensDistortion({'cameraMatrix': lens_ref.camera(64, 48), 'distortionCoeffs': d})
    lens._lens_setup(64, 48)
    assert np.array_equal(seen['dist'], np.arange(1, n + 1) * 1e-3)
    assert len(lens.roi) == 4
