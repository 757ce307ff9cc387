"""CameraCalibration.correct_batch(exposure_time=[...]) refuses per-frame exposure times it cannot use with ValueError, before
any device or engine is involved: another length than the frames, a sequence that is not 1-D, non-numeric values and NaN.
A scalar and None are not per-frame times."""
import time

import numpy as np
import pytest

torch = pytest.importorskip('torch')

from imgprocessor_b200.camera import CameraCalibration  # noqa: E402

H, W, N = 24, 40, 3


@pytest.fixture
def no_engine(monkeypatch):
    """fails the test if correct_batch gets as far as creating an engine"""
    from imgprocessor_b200 import engine

    def refuse(*a, **k):
        raise AssertionError('an engine was requested before the refusal')
    monkeypatch.setattr(engine, 'get_engine', refuse)
    monkeypatch.setattr(engine, 'Engine', refuse)


def _cal():
    """a calibration with a tuple dark-current entry (offset, ascent): the line model"""
    cal = CameraCalibration()
    cal.coeffs['dark current'].append((time.localtime(), '', (np.full((H, W), 0.5), np.full((H, W), 10.0)), None))
    return cal


def _frames():
    return np.zeros((N, H, W), np.uint16)


@pytest.mark.parametrize('times', [[1.0] * (N - 1), [1.0] * (N + 1), []])
def test_wrong_length(no_engine, times):
    with pytest.raises(ValueError, match='times for %d frames' % N):
        _cal().correct_batch(_frames(), exposure_time=times)


def test_wrong_length_on_several_devices(no_engine):
    with pytest.raises(ValueError, match='times for %d frames' % N):
        _cal().correct_batch(_frames(), exposure_time=np.ones(N + 1), devices=[0, 0])


def test_wrong_length_for_tensor_frames(no_engine):
    """a CPU tensor stands in for device frames: the times are refused before the device is looked at"""
    with pytest.raises(ValueError, match='times for %d frames' % N):
        _cal().correct_batch(torch.zeros((N, H, W), dtype=torch.uint16), exposure_time=torch.ones(N - 1))


@pytest.mark.parametrize('times', [np.ones((N, 1)), np.ones((1, N)), [[1.0, 2.0, 3.0]]])
def test_not_1d(no_engine, times):
    with pytest.raises(ValueError, match='1-D sequence'):
        _cal().correct_batch(_frames(), exposure_time=times)


@pytest.mark.parametrize('times', [['1', '2', '3'], [1.0, None, 2.0], [1.0, 'a', 2.0], [1 + 1j] * N, [True] * N])
def test_not_numeric(no_engine, times):
    with pytest.raises(ValueError):
        _cal().correct_batch(_frames(), exposure_time=times)


def test_nan(no_engine):
    with pytest.raises(ValueError, match=r'exposure_time\[1\] is NaN'):
        _cal().correct_batch(_frames(), exposure_time=[1.0, float('nan'), 2.0])


def test_nan_with_array_entry(no_engine):
    """an array dark entry does not use the times, but they are checked all the same"""
    cal = CameraCalibration()
    cal.addDarkCurrent(np.zeros((H, W)))
    with pytest.raises(ValueError, match='NaN'):
        cal.correct_batch(_frames(), exposure_time=[1.0, float('nan'), 2.0])


def test_nan_with_bg_frames(no_engine):
    with pytest.raises(ValueError, match='NaN'):
        _cal().correct_batch(_frames(), exposure_time=[float('nan')] * N, bg_frames=np.zeros((N, H, W), np.uint16))


def test_times_as_float64():
    """integers, float32 and tensors become float64 times; infinities and negative times are times"""
    t = CameraCalibration._exposure_times(np.array([1, 2, 3], np.int32), 3)
    assert t.dtype == np.float64 and list(t) == [1.0, 2.0, 3.0]
    t = CameraCalibration._exposure_times(torch.tensor([0.5, -1.0, float('inf')]), 3)
    assert t.dtype == np.float64 and list(t) == [0.5, -1.0, float('inf')]
    t = CameraCalibration._exposure_times((0.1, 0.2), 2)
    assert list(t) == [0.1, 0.2]


@pytest.mark.parametrize('scalar', [None, 0.0, 3, np.float32(2.5), np.array(1.5)])
def test_scalar_is_not_per_frame(scalar):
    assert CameraCalibration._exposure_times(scalar, N) is None
