"""CameraCalibration.correct_batch(bg_frames=...) refuses backgrounds it cannot pair with the frames with ValueError, before
any device or engine is involved: another shape, bgImages given as well, a numpy / tensor mismatch with the frames, and
(for tensor frames) a tensor on another device."""
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


def _frames():
    return np.zeros((N, H, W), np.uint16)


@pytest.mark.parametrize('shape', [(N - 1, H, W), (N, H, W + 1), (H, W)])
def test_wrong_shape(no_engine, shape):
    with pytest.raises(ValueError, match='bg_frames of shape'):
        CameraCalibration().correct_batch(_frames(), bg_frames=np.zeros(shape, np.uint16))


def test_wrong_shape_on_several_devices(no_engine):
    with pytest.raises(ValueError, match='bg_frames of shape'):
        CameraCalibration().correct_batch(_frames(), bg_frames=np.zeros((N + 1, H, W), np.uint16), devices=[0, 0])


def test_with_bgImages(no_engine):
    with pytest.raises(ValueError, match='bg_frames and bgImages'):
        CameraCalibration().correct_batch(_frames(), bgImages=np.zeros((H, W)), bg_frames=np.zeros((N, H, W), np.uint16))


def test_tensor_for_host_frames(no_engine):
    with pytest.raises(ValueError, match='numpy array for host frames'):
        CameraCalibration().correct_batch(_frames(), bg_frames=torch.zeros((N, H, W), dtype=torch.uint16))


def test_numpy_for_tensor_frames(no_engine):
    """a CPU tensor stands in for device frames: the pairing is refused before the device is looked at"""
    with pytest.raises(ValueError, match='CUDA tensor for tensor frames'):
        CameraCalibration().correct_batch(torch.zeros((N, H, W), dtype=torch.uint16), bg_frames=_frames())


def test_tensor_on_another_device(no_engine):
    frames = torch.zeros((N, H, W), dtype=torch.uint16)          # not on a CUDA device either: refused as well
    with pytest.raises(ValueError, match='bg_frames on cpu'):
        CameraCalibration().correct_batch(frames, bg_frames=torch.zeros((N, H, W), dtype=torch.uint16))


def test_background_dtypes():
    """the frames' dtype and float32 stay; others (float64, uint16 for uint8 frames) become float32; a big-endian array is
    swapped to native order"""
    bg16 = np.arange(N * H * W, dtype=np.uint16).reshape(N, H, W)
    assert CameraCalibration._bg_dtype(bg16, np.dtype(np.uint16)) is bg16
    assert CameraCalibration._bg_dtype(bg16, np.dtype(np.uint8)).dtype == np.float32
    assert CameraCalibration._bg_dtype(bg16.astype(np.float64), np.dtype(np.uint16)).dtype == np.float32
    be = CameraCalibration._bg_dtype(bg16.astype('>u2'), np.dtype(np.uint16))
    assert be.dtype == np.dtype('=u2') and np.array_equal(be, bg16)
