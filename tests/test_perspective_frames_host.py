"""CameraCalibration.correct_batch(perspective=[pc_0, ..., pc_n-1]) refuses a per-frame list it cannot run as one stage
with ValueError, before any device or engine is involved: a length other than the frame count, destination sizes or
border values that differ between the objects, and an object with do_correctIntensity (per-frame tilt factors)."""
import numpy as np
import pytest

pytest.importorskip('torch')

from imgprocessor_b200.camera import CameraCalibration, PerspectiveCorrection  # noqa: E402

H, W, N = 24, 40, 3


def _pcs(n=N, new_size=(20, 36), border=0.0, tilt_at=None):
    out = []
    for i in range(n):
        M = np.array([[1.0, 0.01 * i, 0.5 * i], [0.002 * i, 1.0, -0.25 * i], [1e-5 * i, 0.0, 1.0]])
        pc = PerspectiveCorrection((H, W), new_size=new_size, do_correctIntensity=(i == tilt_at),
                                   cv2_opts={'borderValue': border})
        pc.setReference(M)
        if i == tilt_at:
            pc.setTiltFactor(np.ones((H, W)))
        out.append(pc)
    return out


@pytest.fixture
def no_engine(monkeypatch):
    """fails the test if correct_batch gets as far as creating an engine"""
    from imgprocessor_b200 import engine

    def refuse(*a, **k):
        raise AssertionError('an engine was requested before the refusal')
    monkeypatch.setattr(engine, 'get_engine', refuse)
    monkeypatch.setattr(engine, 'Engine', refuse)


def _call(pcs, **kw):
    frames = np.zeros((N, H, W), np.uint16)
    CameraCalibration().correct_batch(frames, perspective=pcs, **kw)


@pytest.mark.parametrize('n', [0, N - 1, N + 1])
def test_wrong_length(no_engine, n):
    with pytest.raises(ValueError, match='%d PerspectiveCorrection objects for %d frames' % (n, N)):
        _call(_pcs(n))


def test_wrong_length_on_several_devices(no_engine):
    with pytest.raises(ValueError, match='for %d frames' % N):
        _call(_pcs(N + 1), devices=[0, 0])


def test_mixed_dsize(no_engine):
    pcs = _pcs()
    pcs[2] = _pcs(new_size=(21, 36))[2]
    with pytest.raises(ValueError, match=r'perspective\[2\] has dsize'):
        _call(pcs)


def test_mixed_border_value(no_engine):
    pcs = _pcs()
    pcs[1] = _pcs(border=1.5)[1]
    with pytest.raises(ValueError, match=r'perspective\[1\] has dsize .* border value 1.5'):
        _call(pcs)


@pytest.mark.parametrize('out_dtype', [np.float32, np.float64])
def test_tilt_factor(no_engine, out_dtype):
    with pytest.raises(ValueError, match=r'perspective\[1\] has do_correctIntensity'):
        _call(_pcs(tilt_at=1), out_dtype=out_dtype)


def test_consistent_list_is_one_table():
    """the stage a valid list becomes: the homographies stacked in frame order, one dsize and border value, no tilt"""
    pcs = _pcs(border=2.0)
    M, dsize, border, tf = CameraCalibration._perspective_stage(pcs, None, None, N)
    assert M.shape == (N, 3, 3) and M.dtype == np.float64
    for i, pc in enumerate(pcs):
        assert np.array_equal(M[i], pc.homography)
    assert dsize == (36, 20) and border == 2.0 and tf is None
