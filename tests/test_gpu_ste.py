"""SURVEY §8 rows a11 / f1 on the GPU: kernel K4 (csrc/k4_ste.cu) through the C ABI against the STE oracle and the
outputs of the reference's own SingleTimeEffectDetection (tests/golden/ste.npz; MaskedMovingAverage restated — see
oracle/ste.py).  Bar: the float64 average and the STE mask bit-exact; correct() with several exposures within 1e-5 of
full scale of the float64 reference (the average enters the float32 chain)."""
import contextlib
import io

import numpy as np
import pytest

from conftest import load_golden
from oracle import ste

pytestmark = pytest.mark.gpu

torch = pytest.importorskip('torch')


@pytest.fixture(scope='module')
def engine():
    if not torch.cuda.is_available():
        pytest.skip('needs a CUDA device')
    from imgprocessor_b200 import engine
    return engine


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def test_k4_golden(engine):
    g = load_golden('ste')
    fr, nlf = g['frames'], tuple(g['nlf'])
    e = engine.get_engine(*fr.shape[1:])
    for n in (2, 3, 5):
        a, m = e.ste_average(_dev(fr[:n]), nlf, 4, want_mask=True)
        assert np.array_equal(a.cpu().numpy(), g['noSTE_%d' % n])
        assert np.array_equal(m.cpu().numpy(), g['mask_%d' % n])
    a = e.ste_average(_dev(fr.astype(np.float32)), nlf, 3)
    assert np.array_equal(a.cpu().numpy(), g['noSTE_f32_nstd3'])


@pytest.mark.parametrize('shape', [(1, 1), (1, 7), (5, 1), (9, 33), (40, 70), (64, 64), (257, 130)])
@pytest.mark.parametrize('dtype', [np.uint8, np.uint16, np.float32, np.float64])
def test_k4_bit_exact(engine, shape, dtype):
    rng = np.random.default_rng(11)
    e = engine.get_engine(*shape)
    for n in (2, 3, 6):
        f = rng.normal(120, 8, (n,) + shape)
        f[rng.random(f.shape) < 0.05] += 90                     # single pixels and, by chance, clusters
        if shape[0] > 4 and shape[1] > 4:
            f[n - 1, 1:3, 2:4] += 100                            # a 2x2 blob: stays an STE
            f[0, -1, -1] += 100                                  # corner pixel
        f = np.clip(f, 0, 255).astype(dtype) if np.dtype(dtype).kind == 'u' else f.astype(dtype)
        for coeff, nstd in (((2.0, 10.0, 0.8), 4.0), ((0.0, 1e9, 1.0), 3.0), ((3.0, -50.0, 0.0), 2.5)):
            a, m = e.ste_average(_dev(f), coeff, nstd, want_mask=True)
            ra, rm = ste.ste_average(list(f), coeff, nstd, True)
            assert np.array_equal(a.cpu().numpy(), ra), (shape, dtype, n, coeff)
            assert np.array_equal(m.cpu().numpy(), rm)


def test_k4_special_values_and_errors(engine):
    from imgprocessor_b200._lib import ImgcorrError
    e = engine.get_engine(16, 24)
    f = np.random.default_rng(3).normal(100, 5, (4, 16, 24)).astype(np.float32)
    f[0, 3, 3] = np.nan
    f[1, 5, 5] = np.inf
    f[2, 7, 7] = -np.inf
    f[3, 9, 9] = np.nan
    with np.errstate(invalid='ignore'):
        ra, rm = ste.ste_average(list(f), (2.0, 10.0, 0.8), 4, True)
    a, m = e.ste_average(_dev(f), (2.0, 10.0, 0.8), 4, want_mask=True)
    assert np.array_equal(a.cpu().numpy(), ra, equal_nan=True) and np.array_equal(m.cpu().numpy(), rm)
    with pytest.raises(ImgcorrError):
        e.ste_average(_dev(f[:1]), (2.0, 10.0, 0.8))


def test_k4_full_frame_properties(engine):
    """BASELINE frame size: identical exposures average to themselves, a planted blob is rejected, a planted single
    pixel is kept (it is noise by the reference's definition), and the mask equals the oracle's."""
    H, W = 3000, 4096
    e = engine.get_engine(H, W)
    base = (torch.rand((H, W), device='cuda') * 3000 + 500).to(torch.float32)
    frames = base[None].repeat(4, 1, 1).contiguous()
    frames[2, 100:103, 200:204] += 5000
    frames[3, 1500, 2000] += 5000
    nlf = (5.0, 0.0, 0.5)
    avg, mask = e.ste_average(frames, nlf, 4, want_mask=True)
    exp = base.double().clone()
    exp[1500, 2000] += (frames[3, 1500, 2000].double() - exp[1500, 2000]) / 4
    assert torch.equal(mask.nonzero(), torch.stack(torch.meshgrid(torch.arange(100, 103), torch.arange(200, 204), indexing='ij'),
                                                   -1).reshape(-1, 2).cuda())
    assert torch.allclose(avg, exp, rtol=0, atol=1e-9)
    ra, rm = ste.ste_average(list(frames[:, 1400:1600, 1900:2100].cpu().numpy()), nlf, 4, True)
    assert np.array_equal(avg[1400:1600, 1900:2100].cpu().numpy(), ra)


def test_k4_two_streams_share_one_context(engine):
    """two K4 calls of one context on two torch streams, released together by one event after a spin: the second waits
    for the first's scratch (running average, thresholds, counts) instead of overwriting it"""
    H, W, n = 1024, 1024, 6
    rng = np.random.default_rng(23)
    nlf = (2.0, 10.0, 0.8)
    stacks = []
    for level in (3000, 9000):
        f = rng.normal(level, 40, (n, H, W))
        f[rng.random(f.shape) < 0.01] += 2000                   # single pixels and, by chance, clusters
        f[n - 1, 100:103, 200:204] += 5000                      # a blob: stays an STE
        stacks.append(np.clip(f, 0, 65535).astype(np.uint16))
    want = [ste.ste_average(list(f), nlf, 4, True) for f in stacks]
    e = engine.get_engine(H, W)
    a, b = _dev(stacks[0]), _dev(stacks[1])
    e.ste_average(a[:2], nlf, 4)                                 # allocation outside the race
    sa, sb = torch.cuda.Stream(), torch.cuda.Stream()
    go = torch.cuda.Event()
    torch.cuda.synchronize()
    with torch.cuda.stream(sa):
        torch.cuda._sleep(600_000_000)                           # about 0.3 s of device time
        go.record(sa)
        got_a = e.ste_average(a, nlf, 4, want_mask=True)
    with torch.cuda.stream(sb):
        sb.wait_event(go)
        got_b = e.ste_average(b, nlf, 4, want_mask=True)
    torch.cuda.synchronize()
    for tag, (avg, mask), (ra, rm) in zip('ab', (got_a, got_b), want):
        assert np.array_equal(avg.cpu().numpy(), ra), tag
        assert np.array_equal(mask.cpu().numpy(), rm), tag


def test_correct_with_several_exposures():
    """the Python mirror against the reference's correct() (multi-image branches :385-406, :484-498)"""
    if not torch.cuda.is_available():
        pytest.skip('needs a CUDA device')
    from imgprocessor_b200.camera import CameraCalibration, LensDistortion
    g = load_golden('ste')
    fr = g['frames']
    lens = LensDistortion({'cameraMatrix': g['K'], 'distortionCoeffs': g['dist'], 'shape': fr.shape[1:]})
    cal = CameraCalibration()
    cal.addDarkCurrent(g['dark'])
    cal.addFlatField(g['flat'])
    cal.addLens(lens)
    cal.addNoise(tuple(g['nlf']))
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        out = cal.correct(list(fr[:3]), threshold=0.1)
    assert buf.getvalue() == str(g['correct_3_log'])
    ref = g['correct_3']
    assert out.dtype == np.float64 and out.shape == ref.shape
    assert np.abs(out - ref).max() <= 1e-5 * 65535
    with contextlib.redirect_stdout(io.StringIO()):
        assert np.array_equal(cal.correct(fr[:3], threshold=0.1), out)          # a 3-D array is a stack of exposures too
    cal2 = CameraCalibration()
    cal2.addFlatField(g['flat'])
    cal2.addNoise(tuple(g['nlf']))
    # the bgImages branch hands self.noise_level_function to the STE detection as it is (:490-494); the golden run set it to
    # the reference's own lambda — an arbitrary callable here, which goes to K4 as a threshold map
    from imgprocessor_b200.camera import NoiseLevelFunction as nlfmod
    nlf = tuple(g['nlf'])
    cal2.noise_level_function = lambda x: nlfmod.boundedFunction(x, *nlf)
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        out = cal2.correct(fr[0], bgImages=list(g['bgs']), threshold=0.1)
    assert buf.getvalue() == str(g['correct_bg3_log'])
    assert np.array_equal(cal2.temp['bg'], g['correct_bg3_bg'])
    assert np.abs(out - g['correct_bg3']).max() <= 1e-5 * 65535


def test_noise_level_function_estimated_when_uncalibrated():
    """correct([a, b, c]) WITHOUT a 'noise' calibration: the reference estimates the noise level function from the exposures
    (SingleTimeEffectDetection.py:43-45 -> NoiseLevelFunction.oneImageNLF) and keeps it.  Golden: the unmodified reference
    (tests/golden/make_golden.py ste_nlf).  The 3x3 median of the estimate runs on the GPU (K1) and must equal scipy's
    bit for bit; bins, fit parameters, STE-free averages and masks follow bit for bit; the corrected frame within the
    float32 chain's 1e-5 of full scale."""
    if not torch.cuda.is_available():
        pytest.skip('needs a CUDA device')
    from imgprocessor_b200 import engine
    from imgprocessor_b200.camera import CameraCalibration, LensDistortion
    from imgprocessor_b200.camera import NoiseLevelFunction as nlfmod
    g = load_golden('ste_nlf')
    fr = g['frames']
    H, W = fr.shape[1:]
    e = engine.get_engine(H, W)
    assert np.array_equal(e.median3x3(g['avg0']), g['nlf_signal'])
    x, y, w, signal = nlfmod.calcNLF(g['avg0'])
    filled = g['nlf_w'] > 0
    assert np.array_equal(w, g['nlf_w']) and np.array_equal(signal, g['nlf_signal'])
    assert np.array_equal(x[filled], g['nlf_x'][filled]) and np.array_equal(y[filled], g['nlf_y'][filled])
    x2, y2, w2, s2 = nlfmod.calcNLF(fr[0], fr[1])                     # the two-image estimate
    f2 = g['nlf2_w'] > 0
    assert np.array_equal(w2, g['nlf2_w']) and np.array_equal(s2, g['nlf2_signal']) and np.array_equal(y2[f2], g['nlf2_y'][f2])
    fn, _ = nlfmod.oneImageNLF(g['avg0'])
    assert np.array_equal(np.asarray(fn.params), g['nlf_params'])
    assert np.array_equal(fn(g['nlf_curve_x']), g['nlf_curve'])
    for n in (2, 4):
        avg, mask = e.ste_average(torch.from_numpy(fr[:n].copy()).cuda(), fn.params, 4.0, want_mask=True)
        assert np.array_equal(avg.cpu().numpy(), g['noSTE_%d' % n])
        assert np.array_equal(mask.cpu().numpy(), g['mask_%d' % n])
        # the same through a threshold map (what a non-boundedFunction callable gets)
        thr = fn(g['avg0']) * 4.0
        avg2 = e.ste_average(torch.from_numpy(fr[:n].copy()).cuda(), threshold=thr)
        assert np.array_equal(avg2.cpu().numpy(), g['noSTE_%d' % n])
    lens = LensDistortion({'cameraMatrix': g['K'], 'distortionCoeffs': g['dist'], 'shape': (H, W)})
    cal = CameraCalibration()
    cal.addDarkCurrent(g['dark'])
    cal.addFlatField(g['flat'])
    cal.addLens(lens)
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        out = cal.correct(list(fr[:3]), threshold=0.1)
    assert buf.getvalue() == str(g['correct_3_log'])
    assert np.abs(out - g['correct_3']).max() <= 1e-5 * 65535
    assert cal.noise_level_function is not None and np.array_equal(np.asarray(cal.noise_level_function.params), g['nlf_params'])
    with contextlib.redirect_stdout(io.StringIO()):
        again = cal.correct(list(fr[1:4]), threshold=0.1)              # re-uses the kept function, as the reference does
    assert np.abs(again - g['correct_3_again']).max() <= 1e-5 * 65535
