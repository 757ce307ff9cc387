"""OpenCV's 4-, 8-, 12- and 14-coefficient lens models (rational, thin-prism and tilted-sensor terms) through K2, the
map kernel, LensDistortion and CameraCalibration, compared exactly with cv2's own maps and cv2.remap."""
import contextlib
import ctypes
import io

import numpy as np
import pytest

import lens_ref
from quantise_model import quantise
from imgprocessor_b200 import synth
from oracle import models, refpath

pytestmark = pytest.mark.gpu

torch = pytest.importorskip('torch')
cv2 = pytest.importorskip('cv2')

LENSES = dict(lens_ref.LENSES, wide=lens_ref.WIDE, fold=lens_ref.FOLD)


@pytest.fixture(scope='module')
def ip():
    if not torch.cuda.is_available():
        pytest.skip('needs a CUDA device')
    import imgprocessor_b200 as pkg
    from imgprocessor_b200 import engine, _lib
    pkg.engine_mod, pkg.lib_mod = engine, _lib
    return pkg


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()) as buf:
        r = fn(*a, **k)
    return r, buf.getvalue()


def _lens(d, H, W):
    """(K, d as OpenCV keeps it (1, n), mapx, mapy, P, roi) with cv2's own float32 maps"""
    K = lens_ref.camera(W, H)
    d = np.asarray(d, np.float64)[None, :]
    mapx, mapy, P, roi = refpath.undistort_rectify_map(K, d, W, H)
    return K, d, mapx, mapy, P, roi


def _lens_obj(ip, K, d, H, W):
    lens = ip.LensDistortion({})
    lens._coeffs['cameraMatrix'], lens._coeffs['distortionCoeffs'], lens._coeffs['shape'] = K, d, (H, W)
    return lens


def _cv2_correct(img, mapx, mapy, roi, keep):
    out = cv2.remap(img, mapx, mapy, cv2.INTER_LINEAR, borderMode=cv2.BORDER_CONSTANT, borderValue=0)
    if not keep:
        x, y, w, h = roi
        out = out[y:y + h, x:x + w]
    return out


def _image(H, W, dtype, seed):
    if dtype in (np.float32, np.float64):
        return synth.scene(H, W, seed, np.float32).astype(dtype)
    return synth.scene(H, W, seed, dtype)


@pytest.mark.parametrize('name', list(LENSES))
def test_undistort_maps_fixed_point_equal_cv2(ip, name):
    """the map kernel (getUndistortRectifyMap) at 4096x3000: every fixed-point coordinate is cv2's"""
    H, W = 3000, 4096
    K, d, mapx, mapy, P, _ = _lens(LENSES[name], H, W)
    e = ip.engine_mod.get_engine(H, W)
    e.set_lens(K, d, P)
    try:
        mx, my = (m.cpu().numpy() for m in e.undistort_maps())
        assert np.array_equal(lens_ref.fixed(mx), lens_ref.fixed(mapx))
        assert np.array_equal(lens_ref.fixed(my), lens_ref.fixed(mapy))
        ex, ey, _ = lens_ref.emul_maps(K, d, P, H, W)           # the host build of the same core function
        assert np.array_equal(mx, ex) and np.array_equal(my, ey)
    finally:
        e.set_lens(None, None, None)


@pytest.mark.parametrize('name', ['rational8', 'tilted14', 'wide', 'fold'])
def test_lens_correct_equals_cv2_remap(ip, name):
    """LensDistortion.correct for uint8 / uint16 / float32 / float64 frames, keepSize True and False, K2 chosen
    automatically, through L1 gathers (variant 1) and through the staged tiles (variant 2), with the coordinate cache on
    and off on a first and a repeated one-frame call: equal to cv2.remap on cv2's maps"""
    H, W = 1200, 1600
    K, d, mapx, mapy, P, roi = _lens(LENSES[name], H, W)
    lens = _lens_obj(ip, K, d, H, W)
    e = ip.engine_mod.get_engine(H, W)
    L = ip.lib_mod
    try:
        for dtype in (np.uint8, np.uint16, np.float32, np.float64):
            img = _image(H, W, dtype, 3)
            for keep in (True, False):
                want = _cv2_correct(img, mapx, mapy, roi, keep)
                for variant in (0, 1, 2):
                    if variant == 2 and dtype == np.float64:
                        continue                                # the tiles take float32 and integer frames
                    e.set_option(L.OPT_K2_VARIANT, variant)
                    for cache in (1, 0):
                        e.set_option(L.OPT_K2_COORD_CACHE, cache)
                        e.set_lens(None, None, None)           # a fresh lens: the first call writes the cache
                        for rep in range(2):
                            got = lens.correct(img, keepSize=keep)
                            assert got.dtype == want.dtype and np.array_equal(got, want), (dtype, keep, variant, cache, rep)
    finally:
        e.set_option(L.OPT_K2_VARIANT, 0)
        e.set_option(L.OPT_K2_COORD_CACHE, 1)


def test_batches_through_both_variants(ip):
    """several frames per launch (the batch paths of both K2 variants) for the tilted lens, full frame and roi window"""
    H, W, n = 600, 800, 5
    K, d, mapx, mapy, P, roi = _lens(LENSES['tilted14'], H, W)
    e = ip.engine_mod.get_engine(H, W)
    e.set_lens(K, d, P)
    x, y, w, h = (int(v) for v in roi)
    try:
        for dtype in (np.uint8, np.uint16, np.float32):
            frames = np.stack([_image(H, W, dtype, 10 + i) for i in range(n)])
            for variant in (1, 2):
                e.set_option(ip.lib_mod.OPT_K2_VARIANT, variant)
                full = e.undistort(_dev(frames)).cpu().numpy()
                crop = e.undistort(_dev(frames), window=(x, y, w, h)).cpu().numpy()
                for i in range(n):
                    want = _cv2_correct(frames[i], mapx, mapy, roi, True)
                    assert np.array_equal(full[i], want), (dtype, variant, i)
                    assert np.array_equal(crop[i], want[y:y + h, x:x + w]), (dtype, variant, i)
    finally:
        e.set_option(ip.lib_mod.OPT_K2_VARIANT, 0)
        e.set_lens(None, None, None)


def _calibrated(ip, H, W, d):
    cal = ip.CameraCalibration()
    cal.addDarkCurrent(synth.dark_map(H, W, 7))
    cal.addFlatField(synth.flat_map(H, W, 7))
    K = lens_ref.camera(W, H)
    cal.addLens(_lens_obj(ip, K, np.asarray(d, np.float64)[None, :], H, W))
    return cal


@pytest.mark.parametrize('name', ['rational8', 'prism12', 'tilted14'])
def test_correct_batch_vs_oracle_chain(ip, name):
    """CameraCalibration.correct_batch with an extended lens: host frames and CUDA tensors, 19 frames (a partial last
    chain group), keep_size True and False, uint16 output: equal to the float32 oracle chain on cv2's maps; correct()
    within 1e-5 of full scale of the float64 reference path"""
    H, W, n = 240, 320, 19
    d = LENSES[name]
    cal = _calibrated(ip, H, W, d)
    dark, flat = synth.dark_map(H, W, 7), synth.flat_map(H, W, 7)
    K, dd, mapx, mapy, P, roi = _lens(d, H, W)
    raw = np.stack([synth.scene(H, W, 50 + i, np.uint16) for i in range(n)])
    want = np.stack([models.correct_chain_f32(raw[i], dark, flat, 0.1, 3, mapxy=(mapx, mapy))[0] for i in range(n)])
    x, y, w, h = (int(v) for v in roi)
    got = cal.correct_batch(raw, threshold=0.1)
    assert got.dtype == np.float32 and np.array_equal(got, want)
    got = cal.correct_batch(_dev(raw), threshold=0.1).cpu().numpy()
    assert np.array_equal(got, want)
    got = cal.correct_batch(raw, threshold=0.1, keep_size=False)
    assert np.array_equal(got, want[:, y:y + h, x:x + w])
    got = cal.correct_batch(raw, threshold=0.1, out_dtype=np.uint16)
    assert got.dtype == np.uint16 and np.array_equal(got, quantise(want, np.uint16))
    if torch.cuda.device_count() >= 2:
        got = cal.correct_batch(raw, threshold=0.1, devices=list(range(torch.cuda.device_count())))
        assert np.array_equal(got, want)
    got = cal.correct_batch(raw, threshold=0.1, devices=[0, 0])
    assert np.array_equal(got, want)
    one, _ = _quiet(cal.correct, raw[0], threshold=0.1)
    ref = refpath.correct(raw[0], dark, flat, (K, dd), 0.1)
    assert one.shape == ref.shape and np.abs(one - ref).max() / 65535.0 < 1e-5


def test_correct_batch_with_perspective(ip):
    """correct_batch(perspective=pc) with the 14-term lens equals pc.correct(cal.correct(frame)) frame by frame"""
    from imgprocessor_b200.camera import PerspectiveCorrection
    H, W, n = 240, 320, 6
    cal = _calibrated(ip, H, W, LENSES['tilted14'])
    raw = np.stack([synth.scene(H, W, 80 + i, np.uint16) for i in range(n)])
    ref = [_quiet(cal.correct, raw[i], threshold=0.1)[0] for i in range(n)]
    M = np.array([[1.02, 0.03, -4.0], [-0.02, 0.99, 3.0], [1e-5, -2e-5, 1.0]])
    pc = PerspectiveCorrection((H, W), new_size=(H - 8, W - 16))
    pc.setReference(M)
    want = np.stack([_quiet(pc.correct, r)[0] for r in ref])
    got = cal.correct_batch(raw, threshold=0.1, perspective=pc, out_dtype=np.float64)
    assert got.shape == want.shape and np.array_equal(got, want)


@pytest.mark.parametrize('n', [4, 8])
def test_zero_extra_terms_equal_five_term_lens(ip, n):
    """a 4-term lens equals the 5-term lens with k3 = 0, and an 8-term lens whose k4..k6 are zero equals its 5-term
    form, bit for bit (maps and remapped frames)"""
    H, W = 600, 800
    d5 = [-0.2, 0.05, 1e-3, -1e-3, 0.0 if n == 4 else 0.02]
    dn = d5[:4] if n == 4 else d5 + [0.0, 0.0, 0.0]
    K = lens_ref.camera(W, H)
    frames = np.stack([synth.scene(H, W, 90 + i, np.float32) for i in range(3)])
    e = ip.engine_mod.get_engine(H, W)
    P, _ = cv2.getOptimalNewCameraMatrix(K, np.asarray(d5), (W, H), 1, (W, H))
    res = []
    try:
        for d in (d5, dn):
            e.set_lens(K, np.asarray(d)[None, :], P)
            res.append([m.cpu().numpy() for m in e.undistort_maps()] + [e.undistort(_dev(frames)).cpu().numpy(),
                                                                           e.undistort(_dev(frames[0])).cpu().numpy()])
    finally:
        e.set_lens(None, None, None)
    for a, b in zip(*res):
        assert np.array_equal(a, b)


def test_switching_lenses_on_one_engine(ip):
    """one engine switched between a 5-term lens, an 8-term lens and an 8-term lens that differs only in k4: each call
    gives its own lens' result (no shared geometry choice or coordinate cache)"""
    H, W = 600, 800
    d8 = LENSES['rational8']
    d8b = list(d8)
    d8b[5] += 0.01
    lenses = [_lens(d, H, W) for d in (LENSES['moderate5'], d8, d8b)]
    img = synth.scene(H, W, 5, np.float32)
    e = ip.engine_mod.get_engine(H, W)
    try:
        for rep in range(2):
            for K, d, mapx, mapy, P, roi in lenses:
                e.set_lens(K, d, P)
                for k in range(2):                              # the first call writes the coordinate cache, the second reads it
                    got = e.undistort(_dev(img)).cpu().numpy()
                    assert np.array_equal(got, _cv2_correct(img, mapx, mapy, roi, True)), (rep, d.size, k)
    finally:
        e.set_lens(None, None, None)


def test_refusals(ip):
    H, W = 48, 64
    e = ip.engine_mod.get_engine(H, W)
    K = lens_ref.camera(W, H)
    P = K.copy()
    with pytest.raises(ValueError):
        e.set_lens(K, np.zeros(6), P)
    L = ip.lib_mod
    vp = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    d = np.zeros(14)
    for n in (0, 3, 6, 7, 9, 13, 15, -1):
        assert e.lib.imgcorr_set_lens_model(e._h, vp(K), vp(d), n, vp(P)) == L.ERR_INVALID
    assert e.lib.imgcorr_set_lens_model(e._h, vp(K), None, 8, vp(P)) == L.ERR_INVALID
    assert e.lib.imgcorr_set_lens_model(e._h, vp(K), vp(d), 8, None) == L.ERR_INVALID
    assert e.lib.imgcorr_set_lens_model(e._h, vp(K), vp(d), 8, vp(np.zeros((3, 3)))) == L.ERR_INVALID
    assert e.lib.imgcorr_set_lens_model(e._h, vp(K), vp(d), 14, vp(P)) == 0
    assert e.lib.imgcorr_set_lens_model(e._h, None, None, 0, None) == 0


def test_unsupported_count_skips_the_lens_stage_with_a_message(ip):
    """CameraCalibration.correct with a 6-coefficient lens: the lens stage prints its error and is skipped, as any
    failing stage"""
    H, W = 96, 128
    cal = _calibrated(ip, H, W, [-0.2, 0.05, 1e-3, -1e-3, 0.0, 0.01])
    raw = synth.scene(H, W, 2, np.uint16)
    out, log = _quiet(cal.correct, raw, threshold=0.1)
    assert 'Error' in log and '4, 5, 8, 12 or 14' in log
    dark, flat = synth.dark_map(H, W, 7), synth.flat_map(H, W, 7)
    want, _ = models.correct_chain_f32(raw, dark, flat, 0.1, 3)
    assert out.shape == (H, W) and np.array_equal(out, want.astype(np.float64))
