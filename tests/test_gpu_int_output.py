"""uint16 / uint8 output of the batch chain (out_dtype U16 / U8 with an output scale), fused into the chain's last
kernel, for device and host frames.

Every integer result is compared bit for bit with quantise_model.quantise applied to the float32 oracle chain
(models.correct_chain_f32) and to the same call made with float32 output: for any configuration the integer call
equals quantise(F32 call).  Also covered: the launch count (no extra conversion pass), the refusals, and that a float32
call after an integer one on the same engine is unchanged."""
import contextlib
import io

import numpy as np
import pytest

from quantise_model import quantise
from test_gpu_chain import _calibration, _crop, _dev, _file_image, _flags, _frames, _host, _lens, _maps, _Options, _oracle, _same
from test_gpu_perspective_chain import _stage, _warp

pytestmark = pytest.mark.gpu

torch = pytest.importorskip('torch')

# identity (saturate_cast); a negative offset with a gain > 1; a scale that puts integer results exactly on .5
SCALES = [(0.0, 1.0), (-1000.5, 3.0), (0.0, 0.5)]
INT_OUT = [(np.uint16, 'uint16'), (np.uint8, 'uint8')]


@pytest.fixture(scope='module')
def ip():
    if not torch.cuda.is_available():
        pytest.skip('needs a CUDA device')
    import imgprocessor_b200 as pkg
    from imgprocessor_b200 import engine, _lib
    pkg.engine_mod, pkg.lib_mod = engine, _lib
    return pkg


def _tdt(np_dtype):
    return {np.uint16: torch.uint16, np.uint8: torch.uint8, np.float32: torch.float32}[np_dtype]


def _q(v, dt, scale):
    return quantise(v, dt, *scale)


def _setup(ip, H, W, seed):
    e = ip.engine_mod.get_engine(H, W)
    dark, flat = _calibration(H, W, seed)
    e.set_dark(dark)
    e.set_flat(flat)
    roi = _lens(e, H, W)
    return e, dark, flat, roi, _maps(e)


# ---------------------------------------------------------------------------------------------- 1. the device chain
@pytest.mark.parametrize('shape', [(83, 256), (70, 250), (130, 344)])
@pytest.mark.parametrize('thr', [0.1, 0.0])
@pytest.mark.parametrize('ksize', [3, 5])
@pytest.mark.parametrize('dtype', [np.uint8, np.uint16, np.float32])
def test_device_chain_vs_quantised_oracle(ip, shape, thr, ksize, dtype):
    """5 frames (groups of 2: the pair and the one-frame K1 kernels) without a lens (K1 alone), with the full-frame lens
    and with the roi window; uint16 and uint8 output under each scale.  float32 frames carry NaN, +-inf and +-3e38."""
    H, W = shape
    n = 5
    L = ip.lib_mod
    e, dark, flat, roi, maps = _setup(ip, H, W, 3)
    raw = _frames(H, W, n, 40, dtype)
    dev = _dev(raw)
    fl = _flags(L, thr)
    oracle = {lens: [_oracle(raw[i], dark, flat, thr, ksize, maps if lens else None) for i in range(n)] for lens in (False, True)}
    with _Options(ip, e) as o:
        o.set(L.OPT_CHAIN_GROUP, 2)
        for lens, window in ((False, None), (True, None), (True, roi)):
            f32 = _host(e.correct_batch(dev, threshold=thr, ksize=ksize, flags=fl, use_lens=lens, window=window))
            for i in range(n):
                assert _same(f32[i], _crop(oracle[lens][i], window)), ('f32', lens, window, i)
            for dt, _ in INT_OUT:
                for scale in SCALES:
                    got = _host(e.correct_batch(dev, threshold=thr, ksize=ksize, flags=fl, use_lens=lens, window=window,
                                                out_dtype=_tdt(dt), out_scale=scale))
                    assert _same(got, _q(f32, dt, scale)), (lens, window, dt, scale)
                    for i in range(n):
                        assert _same(got[i], _q(_crop(oracle[lens][i], window), dt, scale)), (lens, window, dt, scale, i)


def test_exact_ties_round_half_to_even(ip):
    """integer results (no calibration, no lens: the median of integer samples) under gain 0.5: half of the pixels are
    exact ties, stored to the even neighbour"""
    H, W, n = 70, 250, 3
    L = ip.lib_mod
    e = ip.engine_mod.get_engine(H, W)
    raw = _frames(H, W, n, 60, np.uint16)
    dev = _dev(raw)
    f32 = _host(e.correct_batch(dev, threshold=0.1, ksize=3, flags=L.DO_NAN_TO_NUM, use_lens=False))
    assert np.array_equal(f32, np.floor(f32))
    got = _host(e.correct_batch(dev, threshold=0.1, ksize=3, flags=L.DO_NAN_TO_NUM, use_lens=False,
                                out_dtype=torch.uint16, out_scale=(0.0, 0.5)))
    odd = (f32 % 2) == 1
    assert odd.mean() > 0.2
    assert _same(got, _q(f32, np.uint16, (0.0, 0.5)))
    assert np.array_equal(got[odd], ((f32[odd] - 1) / 2 + ((f32[odd] - 1) / 2) % 2).astype(np.uint16))


def test_group_seams_with_overlap(ip):
    """33 frames in groups of 5 with the overlap stream on: every group seam and the odd last frame"""
    H, W, n = 130, 344, 33
    L = ip.lib_mod
    e, dark, flat, roi, maps = _setup(ip, H, W, 5)
    raw = _frames(H, W, n, 70, np.uint16)
    dev = _dev(raw)
    scale = SCALES[1]
    with _Options(ip, e) as o:
        o.set(L.OPT_CHAIN_GROUP, 5)
        o.set(L.OPT_CHAIN_OVERLAP, 1)
        for window in (None, roi):
            f32 = _host(e.correct_batch(dev, window=window))
            for dt, _ in INT_OUT:
                got = _host(e.correct_batch(dev, window=window, out_dtype=_tdt(dt), out_scale=scale))
                assert _same(got, _q(f32, dt, scale)), (window, dt)
            for i in (0, 4, 5, 9, 10, 30, 32):
                want = _crop(_oracle(raw[i], dark, flat, 0.1, 3, maps), window)
                assert _same(got[i], _q(want, np.uint8, scale)), (window, i)


def test_full_size(ip):
    """4096x3000 uint16 frames, the moderate lens, 3 frames (the one-frame K2 launch reads the coordinate cache)"""
    H, W, n = 3000, 4096, 3
    e, dark, flat, roi, maps = _setup(ip, H, W, 11)
    raw = _frames(H, W, n, 7, np.uint16)
    dev = _dev(raw)
    f32 = _host(e.correct_batch(dev))
    for dt, _ in INT_OUT:
        got = _host(e.correct_batch(dev, out_dtype=_tdt(dt), out_scale=SCALES[1]))
        assert _same(got, _q(f32, dt, SCALES[1])), dt
    got = _host(e.correct_batch(dev, out_dtype=torch.uint16))
    assert _same(got[0], _q(_oracle(raw[0], dark, flat, 0.1, 3, maps), np.uint16, (0.0, 1.0)))


# ---------------------------------------------------------------------------------------------- 2. host frames
@pytest.mark.parametrize('slots', [2, 3, 4])
def test_host_pipeline(ip, slots):
    """correct_host from pageable and pinned buffers into pageable and pinned outputs; 83x256 frames travel in chunks of
    16 per ring slot (21 frames: a partial last chunk)"""
    H, W, n = 83, 256, 21
    L = ip.lib_mod
    e, dark, flat, roi, maps = _setup(ip, H, W, 13)
    raw = _frames(H, W, n, 30, np.uint16)
    pin = ip.engine_mod.pinned_empty(raw.shape, np.uint16)
    pin[...] = raw
    with _Options(ip, e) as o:
        o.set(L.OPT_HOST_SLOTS, slots)
        for window in (None, roi):
            f32 = e.correct_host(raw, window=window)
            for i in (0, 15, 16, 20):
                assert _same(f32[i], _crop(_oracle(raw[i], dark, flat, 0.1, 3, maps), window)), (window, i)
            for dt, _ in INT_OUT:
                for scale in SCALES[1:]:
                    for src in (raw, pin):
                        got = e.correct_host(src, window=window, out_dtype=dt, out_scale=scale)
                        assert _same(got, _q(f32, dt, scale)), (window, dt, scale, src is pin)
                        out = ip.engine_mod.pinned_empty(got.shape, dt)
                        e.correct_host(src, out=out, window=window, out_scale=scale)
                        assert _same(np.asarray(out), got), ('pinned out', window, dt)


def test_file_bytes_big_endian(ip):
    """big-endian uint16 frames with 20-byte gaps as they sit in a file, swapped in K1's load, to uint16 output"""
    H, W, n = 83, 256, 5
    e, dark, flat, roi, maps = _setup(ip, H, W, 17)
    raw = _frames(H, W, n, 50, np.uint16)
    for gap in (0, 20):
        off = 12
        buf = _file_image(raw, off, gap, big_endian=True)
        f32 = _host(e.correct_file_bytes(_dev(buf), off, n, gap=gap, big_endian=True))
        for dt, _ in INT_OUT:
            got = _host(e.correct_file_bytes(_dev(buf), off, n, gap=gap, big_endian=True, out_dtype=_tdt(dt),
                                             out_scale=SCALES[1]))
            assert _same(got, _q(f32, dt, SCALES[1])), (gap, dt)
        for i in range(n):
            assert _same(f32[i], _oracle(raw[i], dark, flat, 0.1, 3, maps)), (gap, i)


def test_perspective_stage(ip):
    """the perspective stage without a tilt factor: the float32 chain frame warped in float32 (Lanczos4), quantised on
    K3's store; full frame and roi window, 7 frames in groups of 4 (K3's staged tiles, then its L1 path)"""
    H, W, n = 96, 256, 7
    L = ip.lib_mod
    e, dark, flat, roi, maps = _setup(ip, H, W, 19)
    raw = _frames(H, W, n, 90, np.uint16)
    dev = _dev(raw)
    fl = _flags(L, 0.1) | L.DO_PERSPECTIVE
    try:
        with _Options(ip, e) as o:
            o.set(L.OPT_CHAIN_GROUP, 4)
            for lens, window in ((True, None), (True, roi), (False, None)):
                sh = (window[3], window[2]) if window else (H, W)
                M, dsize = _stage(*sh, quad='outside', dsize='larger')
                e.set_perspective(M, dsize, 3.25)
                f32 = _host(e.correct_batch(dev, flags=fl, use_lens=lens, window=window))
                for i in (0, 3, 6):
                    want = _warp(_crop(_oracle(raw[i], dark, flat, 0.1, 3, maps if lens else None), window), M, dsize, 3.25)
                    assert _same(f32[i], want), (lens, window, i)
                for dt, _ in INT_OUT:
                    for scale in SCALES:
                        got = _host(e.correct_batch(dev, flags=fl, use_lens=lens, window=window, out_dtype=_tdt(dt),
                                                    out_scale=scale))
                        assert _same(got, _q(f32, dt, scale)), (lens, window, dt, scale)
                        hst = e.correct_host(raw, flags=fl, use_lens=lens, window=window, out_dtype=dt, out_scale=scale)
                        assert _same(hst, got), ('host', lens, window, dt, scale)
    finally:
        e.set_perspective(None, None)


# ---------------------------------------------------------------------------------------------- 3. public API
def test_camera_calibration_correct_batch(ip):
    """cal.correct_batch(out_dtype=uint16 / uint8, out_scale=...) == quantise(the float32 call): host frames, CUDA tensors,
    two contexts on one device (devices=[0, 0]) and every GPU of the machine"""
    H, W, n = 96, 256, 6
    dark, flat = _calibration(H, W, 9)
    cal = ip.CameraCalibration()
    cal.addDarkCurrent(dark)
    cal.addFlatField(flat)
    lens = ip.LensDistortion({})
    from imgprocessor_b200 import synth
    lens.setCameraParams(*synth.lens_moderate(H, W))
    lens._coeffs['shape'] = (H, W)
    cal.addLens(lens)
    raw = _frames(H, W, n, 140, np.uint16)
    ngpu = torch.cuda.device_count()
    with contextlib.redirect_stdout(io.StringIO()):
        for keep_size in (True, False):
            f32 = cal.correct_batch(raw, keep_size=keep_size)
            for dt, _ in INT_OUT:
                for scale in SCALES[1:]:
                    want = _q(f32, dt, scale)
                    assert _same(cal.correct_batch(raw, keep_size=keep_size, out_dtype=dt, out_scale=scale), want)
                    got = _host(cal.correct_batch(_dev(raw), keep_size=keep_size, out_dtype=_tdt(dt), out_scale=scale))
                    assert _same(got, want), ('tensor', keep_size, dt, scale)
                    for devices in ([0, 0], list(range(ngpu)) if ngpu >= 2 else None):
                        if devices is not None:
                            got = cal.correct_batch(raw, keep_size=keep_size, out_dtype=dt, out_scale=scale, devices=devices)
                            assert _same(got, want), (devices, keep_size, dt, scale)
            assert _same(cal.correct_batch(raw, keep_size=keep_size, out_dtype=np.uint16), _q(f32, np.uint16, (0.0, 1.0)))


def test_refusals(ip):
    """a tilt factor with integer output, bad scales, out_scale with float output, and out arrays of other dtypes"""
    H, W, n = 96, 256, 2
    L = ip.lib_mod
    e, dark, flat, roi, maps = _setup(ip, H, W, 21)
    raw = _frames(H, W, n, 10, np.uint16)
    dev = _dev(raw)
    fl = _flags(L, 0.1) | L.DO_PERSPECTIVE
    try:
        M, dsize = _stage(H, W, quad='mild', dsize='same')
        e.set_perspective(M, dsize, 0.0, tilt_factor=0.5 + np.random.default_rng(1).random((H, W)))
        for call in (lambda: e.correct_batch(dev, flags=fl, out_dtype=torch.uint16),
                     lambda: e.correct_host(raw, flags=fl, out_dtype=np.uint8)):
            with pytest.raises(L.ImgcorrError) as err:
                call()
            assert err.value.status == L.ERR_INVALID and 'F64' in str(err.value)
    finally:
        e.set_perspective(None, None)
    for bad in ((np.nan, 1.0), (np.inf, 1.0), (0.0, 0.0), (0.0, -1.0), (0.0, np.inf), (0.0, np.nan)):
        with pytest.raises(L.ImgcorrError) as err:
            e.correct_batch(dev, out_dtype=torch.uint16, out_scale=bad)
        assert err.value.status == L.ERR_INVALID, bad
        with pytest.raises(L.ImgcorrError):
            e.correct_host(raw, out_dtype=np.uint8, out_scale=bad)
    for call in (lambda: e.correct_batch(dev, out_scale=(0.0, 2.0)),
                 lambda: e.correct_batch(dev, out_dtype=torch.float64, out_scale=(0.0, 2.0)),
                 lambda: e.correct_host(raw, out_scale=(0.0, 2.0))):
        with pytest.raises(ValueError, match='out_scale'):
            call()
    with pytest.raises(TypeError):
        e.correct_host(raw, out=np.empty((n, H, W), np.int16))
    with pytest.raises(TypeError):
        e.correct_batch(dev, out=torch.empty((n, H, W), dtype=torch.int32, device='cuda'))


# ---------------------------------------------------------------------------------------------- 4. fusion, no state leak
def test_same_launches_and_no_state_leak(ip):
    """an integer call launches exactly the kernels of the float32 call (no conversion pass), with and without a lens
    and the perspective stage; a float32 call after integer calls with a scale gives the result and launch count of
    the one before"""
    H, W, n = 96, 256, 9
    L = ip.lib_mod
    e, dark, flat, roi, maps = _setup(ip, H, W, 23)
    raw = _frames(H, W, n, 20, np.float32)
    dev = _dev(raw)

    def run(**kw):
        torch.cuda.synchronize()
        before = e.launch_count
        out = _host(e.correct_batch(dev, **kw))
        return out, e.launch_count - before

    try:
        for persp in (False, True):
            fl = _flags(L, 0.1) | (L.DO_PERSPECTIVE if persp else 0)
            if persp:
                e.set_perspective(*_stage(H, W, quad='strong', dsize='smaller'), 0.0)
            for lens, window, ks in ((False, None, 3), (True, None, 3), (True, roi, 5)):
                kw = dict(flags=fl, use_lens=lens, window=window, ksize=ks)
                ref, nl = run(**kw)
                assert nl > 0
                for dt, _ in INT_OUT:
                    got, nq = run(out_dtype=_tdt(dt), out_scale=(-3.0, 7.0), **kw)
                    assert nq == nl, (persp, lens, window, dt)
                    assert _same(got, _q(ref, dt, (-3.0, 7.0)))
                again, na = run(**kw)
                assert na == nl and _same(again, ref), (persp, lens, window)
                assert _same(e.correct_host(raw, **kw), ref)
    finally:
        e.set_perspective(None, None)
    # medianThreshold's own integer output (imgcorr_pointwise_median) ignores the chain's scale
    u16 = _dev(_frames(H, W, 1, 21, np.uint16))
    out, _ = e.pointwise_median(u16, 0.1, 3, flags=0, out_dtype=torch.uint16)
    e.correct_batch(dev, out_dtype=torch.uint16, out_scale=(100.0, 0.25))
    out2, _ = e.pointwise_median(u16, 0.1, 3, flags=0, out_dtype=torch.uint16)
    assert _same(_host(out), _host(out2))
