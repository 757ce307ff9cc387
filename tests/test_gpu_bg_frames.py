"""The chain with one background image per frame (imgcorr_correct_batch_bg / imgcorr_correct_host_bg, Engine.correct_batch /
correct_host with bg=, CameraCalibration.correct_batch(bg_frames=...)) against the oracle, frame by frame and bit for bit.

For uint8 / uint16 / float32 backgrounds, frame i of a call is the float32 oracle chain of raw[i] with the dark map
float32(bg[i]): the oracle computes raw - dark in float64, which is what correct(frame, bgImages=bg) does.  Every comparison
is np.array_equal(..., equal_nan=True).  The full-size case compares against the two-step device composition (the
difference in torch, then the chain without a dark stage), which is exact for uint16 frames."""
import contextlib
import io

import numpy as np
import pytest

from imgprocessor_b200 import synth
from quantise_model import quantise
from test_gpu_chain import (_calibration, _crop, _dev, _flags, _frames, _host, _lens, _maps, _Options, _oracle, _same,
                            ip)  # noqa: F401  (ip is a fixture)
from test_gpu_perspective_chain import _calibrated, _warp
from test_gpu_perspective_frames import MIXED, _table

pytestmark = pytest.mark.gpu

torch = pytest.importorskip('torch')

TDT = {np.float32: torch.float32, np.float64: torch.float64, np.uint16: torch.uint16}


def _bgs(raw, kind, seed):
    """one background per frame: of the frames' dtype ('same') or float32 ('f32').  Integer backgrounds reach twice the
    frame's mean, so that many differences are negative; float32 ones carry NaN, +-inf and +-3e38 on the edges and inside"""
    rng = np.random.default_rng(seed)
    n, H, W = raw.shape
    dt = raw.dtype if kind == 'same' else np.dtype(np.float32)
    top = float(np.nanmean(np.clip(raw[np.isfinite(raw)].astype(np.float64), 0, 65535))) * 2 + 1
    if dt.kind == 'u':
        top = min(top, float(np.iinfo(dt).max))
        return rng.integers(0, int(top) + 1, size=raw.shape).astype(dt)
    bg = (rng.random(raw.shape) * top).astype(np.float32)
    special = [np.nan, np.inf, -np.inf, 3e38, -3e38]
    for i in range(n):
        for k, v in enumerate(special):
            bg[i, (3 * k + i) % H, (7 * k + 2 * i) % W] = v
            bg[i, 0, (11 * k + i) % W] = v
            bg[i, (5 * k + i) % H, W - 1] = v
    return bg


def _want(raw, bg, flat, thr, ksize, maps, window, odt, cal='df'):
    w = _oracle(raw, bg.astype(np.float32), flat, thr, ksize, maps, 0.0, cal)
    if odt == np.uint16:
        return quantise(_crop(w, window), np.uint16)
    return _crop(w, window, odt)


def _setup(ip, H, W, seed):
    e = ip.engine_mod.get_engine(H, W)
    dark, flat = _calibration(H, W, seed)
    e.set_dark(dark)
    e.set_flat(flat)
    roi = _lens(e, H, W)
    return e, dark, flat, roi, _maps(e)


# ---------------------------------------------------------------------------------------------- 1. device frames
@pytest.mark.parametrize('shape', [(83, 256), (70, 264), (70, 250)])    # streaming for all / for 2- and 4-byte frames / none
@pytest.mark.parametrize('kind', ['same', 'f32'])
@pytest.mark.parametrize('dtype', [np.uint8, np.uint16, np.float32])
def test_device_frames_vs_oracle(ip, shape, kind, dtype):
    """11 frames with their own backgrounds.  Base: groups of 5 (frame pairs, a one-frame tail, a one-frame group), overlap
    on, lens on, full frame, float32 out, threshold 0.1, 3x3, dark + flat.  Each other axis alone: one group of 16, groups of
    3 without overlap, no lens (K1 ends the chain) with float32 / uint16 out and with threshold 0, the roi window, float64
    and uint16 out, threshold 0, the 5x5 median, and no flat field."""
    H, W = shape
    n = 11
    L = ip.lib_mod
    e, dark, flat, roi, maps = _setup(ip, H, W, 3)
    raw = _frames(H, W, n, 40, dtype)
    bg = _bgs(raw, kind, 7)
    dev, dbg = _dev(raw), _dev(bg)
    base = dict(group=5, overlap=1, lens=True, window=None, odt=np.float32, thr=0.1, ksize=3, cal='df')
    cases = [base] + [dict(base, **v) for v in (
        {'group': 16}, {'group': 3, 'overlap': 0}, {'lens': False}, {'lens': False, 'odt': np.uint16},
        {'lens': False, 'thr': 0.0}, {'window': roi}, {'odt': np.float64}, {'odt': np.uint16}, {'thr': 0.0},
        {'ksize': 5}, {'cal': 'd'})]
    with _Options(ip, e) as o:
        for c in cases:
            o.set(L.OPT_CHAIN_GROUP, c['group'])
            o.set(L.OPT_CHAIN_OVERLAP, c['overlap'])
            out = e.correct_batch(dev, threshold=c['thr'], ksize=c['ksize'], flags=_flags(L, c['thr'], c['cal']),
                                  use_lens=c['lens'], window=c['window'], out_dtype=TDT[c['odt']], bg=dbg)
            got = _host(out)
            for i in range(n):
                w = _want(raw[i], bg[i], flat, c['thr'], c['ksize'], maps if c['lens'] else None, c['window'], c['odt'],
                          c['cal'])
                assert _same(got[i], w), (c, i)


# ---------------------------------------------------------------------------------------------- 2. the streaming kernel runs
@pytest.mark.parametrize('dtype', [np.uint16, np.float32])
def test_streaming_variant_runs(ip, dtype):
    """IMGCORR_OPT_K1_VARIANT = 3 forces the streaming pipeline: uint16 + uint16 and float32 + float32 backgrounds are
    taken on a streaming shape (frame pairs and the one-frame tail, threshold 0.1 and 0, lens on and off, uint16 out) and
    equal the generic tiles (variant 1) and the oracle; a pair the pipeline does not implement is refused, not run wrong"""
    H, W, n = 83, 256, 7
    L = ip.lib_mod
    e, dark, flat, roi, maps = _setup(ip, H, W, 5)
    raw = _frames(H, W, n, 60, dtype)
    bg = _bgs(raw, 'same', 8)
    dev, dbg = _dev(raw), _dev(bg)
    with _Options(ip, e) as o:
        for lens, thr, odt in ((True, 0.1, np.float32), (False, 0.1, np.float32), (False, 0.0, np.float32),
                               (True, 0.0, np.float32), (False, 0.1, np.uint16)):
            res = {}
            for variant in (3, 1):
                o.set(L.OPT_K1_VARIANT, variant)
                res[variant] = _host(e.correct_batch(dev, threshold=thr, flags=_flags(L, thr), use_lens=lens,
                                                     out_dtype=TDT[odt], bg=dbg))
            assert _same(res[3], res[1]), (lens, thr, odt)
            for i in (0, n - 1):
                assert _same(res[3][i], _want(raw[i], bg[i], flat, thr, 3, maps if lens else None, None, odt)), (lens, thr, i)
        o.set(L.OPT_K1_VARIANT, 3)
        refused = [dict(ksize=5, bg=dbg)]                          # the 5x5 pipeline does not take backgrounds
        if dtype == np.uint16:
            refused.append(dict(bg=_dev(_bgs(raw, 'f32', 9))))     # nor a float32 background of uint16 frames
        for kw in refused:
            with pytest.raises(L.ImgcorrError):
                e.correct_batch(dev, use_lens=False, **kw)
        o.set(L.OPT_K1_VARIANT, 2)                                 # nor the TMA tiles
        with pytest.raises(L.ImgcorrError):
            e.correct_batch(dev, use_lens=False, bg=dbg)


# ---------------------------------------------------------------------------------------------- 3. host pipeline
@pytest.mark.parametrize('slots', [2, 3, 8])
def test_host_pipeline_vs_device(ip, slots):
    """correct_host(bg=) equals correct_batch(bg=): 37 small frames in chunks (backgrounds at chunk offsets), pageable and
    pinned frames and backgrounds, pageable and pinned output; float32 backgrounds of uint16 frames; the roi window with
    float64 out; and a call without backgrounds afterwards still equals its device call"""
    H, W, n = 96, 160, 37
    L = ip.lib_mod
    e, dark, flat, roi, maps = _setup(ip, H, W, 13)
    pe = ip.engine_mod.pinned_empty
    raw = _frames(H, W, n, 200, np.uint16)
    with _Options(ip, e) as o:
        o.set(L.OPT_HOST_SLOTS, slots)
        for kind in ('same', 'f32'):
            bg = _bgs(raw, kind, 21)
            want = _host(e.correct_batch(_dev(raw), bg=_dev(bg)))
            pin_raw, pin_bg = pe(raw.shape, raw.dtype), pe(bg.shape, bg.dtype)
            pin_raw[...] = raw
            pin_bg[...] = bg
            for r, b in ((raw, bg), (pin_raw, pin_bg), (raw, pin_bg), (pin_raw, bg)):
                for pinned_out in (False, True):
                    out = pe(raw.shape, np.float32) if pinned_out else np.empty(raw.shape, np.float32)
                    out[...] = -1
                    got = e.correct_host(r, out=out, bg=b)
                    assert got is out and _same(got, want), (kind, r is pin_raw, b is pin_bg, pinned_out)
            got = e.correct_host(raw, bg=bg, window=roi, out_dtype=np.float64)
            assert _same(got, _host(e.correct_batch(_dev(raw), bg=_dev(bg), window=roi, out_dtype=torch.float64))), kind
        assert _same(e.correct_host(raw), _host(e.correct_batch(_dev(raw))))
    for i in (0, 16, 36):
        assert _same(want[i], _want(raw[i], bg[i], flat, 0.1, 3, maps, None, np.float32)), i


# ---------------------------------------------------------------------------------------------- 4. composition
def test_per_frame_perspective_with_backgrounds(ip):
    """the per-frame perspective table and per-frame backgrounds in one call: frame i is the oracle warp (matrix i) of the
    oracle chain of raw[i] with dark float32(bg[i]); device and host frames"""
    H, W, n = 96, 256, 6
    L = ip.lib_mod
    e, dark, flat, roi, maps = _setup(ip, H, W, 3)
    raw = _frames(H, W, n, 80, np.uint16)
    bg = _bgs(raw, 'same', 4)
    Ms, dsize = _table(H, W, n, MIXED)
    fl = _flags(L, 0.1) | L.DO_PERSPECTIVE
    try:
        e.set_perspective(Ms, dsize, 2.5)
        got = _host(e.correct_batch(_dev(raw), flags=fl, bg=_dev(bg)))
        for i in range(n):
            assert _same(got[i], _warp(_want(raw[i], bg[i], flat, 0.1, 3, maps, None, np.float32), Ms[i], dsize, 2.5)), i
        assert _same(e.correct_host(raw, flags=fl, bg=bg), got)
    finally:
        e.set_perspective(None, None)


def test_camera_calibration_correct_batch(ip):
    """cal.correct_batch(frames, bg_frames=bgs, out_dtype=float64)[i] == cal.correct(frames[i], bgImages=bgs[i]): host
    frames, CUDA tensors, devices=[0] (equal to no devices=) and devices=[0, 0] (two contexts, 3 + 2 frames), keep_size
    False, big-endian frames with big-endian backgrounds, float64 backgrounds (rounded to float32 once, like correct()),
    uint16 output with a scale, and a per-frame perspective list"""
    from imgprocessor_b200.camera import PerspectiveCorrection
    H, W, n = 96, 256, 5
    cal = _calibrated(ip, H, W)
    raw = _frames(H, W, n, 140, np.uint16)
    bgs = _bgs(raw, 'same', 5)
    for keep_size in (True, False):
        with contextlib.redirect_stdout(io.StringIO()):
            want = np.stack([cal.correct(raw[i], bgImages=bgs[i], keep_size=keep_size) for i in range(n)])
        got = cal.correct_batch(raw, bg_frames=bgs, keep_size=keep_size, out_dtype=np.float64)
        assert _same(got, want), keep_size
        got = _host(cal.correct_batch(_dev(raw), bg_frames=_dev(bgs), keep_size=keep_size, out_dtype=torch.float64))
        assert _same(got, want), ('tensor', keep_size)
        for devices in ([0], [0, 0]):
            got = cal.correct_batch(raw, bg_frames=bgs, keep_size=keep_size, out_dtype=np.float64, devices=devices)
            assert _same(got, want), (devices, keep_size)
    with contextlib.redirect_stdout(io.StringIO()):
        want = np.stack([cal.correct(raw[i], bgImages=bgs[i]) for i in range(n)])
    got = cal.correct_batch(raw.astype('>u2'), bg_frames=bgs.astype('>u2'), out_dtype=np.float64)
    assert _same(got, want), 'big-endian'
    got = cal.correct_batch(raw, bg_frames=bgs.astype(np.float64) + 0.3, out_dtype=np.float64)
    with contextlib.redirect_stdout(io.StringIO()):
        w64 = np.stack([cal.correct(raw[i], bgImages=bgs[i].astype(np.float64) + 0.3) for i in range(n)])
    assert _same(got, w64), 'float64 backgrounds'
    got = cal.correct_batch(raw, bg_frames=bgs, out_dtype=np.uint16, out_scale=(10.0, 2.0))
    assert _same(got, quantise(cal.correct_batch(raw, bg_frames=bgs), np.uint16, 10.0, 2.0)), 'uint16 out'
    # a calibration without a dark entry: the backgrounds are the dark stage
    cal2 = ip.CameraCalibration()
    cal2.addFlatField(_calibration(H, W, 9)[1])
    with contextlib.redirect_stdout(io.StringIO()):
        want2 = np.stack([cal2.correct(raw[i], bgImages=bgs[i]) for i in range(n)])
    assert _same(cal2.correct_batch(raw, bg_frames=bgs, out_dtype=np.float64), want2), 'no dark entry'
    # per-frame perspective
    ref = want
    Ms, dsize = _table(H, W, n, ['mild', 'strong', 'outside'], dsize='larger')
    pcs = []
    for i in range(n):
        pc = PerspectiveCorrection((H, W), new_size=(dsize[1], dsize[0]))
        pc.setReference(Ms[i])
        pcs.append(pc)
    with contextlib.redirect_stdout(io.StringIO()):
        wp = np.stack([pcs[i].correct(ref[i]) for i in range(n)])
    assert _same(cal.correct_batch(raw, bg_frames=bgs, perspective=pcs, out_dtype=np.float64), wp), 'perspective'


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='a split over several GPUs needs two or more')
def test_camera_calibration_over_every_gpu(ip):
    H, W = 96, 256
    n = 2 * torch.cuda.device_count() + 1
    cal = _calibrated(ip, H, W)
    raw = _frames(H, W, n, 150, np.uint16)
    bgs = _bgs(raw, 'same', 6)
    want = cal.correct_batch(raw, bg_frames=bgs)
    got = cal.correct_batch(raw, bg_frames=bgs, devices=range(torch.cuda.device_count()))
    assert _same(got, want)


# ---------------------------------------------------------------------------------------------- 5. full size
def test_full_size_against_the_two_step_composition(ip):
    """33 uint16 4096x3000 frames with their backgrounds (groups of 16 and a one-frame group, overlap on) equal the
    difference in torch (exact in float32) followed by the chain without a dark stage"""
    H, W, n = 3000, 4096, 33
    L = ip.lib_mod
    e = ip.engine_mod.get_engine(H, W)
    e.set_dark(synth.dark_map(H, W))
    e.set_flat(synth.flat_map(H, W))
    _lens(e, H, W)
    try:
        d = torch.device('cuda', torch.cuda.current_device())
        raw = synth.scene_torch(n, H, W, 17, d)
        bg = synth.scene_torch(n, H, W, 18, d)
        got = e.correct_batch(raw, bg=bg)
        want = e.correct_batch(raw.float() - bg.float(), flags=L.DO_FLAT | L.DO_NAN_TO_NUM)
        torch.cuda.synchronize()
        assert torch.equal(got, want)
    finally:
        e.set_lens(None, None, None)


# ---------------------------------------------------------------------------------------------- 6. nothing else changes
def test_later_calls_and_the_dark_map_are_unchanged(ip):
    """a call without backgrounds after background calls gives the values and the launch count it gives on a fresh
    engine, and the stored dark map reads back the same (K1 alone on zero float32 frames returns -dark)"""
    H, W, n = 83, 256, 6
    L = ip.lib_mod
    dark, flat = _calibration(H, W, 3)
    raw = _dev(_frames(H, W, n, 90, np.uint16))
    bg = _dev(_bgs(_frames(H, W, n, 90, np.uint16), 'same', 3))
    zeros = torch.zeros((1, H, W), dtype=torch.float32, device=raw.device)
    res = []
    for with_bg in (False, True):
        e = ip.engine_mod.Engine(H, W)
        try:
            e.set_dark(dark)
            e.set_flat(flat)
            _lens(e, H, W)
            before = _host(e.pointwise_median(zeros, 0.0, 0, flags=L.DO_DARK)[0])
            if with_bg:
                e.correct_batch(raw, bg=bg)
                e.correct_host(_host(raw), bg=_host(bg))
                torch.cuda.synchronize()
            after = _host(e.pointwise_median(zeros, 0.0, 0, flags=L.DO_DARK)[0])
            assert _same(before, after) and _same(after[0], -dark), with_bg
            k = e.launch_count
            out = _host(e.correct_batch(raw))
            res.append((out, e.launch_count - k))
        finally:
            e.close()
    assert _same(res[0][0], res[1][0]) and res[0][1] == res[1][1]


# ---------------------------------------------------------------------------------------------- 7. refusals
def test_refusals(ip):
    """bg_dtype other than the raw dtype or F32, and backgrounds without DO_DARK, fail with IMGCORR_ERR_INVALID before
    anything is enqueued (the launch count does not move); the Python wrappers check shape, device and dtype"""
    import ctypes
    H, W, n = 83, 256, 3
    L = ip.lib_mod
    e, dark, flat, roi, maps = _setup(ip, H, W, 3)
    raw = _dev(_frames(H, W, n, 90, np.uint16))
    out = torch.empty((n, H, W), dtype=torch.float32, device=raw.device)
    bg8 = torch.zeros((n, H, W), dtype=torch.uint8, device=raw.device)
    bg16 = torch.zeros((n, H, W), dtype=torch.uint16, device=raw.device)
    lib = e.lib
    k = e.launch_count

    def call(fn, bg, bg_code, flags):
        return fn(e._h, ctypes.c_void_p(raw.data_ptr()), L.U16, ctypes.c_void_p(bg.data_ptr()), bg_code,
                  ctypes.c_void_p(out.data_ptr()), L.F32, n, 0.1, 3, flags, 1, 0.0, 0, 0, W, H, None)

    for bg, code in ((bg8, L.U8), (bg16, L.F64), (bg16, 7)):
        assert call(lib.imgcorr_correct_batch_bg, bg, code, _flags(L, 0.1)) == L.ERR_INVALID
    assert call(lib.imgcorr_correct_batch_bg, bg16, L.U16, L.DO_FLAT | L.DO_NAN_TO_NUM) == L.ERR_INVALID
    assert e.launch_count == k
    with pytest.raises(ValueError):
        e.correct_batch(raw, bg=bg16[:2])
    with pytest.raises(ValueError):
        e.correct_batch(raw, bg=bg16.cpu())
    with pytest.raises(ValueError):
        e.correct_batch(raw, bg=bg8)
    with pytest.raises(ValueError):
        e.correct_host(_host(raw), bg=_host(bg8))
    with pytest.raises(L.ImgcorrError) as err:
        e.correct_host(_host(raw), bg=_host(bg16), flags=L.DO_FLAT)
    assert err.value.status == L.ERR_INVALID
    assert e.launch_count == k
