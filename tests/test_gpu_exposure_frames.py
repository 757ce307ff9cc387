"""Per-frame exposure times for the linear dark model (imgcorr_set_dark_exposures, Engine.set_dark_exposures,
CameraCalibration.correct_batch(exposure_time=[...])) against the oracle and against the same call with the scalar exposure
t_i, frame by frame and bit for bit.

Frame i of a call evaluates bg = offset + ascent * t_i (two float64 roundings, clipped to 2**depth - 1, NaN staying NaN)
exactly as a call with exposure_time = t_i does, so the oracle is oracle.models.pointwise_model(..., dark_ascent=,
exposure_time=t_i) followed by the median and the remap.  Every comparison is np.array_equal(..., equal_nan=True)."""
import contextlib
import io
import os
import time

import numpy as np
import pytest

from imgprocessor_b200 import synth
from oracle import models
from quantise_model import quantise
from test_gpu_chain import _calibration, _crop, _dev, _frames, _host, _lens, _maps, _Options, _same, ip  # noqa: F401
from test_gpu_perspective_frames import _table
from conftest import load_golden

pytestmark = pytest.mark.gpu

torch = pytest.importorskip('torch')

TDT = {np.float32: torch.float32, np.float64: torch.float64, np.uint16: torch.uint16}
ELBIN_FILE = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'stack_3x24x40.elbin')


def _line(H, W, seed):
    """offset and ascent maps of the line model: the ascent holds zeros and a negative value"""
    rng = np.random.default_rng(seed)
    offs = synth.dark_map(H, W, seed)
    asc = (rng.random((H, W)) * 40.0).astype(np.float32)
    asc[1, 2] = 0.0
    asc[H // 2, W // 3] = -7.5
    return offs, asc


def _times(n, seed=0):
    """n exposure times, some of them repeated"""
    base = np.array([0.3, 1.2, 0.0, 4.8, 2.5, 1.2, 0.8], np.float64)
    return np.resize(np.roll(base, seed), n)


def _want(raw, offs, asc, t, flat, thr, ksize, maps, window=None, odt=np.float32, depth=16):
    x = models.pointwise_model(raw, offs, flat, nan_to_num=thr > 0, dark_ascent=asc, exposure_time=t, depth_bits=depth)
    if thr > 0:
        x, _ = models.median_threshold_model(x, thr, ksize)
    if maps is not None:
        x = models.remap_model(x, maps[0], maps[1], 0.0)
    if odt == np.uint16:
        return quantise(_crop(x, window), np.uint16)
    return _crop(x, window, odt)


def _flags(L, thr):
    return L.DO_DARK | L.DO_FLAT | (L.DO_NAN_TO_NUM if thr > 0 else 0)


def _setup(ip, H, W, seed, depth=16):
    e = ip.engine_mod.get_engine(H, W)
    offs, asc = _line(H, W, seed)
    flat = _calibration(H, W, seed)[1]
    e.set_dark(offs, asc, 0.0, depth)
    e.set_flat(flat)
    roi = _lens(e, H, W)
    return e, offs, asc, flat, roi, _maps(e)


# ---------------------------------------------------------------------------------------------- 1. device frames
@pytest.mark.parametrize('shape', [(83, 256), (70, 250)])        # a streaming width and one the streaming kernels refuse
@pytest.mark.parametrize('dtype', [np.uint8, np.uint16, np.float32])
def test_device_frames_vs_oracle(ip, shape, dtype):
    """11 frames with their own times.  Base: groups of 5, overlap on, lens on, full frame, float32 out, threshold 0.1,
    3x3.  Each other axis alone: one group of 16, groups of 3 without overlap, no lens (K1 ends the chain) with float32 /
    uint16 out and with threshold 0, the roi window, float64 and uint16 out, threshold 0, the 5x5 median, and the generic
    tiles forced (K1 variant 1).  The base case also equals the scalar call with t_i, frame by frame."""
    H, W = shape
    n = 11
    L = ip.lib_mod
    e, offs, asc, flat, roi, maps = _setup(ip, H, W, 3)
    raw = _frames(H, W, n, 40, dtype)
    ts = _times(n)
    dev = _dev(raw)
    base = dict(group=5, overlap=1, lens=True, window=None, odt=np.float32, thr=0.1, ksize=3, variant=0)
    cases = [base] + [dict(base, **v) for v in (
        {'group': 16}, {'group': 3, 'overlap': 0}, {'lens': False}, {'lens': False, 'odt': np.uint16},
        {'lens': False, 'thr': 0.0}, {'window': roi}, {'odt': np.float64}, {'odt': np.uint16}, {'thr': 0.0},
        {'ksize': 5}, {'variant': 1}, {'variant': 1, 'lens': False})]
    try:
        e.set_dark_exposures(ts)
        with _Options(ip, e) as o:
            for c in cases:
                o.set(L.OPT_CHAIN_GROUP, c['group'])
                o.set(L.OPT_CHAIN_OVERLAP, c['overlap'])
                o.set(L.OPT_K1_VARIANT, c['variant'])
                got = _host(e.correct_batch(dev, threshold=c['thr'], ksize=c['ksize'], flags=_flags(L, c['thr']),
                                            use_lens=c['lens'], window=c['window'], out_dtype=TDT[c['odt']]))
                for i in range(n):
                    w = _want(raw[i], offs, asc, ts[i], flat, c['thr'], c['ksize'], maps if c['lens'] else None,
                              c['window'], c['odt'])
                    assert _same(got[i], w), (c, i)
        per_frame = _host(e.correct_batch(dev))
        for i in range(n):
            e.set_dark(offs, asc, ts[i], 16)                  # drops the table
            assert _same(per_frame[i], _host(e.correct_batch(dev[i:i + 1]))[0]), i
    finally:
        e.set_dark(None)


@pytest.mark.parametrize('dtype', [np.uint16, np.float32])
def test_streaming_kernel_vs_oracle(ip, dtype):
    """IMGCORR_OPT_K1_VARIANT = 3 forces the streaming pipeline's line-model configuration: 7 frames (frame pairs and the
    one-frame tail), per-frame times and one scalar time, threshold 0.1 and 0 (KS_NOMED), lens on and off, float32, uint16
    and uint8 output.  It equals the generic tiles (variant 1), the automatic choice and the oracle"""
    H, W, n = 83, 256, 7
    L = ip.lib_mod
    e, offs, asc, flat, roi, maps = _setup(ip, H, W, 5)
    raw = _frames(H, W, n, 60, dtype)
    dev = _dev(raw)
    ts = _times(n, 3)
    try:
        with _Options(ip, e) as o:
            for table in (ts, None):
                e.set_dark(offs, asc, 2.5, 16)
                e.set_dark_exposures(table)
                tv = ts if table is not None else [2.5] * n
                for lens, thr, odt in ((True, 0.1, torch.float32), (False, 0.1, torch.float32), (False, 0.0, torch.float32),
                                       (True, 0.0, torch.float32), (False, 0.1, torch.uint16), (False, 0.1, torch.uint8)):
                    res = {}
                    for variant in (3, 1, 0):
                        o.set(L.OPT_K1_VARIANT, variant)
                        res[variant] = _host(e.correct_batch(dev, threshold=thr, flags=_flags(L, thr), use_lens=lens,
                                                             out_dtype=odt))
                    assert _same(res[3], res[1]) and _same(res[0], res[1]), (table is None, lens, thr, odt)
                    if odt == torch.float32:
                        for i in range(n):
                            w = _want(raw[i], offs, asc, tv[i], flat, thr, 3, maps if lens else None)
                            assert _same(res[3][i], w), (table is None, lens, thr, i)
    finally:
        e.set_dark(None)


def test_streaming_kernel_overflow_and_unbounded_times(ip):
    """uint16 frames through the streaming kernel where the overflow proof cannot hold: a very negative ascent on a few
    pixels and a tiny flat value there make |raw - bg| / flat overflow float32 (finite maps: the unchecked kernel with the
    nan_to_num clamp), and an infinite time leaves no bound at all (the checked kernel).  Both equal the tiles and the
    oracle, and the clamp acts"""
    H, W, n = 64, 256, 5
    L = ip.lib_mod
    e = ip.engine_mod.get_engine(H, W)
    offs, asc = _line(H, W, 12)
    flat = _calibration(H, W, 12)[1]
    asc[10:14, 20:30] = -1e30                       # a block, so that the 3x3 median keeps the clamped values
    flat[10:14, 20:30] = np.float32(1e-9)
    raw = _frames(H, W, n, 61, np.uint16)
    e.set_dark(offs, asc, 0.0, 16)
    e.set_flat(flat)
    try:
        with _Options(ip, e) as o:
            for ts in ([1.0, 2.0, 0.5, 3.0, 1.5], [1.0, np.inf, -np.inf, 0.0, 2.0]):
                e.set_dark_exposures(ts)
                res = {}
                for variant in (3, 1):
                    o.set(L.OPT_K1_VARIANT, variant)
                    res[variant] = _host(e.correct_batch(_dev(raw), threshold=0.1, flags=_flags(L, 0.1), use_lens=False))
                assert _same(res[3], res[1]), ts
                for i in range(n):
                    assert _same(res[3][i], _want(raw[i], offs, asc, ts[i], flat, 0.1, 3, None)), (ts, i)
                assert (res[3][0] == np.float32(3.4028235e38)).any() and np.isfinite(res[3][0]).all()
    finally:
        e.set_dark(None)
        e.set_flat(None)


# ---------------------------------------------------------------------------------------------- 2. K1 alone
@pytest.mark.parametrize('dtype', [np.uint8, np.uint16, np.float32, np.float64])
@pytest.mark.parametrize('ksize', [0, 3, 5])
def test_pointwise_median_vs_oracle(ip, dtype, ksize):
    """imgcorr_pointwise_median reads the table too: an odd width, 7 frames, every raw dtype (float64 frames give float64
    output), pointwise only and both medians"""
    H, W, n = 37, 129, 7
    L = ip.lib_mod
    e = ip.engine_mod.get_engine(H, W)
    offs, asc = _line(H, W, 6)
    flat = _calibration(H, W, 6)[1]
    e.set_dark(offs, asc, 0.0, 16)
    e.set_flat(flat)
    raw = _frames(H, W, n, 50, np.float32 if dtype == np.float64 else dtype).astype(dtype)
    ts = _times(n, 2)
    thr = 0.1 if ksize else 0.0
    flags = _flags(L, thr)
    try:
        e.set_dark_exposures(ts)
        got = _host(e.pointwise_median(_dev(raw), thr, ksize, flags=flags)[0])
        for i in range(n):
            if dtype != np.float64:
                assert _same(got[i], _want(raw[i], offs, asc, ts[i], flat, thr, max(ksize, 3), None)), i
        for i in range(n):                             # the scalar call with t_i (float64 frames: float64 output)
            e.set_dark(offs, asc, ts[i], 16)
            want = _host(e.pointwise_median(_dev(raw[i:i + 1]), thr, ksize, flags=flags)[0])[0]
            assert got[i].dtype == want.dtype and _same(got[i], want), i
    finally:
        e.set_dark(None)
        e.set_flat(None)


# ---------------------------------------------------------------------------------------------- 3. host pipeline
@pytest.mark.parametrize('slots', [2, 3, 8])
def test_host_pipeline_vs_oracle(ip, slots):
    """37 small host frames travel in chunks of 16 through a ring of 2, 3 or 8 slots: every chunk reads the times from its
    own offset.  Groups of 5 inside a chunk, lens on; then no lens with uint16 output"""
    H, W, n = 40, 64, 37
    L = ip.lib_mod
    e, offs, asc, flat, roi, maps = _setup(ip, H, W, 7)
    raw = _frames(H, W, n, 70, np.uint16)
    ts = np.linspace(-1.0, 6.0, n)
    try:
        e.set_dark_exposures(ts)
        with _Options(ip, e) as o:
            o.set(L.OPT_HOST_SLOTS, slots)
            o.set(L.OPT_CHAIN_GROUP, 5)
            got = e.correct_host(raw)
            for i in range(n):
                assert _same(got[i], _want(raw[i], offs, asc, ts[i], flat, 0.1, 3, maps)), i
            got = e.correct_host(raw, use_lens=False, out_dtype=np.uint16)
            for i in range(n):
                assert _same(got[i], _want(raw[i], offs, asc, ts[i], flat, 0.1, 3, None, odt=np.uint16)), i
    finally:
        e.set_dark(None)


# ---------------------------------------------------------------------------------------------- 4. clip and edge values
def test_clip_and_special_values(ip):
    """a 12-bit sensor: frames with long times clip the dark image at 4095, short ones do not.  Times 0, negative and
    +-inf; NaN and +-inf in the ascent map; and an overflow: float32 frames near FLT_MAX and a very negative dark image
    make |raw - bg| / flat overflow float32, where nan_to_num must clamp to +-FLT_MAX"""
    H, W = 64, 256
    L = ip.lib_mod
    e = ip.engine_mod.get_engine(H, W)
    offs, asc = _line(H, W, 8)
    flat = _calibration(H, W, 8)[1]
    asc[5, 7] = np.nan
    asc[6, 8] = np.inf
    asc[7, 9] = -np.inf
    asc[0, 0] = np.inf
    ts = np.array([0.5, 200.0, 0.0, -3.0, np.inf, -np.inf, 1.0, 120.0])
    n = ts.size
    raw = _frames(H, W, n, 80, np.uint16) % 4096
    e.set_dark(offs, asc, 0.0, 12)
    e.set_flat(flat)
    try:
        e.set_dark_exposures(ts)
        for thr in (0.1, 0.0):
            got = _host(e.correct_batch(_dev(raw), threshold=thr, flags=_flags(L, thr), use_lens=False))
            for i in range(n):
                assert _same(got[i], _want(raw[i], offs, asc, ts[i], flat, thr, 3, None, depth=12)), (thr, i)
        fin = np.isfinite(asc)
        assert (offs[fin] + asc[fin].astype(np.float64) * 200.0 > 4095).any()               # frame 1 clips
        assert (offs[fin] + asc[fin].astype(np.float64) * 0.5 < 4095).all()                 # frame 0 does not
        # overflow: bg = -3e38 * 1e3 (float64, far below -FLT_MAX) for every pixel, float32 frames of +-3e38
        big = np.full((H, W), -3e38, np.float32)
        e.set_dark(np.zeros((H, W), np.float32), big, 0.0, 12)
        e.set_dark_exposures([1e3, 1e-38, 0.0])
        f32 = np.stack([np.full((H, W), 3e38, np.float32), np.full((H, W), -3e38, np.float32),
                        _frames(H, W, 1, 81, np.float32)[0]])
        got = _host(e.correct_batch(_dev(f32), threshold=0.1, flags=_flags(L, 0.1), use_lens=False))
        for i in range(3):
            w = _want(f32[i], np.zeros((H, W), np.float32), big, [1e3, 1e-38, 0.0][i], flat, 0.1, 3, None, depth=12)
            assert _same(got[i], w), i
        assert np.isfinite(got[0]).all() and (np.abs(got[0]) == np.float32(3.4028235e38)).any()
    finally:
        e.set_dark(None)
        e.set_flat(None)


# ---------------------------------------------------------------------------------------------- 5. refusals and lifetime
def test_refusals_and_lifetime(ip):
    """the table needs the line model (ERR_STATE); n <= 0 and NaN are refused (ERR_INVALID) and leave no table; more frames
    than times are refused before anything runs, by the batch, host and K1-only calls; set_dark drops the table, so a
    scalar call afterwards gives the old result; calls with per-frame backgrounds ignore it"""
    H, W = 40, 64
    L = ip.lib_mod
    e, offs, asc, flat, roi, maps = _setup(ip, H, W, 9)
    raw = _frames(H, W, 5, 90, np.uint16)
    dev = _dev(raw)
    try:
        e.set_dark(offs, None, 0.0, 16)
        with pytest.raises(L.ImgcorrError) as ex:
            e.set_dark_exposures([1.0])
        assert ex.value.status == L.ERR_STATE
        e.set_dark(offs, asc, 1.5, 16)
        scalar = _host(e.correct_batch(dev))
        for bad in ([], [1.0, float('nan')]):
            e.set_dark_exposures([2.0] * 5)
            with pytest.raises(L.ImgcorrError) as ex:
                e.set_dark_exposures(bad)
            assert ex.value.status == L.ERR_INVALID and not e.has_exposures
            assert _same(_host(e.correct_batch(dev)), scalar), bad          # no table left: the scalar time
        e.set_dark_exposures([1.5, 2.0, 3.0])
        out = torch.full((5, H, W), 7.0, device=dev.device)
        with pytest.raises(L.ImgcorrError) as ex:
            e.correct_batch(dev, out=out)
        assert ex.value.status == L.ERR_INVALID
        assert bool((out == 7.0).all())                                      # nothing ran
        with pytest.raises(L.ImgcorrError, match='exposure table'):
            e.correct_host(raw)
        with pytest.raises(L.ImgcorrError, match='exposure table'):
            e.pointwise_median(dev)
        # without the dark stage the table is not read
        e.correct_batch(dev, flags=L.DO_FLAT | L.DO_NAN_TO_NUM)
        # per-frame backgrounds replace the dark stage: the table (3 times) is ignored for 5 frames
        bgs = _frames(H, W, 5, 91, np.uint16)
        got = _host(e.correct_batch(dev, bg=_dev(bgs)))
        for i in range(5):
            w = _want(raw[i], bgs[i].astype(np.float32), None, 0.0, flat, 0.1, 3, maps)
            assert _same(got[i], w), i
        got = _host(e.correct_batch(dev[:3]))
        for i in range(3):
            assert _same(got[i], _want(raw[i], offs, asc, [1.5, 2.0, 3.0][i], flat, 0.1, 3, maps)), i
        e.set_dark(offs, asc, 1.5, 16)
        assert not e.has_exposures
        assert _same(_host(e.correct_batch(dev)), scalar)
        e.set_dark_exposures([4.0] * 5)
        e.set_dark_exposures(None)
        assert _same(_host(e.correct_batch(dev)), scalar)
    finally:
        e.set_dark(None)


# ---------------------------------------------------------------------------------------------- 6. CameraCalibration
def _tuple_cal(ip, H, W, offs, asc, flat=None, lens=True):
    cal = ip.CameraCalibration()
    cal.coeffs['dark current'].append((time.localtime(), '', (offs.copy(), asc.copy()), None))
    cal.coeffs['shape'] = (H, W)
    if flat is not None:
        cal.addFlatField(flat)
    if lens:
        lc = ip.LensDistortion({})
        lc.setCameraParams(*synth.lens_moderate(H, W))
        lc._coeffs['shape'] = (H, W)
        cal.addLens(lc)
    return cal


def _correct_each(cal, raw, ts, **kw):
    with contextlib.redirect_stdout(io.StringIO()):
        return np.stack([cal.correct(raw[i], exposure_time=float(ts[i]), **kw) for i in range(len(ts))])


def test_camera_calibration_correct_batch(ip):
    """cal.correct_batch(frames, exposure_time=ts, out_dtype=float64)[i] == cal.correct(frames[i], exposure_time=ts[i])
    with a tuple dark entry: host frames, CUDA tensors, devices=[0] and [0, 0], keep_size False, big-endian frames, uint16
    output with a scale, and a per-frame perspective list.  A scalar afterwards gives the scalar result; an array entry
    takes the times and ignores them"""
    from imgprocessor_b200.camera import PerspectiveCorrection
    H, W, n = 96, 256, 5
    offs, asc = _line(H, W, 10)
    flat = _calibration(H, W, 10)[1]
    cal = _tuple_cal(ip, H, W, offs, asc, flat)
    raw = _frames(H, W, n, 140, np.uint16)
    ts = [0.5, 3.0, 0.5, 0.0, 12.0]
    for keep_size in (True, False):
        want = _correct_each(cal, raw, ts, keep_size=keep_size)
        got = cal.correct_batch(raw, exposure_time=ts, keep_size=keep_size, out_dtype=np.float64)
        assert _same(got, want), keep_size
        got = _host(cal.correct_batch(_dev(raw), exposure_time=np.array(ts), keep_size=keep_size, out_dtype=torch.float64))
        assert _same(got, want), ('tensor', keep_size)
        for devices in ([0], [0, 0]):
            got = cal.correct_batch(raw, exposure_time=ts, keep_size=keep_size, out_dtype=np.float64, devices=devices)
            assert _same(got, want), (devices, keep_size)
    want = _correct_each(cal, raw, ts)
    assert _same(cal.correct_batch(raw.astype('>u2'), exposure_time=ts, out_dtype=np.float64), want), 'big-endian'
    got = cal.correct_batch(raw, exposure_time=ts, out_dtype=np.uint16, out_scale=(10.0, 2.0))
    assert _same(got, quantise(cal.correct_batch(raw, exposure_time=ts), np.uint16, 10.0, 2.0)), 'uint16 out'
    # per-frame perspective
    Ms, dsize = _table(H, W, n, ['mild', 'strong', 'outside'], dsize='larger')
    pcs = []
    for i in range(n):
        pc = PerspectiveCorrection((H, W), new_size=(dsize[1], dsize[0]))
        pc.setReference(Ms[i])
        pcs.append(pc)
    with contextlib.redirect_stdout(io.StringIO()):
        wp = np.stack([pcs[i].correct(want[i]) for i in range(n)])
    assert _same(cal.correct_batch(raw, exposure_time=ts, perspective=pcs, out_dtype=np.float64), wp), 'perspective'
    # a scalar after the per-frame call, and None (the stage is skipped, as in correct())
    want3 = _correct_each(cal, raw, [3.0] * n)
    assert _same(cal.correct_batch(raw, exposure_time=3.0, out_dtype=np.float64), want3), 'scalar'
    with contextlib.redirect_stdout(io.StringIO()):
        skip = np.stack([cal.correct(raw[i]) for i in range(n)])
    assert _same(cal.correct_batch(raw, out_dtype=np.float64), skip), 'None'
    # an array entry: the times are valid and unused
    cal2 = ip.CameraCalibration()
    cal2.addDarkCurrent(offs)
    cal2.addFlatField(flat)
    assert _same(cal2.correct_batch(raw, exposure_time=ts), cal2.correct_batch(raw)), 'array entry'


def test_legacy_golden_through_a_constant_table(ip):
    """the reference's golden for a tuple entry, through a table that repeats its exposure time, within 1e-5 of full scale"""
    g = load_golden('correct_u16_legacy_dark')
    H, W = g['raw'].shape
    cal = _tuple_cal(ip, H, W, g['offs'], g['ascent'], lens=False)
    t = float(g['exposure_time'])
    got = cal.correct_batch(np.stack([g['raw']] * 3), exposure_time=[t] * 3, out_dtype=np.float64)
    for i in range(3):
        assert np.abs(got[i] - g['out']).max() / 65535.0 < 1e-5, i


def test_elbin_stack_with_its_labels(ip):
    """an .elbin file image through correct_file_bytes (headers skipped in K1's load) with the times its labels give,
    frame by frame equal to correct() of the decoded frame with that time"""
    from imgprocessor_b200 import reader
    lay = reader.elbin_layout(ELBIN_FILE)
    frames, labels = reader.elbin(ELBIN_FILE)
    ts = [l['exposure time[s]'] for l in labels]
    n, (H, W) = lay['frames'], lay['shape']
    offs, asc = _line(H, W, 11)
    asc *= 0.2
    flat = _calibration(H, W, 11)[1]
    cal = _tuple_cal(ip, H, W, offs, asc, flat, lens=False)
    want = _correct_each(cal, frames, ts)
    e = ip.engine_mod.get_engine(H, W)
    try:
        e.set_dark(offs, asc, 0.0, 16)
        e.set_flat(flat)
        e.set_dark_exposures(ts)
        buf = torch.from_numpy(lay['bytes']).cuda()
        got = _host(e.correct_file_bytes(buf, lay['offset'], n, gap=lay['gap'], use_lens=False, out_dtype=torch.float64))
        assert _same(got, want)
    finally:
        e.set_dark(None)
        e.set_flat(None)


# ---------------------------------------------------------------------------------------------- 7. full size
def test_full_size_against_scalar_groups(ip):
    """33 uint16 4096x3000 frames with three exposure times (groups of 16 and a one-frame group, overlap on, the moderate
    lens) equal one scalar call per exposure-time group"""
    H, W, n = 3000, 4096, 33
    e = ip.engine_mod.get_engine(H, W)
    offs = synth.dark_map(H, W)
    asc = np.full((H, W), 3.25, np.float32)
    e.set_dark(offs, asc, 0.0, 16)
    e.set_flat(synth.flat_map(H, W))
    _lens(e, H, W)
    try:
        d = torch.device('cuda', torch.cuda.current_device())
        raw = synth.scene_torch(n, H, W, 17, d)
        ts = np.resize([1.2, 4.8, 0.3], n)
        e.set_dark_exposures(ts)
        got = e.correct_batch(raw)
        for t in np.unique(ts):
            idx = torch.from_numpy(np.flatnonzero(ts == t)).to(d)
            e.set_dark(offs, asc, float(t), 16)
            want = e.correct_batch(raw.index_select(0, idx).contiguous())
            torch.cuda.synchronize()
            assert torch.equal(got.index_select(0, idx), want), t
    finally:
        e.set_dark(None)
        e.set_flat(None)
        e.set_lens(None, None, None)
