"""The perspective warp as the chain's last stage (IMGCORR_DO_PERSPECTIVE, Engine.set_perspective,
CameraCalibration.correct_batch(perspective=...)) against the oracle, frame by frame and bit for bit.

The oracle is the float32 chain of test_gpu_chain (oracle.models.correct_chain_f32 with the engine's own maps), cropped
to the K2 window and widened to float64 where the call returns float64, followed by oracle.warp.warp_perspective_model
(Lanczos4, forward map, constant border; divide_by= for the tilt factor).  Every comparison is
np.array_equal(..., equal_nan=True).  The full-size case compares against the two-step device composition (correct_batch,
then Engine.warp_perspective, which test_gpu_warp pins to the oracle): the numpy model is too slow at 12 Mpx."""
import contextlib
import io

import numpy as np
import pytest

from imgprocessor_b200 import synth
from oracle import warp as warp_model
from test_gpu_chain import (SPIN_CYCLES, _calibration, _crop, _dev, _file_image, _flags, _frames, _host, _lens, _maps,
                            _Options, _oracle, _same, ip)  # noqa: F401  (ip is a fixture)

pytestmark = pytest.mark.gpu

torch = pytest.importorskip('torch')

QUADS = {   # source quads as fractions of the chain frame's (width, height), mapped onto the whole destination
    'mild': [[0.02, 0.015], [0.985, 0.03], [0.97, 0.98], [0.01, 0.96]],
    'strong': [[0.2, 0.1], [0.85, 0.25], [0.95, 0.9], [0.05, 0.75]],
    'outside': [[-0.15, -0.1], [1.1, 0.05], [0.9, 1.2], [0.1, 0.9]],       # parts of the destination map outside the source
}


def _homography(src, dst):
    """the 3x3 matrix that maps the four points `src` onto `dst` (cv2.getPerspectiveTransform's linear system)"""
    A, b = [], []
    for (x, y), (u, v) in zip(src, dst):
        A.append([x, y, 1, 0, 0, 0, -u * x, -u * y])
        A.append([0, 0, 0, x, y, 1, -v * x, -v * y])
        b += [u, v]
    return np.append(np.linalg.solve(np.array(A, float), np.array(b, float)), 1.0).reshape(3, 3)


def _dsize(h, w, kind='same'):
    return {'same': (w, h), 'larger': (w + 37, h + 21), 'smaller': (w // 2 + 3, h // 2 + 1)}[kind]


def _stage(h, w, quad='mild', dsize='same'):
    """(M, dsize) that rectifies a quad of an h x w chain frame onto the whole destination"""
    dw, dh = _dsize(h, w, dsize)
    src = [(fx * w, fy * h) for fx, fy in QUADS[quad]]
    return _homography(src, [(0, 0), (dw, 0), (dw, dh), (0, dh)]), (dw, dh)


def _warp(chain_frame, M, dsize, border, tilt=None):
    return warp_model.warp_perspective_model(chain_frame, M, dsize, 'lanczos4', False, border, divide_by=tilt)


class _Want(object):
    """the oracle for one set of frames and calibration: chain frames cached per (frame, lens)"""

    def __init__(self, raw, dark, flat, maps, thr=0.1):
        self.raw, self.dark, self.flat, self.maps, self.thr = raw, dark, flat, maps, thr
        self.chain = {}

    def __call__(self, i, M, dsize, border, window=None, odt=np.float32, lens=True, tilt=None):
        if (i, lens) not in self.chain:
            self.chain[i, lens] = _oracle(self.raw[i], self.dark, self.flat, self.thr, 3, self.maps if lens else None)
        return _warp(_crop(self.chain[i, lens], window, odt), M, dsize, border, tilt)


def _setup(ip, H, W, seed):
    e = ip.engine_mod.get_engine(H, W)
    dark, flat = _calibration(H, W, seed)
    e.set_dark(dark)
    e.set_flat(flat)
    roi = _lens(e, H, W)
    return e, dark, flat, roi, _maps(e)


def _src_shape(e, window, lens=True):
    return (window[3], window[2]) if (lens and window) else (e.H, e.W)


# ---------------------------------------------------------------------------------------------- 1. the device chain
@pytest.mark.parametrize('shape', [(96, 256), (70, 251)])       # K3's staged tiles (float32 rows of 16-byte multiples) / not
@pytest.mark.parametrize('dtype', [np.uint8, np.uint16, np.float32])
def test_device_chain_with_perspective_vs_oracle(ip, shape, dtype):
    """6 frames in one group through correct_batch with DO_PERSPECTIVE.  Base: lens on, full frame, float32 out, the mild
    quad onto a destination of the source's size, border 2.5.  Each other axis is varied alone: no lens, the roi window,
    float64 out, float64 out with the roi, the strong quad, a quad partly outside the source, a larger and a smaller
    destination."""
    H, W = shape
    n = 6
    L = ip.lib_mod
    e, dark, flat, roi, maps = _setup(ip, H, W, 3)
    raw = _frames(H, W, n, 40, dtype)
    want = _Want(raw, dark, flat, maps)
    dev = _dev(raw)
    base = dict(lens=True, window=None, odt=np.float32, quad='mild', dsize='same')
    cases = [base] + [dict(base, **v) for v in (
        {'lens': False}, {'window': roi}, {'odt': np.float64}, {'odt': np.float64, 'window': roi}, {'quad': 'strong'},
        {'quad': 'outside'}, {'dsize': 'larger'}, {'dsize': 'smaller'})]
    try:
        for c in cases:
            M, dsize = _stage(*_src_shape(e, c['window'], c['lens']), quad=c['quad'], dsize=c['dsize'])
            e.set_perspective(M, dsize, 2.5)
            tdt = torch.float64 if c['odt'] == np.float64 else torch.float32
            out = e.correct_batch(dev, threshold=0.1, ksize=3, flags=_flags(L, 0.1) | L.DO_PERSPECTIVE, use_lens=c['lens'],
                                  window=c['window'], out_dtype=tdt)
            assert tuple(out.shape) == (n, dsize[1], dsize[0])
            got = _host(out)
            for i in range(n):
                assert _same(got[i], want(i, M, dsize, 2.5, c['window'], c['odt'], c['lens'])), (c, i)
    finally:
        e.set_perspective(None, None)


# ---------------------------------------------------------------------------------------------- 2. group seams
def test_group_seams_vs_oracle(ip):
    """11 frames in groups of 4 (4 + 4 + 3), overlap on and off, every frame: with the lens in float32 (K1 of the next
    group overlaps K2, division and K3 of this one) and without it in float64 (K1 writes the warp source)"""
    H, W, n = 96, 256, 11
    L = ip.lib_mod
    e, dark, flat, roi, maps = _setup(ip, H, W, 5)
    raw = _frames(H, W, n, 60, np.uint16)
    want = _Want(raw, dark, flat, maps)
    dev = _dev(raw)
    try:
        with _Options(ip, e) as o:
            o.set(L.OPT_CHAIN_GROUP, 4)
            for lens, window, tdt, odt in ((True, roi, torch.float32, np.float32), (False, None, torch.float64, np.float64)):
                M, dsize = _stage(*_src_shape(e, window, lens), quad='strong', dsize='larger')
                e.set_perspective(M, dsize, 0.0)
                for overlap in (1, 0):
                    o.set(L.OPT_CHAIN_OVERLAP, overlap)
                    got = _host(e.correct_batch(dev, flags=_flags(L, 0.1) | L.DO_PERSPECTIVE, use_lens=lens, window=window,
                                                out_dtype=tdt))
                    for i in range(n):
                        assert _same(got[i], want(i, M, dsize, 0.0, window, odt, lens)), (lens, overlap, i)
    finally:
        e.set_perspective(None, None)


# ---------------------------------------------------------------------------------------------- 3. tilt factor and refusals
def test_tilt_factor_and_refusals(ip):
    """the tilt-factor division in float64 before the warp, with the roi window and without a lens, 7 frames in groups
    of 3; then what the library refuses: float32 output with a tilt, a tilt of another shape, the bit without a stage,
    and the bit after a rejected set_perspective"""
    H, W, n = 96, 256, 7
    L = ip.lib_mod
    e, dark, flat, roi, maps = _setup(ip, H, W, 7)
    raw = _frames(H, W, n, 80, np.uint16)
    want = _Want(raw, dark, flat, maps)
    dev = _dev(raw)
    fl = _flags(L, 0.1) | L.DO_PERSPECTIVE
    rng = np.random.default_rng(3)
    try:
        with _Options(ip, e) as o:
            o.set(L.OPT_CHAIN_GROUP, 3)
            for lens, window in ((True, roi), (False, None)):
                sh = _src_shape(e, window, lens)
                tf = 0.5 + rng.random(sh)
                M, dsize = _stage(*sh, quad='mild', dsize='smaller')
                e.set_perspective(M, dsize, 1.5, tilt_factor=tf)
                got = _host(e.correct_batch(dev, flags=fl, use_lens=lens, window=window, out_dtype=torch.float64))
                for i in range(n):
                    assert _same(got[i], want(i, M, dsize, 1.5, window, np.float64, lens, tf)), (lens, i)
                got = e.correct_host(raw, flags=fl, use_lens=lens, window=window, out_dtype=np.float64)
                for i in range(n):
                    assert _same(got[i], want(i, M, dsize, 1.5, window, np.float64, lens, tf)), ('host', lens, i)
        # the tilt factor now has the full frame's shape
        with pytest.raises(L.ImgcorrError) as err:
            e.correct_batch(dev, flags=fl, out_dtype=torch.float32, use_lens=False)
        assert err.value.status == L.ERR_INVALID and 'F64' in str(err.value)
        with pytest.raises(L.ImgcorrError) as err:
            e.correct_batch(dev, flags=fl, window=roi, out_dtype=torch.float64)
        assert err.value.status == L.ERR_INVALID and 'tilt factor' in str(err.value)
        with pytest.raises(L.ImgcorrError) as err:
            e.correct_host(raw, flags=fl, window=roi, out_dtype=np.float64)
        assert err.value.status == L.ERR_INVALID
        e.set_perspective(None, None)
        for call in (lambda: e.correct_batch(dev, flags=fl), lambda: e.correct_host(raw, flags=fl)):
            with pytest.raises(L.ImgcorrError) as err:
                call()
            assert err.value.status == L.ERR_STATE
        # a rejected set_perspective leaves no stage behind, on either side of the binding: a chain call with the bit is
        # refused instead of writing frames of the previous destination shape into buffers sized for the chain frame
        for bad in (dict(dsize=(0, 40)), dict(dsize=(40, 40), tilt_factor=np.ones((0, 5)))):
            M, dsize = _stage(H, W, quad='mild', dsize='larger')
            e.set_perspective(M, dsize, 0.0)
            with pytest.raises(L.ImgcorrError) as err:
                e.set_perspective(M, **bad)
            assert err.value.status == L.ERR_INVALID and e.perspective_dsize is None
            for call in (lambda: e.correct_batch(dev, flags=fl), lambda: e.correct_host(raw, flags=fl)):
                with pytest.raises(L.ImgcorrError) as err:
                    call()
                assert err.value.status == L.ERR_STATE, bad
    finally:
        e.set_perspective(None, None)


# ---------------------------------------------------------------------------------------------- 4. host pipeline
@pytest.mark.parametrize('slots', [2, 3, 8])
def test_host_pipeline_with_perspective_vs_oracle(ip, slots):
    """correct_host with the stage: 37 small frames in chunks of 16, pageable / pinned input x pageable / pinned output
    into a destination of another size than the chain frame, and float64 out with the roi window"""
    H, W, n = 96, 160, 37
    L = ip.lib_mod
    e, dark, flat, roi, maps = _setup(ip, H, W, 13)
    raw = _frames(H, W, n, 200, np.uint16)
    want = _Want(raw, dark, flat, maps)
    pe = ip.engine_mod.pinned_empty
    fl = _flags(L, 0.1) | L.DO_PERSPECTIVE
    try:
        with _Options(ip, e) as o:
            o.set(L.OPT_HOST_SLOTS, slots)
            M, dsize = _stage(H, W, quad='strong', dsize='larger')
            e.set_perspective(M, dsize, 3.0)
            pin_in = pe(raw.shape, np.uint16)
            pin_in[...] = raw
            oshape = (n, dsize[1], dsize[0])
            for src in (raw, pin_in):
                for pinned_out in (False, True):
                    out = pe(oshape, np.float32) if pinned_out else np.empty(oshape, np.float32)
                    out[...] = -1
                    got = e.correct_host(src, out=out, flags=fl)
                    assert got is out
                    for i in range(n):
                        assert _same(got[i], want(i, M, dsize, 3.0)), (src is pin_in, pinned_out, i)
            M, dsize = _stage(roi[3], roi[2], quad='outside', dsize='smaller')
            e.set_perspective(M, dsize, 0.0)
            got = e.correct_host(raw, flags=fl, window=roi, out_dtype=np.float64)
            for i in range(n):
                assert _same(got[i], want(i, M, dsize, 0.0, roi, np.float64)), ('f64 roi', i)
    finally:
        e.set_perspective(None, None)


# ---------------------------------------------------------------------------------------------- 5. file bytes
def test_file_bytes_with_perspective_vs_oracle(ip):
    """correct_file_bytes on big-endian frames with a 32-byte header and 20-byte gaps, 8 frames in groups of 5"""
    H, W, n = 70, 250, 8
    L = ip.lib_mod
    e, dark, flat, roi, maps = _setup(ip, H, W, 11)
    raw = _frames(H, W, n, 160, np.uint16)
    want = _Want(raw, dark, flat, maps)
    buf = _dev(_file_image(raw, 32, 20, big_endian=True))
    M, dsize = _stage(H, W, quad='mild', dsize='larger')
    try:
        with _Options(ip, e) as o:
            o.set(L.OPT_CHAIN_GROUP, 5)
            e.set_perspective(M, dsize, 0.5)
            got = _host(e.correct_file_bytes(buf, 32, n, gap=20, big_endian=True, dtype=torch.uint16,
                                             flags=_flags(L, 0.1) | L.DO_PERSPECTIVE))
            for i in range(n):
                assert _same(got[i], want(i, M, dsize, 0.5)), i
    finally:
        e.set_perspective(None, None)


# ---------------------------------------------------------------------------------------------- 6. public API
def _calibrated(ip, H, W):
    dark, flat = _calibration(H, W, 9)
    cal = ip.CameraCalibration()
    cal.addDarkCurrent(dark)
    cal.addFlatField(flat)
    lens = ip.LensDistortion({})
    lens.setCameraParams(*synth.lens_moderate(H, W))
    lens._coeffs['shape'] = (H, W)
    cal.addLens(lens)
    return cal


def test_camera_calibration_correct_batch_with_perspective(ip):
    """cal.correct_batch(frames, perspective=pc, out_dtype=float64)[i] == pc.correct(cal.correct(frames[i])) for keep_size
    True and False, with and without the tilt factor; host frames, CUDA tensors, and two contexts on one device
    (devices=[0, 0]) or every GPU of the machine"""
    from imgprocessor_b200.camera import PerspectiveCorrection
    H, W, n = 96, 256, 5
    cal = _calibrated(ip, H, W)
    raw = _frames(H, W, n, 140, np.uint16)
    ngpu = torch.cuda.device_count()
    for keep_size in (True, False):
        for tilt in (False, True):
            quiet = contextlib.redirect_stdout(io.StringIO())
            with quiet:
                ref = [cal.correct(raw[i], keep_size=keep_size) for i in range(n)]
            sh = ref[0].shape
            assert (sh == (H, W)) == keep_size                      # keep_size=False: the roi crop
            M, dsize = _stage(*sh, quad='mild', dsize='larger')
            pc = PerspectiveCorrection(sh, new_size=(dsize[1], dsize[0]), do_correctIntensity=tilt,
                                       cv2_opts={'borderValue': 0.75})
            pc.setReference(M)
            if tilt:
                pc.setTiltFactor(0.5 + np.random.default_rng(4).random(sh))
            with contextlib.redirect_stdout(io.StringIO()):
                want = np.stack([pc.correct(r) for r in ref])
            got = cal.correct_batch(raw, keep_size=keep_size, perspective=pc, out_dtype=np.float64)
            assert _same(got, want), (keep_size, tilt)
            got = _host(cal.correct_batch(_dev(raw), keep_size=keep_size, perspective=pc, out_dtype=torch.float64))
            assert _same(got, want), ('tensor', keep_size, tilt)
            for devices in ([0, 0], list(range(ngpu)) if ngpu >= 2 else None):
                if devices is not None:
                    got = cal.correct_batch(raw, keep_size=keep_size, perspective=pc, out_dtype=np.float64, devices=devices)
                    assert _same(got, want), (devices, keep_size, tilt)
            if tilt:
                with pytest.raises(ValueError, match='float64'):
                    cal.correct_batch(raw, keep_size=keep_size, perspective=pc)
    # float32 output: the float32 chain frame warped in float32
    pc = PerspectiveCorrection((H, W), new_size=(H - 10, W - 20))
    M, _ = _stage(H, W, quad='strong', dsize='same')
    pc.setReference(M)
    maps = _maps(ip.engine_mod.get_engine(H, W))
    dark, flat = _calibration(H, W, 9)
    got = cal.correct_batch(raw, perspective=pc)
    for i in range(n):
        assert _same(got[i], _warp(_oracle(raw[i], dark, flat, 0.1, 3, maps), M, (W - 20, H - 10), 0.0)), i


# ---------------------------------------------------------------------------------------------- 7. two streams
def test_two_streams_with_perspective_share_one_context(ip):
    """two correct_batch calls with the stage on two torch streams, released together by one event after a spin: the
    second waits for the first's scratch (K1 halves and warp source) instead of overwriting it"""
    H, W, n = 128, 256, 12
    L = ip.lib_mod
    e, dark, flat, roi, maps = _setup(ip, H, W, 19)
    dev = torch.device('cuda', torch.cuda.current_device())
    a = synth.scene_torch(n, H, W, 31, dev)
    b = synth.scene_torch(n, H, W, 32, dev)
    wa, wb = _Want(_host(a), dark, flat, maps), _Want(_host(b), dark, flat, maps)
    M, dsize = _stage(H, W, quad='strong', dsize='same')
    fl = _flags(L, 0.1) | L.DO_PERSPECTIVE
    sa, sb = torch.cuda.Stream(), torch.cuda.Stream()
    try:
        e.set_perspective(M, dsize, 0.0)
        with _Options(ip, e) as o:
            o.set(L.OPT_CHAIN_GROUP, 4)
            e.correct_batch(a[:2], flags=fl)                     # allocation and caches outside the race
            bad = []
            for overlap in (0, 1):
                o.set(L.OPT_CHAIN_OVERLAP, overlap)
                go = torch.cuda.Event()
                torch.cuda.synchronize()
                with torch.cuda.stream(sa):
                    torch.cuda._sleep(SPIN_CYCLES)
                    go.record(sa)
                    out_a = e.correct_batch(a, flags=fl)
                with torch.cuda.stream(sb):
                    sb.wait_event(go)
                    out_b = e.correct_batch(b, flags=fl)
                torch.cuda.synchronize()
                for tag, out, want in (('a', _host(out_a), wa), ('b', _host(out_b), wb)):
                    bad += [(overlap, tag, i) for i in range(n) if not _same(out[i], want(i, M, dsize, 0.0))]
        assert not bad, bad
    finally:
        e.set_perspective(None, None)


# ---------------------------------------------------------------------------------------------- 8. nothing else changes
def test_calls_without_the_bit_are_unchanged(ip):
    """after set_perspective (with a tilt factor), a chain call without the bit gives the bits and the launch count of
    the same call on a fresh context: lens with group seams and overlap, no lens, the host pipeline"""
    H, W, n = 96, 256, 11
    L = ip.lib_mod
    dark, flat = _calibration(H, W, 21)
    raw = _frames(H, W, n, 220, np.uint16)
    dev = _dev(raw)
    results = []
    for with_stage in (False, True):
        e = ip.engine_mod.Engine(H, W)
        try:
            e.set_dark(dark)
            e.set_flat(flat)
            _lens(e, H, W)
            e.set_option(L.OPT_CHAIN_GROUP, 4)
            if with_stage:
                M, dsize = _stage(H, W)
                e.set_perspective(M, dsize, 1.0, tilt_factor=np.ones((H, W)))
            r = []
            for kw in (dict(), dict(use_lens=False), dict(out_dtype=torch.float64)):
                before = e.launch_count
                r.append((_host(e.correct_batch(dev, **kw)), e.launch_count - before))
            before = e.launch_count
            r.append((e.correct_host(raw), e.launch_count - before))
            results.append(r)
        finally:
            e.close()
    for (g0, l0), (g1, l1) in zip(*results):
        assert _same(g1, g0) and l1 == l0


# ---------------------------------------------------------------------------------------------- 9. full size
def test_full_size_across_a_group_seam(ip):
    """17 uint16 4096x3000 frames with the moderate lens (groups of 16 + 1, overlap on) through the stage into a
    4000x2900 destination, against correct_batch followed by Engine.warp_perspective; full frame and roi window"""
    H, W, n = 3000, 4096, 17
    L = ip.lib_mod
    e = ip.engine_mod.get_engine(H, W)
    e.set_dark(synth.dark_map(H, W))
    e.set_flat(synth.flat_map(H, W))
    roi = _lens(e, H, W)
    src = synth.scene_torch(n, H, W, 7, torch.device('cuda', torch.cuda.current_device()))
    try:
        for window in (None, roi):
            sh = _src_shape(e, window)
            dsize = (4000, 2900)
            M = _homography([(fx * sh[1], fy * sh[0]) for fx, fy in QUADS['mild']], [(0, 0), (4000, 0), (4000, 2900), (0, 2900)])
            e.set_perspective(M, dsize, 0.0)
            got = e.correct_batch(src, flags=_flags(L, 0.1) | L.DO_PERSPECTIVE, window=window)
            two_step = e.warp_perspective(e.correct_batch(src, window=window), M, dsize)
            assert tuple(got.shape) == (n, 2900, 4000)
            bad = [i for i in range(n) if not torch.equal(got[i], two_step[i])]
            assert not bad, (window, bad)
            del got, two_step
    finally:
        e.set_perspective(None, None)
        e.set_lens(None, None, None)
