"""The K1 -> K2 chain as users call it (Engine.correct_batch, Engine.correct_host, Engine.correct_file_bytes,
CameraCalibration.correct_batch) against the float32 oracle chain, frame by frame and bit for bit.

The oracle's maps are the engine's own (undistort_maps(); test_maps_vs_reference_golden pins their fixed-point
coordinates to OpenCV's), so every comparison is np.array_equal(..., equal_nan=True).  Covered here and nowhere else:
uint8 / float32 frames through the chain, threshold 0 (NaN and inf reach K2), partial calibrations, 5x5 in batches,
batches that cross chain-group seams, big-endian and gapped ingest across groups, the host pipeline's ring slots and
chunking against the oracle (not against the device chain), and one context used from several streams."""
import numpy as np
import pytest

from imgprocessor_b200 import synth
from oracle import bands, models, refpath

pytestmark = pytest.mark.gpu

torch = pytest.importorskip('torch')

SPIN_CYCLES = 600_000_000          # torch.cuda._sleep: about 0.3 s of device time


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


def _host(t):
    torch.cuda.synchronize()
    return t.cpu().numpy()


def _same(got, want):
    return got.shape == want.shape and got.dtype == want.dtype and np.array_equal(got, want, equal_nan=True)


def _maps(e):
    mx, my = e.undistort_maps()
    return _host(mx), _host(my)


def _flags(lib, thr, cal='df'):
    f = (lib.DO_DARK if 'd' in cal else 0) | (lib.DO_FLAT if 'f' in cal else 0)
    return f | (lib.DO_NAN_TO_NUM if thr > 0 else 0)


def _calibration(H, W, seed):
    """dark and flat maps; the flat holds a zero, a denormal and negative values (two of them on frame corners)"""
    dark = synth.dark_map(H, W, seed)
    flat = synth.flat_map(H, W, seed + 1, p_zero=5e-3)
    flat[0, 0] = 0.0
    flat[3, 5] = np.float32(1e-42)
    flat[H - 1, W - 1] = np.float32(-1e-40)
    flat[H // 2, 0] = -0.5
    return dark, flat


def _frames(H, W, n, seed, dtype):
    """n frames; float32 ones carry NaN, +-inf and +-3e38 on the first / last rows and columns and inside, and two 6x6
    blocks of +-3e38 (a corner, the bottom edge) that the median keeps, so that K2 blends +-FLT_MAX there as well"""
    f = np.stack([synth.scene(H, W, seed + i, dtype) for i in range(n)])
    if f.dtype == np.float32:
        edge = [np.nan, np.inf, -np.inf, 3e38, -3e38]
        for i in range(n):
            f[i, :6, :6] = 3e38
            f[i, H - 6:, W // 2 + i:W // 2 + i + 6] = -3e38
            for k, v in enumerate(edge):
                j = (i + k) % len(edge)
                f[i, 0, (7 * k + i) % W] = edge[j]
                f[i, H - 1, (11 * k + 2 * i) % W] = edge[(j + 1) % 5]
                f[i, (5 * k + i) % H, 0] = edge[(j + 2) % 5]
                f[i, (13 * k + i) % H, W - 1] = edge[(j + 3) % 5]
                f[i, H // 2 + k, W // 3 + i] = edge[(j + 4) % 5]
    return f


def _lens(e, H, W, strong=False):
    p = synth.lens_strong(H, W) if strong else synth.lens_moderate(H, W)
    K, d = synth.camera_matrix(p), synth.dist_coeffs(p)
    _, _, P, roi = refpath.undistort_rectify_map(K, d, W, H)
    e.set_lens(K, d, P)
    return tuple(int(v) for v in roi)


class _Options(object):
    """set engine options inside a block; the library defaults are restored when it ends, also on failure"""

    def __init__(self, ip, e):
        L = ip.lib_mod
        self.e = e
        self.defaults = {L.OPT_CHAIN_GROUP: 16, L.OPT_CHAIN_OVERLAP: 1, L.OPT_HOST_SLOTS: 4, L.OPT_K1_VARIANT: 0,
                         L.OPT_RAW_BIG_ENDIAN: 0, L.OPT_RAW_FRAME_GAP: 0}

    def set(self, key, value):
        self.e.set_option(key, value)

    def __enter__(self):
        return self

    def __exit__(self, *a):
        for k, v in self.defaults.items():
            self.e.set_option(k, v)


def _oracle(raw, dark, flat, thr, ksize, maps, border=0.0, cal='df'):
    want, _ = models.correct_chain_f32(raw, dark if 'd' in cal else None, flat if 'f' in cal else None, thr, ksize,
                                       border_value=border, mapxy=maps)
    return want


def _crop(a, window, dtype=np.float32):
    if window is not None:
        x, y, w, h = window
        a = a[y:y + h, x:x + w]
    return a.astype(dtype)


# ---------------------------------------------------------------------------------------------- a. chain matrix
@pytest.mark.parametrize('shape', [(83, 256), (130, 344), (70, 250)])
@pytest.mark.parametrize('thr', [0.1, 0.0])
@pytest.mark.parametrize('ksize', [3, 5])
@pytest.mark.parametrize('dtype', [np.uint8, np.uint16, np.float32])
def test_chain_matrix_vs_oracle(ip, shape, thr, ksize, dtype):
    """11 frames through correct_batch against the oracle, frame by frame.  Base: groups of 5 (5 + 5 + 1 frames: the pair
    kernel, the one-frame kernel, and a one-frame group that reads K2's coordinate cache), overlap on, full frame, float32
    out, border 0, dark + flat.  Each other axis is varied alone: one group of 11, overlap off, the roi window, float64
    out, border 7.5, flat only, dark only, no lens (K1 only)."""
    H, W = shape
    n = 11
    L = ip.lib_mod
    e = ip.engine_mod.get_engine(H, W)
    dark, flat = _calibration(H, W, 3)
    raw = _frames(H, W, n, 40, dtype)
    e.set_dark(dark)
    e.set_flat(flat)
    roi = _lens(e, H, W)
    maps = _maps(e)
    dev = _dev(raw)
    oracle = {}

    def want(i, cal='df', border=0.0, lens=True):
        k = (i, cal, border, lens)
        if k not in oracle:
            oracle[k] = _oracle(raw[i], dark, flat, thr, ksize, maps if lens else None, border, cal)
        return oracle[k]

    base = dict(group=5, overlap=1, window=None, out_dtype=torch.float32, border=0.0, cal='df', lens=True)
    cases = [base] + [dict(base, **v) for v in (
        {'group': 16}, {'overlap': 0}, {'window': roi}, {'out_dtype': torch.float64}, {'border': 7.5},
        {'cal': 'f'}, {'cal': 'd'}, {'lens': False})]
    with _Options(ip, e) as o:
        for c in cases:
            o.set(L.OPT_CHAIN_GROUP, c['group'])
            o.set(L.OPT_CHAIN_OVERLAP, c['overlap'])
            out = e.correct_batch(dev, threshold=thr, ksize=ksize, flags=_flags(L, thr, c['cal']), use_lens=c['lens'],
                                  border_value=c['border'], window=c['window'], out_dtype=c['out_dtype'])
            got = _host(out)
            odt = np.float64 if c['out_dtype'] == torch.float64 else np.float32
            for i in range(n):
                w = _crop(want(i, c['cal'], c['border'], c['lens']), c['window'], odt)
                assert _same(got[i], w), (c, i)


@pytest.mark.parametrize('dtype', [np.uint16, np.float32])
def test_chain_strong_lens_vs_oracle(ip, dtype):
    """the strong lens at 200x328: the larger staged K2 box, several frames per launch, both thresholds"""
    H, W, n = 200, 328, 7
    L = ip.lib_mod
    e = ip.engine_mod.get_engine(H, W)
    dark, flat = _calibration(H, W, 5)
    raw = _frames(H, W, n, 90, dtype)
    e.set_dark(dark)
    e.set_flat(flat)
    roi = _lens(e, H, W, strong=True)
    try:
        maps = _maps(e)
        for thr in (0.1, 0.0):
            for window in (None, roi):
                got = _host(e.correct_batch(_dev(raw), threshold=thr, ksize=3, flags=_flags(L, thr), window=window,
                                            border_value=2.5))
                for i in range(n):
                    assert _same(got[i], _crop(_oracle(raw[i], dark, flat, thr, 3, maps, 2.5), window)), (thr, window, i)
    finally:
        e.set_lens(None, None, None)


# ---------------------------------------------------------------------------------------------- b. ingest
@pytest.mark.parametrize('ksize', [3, 5])
@pytest.mark.parametrize('variant', [0, 3])
def test_big_endian_batches_vs_oracle(ip, ksize, variant):
    """big-endian uint16 frames, byte-swapped in K1's load: five frames in one launch of the streaming kernels (3x3 and
    5x5), through correct_batch and through correct_host from pageable and pinned buffers"""
    H, W, n = 83, 256, 5
    L = ip.lib_mod
    e = ip.engine_mod.get_engine(H, W)
    dark, flat = _calibration(H, W, 7)
    raw = _frames(H, W, n, 120, np.uint16)
    e.set_dark(dark)
    e.set_flat(flat)
    _lens(e, H, W)
    maps = _maps(e)
    want = [_oracle(raw[i], dark, flat, 0.1, ksize, maps) for i in range(n)]
    be = raw.astype('>u2')
    with _Options(ip, e) as o:
        o.set(L.OPT_K1_VARIANT, variant)
        with e.ingest(big_endian=True):
            got = _host(e.correct_batch(_dev(be.view(np.uint16)), threshold=0.1, ksize=ksize))
        for i in range(n):
            assert _same(got[i], want[i]), ('batch', i)
        pin = ip.engine_mod.pinned_empty(be.shape, '>u2')
        pin[...] = be
        for src in (be, pin):
            got = e.correct_host(src, threshold=0.1, ksize=ksize)
            for i in range(n):
                assert _same(got[i], want[i]), ('host', src is pin, i)
    # ingest options are per call: the next little-endian batch is read as such
    got = _host(e.correct_batch(_dev(raw), threshold=0.1, ksize=ksize))
    assert _same(got[0], want[0])


def test_big_endian_camera_calibration_correct_batch(ip):
    """CameraCalibration.correct_batch on a '>u2' host array at a TMA-eligible width"""
    H, W, n = 96, 256, 6
    dark, flat = _calibration(H, W, 9)
    raw = _frames(H, W, n, 140, np.uint16)
    cal = ip.CameraCalibration()
    cal.addDarkCurrent(dark)
    cal.addFlatField(flat)
    lens = ip.LensDistortion({})
    lens.setCameraParams(*synth.lens_moderate(H, W))
    lens._coeffs['shape'] = (H, W)
    cal.addLens(lens)
    got = cal.correct_batch(raw.astype('>u2'), threshold=0.1)
    maps = _maps(ip.engine_mod.get_engine(H, W))
    for i in range(n):
        assert _same(got[i], _oracle(raw[i], dark, flat, 0.1, 3, maps)), i
    native = cal.correct_batch(raw, threshold=0.1)
    assert _same(got, native)


def _file_image(raw, offset, gap, big_endian=False):
    """the bytes of a file holding `raw`'s frames: `offset` header bytes, then frames `gap` bytes apart; headers and gaps
    hold 0xA5 so that a read from them shows"""
    n = raw.shape[0]
    fb = raw[0].nbytes
    buf = np.full(offset + n * fb + (n - 1) * gap, 0xA5, np.uint8)
    data = raw.astype(raw.dtype.newbyteorder('>')) if big_endian else raw
    for i in range(n):
        p = offset + i * (fb + gap)
        buf[p:p + fb] = np.frombuffer(data[i].tobytes(), np.uint8)
    return buf


def test_frame_gap_across_groups_vs_oracle(ip):
    """correct_file_bytes with a 32-byte header and 20-byte per-frame gaps: 11 frames in groups of 5, so the gap enters the
    stride of every group after the first; little- and big-endian, with and without overlap"""
    H, W, n = 70, 250, 11
    L = ip.lib_mod
    e = ip.engine_mod.get_engine(H, W)
    dark, flat = _calibration(H, W, 11)
    raw = _frames(H, W, n, 160, np.uint16)
    e.set_dark(dark)
    e.set_flat(flat)
    _lens(e, H, W)
    maps = _maps(e)
    want = [_oracle(raw[i], dark, flat, 0.1, 3, maps) for i in range(n)]
    with _Options(ip, e) as o:
        o.set(L.OPT_CHAIN_GROUP, 5)
        for be in (False, True):
            buf = _dev(_file_image(raw, 32, 20, be))
            for overlap in (1, 0):
                o.set(L.OPT_CHAIN_OVERLAP, overlap)
                got = _host(e.correct_file_bytes(buf, 32, n, gap=20, big_endian=be, dtype=torch.uint16))
                for i in range(n):
                    assert _same(got[i], want[i]), (be, overlap, i)
        # a gap that is not a multiple of the sample size: refused by the wrapper and by the library
        with pytest.raises(ValueError):
            e.correct_file_bytes(buf, 32, n, gap=21, dtype=torch.uint16)
        o.set(L.OPT_RAW_FRAME_GAP, 3)
        with pytest.raises(L.ImgcorrError):
            e.correct_batch(_dev(raw), threshold=0.1)
        # host frames are passed as pixel blocks: a gap is refused
        o.set(L.OPT_RAW_FRAME_GAP, 20)
        with pytest.raises(L.ImgcorrError):
            e.correct_host(raw, threshold=0.1)
        o.set(L.OPT_RAW_FRAME_GAP, 0)
        # big-endian ingest is for integer frames only
        fbuf = _dev(_file_image(raw.astype(np.float32), 0, 0))
        with pytest.raises(L.ImgcorrError):
            e.correct_file_bytes(fbuf, 0, n, big_endian=True, dtype=torch.float32)
    got = _host(e.correct_batch(_dev(raw), threshold=0.1))          # options are back to dense little-endian frames
    assert _same(got[n - 1], want[n - 1])


# ---------------------------------------------------------------------------------------------- c. host pipeline
@pytest.mark.parametrize('slots', [2, 3, 8])
def test_host_pipeline_vs_oracle(ip, slots):
    """correct_host against the oracle: 37 small frames travel in chunks of 16 (more chunks than two slots, a ragged last
    chunk), pageable / pinned input x pageable / pinned output, float64 out with the roi window, uint8 and float32 input"""
    H, W, n = 96, 160, 37
    L = ip.lib_mod
    e = ip.engine_mod.get_engine(H, W)
    dark, flat = _calibration(H, W, 13)
    e.set_dark(dark)
    e.set_flat(flat)
    roi = _lens(e, H, W)
    maps = _maps(e)
    pe = ip.engine_mod.pinned_empty
    with _Options(ip, e) as o:
        o.set(L.OPT_HOST_SLOTS, slots)
        raw = _frames(H, W, n, 200, np.uint16)
        want = [_oracle(raw[i], dark, flat, 0.1, 3, maps) for i in range(n)]
        pin_in = pe(raw.shape, np.uint16)
        pin_in[...] = raw
        for src in (raw, pin_in):
            for pinned_out in (False, True):
                out = pe(raw.shape, np.float32) if pinned_out else np.empty(raw.shape, np.float32)
                out[...] = -1
                got = e.correct_host(src, out=out, threshold=0.1)
                assert got is out
                for i in range(n):
                    assert _same(got[i], want[i]), (src is pin_in, pinned_out, i)
        got = e.correct_host(raw, threshold=0.1, window=roi, out_dtype=np.float64)
        for i in range(n):
            assert _same(got[i], _crop(want[i], roi, np.float64)), ('f64 roi', i)
        for dtype, thr in ((np.uint8, 0.1), (np.float32, 0.1), (np.float32, 0.0)):
            r = _frames(H, W, n, 300, dtype)
            got = e.correct_host(r, threshold=thr, flags=_flags(L, thr))
            for i in range(n):
                assert _same(got[i], _oracle(r[i], dark, flat, thr, 3, maps)), (dtype, thr, i)


def _full_size_setup(ip, H, W):
    e = ip.engine_mod.get_engine(H, W)
    dark, flat = synth.dark_map(H, W), synth.flat_map(H, W)
    e.set_dark(dark)
    e.set_flat(flat)
    _lens(e, H, W)
    return e, dark, flat, _maps(e)


def _check_bands(got, raw, dark, flat, maps, ksize, what):
    for r0, r1 in bands.default_bands(raw.shape[0]):
        want = bands.chain_band(raw, dark, flat, maps[0], maps[1], r0, r1, 0.1, ksize)
        assert _same(got[r0:r1], want), (what, r0, r1)


def test_host_pipeline_full_size_vs_oracle(ip):
    """five 3000x4096 uint16 frames through two ring slots, one frame per slot"""
    H, W, n = 3000, 4096, 5
    L = ip.lib_mod
    e, dark, flat, maps = _full_size_setup(ip, H, W)
    try:
        raw = _host(synth.scene_torch(n, H, W, 21, torch.device('cuda', torch.cuda.current_device())))
        with _Options(ip, e) as o:
            o.set(L.OPT_HOST_SLOTS, 2)
            got = e.correct_host(raw, threshold=0.1)
        for i in range(n):
            _check_bands(got[i], raw[i], dark, flat, maps, 3, i)
    finally:
        e.set_lens(None, None, None)


# ---------------------------------------------------------------------------------------------- d. headline configuration
def test_headline_batch_across_group_seams(ip):
    """33 uint16 4096x3000 frames with the defaults (groups of 16, overlap on): frames on both sides of each group seam
    and the one-frame last group, then 5 frames with the 5x5 median"""
    H, W = 3000, 4096
    e, dark, flat, maps = _full_size_setup(ip, H, W)
    try:
        src = synth.scene_torch(33, H, W, 7, torch.device('cuda', torch.cuda.current_device()))
        out = e.correct_batch(src)
        for i in (0, 15, 16, 31, 32):
            _check_bands(_host(out[i]), _host(src[i]), dark, flat, maps, 3, i)
        del out
        out = e.correct_batch(src[:5], ksize=5)
        for i in (0, 4):
            _check_bands(_host(out[i]), _host(src[i]), dark, flat, maps, 5, ('5x5', i))
    finally:
        e.set_lens(None, None, None)


# ---------------------------------------------------------------------------------------------- e. one context, several streams
def test_host_pipeline_waits_for_earlier_batch(ip):
    """correct_host after a correct_batch that has not run yet (a spin holds the caller's stream): both use the
    context's K1 scratch, so the host pipeline must wait for the earlier batch — when it returns, the caller's stream is
    idle — and both results equal the oracle"""
    H, W, n = 128, 256, 9
    e = ip.engine_mod.get_engine(H, W)
    dark, flat = _calibration(H, W, 17)
    e.set_dark(dark)
    e.set_flat(flat)
    _lens(e, H, W)
    maps = _maps(e)
    a = _frames(H, W, n, 400, np.uint16)
    b = _frames(H, W, n, 500, np.uint16)
    dev = _dev(a)
    # first calls allocate the scratch, the ring slots and K2's caches (allocation synchronises the device)
    e.correct_batch(dev, threshold=0.1)
    e.correct_host(b, threshold=0.1)
    torch.cuda.synchronize()
    torch.cuda._sleep(SPIN_CYCLES)
    out_a = e.correct_batch(dev, threshold=0.1)
    out_b = e.correct_host(b, threshold=0.1)
    assert torch.cuda.current_stream().query(), 'correct_host returned before the earlier batch had used the scratch'
    got_a = _host(out_a)
    for i in range(n):
        assert _same(got_a[i], _oracle(a[i], dark, flat, 0.1, 3, maps)), ('batch', i)
        assert _same(out_b[i], _oracle(b[i], dark, flat, 0.1, 3, maps)), ('host', i)


def test_batches_on_two_streams_share_one_context(ip):
    """two correct_batch calls on two torch streams, released together by one event after a spin: the second waits for
    the first's K1 scratch instead of overwriting it.  Without overlap both calls alternate K1 and K2 on the same two
    buffers; with overlap their K1s share the internal stream and only the tail of the first call is exposed."""
    H, W, n = 512, 1024, 24
    L = ip.lib_mod
    e = ip.engine_mod.get_engine(H, W)
    dark, flat = _calibration(H, W, 19)
    e.set_dark(dark)
    e.set_flat(flat)
    _lens(e, H, W)
    maps = _maps(e)
    dev = torch.device('cuda', torch.cuda.current_device())
    a = synth.scene_torch(n, H, W, 31, dev)
    b = synth.scene_torch(n, H, W, 32, dev)
    sa, sb = torch.cuda.Stream(), torch.cuda.Stream()
    ra, rb = _host(a), _host(b)
    want = {(tag, i): _oracle(raw[i], dark, flat, 0.1, 3, maps) for tag, raw in (('a', ra), ('b', rb)) for i in range(n)}
    with _Options(ip, e) as o:
        o.set(L.OPT_CHAIN_GROUP, 1)
        e.correct_batch(a[:2])                                   # allocation and caches outside the race
        bad = []
        for overlap in (0, 1):
            o.set(L.OPT_CHAIN_OVERLAP, overlap)
            go = torch.cuda.Event()
            torch.cuda.synchronize()
            with torch.cuda.stream(sa):
                torch.cuda._sleep(SPIN_CYCLES)
                go.record(sa)
                out_a = e.correct_batch(a)
            with torch.cuda.stream(sb):
                sb.wait_event(go)
                out_b = e.correct_batch(b)
            torch.cuda.synchronize()
            for tag, out in (('a', _host(out_a)), ('b', _host(out_b))):
                bad += [(overlap, tag, i) for i in range(n) if not _same(out[i], want[tag, i])]
    assert not bad, bad
