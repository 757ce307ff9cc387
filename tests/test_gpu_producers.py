"""Kernel K5 (csrc/k5_producers.cu) and Engine.median3x3 against plain float64 references, bit for bit, at full size and at
the edges: the calibration-map producers behind flatFieldFromCloseDistance and getLinearityFunction.

The K5 kernels are grid-stride loops over at most sm_count * 16 blocks of 256 threads.  The large cases use
2 * cap + 37 outputs (cap = that thread count on this device), so every loop runs at least twice and its last pass is
partial.  The kernels use IEEE float64 operations in the reference's order, so results match bit for bit, and the sign
of a zero result must match too, with two exceptions compared by value only.  The luminance of gray3 is numpy's sum
over the channel axis, which turns a sum of three -0.0 into +0.0.  The sign of a zero median is whichever zero scipy's
selection picks; NaN inputs to median3x3 are excluded for the same reason."""
import numpy as np
import pytest
from scipy.ndimage import median_filter

from oracle import producers

pytestmark = pytest.mark.gpu

torch = pytest.importorskip('torch')

FLT_MAX = float(np.finfo(np.float32).max)


@pytest.fixture(scope='module')
def engine():
    if not torch.cuda.is_available():
        pytest.skip('needs a CUDA device')
    from imgprocessor_b200 import engine
    return engine


@pytest.fixture(scope='module')
def cap(engine):
    """threads of one pass of the K5 grid-stride loops (grid_for() in k5_producers.cu)"""
    return torch.cuda.get_device_properties(0).multi_processor_count * 16 * 256


@pytest.fixture(scope='module')
def k5(engine):
    return engine.get_engine(16, 16)             # K5 takes free shapes: the engine supplies the device


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _same(got, want, signed_zero=True):
    got = got.cpu().numpy() if isinstance(got, torch.Tensor) else np.asarray(got)
    want = np.asarray(want)
    if got.shape != want.shape or got.dtype != want.dtype or not np.array_equal(got, want, equal_nan=True):
        return False
    keep = ~np.isnan(want)
    return not signed_zero or np.array_equal(np.signbit(got[keep]), np.signbit(want[keep]))


def _random(rng, dtype, shape, scale=1000.0):
    if dtype == np.uint8:
        return rng.integers(0, 256, shape, dtype=np.uint8)
    if dtype == np.uint16:
        return rng.integers(0, 65536, shape, dtype=np.uint16)
    return rng.normal(0, scale, shape).astype(dtype)


# ---- A. stack_mean: imgAverage(frames) [- minus] [-> toGray] -------------------------------------------------------------
def _stack_ref(frames, minus=None, gray3=False):
    with np.errstate(all='ignore'):
        x = producers.img_average(list(frames))
        if minus is not None:
            x -= minus
        if gray3:
            x = np.average(x, axis=-1, weights=(0.299, 0.587, 0.114))
    return x


def _minus_values(rng, shape):
    bg = rng.normal(0, 50, shape)
    flat = bg.reshape(-1)
    flat[:: 5] = np.nan
    flat[1:: 7] = np.inf
    flat[2:: 11] = -np.inf
    return [None, 0, -17, -3.25, float('nan'), bg]


@pytest.mark.parametrize('gray3,shape', [(False, (1,)), (False, (1, 1)), (False, (7, 13)),
                                         (True, (3,)), (True, (1, 1, 3)), (True, (7, 13, 3))])
@pytest.mark.parametrize('n', [1, 2, 7])
@pytest.mark.parametrize('dtype', [np.uint8, np.uint16, np.float32, np.float64])
def test_stack_mean(k5, dtype, n, gray3, shape):
    rng = np.random.default_rng(n * 100 + len(shape))
    frames = _random(rng, dtype, (n,) + shape)
    for minus in _minus_values(rng, shape):
        got = k5.stack_mean(_dev(frames), minus=minus, gray3=gray3)
        assert _same(got, _stack_ref(frames, minus, gray3), not gray3), 'array' if isinstance(minus, np.ndarray) else minus


@pytest.mark.parametrize('gray3', [False, True])
def test_stack_mean_float_edges(k5, gray3):
    """float32 frames with NaN, +-inf and +-FLT_MAX; float64 frames near 1e308 whose running sum overflows (or not) in
    frame order"""
    rng = np.random.default_rng(7)
    f = rng.normal(0, 100, (3, 7, 13, 3)).astype(np.float32)
    f[0, 0, 0, 0], f[1, 0, 1, 1], f[2, 0, 2, 2] = np.nan, np.inf, -np.inf
    f[:, 1, 0, :] = FLT_MAX
    f[:, 1, 1, :] = -FLT_MAX
    f[0, 1, 2, 0], f[1, 1, 2, 0] = np.inf, -np.inf                # inf + -inf = NaN
    if not gray3:
        f = f[..., 0]
    for minus in (None, 1.5, _minus_values(rng, f.shape[1:])[-1]):
        assert _same(k5.stack_mean(_dev(f), minus=minus, gray3=gray3), _stack_ref(f, minus, gray3), not gray3)
    big = np.full((3, 4, 5, 3), 1.0)
    big[:, 0, 0, :] = np.array([1e308, 1e308, -1e308])[:, None]        # overflows to inf after frame 2, stays inf
    big[:, 0, 1, :] = np.array([1e308, -1e308, 1e308])[:, None]        # no overflow in this order: 1e308 / 3
    big[:, 0, 2, :] = np.array([-1e308, -1e308, 1e308])[:, None]       # -inf
    big[:, 0, 3, :] = np.array([1.7e308, 1e307, -1e308])[:, None]      # overflows by a little
    big[:, 1, 0, :] = np.array([[1e308, -1e308, 1e308], [1e308, 1e308, 1e308], [1e308, 1e308, -1e308]])
    big[:, 1, 1, :] = np.array([8e307, 8e307, 8e307])[:, None]         # the mean fits, the sum does not
    if not gray3:
        big = big[..., 1]
    for minus in (None, -1e308, np.nan):
        assert _same(k5.stack_mean(_dev(big), minus=minus, gray3=gray3), _stack_ref(big, minus, gray3), not gray3)


@pytest.mark.parametrize('dtype,gray3', [(np.uint16, True), (np.float32, False)])
def test_stack_mean_grid_stride(k5, cap, dtype, gray3):
    n_out = 2 * cap + 37
    shape = (n_out, 3) if gray3 else (n_out,)
    rng = np.random.default_rng(9)
    frames = _random(rng, dtype, (3,) + shape)
    bg = _minus_values(rng, shape)[-1]
    for minus in (None, bg):
        assert _same(k5.stack_mean(_dev(frames), minus=minus, gray3=gray3), _stack_ref(frames, minus, gray3), not gray3)


# ---- B. scale_: data /= divisor in place -----------------------------------------------------------------------------
DIVISORS = [1.0, 3.0, -7.0, 0.0, float('nan'), 5e-324, 1e300]


def _scale_data(rng, size):
    a = rng.normal(0, 1e3, size)
    specials = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, 5e-324, -5e-324, 1e308, -1e308, 2.2e-308, 1.0, -3.0])
    k = min(size, specials.size)
    a[:k] = specials[:k]
    a[size // 2] = -0.0
    return a


@pytest.mark.parametrize('size', ['one', 'odd', 'grid_stride'])
def test_scale(k5, cap, size):
    n = {'one': 1, 'odd': 1001, 'grid_stride': 2 * cap + 37}[size]
    a = _scale_data(np.random.default_rng(n), n)
    for d in DIVISORS:
        t = _dev(a)
        assert k5.scale_(t, d) is t
        with np.errstate(all='ignore'):
            want = a / d
        assert _same(t, want), d


# ---- C. subsample: img[::sy, ::sx] ------------------------------------------------------------------------------------
@pytest.mark.parametrize('shape', [(1, 1), (1, 37), (29, 1), (7, 13), (90, 130)])
def test_subsample(k5, shape):
    H, W = shape
    img = np.random.default_rng(H * W).normal(0, 1, shape)
    d = _dev(img)
    for sy, sx in ((1, 1), (2, 2), (3, 3), (10, 10), (H + 1, W + 1), (H + 7, 1), (1, W + 3), (3, 7), (10, 3), (4, 1)):
        assert _same(k5.subsample(d, sy, sx), img[::sy, ::sx]), (sy, sx)


def test_subsample_full_frame(k5):
    img = np.random.default_rng(1).normal(0, 1, (3000, 4096))
    d = _dev(img)
    for sy, sx in ((10, 10), (7, 3), (1, 1)):
        assert _same(k5.subsample(d, sy, sx), img[::sy, ::sx]), (sy, sx)


def test_subsample_takes_views(k5):
    """a strided view is subsampled as the image it shows, not as the storage under it"""
    img = np.random.default_rng(2).normal(0, 1, (37, 52))
    d = _dev(img)
    assert _same(k5.subsample(d.t(), 3, 2), img.T[::3, ::2])
    assert _same(k5.subsample(d[1::2, 3:], 2, 5), img[1::2, 3:][::2, ::5])


# ---- D. linear_fit: per-pixel least-squares line (getLinearityFunction) ----------------------------------------------
def _times(kind, n):
    if kind == 'sorted':
        return [0.5 * 2 ** k for k in range(n)]
    if kind == 'negative_unsorted':
        return list(np.random.default_rng(n).permutation(np.linspace(-3.0, 5.0, n)))
    if kind == 'equal':
        return [2.0] * n                                     # denominator exactly 0
    return [1.0 + k * 2.0 ** -50 for k in range(n)]          # denominator nearly 0


def _series(rng, dtype, x, shape):
    """frames[k] = offset + ascent * x[k] + noise, with pixels of 0, 1 and 2 samples at or below the returned mx and NaN
    samples in float frames"""
    x = np.asarray(x)
    hi = {np.uint8: 255, np.uint16: 65535}.get(dtype, 1e6)
    mx = {np.uint8: 250, np.uint16: 65534}.get(dtype, 1e4)
    lo = 0.2 * mx
    base = lo + rng.random(shape) * 0.2 * mx
    slope = rng.normal(0, 0.02 * mx / max(np.ptp(x), 1.0), shape)
    y = base[None] + slope[None] * (x - x.min())[:, None, None] + rng.normal(0, 0.01 * mx, (len(x),) + shape)
    y = np.rint(y) if np.dtype(dtype).kind == 'u' else y
    y[:, 0, 0] = hi                                         # 0 unmasked samples: 0/0
    y[1:, 0, 1] = hi                                        # 1 unmasked sample
    y[2:, 0, 2] = hi                                        # 2 unmasked samples
    y[:, 0, 3] = y[0, 0, 3]                                 # flat line: ascent 0
    y[-1, 0, 4] = hi                                        # the last sample saturated
    if np.dtype(dtype).kind == 'f':
        y[0, 1, 0] = np.nan                                 # NaN samples are not masked (NaN > mx is False)
        y[:, 1, 1] = np.nan
        y[-1, 1, 2] = np.inf
        y[0, 1, 3] = -np.inf
    return y.astype(dtype), mx


@pytest.mark.parametrize('times', ['sorted', 'negative_unsorted', 'equal', 'nearly_equal'])
@pytest.mark.parametrize('n', [2, 3, 16])
@pytest.mark.parametrize('dtype', [np.uint8, np.uint16, np.float32, np.float64])
def test_linear_fit(k5, dtype, n, times):
    rng = np.random.default_rng(n)
    x = _times(times, n)
    frames, mx = _series(rng, dtype, x, (9, 13))
    d = _dev(frames)
    for min_ascent in (0.0, 0.001, 0.5, -1.0):
        with np.errstate(all='ignore'):
            woff, wasc, werr = producers.get_linearity_function(x, frames, mx, min_ascent)
        off, asc, err = k5.linear_fit(d, x, mx, min_ascent)
        assert _same(off, woff) and _same(asc, wasc) and _same(err, werr), min_ascent
        off2, asc2 = k5.linear_fit(d, x, mx, min_ascent, want_rmse=False)
        assert _same(off2, woff) and _same(asc2, wasc)


def test_linear_fit_grid_stride(k5, cap):
    rng = np.random.default_rng(4)
    x = [3.0, 0.5, 1.0, 8.0]
    frames, mx = _series(rng, np.float32, x, (2, cap + 19))          # 2 * cap + 38 pixels
    frames = frames.reshape(len(x), -1)[:, :2 * cap + 37]
    with np.errstate(all='ignore'):
        want = producers.get_linearity_function(x, frames, mx, 0.001)
    got = k5.linear_fit(_dev(frames), x, mx, 0.001)
    assert all(_same(g, w) for g, w in zip(got, want))


def test_linear_fit_refusals(k5, engine):
    from imgprocessor_b200._lib import ImgcorrError
    frames = np.random.default_rng(5).integers(0, 1000, (4, 6, 7)).astype(np.uint16)
    with pytest.raises(ImgcorrError):
        k5.linear_fit(_dev(frames[:1]), [1.0])               # a line needs two exposure times
    with pytest.raises(ValueError):
        k5.linear_fit(torch.from_numpy(frames), [1.0, 2.0, 3.0, 4.0])      # host tensor


def test_linear_fit_needs_one_time_per_frame(k5):
    """too few exposure times would be padded with zeros by ctypes and fit a wrong line"""
    frames = _dev(np.random.default_rng(6).integers(0, 1000, (4, 6, 7)).astype(np.uint16))
    with pytest.raises(ValueError):
        k5.linear_fit(frames, [1.0, 2.0, 3.0])
    with pytest.raises(ValueError):
        k5.linear_fit(frames, [1.0, 2.0, 3.0, 4.0, 5.0])


# ---- refusals of the K5 wrappers (each of these would read or write the wrong memory if it reached a kernel) -------------
def test_k5_wrappers_refuse_bad_tensors(k5):
    f64 = _dev(np.zeros((6, 9)))
    with pytest.raises(TypeError):
        k5.scale_(f64.float(), 2.0)
    with pytest.raises(ValueError):
        k5.scale_(f64.t(), 2.0)                              # in place: a copy would not be the caller's tensor
    with pytest.raises(ValueError):
        k5.scale_(f64.cpu(), 2.0)
    with pytest.raises(TypeError):
        k5.subsample(f64.float(), 2, 2)
    with pytest.raises(ValueError):
        k5.subsample(f64.cpu(), 2, 2)
    with pytest.raises(ValueError):
        k5.subsample(f64, 0, 2)
    with pytest.raises(ValueError):
        k5.stack_mean(torch.zeros((2, 4, 3), dtype=torch.uint16), gray3=True)
    with pytest.raises(ValueError):
        k5.stack_mean(_dev(np.zeros((2, 4, 6), np.uint16)), gray3=True)     # 24 samples: divisible by 3, not colour
    with pytest.raises(ValueError):
        k5.stack_mean(_dev(np.zeros((2, 4), np.uint16)), gray3=True)
    with pytest.raises(ValueError):
        k5.stack_mean(_dev(np.zeros((2, 4, 3), np.uint16)), minus=np.zeros(11), gray3=True)
    assert _same(f64, np.zeros((6, 9)))


# ---- E. median3x3: scipy.ndimage.median_filter(img, 3) --------------------------------------------------------------------
MEDIAN_SHAPES = [(1, 1), (1, 16), (2, 16), (3, 32), (4, 16), (16, 1), (9, 13), (300, 410)]


def _median_engine(engine, shape):
    from imgprocessor_b200 import _lib
    e = engine.get_engine(*shape)
    e.set_option(_lib.OPT_K1_VARIANT, 0)                     # the default dispatch, whatever an earlier test selected
    return e


def _median_image(rng, dtype, shape, kind):
    if kind == 'random':
        return rng.normal(0, 100, shape).astype(dtype)
    if kind == 'plateaus':
        return rng.integers(-2, 3, shape).astype(dtype)       # runs of equal values: medians tie with their neighbours
    tiny = float(np.finfo(dtype).smallest_subnormal)
    big = 1e308 if dtype == np.float64 else FLT_MAX
    vals = np.array([0.0, -0.0, tiny, -tiny, 3 * tiny, big, -big, 1.0, -1.0], dtype)
    return vals[rng.integers(0, vals.size, shape)]


@pytest.mark.parametrize('shape', MEDIAN_SHAPES)
@pytest.mark.parametrize('dtype', [np.float64, np.float32])
def test_median3x3(engine, dtype, shape):
    rng = np.random.default_rng(shape[0] * 1000 + shape[1])
    e = _median_engine(engine, shape)
    for kind in ('random', 'plateaus', 'edges'):
        img = _median_image(rng, dtype, shape, kind)
        got = e.median3x3(img)
        assert got.dtype == dtype and _same(got, median_filter(img, 3), signed_zero=False), kind


@pytest.mark.parametrize('dtype', [np.float64, np.float32])
def test_median3x3_infinite_medians(engine, dtype):
    """finite pixels inside regions of +-inf take the infinite median, and infinite pixels next to such regions the
    finite one"""
    rng = np.random.default_rng(12)
    for shape in ((9, 13), (4, 16), (1, 16), (300, 410)):
        e = _median_engine(engine, shape)
        H = shape[0]
        img = rng.normal(0, 10, shape).astype(dtype)
        img[H // 3:H // 3 + 5, 3:9] = np.inf
        img[min(H // 3 + 2, H - 1), 5] = 0.5                 # one finite pixel in a block of +inf
        img[-5:, -6:] = -np.inf
        img[-min(H, 3), -3] = 2.0                            # and one in a block of -inf
        img[0, :3] = np.inf
        r = rng.random(shape)
        img[r < 0.05] = np.inf
        img[r > 0.95] = -np.inf
        got = e.median3x3(img)
        assert _same(got, median_filter(img, 3), signed_zero=False), shape
    e = _median_engine(engine, (9, 13))
    img = np.full((9, 13), -np.inf, dtype)
    img[::2, ::2] = np.inf
    img[4, 4] = 1.0
    assert _same(e.median3x3(img), median_filter(img, 3), signed_zero=False)


def test_median3x3_full_frame_float64(engine):
    """the noise-level-function path: a float64 frame through K1's float64 path at full size"""
    rng = np.random.default_rng(13)
    img = rng.normal(1000, 30, (3000, 4096))
    img[::97, ::89] = 0.0
    img[1000:1010, 2000:2040] = 2500.0
    got = _median_engine(engine, img.shape).median3x3(img)
    assert _same(got, median_filter(img, 3), signed_zero=False)


# ---- F. end to end ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('shape', [(7, 130), (35, 9), (41, 43)])
@pytest.mark.parametrize('dtype', [np.uint16, np.float32, np.float64])
def test_flat_field_small_subsamples(engine, shape, dtype):
    """the median of the every-tenth-pixel image at 1 - 5 rows or columns"""
    from imgprocessor_b200.camera.flatField import flatFieldFromCloseDistance
    rng = np.random.default_rng(shape[0] + shape[1])
    scale = 4000.0 if dtype == np.uint16 else 1.0
    imgs = [(scale * (0.5 + rng.random(shape + (3,)))).astype(dtype) for _ in range(2)]
    bgs = [(scale * 0.1 * rng.random(shape + (3,))).astype(dtype) for _ in range(2)]
    for bg in (bgs, 41.5 if dtype == np.uint16 else 0.05):
        with np.errstate(all='ignore'):
            want = producers.flat_field_from_close_distance(imgs, bg)
        assert _same(flatFieldFromCloseDistance(imgs, bg), want)


def test_flat_field_full_frame(engine):
    from imgprocessor_b200.camera.flatField import flatFieldFromCloseDistance
    rng = np.random.default_rng(14)
    shape = (3000, 4096, 3)
    imgs = [rng.integers(20000, 40000, shape, dtype=np.uint16) for _ in range(2)]
    bgs = [rng.integers(0, 2000, shape, dtype=np.uint16) for _ in range(2)]
    got = flatFieldFromCloseDistance(imgs, bgs)
    assert _same(got, producers.flat_field_from_close_distance(imgs, bgs))


def test_linearity_function_full_frame(engine):
    """DarkCurrentMap.getLinearityFunction on a 4096x3000 uint16 series of 6 exposures, with saturated samples"""
    from imgprocessor_b200.camera import DarkCurrentMap as dcm
    rng = np.random.default_rng(15)
    x = [0.5, 1.0, 2.0, 4.0, 8.0, 16.0]
    frames, mx = _series(rng, np.uint16, x, (3000, 4096))
    frames[-1, ::13, ::7] = 65535
    got = dcm.getLinearityFunction(x, frames, mxIntensity=mx, min_ascent=0.001)
    want = producers.get_linearity_function(x, frames, mx, 0.001)
    assert all(_same(g, w) for g, w in zip(got, want))
