"""Parity tests proper: the CUDA path, called through the C ABI (ctypes -> libimgcorr.so), against the
oracle on the same seeded inputs and against the golden outputs of the unmodified reference.
Bars (BASELINE.json north star): median + mask bit-exact; pointwise float32 <= 1 ulp of the float64
reference (we require 0 ulp: correctly rounded); remap bit-exact given the same fixed-point coordinates;
end to end vs the float64 reference <= 1e-3 of full scale (we require 1e-5)."""
import contextlib
import io

import numpy as np
import pytest

from conftest import load_golden, ulp_diff_f32
from imgprocessor_b200 import synth
from oracle import models, refpath

pytestmark = pytest.mark.gpu

torch = pytest.importorskip('torch')


@pytest.fixture(scope='module')
def ip():
    if not torch.cuda.is_available():
        pytest.skip('needs a CUDA device')
    import imgprocessor_b200 as pkg
    from imgprocessor_b200 import engine, _lib
    pkg.engine_mod, pkg.lib_mod = engine, _lib
    return pkg


def _eng(ip, H, W, variant=0):
    e = ip.engine_mod.get_engine(H, W)
    e.set_option(ip.lib_mod.OPT_K1_VARIANT, variant)
    return e


def _case(H, W, seed, dtype=np.uint16):
    raw = synth.scene(H, W, seed, dtype)
    dark = synth.dark_map(H, W, seed)
    flat = synth.flat_map(H, W, seed, p_zero=5e-3)
    return raw, dark, flat


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


SHAPES = [(1, 1), (2, 3), (5, 4), (33, 130), (96, 128), (70, 257), (300, 520), (257, 1024)]


@pytest.mark.parametrize('shape', SHAPES)
@pytest.mark.parametrize('dtype', [np.uint8, np.uint16, np.float32])
@pytest.mark.parametrize('ksize', [3, 5])
def test_k1_bit_exact_generic(ip, shape, dtype, ksize):
    H, W = shape
    raw, dark, flat = _case(H, W, 3, dtype)
    e = _eng(ip, H, W, 1)
    e.set_dark(dark)
    e.set_flat(flat)
    out, mask = e.pointwise_median(_dev(raw), 0.1, ksize, want_mask=True)
    x = models.pointwise_model(raw, dark, flat, nan_to_num=True)
    want, wmask = models.median_threshold_model(x, 0.1, ksize)
    assert np.array_equal(out.cpu().numpy(), want)
    assert np.array_equal(mask.cpu().numpy().astype(bool), wmask)


@pytest.mark.parametrize('shape', [(1, 16), (2, 16), (3, 32), (4, 16), (5, 16), (33, 144), (96, 128), (70, 272), (300, 528),
                                   (257, 1024), (64, 4096)])
@pytest.mark.parametrize('dtype', [np.uint8, np.uint16, np.float32])
@pytest.mark.parametrize('ksize,variant', [(3, 2), (5, 2), (3, 3)])
def test_k1_bit_exact_tma(ip, shape, dtype, ksize, variant):
    """variant 2 = TMA-staged tiles, 3 = TMA streaming pipeline.  Heights 1 - 4 are below the stencil: the TMA tiles
    rebuild reflect rows from zero-filled boxes, and the 3x3 streaming kernel takes its prime / bottom step at height 1"""
    H, W = shape
    raw, dark, flat = _case(H, W, 4, dtype)
    e = _eng(ip, H, W, variant)
    try:
        e.set_dark(dark)
        e.set_flat(flat)
        x = models.pointwise_model(raw, dark, flat, nan_to_num=True)
        want, wmask = models.median_threshold_model(x, 0.1, ksize)
        out, mask = e.pointwise_median(_dev(raw), 0.1, ksize, want_mask=True)
        assert np.array_equal(out.cpu().numpy(), want)
        assert np.array_equal(mask.cpu().numpy().astype(bool), wmask)
        # partial calibrations through the TMA path as well
        e.set_dark(None)
        out, _ = e.pointwise_median(_dev(raw), 0.1, ksize)
        want, _ = models.median_threshold_model(models.pointwise_model(raw, None, flat, True), 0.1, ksize)
        assert np.array_equal(out.cpu().numpy(), want)
        e.set_flat(None)
        out, _ = e.pointwise_median(_dev(raw), 0.1, ksize)
        want, _ = models.median_threshold_model(models.pointwise_model(raw, None, None, True), 0.1, ksize)
        assert np.array_equal(out.cpu().numpy(), want)
    finally:
        e.set_option(ip.lib_mod.OPT_K1_VARIANT, 0)


def test_k1_tma_refused_when_not_eligible(ip):
    for variant in (2, 3):
        e = _eng(ip, 33, 130, variant)
        with pytest.raises(ip.lib_mod.ImgcorrError):
            e.pointwise_median(_dev(np.zeros((33, 130), np.uint16)), 0.1, 3)
    e.set_option(ip.lib_mod.OPT_K1_VARIANT, 0)


@pytest.mark.parametrize('seg_rows', [0, 4, 5, 7, 8, 9, 16, 33, 1000])
@pytest.mark.parametrize('W', [256, 240, 248, 496, 504, 1000])
def test_k1_stream_pair_seams_and_strip_edges(ip, seg_rows, W):
    """batches of the chain configuration run two frames per work unit (shared dark / flat arithmetic) and an odd last
    frame through the one-frame kernel: row segments and 120-column strips meet without seams, the right frame edge may
    fall anywhere inside a strip / warp, frames do not leak into each other; tiny flats make the quotient overflow
    (clamp path), non-finite maps and float32 frames take the checked instantiation"""
    H, n = 83, 5
    _, dark, flat = _case(H, W, 8, np.uint16)
    frames = np.stack([synth.scene(H, W, 50 + i, np.uint16) for i in range(n)])
    e = _eng(ip, H, W, 3)
    e.set_option(ip.lib_mod.OPT_K1_SEG_ROWS, seg_rows)
    try:
        for tweak in ('plain', 'overflow', 'nonfinite'):
            d2, f2 = dark.copy(), flat.copy()
            if tweak == 'overflow':
                f2[3, 5] = np.float32(1e-42)
                f2[H - 1, W - 1] = np.float32(-1e-40)
            if tweak == 'nonfinite':
                f2[7, 9], f2[8, 9], d2[20, 20] = np.inf, np.nan, -np.inf
            e.set_dark(d2)
            e.set_flat(f2)
            for nn in (n, n - 1):
                out, _ = e.pointwise_median(_dev(frames[:nn]), 0.1, 3)
                for i in range(nn):
                    want, _ = models.median_threshold_model(models.pointwise_model(frames[i], d2, f2, True), 0.1, 3)
                    assert np.array_equal(out[i].cpu().numpy(), want), (tweak, nn, i)
        rawf = np.stack([synth.scene(H, W, 60 + i, np.float32) for i in range(4)])
        rawf[1, 5, 5], rawf[2, 6, 7] = np.inf, np.nan
        e.set_dark(dark)
        e.set_flat(flat)
        out, _ = e.pointwise_median(_dev(rawf), 0.1, 3)
        for i in range(4):
            want, _ = models.median_threshold_model(models.pointwise_model(rawf[i], dark, flat, True), 0.1, 3)
            assert np.array_equal(out[i].cpu().numpy(), want), i
    finally:
        e.set_option(ip.lib_mod.OPT_K1_SEG_ROWS, 0)
        e.set_option(ip.lib_mod.OPT_K1_VARIANT, 0)


@pytest.mark.parametrize('seg_rows', [4, 7, 8, 9, 16, 33, 1000])
def test_k1_stream_segment_seams(ip, seg_rows):
    """row segments of the streaming kernel meet without seams, whatever their height; non-finite
    calibration values and the mask / '<' paths go through the run-time-flag instantiation"""
    H, W = 75, 256
    raw, dark, flat = _case(H, W, 6, np.uint16)
    e = _eng(ip, H, W, 3)
    e.set_option(ip.lib_mod.OPT_K1_SEG_ROWS, seg_rows)
    e.set_dark(dark)
    e.set_flat(flat)
    out, _ = e.pointwise_median(_dev(raw), 0.1, 3)
    want, _ = models.median_threshold_model(models.pointwise_model(raw, dark, flat, True), 0.1, 3)
    assert np.array_equal(out.cpu().numpy(), want)
    flat2 = flat.copy()
    flat2[7, 9], flat2[8, 9], dark2 = np.inf, np.nan, dark.copy()
    dark2[20, 20] = -np.inf
    e.set_dark(dark2)
    e.set_flat(flat2)
    for cond in ('>', '<'):
        out, mask = e.pointwise_median(_dev(raw), 0.1, 3, cond, want_mask=True)
        want, wmask = models.median_threshold_model(models.pointwise_model(raw, dark2, flat2, True), 0.1, 3, cond)
        assert np.array_equal(out.cpu().numpy(), want) and np.array_equal(mask.cpu().numpy().astype(bool), wmask)
    e.set_option(ip.lib_mod.OPT_K1_SEG_ROWS, 0)
    e.set_option(ip.lib_mod.OPT_K1_VARIANT, 0)


@pytest.mark.parametrize('seg_rows', [0, 8, 9, 11, 16, 37, 1000])
@pytest.mark.parametrize('shape', [(8, 16), (75, 256), (37, 112), (64, 120), (130, 344)])
def test_k1_stream5_bit_exact(ip, seg_rows, shape):
    """the 5x5 streaming kernel: segment seams at any height (incl. heights that leave a 1-row tail, which the launcher
    avoids), strip edges at non-multiples of 112 columns, top / bottom / left / right 'reflect', every instantiation"""
    H, W = shape
    raw, dark, flat = _case(H, W, 16, np.uint16)
    e = _eng(ip, H, W, 3)                      # variant 3 = streaming pipeline or an error: never a silent tile fallback
    e.set_option(ip.lib_mod.OPT_K1_SEG_ROWS, seg_rows)
    try:
        e.set_dark(dark)
        e.set_flat(flat)
        out, _ = e.pointwise_median(_dev(raw), 0.1, 5)                                  # chain instantiation
        want, _ = models.median_threshold_model(models.pointwise_model(raw, dark, flat, True), 0.1, 5)
        assert np.array_equal(out.cpu().numpy(), want)
        rawf = synth.scene(H, W, 17, np.float32)
        out, mask = e.pointwise_median(_dev(rawf), 0.1, 5, want_mask=True)              # float32 frames: checked instantiation
        want, wmask = models.median_threshold_model(models.pointwise_model(rawf, dark, flat, True), 0.1, 5)
        assert np.array_equal(out.cpu().numpy(), want) and np.array_equal(mask.cpu().numpy().astype(bool), wmask)
        flat2, dark2 = flat.copy(), dark.copy()
        flat2[min(7, H - 1), 9], flat2[min(8, H - 1), 9], dark2[H // 2, W // 2] = np.inf, np.nan, -np.inf
        e.set_dark(dark2)
        e.set_flat(flat2)
        for cond in ('>', '<'):                                                         # run-time-flag instantiation
            out, mask = e.pointwise_median(_dev(raw), 0.1, 5, cond, want_mask=True)
            want, wmask = models.median_threshold_model(models.pointwise_model(raw, dark2, flat2, True), 0.1, 5, cond)
            assert np.array_equal(out.cpu().numpy(), want) and np.array_equal(mask.cpu().numpy().astype(bool), wmask)
        # direct medianThreshold on the image dtype (no calibration): uint16 -> uint16 and uint8 -> uint8 with mask
        e.set_dark(None)
        e.set_flat(None)
        for dt in (np.uint16, np.uint8) if W % 16 == 0 else (np.uint16,):
            img = synth.scene(H, W, 18, dt)
            out, mask = e.pointwise_median(_dev(img), 0.1, 5, flags=0, out_dtype=_dev(img).dtype, want_mask=True)
            want, wmask = models.median_threshold_model(img, 0.1, 5)
            assert np.array_equal(out.cpu().numpy(), want) and np.array_equal(mask.cpu().numpy().astype(bool), wmask)
    finally:
        e.set_option(ip.lib_mod.OPT_K1_SEG_ROWS, 0)
        e.set_option(ip.lib_mod.OPT_K1_VARIANT, 0)


def test_k1_stream5_batch_and_guard_band(ip):
    H, W, n = 70, 272, 5
    e = _eng(ip, H, W, 3)
    _, dark, flat = _case(H, W, 1)
    e.set_dark(dark)
    e.set_flat(flat)
    frames = np.stack([synth.scene(H, W, 30 + i, np.uint16) for i in range(n)])
    out, mask = e.pointwise_median(_dev(frames), 0.1, 5, want_mask=True)
    for i in range(n):
        want, wmask = models.median_threshold_model(models.pointwise_model(frames[i], dark, flat, True), 0.1, 5)
        assert np.array_equal(out[i].cpu().numpy(), want) and np.array_equal(mask[i].cpu().numpy().astype(bool), wmask)
    # pixels engineered onto the threshold from both sides: the float32 guard band must hand them to the exact path
    e.set_dark(None)
    e.set_flat(None)
    rng = np.random.default_rng(5)
    img = np.full((H, W), 1000.0, np.float32) + rng.random((H, W)).astype(np.float32)
    ys, xs = rng.integers(3, H - 3, 200), rng.integers(3, W - 3, 200)
    img[ys, xs] = np.float32(1100.0) * (1 + rng.integers(-4, 5, 200).astype(np.float32) * np.float32(2.0 ** -23))
    out, mask = e.pointwise_median(_dev(img), 0.1, 5, flags=0, want_mask=True)
    want, wmask = models.median_threshold_model(img, 0.1, 5)
    assert np.array_equal(out.cpu().numpy(), want) and np.array_equal(mask.cpu().numpy().astype(bool), wmask)
    e.set_option(ip.lib_mod.OPT_K1_VARIANT, 0)


@pytest.mark.parametrize('seg_rows', [0, 4, 7, 16, 33])
@pytest.mark.parametrize('dtype', [np.uint16, np.float32, np.uint8])
def test_k1_stream_pointwise_only(ip, seg_rows, dtype):
    """threshold <= 0 (no artefact step, no nan_to_num) through the streaming pipeline: 0 ulp of the float64 result at
    every segment seam, with finite and non-finite calibration values, several frames per launch"""
    H, W, n = 61, 272, 3
    _, dark, flat = _case(H, W, 8)
    frames = np.stack([synth.scene(H, W, 40 + i, dtype) for i in range(n)])
    e = _eng(ip, H, W, 3)
    e.set_option(ip.lib_mod.OPT_K1_SEG_ROWS, seg_rows)
    try:
        for d, f in ((dark, flat), (np.where(dark > 105, np.inf, dark).astype(np.float32), np.where(flat > 0.9, np.nan, flat).astype(np.float32))):
            e.set_dark(d)
            e.set_flat(f)
            out, _ = e.pointwise_median(_dev(frames), 0.0, 3, flags=ip.lib_mod.DO_DARK | ip.lib_mod.DO_FLAT)
            for i in range(n):
                with np.errstate(all='ignore'):
                    want = models.pointwise_model(frames[i], d, f, False)
                assert np.array_equal(out[i].cpu().numpy(), want, equal_nan=True), (seg_rows, dtype, i)
    finally:
        e.set_option(ip.lib_mod.OPT_K1_SEG_ROWS, 0)
        e.set_option(ip.lib_mod.OPT_K1_VARIANT, 0)


def test_ddiv_selftest(ip):
    """the float64 division K1 / K4 run (MUFU.RCP64H seed + ONE Newton step + residual correction) equals IEEE division
    for every float32 significand pattern of the divisor (2^24 patterns incl. sign, exponents over the float32 range and
    small integers) x 64 numerators of the shapes the kernels produce; the seed is good to better than 2^-16 (the
    proof in imgcorr_core.cuh needs 2^-14)"""
    e = _eng(ip, 16, 16)
    bad, worst = e.selftest_division(64, 2024)
    assert bad == 0, '%d of 2^30 quotients differ from IEEE division' % bad
    assert 0.0 < worst < 2.0 ** -16, worst


def test_k1_multi_frame_batch(ip):
    H, W, n = 70, 272, 5
    e = _eng(ip, H, W, 0)
    _, dark, flat = _case(H, W, 1)
    e.set_dark(dark)
    e.set_flat(flat)
    frames = np.stack([synth.scene(H, W, 10 + i, np.uint16) for i in range(n)])
    for variant in (1, 2, 3):
        e.set_option(ip.lib_mod.OPT_K1_VARIANT, variant)
        out, mask = e.pointwise_median(_dev(frames), 0.1, 3, want_mask=True)
        for i in range(n):
            want, wmask = models.median_threshold_model(models.pointwise_model(frames[i], dark, flat, True), 0.1, 3)
            assert np.array_equal(out[i].cpu().numpy(), want)
            assert np.array_equal(mask[i].cpu().numpy().astype(bool), wmask)
    e.set_option(ip.lib_mod.OPT_K1_VARIANT, 0)


def test_k1_pointwise_zero_ulp(ip):
    H, W = 64, 96
    raw, dark, flat = _case(H, W, 9)
    flat[3, 3] = np.float32(1e-42)
    flat[4, 4] = np.float32(-2.0)
    e = _eng(ip, H, W)
    e.set_dark(dark)
    e.set_flat(flat)
    out, _ = e.pointwise_median(_dev(raw), 0.0, 0, flags=3)
    x = refpath.to_float_image(raw)
    refpath.correct_dark_current(x, dark)
    refpath.correct_vignetting(x, flat)
    with np.errstate(over='ignore'):
        ref32 = x.astype(np.float32)
    got = out.cpu().numpy()
    fin = np.isfinite(ref32)
    assert ulp_diff_f32(got[fin], ref32[fin]).max() == 0          # north star asks for <= 1
    assert np.array_equal(got, ref32)
    out, _ = e.pointwise_median(_dev(raw), 0.0, 0, flags=7)
    assert out[3, 3].item() == np.finfo(np.float32).max
    # float64 widening output
    out, _ = e.pointwise_median(_dev(raw), 0.0, 0, flags=3, out_dtype=torch.float64)
    assert np.array_equal(out.cpu().numpy(), ref32.astype(np.float64))


def test_k1_legacy_linear_dark(ip):
    g = load_golden('correct_u16_legacy_dark')
    offs, asc = g['offs'].astype(np.float32), g['ascent'].astype(np.float32)
    H, W = offs.shape
    e = _eng(ip, H, W)
    e.set_dark(offs, asc, float(g['exposure_time']), 16)
    e.set_flat(None)
    out, _ = e.pointwise_median(_dev(g['raw']), 0.0, 0, flags=1)
    want = models.pointwise_model(g['raw'], offs, None, False, dark_ascent=asc, exposure_time=float(g['exposure_time']))
    assert np.array_equal(out.cpu().numpy(), want)
    out, _ = e.pointwise_median(_dev(g['raw']), 0.1, 3, flags=5)
    want, _ = models.median_threshold_model(models.nan_to_num_f32(want), 0.1, 3)
    assert np.array_equal(out.cpu().numpy(), want)
    # and against the float64 reference output itself
    assert np.abs(out.cpu().numpy() - g['out']).max() / 65535.0 < 1e-5


@pytest.mark.parametrize('name', ['median_u16_s3_gt', 'median_u16_s3_lt', 'median_u16_s5_gt', 'median_u16_s5_lt',
                                  'median_f32_s3_gt', 'median_f32_s3_lt', 'median_f32_s5_gt', 'median_f32_s5_lt'])
def test_medianThreshold_api_vs_reference_golden(ip, name):
    g = load_golden(name)
    size = 3 if '_s3_' in name else 5
    cond = '>' if name.endswith('gt') else '<'
    img = g['img'].copy()
    out, ind = ip.medianThreshold(img, threshold=0.1, size=size, condition=cond, copy=True)
    assert out is not img and np.array_equal(img, g['img'])
    assert out.dtype == g['out'].dtype and np.array_equal(out, g['out'])
    assert ind.dtype == bool and np.array_equal(ind, g['ind'])
    same, ind2 = ip.medianThreshold(img, threshold=0.1, size=size, condition=cond, copy=False)
    assert same is img and np.array_equal(img, g['out']) and np.array_equal(ind2, g['ind'])
    untouched, none = ip.medianThreshold(img, threshold=0)
    assert untouched is img and none is None


def test_medianThreshold_zero_medians_f64_and_extremes(ip):
    g = load_golden('median_f32_zeros')
    out, ind = ip.medianThreshold(g['img'], float(g['threshold']), 3)
    assert np.array_equal(out, g['out']) and np.array_equal(ind, g['ind'])
    rng = np.random.default_rng(4)
    img = rng.normal(1000, 300, (40, 50))
    img[rng.random(img.shape) < 0.01] *= 5
    for size in (3, 5):
        out, ind = ip.medianThreshold(img, 0.2, size)
        want, wmask = models.median_threshold_model(img, 0.2, size)
        assert out.dtype == np.float64 and np.array_equal(out, want) and np.array_equal(ind, wmask)
    ext = np.array([[3e38, -3e38, 1e-40, 0, 5], [1e30, -1e30, 7, 1, 2], [0, 0, 0, 0, 0]], np.float32)
    for thr in (0.1, 5.0):
        out, ind = ip.medianThreshold(ext, thr, 3)
        want, wmask = models.median_threshold_model(ext, thr, 3)
        assert np.array_equal(ind, wmask) and np.array_equal(out, want)


def test_predicate_guard_band(ip):
    """pixels engineered to sit on the threshold from both sides, many seeds, one launch per seed"""
    for seed in range(40):
        rng = np.random.default_rng(seed)
        H, W = 24, 40
        thr = float(rng.choice([0.01, 0.1, 0.3, 1.0, 1.5]))
        img = (rng.random((H, W)) * 100 + 1).astype(np.float32)
        med = models.median_filter_reflect(img, 3)
        for _ in range(40):
            y, x = rng.integers(0, H), rng.integers(0, W)
            b = np.float64(med[y, x])
            img[y, x] = np.float32(b * (1 + thr * rng.choice([-1, 1])) * (1 + rng.choice([-1, 0, 1]) * 6e-8))
        for cond in ('>', '<'):
            out, ind = ip.medianThreshold(img, thr, 3, cond)
            want, wmask = models.median_threshold_model(img, thr, 3, cond)
            assert np.array_equal(ind, wmask) and np.array_equal(out, want)


# ---------------------------------------------------------------------------- K2
@pytest.mark.parametrize('tag', ['moderate', 'strong', 'realistic'])
def test_maps_vs_reference_golden(ip, tag):
    g = load_golden('maps_' + tag)
    H, W = (int(v) for v in g['shape'])
    l = ip.LensDistortion({})
    l._coeffs['cameraMatrix'], l._coeffs['distortionCoeffs'] = g['K'], g['dist']
    mx, my = l.getUndistortRectifyMap(W, H)
    assert mx.dtype == np.float32 and tuple(l.roi) == tuple(g['roi'])
    for a, b in zip(models.fixed_point_coords(mx, my), models.fixed_point_coords(g['mapx'], g['mapy'])):
        assert np.array_equal(a, b)
    assert (mx != g['mapx']).mean() < 1e-3 and (my != g['mapy']).mean() < 1e-3
    assert np.abs(mx.astype(np.float64) - g['mapx']).max() < 2e-4


@pytest.mark.parametrize('tag', ['u8', 'u16', 'f32', 'f64'])
@pytest.mark.parametrize('keep', [0, 1])
def test_LensDistortion_correct_vs_reference_golden(ip, tag, keep):
    g = load_golden('lens_%s_keep%d' % (tag, keep))
    l = ip.LensDistortion({})
    l._coeffs['cameraMatrix'], l._coeffs['distortionCoeffs'] = g['K'], g['dist']
    out = l.correct(g['img'], keepSize=bool(keep), borderValue=float(g['border']))
    assert out.dtype == g['out'].dtype and out.shape == g['out'].shape
    assert tuple(l.roi) == tuple(g['roi'])
    assert np.array_equal(out, g['out'])          # bit-exact incl. the analytic map on this fixture
    assert l.img is out


@pytest.mark.parametrize('dtype', [np.uint8, np.uint16, np.float32, np.float64])
def test_remap_explicit_maps_vs_model(ip, dtype):
    rng = np.random.default_rng(3)
    H, W = 70, 90
    if np.dtype(dtype).kind == 'u':
        src = rng.integers(0, np.iinfo(dtype).max + 1, (H, W)).astype(dtype)
    else:
        src = ((rng.random((H, W)) - 0.3) * 4000).astype(dtype)
    mapx = np.arange(W, dtype=np.float32)[None, :] + rng.normal(0, 4, (H, W)).astype(np.float32)
    mapy = np.arange(H, dtype=np.float32)[:, None] + rng.normal(0, 4, (H, W)).astype(np.float32)
    mapx[0, :6] = [-1.0, -0.5, W - 1, W - 0.5, W, 1e9]
    mapy[1, :4] = [-1.0, H - 1, H, -1e9]
    mapx[2, :3] = [np.nan, np.inf, -np.inf]
    mapx[3, :4] = np.float32(10) + np.array([0.5, 1.5, 2.5, 3.5], np.float32) / np.float32(32)
    e = _eng(ip, H, W)
    for border in (0, 7, 0.1234567):
        out = e.remap(_dev(src), _dev(mapx), _dev(mapy), border).cpu().numpy()
        assert out.dtype == src.dtype
        assert np.array_equal(out, models.remap_model(src, mapx, mapy, border))
    if dtype == np.float32:
        wide = e.remap(_dev(src), _dev(mapx), _dev(mapy), 0.0, out_dtype=torch.float64).cpu().numpy()
        assert np.array_equal(wide, models.remap_model(src, mapx, mapy, 0).astype(np.float64))


@pytest.mark.parametrize('shape', [(200, 328), (96, 128), (333, 1000), (1500, 2048)])
@pytest.mark.parametrize('lens_kind', ['moderate', 'strong', 'extreme'])
def test_k2_coordinate_cache(ip, shape, lens_kind):
    """the tiled K2 stores the packed source coordinates of a lens / output window on its first launch and reads them on
    the following ones (IMGCORR_OPT_K2_COORD_CACHE): first launch, cached launches, cache switched off and the oracle all
    agree bit for bit — whole frame and roi window, float32 / float64 / uint16 outputs, any box geometry (the strong and
    the extreme lens need the larger staged boxes; tiles the box cannot cover fall back to gathers), border values;
    a new lens drops the cache.  Option key 12 (retired) is refused."""
    H, W = shape
    p = {'moderate': synth.lens_moderate(H, W), 'strong': synth.lens_strong(H, W),
         'extreme': (0.45 * W, 0.45 * W, W / 2.0 + 3, H / 2.0 - 2, -0.3, 0.12, -0.02, 4e-3, -3e-3)}[lens_kind]
    K, d = synth.camera_matrix(p), synth.dist_coeffs(p)
    mapx, mapy, P, roi = refpath.undistort_rectify_map(K, d, W, H)
    e = _eng(ip, H, W)
    rng = np.random.default_rng(11)
    src = (rng.random((5, H, W)) * 4000).astype(np.float32)
    x0, y0, ww, hh = (int(v) for v in roi)
    with pytest.raises(ip.lib_mod.ImgcorrError) as err:
        e.set_option(12, 1)
    assert err.value.status == ip.lib_mod.ERR_INVALID
    try:
        for cache in (1, 0):
            e.set_option(ip.lib_mod.OPT_K2_COORD_CACHE, cache)
            e.set_lens(K, d, P)                                    # drops any cache of an earlier test
            for rep in range(3):                                   # 1st: computes (and writes), 2nd / 3rd: read
                for border in (0.0, 7.5):
                    out = e.undistort(_dev(src[:1 + rep]), border_value=border).cpu().numpy()
                    for i in range(1 + rep):
                        got, want = out[i], models.remap_model(src[i], mapx, mapy, border)
                        # analytic map vs cv2's: at most a stray 1/32-px flip
                        assert (got != want).mean() < 1e-5, (cache, rep, border, i)
                if ww > 0 and hh > 0:
                    win = e.undistort(_dev(src[0]), window=(x0, y0, ww, hh)).cpu().numpy()
                    full = e.undistort(_dev(src[0])).cpu().numpy()
                    assert np.array_equal(win, full[y0:y0 + hh, x0:x0 + ww]), (cache, rep)
            a = e.undistort(_dev(src[:4])).cpu().numpy()
            if cache == 1:
                cached = a
            else:
                assert np.array_equal(a, cached)                   # cache on == cache off, bit for bit
            wide = e.undistort(_dev(src[0]), out_dtype=torch.float64).cpu().numpy()
            assert np.array_equal(wide, a[0].astype(np.float64))
        e.set_option(ip.lib_mod.OPT_K2_COORD_CACHE, 1)
        u16 = rng.integers(0, 65536, (4, H, W)).astype(np.uint16)
        if W % 8 == 0:
            for rep in range(2):
                out = e.undistort(_dev(u16)).cpu().numpy()
                for i in range(4):
                    assert (out[i] != models.remap_model(u16[i], mapx, mapy, 0)).mean() < 1e-5
        # the same lens set again (every correct() call of the mirror does that) keeps the cache: same bits
        e.set_lens(K, d, P)
        again = e.undistort(_dev(src[:1])).cpu().numpy()
        e.set_lens(K, d, P)
        assert np.array_equal(again, e.undistort(_dev(src[:1])).cpu().numpy()) and np.array_equal(again[0], cached[0])
        # another lens: the cached coordinates of the first must not survive
        p2 = synth.lens_moderate(H, W) if lens_kind != 'moderate' else synth.lens_strong(H, W)
        K2, d2 = synth.camera_matrix(p2), synth.dist_coeffs(p2)
        mapx2, mapy2, P2, _ = refpath.undistort_rectify_map(K2, d2, W, H)
        e.set_lens(K2, d2, P2)
        got = e.undistort(_dev(src[0])).cpu().numpy()
        assert (got != models.remap_model(src[0], mapx2, mapy2, 0)).mean() < 1e-5
    finally:
        e.set_option(ip.lib_mod.OPT_K2_COORD_CACHE, 1)
        e.set_lens(None, None, None)


@pytest.mark.parametrize('k2_variant', [1, 2])
@pytest.mark.parametrize('lens_kind', ['moderate', 'strong'])
def test_k2_variants_bit_identical(ip, k2_variant, lens_kind):
    """K2 through L1 gathers (1) and through TMA-staged shared-memory tiles (2): same bits, several frames per launch,
    roi window, float64 widening; the strong lens and the jittered explicit maps overflow the staged box -> fallback"""
    H, W, n = 200, 328, 3
    p = synth.lens_moderate(H, W) if lens_kind == 'moderate' else synth.lens_strong(H, W)
    K, d = synth.camera_matrix(p), synth.dist_coeffs(p)
    mapx, mapy, P, roi = refpath.undistort_rectify_map(K, d, W, H)
    e = _eng(ip, H, W)
    e.set_lens(K, d, P)
    e.set_option(ip.lib_mod.OPT_K2_VARIANT, k2_variant)
    try:
        frames = np.stack([synth.scene(H, W, 40 + i, np.float32) for i in range(n)])
        mx, my = (m.cpu().numpy() for m in e.undistort_maps())
        full = e.undistort(_dev(frames), border_value=3.5).cpu().numpy()
        x, y, w, h = (int(v) for v in roi)
        crop = e.undistort(_dev(frames), window=(x, y, w, h), out_dtype=torch.float64).cpu().numpy()
        for i in range(n):
            want = models.remap_model(frames[i], mx, my, 3.5)
            assert np.array_equal(full[i], want)
            want0 = models.remap_model(frames[i], mx, my, 0.0)
            assert crop.dtype == np.float64 and np.array_equal(crop[i], want0[y:y + h, x:x + w].astype(np.float64))
        rng = np.random.default_rng(5)
        jx = np.arange(W, dtype=np.float32)[None, :] + rng.normal(0, 6, (H, W)).astype(np.float32)
        jy = np.arange(H, dtype=np.float32)[:, None] + rng.normal(0, 6, (H, W)).astype(np.float32)
        jx[0, :3] = [np.nan, -5.0, W + 3.0]
        got = e.remap(_dev(frames), _dev(jx), _dev(jy), 1.25).cpu().numpy()
        for i in range(n):
            assert np.array_equal(got[i], models.remap_model(frames[i], jx, jy, 1.25))
    finally:
        e.set_option(ip.lib_mod.OPT_K2_VARIANT, 0)


@pytest.mark.parametrize('k2_variant', [0, 1, 2])
@pytest.mark.parametrize('dtype', [np.uint16, np.uint8])
def test_k2_integer_frames_all_variants(ip, k2_variant, dtype):
    """uint16 / uint8 frames (int16 fixed-point weights for uint8) through L1 gathers, the staged tiles and the automatic
    choice (tiles from 4 frames per launch): bit-exact vs the model, border value rounded to the image type, roi window"""
    H, W = 200, 336                                             # 336 uint8 columns = 21 x 16 bytes: tiles eligible for both types
    p = synth.lens_moderate(H, W)
    K, d = synth.camera_matrix(p), synth.dist_coeffs(p)
    mapx, mapy, P, roi = refpath.undistort_rectify_map(K, d, W, H)
    e = _eng(ip, H, W)
    e.set_lens(K, d, P)
    e.set_option(ip.lib_mod.OPT_K2_VARIANT, k2_variant)
    try:
        mx, my = (m.cpu().numpy() for m in e.undistort_maps())
        x, y, w, h = (int(v) for v in roi)
        for n in (1, 6):
            frames = np.stack([synth.scene(H, W, 60 + i, dtype) for i in range(n)])
            full = e.undistort(_dev(frames), border_value=77.6).cpu().numpy()
            crop = e.undistort(_dev(frames), window=(x, y, w, h)).cpu().numpy()
            assert full.dtype == dtype
            for i in range(n):
                assert np.array_equal(full[i], models.remap_model(frames[i], mx, my, 77.6)), (k2_variant, dtype, n, i)
                assert np.array_equal(crop[i], models.remap_model(frames[i], mx, my, 0.0)[y:y + h, x:x + w])
    finally:
        e.set_option(ip.lib_mod.OPT_K2_VARIANT, 0)


def test_undistort_multi_frame_and_window(ip):
    H, W, n = 125, 166, 4
    p = synth.lens_moderate(H, W)
    K, d = synth.camera_matrix(p), synth.dist_coeffs(p)
    mapx, mapy, P, roi = refpath.undistort_rectify_map(K, d, W, H)
    e = _eng(ip, H, W)
    e.set_lens(K, d, P)
    frames = np.stack([synth.scene(H, W, 20 + i, np.float32) for i in range(n)])
    mx, my = (m.cpu().numpy() for m in e.undistort_maps())
    full = e.undistort(_dev(frames)).cpu().numpy()
    x, y, w, h = (int(v) for v in roi)
    crop = e.undistort(_dev(frames), window=(x, y, w, h)).cpu().numpy()
    for i in range(n):
        want = models.remap_model(frames[i], mx, my, 0.0)
        assert np.array_equal(full[i], want)
        assert np.array_equal(crop[i], want[y:y + h, x:x + w])
    with pytest.raises(ip.lib_mod.ImgcorrError):
        e.undistort(_dev(frames), window=(0, 0, W + 1, H))


# ---------------------------------------------------------------------------- the chain, reference API
def _cal(ip, g, lens=True):
    cal = ip.CameraCalibration()
    if 'dark' in g:
        cal.addDarkCurrent(g['dark'])
    if 'flat' in g:
        cal.addFlatField(g['flat'])
    if lens and 'K' in g:
        l = ip.LensDistortion({})
        l._coeffs['cameraMatrix'], l._coeffs['distortionCoeffs'] = g['K'], g['dist']
        l._coeffs['shape'] = g['raw'].shape
        cal.addLens(l)
    return cal


def _quiet(fn, *a, **k):
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        r = fn(*a, **k)
    return r, buf.getvalue()


@pytest.mark.parametrize('keep', [1, 0])
def test_correct_vs_unmodified_reference(ip, keep):
    g = load_golden('correct_u16_keep%d' % keep)
    cal = _cal(ip, g)
    raw = g['raw'].copy()
    out, log = _quiet(cal.correct, raw, threshold=0.1, keep_size=bool(keep))
    assert np.array_equal(raw, g['raw'])                          # input never mutated
    assert out.dtype == np.float64 and out.shape == g['out'].shape
    assert log == str(g['log'])                                   # same progress lines
    ok = np.abs(g['out']) < 1e6                                   # denormal-flat pixel overflows float32
    assert (~ok).sum() <= 4
    assert np.abs(out[ok] - g['out'][ok]).max() / 65535.0 < 1e-5  # north star bar: 1e-3
    # bit-exact against the float32 staged oracle chain
    mx, my = models.undistort_map_model(g['K'], g['dist'], refpath.undistort_rectify_map(g['K'], g['dist'], 128, 96)[2], 128, 96)
    l = cal.getLens(None, None)
    gmx, gmy = l.getUndistortRectifyMap(128, 96)
    want, _ = models.correct_chain_f32(g['raw'], g['dark'], g['flat'], 0.1, 3, mapxy=(gmx, gmy))
    if not keep:
        x, y, w, h = (int(v) for v in l.roi)
        want = want[y:y + h, x:x + w]
    assert np.array_equal(out, want.astype(np.float64))
    # last_img: the dark+flat corrected, pre-median image
    li = cal.last_img
    fin = np.isfinite(g['last_img']) & (np.abs(g['last_img']) < 3e38)
    assert np.array_equal(li[fin], g['last_img'][fin].astype(np.float32).astype(np.float64))
    assert np.array_equal(cal.temp['bg'], g['bg'])


def test_correct_partial_calibrations_and_thr0(ip):
    g = load_golden('correct_f32_thr0')
    out, log = _quiet(_cal(ip, g).correct, g['raw'], threshold=0)
    assert log == str(g['log'])
    fin = np.isfinite(g['out']) & (np.abs(g['out']) < 1e6)
    assert np.abs(out[fin] - g['out'][fin]).max() / 4095.0 < 1e-5
    g = load_golden('correct_f32_flat_only')
    out, log = _quiet(_cal(ip, g).correct, g['raw'], threshold=0.25)
    assert log == str(g['log'])
    ok = np.abs(g['out']) < 1e6
    assert np.abs(out[ok] - g['out'][ok]).max() / 4095.0 < 1e-5
    g = load_golden('correct_u16_nothing')
    out, log = _quiet(ip.CameraCalibration().correct, g['raw'], threshold=0.1)
    assert log == str(g['log'])
    assert np.array_equal(out, g['out'])          # integers: float32 chain == float64 chain exactly


def test_correct_legacy_tuple_dark_and_dates(ip):
    import time
    g = load_golden('correct_u16_legacy_dark')
    cal = ip.CameraCalibration()
    cal.coeffs['dark current'].append((time.localtime(), '', (g['offs'].copy(), g['ascent'].copy()), None))
    cal.coeffs['shape'] = g['raw'].shape
    out, log = _quiet(cal.correct, g['raw'], exposure_time=float(g['exposure_time']), threshold=0.1)
    assert log == str(g['log'])
    assert np.abs(out - g['out']).max() / 65535.0 < 1e-5
    # exposure_time=None with a tuple entry: TypeError swallowed, stage skipped (SURVEY §8b)
    out, log = _quiet(cal.correct, g['raw'], threshold=0)
    assert 'Error:' in log and np.array_equal(out, g['raw'].astype(np.float64))
    g = load_golden('correct_u16_dates')
    cal = ip.CameraCalibration()
    cal.addDarkCurrent(g['d1'], date='01 Jan 15 - 10:00')
    cal.addDarkCurrent(g['d3'], date='01 Jan 17 - 10:00')
    cal.addDarkCurrent(g['d2'], date='01 Jan 16 - 10:00')
    for tag, date in (('none', None), ('mid', '01 Jun 16 - 00:00'), ('old', '01 Jan 14 - 00:00'),
                      ('new', '01 Jan 18 - 00:00'), ('bad', 'not a date')):
        out, _ = _quiet(cal.correct, g['raw'], threshold=0, date=date)
        # float32 dark maps: the float64 reference keeps raw - dark exactly, the float32 chain rounds it once
        assert np.array_equal(out, g['out_' + tag].astype(np.float32).astype(np.float64)), tag


def test_correct_error_conventions(ip):
    cal = ip.CameraCalibration()
    cal.addDarkCurrent(np.zeros((8, 8), np.float32))
    with pytest.raises(Exception, match='array shapes are different'):
        _quiet(cal.correct, np.zeros((8, 9), np.uint16))
    with pytest.raises(Exception):           # no noise calibration: the function is estimated from the exposures, which
        _quiet(cal.correct, [np.zeros((8, 8), np.uint16)] * 2)     # two all-zero 8x8 frames cannot support (the reference fails in curve_fit too)
    out, log = _quiet(cal.correct, [np.ones((8, 8), np.uint16)], threshold=0)
    assert np.array_equal(out, np.ones((8, 8)))
    # a dark map of the wrong shape slipped into the store: printed, stage skipped, pipeline continues
    cal.coeffs['dark current'][0][2] = np.zeros((3, 3), np.float32)
    out, log = _quiet(cal.correct, np.ones((8, 8), np.uint16), threshold=0)
    assert 'Error:' in log and np.array_equal(out, np.ones((8, 8)))


# ---------------------------------------------------------------------------- batches
def test_correct_batch_device_and_host(ip):
    H, W, n = 96, 128, 7
    g = load_golden('correct_u16_keep1')
    cal = _cal(ip, g)
    frames = np.stack([synth.scene(H, W, 30 + i, np.uint16) for i in range(n)])
    single = []
    for i in range(n):
        o, _ = _quiet(cal.correct, frames[i], threshold=0.1)
        single.append(o)
    single = np.stack(single)
    dev_out = cal.correct_batch(_dev(frames), threshold=0.1)
    assert dev_out.dtype == torch.float32 and dev_out.is_cuda
    assert np.array_equal(dev_out.cpu().numpy().astype(np.float64), single)
    host_out = cal.correct_batch(frames, threshold=0.1)
    assert host_out.dtype == np.float32 and np.array_equal(host_out.astype(np.float64), single)
    host64 = cal.correct_batch(frames, threshold=0.1, out_dtype=np.float64)
    assert np.array_equal(host64, single)
    # pinned buffers + cropped output + more frames than ring slots
    from imgprocessor_b200.engine import pinned_empty
    pin_in = pinned_empty(frames.shape, np.uint16)
    pin_in[...] = frames
    l = cal.getLens(None, None)
    l.getUndistortRectifyMap(W, H)
    x, y, w, h = (int(v) for v in l.roi)
    pin_out = pinned_empty((n, h, w), np.float32)
    r = cal.correct_batch(pin_in, threshold=0.1, keep_size=False, out=pin_out)
    assert r is pin_out and np.array_equal(pin_out.astype(np.float64), single[:, y:y + h, x:x + w])


@pytest.mark.parametrize('ndev', [2, 3])
def test_correct_batch_sharded_over_devices(ip, ndev):
    """CameraCalibration.correct_batch(frames, devices=...): host frames split contiguously over several contexts, one host
    thread each, results in one output array — equal to the one-device result.  With fewer physical GPUs than requested the
    same device is used twice (a second context), which exercises the sharding / threading logic on a one-GPU box; with
    >= 2 GPUs the shards really run on different devices (contexts, calibration upload, attribute caches per device)."""
    H, W, n = 96, 128, 11
    g = load_golden('correct_u16_keep1')
    cal = _cal(ip, g)
    frames = np.stack([synth.scene(H, W, 70 + i, np.uint16) for i in range(n)])
    one = cal.correct_batch(frames, threshold=0.1)
    have = torch.cuda.device_count()
    devices = [i % have for i in range(ndev)]
    got = cal.correct_batch(frames, threshold=0.1, devices=devices)
    assert got.dtype == np.float32 and np.array_equal(got, one)
    l = cal.getLens(None, None)
    l.getUndistortRectifyMap(W, H)
    x, y, w, h = (int(v) for v in l.roi)
    from imgprocessor_b200.engine import pinned_empty
    pin_out = pinned_empty((n, h, w), np.float64)
    r = cal.correct_batch(frames, threshold=0.1, keep_size=False, out=pin_out, out_dtype=np.float64, devices=devices)
    assert r is pin_out and np.array_equal(pin_out, one[:, y:y + h, x:x + w].astype(np.float64))
    assert np.array_equal(cal.correct_batch(frames[:1], threshold=0.1, devices=devices), one[:1])     # fewer frames than devices
    assert np.array_equal(cal.correct_batch(frames, threshold=0.1, devices=[0]), one)
    with pytest.raises(ValueError):
        cal.correct_batch(_dev(frames), devices=devices)


def test_two_contexts_on_two_devices_in_one_process(ip):
    """the shared-memory opt-in of the TMA kernels (cudaFuncSetAttribute) is per device: a context on a second device of the
    same process must launch them as well (ADVICE r1: the attribute used to be cached process-wide)"""
    if torch.cuda.device_count() < 2:
        pytest.skip('needs two CUDA devices')
    H, W = 96, 128
    raw, dark, flat = _case(H, W, 5)
    outs = []
    for dev in (0, 1):
        e = ip.engine_mod.Engine(H, W, dev)
        e.set_dark(dark)
        e.set_flat(flat)
        p = synth.lens_moderate(H, W)
        import cv2
        K, d = synth.camera_matrix(p), synth.dist_coeffs(p)
        P, _ = cv2.getOptimalNewCameraMatrix(K, d, (W, H), 1, (W, H))
        e.set_lens(K, d, P)
        frames = torch.from_numpy(np.stack([raw] * 5)).to('cuda:%d' % dev)
        with torch.cuda.device(dev):
            outs.append(e.correct_batch(frames, 0.1, 3).cpu().numpy())
            out5, _ = e.pointwise_median(frames, 0.1, 5)
            outs.append(out5.cpu().numpy())
        e.close()
    assert np.array_equal(outs[0], outs[2]) and np.array_equal(outs[1], outs[3])


def test_out_tensors_are_validated(ip):
    """caller-supplied output tensors reach the kernels by pointer: wrong shape / device / layout must raise, not scribble"""
    H, W, n = 64, 96, 3
    e = _eng(ip, H, W)
    frames = _dev(np.stack([synth.scene(H, W, i, np.uint16) for i in range(n)]))
    good = torch.empty((n, H, W), dtype=torch.float32, device='cuda')
    e.correct_batch(frames, 0.1, 3, out=good)
    for bad in (torch.empty((n - 1, H, W), dtype=torch.float32, device='cuda'),
                torch.empty((n, H, W + 1), dtype=torch.float32, device='cuda')[:, :, :W],
                torch.empty((n, H, W), dtype=torch.float32)):
        with pytest.raises(ValueError):
            e.correct_batch(frames, 0.1, 3, out=bad)
        with pytest.raises(ValueError):
            e.pointwise_median(frames, 0.1, 3, out=bad)


def test_correct_host_chunks_small_frames(ip):
    """small frames go through the host pipeline in chunks of up to 16 per ring slot: more chunks than slots, a ragged last
    chunk, pinned and pageable buffers — same output as the device-resident chain"""
    H, W, n = 96, 128, 103
    g = load_golden('correct_u16_keep1')
    cal = _cal(ip, g)
    _quiet(cal.correct, g['raw'], threshold=0.1)                         # uploads the calibration into the engine
    e = ip.engine_mod.get_engine(H, W)
    rng = np.random.default_rng(8)
    frames = (synth.scene(H, W, 70, np.uint16)[None].astype(np.int64) + rng.integers(-200, 200, (n, H, W))).clip(0, 65535).astype(np.uint16)
    want = e.correct_batch(_dev(frames), threshold=0.1).cpu().numpy()
    got = e.correct_host(frames, threshold=0.1)                          # pageable
    assert np.array_equal(got, want)
    pin_in = ip.engine_mod.pinned_empty(frames.shape, np.uint16)
    pin_out = ip.engine_mod.pinned_empty(frames.shape, np.float32)
    pin_in[...] = frames
    pin_out[...] = -1
    e.correct_host(pin_in, out=pin_out, threshold=0.1)
    assert np.array_equal(pin_out, want)
    assert np.array_equal(e.correct_host(frames[:5], threshold=0.1), want[:5])     # fewer frames than one chunk


def test_calibration_modified_in_place_is_uploaded_again(ip):
    """the reference reads its calibration arrays on every call; the engine's upload cache must notice an in-place edit"""
    g = dict(load_golden('correct_u16_keep1'))
    g['dark'] = g['dark'].copy()
    cal = _cal(ip, g, lens=False)
    raw = g['raw']
    out1, _ = _quiet(cal.correct, raw, threshold=0.1)
    g['dark'] += 50.0                                                # same array object, new content
    out2, _ = _quiet(cal.correct, raw, threshold=0.1)
    want = refpath.correct(raw, g['dark'], g['flat'], None, 0.1)
    assert not np.array_equal(out1, out2)
    assert np.abs(out2 - want).max() <= 1e-5 * 65535
    g['dark'][11, 13] += 4000.0                                      # a single patched pixel must be noticed as well
    out3, _ = _quiet(cal.correct, raw, threshold=0.1)
    want = refpath.correct(raw, g['dark'], g['flat'], None, 0.1)
    assert np.abs(out3 - want).max() <= 1e-5 * 65535 and not np.array_equal(out2, out3)


def test_chain_overlap_mode_is_identical(ip):
    """IMGCORR_OPT_CHAIN_OVERLAP: K1 of group g+1 on the internal high-priority stream while K2 of group g runs — same
    output for every group size (buffer hand-off by events), with and without profiling brackets"""
    H, W, n = 96, 128, 11
    g = load_golden('correct_u16_keep1')
    cal = _cal(ip, g)
    frames = _dev(np.stack([synth.scene(H, W, 50 + i, np.uint16) for i in range(n)]))
    e = ip.engine_mod.get_engine(H, W)
    _quiet(cal.correct, frames[0].cpu().numpy(), threshold=0.1)            # uploads the calibration into the engine
    e.set_option(ip.lib_mod.OPT_CHAIN_OVERLAP, 0)                          # reference result: everything on one stream
    want = e.correct_batch(frames, threshold=0.1).cpu().numpy()
    try:
        e.set_option(ip.lib_mod.OPT_CHAIN_OVERLAP, 1)
        for group in (1, 2, 3, 4, 16):
            e.set_option(ip.lib_mod.OPT_CHAIN_GROUP, group)
            for prof in (0, 1, 2):
                e.set_option(ip.lib_mod.OPT_PROFILE, prof)
                for rep in range(3):
                    got = e.correct_batch(frames, threshold=0.1)
                assert np.array_equal(got.cpu().numpy(), want), (group, prof)
                e.profile_read()
    finally:
        e.set_option(ip.lib_mod.OPT_PROFILE, 0)
        e.set_option(ip.lib_mod.OPT_CHAIN_OVERLAP, 1)                      # the library default
        e.set_option(ip.lib_mod.OPT_CHAIN_GROUP, 16)


# ---------------------------------------------------------------------------- BASELINE.json sizes
def test_config1_1024_f32_full_chain(ip):
    """configs[0]: one 1024x1024 float32 frame, dark + flat + 3x3 + 5-coefficient lens, vs the float64
    reference path (refpath == unmodified reference, pinned by test_oracle_golden)."""
    H = W = 1024
    raw = synth.scene(H, W, 0, np.float32)
    dark, flat = synth.dark_map(H, W), synth.flat_map(H, W)
    p = synth.lens_moderate(H, W)
    K, d = synth.camera_matrix(p), synth.dist_coeffs(p)
    cal = ip.CameraCalibration()
    cal.addDarkCurrent(dark)
    cal.addFlatField(flat)
    l = ip.LensDistortion({})
    l.setCameraParams(*p)
    l._coeffs['shape'] = (H, W)
    cal.addLens(l)
    out, _ = _quiet(cal.correct, raw, threshold=0.1)
    ref = refpath.correct(raw, dark, flat, (K, d), 0.1)
    assert np.abs(out - ref).max() / 4095.0 < 1e-5
    mapx, mapy, P, roi = refpath.undistort_rectify_map(K, d, W, H)
    want, mask = models.correct_chain_f32(raw, dark, flat, 0.1, 3, mapxy=(mapx, mapy))   # cv2's own maps
    assert (out != want).sum() == 0


@pytest.mark.parametrize('variant', [1, 2, 3])
def test_config2_4096x3000_u16_k1(ip, variant):
    """configs[1]: a 4096x3000 uint16 frame through K1, bit-exact against the oracle at full size."""
    H, W = 3000, 4096
    raw, dark, flat = synth.scene(H, W, 1, np.uint16), synth.dark_map(H, W), synth.flat_map(H, W)
    e = _eng(ip, H, W, variant)
    e.set_dark(dark)
    e.set_flat(flat)
    out, mask = e.pointwise_median(_dev(raw), 0.1, 3, want_mask=True)
    x = models.pointwise_model(raw, dark, flat, True)
    want, wmask = models.median_threshold_model(x, 0.1, 3)
    assert np.array_equal(out.cpu().numpy(), want)
    if mask is not None:
        assert np.array_equal(mask.cpu().numpy().astype(bool), wmask)
    assert 0.001 < wmask.mean() < 0.05
    e.set_option(ip.lib_mod.OPT_K1_VARIANT, 0)


def test_config3_chain_full_size_properties(ip):
    """configs[2] frame size: full chain on a few 4096x3000 frames; frame independence (batch == single),
    remap against cv2's own maps at full size, linearity of the border (no lens -> identity)."""
    H, W, n = 3000, 4096, 3
    dark, flat = synth.dark_map(H, W), synth.flat_map(H, W)
    p = synth.lens_moderate(H, W)
    K, d = synth.camera_matrix(p), synth.dist_coeffs(p)
    mapx, mapy, P, roi = refpath.undistort_rectify_map(K, d, W, H)
    e = _eng(ip, H, W, 0)
    e.set_dark(dark)
    e.set_flat(flat)
    e.set_lens(K, d, P)
    frames = torch.stack([_dev(synth.scene(H, W, 100 + i, np.uint16)) for i in range(n)])
    out = e.correct_batch(frames, 0.1, 3)
    one = e.correct_batch(frames[1], 0.1, 3)
    assert torch.equal(out[1], one)
    raw1 = frames[1].cpu().numpy()
    want, _ = models.correct_chain_f32(raw1, dark, flat, 0.1, 3, mapxy=(mapx, mapy))
    assert np.array_equal(one.cpu().numpy(), want)


def test_config4_f32_5x5_strong_lens(ip):
    """configs[3] at 2048x2048 (the oracle's 5x5 partition at 8192^2 needs ~7 GB): float32 frame, direct
    medianThreshold(size=5) then LensDistortion.correct with the strong lens."""
    H = W = 2048
    raw = synth.scene(H, W, 2, np.float32)
    med, ind = ip.medianThreshold(raw, 0.1, 5)
    want, wmask = models.median_threshold_model(raw, 0.1, 5)
    assert np.array_equal(med, want) and np.array_equal(ind, wmask)
    p = synth.lens_strong(H, W)
    l = ip.LensDistortion({})
    l.setCameraParams(*p)
    out = l.correct(med, keepSize=True)
    ref = refpath.lens_correct(want, synth.camera_matrix(p), synth.dist_coeffs(p), keep_size=True)
    assert (out != ref).mean() < 1e-6          # analytic map vs cv2's: at most a stray 1/32-px flip
    assert np.abs(out - ref).max() / 4095.0 < 1e-3


def test_config4_8192_full_size(ip):
    """configs[3] at its FULL size: one 8192x8192 float32 frame through dark + flat + 5x5 medianThreshold + the strong lens.
    (1) every 5-bit fixed-point coordinate of the analytic map equals OpenCV's (67 M pixels, compared in slabs);
    (2) bands of the chain's output (top edge, two interior, bottom edge) equal the band-wise oracle chain evaluated with
    cv2's own maps, bit for bit — the oracle never holds more than a band, so the test stays within a few GB of host memory."""
    import cv2
    from oracle import bands
    H = W = 8192
    raw = synth.scene(H, W, 2, np.float32)
    dark, flat = synth.dark_map(H, W), synth.flat_map(H, W)
    p = synth.lens_strong(H, W)
    K, d = synth.camera_matrix(p), synth.dist_coeffs(p)
    P, roi = cv2.getOptimalNewCameraMatrix(K, d, (W, H), 1, (W, H))
    mapx, mapy = cv2.initUndistortRectifyMap(K, d, None, P, (W, H), cv2.CV_32FC1)
    e = ip.engine_mod.Engine(H, W, 0)
    try:
        e.set_dark(dark)
        e.set_flat(flat)
        e.set_lens(K, d, P)
        mx, my = e.undistort_maps()
        mx, my = mx.cpu().numpy(), my.cpu().numpy()
        for r0 in range(0, H, 1024):
            a = models.fixed_point_coords(mx[r0:r0 + 1024], my[r0:r0 + 1024])
            b = models.fixed_point_coords(mapx[r0:r0 + 1024], mapy[r0:r0 + 1024])
            for u, v in zip(a, b):
                assert np.array_equal(u, v), r0
        del mx, my
        out = e.correct_batch(_dev(raw), 0.1, 5)
        again = e.correct_batch(_dev(raw), 0.1, 5)                  # second call: K2 reads its coordinate cache
        assert torch.equal(out, again)
        for r0, r1 in bands.default_bands(H, 32) + [(1500, 1532), (6000, 6032)]:
            want = bands.chain_band(raw, dark, flat, mapx, mapy, r0, r1, 0.1, 5)
            assert np.array_equal(out[r0:r1].cpu().numpy(), want), (r0, r1)
        k1, mask = e.pointwise_median(_dev(raw), 0.1, 5, flags=0, want_mask=True)          # direct medianThreshold(size=5)
        for r0, r1 in ((0, 40), (4000, 4040), (H - 40, H)):
            want = bands.k1_band(raw, None, None, r0, r1, 0.1, 5)
            assert np.array_equal(k1[r0:r1].cpu().numpy(), want), (r0, r1)
    finally:
        e.close()


def test_config5_6000x4000_streamed_from_pinned_pool(ip):
    """configs[4]: 6000x4000 uint16 frames cycled from a small pool of pinned buffers through the host-buffer chain; the
    streamed result equals the device-resident chain, and K1 of that chain equals the oracle on a band of rows"""
    import cv2
    H, W, pool = 4000, 6000, 3
    e = ip.engine_mod.get_engine(H, W)
    dark, flat = synth.dark_map(H, W), synth.flat_map(H, W)
    e.set_dark(dark)
    e.set_flat(flat)
    p = synth.lens_moderate(H, W)
    K, d = synth.camera_matrix(p), synth.dist_coeffs(p)
    P, _ = cv2.getOptimalNewCameraMatrix(K, d, (W, H), 1, (W, H))
    e.set_lens(K, d, P)
    src = synth.scene_torch(pool, H, W, 3, torch.device('cuda', 0), 'uint16')
    h_in = ip.engine_mod.pinned_empty((pool, H, W), np.uint16)
    h_out = ip.engine_mod.pinned_empty((pool, H, W), np.float32)
    h_in[...] = src.cpu().numpy()
    for rep in range(3):                                     # the pool is reused, as the streaming config does
        h_out[...] = -1
        e.correct_host(h_in, out=h_out)
        assert np.array_equal(h_out, e.correct_batch(src).cpu().numpy())
    k1, _ = e.pointwise_median(src[0], 0.1, 3)
    rows = slice(1990, 2060)
    band = slice(rows.start - 1, rows.stop + 1)
    want, _ = models.median_threshold_model(models.pointwise_model(h_in[0][band], dark[band], flat[band], True), 0.1, 3)
    assert np.array_equal(k1[rows].cpu().numpy(), want[1:-1])
    e.set_lens(None, None, None)


def test_to_numpy_staged_copy(ip):
    """engine.to_numpy (pinned staging + threaded copy for large results) returns exactly tensor.cpu().numpy()"""
    for shape, dt in (((3000, 4096), torch.float64), ((5, 700, 900), torch.float32), ((1200, 1100), torch.uint16),
                      ((10, 10), torch.float64), ((2049, 1025), torch.uint8)):
        t = (torch.rand(shape, device='cuda') * 200).to(dt)
        a = ip.engine_mod.to_numpy(t)
        assert a.flags.writeable and np.array_equal(a, t.cpu().numpy())
    t = torch.rand((2000, 3000), device='cuda', dtype=torch.float64)[:, ::2]          # non-contiguous view
    assert np.array_equal(ip.engine_mod.to_numpy(t), t.cpu().numpy())
    b = ip.engine_mod.to_numpy(torch.zeros((1500, 1500), device='cuda', dtype=torch.float64))   # staging reuse must not alias
    assert not b.any() and a.any()
