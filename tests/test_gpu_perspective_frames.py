"""The chain's perspective stage with one homography per frame (imgcorr_set_perspective_frames, Engine.set_perspective
with M of shape (n, 3, 3), CameraCalibration.correct_batch(perspective=[pc_0, ..., pc_n-1])) against the oracle, frame
by frame and bit for bit: frame i of a call is oracle.warp.warp_perspective_model of the float32 oracle chain frame i
(widened to float64 where the call returns float64) with matrix i.  Every comparison is np.array_equal(...,
equal_nan=True).  The full-size case compares against the per-frame two-step device composition (correct_batch, then
Engine.warp_perspective with each frame's matrix): the numpy model is too slow at 12 Mpx."""
import contextlib
import io

import numpy as np
import pytest

from imgprocessor_b200 import synth
from quantise_model import quantise
from test_gpu_chain import (SPIN_CYCLES, _calibration, _crop, _dev, _file_image, _flags, _frames, _host, _lens, _maps,
                            _Options, _oracle, _same, ip)  # noqa: F401  (ip is a fixture)
from test_gpu_perspective_chain import QUADS, _calibrated, _homography, _stage, _Want, _warp

pytestmark = pytest.mark.gpu

torch = pytest.importorskip('torch')

SINGULAR = np.array([[1.0, 2.0, 0.0], [2.0, 4.0, 0.0], [0.0, 0.0, 1.0]])      # det == 0: cv::invert gives zeros


def _jitter(M, i, h, w):
    """M followed by a shift of a few pixels and a rotation of a fraction of a degree about the destination's centre,
    different for every i"""
    a = np.deg2rad(0.3 * np.sin(1.7 * i + 0.4))
    tx, ty = 3.0 * np.sin(0.9 * i + 1.0), 2.0 * np.cos(1.3 * i)
    cx, cy = w / 2.0, h / 2.0
    c, s = np.cos(a), np.sin(a)
    R = np.array([[c, -s, cx - c * cx + s * cy + tx], [s, c, cy - s * cx - c * cy + ty], [0.0, 0.0, 1.0]])
    return R @ M


def _table(h, w, n, kinds, dsize='same'):
    """(n x 3 x 3 matrices, dsize) for an h x w chain frame: frame i takes kinds[i % len(kinds)] — a quad of QUADS jittered
    per frame, 'singular', or 'zoomout' (a 0.3x shrink: a 32-pixel tile reads ~107 source columns, more than K3's staged
    box holds, so that frame falls back to the global gathers)"""
    M0, ds = _stage(h, w, quad='mild', dsize=dsize)
    out = []
    for i in range(n):
        k = kinds[i % len(kinds)]
        if k == 'singular':
            out.append(SINGULAR)
        elif k == 'zoomout':
            out.append(np.array([[0.3, 0.02, 1.5], [-0.01, 0.3, 2.0], [0.0, 0.0, 1.0]]))
        else:
            out.append(_jitter(_stage(h, w, quad=k, dsize=dsize)[0], i, ds[1], ds[0]))
    return np.stack(out), ds


MIXED = ['mild', 'strong', 'outside', 'singular', 'zoomout', 'mild']


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
def test_device_frames_vs_oracle(ip, shape, dtype):
    """6 frames in one group, every frame with its own matrix: mild, strong and partly-outside quads, a singular matrix and
    a zoom-out whose windows do not fit K3's staged box, next to frames whose windows fit.  Base: lens on, full frame,
    float32 out, K3 variant auto (its L1 gathers for a table).  Then the lens off, the roi window, float64 out (with and
    without the roi), uint16 out (quantise of the float32 result), and K3 forced to its L1 gathers (1) and to its staged
    tiles (2: refused, a table is never eligible for them)."""
    H, W = shape
    n = 6
    L = ip.lib_mod
    e, dark, flat, roi, maps = _setup(ip, H, W, 3)
    raw = _frames(H, W, n, 40, dtype)
    want = _Want(raw, dark, flat, maps)
    dev = _dev(raw)
    base = dict(lens=True, window=None, odt=np.float32, variant=0)
    cases = [base] + [dict(base, **v) for v in (
        {'lens': False}, {'window': roi}, {'odt': np.float64}, {'odt': np.float64, 'window': roi}, {'odt': np.uint16},
        {'variant': 1}, {'variant': 2}, {'variant': 2, 'odt': np.uint16, 'window': roi})]
    fl = _flags(L, 0.1) | L.DO_PERSPECTIVE
    try:
        with _Options(ip, e) as o:
            for c in cases:
                o.set(L.OPT_K3_VARIANT, c['variant'])
                Ms, dsize = _table(*_src_shape(e, c['window'], c['lens']), n, MIXED)
                e.set_perspective(Ms, dsize, 2.5)
                tdt = {np.float32: torch.float32, np.float64: torch.float64, np.uint16: torch.uint16}[c['odt']]
                call = lambda: e.correct_batch(dev, flags=fl, use_lens=c['lens'], window=c['window'], out_dtype=tdt)  # noqa: E731
                if c['variant'] == 2:
                    with pytest.raises(L.ImgcorrError) as err:
                        call()
                    assert err.value.status == L.ERR_INVALID
                    continue
                got = _host(call())
                assert got.shape == (n, dsize[1], dsize[0])
                for i in range(n):
                    wdt = np.float64 if c['odt'] == np.float64 else np.float32
                    w = want(i, Ms[i], dsize, 2.5, c['window'], wdt, c['lens'])
                    if c['odt'] == np.uint16:
                        w = quantise(w, np.uint16)
                    assert _same(got[i], w), (c, i)
    finally:
        e.set_option(L.OPT_K3_VARIANT, 0)
        e.set_perspective(None, None)


# ---------------------------------------------------------------------------------------------- 2. group seams
def test_group_seams_vs_oracle(ip):
    """11 frames in groups of 4 (4 + 4 + 3), overlap on and off: with the lens and the roi in float32, with the lens on
    the full frame in float32, and without a lens in float64.  Frame i of the call takes matrix i across every seam."""
    H, W, n = 96, 256, 11
    L = ip.lib_mod
    e, dark, flat, roi, maps = _setup(ip, H, W, 5)
    raw = _frames(H, W, n, 60, np.uint16)
    want = _Want(raw, dark, flat, maps)
    dev = _dev(raw)
    try:
        with _Options(ip, e) as o:
            o.set(L.OPT_CHAIN_GROUP, 4)
            for lens, window, tdt, odt in ((True, roi, torch.float32, np.float32), (True, None, torch.float32, np.float32),
                                           (False, None, torch.float64, np.float64)):
                Ms, dsize = _table(*_src_shape(e, window, lens), n, ['strong', 'mild', 'outside'], dsize='larger')
                e.set_perspective(Ms, dsize, 0.0)
                for overlap in (1, 0):
                    o.set(L.OPT_CHAIN_OVERLAP, overlap)
                    got = _host(e.correct_batch(dev, flags=_flags(L, 0.1) | L.DO_PERSPECTIVE, use_lens=lens, window=window,
                                                out_dtype=tdt))
                    for i in range(n):
                        assert _same(got[i], want(i, Ms[i], dsize, 0.0, window, odt, lens)), (lens, window, overlap, i)
    finally:
        e.set_perspective(None, None)


# ---------------------------------------------------------------------------------------------- 3. a table of one matrix
@pytest.mark.parametrize('variant', [0, 1, 2])
def test_equal_table_is_the_single_matrix_stage(ip, variant):
    """a table whose n matrices are all M gives the output of imgcorr_set_perspective(M), for float32, float64 and uint16
    output; and the two setters replace each other in both directions.  With K3 forced to its staged tiles (2) the single
    matrix runs them and the table is refused."""
    H, W, n = 96, 256, 9
    L = ip.lib_mod
    e, dark, flat, roi, maps = _setup(ip, H, W, 23)
    dev = _dev(_frames(H, W, n, 70, np.uint16))
    M, dsize = _stage(H, W, quad='strong', dsize='smaller')
    fl = _flags(L, 0.1) | L.DO_PERSPECTIVE
    try:
        with _Options(ip, e) as o:
            o.set(L.OPT_K3_VARIANT, variant)
            o.set(L.OPT_CHAIN_GROUP, 5)
            for tdt in (torch.float32, torch.float64, torch.uint16):
                if variant == 2 and tdt == torch.float64:
                    continue                                     # float64 frames have no staged tiles
                e.set_perspective(M, dsize, 1.25)
                one = e.correct_batch(dev, flags=fl, out_dtype=tdt)
                e.set_perspective(np.stack([M] * n), dsize, 1.25)
                if variant == 2:
                    with pytest.raises(L.ImgcorrError) as err:
                        e.correct_batch(dev, flags=fl, out_dtype=tdt)
                    assert err.value.status == L.ERR_INVALID, tdt
                    table = one
                else:
                    table = e.correct_batch(dev, flags=fl, out_dtype=tdt)
                e.set_perspective(M, dsize, 1.25)
                again = e.correct_batch(dev, flags=fl, out_dtype=tdt)
                assert torch.equal(one, table) and torch.equal(one, again), tdt
    finally:
        e.set_option(L.OPT_K3_VARIANT, 0)
        e.set_perspective(None, None)


# ---------------------------------------------------------------------------------------------- 4. host pipeline
@pytest.mark.parametrize('slots', [2, 3, 8])
def test_host_pipeline_vs_oracle(ip, slots):
    """correct_host with a table: 37 small frames in chunks of 16 per ring slot (16 + 16 + 5), pageable / pinned input x
    pageable / pinned output, float32 out; then float64 out with the roi window.  Chunk k's frames take matrices 16k..."""
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
            Ms, dsize = _table(H, W, n, ['strong', 'mild', 'outside', 'singular'], dsize='larger')
            e.set_perspective(Ms, dsize, 3.0)
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
                        assert _same(got[i], want(i, Ms[i], dsize, 3.0)), (src is pin_in, pinned_out, i)
            Ms, dsize = _table(roi[3], roi[2], n, ['outside', 'mild'], dsize='smaller')
            e.set_perspective(Ms, dsize, 0.0)
            got = e.correct_host(raw, flags=fl, window=roi, out_dtype=np.float64)
            for i in range(n):
                assert _same(got[i], want(i, Ms[i], dsize, 0.0, roi, np.float64)), ('f64 roi', i)
    finally:
        e.set_perspective(None, None)


# ---------------------------------------------------------------------------------------------- 5. file bytes
def test_file_bytes_vs_oracle(ip):
    """correct_file_bytes on big-endian frames with a 32-byte header and 20-byte gaps, 8 frames in groups of 5"""
    H, W, n = 70, 250, 8
    L = ip.lib_mod
    e, dark, flat, roi, maps = _setup(ip, H, W, 11)
    raw = _frames(H, W, n, 160, np.uint16)
    want = _Want(raw, dark, flat, maps)
    buf = _dev(_file_image(raw, 32, 20, big_endian=True))
    Ms, dsize = _table(H, W, n, ['mild', 'strong'], dsize='larger')
    try:
        with _Options(ip, e) as o:
            o.set(L.OPT_CHAIN_GROUP, 5)
            e.set_perspective(Ms, dsize, 0.5)
            got = _host(e.correct_file_bytes(buf, 32, n, gap=20, big_endian=True, dtype=torch.uint16,
                                             flags=_flags(L, 0.1) | L.DO_PERSPECTIVE))
            for i in range(n):
                assert _same(got[i], want(i, Ms[i], dsize, 0.5)), i
    finally:
        e.set_perspective(None, None)


# ---------------------------------------------------------------------------------------------- 6. public API
def test_camera_calibration_correct_batch_with_a_list(ip):
    """cal.correct_batch(frames, perspective=[pc_0, ...], out_dtype=float64)[i] == pcs[i].correct(cal.correct(frames[i]))
    for keep_size True and False: host frames, CUDA tensors and two contexts on one device (devices=[0, 0], 5 frames split
    3 + 2, so the second context's frame 0 is the batch's frame 3); float32 output against the oracle.  A single
    PerspectiveCorrection after the list is the single-matrix stage again."""
    from imgprocessor_b200.camera import PerspectiveCorrection
    H, W, n = 96, 256, 5
    cal = _calibrated(ip, H, W)
    raw = _frames(H, W, n, 140, np.uint16)
    for keep_size in (True, False):
        ref, pcs, want = _list_case(cal, raw, keep_size)
        got = cal.correct_batch(raw, keep_size=keep_size, perspective=pcs, out_dtype=np.float64)
        assert _same(got, want), keep_size
        got = _host(cal.correct_batch(_dev(raw), keep_size=keep_size, perspective=pcs, out_dtype=torch.float64))
        assert _same(got, want), ('tensor', keep_size)
        got = cal.correct_batch(raw, keep_size=keep_size, perspective=pcs, out_dtype=np.float64, devices=[0, 0])
        assert _same(got, want), ('devices=[0, 0]', keep_size)
        # a single PerspectiveCorrection: every frame with pcs[1]'s matrix
        got = cal.correct_batch(raw, keep_size=keep_size, perspective=pcs[1], out_dtype=np.float64)
        with contextlib.redirect_stdout(io.StringIO()):
            assert _same(got, np.stack([pcs[1].correct(r) for r in ref])), ('single', keep_size)
    # float32 output: the float32 chain frame warped in float32 with its own matrix
    maps = _maps(ip.engine_mod.get_engine(H, W))
    dark, flat = _calibration(H, W, 9)
    Ms, dsize = _table(H, W, n, MIXED, dsize='smaller')
    pcs = []
    for i in range(n):
        pc = PerspectiveCorrection((H, W), new_size=(dsize[1], dsize[0]))
        pc.setReference(Ms[i])
        pcs.append(pc)
    got = cal.correct_batch(raw, perspective=pcs)
    for i in range(n):
        assert _same(got[i], _warp(_oracle(raw[i], dark, flat, 0.1, 3, maps), Ms[i], dsize, 0.0)), i


def _list_case(cal, raw, keep_size):
    """(the corrected frames, one PerspectiveCorrection per frame, pcs[i].correct(corrected frame i) stacked)"""
    from imgprocessor_b200.camera import PerspectiveCorrection
    n = raw.shape[0]
    with contextlib.redirect_stdout(io.StringIO()):
        ref = [cal.correct(raw[i], keep_size=keep_size) for i in range(n)]
    sh = ref[0].shape
    Ms, dsize = _table(*sh, n, ['mild', 'strong', 'outside'], dsize='larger')
    pcs = []
    for i in range(n):
        pc = PerspectiveCorrection(sh, new_size=(dsize[1], dsize[0]), cv2_opts={'borderValue': 0.75})
        pc.setReference(Ms[i])
        pcs.append(pc)
    with contextlib.redirect_stdout(io.StringIO()):
        want = np.stack([pcs[i].correct(ref[i]) for i in range(n)])
    return ref, pcs, want


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='a split over several GPUs needs two or more')
def test_camera_calibration_list_over_every_gpu(ip):
    """devices=range(number of GPUs): every device gets the matrices of its own shard"""
    H, W, n = 96, 256, 7
    cal = _calibrated(ip, H, W)
    raw = _frames(H, W, n, 150, np.uint16)
    for keep_size in (True, False):
        _, pcs, want = _list_case(cal, raw, keep_size)
        got = cal.correct_batch(raw, keep_size=keep_size, perspective=pcs, out_dtype=np.float64,
                                devices=range(torch.cuda.device_count()))
        assert _same(got, want), keep_size


# ---------------------------------------------------------------------------------------------- 7. refusals and replacement
def test_refusals_and_replacement(ip):
    """too few matrices: correct_batch, correct_host and correct_file_bytes fail with ERR_INVALID and write nothing to
    `out`; a tilt factor with a table, and a table of the wrong shape, raise ValueError; replacing the table with a single
    matrix and back gives each stage's own warp; removing the stage refuses the bit"""
    H, W, n = 96, 256, 6
    L = ip.lib_mod
    e, dark, flat, roi, maps = _setup(ip, H, W, 29)
    raw = _frames(H, W, n, 300, np.uint16)
    want = _Want(raw, dark, flat, maps)
    dev = _dev(raw)
    fl = _flags(L, 0.1) | L.DO_PERSPECTIVE
    Ms, dsize = _table(H, W, n, ['mild', 'strong'])
    try:
        e.set_perspective(Ms[:n - 1], dsize, 0.0)
        out = torch.full((n, dsize[1], dsize[0]), -7.0, device=dev.device)
        hout = np.full((n, dsize[1], dsize[0]), -7.0, np.float32)
        buf = _dev(_file_image(raw, 0, 0))
        for call in (lambda: e.correct_batch(dev, flags=fl, out=out), lambda: e.correct_host(raw, out=hout, flags=fl),
                     lambda: e.correct_file_bytes(buf, 0, n, dtype=torch.uint16, flags=fl, out=out)):
            with pytest.raises(L.ImgcorrError) as err:
                call()
            assert err.value.status == L.ERR_INVALID and 'matrices' in str(err.value)
        torch.cuda.synchronize()
        assert bool((out == -7.0).all()) and (hout == -7.0).all()
        got = _host(e.correct_batch(dev[:n - 1], flags=fl))      # as many frames as matrices is fine
        for i in range(n - 1):
            assert _same(got[i], want(i, Ms[i], dsize, 0.0)), i
        with pytest.raises(ValueError, match='tilt factor'):
            e.set_perspective(Ms, dsize, 0.0, tilt_factor=np.ones((H, W)))
        with pytest.raises(ValueError, match=r'\(n, 3, 3\)'):
            e.set_perspective(np.zeros((n, 2, 3)), dsize, 0.0)
        # table -> single matrix -> table
        e.set_perspective(Ms, dsize, 0.0)
        e.set_perspective(Ms[2], dsize, 0.0)
        got = _host(e.correct_batch(dev, flags=fl))
        for i in range(n):
            assert _same(got[i], want(i, Ms[2], dsize, 0.0)), ('single', i)
        e.set_perspective(Ms, dsize, 0.0)
        got = _host(e.correct_batch(dev, flags=fl))
        for i in range(n):
            assert _same(got[i], want(i, Ms[i], dsize, 0.0)), ('table', i)
        # a single matrix with a tilt factor, then a table: the tilt factor is gone (float32 output is accepted again)
        e.set_perspective(Ms[0], dsize, 0.0, tilt_factor=np.ones((H, W)))
        e.set_perspective(Ms, dsize, 0.0)
        got = _host(e.correct_batch(dev, flags=fl, out_dtype=torch.float32))
        assert _same(got[n - 1], want(n - 1, Ms[n - 1], dsize, 0.0))
        e.set_perspective(None, None)
        with pytest.raises(L.ImgcorrError) as err:
            e.correct_batch(dev, flags=fl)
        assert err.value.status == L.ERR_STATE
    finally:
        e.set_perspective(None, None)


def test_replacing_the_table_while_a_call_is_queued(ip):
    """a chain call queued behind a spin kernel on another stream still returns the old table's warp when the table is
    replaced (same and another number of matrices) or swapped for a single matrix before the call has run"""
    H, W, n = 96, 256, 8
    L = ip.lib_mod
    e, dark, flat, roi, maps = _setup(ip, H, W, 31)
    raw = _frames(H, W, n, 400, np.uint16)
    want = _Want(raw, dark, flat, maps)
    dev = _dev(raw)
    fl = _flags(L, 0.1) | L.DO_PERSPECTIVE
    old, dsize = _table(H, W, n, ['strong', 'outside', 'mild'])
    new, _ = _table(H, W, n + 3, ['mild'])
    s = torch.cuda.Stream()
    try:
        with _Options(ip, e) as o:
            o.set(L.OPT_CHAIN_GROUP, 4)
            for replace in (lambda: e.set_perspective(new[:n], dsize, 0.0), lambda: e.set_perspective(new, dsize, 0.0),
                            lambda: e.set_perspective(new[0], dsize, 0.0)):
                e.set_perspective(old, dsize, 0.0)
                e.correct_batch(dev[:2], flags=fl)               # allocation and caches outside the race
                torch.cuda.synchronize()
                with torch.cuda.stream(s):
                    torch.cuda._sleep(SPIN_CYCLES)
                    out = e.correct_batch(dev, flags=fl)
                replace()
                torch.cuda.synchronize()
                got = _host(out)
                bad = [i for i in range(n) if not _same(got[i], want(i, old[i], dsize, 0.0))]
                assert not bad, bad
    finally:
        e.set_perspective(None, None)


# ---------------------------------------------------------------------------------------------- 8. full size
def test_full_size_against_the_two_step_composition(ip):
    """17 uint16 4096x3000 frames with the moderate lens (groups of 16 + 1) through a table of jittered mild homographies
    onto 4000x2900, against correct_batch followed by Engine.warp_perspective of each frame with its own matrix: the full
    frame and the roi window"""
    H, W, n = 3000, 4096, 17
    L = ip.lib_mod
    e = ip.engine_mod.get_engine(H, W)
    e.set_dark(synth.dark_map(H, W))
    e.set_flat(synth.flat_map(H, W))
    roi = _lens(e, H, W)
    src = synth.scene_torch(n, H, W, 7, torch.device('cuda', torch.cuda.current_device()))
    dsize = (4000, 2900)
    try:
        for window in (None, roi):
            sh = _src_shape(e, window)
            M = _homography([(fx * sh[1], fy * sh[0]) for fx, fy in QUADS['mild']],
                            [(0, 0), (4000, 0), (4000, 2900), (0, 2900)])
            Ms = np.stack([_jitter(M, i, 2900, 4000) for i in range(n)])
            e.set_perspective(Ms, dsize, 0.0)
            got = e.correct_batch(src, flags=_flags(L, 0.1) | L.DO_PERSPECTIVE, window=window)
            mid = e.correct_batch(src, window=window)
            assert tuple(got.shape) == (n, 2900, 4000)
            bad = [i for i in range(n) if not torch.equal(got[i], e.warp_perspective(mid[i], Ms[i], dsize))]
            assert not bad, (window, bad)
            del got, mid
    finally:
        e.set_perspective(None, None)
        e.set_lens(None, None, None)
