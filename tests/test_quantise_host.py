"""The quantiser of the chain's integer output (quantise<T> in imgcorr_core.cuh), compiled with g++ into a small host
harness, against the numpy model quantise_model.quantise, bit for bit.  No GPU needed."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
from hypothesis import given, settings, strategies as st

from quantise_model import quantise

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, 'imgprocessor_b200', 'csrc')

HARNESS = r'''
#include "imgcorr_core.cuh"
#define EXPORT extern "C" __attribute__((visibility("default")))
EXPORT void quantise_u16(const float* v, long n, double offset, double gain, uint16_t* out) {
    for (long i = 0; i < n; ++i) out[i] = imgcorr::quantise<uint16_t>(v[i], offset, gain);
}
EXPORT void quantise_u8(const float* v, long n, double offset, double gain, uint8_t* out) {
    for (long i = 0; i < n; ++i) out[i] = imgcorr::quantise<uint8_t>(v[i], offset, gain);
}
EXPORT void sat_u16(const float* v, long n, uint16_t* out) { for (long i = 0; i < n; ++i) out[i] = imgcorr::sat_u16(v[i]); }
EXPORT void sat_u8(const float* v, long n, uint8_t* out) { for (long i = 0; i < n; ++i) out[i] = imgcorr::sat_u8(v[i]); }
'''


@pytest.fixture(scope='module')
def harness(tmp_path_factory):
    d = tmp_path_factory.mktemp('quantise')
    src, so = d / 'harness.cpp', d / 'libquantise.so'
    src.write_text(HARNESS)
    subprocess.check_call(['g++', '-O2', '-std=c++17', '-ffp-contract=off', '-fPIC', '-shared', '-fvisibility=hidden',
                           '-I', CSRC, '-o', str(so), str(src), '-lm'])
    return ctypes.CDLL(str(so))


def _run(lib, v, dtype, offset, gain):
    v = np.ascontiguousarray(v, np.float32)
    out = np.empty(v.shape, dtype)
    fn = lib.quantise_u16 if np.dtype(dtype) == np.uint16 else lib.quantise_u8
    fn(v.ctypes.data_as(ctypes.c_void_p), ctypes.c_long(v.size), ctypes.c_double(offset), ctypes.c_double(gain),
       out.ctypes.data_as(ctypes.c_void_p))
    return out


def _check(lib, v, dtype, offset=0.0, gain=1.0):
    got = _run(lib, v, dtype, offset, gain)
    want = quantise(v, dtype, offset, gain)
    bad = np.flatnonzero(got != want)
    assert bad.size == 0, 'v=%r offset=%r gain=%r: harness %r, model %r' % (
        np.asarray(v, np.float32).ravel()[bad[:4]], offset, gain, got.ravel()[bad[:4]], want.ravel()[bad[:4]])
    return got


def _f32(*xs):
    return np.array(xs, np.float32)


SPECIAL = _f32(0.0, -0.0, 0.5, 1.5, 2.5, -0.5, -1.5, 0.49999997, 0.50000006, 254.5, 255.5, 256.0, 65534.5, 65535.0,
               65535.5, 65536.0, 1e-45, -1e-45, 1.17549435e-38, 1e-38, np.inf, -np.inf, np.nan, 3e38, -3e38, 3.4028235e38,
               -3.4028235e38, 1.0, 100.25, 7.5)


@pytest.mark.parametrize('dtype', [np.uint16, np.uint8])
def test_special_values_identity_scale(harness, dtype):
    got = _check(harness, SPECIAL, dtype)
    mx = np.iinfo(dtype).max
    by = dict(zip(SPECIAL.tolist(), got.tolist()))
    assert by[0.5] == 0 and by[1.5] == 2 and by[2.5] == 2 and by[-0.5] == 0                 # ties to even, -0.5 -> 0
    assert by[float(np.float32(-0.0))] == 0 and by[float('inf')] == mx and by[float('-inf')] == 0
    assert got[np.isnan(SPECIAL)][0] == 0
    if dtype == np.uint16:
        assert by[65534.5] == 65534 and by[65535.5] == 65535 and by[65536.0] == 65535
    else:
        assert by[254.5] == 254 and by[255.5] == 255


@pytest.mark.parametrize('dtype', [np.uint16, np.uint8])
def test_identity_scale_is_saturate_cast(harness, dtype):
    """with (0, 1) the quantiser is the existing sat_u16 / sat_u8 bit for bit"""
    rng = np.random.default_rng(7)
    v = np.concatenate([SPECIAL, rng.uniform(-10, 70000, 20000).astype(np.float32),
                        (rng.integers(-4, 131080, 20000) * 0.5).astype(np.float32)])
    got = _check(harness, v, dtype)
    sat = np.empty(v.shape, dtype)
    fn = harness.sat_u16 if dtype == np.uint16 else harness.sat_u8
    fn(v.ctypes.data_as(ctypes.c_void_p), ctypes.c_long(v.size), sat.ctypes.data_as(ctypes.c_void_p))
    assert np.array_equal(got, sat)


@pytest.mark.parametrize('dtype', [np.uint16, np.uint8])
@pytest.mark.parametrize('offset,gain', [(0.0, 1.0), (-100.5, 1.0), (1000.0, 0.5), (0.25, 2.0), (0.0, 1e-300),
                                         (0.0, 1e300), (-1e300, 1e-300), (12.5, 1.0 / 3.0), (0.0, 65535.0 / 4095.0),
                                         (1e20, 1e-20), (-3e38, 1e-33)])
def test_scales(harness, dtype, offset, gain):
    rng = np.random.default_rng(abs(hash((offset, gain))) % 2 ** 32)
    v = np.concatenate([SPECIAL, rng.normal(0, 3e4, 5000).astype(np.float32),
                        rng.uniform(-1e6, 1e6, 5000).astype(np.float32)])
    _check(harness, v, dtype, offset, gain)


@pytest.mark.parametrize('dtype', [np.uint16, np.uint8])
def test_exact_ties_after_scaling(harness, dtype):
    """offset / gain that put (v - offset) * gain exactly on .5: round half to even, not half up"""
    k = np.arange(0, 300, dtype=np.float32)
    _check(harness, k + 0.25, dtype, offset=-0.75, gain=0.5)           # (k + 1) * 0.5: a tie for every even k
    got = _check(harness, 2 * k + 1, dtype, offset=0.0, gain=0.5)       # k + 0.5 exactly
    mx = np.iinfo(dtype).max
    want = np.minimum(np.where(k % 2 == 0, k, k + 1), mx).astype(dtype)
    assert np.array_equal(got, want)


def test_float32_value_is_widened_before_the_offset(harness):
    """the offset is subtracted in float64: 16777217 - 16777216 is exact there but not in float32 arithmetic"""
    v = _f32(16777216.0)
    assert _check(harness, v, np.uint16, offset=16777215.0, gain=1.0)[0] == 1
    assert _check(harness, _f32(1.0), np.uint16, offset=0.5, gain=1.0)[0] == 0        # 0.5 -> 0 (even)


finite32 = st.floats(width=32, allow_nan=True, allow_infinity=True, allow_subnormal=True)


@settings(max_examples=400, deadline=None)
@given(v=st.lists(finite32, min_size=1, max_size=64),
       offset=st.floats(min_value=-1e30, max_value=1e30, allow_nan=False, allow_infinity=False),
       gain=st.floats(min_value=1e-300, max_value=1e300, allow_nan=False, allow_infinity=False),
       u8=st.booleans())
def test_hypothesis_values_and_scales(harness, v, offset, gain, u8):
    _check(harness, np.array(v, np.float32), np.uint8 if u8 else np.uint16, offset, gain)


@settings(max_examples=300, deadline=None)
@given(k=st.integers(min_value=-10, max_value=140000), u8=st.booleans())
def test_hypothesis_half_integers(harness, k, u8):
    v = _f32(k * 0.5, k * 0.5 + 0.25, np.nextafter(np.float32(k * 0.5), np.float32(np.inf)))
    _check(harness, v, np.uint8 if u8 else np.uint16)
