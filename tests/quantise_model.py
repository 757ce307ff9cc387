"""numpy model of the chain's scaled integer output (out_dtype U16 / U8, imgcorr_set_output_scale), used by the tests and
tools/int_output.py as the reference for quantise<T> in imgprocessor_b200/csrc/imgcorr_core.cuh."""
import numpy as np


def quantise(v, dtype, offset=0.0, gain=1.0):
    """The uint16 / uint8 image the chain returns for the float32 result ``v`` with output scale (offset, gain):
    t = (float64(v) - offset) * gain, two separately rounded float64 operations; 0 where t is NaN or <= 0, the
    dtype's maximum where t >= it (+inf included), t rounded half to even elsewhere.  The scale (0, 1) is OpenCV's
    saturate_cast<T>(v)."""
    dtype = np.dtype(dtype)
    mx = float(np.iinfo(dtype).max)
    with np.errstate(invalid='ignore', over='ignore'):
        t = (np.asarray(v, np.float32).astype(np.float64) - float(offset)) * float(gain)
        return np.where(np.isnan(t), 0.0, np.clip(np.rint(t), 0.0, mx)).astype(dtype)
