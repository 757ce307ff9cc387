"""float32 vs uint16 output of the batch chain: end-to-end on pinned host frames and device resident.

    python tools/int_output.py [--frames 64] [--reps 5] [--devices N] [--out FILE]

Full chain (dark + flat + nan_to_num + 3x3 median-threshold + moderate lens) on pinned uint16 frames at 4096x3000 and
6000x4000, more frames than the 126 MB L2 holds.  Each rep runs the float32 call and then the uint16 call (identity
output scale), so drifts of the shared machine hit both alike.  Reported per shape and output dtype: the median per-frame
time, Mpx/s and the PCIe bytes per second (raw frames in + results out) of the host-buffer call, and the CUDA-event
time of the same chain on device-resident frames.  --devices N adds the host path sharded over N GPUs
(CameraCalibration.correct_batch(devices=range(N))).  The uint16 results are checked against
quantise(float32 results) of tests/quantise_model.py bit for bit.  Prints the GPU name and power limit, then one JSON object."""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        r = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                           text=True, timeout=60)
        return r.stdout.strip().splitlines()
    except Exception as e:                             # noqa: BLE001 - informational only
        return ['nvidia-smi unavailable: %s' % e]


def frames(H, W, n, pinned_empty):
    from imgprocessor_b200 import synth
    base = [synth.scene(H, W, 100 + i, np.uint16) for i in range(4)]
    out = pinned_empty((n, H, W), np.uint16)
    for i in range(n):
        np.add(base[i % 4], np.uint16(i // 4), out=out[i])
    return out


def calibration(H, W):
    from imgprocessor_b200 import synth
    from oracle import refpath
    p = synth.lens_moderate(H, W)
    K, d = synth.camera_matrix(p), synth.dist_coeffs(p)
    _, _, P, _ = refpath.undistort_rectify_map(K, d, W, H)
    return synth.dark_map(H, W), synth.flat_map(H, W), (K, d, P)


def med(xs):
    return float(np.median(xs))


def run_shape(H, W, n, reps, n_dev):
    import torch
    from imgprocessor_b200 import engine
    from imgprocessor_b200.camera import CameraCalibration, LensDistortion
    from imgprocessor_b200 import synth
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    from quantise_model import quantise
    dark, flat, (K, d, P) = calibration(H, W)
    e = engine.get_engine(H, W)
    e.set_dark(dark)
    e.set_flat(flat)
    e.set_lens(K, d, P)
    raw = frames(H, W, n, engine.pinned_empty)
    out = {np.float32: engine.pinned_empty((n, H, W), np.float32), np.uint16: engine.pinned_empty((n, H, W), np.uint16)}
    mpx = n * H * W / 1e6
    res = {'shape': [H, W], 'frames': n}

    # host frames, one GPU
    host = {np.float32: [], np.uint16: []}
    for dt in out:                                      # warm-up: ring allocation, module load
        e.correct_host(raw[:4], out=out[dt][:4])
    for _ in range(reps):
        for dt in (np.float32, np.uint16):
            t0 = time.perf_counter()
            e.correct_host(raw, out=out[dt])
            host[dt].append(time.perf_counter() - t0)
    assert np.array_equal(out[np.uint16], quantise(out[np.float32], np.uint16)), 'U16 != quantise(F32), host'
    for dt, name in ((np.float32, 'f32'), (np.uint16, 'u16')):
        t = med(host[dt])
        res['host_' + name] = {'ms_per_frame': 1e3 * t / n, 'mpx_s': mpx / t,
                               'pcie_gb_s': n * H * W * (2 + np.dtype(dt).itemsize) / t / 1e9,
                               'spread_ms_per_frame': [1e3 * min(host[dt]) / n, 1e3 * max(host[dt]) / n]}
    res['host_speedup_u16'] = med(host[np.float32]) / med(host[np.uint16])

    # device-resident frames, CUDA events
    dev = torch.from_numpy(np.asarray(raw)).cuda()
    dout = {np.float32: torch.empty((n, H, W), dtype=torch.float32, device='cuda'),
            np.uint16: torch.empty((n, H, W), dtype=torch.uint16, device='cuda')}
    for dt in dout:
        e.correct_batch(dev, out=dout[dt])
    ev = {dt: [] for dt in dout}
    for _ in range(reps):
        for dt in (np.float32, np.uint16):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            e.correct_batch(dev, out=dout[dt])
            b.record()
            b.synchronize()
            ev[dt].append(a.elapsed_time(b) / 1e3)
    assert np.array_equal(dout[np.uint16].cpu().numpy(), quantise(dout[np.float32].cpu().numpy(), np.uint16)), \
        'U16 != quantise(F32), device'
    for dt, name in ((np.float32, 'f32'), (np.uint16, 'u16')):
        t = med(ev[dt])
        res['device_' + name] = {'ms_per_frame': 1e3 * t / n, 'mpx_s': mpx / t}
    del dev, dout

    if n_dev:
        cal = CameraCalibration()
        cal.addDarkCurrent(dark)
        cal.addFlatField(flat)
        lens = LensDistortion({})
        lens.setCameraParams(*synth.lens_moderate(H, W))
        lens._coeffs['shape'] = (H, W)
        cal.addLens(lens)
        devices = list(range(n_dev))
        sh = {np.float32: [], np.uint16: []}
        with contextlib.redirect_stdout(io.StringIO()):
            for dt in out:
                cal.correct_batch(raw, out=out[dt], devices=devices)
            for _ in range(reps):
                for dt in (np.float32, np.uint16):
                    t0 = time.perf_counter()
                    cal.correct_batch(raw, out=out[dt], devices=devices)
                    sh[dt].append(time.perf_counter() - t0)
        assert np.array_equal(out[np.uint16], quantise(out[np.float32], np.uint16)), 'U16 != quantise(F32), sharded'
        for dt, name in ((np.float32, 'f32'), (np.uint16, 'u16')):
            t = med(sh[dt])
            res['sharded_%d_%s' % (n_dev, name)] = {'ms_per_frame': 1e3 * t / n, 'mpx_s': mpx / t,
                                                     'pcie_gb_s': n * H * W * (2 + np.dtype(dt).itemsize) / t / 1e9}
        res['sharded_speedup_u16'] = med(sh[np.float32]) / med(sh[np.uint16])
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--frames', type=int, default=64)
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--devices', type=int, default=0, help='also time the host path sharded over this many GPUs')
    ap.add_argument('--shapes', default='3000x4096,4000x6000', help='HxW,...')
    ap.add_argument('--out', help='also write the JSON object to this file')
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('tools/int_output.py needs a CUDA device')
    info = gpu_info()
    for line in info:
        print('gpu: %s' % line, flush=True)
    n_dev = min(a.devices, torch.cuda.device_count()) if a.devices else 0
    result = {'gpu': info, 'devices_sharded': n_dev, 'shapes': []}
    for s in a.shapes.split(','):
        H, W = (int(v) for v in s.split('x'))
        r = run_shape(H, W, a.frames, a.reps, n_dev if n_dev > 1 else 0)
        print(json.dumps(r), flush=True)
        result['shapes'].append(r)
    if a.out:
        with open(a.out, 'w') as f:
            json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == '__main__':
    main()
