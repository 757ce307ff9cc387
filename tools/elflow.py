"""Per-frame time of the EL workflow's correction and rectification on one GPU: dark, flat, 3x3 median-threshold, lens
and perspective, for a batch of uint16 frames.

    python tools/elflow.py [--frames 64] [--reps 3] [--device 0]

64 uint16 4096x3000 frames by default (1.5 GB, larger than L2), the moderate lens, full-frame output, and a mild
homography onto a 4000x2900 destination, float32 output.  Four ways to the same result, every one warmed up first:
  a  device frames, the chain with its perspective stage:  cal.correct_batch(frames_dev, perspective=pc)
  b  device frames, two steps:  cal.correct_batch(frames_dev), then Engine.warp_perspective of the whole batch
  c  pinned host frames, the chain with its perspective stage:  cal.correct_batch(frames_host, perspective=pc)
  d  pinned host frames, two steps:  cal.correct_batch(frames_host), then pc.correct(frame) for every frame
Prints one JSON line: the GPU's name and power limit, and per path the median over --reps of the call's wall time divided
by the frame count (each call ends in a device synchronise or returns host arrays).  Asserts a == b and c == d bit for
bit."""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402


def gpu_info(device):
    q = subprocess.run(['nvidia-smi', '-i', str(device), '--query-gpu=name,power.limit', '--format=csv,noheader'],
                       capture_output=True, text=True)
    name, power = (v.strip() for v in q.stdout.strip().split(',', 1))
    return name, power


def homography(src, dst):
    A, b = [], []
    for (x, y), (u, v) in zip(src, dst):
        A.append([x, y, 1, 0, 0, 0, -u * x, -u * y])
        A.append([0, 0, 0, x, y, 1, -v * x, -v * y])
        b += [u, v]
    return np.append(np.linalg.solve(np.array(A, float), np.array(b, float)), 1.0).reshape(3, 3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--frames', type=int, default=64)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--device', type=int, default=0)
    args = ap.parse_args()
    import torch
    from imgprocessor_b200 import engine, synth
    from imgprocessor_b200.camera import CameraCalibration, LensDistortion, PerspectiveCorrection
    if not torch.cuda.is_available():
        raise SystemExit('elflow.py measures on a CUDA device; none found')
    torch.cuda.set_device(args.device)
    dev = torch.device('cuda', args.device)
    H, W, n = 3000, 4096, args.frames
    dh, dw = 2900, 4000
    cal = CameraCalibration()
    cal.addDarkCurrent(synth.dark_map(H, W))
    cal.addFlatField(synth.flat_map(H, W))
    lens = LensDistortion({})
    lens.setCameraParams(*synth.lens_moderate(H, W))
    lens._coeffs['shape'] = (H, W)
    cal.addLens(lens)
    quad = [(0.02 * W, 0.015 * H), (0.985 * W, 0.03 * H), (0.97 * W, 0.98 * H), (0.01 * W, 0.96 * H)]
    M = homography(quad, [(0, 0), (dw, 0), (dw, dh), (0, dh)])
    pc = PerspectiveCorrection((H, W), new_size=(dh, dw))
    pc.setReference(M)

    frames_dev = synth.scene_torch(n, H, W, 11, dev)
    frames_host = engine.pinned_empty((n, H, W), np.uint16)
    frames_host[...] = frames_dev.cpu().numpy()
    out_c = np.empty((n, dh, dw), np.float32)
    mid_d = np.empty((n, H, W), np.float32)
    out_c[...] = 0
    mid_d[...] = 0

    def path_a():
        r = cal.correct_batch(frames_dev, perspective=pc)
        torch.cuda.synchronize()
        return r

    def path_b():
        mid = cal.correct_batch(frames_dev)
        r = engine.get_engine(H, W, args.device).warp_perspective(mid, M, (dw, dh))
        torch.cuda.synchronize()
        return r

    def path_c():
        return cal.correct_batch(frames_host, perspective=pc, out=out_c)

    def path_d():
        mid = cal.correct_batch(frames_host, out=mid_d)
        with contextlib.redirect_stdout(io.StringIO()):
            return [pc.correct(mid[i]) for i in range(n)]

    paths = {'a_device_chain_with_stage': path_a, 'b_device_two_steps': path_b, 'c_host_chain_with_stage': path_c,
             'd_host_two_steps': path_d}
    result, per_frame_ms = {}, {}
    for name, fn in paths.items():
        result[name] = fn()                                # warm-up; its output is the one compared below
        times = []
        for _ in range(args.reps):
            t0 = time.perf_counter()
            fn()
            times.append(time.perf_counter() - t0)
        per_frame_ms[name] = round(1e3 * float(np.median(times)) / n, 3)
    a, b = result['a_device_chain_with_stage'], result['b_device_two_steps']
    assert a.shape == b.shape == (n, dh, dw) and torch.equal(a, b), 'a != b'
    c, d = result['c_host_chain_with_stage'], np.stack(result['d_host_two_steps'])
    assert c.shape == d.shape == (n, dh, dw) and np.array_equal(c, d, equal_nan=True), 'c != d'
    name, power = gpu_info(args.device)
    print(json.dumps({'gpu': name, 'power_limit': power, 'frames': n, 'frame': [H, W], 'dst': [dh, dw], 'raw_dtype': 'uint16',
                      'out_dtype': 'float32', 'reps': args.reps, 'per_frame_ms': per_frame_ms,
                      'a_equals_b': True, 'c_equals_d': True}))


if __name__ == '__main__':
    main()
