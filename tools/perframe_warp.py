"""Per-frame time of the batch chain's perspective stage when every frame has its own homography (the EL workflow: the
module sits at a slightly different place in each image, and pc_i.setReference(quad_i) is called per frame).

    python tools/perframe_warp.py [--frames 64] [--reps 3] [--device 0]

64 uint16 4096x3000 frames by default (1.5 GB, larger than L2), the moderate lens, full-frame output, float32 output.
Frame i's homography maps a mild quad, jittered by a few pixels and a fraction of a degree per frame, onto a 4000x2900
destination.  Every path is warmed up first:
  a   device frames, the per-frame stage:  cal.correct_batch(frames_dev, perspective=[pc_0, ..., pc_n-1])
  b   device frames, the stage with one shared matrix (pc_0 for every frame): the cost of per-frame coordinates is a - b
  c   device frames, two steps:  cal.correct_batch(frames_dev), then Engine.warp_perspective of each frame with its matrix
  d   pinned host frames, the per-frame stage:  cal.correct_batch(frames_host, perspective=[pc_0, ..., pc_n-1])
  e   pinned host frames, two steps:  cal.correct_batch(frames_host), then pc_i.correct(frame_i) for every frame
Prints one JSON line: the GPU's name and power limit, and per path the median over --reps of the call's wall time divided
by the frame count (each call ends in a device synchronise or returns host arrays).  Asserts a == c and d == e bit for
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


def jittered_quads(H, W, n, seed=5):
    """the mild quad of tools/elflow.py, each frame's copy shifted by up to 4 pixels and rotated by up to 0.5 degree"""
    base = np.array([(0.02 * W, 0.015 * H), (0.985 * W, 0.03 * H), (0.97 * W, 0.98 * H), (0.01 * W, 0.96 * H)])
    rng = np.random.default_rng(seed)
    centre = base.mean(axis=0)
    out = []
    for _ in range(n):
        a = np.deg2rad(rng.uniform(-0.5, 0.5))
        R = np.array([[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]])
        out.append((base - centre) @ R.T + centre + rng.uniform(-4.0, 4.0, size=2))
    return out


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
        raise SystemExit('perframe_warp.py measures on a CUDA device; none found')
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
    Ms = [homography(q, [(0, 0), (dw, 0), (dw, dh), (0, dh)]) for q in jittered_quads(H, W, n)]
    pcs = []
    for M in Ms:
        pc = PerspectiveCorrection((H, W), new_size=(dh, dw))
        pc.setReference(M)
        pcs.append(pc)
    eng = engine.get_engine(H, W, args.device)

    frames_dev = synth.scene_torch(n, H, W, 11, dev)
    frames_host = engine.pinned_empty((n, H, W), np.uint16)
    frames_host[...] = frames_dev.cpu().numpy()
    out_d = np.empty((n, dh, dw), np.float32)
    mid_e = np.empty((n, H, W), np.float32)
    out_d[...] = 0
    mid_e[...] = 0

    def path_a():
        r = cal.correct_batch(frames_dev, perspective=pcs)
        torch.cuda.synchronize()
        return r

    def path_b():
        r = cal.correct_batch(frames_dev, perspective=pcs[0])
        torch.cuda.synchronize()
        return r

    def path_c():
        mid = cal.correct_batch(frames_dev)
        r = torch.stack([eng.warp_perspective(mid[i], Ms[i], (dw, dh)) for i in range(n)])
        torch.cuda.synchronize()
        return r

    def path_d():
        return cal.correct_batch(frames_host, perspective=pcs, out=out_d)

    def path_e():
        mid = cal.correct_batch(frames_host, out=mid_e)
        with contextlib.redirect_stdout(io.StringIO()):
            return [pcs[i].correct(mid[i]) for i in range(n)]

    paths = {'a_device_per_frame_stage': path_a, 'b_device_shared_matrix_stage': path_b, 'c_device_two_steps': path_c, 'd_host_per_frame_stage': path_d,
             'e_host_two_steps': path_e}
    per_frame_ms, checks = {}, {}
    for name, fn in paths.items():
        first = fn()                                       # warm-up; its output is the one compared below
        times = []
        for _ in range(args.reps):
            t0 = time.perf_counter()
            fn()
            times.append(time.perf_counter() - t0)
        per_frame_ms[name] = round(1e3 * float(np.median(times)) / n, 3)
        if name == 'a_device_per_frame_stage':
            a = first.clone()
        elif name == 'c_device_two_steps':
            checks['a_equals_c'] = bool(first.shape == (n, dh, dw) and torch.equal(a, first))
        elif name == 'd_host_per_frame_stage':
            d = first.copy()
        elif name == 'e_host_two_steps':
            checks['d_equals_e'] = bool(np.array_equal(d, np.stack(first), equal_nan=True))
        del first
    name, power = gpu_info(args.device)
    print(json.dumps({'gpu': name, 'power_limit': power, 'frames': n, 'frame': [H, W], 'dst': [dh, dw], 'raw_dtype': 'uint16',
                      'out_dtype': 'float32', 'reps': args.reps, 'per_frame_ms': per_frame_ms, **checks}))
    assert all(checks.values()), checks


if __name__ == '__main__':
    main()
