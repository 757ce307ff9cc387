"""Per-frame time of the batch chain when every frame brings its own background image (the EL workflow: each image is taken
together with the same exposure at zero module current).

    python tools/bg_frames.py [--frames 64] [--reps 3] [--device 0]

64 uint16 4096x3000 frames and as many uint16 backgrounds by default (1.5 GB each, larger than L2), the moderate lens,
full-frame float32 output.  Every path is warmed up first:
  a  device frames, backgrounds in the chain:  cal.correct_batch(frames_dev, bg_frames=bgs_dev)
  b  device frames, two steps:  frames_dev.float() - bgs_dev.float() in torch, then the chain without a dark stage
  c  device frames, one shared dark map:  cal.correct_batch(frames_dev) (what per-frame backgrounds cost is a - c)
  d  pinned host frames and backgrounds through imgcorr_correct_host_bg:  cal.correct_batch(frames_host, bg_frames=bgs_host)
  e  pinned host frames, what users did before:  cal.correct_batch(frames_host[i:i+1], bgImages=bgs_host[i]) per frame
and K1 alone (no lens: one K1 launch for the batch), event-timed, with the per-frame backgrounds and with the shared dark.
Prints one JSON line: the GPU's name and power limit, and per path the median over --reps of the call's wall time (or
event time for K1) divided by the frame count.  Asserts a == b and d == e bit for bit."""
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--frames', type=int, default=64)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--device', type=int, default=0)
    args = ap.parse_args()
    import torch
    from imgprocessor_b200 import _lib, engine, synth
    from imgprocessor_b200.camera import CameraCalibration, LensDistortion
    if not torch.cuda.is_available():
        raise SystemExit('bg_frames.py measures on a CUDA device; none found')
    torch.cuda.set_device(args.device)
    dev = torch.device('cuda', args.device)
    H, W, n = 3000, 4096, args.frames
    cal = CameraCalibration()
    cal.addDarkCurrent(synth.dark_map(H, W))
    cal.addFlatField(synth.flat_map(H, W))
    lens = LensDistortion({})
    lens.setCameraParams(*synth.lens_moderate(H, W))
    lens._coeffs['shape'] = (H, W)
    cal.addLens(lens)
    eng = engine.get_engine(H, W, args.device)

    frames_dev = synth.scene_torch(n, H, W, 11, dev)
    bgs_dev = synth.scene_torch(n, H, W, 12, dev)
    frames_host = engine.pinned_empty((n, H, W), np.uint16)
    frames_host[...] = frames_dev.cpu().numpy()
    bgs_host = engine.pinned_empty((n, H, W), np.uint16)
    bgs_host[...] = bgs_dev.cpu().numpy()
    out_d = engine.pinned_empty((n, H, W), np.float32)
    out_e = engine.pinned_empty((n, H, W), np.float32)
    out_d[...] = 0
    out_e[...] = 0
    chain = _lib.DO_DARK | _lib.DO_FLAT | _lib.DO_NAN_TO_NUM

    def sync(r):
        torch.cuda.synchronize()
        return r

    def path_a():
        return sync(cal.correct_batch(frames_dev, bg_frames=bgs_dev))

    def path_b():
        return sync(eng.correct_batch(frames_dev.float() - bgs_dev.float(), flags=_lib.DO_FLAT | _lib.DO_NAN_TO_NUM))

    def path_c():
        return sync(cal.correct_batch(frames_dev))

    def path_d():
        return cal.correct_batch(frames_host, bg_frames=bgs_host, out=out_d)

    def path_e():
        with contextlib.redirect_stdout(io.StringIO()):
            for i in range(n):
                cal.correct_batch(frames_host[i:i + 1], bgImages=bgs_host[i], out=out_e[i:i + 1])
        return out_e

    paths = {'a_device_bg_in_chain': path_a, 'b_device_two_steps': path_b, 'c_device_shared_dark': path_c,
             'd_host_bg_in_chain': path_d, 'e_host_per_frame_calls': path_e}
    per_frame_ms, checks = {}, {}
    for name, fn in paths.items():
        first = fn()                                       # warm-up; its output is the one compared below
        first = first.clone() if isinstance(first, torch.Tensor) else first.copy()
        times = []
        for _ in range(args.reps):
            t0 = time.perf_counter()
            fn()
            times.append(time.perf_counter() - t0)
        per_frame_ms[name] = round(1e3 * float(np.median(times)) / n, 3)
        if name == 'a_device_bg_in_chain':
            a = first
        elif name == 'b_device_two_steps':
            checks['a_equals_b'] = bool(torch.equal(a, first))
        elif name == 'd_host_bg_in_chain':
            d = first
        elif name == 'e_host_per_frame_calls':
            checks['d_equals_e'] = bool(np.array_equal(d, first, equal_nan=True))
        del first
    del a

    # K1 alone (no lens): one launch for the batch, event-timed
    cal.correct_batch(frames_dev[:1])                      # the calibrated dark map back on the engine
    k1_us = {}
    for name, kw in (('k1_bg_frames', dict(bg=bgs_dev)), ('k1_shared_dark', {})):
        out = torch.empty((n, H, W), dtype=torch.float32, device=dev)
        eng.correct_batch(frames_dev, flags=chain, use_lens=False, out=out, **kw)
        times = []
        for _ in range(max(args.reps, 5)):
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            ev[0].record()
            eng.correct_batch(frames_dev, flags=chain, use_lens=False, out=out, **kw)
            ev[1].record()
            torch.cuda.synchronize()
            times.append(ev[0].elapsed_time(ev[1]))
        k1_us[name] = round(1e3 * float(np.median(times)) / n, 2)
        del out
    name, power = gpu_info(args.device)
    print(json.dumps({'gpu': name, 'power_limit': power, 'frames': n, 'frame': [H, W], 'raw_dtype': 'uint16',
                      'bg_dtype': 'uint16', 'out_dtype': 'float32', 'reps': args.reps, 'per_frame_ms': per_frame_ms,
                      'k1_per_frame_us': k1_us, **checks}))
    assert all(checks.values()), checks


if __name__ == '__main__':
    main()
