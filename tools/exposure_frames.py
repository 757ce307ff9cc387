"""Per-frame time of the batch chain when the frames of one batch were taken at different exposure times and the dark
current is the line model bg = offset + ascent * t (a tuple dark-current entry).

    python tools/exposure_frames.py [--frames 64] [--reps 3] [--device 0]

64 uint16 4096x3000 frames by default (1.5 GB, larger than L2) with four exposure times, the moderate lens, full-frame
float32 output.  Every path is warmed up first:
  a  device frames, one time per frame:  cal.correct_batch(frames_dev, exposure_time=ts)
  b  device frames, one scalar time:  cal.correct_batch(frames_dev, exposure_time=t0)
  c  as b with K1 forced to the generic tiles (IMGCORR_OPT_K1_VARIANT = 1)
  d  device frames, one scalar call per exposure-time group (what users did before):  the frames of each time gathered,
     corrected with that time, scattered back
  e  pinned host frames, one time per frame:  cal.correct_batch(frames_host, exposure_time=ts)
and K1 alone (no lens: one K1 launch for the batch), event-timed, with the line model and per-frame times, with the line
model and one time (each on the streaming kernel and on the generic tiles), and with a plain dark map.  Prints one JSON
line: the GPU's name and power limit, and per path the median over --reps of the call's wall time (or event time for K1)
divided by the frame count.  Asserts a == d bit for bit
and that the host path e equals a."""
import argparse
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
        raise SystemExit('exposure_frames.py measures on a CUDA device; none found')
    torch.cuda.set_device(args.device)
    dev = torch.device('cuda', args.device)
    H, W, n = 3000, 4096, args.frames
    offs = synth.dark_map(H, W)
    asc = (np.random.default_rng(5).random((H, W)) * 2.0).astype(np.float32)
    cal = CameraCalibration()
    cal.coeffs['dark current'].append((time.localtime(), '', (offs, asc), None))
    cal.coeffs['shape'] = (H, W)
    cal.addFlatField(synth.flat_map(H, W))
    lens = LensDistortion({})
    lens.setCameraParams(*synth.lens_moderate(H, W))
    lens._coeffs['shape'] = (H, W)
    cal.addLens(lens)
    eng = engine.get_engine(H, W, args.device)
    ts = np.resize([0.3, 1.2, 4.8, 19.2], n)
    groups = [(float(t), torch.from_numpy(np.flatnonzero(ts == t)).to(dev)) for t in np.unique(ts)]

    frames_dev = synth.scene_torch(n, H, W, 11, dev)
    frames_host = engine.pinned_empty((n, H, W), np.uint16)
    frames_host[...] = frames_dev.cpu().numpy()
    out_e = engine.pinned_empty((n, H, W), np.float32)
    out_e[...] = 0
    chain = _lib.DO_DARK | _lib.DO_FLAT | _lib.DO_NAN_TO_NUM

    def sync(r):
        torch.cuda.synchronize()
        return r

    def path_a():
        return sync(cal.correct_batch(frames_dev, exposure_time=ts))

    def path_b():
        return sync(cal.correct_batch(frames_dev, exposure_time=float(ts[0])))

    def path_c():
        eng.set_option(_lib.OPT_K1_VARIANT, 1)
        try:
            return sync(cal.correct_batch(frames_dev, exposure_time=float(ts[0])))
        finally:
            eng.set_option(_lib.OPT_K1_VARIANT, 0)

    def path_d():
        out = torch.empty((n, H, W), dtype=torch.float32, device=dev)
        for t, idx in groups:
            out.index_copy_(0, idx, cal.correct_batch(frames_dev.index_select(0, idx), exposure_time=t))
        return sync(out)

    def path_e():
        return cal.correct_batch(frames_host, exposure_time=ts, out=out_e)

    paths = {'a_device_per_frame_times': path_a, 'b_device_scalar_time': path_b,
             'c_device_scalar_time_generic_tiles': path_c, 'd_device_scalar_call_per_group': path_d,
             'e_host_per_frame_times': path_e}
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
        if name == 'a_device_per_frame_times':
            a = first
        elif name == 'b_device_scalar_time':
            checks['b_equals_c'] = None
            b = first
        elif name == 'c_device_scalar_time_generic_tiles':
            checks['b_equals_c'] = bool(torch.equal(b, first))
            del b
        elif name == 'd_device_scalar_call_per_group':
            checks['a_equals_d'] = bool(torch.equal(a, first))
        elif name == 'e_host_per_frame_times':
            checks['e_equals_a'] = bool(np.array_equal(a.cpu().numpy(), first, equal_nan=True))
        del first
    del a

    # K1 alone (no lens): one launch for the batch, event-timed
    k1_us = {}
    for name in ('k1_line_per_frame_times', 'k1_line_per_frame_times_generic_tiles', 'k1_line_scalar_time',
                 'k1_line_scalar_time_generic_tiles', 'k1_plain_dark'):
        if name == 'k1_plain_dark':
            eng.set_dark(offs)
        else:
            eng.set_dark(offs, asc, float(ts[0]), 16)
            if name.startswith('k1_line_per_frame_times'):
                eng.set_dark_exposures(ts)
        eng.set_option(_lib.OPT_K1_VARIANT, 1 if name.endswith('generic_tiles') else 0)
        out = torch.empty((n, H, W), dtype=torch.float32, device=dev)
        eng.correct_batch(frames_dev, flags=chain, use_lens=False, out=out)
        times = []
        for _ in range(max(args.reps, 5)):
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            ev[0].record()
            eng.correct_batch(frames_dev, flags=chain, use_lens=False, out=out)
            ev[1].record()
            torch.cuda.synchronize()
            times.append(ev[0].elapsed_time(ev[1]))
        k1_us[name] = round(1e3 * float(np.median(times)) / n, 2)
        del out
    eng.set_option(_lib.OPT_K1_VARIANT, 0)
    eng.set_dark(None)
    name, power = gpu_info(args.device)
    print(json.dumps({'gpu': name, 'power_limit': power, 'frames': n, 'frame': [H, W], 'raw_dtype': 'uint16',
                      'out_dtype': 'float32', 'exposure_times': sorted(set(float(t) for t in ts)), 'reps': args.reps,
                      'per_frame_ms': per_frame_ms, 'k1_per_frame_us': k1_us, **checks}))
    assert all(checks.values()), checks


if __name__ == '__main__':
    main()
