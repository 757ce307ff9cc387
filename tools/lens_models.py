"""Cost of OpenCV's extended lens models in K2: the 5-term lens against an 8-term (rational) and a 14-term (rational,
thin prism, tilted sensor) lens, in the same run.  The 8- and 14-term lenses are stronger (159 and 166 px largest shift
against 87) and need K2's 96x32 staged boxes where the 5-term lens fits 80x28 ones; '8-term, same map' is the 5-term lens
with k4 = 1e-12: the same boxes and (to the pixel) the same map, evaluated by the extended kernels.  It isolates the cost
of the model's arithmetic from the cost of a stronger lens.

    python tools/lens_models.py [--reps 7] [--device 0]

4096x3000 float32 frames, K = [[4096, 0, 2048], [0, 4096, 1500], [0, 0, 1]], P from cv2.getOptimalNewCameraMatrix.
Per lens, lenses alternating within every rep, CUDA-event times:
  batch16 / batch32   K2 alone (Engine.undistort) on launches of 16 and 32 frames, per frame
  single_nocache      one frame with the coordinate cache off: evaluates the map on every call
  first               one frame, the first call for the lens: evaluates the map and writes the coordinate cache; includes
                      allocating the cache (the staged-box geometry is chosen beforehand by an untimed call)
  repeat              one frame, a repeated call: reads the cache
  chain_mpxs          the device-resident chain (CameraCalibration.correct_batch, 32 uint16 frames, dark + flat + 3x3
                      median + lens, float32 output) in Mpx/s
Prints one JSON line with the GPU's name and power limit, read in the same call, and per lens the median over --reps."""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402

_R8 = [-0.25, 0.06, 1e-3, -1e-3, -0.01, 0.05, 0.01, -0.004]
LENSES = {
    '5-term': [-0.2, 0.05, 1e-3, -1e-3, 0.0],
    '8-term, same map': [-0.2, 0.05, 1e-3, -1e-3, 0.0, 1e-12, 0.0, 0.0],
    '8-term': _R8,
    '14-term': _R8 + [1e-3, -2e-4, 5e-4, 1e-4, 0.01, -0.008],
}


def gpu_info(device):
    q = subprocess.run(['nvidia-smi', '-i', str(device), '--query-gpu=name,power.limit', '--format=csv,noheader'],
                       capture_output=True, text=True)
    name, power = (v.strip() for v in q.stdout.strip().split(',', 1))
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=7)
    ap.add_argument('--device', type=int, default=0)
    args = ap.parse_args()
    import cv2
    import torch
    from imgprocessor_b200 import _lib, engine, synth
    from imgprocessor_b200.camera import CameraCalibration, LensDistortion
    if not torch.cuda.is_available():
        raise SystemExit('lens_models.py measures on a CUDA device; none found')
    torch.cuda.set_device(args.device)
    dev = torch.device('cuda', args.device)
    H, W, nb = 3000, 4096, 32
    K = np.array([[W, 0, W / 2.0], [0, W, H / 2.0], [0, 0, 1.0]])
    lenses = {}
    for name, d in LENSES.items():
        d = np.asarray(d, np.float64)[None, :]
        P, _ = cv2.getOptimalNewCameraMatrix(K, d, (W, H), 1, (W, H))
        lenses[name] = (d, P)
    e = engine.get_engine(H, W, args.device)
    src = torch.rand((nb, H, W), device=dev, dtype=torch.float32) * 4000     # 1.5 GB: larger than L2
    out = torch.empty_like(src)
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn):
        start.record()
        fn()
        stop.record()
        stop.synchronize()
        return start.elapsed_time(stop)

    raw = synth.scene_torch(nb, H, W, 3, dev)
    cals = {}
    for name, (d, _) in lenses.items():
        cal = CameraCalibration()
        cal.addDarkCurrent(synth.dark_map(H, W))
        cal.addFlatField(synth.flat_map(H, W))
        lens = LensDistortion({'cameraMatrix': K, 'distortionCoeffs': d, 'shape': (H, W)})
        cal.addLens(lens)
        cals[name] = cal
    res = {name: {k: [] for k in ('batch16', 'batch32', 'single_nocache', 'first', 'repeat', 'chain_mpxs')} for name in lenses}
    quiet = lambda: contextlib.redirect_stdout(io.StringIO())
    for rep in range(args.reps + 1):                       # rep 0 warms up every shape and kernel
        for name, (d, P) in lenses.items():
            r = res[name]
            e.set_lens(K, d, P)
            e.undistort(src[:32], out=out[:32])            # chooses the geometry for the lens (host), untimed
            for n in (16, 32):
                t = timed(lambda: e.undistort(src[:n], out=out[:n]))
                if rep:
                    r['batch%d' % n].append(t / n)
            e.set_lens(None, None, None)
            e.set_lens(K, d, P)                            # a fresh lens: no geometry, no coordinate cache
            e.set_option(_lib.OPT_K2_COORD_CACHE, 0)
            e.undistort(src[:1], out=out[:1])              # chooses the geometry (host), untimed
            nocache = timed(lambda: e.undistort(src[:1], out=out[:1]))
            e.set_option(_lib.OPT_K2_COORD_CACHE, 1)
            first = timed(lambda: e.undistort(src[:1], out=out[:1]))
            again = timed(lambda: e.undistort(src[:1], out=out[:1]))
            with quiet():
                cals[name].correct_batch(raw[:1], threshold=0.1)       # sets the calibration's lens
                t = timed(lambda: cals[name].correct_batch(raw, threshold=0.1))
            if rep:
                r['single_nocache'].append(nocache)
                r['first'].append(first)
                r['repeat'].append(again)
                r['chain_mpxs'].append(nb * H * W / (t * 1e-3) / 1e6)
    gpu, power = gpu_info(args.device)
    summary = {name: {k: round(float(np.median(v)), 4 if k != 'chain_mpxs' else 0) for k, v in r.items()}
               for name, r in res.items()}
    print(json.dumps({'gpu': gpu, 'power_limit': power, 'frame': [H, W], 'reps': args.reps,
                      'units': {'batch16': 'ms/frame', 'batch32': 'ms/frame', 'single_nocache': 'ms', 'first': 'ms', 'repeat': 'ms',
                                'chain_mpxs': 'Mpx/s'}, 'lenses': summary}))


if __name__ == '__main__':
    main()
