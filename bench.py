#!/usr/bin/env python
"""bench.py — corrected Mpx/s of the CameraCalibration.correct() chain on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--frames F] [--impl reference] [--dump-outputs DIR]

Headline workload (BASELINE.json configs[2]): a batch of 4096x3000 uint16 frames per GPU through the full chain
(dark subtract, flat-field divide, nan_to_num, 3x3 median-threshold, lens undistortion).  One step = one pass
over the whole batch.  Frames are sharded over ranks (weak scaling: F frames on every GPU), calibration maps
are built on rank 0 and broadcast once; there is no collective in the timed region.

One JSON line on rank 0:
  value        device-resident whole-job Mpx/s (inputs in HBM, CUDA-event timed, max over ranks)
  e2e          the same metric through the C-ABI host-buffer call (pinned host frames, H2D + kernels + D2H
               overlapped inside libimgcorr), host wall clock, max over ranks; with the box's raw pinned-copy ceiling
               measured in the same run (all ranks copying at once) and the fraction of it the pipeline reaches
  roofline     the dominant kernel (K1): algorithmic bytes (14 B/px, SURVEY §8d) / event-timed launch duration
               inside the timed region, against the measured HBM copy peak (MEASURED_PEAKS.json)
  configs      the other BASELINE configs, measured the same way (CUDA events on the launching stream, inputs larger
               than L2 by rotating over frames): c0 1024x1024 float32 single frame, c1 single 4096x3000 uint16 K1 only,
               c3 8192x8192 float32 5x5 + strong lens, c4 6000x4000 uint16 streamed from a 16-buffer pinned pool, and the
               strong-scaling point (256 frames in total over the N GPUs)
  parity_check "ok" when, on EVERY rank, row bands of the first and last frame of each measured output equal the
               float32 oracle chain (oracle/bands.py, cv2's own maps) bit for bit; anything else makes the run fail
  cpu_baseline the oracle's restatement of the reference path (scipy + OpenCV, float64) on one host core
`--impl reference` times that reference path on all host cores instead (rank 0 only), after re-checking it against the
golden outputs of the unmodified reference (tests/golden).

`--dump-outputs DIR` writes, after the timed steps, what the headline correct_batch() call returned in its last step on
rank 0, as float32 .npy files (see dump_outputs).  The inputs are seeded, so two builds run with the same arguments can
be compared file for file.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H, W = 3000, 4096
METRIC = 'corrected Mpx/s, CameraCalibration.correct() chain'
K1_BYTES_PER_PX = 14.0      # raw u16 2 + dark 4 + flat 4 + out 4   (SURVEY.md §8d)
K2_BYTES_PER_PX = 8.0       # src 4 + dst 4
FALLBACK_HBM_GBS = 6650.0   # /opt/skills/guides/B200_PROFILING.md


def workload_config(frames, n_gpus):
    return {
        'workload': 'BASELINE configs[2]: batch of %d 4096x3000 uint16 frames per GPU, full correct() chain '
                    '(dark + flat + nan_to_num + 3x3 medianThreshold + LensDistortion remap), moderate 5-coeff lens' % frames,
        'frame_shape': [H, W], 'frames_per_gpu': frames, 'global_frames': frames * n_gpus,
        'threshold': 0.1, 'keep_size': True, 'out_dtype': 'float32',
        'l2': 'inputs (%.1f GB of raw frames per GPU) are far larger than the 126 MB L2; no flush needed' % (frames * H * W * 2 / 1e9),
        'sharding': 'frames split contiguously over ranks, calibration broadcast once, no steady-state collective',
    }


def measured_peak():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            return float(json.load(f)['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    except Exception:
        return FALLBACK_HBM_GBS, 'fallback (B200_PROFILING.md)'


class ClockSampler(object):
    """SM clock + throttle reasons of one GPU, sampled while the timed region runs."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {}
        for n in dir(nv):
            if n.startswith('nvmlClocksThrottleReason') or n.startswith('nvmlClocksEventReason'):
                v = getattr(nv, n)
                if isinstance(v, int) and v:
                    names[v] = n.replace('nvmlClocksThrottleReason', '').replace('nvmlClocksEventReason', '')
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    bits = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    bits = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for b, n in names.items():
                    if bits & b and n not in ('None', 'GpuIdle', 'All'):
                        self.reasons.add(n)
            except Exception:
                pass
            self._stop.wait(0.005)

    def __enter__(self):
        if self.nv is not None:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thread is not None:
            self._thread.join()

    def summary(self):
        if not self.samples:
            return {'sm_mhz': None, 'sm_max_mhz': self.max_mhz, 'reasons': ['unavailable']}
        s = sorted(self.samples)
        return {'sm_mhz': s[len(s) // 2], 'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons), 'samples': len(s)}


# ------------------------------------------------------------------------------------------------ reference arm
def _ref_inputs(seed):
    import numpy as np
    from imgprocessor_b200 import synth
    raw = synth.scene(H, W, seed, np.uint16)
    dark, flat = synth.dark_map(H, W), synth.flat_map(H, W)
    p = synth.lens_moderate(H, W)
    return raw, dark, flat, (synth.camera_matrix(p), synth.dist_coeffs(p))


_REF_STATE = {}


def _ref_worker_init():
    import cv2
    cv2.setNumThreads(1)
    raw, dark, flat, lens = _ref_inputs(100 + os.getpid() % 7)
    _REF_STATE.update(raw=raw, dark=dark, flat=flat, lens=lens)


def _ref_worker_step(_):
    from oracle import refpath
    s = _REF_STATE
    out = refpath.correct(s['raw'], s['dark'], s['flat'], s['lens'], 0.1, True)
    return float(out[0, 0])


def golden_check():
    """the timed port (oracle.refpath) against outputs of the UNMODIFIED reference (tests/golden/*.npz, generated in the
    build container by tests/golden/make_golden.py): re-asserted on the box that does the timing.  Returns a description."""
    import numpy as np
    from oracle import refpath
    gdir = os.path.join(ROOT, 'tests', 'golden')
    n = 0
    for keep in (1, 0):
        g = np.load(os.path.join(gdir, 'correct_u16_keep%d.npz' % keep))
        out = refpath.correct(g['raw'], g['dark'], g['flat'], (g['K'], g['dist']), threshold=0.1, keep_size=bool(keep))
        if not np.array_equal(out, g['out']):
            raise SystemExit('bench.py: oracle.refpath.correct differs from the golden output of the reference (correct_u16_keep%d)' % keep)
        n += 1
    for name, kw in (('correct_f32_thr0', dict(threshold=0)),):
        g = np.load(os.path.join(gdir, name + '.npz'))
        out = refpath.correct(g['raw'], g['dark'], g['flat'], (g['K'], g['dist']), **kw)
        if not np.array_equal(out, g['out'], equal_nan=True):
            raise SystemExit('bench.py: oracle.refpath.correct differs from the golden output of the reference (%s)' % name)
        n += 1
    for tag in ('u16', 'f32'):
        for size in (3, 5):
            g = np.load(os.path.join(gdir, 'median_%s_s%d_gt.npz' % (tag, size)))
            o, ind = refpath.median_threshold(g['img'], 0.1, size, '>', copy=True)
            if not (np.array_equal(o, g['out']) and np.array_equal(ind, g['ind'])):
                raise SystemExit('bench.py: oracle.refpath.median_threshold differs from the golden output (%s, %d)' % (tag, size))
            n += 1
    return 'ok: oracle.refpath == %d golden outputs of the unmodified reference, re-checked on this box before timing' % n


def run_reference(args):
    """the reference's own CPU implementation of the path (oracle.refpath = its Python chain restated over the
    same scipy / OpenCV / numpy natives), one frame per worker per step, all host cores."""
    import multiprocessing as mp
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    ctx = mp.get_context('fork')
    # the workers are forked BEFORE this process touches OpenCV / scipy: forking a process whose OpenCV thread pool already
    # runs can deadlock the children.  The golden check then runs here, in the parent, before anything is timed.
    with ctx.Pool(cores, initializer=_ref_worker_init) as pool:
        golden = golden_check()
        for _ in range(max(args.warmup, 1)):
            pool.map(_ref_worker_step, range(cores))
        t0 = time.perf_counter()
        for _ in range(args.steps):
            pool.map(_ref_worker_step, range(cores))
        dt = time.perf_counter() - t0
    px = float(cores) * H * W * args.steps
    val = px / dt / 1e6
    import cv2
    import numpy
    import scipy
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': val, 'unit': 'Mpx/s', 'n_gpus': args.gpus, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': dt / args.steps * 1e3, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': workload_config(args.frames, args.gpus),
        'cpu_baseline': {'value': val, 'unit': 'Mpx/s', 'cores': cores, 'kind': 'port',
                         'sample': 'each step = one 4096x3000 uint16 frame per worker through the float64 reference chain '
                                   '(oracle.refpath: scipy %s median_filter, OpenCV %s remap, numpy %s), %d worker processes'
                                   % (scipy.__version__, cv2.__version__, numpy.__version__, cores),
                         'golden_check': golden},
        'e2e': {'value': val, 'unit': 'Mpx/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


def cpu_baseline_single(frames=3):
    """the oracle's reference-path restatement, one process, one thread, `frames` frames"""
    import cv2
    import numpy
    import scipy
    from oracle import refpath
    cv2.setNumThreads(1)
    raw, dark, flat, lens = _ref_inputs(100)
    refpath.correct(raw[:256, :256], dark[:256, :256], flat[:256, :256], None, 0.1)      # import / warm-up
    best = None
    for _ in range(frames):
        t0 = time.perf_counter()
        refpath.correct(raw, dark, flat, lens, 0.1, True)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return {'value': H * W / best / 1e6, 'unit': 'Mpx/s', 'cores': 1, 'kind': 'port',
            'sample': 'best of %d single 4096x3000 uint16 frames through oracle.refpath.correct (float64; scipy %s '
                      'median_filter single-threaded, OpenCV %s with 1 thread, numpy %s), %.2f s/frame'
                      % (frames, scipy.__version__, cv2.__version__, numpy.__version__, best)}


# ------------------------------------------------------------------------------------------------ our arm
class Parity(object):
    """in-run parity check: row bands of GPU outputs against the float32 oracle chain, collected per rank"""

    def __init__(self):
        self.failures, self.bands, self.pixels = [], 0, 0

    def check(self, tag, got_rows, want_rows):
        import numpy as np
        self.bands += 1
        self.pixels += int(want_rows.size)
        if got_rows.shape != want_rows.shape or not np.array_equal(got_rows, want_rows, equal_nan=True):
            bad = int((got_rows != want_rows).sum()) if got_rows.shape == want_rows.shape else -1
            self.failures.append('%s: %d pixels differ' % (tag, bad))

    def chain(self, tag, raw_host, out_dev_or_host, dark, flat, maps, ksize=3, threshold=0.1, nbands=48):
        """raw_host: the full input frame on the host; out: the chain's full output frame (device tensor or numpy)"""
        from oracle import bands
        h = raw_host.shape[0]
        for r0, r1 in bands.default_bands(h, nbands):
            want = bands.chain_band(raw_host, dark, flat, maps[0], maps[1], r0, r1, threshold, ksize)
            got = out_dev_or_host[r0:r1]
            got = got.cpu().numpy() if hasattr(got, 'cpu') else got
            self.check('%s rows %d:%d' % (tag, r0, r1), got, want)

    def k1(self, tag, raw_host, out_dev, dark, flat, ksize=3, threshold=0.1, nbands=48):
        from oracle import bands
        h = raw_host.shape[0]
        for r0, r1 in bands.default_bands(h, nbands):
            want = bands.k1_band(raw_host, dark, flat, r0, r1, threshold, ksize)
            self.check('%s rows %d:%d' % (tag, r0, r1), out_dev[r0:r1].cpu().numpy(), want)


def event_times_us(fn, iters, warm=3):
    """median / min duration in us of fn(i), each call bracketed by CUDA events on the current stream.  A ~20 ms spin
    kernel is queued first so that the calls pile up behind it: the events then time the GPU, not the Python call rate
    (a one-frame call costs ~50 us of host time, more than the kernels of a small frame)."""
    import torch
    for i in range(warm):
        fn(i)
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(iters + 1)]
    torch.cuda._sleep(40000000)
    ev[0].record()
    for i in range(iters):
        fn(i)
        ev[i + 1].record()
    torch.cuda.synchronize()
    ts = sorted(ev[i].elapsed_time(ev[i + 1]) * 1e3 for i in range(iters))
    return ts[len(ts) // 2], ts[0]


def pcie_probe(dev, in_bytes, out_bytes, seconds=0.25):
    """raw page-locked copies of the box, the ceiling of every host-buffer number: H2D alone, D2H alone and both at once
    (two streams, chunks of the e2e frame sizes, several in flight), GB/s each.  All ranks call this at the same time."""
    import torch
    h_in = torch.empty(in_bytes, dtype=torch.uint8, pin_memory=True)
    h_out = torch.empty(out_bytes, dtype=torch.uint8, pin_memory=True)
    d_in = torch.empty(in_bytes, dtype=torch.uint8, device=dev)
    d_out = torch.empty(out_bytes, dtype=torch.uint8, device=dev)
    s1, s2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)

    def run(do_in, do_out, reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            if do_in:
                with torch.cuda.stream(s1):
                    d_in.copy_(h_in, non_blocking=True)
            if do_out:
                with torch.cuda.stream(s2):
                    h_out.copy_(d_out, non_blocking=True)
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    res = {}
    for name, di, do in (('h2d', True, False), ('d2h', False, True), ('both', True, True)):
        run(di, do, 2)
        t = run(di, do, 4)
        reps = max(4, int(seconds / max(t / 4, 1e-6)))
        t = run(di, do, reps)
        res[name] = (reps * ((in_bytes if di else 0) + (out_bytes if do else 0)) / t / 1e9, t)
    return res


DUMP_SAMPLE = 1 << 21      # pixels in the seeded sample of the whole batch: 8 MB of float32


def dump_outputs(path, out):
    """write the (F, H, W) float32 result of the timed call as two .npy files, 57.5 MB in all at the 4096x3000 frame size:
    out_last_frame.npy, the whole last frame (every tile and strip seam of one frame), and out_sample.npy, the values at
    DUMP_SAMPLE flat positions of the batch drawn by a fixed-seed generator (every frame group).  The positions depend on
    the output's shape only."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    idx = np.sort(np.random.default_rng(20240607).integers(0, out.numel(), DUMP_SAMPLE))
    sample = out.reshape(-1)[torch.from_numpy(idx).to(out.device)]
    np.save(os.path.join(path, 'out_last_frame.npy'), out[-1].cpu().numpy())
    np.save(os.path.join(path, 'out_sample.npy'), sample.cpu().numpy())


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from imgprocessor_b200 import _lib, engine, sharding, synth
    import cv2

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise RuntimeError('bench.py needs a CUDA device; there is no CPU fallback (use --impl reference for the CPU arm)')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    distributed = world > 1
    if distributed:
        dist.init_process_group('nccl', device_id=dev)
    peak, peak_src = measured_peak()
    parity = Parity()

    def barrier():
        if distributed:
            dist.barrier(device_ids=[local])
        torch.cuda.synchronize()

    def rmax(v):
        return sharding.reduce_max(v, dev) if distributed else float(v)

    def rsum(v):
        return sharding.reduce_sum(v, dev) if distributed else float(v)

    def lens_setup(eng, h, w, params):
        Kmat, dvec = synth.camera_matrix(params), synth.dist_coeffs(params)
        P, _roi = cv2.getOptimalNewCameraMatrix(Kmat, dvec, (w, h), 1, (w, h))
        eng.set_lens(Kmat, dvec, P)
        return cv2.initUndistortRectifyMap(Kmat, dvec, None, P, (w, h), cv2.CV_32FC1)      # cv2's own maps: the oracle's

    F = args.frames
    eng = engine.Engine(H, W, local)

    # calibration: built on rank 0, broadcast once over NCCL, uploaded into the library's per-device copies
    if distributed:
        maps = {'dark': synth.dark_map(H, W), 'flat': synth.flat_map(H, W)} if rank == 0 else {'dark': None, 'flat': None}
        cal = sharding.broadcast_calibration(maps, src=0, device=dev)
        eng.set_dark(cal['dark'])
        eng.set_flat(cal['flat'])
        dark_h, flat_h = cal['dark'].cpu().numpy(), cal['flat'].cpu().numpy()
    else:
        dark_h, flat_h = synth.dark_map(H, W), synth.flat_map(H, W)
        eng.set_dark(dark_h)
        eng.set_flat(flat_h)
    cvmaps = lens_setup(eng, H, W, synth.lens_moderate(H, W))
    eng.set_option(_lib.OPT_CHAIN_GROUP, args.group)
    eng.set_option(_lib.OPT_CHAIN_OVERLAP, int(args.overlap))
    if args.host_slots:
        eng.set_option(_lib.OPT_HOST_SLOTS, args.host_slots)

    numa = {'bound': False} if os.environ.get('IMGCORR_NO_NUMA_BIND') else sharding.bind_host_to_gpu(local)
    raw = synth.scene_torch(F, H, W, 1000 + rank, dev, 'uint16')
    out = torch.empty((F, H, W), dtype=torch.float32, device=dev)
    px_step = float(F) * H * W

    def step():
        eng.correct_batch(raw, threshold=0.1, ksize=3, out=out)

    # ---- device-resident timing (headline) ---------------------------------------------------------
    for _ in range(args.warmup):
        step()
    eng.set_option(_lib.OPT_PROFILE, max(1, F // 32))      # event-bracket ~32 K1 / K2 launches per step
    eng.profile_read()
    launches0 = eng.launch_count
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clocks:
        ev0.record()
        for _ in range(args.steps):
            step()
        ev1.record()
        torch.cuda.synchronize()
    ms_total = ev0.elapsed_time(ev1)
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out)
    launches = eng.launch_count - launches0
    k1_ms, k1_frames, k2_ms, k2_frames = eng.profile_read()
    eng.set_option(_lib.OPT_PROFILE, 0)
    ms_total = rmax(ms_total)
    launches = rsum(launches)
    value = px_step * world * args.steps / (ms_total * 1e-3) / 1e6
    # parity of what was just timed: first and last frame of this rank's shard
    for fi in sorted({0, F - 1}):
        parity.chain('c2 rank %d frame %d' % (rank, fi), raw[fi].cpu().numpy(), out[fi], dark_h, flat_h, cvmaps)

    # ---- strong scaling: 256 frames in total over the N GPUs -----------------------------------------
    strong = None
    Fs = max(1, args.strong_total // world)
    if world > 1 and Fs <= F:
        for _ in range(2):
            eng.correct_batch(raw[:Fs], threshold=0.1, ksize=3, out=out[:Fs])
        barrier()
        ev0.record()
        for _ in range(args.steps):
            eng.correct_batch(raw[:Fs], threshold=0.1, ksize=3, out=out[:Fs])
        ev1.record()
        torch.cuda.synchronize()
        ms_s = rmax(ev0.elapsed_time(ev1))
        barrier()
        us_frame = ms_s * 1e3 / (args.steps * Fs)
        strong = {'total_frames': Fs * world, 'frames_per_gpu': Fs, 'ms_per_step': ms_s / args.steps,
                  'value': float(Fs) * world * H * W * args.steps / (ms_s * 1e-3) / 1e6, 'unit': 'Mpx/s',
                  'us_per_frame_per_gpu': us_frame, 'algorithmic_bytes_per_frame': 22.0 * H * W,
                  'frac': 22.0 * H * W / (us_frame * 1e-6) / 1e9 / peak, 'batched': True,
                  'frames_per_launch': min(args.group, Fs)}
    elif world == 1:
        strong = {'total_frames': F, 'frames_per_gpu': F, 'note': 'N = 1: identical to the headline measurement',
                  'ms_per_step': ms_total / args.steps, 'value': value, 'unit': 'Mpx/s', 'batched': True}

    # ---- end to end: host frames through the C-ABI host call ----------------------------------------
    pool = min(F, args.e2e_pool)
    h_in = engine.pinned_empty((pool, H, W), np.uint16)
    h_out = engine.pinned_empty((pool, H, W), np.float32)
    h_in[...] = raw[:pool].cpu().numpy()
    reps = max(1, F // pool)

    def e2e_step():
        for _ in range(reps):
            eng.correct_host(h_in, out=h_out, threshold=0.1, ksize=3)

    e2e_step()
    barrier()
    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    e2e_s = rmax(time.perf_counter() - t0)
    e2e_px_step = float(reps * pool) * H * W
    e2e_value = e2e_px_step * world * e2e_steps / e2e_s / 1e6
    for fi in sorted({0, pool - 1}):
        parity.chain('e2e rank %d frame %d' % (rank, fi), h_in[fi], h_out[fi], dark_h, flat_h, cvmaps)
    # the box's raw pinned-copy ceiling for this traffic mix, all ranks copying at the same time
    barrier()
    probe = pcie_probe(dev, H * W * 2 * 4, H * W * 4 * 4)
    barrier()
    ceil_both = rsum(probe['both'][0])
    ceil_h2d = rsum(probe['h2d'][0])
    ceil_d2h = rsum(probe['d2h'][0])
    e2e_gbs = e2e_value * 1e6 * 6.0 / 1e9                       # 2 B/px in + 4 B/px out
    del h_in, h_out

    k1_us = k1_ms * 1e3 / max(k1_frames, 1.0)
    k2_us = k2_ms * 1e3 / max(k2_frames, 1.0)
    achieved = K1_BYTES_PER_PX * H * W / (k1_us * 1e-6) / 1e9 if k1_us > 0 else 0.0
    k2_achieved = K2_BYTES_PER_PX * H * W / (k2_us * 1e-6) / 1e9 if k2_us > 0 else 0.0

    # ---- the other BASELINE configs ------------------------------------------------------------------
    configs = {}

    def record(name, desc, us, us_min, bytes_frame, frames_per_launch, batched, extra=None):
        us = rmax(us)
        r = {'workload': desc, 'us_per_frame': us, 'us_per_frame_min': us_min, 'algorithmic_bytes_per_frame': bytes_frame,
             'achieved_gbs': bytes_frame / (us * 1e-6) / 1e9, 'frac': bytes_frame / (us * 1e-6) / 1e9 / peak,
             'mpx_s': (extra or {}).get('px', 0) / us, 'frames_per_launch': frames_per_launch, 'batched': batched}
        if extra:
            r.update({k: v for k, v in extra.items() if k != 'px'})
        configs[name] = r

    if not args.no_configs:
        # c1: single 4096x3000 uint16 frame, K1 only (one frame per launch, rotating over 32 frames: 2.4 GB >> L2)
        n1 = min(F, 32)
        mid = out                                             # reuse the output buffer as K1's destination
        us, us_min = event_times_us(lambda i: eng.pointwise_median(raw[i % n1], 0.1, 3, out=mid[i % n1:i % n1 + 1]), 48)
        parity.k1('c1 rank %d' % rank, raw[0].cpu().numpy(), mid[0], dark_h, flat_h)
        record('c1_single_4096x3000_u16_k1', 'BASELINE configs[1]: ONE 4096x3000 uint16 frame per launch, dark + flat + 3x3 '
               'medianThreshold (K1 only)', us, us_min, K1_BYTES_PER_PX * H * W, 1, False, {'px': H * W})
        # the full chain one frame per call (the drop-in's single-frame path, device resident)
        us, us_min = event_times_us(lambda i: eng.correct_batch(raw[i % n1], 0.1, 3, out=out[i % n1:i % n1 + 1]), 48)
        record('c2_single_frame_chain', 'configs[2] frame, full chain, ONE frame per call (K1 + K2 launches of one frame)',
               us, us_min, 22.0 * H * W, 1, False, {'px': H * W})
        del mid
    del raw, out
    torch.cuda.empty_cache()

    def small_config(name, desc, h, w, dtype, lens_params, ksize, nrot, iters, raw_bytes):
        e = engine.Engine(h, w, local)
        d_h, f_h = synth.dark_map(h, w), synth.flat_map(h, w)
        e.set_dark(d_h)
        e.set_flat(f_h)
        maps = lens_setup(e, h, w, lens_params)
        r = synth.scene_torch(nrot, h, w, 2000 + rank, dev, dtype)
        o = torch.empty((nrot, h, w), dtype=torch.float32, device=dev)
        bytes_frame = (raw_bytes + 8.0 + 4.0 + 8.0) * h * w        # raw + dark + flat + K1 out | K2 src + dst
        us, us_min = event_times_us(lambda i: e.correct_batch(r[i % nrot], 0.1, ksize, out=o[i % nrot:i % nrot + 1]), iters)
        parity.chain('%s rank %d frame 0' % (name, rank), r[0].cpu().numpy(), o[0], d_h, f_h, maps, ksize)
        extra = {'px': h * w, 'rotating_frames': nrot}
        if nrot >= 4:
            e.set_option(_lib.OPT_CHAIN_GROUP, min(nrot, 32))
            usb, _ = event_times_us(lambda i: e.correct_batch(r, 0.1, ksize, out=o), 6, warm=2)
            extra['batched_us_per_frame'] = rmax(usb / nrot)
            extra['batched_frac'] = bytes_frame / (extra['batched_us_per_frame'] * 1e-6) / 1e9 / peak
            parity.chain('%s rank %d batch frame %d' % (name, rank, nrot - 1), r[nrot - 1].cpu().numpy(), o[nrot - 1], d_h, f_h, maps, ksize)
        record(name, desc, us, us_min, bytes_frame, 1, False, extra)
        e.close()
        del r, o
        torch.cuda.empty_cache()

    if not args.no_configs:
        small_config('c0_1024x1024_f32_chain', 'BASELINE configs[0]: ONE 1024x1024 float32 frame per call, full chain (dark + flat + 3x3 '
                     'medianThreshold + moderate lens); rotating over 64 frames (512 MB of raw + output)', 1024, 1024, 'float32',
                     synth.lens_moderate(1024, 1024), 3, 64, 64, 4.0)
        small_config('c3_8192x8192_f32_5x5_strong_lens', 'BASELINE configs[3]: ONE 8192x8192 float32 frame per call, dark + flat + 5x5 '
                     'medianThreshold + strong radial/tangential lens; rotating over 4 frames', 8192, 8192, 'float32',
                     synth.lens_strong(8192, 8192), 5, 4, 12, 4.0)

        # c4: 6000x4000 uint16 frames streamed from a pool of 16 pinned buffers through the host-buffer chain
        h4, w4, pool4 = 4000, 6000, 16
        e4 = engine.Engine(h4, w4, local)
        d4, f4 = synth.dark_map(h4, w4), synth.flat_map(h4, w4)
        e4.set_dark(d4)
        e4.set_flat(f4)
        maps4 = lens_setup(e4, h4, w4, synth.lens_moderate(h4, w4))
        r4 = synth.scene_torch(pool4, h4, w4, 3000 + rank, dev, 'uint16')
        hin4 = engine.pinned_empty((pool4, h4, w4), np.uint16)
        hout4 = engine.pinned_empty((pool4, h4, w4), np.float32)
        hin4[...] = r4.cpu().numpy()
        o4 = torch.empty((pool4, h4, w4), dtype=torch.float32, device=dev)
        e4.set_option(_lib.OPT_CHAIN_GROUP, 16)
        usk, _ = event_times_us(lambda i: e4.correct_batch(r4, 0.1, 3, out=o4), 6, warm=2)
        kern_us = rmax(usk / pool4)
        e4.correct_host(hin4, out=hout4, threshold=0.1, ksize=3)
        cycles = max(1, args.c4_frames // pool4)
        barrier()
        t0 = time.perf_counter()
        for _ in range(cycles):
            e4.correct_host(hin4, out=hout4, threshold=0.1, ksize=3)
        t4 = rmax(time.perf_counter() - t0)
        nfr = cycles * pool4
        for fi in (0, pool4 - 1):
            parity.chain('c4 rank %d frame %d' % (rank, fi), hin4[fi], hout4[fi], d4, f4, maps4)
        barrier()
        probe4 = pcie_probe(dev, h4 * w4 * 2 * 2, h4 * w4 * 4 * 2)
        barrier()
        per_frame_us = t4 / nfr * 1e6
        in_b, out_b = h4 * w4 * 2.0, h4 * w4 * 4.0
        h2d_us = in_b / (probe4['h2d'][0] * 1e9) * 1e6
        d2h_us = out_b / (probe4['d2h'][0] * 1e9) * 1e6
        slowest = max(h2d_us, d2h_us, kern_us)
        serial = h2d_us + d2h_us + kern_us
        ceil4 = rsum(probe4['both'][0])
        gbs4 = (in_b + out_b) * nfr * world / t4 / 1e9
        configs['c4_6000x4000_u16_streamed'] = {
            'workload': 'BASELINE configs[4]: 6000x4000 uint16 frames streamed from a pool of %d pinned host buffers per GPU through '
                        'imgcorr_correct_host (H2D, K1 + K2, D2H on three streams), %d frames per GPU in the timed region '
                        '(the config names 4096: the pool is cycled, the rate is steady after the first cycle)' % (pool4, nfr),
            'frames_per_s': nfr * world / t4, 'mpx_s': nfr * world * h4 * w4 / t4 / 1e6, 'us_per_frame_per_gpu': per_frame_us,
            'pcie_gbs_achieved': gbs4, 'pcie_ceiling_gbs': ceil4, 'frac_of_ceiling': gbs4 / ceil4 if ceil4 > 0 else None,
            'stage_us_per_frame': {'h2d_alone': h2d_us, 'kernels_device_resident': kern_us, 'd2h_alone': d2h_us},
            'overlap_pct': 100.0 * (serial - per_frame_us) / (serial - slowest) if serial > slowest else None,
            'overlap_note': '100 % = the pipeline runs at the speed of its slowest stage (copies of one direction alone), 0 % = the three '
                            'stages run one after the other; with both directions active the link itself gives less than either alone',
            'kernel_frac_of_hbm_peak': 22.0 * h4 * w4 / (kern_us * 1e-6) / 1e9 / peak,
        }
        e4.close()
        del r4, o4, hin4, hout4
        torch.cuda.empty_cache()

    bad = rsum(len(parity.failures))
    nb = rsum(parity.bands)
    npx = rsum(parity.pixels)
    parity_line = 'ok' if bad == 0 else 'FAILED'

    if rank == 0:
        line = {
            'metric': METRIC, 'value': value, 'unit': 'Mpx/s', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': ms_total / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f32', 'data': 'synthetic', 'config': workload_config(F, world),
            'clocks': clocks.summary(),
            'parity_check': parity_line,
            'parity_detail': {'bands_checked': int(nb), 'pixels_checked': int(npx), 'ranks': world,
                              'failures': parity.failures[:8] if bad else [],
                              'what': 'bit-exact against the float32 oracle chain (oracle/bands.py, cv2 maps): 3 bands of 48 rows of the '
                                      'first and last frame of every measured output (headline shard, e2e pool, c0, c1, c3, c4), every rank'},
            'e2e': {'value': e2e_value, 'unit': 'Mpx/s', 'h2d_bytes_per_step': int(reps * pool * H * W * 2),
                    'd2h_bytes_per_step': int(reps * pool * H * W * 4), 'frames_per_step_per_gpu': reps * pool,
                    'steps': e2e_steps, 'pinned_pool_frames': pool, 'result_dtype': 'float32 (the north star\'s arithmetic; the '
                    'drop-in CameraCalibration.correct() widens to float64 on the host side, outside this number)',
                    'api': 'imgcorr_correct_host (C ABI) with pinned host buffers; copies inside the timed region',
                    'pcie_gbs_achieved': e2e_gbs, 'pcie_ceiling_gbs': ceil_both, 'frac_of_ceiling': e2e_gbs / ceil_both if ceil_both else None,
                    'pcie_ceiling_detail': {'h2d_alone_gbs': ceil_h2d, 'd2h_alone_gbs': ceil_d2h, 'both_directions_gbs': ceil_both,
                                            'how': 'raw cudaMemcpyAsync of page-locked buffers (4 frames in, 4 frames out per round, two '
                                                   'streams), all %d ranks at the same time, summed over ranks' % world},
                    'host_numa_binding': numa},
            'gpu_launches': int(launches),
            'roofline': {'bound': 'hbm', 'kernel': 'K1 k1_stream_kernel (fused dark/flat/nan_to_num/3x3 median-threshold)',
                         'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak, 'traffic': args.k1_traffic,
                         'peak_source': peak_src, 'algorithmic_bytes_per_px': K1_BYTES_PER_PX,
                         'us_per_frame': k1_us, 'frames_timed': k1_frames, 'frames_per_launch': min(args.group, F),
                         'launch_us': k1_us * min(args.group, F),
                         'algorithmic_bytes_per_launch': K1_BYTES_PER_PX * H * W * min(args.group, F),
                         'k2': {'achieved': k2_achieved, 'frac': k2_achieved / peak, 'us_per_frame': k2_us,
                                'algorithmic_bytes_per_px': K2_BYTES_PER_PX},
                         'chain_frac': (K1_BYTES_PER_PX + K2_BYTES_PER_PX) * H * W / ((k1_us + k2_us) * 1e-6) / 1e9 / peak
                                       if k1_us + k2_us > 0 else 0.0,
                         'chain_overlap': bool(args.overlap),
                         'note': 'K1 reads dark / flat from DRAM once per launch (frame pairs of one strip run back to back, the maps '
                                 'stay in L2): its DRAM traffic (`traffic`, ncu) is below the algorithmic bytes, so `frac` can exceed 1',
                         'timing_note': 'K1 / K2 durations are event-bracketed launches inside the timed region; with chain_overlap '
                                        'the bracketed frame groups run unoverlapped (kernel alone), the others overlap K1 of group '
                                        'g+1 with K2 of group g, so ms_per_step can be below frames * (K1 + K2)'},
            'configs': configs,
            'strong_scaling': strong,
        }
        if world == 1 and not args.no_cpu_baseline:
            line['cpu_baseline'] = cpu_baseline_single()
        print(json.dumps(line), flush=True)
    if distributed:
        dist.barrier(device_ids=[local])
        dist.destroy_process_group()
    if bad:
        sys.stderr.write('bench.py: PARITY CHECK FAILED on rank %d: %s\n' % (rank, '; '.join(parity.failures[:8])))
        raise SystemExit(1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--frames', type=int, default=256, help='frames per GPU per step')
    ap.add_argument('--group', type=int, default=32, help='frames per K1/K2 launch inside the chain')
    ap.add_argument('--overlap', type=int, default=1, help='1 (library default): K1 of the next group overlaps K2 of the current one')
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--e2e-pool', type=int, default=32, help='pinned host frames cycled by the end-to-end leg')
    ap.add_argument('--e2e-steps', type=int, default=3)
    ap.add_argument('--host-slots', type=int, default=0, help='depth of the pinned / device staging ring of the host-buffer pipeline (0 = library default)')
    ap.add_argument('--strong-total', type=int, default=256, help='frames in total for the strong-scaling point')
    ap.add_argument('--c4-frames', type=int, default=256, help='6000x4000 frames streamed per GPU in the timed region of c4')
    ap.add_argument('--no-configs', action='store_true', help='headline only (skip c0 / c1 / c3 / c4)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the last timed step\'s output (rank 0) as .npy files into DIR')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs needs --impl ours')
    if args.gpus > 1 and 'WORLD_SIZE' not in os.environ and args.impl == 'ours':
        # started as plain `python bench.py --gpus N`: relaunch under torchrun, one rank per GPU (the driver does this itself)
        import socket
        with socket.socket() as sk:
            sk.bind(('127.0.0.1', 0))
            port = sk.getsockname()[1]
        os.execv(sys.executable, [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', str(args.gpus),
                                  '--master-addr', '127.0.0.1', '--master-port', str(port), os.path.abspath(__file__)] + sys.argv[1:])
    if 'WORLD_SIZE' in os.environ and int(os.environ['WORLD_SIZE']) != args.gpus and args.impl == 'ours':
        raise SystemExit('bench.py: --gpus %d but WORLD_SIZE=%s' % (args.gpus, os.environ['WORLD_SIZE']))
    args.k1_traffic = None
    try:        # dram__bytes_read.sum + dram__bytes_write.sum of one K1 launch from the committed ncu --set full capture
        with open(os.path.join(ROOT, 'profiles', 'roofline_traffic.json')) as f:
            t = json.load(f)
        if int(t['frames_per_launch']) == args.group:          # the capture is of a launch of that many frames
            args.k1_traffic = float(t['k1_dram_bytes_per_launch'])
    except Exception:
        pass
    if args.warmup < 3 and args.impl == 'ours':
        args.warmup = 3
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
